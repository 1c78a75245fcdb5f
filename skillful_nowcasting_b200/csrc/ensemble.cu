// Ensemble statistics of K-member forecasts in one pass over the ensemble (include/dgmr_b200.h: dgmr_ensemble_stats).
//
// One CTA owns the 16-row band [16*band, 16*band + 16) x [0, W) of one (b, t*C + c) frame and walks it in 16x16 tiles.  Thread t of a
// tile holds pixel (4*(w/4) + p/4, 4*(w%4) + p%4) with w = t/16, p = t%16, so the 16 threads of each 4x4 window are consecutive; a warp
// reads 4 rows x 8 columns of every member (4 full 32-byte sectors).  Each thread loads its pixel's K member values into registers once,
// writes the mean and the exceedance fractions, and (with a target) the pixel CRPS from the register-sorted members.  The members are
// also staged in shared memory, from which the pooled member values of the 16 4x4 windows and the 16x16 window of the tile are formed;
// threads 0..33 then evaluate the 34 pooled cells (avg 4x4, max 4x4, avg 16x16, max 16x16) the same way.  CRPS sums are fp64, reduced in
// a fixed order per CTA into ws[frame][band][5]; a second launch sums the bands of every frame in order: results are bitwise repeatable.
#include "common.cuh"

#include <float.h>

namespace dgmr {

constexpr int ENS_TILE = 16;            // tile edge = largest pooling window
constexpr int ENS_PIX = ENS_TILE * ENS_TILE;
constexpr int ENS_MAX_K = 64;
constexpr int ENS_MAX_THR = 8;
constexpr int ENS_SCALES = 5;           // 1, avg 4x4, max 4x4, avg 16x16, max 16x16
constexpr int ENS_XS_LD = ENS_PIX + 4;  // member rows of the staged tile: +4 floats keeps the float4 window reads conflict-free

// ascending bitonic sort of KM register values (fully unrolled: stays in registers)
template <int KM>
__device__ __forceinline__ void sort_regs(float (&x)[KM]) {
#pragma unroll
  for (int k = 2; k <= KM; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
      for (int i = 0; i < KM; ++i) {
        const int l = i ^ j;
        if (l > i) {
          const float a = x[i], b = x[l];
          const bool up = (i & k) == 0;
          x[i] = up ? fminf(a, b) : fmaxf(a, b);
          x[l] = up ? fmaxf(a, b) : fminf(a, b);
        }
      }
    }
  }
}

// CRPS of one cell: (1/K) sum_k |x_k - y| - (1/K^2) sum_i (2i - K + 1) x_(i)   (x sorted in place; entries >= K are +FLT_MAX pads)
template <int KM>
__device__ __forceinline__ double cell_crps(float (&x)[KM], int K, float y) {
  double a = 0.0;
#pragma unroll
  for (int k = 0; k < KM; ++k)
    if (k < K) a += fabs((double)x[k] - (double)y);
  sort_regs<KM>(x);
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < KM; ++i)
    if (i < K) s += (double)(2 * i - K + 1) * (double)x[i];
  return a / K - s / ((double)K * K);
}

template <int KM>
__global__ void __launch_bounds__(ENS_PIX, 2) ensemble_stats_kernel(const float* __restrict__ ens, const float* __restrict__ target,
                                                                 const float* __restrict__ thr, int n_thr, float* __restrict__ mean,
                                                                 float* __restrict__ prob, double* __restrict__ ws, int B, int K, int TC,
                                                                 int H, int W) {
  extern __shared__ float smem[];
  float* xs = smem;                                  // [K][ENS_XS_LD]   (target only)
  float* pool4 = xs + (size_t)K * ENS_XS_LD;         // [2][16][K]       window sums / maxima per member
  float* pool16 = pool4 + 2 * 16 * K;                // [2][K]
  float* ys = pool16 + 2 * K;                        // [ENS_PIX]
  float* ypool = ys + ENS_PIX;                       // [2][16 + 1]
  __shared__ float s_thr[ENS_MAX_THR];
  __shared__ double s_red[ENS_PIX / 32][ENS_SCALES];

  const int t = threadIdx.x;
  const int band = blockIdx.x, tc = blockIdx.y, b = blockIdx.z;
  if (t < n_thr) s_thr[t] = thr[t];
  __syncthreads();
  const int64_t P = (int64_t)TC * H * W;
  const int64_t frame = (int64_t)tc * H * W;
  const float* e0 = ens + (int64_t)b * K * P + frame;  // member k: e0 + k * P
  const int win = t >> 4, p = t & 15;
  const int row = band * ENS_TILE + (win >> 2) * 4 + (p >> 2);
  const int tiles = (W + ENS_TILE - 1) / ENS_TILE;
  double acc[ENS_SCALES] = {0.0, 0.0, 0.0, 0.0, 0.0};

  for (int tile = 0; tile < tiles; ++tile) {
    const int col = tile * ENS_TILE + (win & 3) * 4 + (p & 3);
    const bool valid = row < H && col < W;
    const int64_t pix = (int64_t)row * W + col;
    float x[KM];
#pragma unroll
    for (int k = 0; k < KM; ++k) x[k] = (valid && k < K) ? __ldg(e0 + (int64_t)k * P + pix) : FLT_MAX;
    if (valid) {
      float s = 0.0f;
#pragma unroll
      for (int k = 0; k < KM; ++k)
        if (k < K) s += x[k];                        // member order
      const int64_t o = (int64_t)b * P + frame + pix;
      mean[o] = s / (float)K;
      for (int i = 0; i < n_thr; ++i) {
        int c = 0;
#pragma unroll
        for (int k = 0; k < KM; ++k)
          if (k < K) c += x[k] >= s_thr[i];
        prob[(int64_t)i * B * P + o] = (float)c / (float)K;
      }
    }
    if (target == nullptr) continue;                 // (uniform over the CTA: no barrier is skipped by a subset of threads)

    // ---- CRPS (the caller guarantees H, W multiples of 16: every thread holds a valid pixel)
    const float y = __ldg(target + (int64_t)b * P + frame + pix);
#pragma unroll
    for (int k = 0; k < KM; ++k)
      if (k < K) xs[k * ENS_XS_LD + t] = x[k];
    ys[t] = y;
    acc[0] += cell_crps<KM>(x, K, y);
    __syncthreads();
    // member pools of the 16 4x4 windows: (window, member) pairs over the CTA, four float4 reads of the window's 16 values each
    for (int q = t; q < 16 * K; q += ENS_PIX) {
      const int w = q / K, k = q - w * K;
      const float4* v = reinterpret_cast<const float4*>(xs + k * ENS_XS_LD + w * 16);
      float s = 0.0f, m = -FLT_MAX;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 f = v[i];
        s += (f.x + f.y) + (f.z + f.w);
        m = fmaxf(m, fmaxf(fmaxf(f.x, f.y), fmaxf(f.z, f.w)));
      }
      pool4[w * K + k] = s;
      pool4[(16 + w) * K + k] = m;
    }
    if (t < 16) {
      float s = 0.0f, m = -FLT_MAX;
      for (int i = 0; i < 16; ++i) { const float v = ys[t * 16 + i]; s += v; m = fmaxf(m, v); }
      ypool[t] = s;
      ypool[17 + t] = m;
    }
    __syncthreads();
    for (int k = t; k < K; k += ENS_PIX) {
      float s = 0.0f, m = -FLT_MAX;
      for (int w = 0; w < 16; ++w) { s += pool4[w * K + k]; m = fmaxf(m, pool4[(16 + w) * K + k]); }
      pool16[k] = s;
      pool16[K + k] = m;
    }
    if (t == 0) {
      float s = 0.0f, m = -FLT_MAX;
      for (int w = 0; w < 16; ++w) { s += ypool[w]; m = fmaxf(m, ypool[17 + w]); }
      ypool[16] = s;
      ypool[33] = m;
    }
    __syncthreads();
    // the 34 pooled cells of the tile, one per thread of the first two warps (sums / 16 and / 256 are exact scalings)
    if (t < 34) {
      const float* src;
      float scale, yc;
      int slot;
      if (t < 16) { src = pool4 + t * K; scale = 1.0f / 16; yc = ypool[t] * scale; slot = 1; }
      else if (t < 32) { src = pool4 + t * K; scale = 1.0f; yc = ypool[17 + t - 16]; slot = 2; }
      else if (t == 32) { src = pool16; scale = 1.0f / 256; yc = ypool[16] * scale; slot = 3; }
      else { src = pool16 + K; scale = 1.0f; yc = ypool[33]; slot = 4; }
#pragma unroll
      for (int k = 0; k < KM; ++k) x[k] = k < K ? src[k] * scale : FLT_MAX;
      const double c = cell_crps<KM>(x, K, yc);
#pragma unroll
      for (int i = 1; i < ENS_SCALES; ++i) acc[i] += i == slot ? c : 0.0;   // (static indices: acc stays in registers)
    }
    __syncthreads();                                 // the next tile overwrites the staged members
  }
  if (target == nullptr) return;
  // fixed-order CTA reduction of the five partial sums
  const int lane = t & 31, wid = t >> 5;
#pragma unroll
  for (int s = 0; s < ENS_SCALES; ++s) {
    const double v = warp_sum_d(acc[s]);
    if (lane == 0) s_red[wid][s] = v;
  }
  __syncthreads();
  if (t < ENS_SCALES) {
    double v = 0.0;
    for (int w = 0; w < ENS_PIX / 32; ++w) v += s_red[w][t];
    ws[(((int64_t)b * TC + tc) * gridDim.x + band) * ENS_SCALES + t] = v;
  }
}

// crps[frame][s] = sum over the bands of frame (in band order) / number of cells at scale s
__global__ void ensemble_crps_final_kernel(const double* __restrict__ ws, float* __restrict__ crps, int frames, int bands, int H, int W) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= frames * ENS_SCALES) return;
  const int f = i / ENS_SCALES, s = i - f * ENS_SCALES;
  double v = 0.0;
  for (int bd = 0; bd < bands; ++bd) v += ws[((int64_t)f * bands + bd) * ENS_SCALES + s];
  const double cells = (double)H * W / (s == 0 ? 1.0 : s <= 2 ? 16.0 : 256.0);
  crps[i] = (float)(v / cells);
}

template <int KM>
static int launch_ensemble(const float* ens, const float* target, const float* thr, int n_thr, float* mean, float* prob, double* ws, int B,
                           int K, int TC, int H, int W, cudaStream_t st) {
  const size_t smem = target ? sizeof(float) * ((size_t)K * ENS_XS_LD + 2 * 16 * K + 2 * K + ENS_PIX + 2 * 17) : 0;
  if (smem > 48 * 1024) DGMR_CUDA(cudaFuncSetAttribute(ensemble_stats_kernel<KM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const dim3 grid((unsigned)((H + ENS_TILE - 1) / ENS_TILE), (unsigned)TC, (unsigned)B);
  ensemble_stats_kernel<KM><<<grid, ENS_PIX, smem, st>>>(ens, target, thr, n_thr, mean, prob, ws, B, K, TC, H, W);
  DGMR_CHECK_LAUNCH("dgmr_ensemble_stats");
  return 0;
}

}  // namespace dgmr

using namespace dgmr;

extern "C" {

int dgmr_ensemble_stats(const float* ens, const float* target, const float* thr, int n_thr, float* mean, float* prob, float* crps, double* ws,
                        int B, int K, int T, int C, int H, int W, dgmr_stream_t stream) {
  DGMR_REQUIRE(B > 0 && T > 0 && C > 0 && H > 0 && W > 0, "dgmr_ensemble_stats: bad dims B=%d T=%d C=%d H=%d W=%d", B, T, C, H, W);
  DGMR_REQUIRE(K >= 1 && K <= ENS_MAX_K, "dgmr_ensemble_stats: K = %d members (1 <= K <= %d)", K, ENS_MAX_K);
  DGMR_REQUIRE(n_thr >= 0 && n_thr <= ENS_MAX_THR, "dgmr_ensemble_stats: n_thr = %d thresholds (at most %d)", n_thr, ENS_MAX_THR);
  DGMR_REQUIRE(ens && mean, "dgmr_ensemble_stats: ens and mean are required");
  DGMR_REQUIRE(n_thr == 0 || (thr && prob), "dgmr_ensemble_stats: thresholds need thr and prob");
  DGMR_REQUIRE((int64_t)T * C <= 65535 && B <= 65535, "dgmr_ensemble_stats: T*C and B must be <= 65535");
  if (target) {
    DGMR_REQUIRE(crps && ws, "dgmr_ensemble_stats: a target needs crps and ws");
    DGMR_REQUIRE(H % ENS_TILE == 0 && W % ENS_TILE == 0, "dgmr_ensemble_stats: CRPS needs H and W multiples of 16 (got %d x %d)", H, W);
  }
  const int TC = T * C;
  cudaStream_t st = S(stream);
  int rc;
  if (K <= 8) rc = launch_ensemble<8>(ens, target, thr, n_thr, mean, prob, ws, B, K, TC, H, W, st);
  else if (K <= 16) rc = launch_ensemble<16>(ens, target, thr, n_thr, mean, prob, ws, B, K, TC, H, W, st);
  else if (K <= 32) rc = launch_ensemble<32>(ens, target, thr, n_thr, mean, prob, ws, B, K, TC, H, W, st);
  else rc = launch_ensemble<64>(ens, target, thr, n_thr, mean, prob, ws, B, K, TC, H, W, st);
  if (rc || !target) return rc;
  const int frames = B * TC;
  ensemble_crps_final_kernel<<<(unsigned)ceil_div((int64_t)frames * ENS_SCALES, 256), 256, 0, st>>>(ws, crps, frames, H / ENS_TILE, H, W);
  DGMR_CHECK_LAUNCH("dgmr_ensemble_crps_final");
  return 0;
}

}  // extern "C"
