/*
 * dgmr_b200.h -- C ABI of the B200-native DGMR hot path (libdgmr_b200.so).
 *
 * Drop-in boundary (SURVEY.md 8b): the reference has no native code; its hot path is the
 * PyTorch op call sites listed in SURVEY.md 2.2.  Each entry point below replaces one family
 * of those call sites and cites it (paths relative to the reference repo root, `ref:`).
 * The Python package `skillful_nowcasting_b200` binds these with ctypes (see INTEGRATION.md)
 * and mirrors the reference's module API (DGMR, Generator, Sampler, ... dgmr/__init__.py:3-6).
 *
 * Conventions
 *  - All pointers are DEVICE pointers owned by the caller (PyTorch allocates everything,
 *    including workspaces); the library never allocates or frees caller-visible memory.
 *  - Activations are fp32, channels-last: [N, D, H, W, C] contiguous (2-D convs: D == 1).
 *    "Groups" G: the N images are G consecutive groups of N/G images; a group is one
 *    *reference call* (one timestep / one frame).  Per-call quantities of the reference
 *    (spectral-norm sigma, BatchNorm batch statistics) are per group here, which is how the
 *    T calls of e.g. `[self.g1(h) for h in hidden_states]` (ref: dgmr/generators.py:154)
 *    run as ONE launch with identical results.
 *  - Every function is asynchronous on `stream` (a cudaStream_t), never synchronises the host,
 *    returns 0 on success and a non-zero code on error; dgmr_last_error() gives the message
 *    (thread-local).  Nothing aborts.
 *  - Conv weights are consumed "packed": [tap][Cout][Cin] fp32 (tap = (kd*KH + kh)*KW + kw),
 *    produced from the state-dict OIHW tensor by dgmr_pack_weight.
 */
#ifndef DGMR_B200_H
#define DGMR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dgmr_stream_t; /* cudaStream_t */

enum { DGMR_ACT_NONE = 0, DGMR_ACT_RELU = 1 };
/* OR-able flag: round the produced tensor-core operand (packed weights in dgmr_pack_weight's `mode`, dz in
 * dgmr_conv_bwd_prep's `act`) to the nearest TF32 value.  tcgen05 kind::tf32 ignores the low 13 mantissa bits of its
 * fp32 operands (truncation, biased); feeding it round-to-nearest values gives the unbiased rounding cuDNN applies
 * for the reference's TF32 convolutions. */
enum { DGMR_FLAG_ROUND_TF32 = 256 };
/* OR-able into dgmr_conv_fwd's `act`: y += conv(x, wp) * scale  (bias, res must be NULL, act NONE; y pre-initialised by the
 * caller, e.g. with the residual).  The tensor-core path then splits the K loop over filter taps across CTAs (fp32 red.add
 * into y), which is what fills the SMs for the small-M, large-K convolutions of the ConvGRU steps. */
enum { DGMR_FLAG_ACCUMULATE = 512 };
/* OR-able into dgmr_conv_fwd's `act`: y is written TF32-rounded (round-to-nearest) -- for outputs that feed tensor-core convolutions
 * only, instead of a separate dgmr_round_tf32 pass over them. */
enum { DGMR_FLAG_ROUND_OUT = 1024 };
/* OR-able into dgmr_conv_fwd's `act`: `res` is a HALF-resolution tensor [N, D, H/2, W/2, Cout] and is added nearest-upsampled, i.e. read
 * at (h/2, w/2): the shortcut of UpsampleGBlock, conv1x1(up2(x)) = up2(conv1x1(x)) (ref: dgmr/common.py:141-143), without ever
 * materialising the upsampled tensor.  H and W must be even. */
enum { DGMR_FLAG_RES_UP2 = 2048 };
/* conv algorithm selector */
enum { DGMR_ALGO_AUTO = 0, DGMR_ALGO_SIMT = 1, DGMR_ALGO_UMMA = 2 /* plain tcgen05 kernel */, DGMR_ALGO_UMMA_PATCH = 3 /* halo-patch tcgen05 kernel */,
       DGMR_ALGO_UMMA_KWSTACK = 4 /* narrow outputs: column taps stacked along N (conv_kwstack.cu) */,
       DGMR_ALGO_UMMA_PAIR = 5 /* persistent whole-row tiles, CTA pairs sharing each weight tile (conv_kwstack.cu, STACK = false) */ };
/* tensor-core operand precision: 1xTF32 (what cuDNN does by default for the reference) or
 * 3xTF32 error-compensated (hi*hi + hi*lo + lo*hi), ~fp32 accuracy */
enum { DGMR_PREC_TF32 = 0, DGMR_PREC_3XTF32 = 1 };

const char* dgmr_last_error(void);
int dgmr_abi_version(void);
/* 1 if the tcgen05/TMA implicit-GEMM path can serve this conv shape (else the SIMT kernel is used) */
int dgmr_conv_umma_supported(int N, int D, int H, int W, int Cin, int Cout, int kd, int kh, int kw);
int dgmr_wgrad_umma_supported(int N, int D, int H, int W, int Cin, int Cout, int kd, int kh, int kw);

/* Process-wide tuning / test options of the tensor-core launchers (-1 restores the heuristic default): "umma_cg", "umma_persist",
 * "umma_persist_r", "patch_pair", "patch_mt", "patch_tg", "prefer_patch" (1: AUTO dispatch uses the halo-patch kernel for every
 * shape it supports -- lets small parity cases exercise the kernels the benchmark shapes use).  Not a per-launch argument on
 * purpose: results never depend on them, only which kernel variant computes them. */
int dgmr_set_option(const char* name, int value);

/* debug probe (tests only): C[128][N] = A[r0:r0+128, 0:32] . B[N, 0:32]^T through TMA + tcgen05 with the A descriptor
 * starting r0 rows into a swizzled 256-row tile; mode bit0 sets the descriptor base_offset field */
int dgmr_debug_umma_shift(const float* A, const float* B, float* C, int N, int r0, int mode, dgmr_stream_t stream);
/* tuning probe: cycles per kind::tf32 MMA (M=128, N, K=8) issued by one thread per CTA; mode 0 back to back, 1 commit per 8, 2 commit+wait per 8;
 * shift_rows: the A descriptor starts that many 128-byte rows into the swizzled tile (the halo-patch kernels' tap offsets) */
int dgmr_debug_umma_rate(float* out, int blocks, int N, int iters, int mode, int shift_rows, dgmr_stream_t stream);

/* ---- layout: generic strided gather  dst[i0..] (+)= src[i0..]
 * replaces ref: PixelUnshuffle/PixelShuffle (dgmr/common.py:326,393; generators.py:123,178;
 * discriminators.py:69,166), einops rearrange "b t c h w -> b (c t) h w" (common.py:423),
 * torch.cat / torch.stack / permute (ConvGRU.py:69,78; discriminators.py:110,116), and the
 * NCHW<->NHWC transposes at the module boundary.  Pure index permutation: bit-exact. */
int dgmr_permute(const float* src, float* dst, int ndim, const int64_t* shape,
                 const int64_t* src_strides, const int64_t* dst_strides, int accumulate,
                 dgmr_stream_t stream);

/* y[a][c] (+)= sum_r x[a][r][c]   (ref: torch.sum over stacked frame scores, discriminators.py:229-231,
 * 135-137; backward of the latent batch-repeat generators.py:146-148) */
int dgmr_reduce_mid(const float* x, float* y, int64_t A, int64_t R, int64_t C, int accumulate, dgmr_stream_t stream);

/* ---- pointwise */
/* out = a*x + b*y (y may be NULL) ; ref: residual adds, torch.stack(...).mean(0) (dgmr/dgmr.py:180) */
int dgmr_axpby(float a, const float* x, float b, const float* y, float* out, int64_t n, dgmr_stream_t stream);
int dgmr_fill(float* x, float value, int64_t n, dgmr_stream_t stream);
/* ref: torch.nn.ReLU / F.relu (dgmr/common.py:229-233) */
int dgmr_relu_fwd(const float* x, float* y, int64_t n, dgmr_stream_t stream);
int dgmr_relu_bwd(const float* dy, const float* x, float* dx, int64_t n, dgmr_stream_t stream);
/* sum-pool with window (pd,ph,pw) in {1,2}, floor output dims, times `scale`.
 * scale=1/(pd*ph*pw): AvgPool2d/3d forward (ref: dgmr/common.py:189-191, discriminators.py:68,165);
 * scale=1: backward of nearest Upsample. */
int dgmr_pool_sum(const float* x, float* y, int N, int D, int H, int W, int C, int pd, int ph, int pw,
                  float scale, dgmr_stream_t stream);
/* nearest replicate by (ud,uh,uw) times `scale`, x:[N,D,H,W,C] -> y:[N,D*ud,H*uh,W*uw,C] (output dims
 * Do,Ho,Wo given explicitly so floor-pooled odd sizes back-propagate zeros to the dropped rim).
 * scale=1: Upsample(nearest) forward (ref: dgmr/common.py:121,142,148); scale=1/window: AvgPool backward. */
int dgmr_upsample(const float* x, float* y, int N, int D, int H, int W, int C, int ud, int uh, int uw,
                  int Do, int Ho, int Wo, float scale, dgmr_stream_t stream);

/* ---- ConvGRU gate arithmetic (ref: dgmr/layers/ConvGRU.py:72-82); `ld` = row pitch (floats) of the
 * pre-activation tensors so that r|u can live side by side in one [rows, 2*Ch] conv output. */
/* flags & DGMR_FLAG_ROUND_TF32: rh (a conv-only operand) is emitted tf32-rounded.
 * x_r (nullable, pitch ld): the input-dependent part of the pre-activation (ConvGRU.py:66-70: the conv over cat(x, h) split by input
 * channels); when given, pre_r holds only the h part, the sum is formed here AND written back to pre_r (the backward reads it). */
int dgmr_gru_gate_fwd(float* pre_r, int ld, const float* x_r, const float* h, float* rh, int64_t rows, int Ch, int flags, dgmr_stream_t stream);
/* relu_c != 0: `c` holds the candidate pre-activation and relu is applied here (ref: ConvGRU.py:81) */
/* hnew_tf32 (nullable): tf32-rounded copy of hnew = the next step's conv operand */
/* x_u (pitch ld) / x_c (dense), nullable: as x_r above, for the update gate and the candidate; pre_u / c are completed in place */
int dgmr_gru_blend_fwd(float* pre_u, int ld, const float* x_u, const float* h, float* c, const float* x_c, float* hnew, float* hnew_tf32,
                       int64_t rows, int Ch, int relu_c, dgmr_stream_t stream);
/* d_rh -> d_pre_r, dh (+= if accumulate).  dz_scale [Ch] / dz (nullable, leading dimension ldd like d_pre_r): additionally dz = d_pre_r * dz_scale[c]
 * (tf32-rounded if dz_round) -- the recurrent convolution's backward operand, so the walk over the steps needs no dgmr_conv_bwd_prep per step */
int dgmr_gru_gate_bwd(const float* d_rh, const float* pre_r, int ld, const float* h, float* d_pre_r, int ldd,
                      float* dh, int accumulate, int64_t rows, int Ch, const float* dz_scale, float* dz, int dz_round, dgmr_stream_t stream);
/* d_hnew -> d_pre_u, dc, dh (+= if accumulate); dz_u (ldd) = d_pre_u * dz_u_scale[c], dz_c (contiguous) = dc * dz_c_scale[c] as above (nullable) */
int dgmr_gru_blend_bwd(const float* d_hnew, const float* pre_u, int ld, const float* h, const float* c,
                       float* d_pre_u, int ldd, float* dc, float* dh, int accumulate,
                       int64_t rows, int Ch, int relu_c, const float* dz_u_scale, float* dz_u, const float* dz_c_scale, float* dz_c, int dz_round,
                       dgmr_stream_t stream);

/* ---- BatchNorm (ref: BatchNorm2d dgmr/common.py:38-39,108-109, generators.py:113; BatchNorm1d
 * discriminators.py:102,194).  x: [G*rows, C]; batch statistics per (group, channel). */
int dgmr_bn_stats(const float* x, double* sums /*[G][C][2], zeroed inside*/, int64_t rows, int G, int C, dgmr_stream_t stream);
/* training: mean/var from sums, running stats updated sequentially over g (momentum, unbiased var);
 * eval: running stats.  Outputs mean,invstd,a,b : [G][C], y = a*x + b. */
int dgmr_bn_finalize(const double* sums, const float* gamma, const float* beta, float* running_mean,
                     float* running_var, int64_t rows, int G, int C, float eps, float momentum, int training,
                     float* mean, float* invstd, float* a, float* b, dgmr_stream_t stream);
/* y = act(a[g,c]*x + b[g,c]); if up2: x is [G*Ng, H, W, C] and y is [G*Ng, 2H, 2W, C] (nearest).
 * relu | DGMR_FLAG_ROUND_TF32: y is written tf32-rounded (it feeds tensor-core convolutions only).
 * x_rounded (nullable, not with up2): the tf32-rounded copy of x itself, for x's OTHER consumer in a residual block (the 1x1 shortcut
 * convolution, ref: dgmr/common.py:71-74,140-143) -- written by the pass that reads x anyway instead of by a separate rounding pass. */
int dgmr_bn_apply(const float* x, const float* a, const float* b, float* y, float* x_rounded, int64_t rows, int G, int C,
                  int relu, int up2, int H, int W, dgmr_stream_t stream);
/* red[g][c] = (sum dpre, sum dpre*xhat), dpre = dy*(y>0 if relu), dy pooled over the 2x2 replicas if up2 */
int dgmr_bn_bwd_reduce(const float* dy, const float* x, const float* a, const float* b, const float* mean,
                       const float* invstd, double* red /*[G][C][2], zeroed inside*/, int64_t rows, int G, int C,
                       int relu, int up2, int H, int W, dgmr_stream_t stream);
/* dx (training: full batch-stat backward; eval: a*dpre); dgamma/dbeta [C] (+= if accumulate).
 * out_scale (nullable, [G][C]): dx is multiplied by it, and with relu | DGMR_FLAG_ROUND_TF32 written tf32-rounded -- when the BatchNorm
 * input is the output of a spectrally normalised convolution y = z/sigma_g + b, this IS that convolution's scaled, rounded output
 * gradient dz (its bias / scale gradients vanish identically under train-mode BatchNorm), so no separate dgmr_conv_bwd_prep pass runs.
 * dx_add (nullable, same shape as dx): added to dx before the optional rounding -- the gradient that reaches the BatchNorm input through its
 * OTHER consumer (the residual shortcut of GBlock / UpsampleGBlock, ref: dgmr/common.py:70-84), instead of a separate accumulation pass. */
int dgmr_bn_bwd_apply(const float* dy, const float* x, const float* a, const float* b, const float* mean,
                      const float* invstd, const float* out_scale, const double* red, float* dx, const float* dx_add,
                      float* dgamma, float* dbeta, int accumulate, int64_t rows, int G, int C, int relu, int up2, int H,
                      int W, int training, dgmr_stream_t stream);

/* ---- spectral norm (ref: torch/nn/utils/parametrizations.py:495-527, applied at
 * dgmr/layers/ConvGRU.py:29-55, common.py:43-66,113-137,192-215,350-384,451-455,
 * generators.py:52,67,84,101,115, discriminators.py:100,192).
 * W: [R][K] row-major (= weight.flatten(1)).  Performs the power iterations of `G` consecutive
 * reference calls in one launch: for g in 0..G-1: (training) u<-norm(W v), v<-norm(W^T u);
 * sigma_g = u.(W v).  Emits inv_sigma[g] and the (u_g, v_g) used, and leaves the final u,v in place.
 * ws: >= (G+2)*R + 2*G + 8 floats of scratch. */
int dgmr_sn_power_iter(const float* w, float* u, float* v, int R, int K, int G, float eps, int training,
                       float* inv_sigma, float* u_hist, float* v_hist, float* ws, dgmr_stream_t stream);
/* All spectrally normalised layers of a module in ONE launch (CTAs split over the weights by size, each weight's CTA group
 * iterating independently): `items` is a HOST array; every `ws` must be zero-initialised by the caller (same size rule). */
typedef struct {
  const float* w; float* u; float* v;            /* as in dgmr_sn_power_iter */
  float* inv_sigma; float* u_hist; float* v_hist;
  float* ws;
  int R, K, G, training;
  float eps;
} dgmr_sn_item;
int dgmr_sn_power_iter_multi(const dgmr_sn_item* items, int n, dgmr_stream_t stream);
/* dW[r][k] += sum_g d_inv_sigma[g] * (-inv_sigma[g]^2) * u_g[r] v_g[k]  (u,v constants, as in torch) */
int dgmr_sn_bwd(const float* d_inv_sigma, const float* inv_sigma, const float* u_hist, const float* v_hist,
                float* dw, int R, int K, int G, int accumulate, dgmr_stream_t stream);

/* out[r] = <a[r][offset : offset+cols], b[r][offset : offset+cols]> / denom[r]   (a, b: [rows][ld]; denom nullable)
 * The gradient of a G = 1 spectrally normalised convolution's output scale s = 1/sigma from its weight gradient:
 * dL/ds[co] = <dW[co], W[co]> / s[co]  (replaces the activation-side reduction of dgmr_conv_bwd_prep where one sigma serves the whole
 * batch; ref: torch.nn.utils.parametrizations.spectral_norm as used in dgmr/common.py:174-201, dgmr/layers/ConvGRU.py:37-52) */
int dgmr_rowdot_div(const float* a, const float* b, const float* denom, float* out, int rows, int64_t cols, int64_t ld, int64_t offset,
                    dgmr_stream_t stream);

/* dgmr_sn_bwd for all the spectrally normalised weights of a module in one launch (`items`: HOST array) */
typedef struct {
  const float* d_inv_sigma; const float* inv_sigma; const float* u_hist; const float* v_hist;
  float* dw;
  int R, K, G, accumulate;
} dgmr_sn_bwd_item;
int dgmr_sn_bwd_multi(const dgmr_sn_bwd_item* items, int n, dgmr_stream_t stream);

/* ---- convolution (ref: every Conv2d/Conv3d call site: dgmr/layers/ConvGRU.py:72-81,
 * common.py:71-83,141-154,222-236,290-300,413-424,486, generators.py:153,176-177,
 * discriminators.py:113-133,203-211; F.linear heads as 1x1).  Stride 1, "same" zero padding,
 * kernel extent 1 or 3 per dim. */
/* w: OIHW(/OIDHW) [Cout][CinTot][taps]; packs input-channel slice [ci0, ci0+Cin).
 * mode 0: forward pack  packed[tap][co][ci];  mode 1: dgrad pack  packed[taps-1-tap][ci][co]. */
int dgmr_pack_weight(const float* w, float* packed, int Cout, int CinTot, int ci0, int Cin, int taps, int mode,
                     dgmr_stream_t stream);
/* Many packs in ONE launch (all the weights of a network right after its optimiser step).  `items` is a HOST array.  Compared with
 * dgmr_pack_weight the destination may be wider than the slice: CinPad >= Cin input channels per row (the pad is not written: the
 * caller zeroes the buffer once) and rows [co0, co0 + Cout) of CoutTot (several weights side by side along Cout: the read|update gate
 * convolution of a ConvGRU, ref: dgmr/layers/ConvGRU.py:72-75).  mode as in dgmr_pack_weight (| DGMR_FLAG_ROUND_TF32). */
typedef struct {
  const float* w; float* packed;
  int Cout, CinTot, ci0, Cin, taps, mode;
  int CinPad, co0, CoutTot;
} dgmr_pack_item;
int dgmr_pack_weight_multi(const dgmr_pack_item* items, int n, dgmr_stream_t stream);
/* inverse of mode 0 for gradients: gw[co][ci0+ci][tap] (+)= packed[tap][co][ci] */
int dgmr_unpack_wgrad(const float* packed, float* gw, int Cout, int CinTot, int ci0, int Cin, int taps,
                      int accumulate, dgmr_stream_t stream);
/* y = act( conv(x, wp) * scale[g][co] + bias[co] + res )   (scale, bias, res optional = NULL)
 * x:[N,D,H,W,Cin]  y,res:[N,D,H,W,Cout]  scale:[G][Cout]  g = n / (N/G) */
/* precision DGMR_PREC_3XTF32 ("parity mode"): on the tensor-core path x/wp hold the hi parts and x_lo/wp_lo the lo parts
 * (dgmr_split_tf32) and every k-step issues lo*hi + hi*lo + hi*hi into the fp32 accumulator; with x_lo == wp_lo == NULL the
 * operands are full fp32 and the fp32-FMA kernel serves the call.  DGMR_PREC_TF32: x_lo/wp_lo are NULL. */
int dgmr_conv_fwd(const float* x, const float* x_lo, const float* wp, const float* wp_lo, const float* bias,
                  const float* scale, const float* res, float* y, int N, int D, int H, int W, int Cin, int Cout,
                  int kd, int kh, int kw, int G, int act, int algo, int precision, dgmr_stream_t stream);
/* backward prologue: dpre = dy*act'(y); dz = dpre*scale; dbias[co] (+)= sum dpre;
 * dscale[g][co] = sum dpre*(y - bias - res)/scale  (the <dY, Y-b> identity of SURVEY.md 8a/a13).
 * rows = pixels per group.  Any of dbias/dscale may be NULL.  up_h, up_w > 0: the forward ran with DGMR_FLAG_RES_UP2 on up_h x up_w
 * images, i.e. `res` is the half-resolution tensor and is read at (h/2, w/2); 0, 0 otherwise.
 * pool_d, pool_h, pool_w > 0 (with the convolution's output geometry D, H, W): the convolution output went through AvgPool (window
 * pool_d x pool_h x pool_w, floor; ref: DBlock, dgmr/common.py:234-236) and `dy` is the gradient of the POOLED tensor [N, D/pd, H/ph, W/pw, Cout]:
 * it is read at (d/pd, h/ph, w/pw) and divided by the window size here, instead of a separate upsample pass. */
int dgmr_conv_bwd_prep(const float* dy, const float* y, const float* res, const float* bias, const float* scale,
                       float* dz, float* dpre /*optional: unscaled dpre, = grad of res*/, float* dbias, float* dscale,
                       int64_t rows, int G, int Cout, int act, int accumulate_dbias, int up_h, int up_w,
                       int pool_d, int pool_h, int pool_w, int D, int H, int W, dgmr_stream_t stream);
/* dwp[tap][co][ci] = sum_pixels dz[p][co] * x[p+tap][ci]   (dwp fully overwritten).  Both operands are read straight from the
 * channels-last tensors (MN-major tensor-core tiles).  x_lo/dz_lo: lo parts for DGMR_PREC_3XTF32 (as in dgmr_conv_fwd), else NULL. */
int dgmr_conv_wgrad(const float* x, const float* x_lo, const float* dz, const float* dz_lo, float* dwp, int N, int D, int H, int W,
                    int Cin, int Cout, int kd, int kh, int kw, int algo, int precision, dgmr_stream_t stream);

/* ---- "nearest x2 upsample -> 3x3 convolution" in sub-pixel form (ref: UpsampleGBlock.first_conv_3x3 on the upsampled input,
 * dgmr/common.py:146-149): every output phase (2h+i, 2w+j) is a 2x2-tap convolution of the LOW-resolution input with pre-summed taps --
 * 16 instead of 36 MACs per low-resolution pixel, and the upsampled activation is never materialised (csrc/conv_subpix.cu).
 * x: [N,H,W,Cin] low resolution; y, res, dz: [N,2H,2W,Cout]; scale: [G][Cout].  All tensor-core only (no SIMT form): check
 * dgmr_upconv_supported first and use dgmr_upsample + dgmr_conv_fwd otherwise. */
int dgmr_upconv_supported(int N, int H, int W, int Cin, int Cout);
/* w: OIHW [Cout][CinTot][3][3] -> packed[16][Cout][Cin] (mode 0, forward) or packed[16][Cin][Cout] (mode 1, dgrad); tile z = ((i*2+j)*2+a)*2+b holds
 * sum_{kh in S(i,a), kw in S(j,b)} w[:, :, kh, kw], S(0,0) = {0}, S(0,1) = {1,2}, S(1,0) = {0,1}, S(1,1) = {2}; mode | DGMR_FLAG_ROUND_TF32 rounds the sums. */
int dgmr_pack_weight_subpix(const float* w, float* packed, int Cout, int CinTot, int ci0, int Cin, int mode, dgmr_stream_t stream);
/* gw[co][ci0+ci][kh][kw] (+)= sum of the tiles dwsp[z][co][ci] whose tap sets contain (kh, kw) */
int dgmr_unpack_wgrad_subpix(const float* dwsp, float* gw, int Cout, int CinTot, int ci0, int Cin, int accumulate, dgmr_stream_t stream);
/* y = act( upconv(x, wsp) * scale[g][co] + bias + res );  act may carry DGMR_FLAG_ROUND_OUT */
int dgmr_upconv_fwd(const float* x, const float* wsp, const float* bias, const float* scale, const float* res, float* y, int N, int H, int W,
                    int Cin, int Cout, int G, int act, dgmr_stream_t stream);
/* dx[N,H,W,Cin] = transpose of the above applied to dz (already scaled, tf32-rounded); wspt: the mode-1 pack */
int dgmr_upconv_dgrad(const float* dz, const float* wspt, float* dx, int N, int H, int W, int Cin, int Cout, dgmr_stream_t stream);
/* dwsp[16][Cout][Cin] = weight gradient of the pre-summed tiles (fold with dgmr_unpack_wgrad_subpix) */
int dgmr_upconv_wgrad(const float* x, const float* dz, float* dwsp, int N, int H, int W, int Cin, int Cout, dgmr_stream_t stream);

/* ---- discriminator head (ref: dgmr/discriminators.py:129,209: sum(relu(x)) over H,W) */
int dgmr_sumpool_relu_fwd(const float* x, float* y, int N, int HW, int C, dgmr_stream_t stream);
int dgmr_sumpool_relu_bwd(const float* dy, const float* x, float* dx, int N, int HW, int C, dgmr_stream_t stream);

/* ---- latent-stack attention (ref: dgmr/layers/Attention.py:9-20,71-85; note the reference
 * feeds [C,H,W] tensors to einsums labelled "h w c": positions are (channel,row) pairs, the
 * contracted axis is the image column).  q,k,v,out: [B,H,W,C] channels-last; beta: [B][L][L], L=C*H. */
int dgmr_attention_fwd(const float* q, const float* k, const float* v, float* out, float* beta,
                       int B, int H, int W, int C, dgmr_stream_t stream);
int dgmr_attention_bwd(const float* dout, const float* q, const float* k, const float* v, const float* beta,
                       float* dq, float* dk, float* dv, float* ws /*[B][L][L]*/, int B, int H, int W, int C,
                       dgmr_stream_t stream);

/* ---- losses (ref: dgmr/losses.py:307-319 hinge; :172-192 GridCellLoss + dgmr/dgmr.py:20-33 weight_fn) */
/* scores: [2B][cols] (real rows then generated rows; training uses cols=2: col 0 spatial, col 1 temporal).
 * loss = sum_col ( mean relu(1-real) + mean relu(1+gen) );  dscores = d loss/d scores */
int dgmr_hinge_disc(const float* scores, int B, int cols, float* loss, float* dscores, dgmr_stream_t stream);
/* loss = -mean(scores_gen) over n values; dscores = -1/n */
int dgmr_hinge_gen(const float* scores, int n, float* loss, float* dscores, dgmr_stream_t stream);
/* loss = sum |(gen-target)*max(target+1,cap)| * coef ; gen/target n elements */
int dgmr_grid_cell_fwd(const float* gen, const float* target, float cap, float coef, float* loss,
                       double* acc_ws /*1 double scratch*/, int64_t n, dgmr_stream_t stream);
/* dgen = sign(gen-target)*max(target+1,cap)*coef*(*gout)   (gout: device scalar) */
int dgmr_grid_cell_bwd(const float* gen, const float* target, float cap, float coef, const float* gout,
                       float* dgen, int64_t n, dgmr_stream_t stream);

/* ---- optimiser (ref: torch.optim.Adam built at dgmr/dgmr.py:292-300; eps 1e-8) on a flat buffer;
 * g is multiplied by grad_scale first (1/world_size after the NCCL all-reduce). */
int dgmr_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
              float eps, int step, float grad_scale, dgmr_stream_t stream);

/* ---- ensemble statistics of K-member forecasts (Generator.sample; the ensemble the reference's unused DGMR(num_samples=6) describes,
 * dgmr/dgmr.py:102), one pass over the ensemble.  P = T*C*H*W.
 * ens [B][K][P] (the layout Generator.sample returns); target [B][P] or NULL; thr [n_thr] (device); mean [B][P];
 * prob [n_thr][B][P] or NULL when n_thr == 0; crps [B][T*C][5] and ws (fp64, B*T*C*(H/16)*5 doubles) when target != NULL, else NULL
 * (the target pointer is then never read).
 *   mean[b][p]    = (sum of the members in member order) / K
 *   prob[i][b][p] = count(ens[b][k][p] >= thr[i]) / K
 *   crps[b][tc][s] = mean over the cells of frame (b, tc) at scale s of the ensemble CRPS
 *                    (1/K) sum_k |x_k - y| - (1/(2K^2)) sum_{j,k} |x_j - x_k|,   sum_{j,k} |x_j - x_k| = 2 sum_i (2i - K + 1) x_(i)
 *                    (x_(i) ascending, 0-based); scales s: 1 (pixels), 4x4 average, 4x4 maximum, 16x16 average, 16x16 maximum -- members and
 *                    target pooled the same way over non-overlapping windows.
 * 1 <= K <= 64, n_thr <= 8; with a target H and W must be multiples of 16.  No atomics: results are bitwise repeatable. */
int dgmr_ensemble_stats(const float* ens, const float* target, const float* thr, int n_thr, float* mean, float* prob, float* crps, double* ws,
                        int B, int K, int T, int C, int H, int W, dgmr_stream_t stream);

/* y <- nearest TF32-representable value of x (cvt.rna.tf32.f32; y may alias x; idempotent); applied to activations before
 * they enter a tensor-core convolution: in place when the tensor feeds convolutions only, into a copy otherwise */
int dgmr_round_tf32(const float* x, float* y, int64_t n, dgmr_stream_t stream);

/* ---- 3xTF32 support: hi = nearest TF32 of x, lo = nearest TF32 of (x - hi); hi + lo reproduces x to 2^-22 relative */
int dgmr_split_tf32(const float* x, float* hi, float* lo, int64_t n, dgmr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif
