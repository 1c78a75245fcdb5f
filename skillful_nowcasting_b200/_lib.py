"""ctypes binding of libdgmr_b200.so (the C ABI declared in include/dgmr_b200.h).

PyTorch tensors cross this boundary as raw device pointers + the current CUDA stream; nothing
else of torch is visible to the library.  There is NO CPU or library fallback: if the shared
object is missing, or a tensor is not a contiguous fp32 CUDA tensor, calls raise RuntimeError.

The argument types of every entry point are derived from the header itself, so the binding
cannot drift from the ABI; `load()` also verifies that every declared symbol is exported.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import Dict, List, Optional, Sequence, Tuple

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(_HERE), "include", "dgmr_b200.h")
LIB_PATH = os.path.join(_HERE, "libdgmr_b200.so")

ACT_NONE, ACT_RELU = 0, 1
ALGO_AUTO, ALGO_SIMT, ALGO_UMMA, ALGO_UMMA_PATCH, ALGO_UMMA_KWSTACK, ALGO_UMMA_PAIR = 0, 1, 2, 3, 4, 5
PREC_TF32, PREC_3XTF32 = 0, 1
FLAG_ROUND_TF32 = 256
FLAG_ACCUMULATE = 512
FLAG_ROUND_OUT = 1024
FLAG_RES_UP2 = 2048

_CTYPES = {
    "int": ctypes.c_int,
    "int64_t": ctypes.c_int64,
    "float": ctypes.c_float,
    "dgmr_stream_t": ctypes.c_void_p,
    "char*": ctypes.c_char_p,
}


def parse_header(path: str = HEADER) -> Dict[str, Tuple[str, List[Tuple[str, str]]]]:
    """{name: (return type, [(ctype string, arg name), ...])} for every dgmr_* declaration."""
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    out = {}
    for m in re.finditer(r"\b(int|const char\*)\s+(dgmr_\w+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S):
        ret, name, args = m.group(1), m.group(2), " ".join(m.group(3).split())
        alist = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                mm = re.match(r"(.*?)(\w+)$", a)
                alist.append((mm.group(1).strip(), mm.group(2)))
        out[name] = (ret, alist)
    return out


def _to_ctype(t: str):
    t = t.replace("const ", "").strip()
    if t == "char*":
        return ctypes.c_char_p
    if t.endswith("*"):
        return ctypes.c_void_p
    return _CTYPES[t]


_lib: Optional[ctypes.CDLL] = None
_decls = None


def load() -> ctypes.CDLL:
    """dlopen the library and check every symbol declared in the header (works without a GPU)."""
    global _lib, _decls
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
            "(the B200 path has no CPU or library fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    decls = parse_header()
    for name, (ret, args) in decls.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # pragma: no cover
            raise RuntimeError(f"libdgmr_b200.so does not export {name} declared in {HEADER}") from e
        fn.restype = ctypes.c_char_p if ret != "int" else ctypes.c_int
        fn.argtypes = [_to_ctype(t) for t, _ in args]
    _lib, _decls = lib, decls
    return lib


def _ptr(t: Optional[torch.Tensor], name: str = "tensor") -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError(f"dgmr_b200: {name} must be a CUDA tensor (no CPU fallback exists)")
    if not t.is_contiguous():
        raise RuntimeError(f"dgmr_b200: {name} must be contiguous")
    return t.data_ptr()


def _f32(t: Optional[torch.Tensor], name: str):
    if t is not None and t.dtype != torch.float32:
        raise RuntimeError(f"dgmr_b200: {name} must be float32, got {t.dtype}")
    return _ptr(t, name)


def _f64(t: Optional[torch.Tensor], name: str):
    if t is not None and t.dtype != torch.float64:
        raise RuntimeError(f"dgmr_b200: {name} must be float64, got {t.dtype}")
    return _ptr(t, name)


class SnItem(ctypes.Structure):
    """dgmr_sn_item of include/dgmr_b200.h."""
    _fields_ = [("w", ctypes.c_void_p), ("u", ctypes.c_void_p), ("v", ctypes.c_void_p), ("inv_sigma", ctypes.c_void_p),
                ("u_hist", ctypes.c_void_p), ("v_hist", ctypes.c_void_p), ("ws", ctypes.c_void_p), ("R", ctypes.c_int),
                ("K", ctypes.c_int), ("G", ctypes.c_int), ("training", ctypes.c_int), ("eps", ctypes.c_float)]


class PackItem(ctypes.Structure):
    """dgmr_pack_item of include/dgmr_b200.h."""
    _fields_ = [("w", ctypes.c_void_p), ("packed", ctypes.c_void_p), ("Cout", ctypes.c_int), ("CinTot", ctypes.c_int), ("ci0", ctypes.c_int),
                ("Cin", ctypes.c_int), ("taps", ctypes.c_int), ("mode", ctypes.c_int), ("CinPad", ctypes.c_int), ("co0", ctypes.c_int),
                ("CoutTot", ctypes.c_int)]


class SnBwdItem(ctypes.Structure):
    """dgmr_sn_bwd_item of include/dgmr_b200.h."""
    _fields_ = [("d_inv_sigma", ctypes.c_void_p), ("inv_sigma", ctypes.c_void_p), ("u_hist", ctypes.c_void_p), ("v_hist", ctypes.c_void_p),
                ("dw", ctypes.c_void_p), ("R", ctypes.c_int), ("K", ctypes.c_int), ("G", ctypes.c_int), ("accumulate", ctypes.c_int)]


class CudaBackend:
    """Thin tensor-level view of the C ABI.  Method names/arguments mirror include/dgmr_b200.h.
    `launches` counts kernel-launching entry-point calls (reported by bench.py as gpu_launches)."""

    name = "cuda"

    def __init__(self):
        self.lib = load()
        self.launches = 0
        self.profile = None  # bench.py sets a list: (name, flops, ev0, ev1, tag) per call, CUDA events on the launch stream

    # -- plumbing
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def _call(self, name, *args, _tag=None, _flops=0.0, _info=""):
        self.launches += 1
        prof = self.profile
        if prof is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        rc = getattr(self.lib, name)(*args, self._stream())
        if prof is not None:
            e1.record()
            prof.append((name, _flops, e0, e1, _tag or name.replace("dgmr_", ""), _info))
        if rc != 0:
            raise RuntimeError(f"{name} failed ({rc}): {self.lib.dgmr_last_error().decode()}")

    def _query(self, name, *args) -> int:
        return int(getattr(self.lib, name)(*args))

    # -- queries / options
    def set_option(self, name: str, value: int):
        """Tuning / test option of the tensor-core launchers (include/dgmr_b200.h: dgmr_set_option); -1 = heuristic default."""
        if self.lib.dgmr_set_option(name.encode(), int(value)) != 0:
            raise RuntimeError(self.lib.dgmr_last_error().decode())

    def conv_umma_supported(self, N, D, H, W, Cin, Cout, kd, kh, kw) -> bool:
        return bool(self._query("dgmr_conv_umma_supported", N, D, H, W, Cin, Cout, kd, kh, kw))

    def wgrad_umma_supported(self, N, D, H, W, Cin, Cout, kd, kh, kw) -> bool:
        return bool(self._query("dgmr_wgrad_umma_supported", N, D, H, W, Cin, Cout, kd, kh, kw))

    # -- layout
    def permute(self, src, dst, shape: Sequence[int], sstr: Sequence[int], dstr: Sequence[int], accumulate=False,
                src_off: int = 0, dst_off: int = 0):
        """src_off/dst_off: element offsets added to the base pointers (slices without torch views)."""
        n = len(shape)
        arr = ctypes.c_int64 * n
        self._call("dgmr_permute", _f32(src, "src") + 4 * src_off, _f32(dst, "dst") + 4 * dst_off, n, arr(*shape), arr(*sstr),
                   arr(*dstr), int(accumulate), _info=f"{tuple(shape)} s{tuple(sstr)} d{tuple(dstr)}")

    def reduce_mid(self, x, y, A, R, C, accumulate=False):
        self._call("dgmr_reduce_mid", _f32(x, "x"), _f32(y, "y"), A, R, C, int(accumulate))

    # -- pointwise
    def axpby(self, a, x, b, y, out):
        self._call("dgmr_axpby", float(a), _f32(x, "x"), float(b), _f32(y, "y"), _f32(out, "out"), out.numel())

    def fill(self, x, value):
        self._call("dgmr_fill", _f32(x, "x"), float(value), x.numel())

    def relu_fwd(self, x, y):
        self._call("dgmr_relu_fwd", _f32(x, "x"), _f32(y, "y"), x.numel())

    def relu_bwd(self, dy, x, dx):
        self._call("dgmr_relu_bwd", _f32(dy, "dy"), _f32(x, "x"), _f32(dx, "dx"), x.numel())

    def round_tf32(self, x, y=None):
        self._call("dgmr_round_tf32", _f32(x, "x"), _f32(x if y is None else y, "y"), x.numel(), _info=f"n{x.numel()} {'inplace' if y is None else 'copy'}")

    def split_tf32(self, x, hi, lo):
        self._call("dgmr_split_tf32", _f32(x, "x"), _f32(hi, "hi"), _f32(lo, "lo"), x.numel())

    def pool_sum(self, x, y, N, D, H, W, C, pd, ph, pw, scale):
        self._call("dgmr_pool_sum", _f32(x, "x"), _f32(y, "y"), N, D, H, W, C, pd, ph, pw, float(scale), _info=f"{N}x{D}x{H}x{W}x{C} /{pd}{ph}{pw}")

    def upsample(self, x, y, N, D, H, W, C, ud, uh, uw, Do, Ho, Wo, scale):
        self._call("dgmr_upsample", _f32(x, "x"), _f32(y, "y"), N, D, H, W, C, ud, uh, uw, Do, Ho, Wo, float(scale), _info=f"{N}x{D}x{H}x{W}x{C} *{ud}{uh}{uw}")

    # -- GRU
    def gru_gate_fwd(self, pre_r, ld, h, rh, rows, Ch, flags=0, x_r=None):
        self._call("dgmr_gru_gate_fwd", _f32(pre_r, "pre_r"), ld, _f32(x_r, "x_r"), _f32(h, "h"), _f32(rh, "rh"), rows, Ch, int(flags))

    def gru_blend_fwd(self, pre_u, ld, h, c, hnew, hnew_tf32, rows, Ch, relu_c=False, x_u=None, x_c=None):
        self._call("dgmr_gru_blend_fwd", _f32(pre_u, "pre_u"), ld, _f32(x_u, "x_u"), _f32(h, "h"), _f32(c, "c"), _f32(x_c, "x_c"), _f32(hnew, "hnew"),
                   _f32(hnew_tf32, "hnew_tf32"), rows, Ch, int(relu_c))

    def gru_gate_bwd(self, d_rh, pre_r, ld, h, d_pre_r, ldd, dh, accumulate, rows, Ch, dz_scale=None, dz=None, dz_round=False):
        self._call("dgmr_gru_gate_bwd", _f32(d_rh, "d_rh"), _f32(pre_r, "pre_r"), ld, _f32(h, "h"), _f32(d_pre_r, "d_pre_r"), ldd,
                   _f32(dh, "dh"), int(accumulate), rows, Ch, _f32(dz_scale, "dz_scale"), _f32(dz, "dz"), int(dz_round))

    def gru_blend_bwd(self, d_hnew, pre_u, ld, h, c, d_pre_u, ldd, dc, dh, accumulate, rows, Ch, relu_c=False, dz_u_scale=None, dz_u=None,
                      dz_c_scale=None, dz_c=None, dz_round=False):
        self._call("dgmr_gru_blend_bwd", _f32(d_hnew, "d_hnew"), _f32(pre_u, "pre_u"), ld, _f32(h, "h"), _f32(c, "c"),
                   _f32(d_pre_u, "d_pre_u"), ldd, _f32(dc, "dc"), _f32(dh, "dh"), int(accumulate), rows, Ch, int(relu_c),
                   _f32(dz_u_scale, "dz_u_scale"), _f32(dz_u, "dz_u"), _f32(dz_c_scale, "dz_c_scale"), _f32(dz_c, "dz_c"), int(dz_round))

    # -- BatchNorm
    def bn_stats(self, x, sums, rows, G, C):
        self._call("dgmr_bn_stats", _f32(x, "x"), _f64(sums, "sums"), rows, G, C, _flops=4.0 * rows * G * C, _info=f"rows{rows} G{G} C{C} (GB/s)")

    def bn_finalize(self, sums, gamma, beta, rmean, rvar, rows, G, C, eps, momentum, training, mean, invstd, a, b):
        self._call("dgmr_bn_finalize", _f64(sums, "sums"), _f32(gamma, "gamma"), _f32(beta, "beta"), _f32(rmean, "running_mean"),
                   _f32(rvar, "running_var"), rows, G, C, float(eps), float(momentum), int(training), _f32(mean, "mean"),
                   _f32(invstd, "invstd"), _f32(a, "a"), _f32(b, "b"))

    def bn_apply(self, x, a, b, y, rows, G, C, relu, up2, H, W, x_rounded=None):
        self._call("dgmr_bn_apply", _f32(x, "x"), _f32(a, "a"), _f32(b, "b"), _f32(y, "y"), _f32(x_rounded, "x_rounded"), rows, G, C, int(relu), int(up2), H, W,  # relu may carry FLAG_ROUND_TF32
                   _flops=4.0 * rows * G * C * (5 if up2 else 2 + (x_rounded is not None)), _info=f"rows{rows} G{G} C{C} up{int(up2)}{' +xr' if x_rounded is not None else ''} (GB/s)")

    def bn_bwd_reduce(self, dy, x, a, b, mean, invstd, red, rows, G, C, relu, up2, H, W):
        self._call("dgmr_bn_bwd_reduce", _f32(dy, "dy"), _f32(x, "x"), _f32(a, "a"), _f32(b, "b"), _f32(mean, "mean"),
                   _f32(invstd, "invstd"), _f64(red, "red"), rows, G, C, int(relu), int(up2), H, W)

    def bn_bwd_apply(self, dy, x, a, b, mean, invstd, out_scale, red, dx, dgamma, dbeta, accumulate, rows, G, C, relu, up2, H, W, training,
                     dx_add=None):
        """relu may carry FLAG_ROUND_TF32 (dx written tf32-rounded); out_scale [G, C] (nullable) multiplies dx; dx_add (nullable) is added."""
        self._call("dgmr_bn_bwd_apply", _f32(dy, "dy"), _f32(x, "x"), _f32(a, "a"), _f32(b, "b"), _f32(mean, "mean"),
                   _f32(invstd, "invstd"), _f32(out_scale, "out_scale"), _f64(red, "red"), _f32(dx, "dx"), _f32(dx_add, "dx_add"), _f32(dgamma, "dgamma"),
                   _f32(dbeta, "dbeta"), int(accumulate), rows, G, C, int(relu), int(up2), H, W, int(training), _info=f"rows{rows} G{G} C{C} up{int(up2)}")

    # -- spectral norm
    def sn_power_iter(self, w, u, v, R, K, G, eps, training, inv_sigma, u_hist, v_hist, ws):
        self._call("dgmr_sn_power_iter", _f32(w, "w"), _f32(u, "u"), _f32(v, "v"), R, K, G, float(eps), int(training),
                   _f32(inv_sigma, "inv_sigma"), _f32(u_hist, "u_hist"), _f32(v_hist, "v_hist"), _f32(ws, "ws"),
                   _info=f"{R}x{K} G{G} train{int(training)}")

    def sn_power_iter_multi(self, items):
        """items: list of dicts(w,u,v,R,K,G,eps,training,inv_sigma,u_hist,v_hist,ws) -- every `ws` already zeroed."""
        arr = (SnItem * len(items))()
        for a, it in zip(arr, items):
            for k in ("w", "u", "v", "inv_sigma", "u_hist", "v_hist", "ws"):
                setattr(a, k, _f32(it[k], k))
            a.R, a.K, a.G, a.training, a.eps = it["R"], it["K"], it["G"], int(it["training"]), float(it["eps"])
        self._call("dgmr_sn_power_iter_multi", arr, len(items), _info=f"{len(items)} weights")

    def sn_bwd(self, d_inv_sigma, inv_sigma, u_hist, v_hist, dw, R, K, G, accumulate):
        self._call("dgmr_sn_bwd", _f32(d_inv_sigma, "d_inv_sigma"), _f32(inv_sigma, "inv_sigma"), _f32(u_hist, "u_hist"),
                   _f32(v_hist, "v_hist"), _f32(dw, "dw"), R, K, G, int(accumulate))

    def rowdot_div(self, a, b, denom, out, rows, cols, ld, offset=0):
        self._call("dgmr_rowdot_div", _f32(a, "a"), _f32(b, "b"), _f32(denom, "denom"), _f32(out, "out"), int(rows), int(cols), int(ld), int(offset))

    def sn_bwd_multi(self, items):
        """items: list of dicts(d_inv_sigma, inv_sigma, u_hist, v_hist, dw, R, K, G, accumulate): one launch per 48 weights."""
        arr = (SnBwdItem * len(items))()
        for a, it in zip(arr, items):
            for k in ("d_inv_sigma", "inv_sigma", "u_hist", "v_hist", "dw"):
                setattr(a, k, _f32(it[k], k))
            a.R, a.K, a.G, a.accumulate = it["R"], it["K"], it["G"], int(it["accumulate"])
        self._call("dgmr_sn_bwd_multi", arr, len(items), _info=f"{len(items)} weights")

    # -- conv
    def pack_weight(self, w, packed, Cout, CinTot, ci0, Cin, taps, mode):
        self._call("dgmr_pack_weight", _f32(w, "w"), _f32(packed, "packed"), Cout, CinTot, ci0, Cin, taps, mode)

    def pack_weight_multi(self, items):
        """items: list of dicts(w, packed, Cout, CinTot, ci0, Cin, taps, mode, CinPad, co0, CoutTot): all of them in one launch
        (per 64 items)."""
        arr = (PackItem * len(items))()
        for a, it in zip(arr, items):
            a.w, a.packed = _f32(it["w"], "w"), _f32(it["packed"], "packed")
            for k in ("Cout", "CinTot", "ci0", "Cin", "taps", "mode", "CinPad", "co0", "CoutTot"):
                setattr(a, k, int(it[k]))
        self._call("dgmr_pack_weight_multi", arr, len(items), _info=f"{len(items)} packs")

    def unpack_wgrad(self, packed, gw, Cout, CinTot, ci0, Cin, taps, accumulate):
        self._call("dgmr_unpack_wgrad", _f32(packed, "packed"), _f32(gw, "gw"), Cout, CinTot, ci0, Cin, taps, int(accumulate))

    def conv_fwd(self, x, wp, bias, scale, res, y, N, D, H, W, Cin, Cout, kd, kh, kw, G, act, algo=ALGO_AUTO, precision=PREC_TF32,
                 x_lo=None, wp_lo=None):
        tag = None
        if self.profile is not None:
            umma = algo == ALGO_UMMA or (algo == ALGO_AUTO and self.conv_umma_supported(N, D, H, W, Cin, Cout, kd, kh, kw))
            tag = ("conv_umma_splitk" if act & FLAG_ACCUMULATE else "conv_umma") if umma else "conv_simt"
        if x_lo is not None:
            tag = "conv_umma_3x"
        self._call("dgmr_conv_fwd", _f32(x, "x"), _f32(x_lo, "x_lo"), _f32(wp, "wp"), _f32(wp_lo, "wp_lo"), _f32(bias, "bias"),
                   _f32(scale, "scale"), _f32(res, "res"), _f32(y, "y"), N, D, H, W, Cin, Cout, kd, kh, kw, G, act, algo, precision,
                   _tag=tag, _flops=2.0 * N * D * H * W * Cin * Cout * kd * kh * kw,
                   _info=f"{N}x{D}x{H}x{W} {Cin}->{Cout} k{kd}{kh}{kw} G{G}")

    # -- sub-pixel up-convolution (nearest x2 -> 3x3 conv on the low-resolution input; csrc/conv_subpix.cu)
    def upconv_supported(self, N, H, W, Cin, Cout) -> bool:
        return bool(self._query("dgmr_upconv_supported", N, H, W, Cin, Cout))

    def pack_weight_subpix(self, w, packed, Cout, CinTot, ci0, Cin, mode):
        self._call("dgmr_pack_weight_subpix", _f32(w, "w"), _f32(packed, "packed"), Cout, CinTot, ci0, Cin, mode, _tag="pack_weight")

    def unpack_wgrad_subpix(self, dwsp, gw, Cout, CinTot, ci0, Cin, accumulate):
        self._call("dgmr_unpack_wgrad_subpix", _f32(dwsp, "dwsp"), _f32(gw, "gw"), Cout, CinTot, ci0, Cin, int(accumulate), _tag="unpack_wgrad")

    def upconv_fwd(self, x, wsp, bias, scale, res, y, N, H, W, Cin, Cout, G, act):
        self._call("dgmr_upconv_fwd", _f32(x, "x"), _f32(wsp, "wsp"), _f32(bias, "bias"), _f32(scale, "scale"), _f32(res, "res"), _f32(y, "y"),
                   N, H, W, Cin, Cout, G, act, _tag="conv_umma", _flops=2.0 * N * H * W * 16 * Cin * Cout,
                   _info=f"{N}x1x{H}x{W} {Cin}->{Cout} up2+k133 (sub-pixel: 16 taps) G{G}")

    def upconv_dgrad(self, dz, wspt, dx, N, H, W, Cin, Cout):
        self._call("dgmr_upconv_dgrad", _f32(dz, "dz"), _f32(wspt, "wspt"), _f32(dx, "dx"), N, H, W, Cin, Cout, _tag="conv_umma",
                   _flops=2.0 * N * H * W * 16 * Cin * Cout, _info=f"{N}x1x{H}x{W} {Cout}->{Cin} up2+k133 dgrad (sub-pixel: 16 taps)")

    def upconv_wgrad(self, x, dz, dwsp, N, H, W, Cin, Cout):
        self._call("dgmr_upconv_wgrad", _f32(x, "x"), _f32(dz, "dz"), _f32(dwsp, "dwsp"), N, H, W, Cin, Cout, _tag="wgrad_umma",
                   _flops=2.0 * N * H * W * 16 * Cin * Cout, _info=f"{N}x1x{H}x{W} {Cin}->{Cout} up2+k133 (sub-pixel: 16 taps)")

    def conv_bwd_prep(self, dy, y, res, bias, scale, dz, dpre, dbias, dscale, rows, G, Cout, act, accumulate_dbias=False, up_hw=(0, 0),
                      pool=None):
        """pool: (pd, ph, pw, D, H, W): dy is the gradient of the average-pooled conv output (see the header)."""
        pool = tuple(int(v) for v in pool) if pool else (0, 0, 0, 0, 0, 0)
        nb = sum(t is not None for t in (dy, y, res, dz, dpre)) * 4.0 * rows * G * Cout   # bytes moved (profile only)
        self._call("dgmr_conv_bwd_prep", _f32(dy, "dy"), _f32(y, "y"), _f32(res, "res"), _f32(bias, "bias"), _f32(scale, "scale"),
                   _f32(dz, "dz"), _f32(dpre, "dpre"), _f32(dbias, "dbias"), _f32(dscale, "dscale"), rows, G, Cout, act,
                   int(accumulate_dbias), int(up_hw[0]), int(up_hw[1]), *pool, _flops=nb, _info=f"rows{rows} G{G} C{Cout} (GB/s)")

    def conv_wgrad(self, x, dz, dwp, N, D, H, W, Cin, Cout, kd, kh, kw, algo=ALGO_AUTO, precision=PREC_TF32, x_lo=None, dz_lo=None):
        tag = None
        if self.profile is not None:
            umma = algo == ALGO_UMMA or (algo == ALGO_AUTO and self.wgrad_umma_supported(N, D, H, W, Cin, Cout, kd, kh, kw))
            tag = "wgrad_umma" if umma else "wgrad_simt"
        self._call("dgmr_conv_wgrad", _f32(x, "x"), _f32(x_lo, "x_lo"), _f32(dz, "dz"), _f32(dz_lo, "dz_lo"), _f32(dwp, "dwp"),
                   N, D, H, W, Cin, Cout, kd, kh, kw, algo, precision,
                   _tag=tag, _flops=2.0 * N * D * H * W * Cin * Cout * kd * kh * kw,
                   _info=f"{N}x{D}x{H}x{W} {Cin}->{Cout} k{kd}{kh}{kw}")

    # -- D head / attention / losses / optimiser
    def sumpool_relu_fwd(self, x, y, N, HW, C):
        self._call("dgmr_sumpool_relu_fwd", _f32(x, "x"), _f32(y, "y"), N, HW, C)

    def sumpool_relu_bwd(self, dy, x, dx, N, HW, C):
        self._call("dgmr_sumpool_relu_bwd", _f32(dy, "dy"), _f32(x, "x"), _f32(dx, "dx"), N, HW, C)

    def attention_fwd(self, q, k, v, out, beta, B, H, W, C):
        self._call("dgmr_attention_fwd", _f32(q, "q"), _f32(k, "k"), _f32(v, "v"), _f32(out, "out"), _f32(beta, "beta"), B, H, W, C)

    def attention_bwd(self, dout, q, k, v, beta, dq, dk, dv, ws, B, H, W, C):
        self._call("dgmr_attention_bwd", _f32(dout, "dout"), _f32(q, "q"), _f32(k, "k"), _f32(v, "v"), _f32(beta, "beta"),
                   _f32(dq, "dq"), _f32(dk, "dk"), _f32(dv, "dv"), _f32(ws, "ws"), B, H, W, C)

    def hinge_disc(self, scores, B, cols, loss, dscores):
        self._call("dgmr_hinge_disc", _f32(scores, "scores"), B, cols, _f32(loss, "loss"), _f32(dscores, "dscores"))

    def hinge_gen(self, scores, n, loss, dscores):
        self._call("dgmr_hinge_gen", _f32(scores, "scores"), n, _f32(loss, "loss"), _f32(dscores, "dscores"))

    def grid_cell_fwd(self, gen, target, cap, coef, loss, acc_ws):
        self._call("dgmr_grid_cell_fwd", _f32(gen, "gen"), _f32(target, "target"), float(cap), float(coef), _f32(loss, "loss"),
                   _f64(acc_ws, "acc_ws"), gen.numel())

    def grid_cell_bwd(self, gen, target, cap, coef, gout, dgen):
        self._call("dgmr_grid_cell_bwd", _f32(gen, "gen"), _f32(target, "target"), float(cap), float(coef), _f32(gout, "gout"),
                   _f32(dgen, "dgen"), gen.numel())

    # -- ensemble statistics
    def ensemble_stats(self, ens, target, thr, mean, prob, crps, ws, B, K, T, C, H, W):
        n_thr = 0 if thr is None else thr.numel()
        nb = 4.0 * B * T * C * H * W * (K + (target is not None) + 1 + n_thr)   # algorithmic bytes (profile only)
        self._call("dgmr_ensemble_stats", _f32(ens, "ens"), _f32(target, "target"), _f32(thr, "thr"), n_thr, _f32(mean, "mean"),
                   _f32(prob, "prob"), _f32(crps, "crps"), _f64(ws, "ws"), B, K, T, C, H, W, _flops=nb,
                   _info=f"B{B} K{K} T{T} C{C} {H}x{W} thr{n_thr}{' +crps' if target is not None else ''} (GB/s)")

    def adam(self, p, g, m, v, lr, beta1, beta2, eps, step, grad_scale=1.0):
        self._call("dgmr_adam", _f32(p, "p"), _f32(g, "g"), _f32(m, "m"), _f32(v, "v"), p.numel(), float(lr), float(beta1),
                   float(beta2), float(eps), int(step), float(grad_scale))


_backend = None


def backend():
    """The active backend.  Product code gets the CUDA library or an error — never a fallback.
    (tests/ may inject a host emulator of the ABI through set_backend() to exercise host logic.)"""
    global _backend
    if _backend is None:
        _backend = CudaBackend()
    return _backend


def set_backend(b):
    global _backend
    old = _backend
    _backend = b
    return old
