"""Autograd layer over the C ABI: every function here is one (fused) kernel family of
include/dgmr_b200.h with a hand-written backward that also runs through the C ABI.

Internal activation format: contiguous fp32 channels-last tensors [N, D, H, W, C] (2-D: D == 1),
images ordered group-major: N = G * (N // G), one *group* per reference call (timestep / frame).
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
from torch.autograd import Function

from . import _lib
from ._lib import (ACT_NONE, ACT_RELU, ALGO_AUTO, ALGO_SIMT, ALGO_UMMA, FLAG_ACCUMULATE, FLAG_RES_UP2, FLAG_ROUND_OUT, FLAG_ROUND_TF32,
                   PREC_3XTF32, PREC_TF32)

FLAG_SPLIT = 1024   # packed_weight(): return the [hi | lo] 3xTF32 pair (host-side flag, never crosses the ABI)


class config:
    """Runtime knobs (tests flip these to cross-check the tensor-core path against the SIMT kernels)."""
    conv_algo = ALGO_AUTO
    wgrad_algo = ALGO_AUTO
    # PREC_TF32: 1xTF32 operands (what cuDNN does by default for the reference's convolutions) -- the fast mode every benchmark
    # number comes from.  PREC_3XTF32: "parity mode": error-compensated operand pairs (hi*hi + hi*lo + lo*hi, ~fp32 accuracy) on
    # the plain tcgen05 kernels; nothing is rounded to tf32 anywhere.
    precision = PREC_TF32
    # operands of tensor-core convs are rounded to the NEAREST tf32 value first (the MMA itself truncates, which is
    # biased): weights while packing, activations in place (idempotent), dz in the backward prologue
    round_tf32 = True
    _dbg_round_act = True   # debug knobs (finer control of what round_tf32 applies to)
    _dbg_round_w = True
    _dbg_round_dz = True
    # small-M / large-K convs (the ConvGRU steps) run split over the filter taps with fp32 red.add into the output
    split_taps = True
    # ConvGRU: fused read|update gate conv + whole recurrence as one autograd node (False: the per-step reference wiring)
    gru_sequence = True
    # ... in the tap-split mode its step convolutions accumulate into buffers zeroed once per sequence and the gate kernels add the x parts
    # (False: one copy of the x part per convolution and step)
    gru_defer_x = True
    # "nearest x2 -> 3x3 conv" in sub-pixel form (csrc/conv_subpix.cu) wherever the tensor-core kernels serve the shape (1xTF32 mode)
    upconv = True
    # 3x3x3 weight gradients of narrow layers with the depth taps folded into the channel axis (see _Conv.backward)
    fold_depth_wgrad = True
    # G = 1 spectrally normalised convolutions: scale gradient from the weight gradient (<dW, W>/s per output channel) instead of an
    # activation-side reduction in the backward prologue (see _Conv.forward)
    dscale_from_wgrad = True
    _force_upconv = False   # tests: take the sub-pixel path on the host emulator too


def _be():
    return _lib.backend()


def _new(shape, like: torch.Tensor, dtype=torch.float32):
    return torch.empty(tuple(shape), device=like.device, dtype=dtype)


def _zeros(shape, like: torch.Tensor, dtype=torch.float32):
    return torch.zeros(tuple(shape), device=like.device, dtype=dtype)


def _c(t: Optional[torch.Tensor]):
    return None if t is None else (t if t.is_contiguous() else t.contiguous())


def contig_strides(shape: Sequence[int]) -> List[int]:
    st, acc = [], 1
    for s in reversed(shape):
        st.append(acc)
        acc *= s
    return list(reversed(st))


def _numel(shape):
    n = 1
    for s in shape:
        n *= s
    return n


# ----------------------------------------------------------------------------- layout
class _Permute(Function):
    """dst[dstr . i] = src[sstr . i] for i in `shape`; backward gathers the other way.
    The map must be injective on src (every src element read at most once)."""

    @staticmethod
    def forward(ctx, src, out_shape, shape, sstr, dstr, src_off, dst_off):
        src = _c(src)
        full = _numel(shape) == _numel(out_shape)
        dst = _new(out_shape, src) if full else _zeros(out_shape, src)
        _be().permute(src, dst, shape, sstr, dstr, False, src_off, dst_off)
        ctx.meta = (tuple(src.shape), tuple(shape), tuple(sstr), tuple(dstr), src_off, dst_off)
        return dst

    @staticmethod
    def backward(ctx, g):
        src_shape, shape, sstr, dstr, src_off, dst_off = ctx.meta
        g = _c(g)
        full = _numel(shape) == _numel(src_shape)
        gs = _new(src_shape, g) if full else _zeros(src_shape, g)
        _be().permute(g, gs, shape, dstr, sstr, False, dst_off, src_off)
        return gs, None, None, None, None, None, None


def permute(src, out_shape, shape, sstr, dstr, src_off=0, dst_off=0):
    return _Permute.apply(src, tuple(out_shape), tuple(shape), tuple(sstr), tuple(dstr), src_off, dst_off)


def permute_into(src, dst, shape, sstr, dstr, dst_off=0):
    """`permute` without autograd into an existing tensor at element offset dst_off (inference outputs assembled in place)."""
    _be().permute(_c(src), dst, tuple(shape), tuple(sstr), tuple(dstr), False, 0, dst_off)


def nchw_to_cl(x: torch.Tensor) -> torch.Tensor:
    """[N,C,H,W] or [N,C,D,H,W] -> [N,D,H,W,C]."""
    if x.dim() == 4:
        n, c, h, w = x.shape
        d = 1
    else:
        n, c, d, h, w = x.shape
    if c == 1:  # same memory order; private copy because conv inputs may be rounded to tf32 in place
        return permute(x, (n, d, h, w, 1), (n * d * h * w,), (1,), (1,))
    sp = d * h * w
    return permute(x, (n, d, h, w, c), (n, sp, c), (c * sp, 1, sp), (sp * c, c, 1))


def cl_to_nchw(x: torch.Tensor, keep_depth: bool = False) -> torch.Tensor:
    """[N,D,H,W,C] -> [N,C,H,W] (D == 1 and not keep_depth) or [N,C,D,H,W]."""
    n, d, h, w, c = x.shape
    out_shape = (n, c, d, h, w) if (keep_depth or d != 1) else (n, c, h, w)
    if c == 1:
        return x.reshape(out_shape)
    sp = d * h * w
    return permute(x, out_shape, (n, sp, c), (sp * c, c, 1), (c * sp, 1, sp))


def pad8(c: int) -> int:
    return (c + 7) // 8 * 8


def space_to_depth(x: torch.Tensor, pad: bool = True) -> torch.Tensor:
    """PixelUnshuffle(2) on channels-last: [N,D,H,W,C] -> [N,D,H/2,W/2,4C], channel c*4 + i*2 + j
    (ref: torch PixelUnshuffle at dgmr/common.py:326,393; discriminators.py:69,166).  With `pad` the channel axis is
    zero-padded to a multiple of 8 (4 -> 8 for single-channel radar) so the tensor-core convs can consume it."""
    n, d, h, w, c = x.shape
    h2, w2 = h // 2, w // 2
    co = pad8(4 * c) if pad else 4 * c
    ss = contig_strides((n, d, h, w, c))
    ds = contig_strides((n, d, h2, w2, co))
    return permute(x, (n, d, h2, w2, co), (n, d, h2, w2, c, 2, 2),
                   (ss[0], ss[1], 2 * ss[2], 2 * ss[3], 1, ss[2], ss[3]), (ds[0], ds[1], ds[2], ds[3], 4, 2, 1))


class _FoldDepth3(Function):
    """x [N,D,H,W,Cp] (first `c` channels real) -> [N,D,H,W,pad8(3c)] with channel kd*c + i = x[d + kd - 1][i] (zero outside the depth
    range): the depth taps of a 3x3x3 convolution over a FEW-channel input folded into the channel axis, so that the convolution becomes
    a 1x3x3 one with 3c input channels (first temporal-discriminator block: 4 -> 12 real channels in 16 instead of 27 taps x 8 half-empty
    channels; ref: dgmr/discriminators.py:113, common.py:187-191).  Pure index map: bit-exact."""

    @staticmethod
    def forward(ctx, x, c):
        x = _c(x)
        n, d, h, w, cp = x.shape
        co = pad8(3 * c)
        hw = h * w
        if c % 4 == 0 and d >= 2:
            # every element is written exactly once (float4 permutes): the three shifted copies, the two out-of-range depth slices and
            # the padding channels from a zero row -- no full-tensor memset
            out = _new((n, d, h, w, co), x)
            zrow = _zeros((max(c, co - 3 * c, 4),), x)
            _be().permute(zrow, out, (n, hw, c), (0, 0, 1), (d * hw * co, co, 1), False, 0, 0)                               # kd = 0 at d = 0
            _be().permute(zrow, out, (n, hw, c), (0, 0, 1), (d * hw * co, co, 1), False, 0, (d - 1) * hw * co + 2 * c)       # kd = 2 at d = D-1
            if co > 3 * c:
                _be().permute(zrow, out, (n * d * hw, co - 3 * c), (0, 1), (co, 1), False, 0, 3 * c)
        else:
            out = _zeros((n, d, h, w, co), x)
        for kd in range(3):
            sh = kd - 1                                   # out[d] <- x[d + sh]
            d0, d1 = max(0, -sh), min(d, d - sh)          # valid output depths
            if d1 > d0:
                _be().permute(x, out, (n, d1 - d0, hw, c), (d * hw * cp, hw * cp, cp, 1), (d * hw * co, hw * co, co, 1), False,
                              (d0 + sh) * hw * cp, d0 * hw * co + kd * c)
        ctx.meta = (tuple(x.shape), c)
        return out

    @staticmethod
    def backward(ctx, g):
        (n, d, h, w, cp), c = ctx.meta
        g = _c(g)
        co = g.shape[-1]
        gx = _zeros((n, d, h, w, cp), g)
        hw = h * w
        for kd in range(3):
            sh = kd - 1
            d0, d1 = max(0, -sh), min(d, d - sh)
            if d1 > d0:
                _be().permute(g, gx, (n, d1 - d0, hw, c), (d * hw * co, hw * co, co, 1), (d * hw * cp, hw * cp, cp, 1), True,
                              d0 * hw * co + kd * c, (d0 + sh) * hw * cp)
        return gx, None


def fold_depth3(x, c):
    return _FoldDepth3.apply(x, c)


class _ConcatC(Function):
    @staticmethod
    def forward(ctx, a, b):
        a, b = _c(a), _c(b)
        ca, cb = a.shape[-1], b.shape[-1]
        rows = a.numel() // ca
        out = _new(tuple(a.shape[:-1]) + (ca + cb,), a)
        _be().permute(a, out, (rows, ca), (ca, 1), (ca + cb, 1), False, 0, 0)
        _be().permute(b, out, (rows, cb), (cb, 1), (ca + cb, 1), False, 0, ca)
        ctx.meta = (tuple(a.shape), tuple(b.shape))
        return out

    @staticmethod
    def backward(ctx, g):
        sa, sb = ctx.meta
        g = _c(g)
        ca, cb = sa[-1], sb[-1]
        rows = _numel(sa) // ca
        ga, gb = _new(sa, g), _new(sb, g)
        _be().permute(g, ga, (rows, ca), (ca + cb, 1), (ca, 1), False, 0, 0)
        _be().permute(g, gb, (rows, cb), (ca + cb, 1), (cb, 1), False, ca, 0)
        return ga, gb


def concat_channels(a, b):
    return _ConcatC.apply(a, b)


class _GatherFrames(Function):
    """x: [N,T,P] (P = pixels*channels per frame) -> [G*N, P] with group g = frame idxs[g]
    (ref: dgmr/discriminators.py:199-202; indices may repeat, so backward accumulates per group)."""

    @staticmethod
    def forward(ctx, x, idxs):
        x = _c(x)
        n, t, p = x.shape
        out = _new((len(idxs) * n, p), x)
        for g, i in enumerate(idxs):
            _be().permute(x, out, (n, p), (t * p, 1), (p, 1), False, i * p, g * n * p)
        ctx.meta = (tuple(x.shape), tuple(idxs))
        return out

    @staticmethod
    def backward(ctx, go):
        (n, t, p), idxs = ctx.meta
        go = _c(go)
        gx = _zeros((n, t, p), go)
        for g, i in enumerate(idxs):
            _be().permute(go, gx, (n, p), (p, 1), (t * p, 1), True, g * n * p, i * p)
        return gx, None


def gather_frames(x, idxs):
    return _GatherFrames.apply(x, tuple(int(i) for i in idxs))


class _RepeatMid(Function):
    """x [A, P] -> [A, R, P] (broadcast); backward sums over R (ref: latent batch repeat generators.py:146-148)."""

    @staticmethod
    def forward(ctx, x, r):
        x = _c(x)
        a, p = x.shape
        out = _new((a, r, p), x)
        _be().permute(x, out, (a, r, p), (p, 0, 1), (r * p, p, 1), False, 0, 0)
        ctx.r = r
        return out

    @staticmethod
    def backward(ctx, g):
        g = _c(g)
        a, r, p = g.shape
        gx = _new((a, p), g)
        _be().reduce_mid(g, gx, a, r, p, False)
        return gx, None


def repeat_mid(x, r):
    return _RepeatMid.apply(x, r)


class _ReduceMid(Function):
    """x [A, R, C] -> [A, C] sum over R (ref: torch.sum over stacked per-frame scores, discriminators.py:229-231)."""

    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        a, r, c = x.shape
        y = _new((a, c), x)
        _be().reduce_mid(x, y, a, r, c, False)
        ctx.r = r
        return y

    @staticmethod
    def backward(ctx, g):
        g = _c(g)
        a, c = g.shape
        gx = _new((a, ctx.r, c), g)
        _be().permute(g, gx, (a, ctx.r, c), (c, 0, 1), (ctx.r * c, c, 1), False, 0, 0)
        return gx


def reduce_mid(x):
    return _ReduceMid.apply(x)


# ----------------------------------------------------------------------------- pointwise
class _Relu(Function):
    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        y = torch.empty_like(x)
        _be().relu_fwd(x, y)
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        g = _c(g)
        dx = torch.empty_like(x)
        _be().relu_bwd(g, x, dx)
        return dx


def relu(x):
    return _Relu.apply(x)


class _Pool(Function):
    """sum-pool * scale; backward = nearest upsample * scale."""

    @staticmethod
    def forward(ctx, x, pd, ph, pw, scale):
        x = _c(x)
        n, d, h, w, c = x.shape
        y = _new((n, d // pd, h // ph, w // pw, c), x)
        _be().pool_sum(x, y, n, d, h, w, c, pd, ph, pw, scale)
        ctx.meta = (tuple(x.shape), pd, ph, pw, scale)
        return y

    @staticmethod
    def backward(ctx, g):
        (n, d, h, w, c), pd, ph, pw, scale = ctx.meta
        g = _c(g)
        gx = _new((n, d, h, w, c), g)
        _be().upsample(g, gx, n, d // pd, h // ph, w // pw, c, pd, ph, pw, d, h, w, scale)
        return gx, None, None, None, None


def avg_pool(x, pd, ph, pw):
    """AvgPool2d(2) / AvgPool3d(2) / AvgPool3d((1,2,2)) (ref: dgmr/common.py:189-191; discriminators.py:68,165)."""
    return _Pool.apply(x, pd, ph, pw, 1.0 / (pd * ph * pw))


class _Upsample2(Function):
    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        n, d, h, w, c = x.shape
        y = _new((n, d, 2 * h, 2 * w, c), x)
        _be().upsample(x, y, n, d, h, w, c, 1, 2, 2, d, 2 * h, 2 * w, 1.0)
        return y

    @staticmethod
    def backward(ctx, g):
        g = _c(g)
        n, d, h2, w2, c = g.shape
        gx = _new((n, d, h2 // 2, w2 // 2, c), g)
        _be().pool_sum(g, gx, n, d, h2, w2, c, 1, 2, 2, 1.0)
        return gx


def upsample2(x):
    """Upsample(scale_factor=2, nearest) (ref: dgmr/common.py:121)."""
    return _Upsample2.apply(x)


# ----------------------------------------------------------------------------- spectral norm
class _SpectralSigma(Function):
    """inv_sigma[g] for G consecutive reference calls of one spectrally normalised weight
    (ref: torch/nn/utils/parametrizations.py:495-527).  u, v buffers are updated in place in training."""

    @staticmethod
    def forward(ctx, w, u, v, G, eps, training):
        w = _c(w)
        R = w.shape[0]
        K = w.numel() // R
        inv_sigma = _new((G,), w)
        u_hist, v_hist = _new((G, R), w), _new((G, K), w)
        ws = _new(((G + 2) * R + 2 * G + 8,), w)
        _be().sn_power_iter(w, u, v, R, K, G, eps, training, inv_sigma, u_hist, v_hist, ws)
        ctx.save_for_backward(inv_sigma, u_hist, v_hist)
        ctx.meta = (tuple(w.shape), R, K, G)
        ctx.mark_non_differentiable(u_hist, v_hist)
        return inv_sigma, u_hist, v_hist

    @staticmethod
    def backward(ctx, g_is, _gu, _gv):
        inv_sigma, u_hist, v_hist = ctx.saved_tensors
        wshape, R, K, G = ctx.meta
        dw = _new(wshape, inv_sigma)
        _be().sn_bwd(_c(g_is), inv_sigma, u_hist, v_hist, dw, R, K, G, False)
        return dw, None, None, None, None, None


def spectral_inv_sigma(w, u, v, G, eps, training):
    return _SpectralSigma.apply(w, u, v, G, eps, training)[0]


class _SpectralSigmaMulti(Function):
    """_SpectralSigma for many weights in ONE launch (dgmr_sn_power_iter_multi).  Inputs: the n weights; meta carries the
    (u, v, G, eps) of each.  Outputs: n inv_sigma tensors (views of one allocation)."""

    @staticmethod
    def forward(ctx, meta, training, *ws_):
        n = len(ws_)
        sizes, items = [], []
        for w, (u, v, G, eps) in zip(ws_, meta):
            R = w.shape[0]
            K = w.numel() // R
            sizes.append((R, K, G))
        out_tot = sum(G + G * R + G * K for R, K, G in sizes)
        ws_tot = sum((G + 2) * R + 2 * G + 8 for R, K, G in sizes)
        out = _new((out_tot,), ws_[0])
        scratch = _zeros((ws_tot,), ws_[0])
        o = s = 0
        res, hist = [], []
        for w, (u, v, G, eps), (R, K, _) in zip(ws_, meta, sizes):
            inv_sigma = out[o:o + G]; o += G
            u_hist = out[o:o + G * R].view(G, R); o += G * R
            v_hist = out[o:o + G * K].view(G, K); o += G * K
            wsz = (G + 2) * R + 2 * G + 8
            items.append(dict(w=_c(w.detach()), u=u, v=v, R=R, K=K, G=G, eps=eps, training=training, inv_sigma=inv_sigma,
                              u_hist=u_hist, v_hist=v_hist, ws=scratch[s:s + wsz]))
            s += wsz
            res.append(inv_sigma)
            hist.append((u_hist, v_hist))
        _be().sn_power_iter_multi(items)
        ctx.hist = hist
        ctx.sizes = sizes
        ctx.shapes = [tuple(w.shape) for w in ws_]
        ctx.save_for_backward(*res)
        return tuple(r.clone() for r in res) if False else tuple(res)

    @staticmethod
    def backward(ctx, *gs):
        inv = ctx.saved_tensors
        todo = [(i, g, inv_sigma, hist, size, shape) for i, (g, inv_sigma, hist, size, shape, need) in
                enumerate(zip(gs, inv, ctx.hist, ctx.sizes, ctx.shapes, ctx.needs_input_grad[2:])) if g is not None and need]
        outs = [None] * len(gs)
        if todo:   # the rank-G corrections of all the weights in ONE launch, into views of one allocation
            flat = _new((sum(R * K for _, _, _, _, (R, K, G), _ in todo),), inv[0])
            o, items = 0, []
            for i, g, inv_sigma, (u_hist, v_hist), (R, K, G), shape in todo:
                dw = flat[o:o + R * K].view(shape); o += R * K
                items.append(dict(d_inv_sigma=_c(g), inv_sigma=_c(inv_sigma), u_hist=u_hist, v_hist=v_hist, dw=dw, R=R, K=K, G=G, accumulate=False))
                outs[i] = dw
            _be().sn_bwd_multi(items)
        return (None, None) + tuple(outs)


def spectral_inv_sigma_multi(entries, training):
    """entries: list of (w, u, v, G, eps) -> list of inv_sigma[G] tensors, one kernel launch for all of them."""
    meta = tuple((u, v, G, eps) for (_, u, v, G, eps) in entries)
    return list(_SpectralSigmaMulti.apply(meta, training, *[e[0] for e in entries]))


# ----------------------------------------------------------------------------- convolution
import weakref  # noqa: E402

_packed_params = {}   # id(Parameter) -> weakref: the Parameters that carry a pack cache (only so that clear_pack_cache can find them)


def mark_conv_only(t: torch.Tensor) -> torch.Tensor:
    """Declare that `t` is consumed by convolutions only (or through sign-preserving ops such as ReLU), so its tf32
    rounding may happen in place.  Anything else that reads a tensor (BatchNorm statistics, gate arithmetic, residuals)
    must see the unrounded fp32 values, like in the reference, so unmarked conv inputs are rounded into a private copy."""
    t._dgmr_conv_only = True
    return t


def _round_(t: torch.Tensor) -> torch.Tensor:
    """The tf32-rounded version of a conv operand: `t` itself if already rounded, rounded in place if it is conv-only
    (flag rides on the Python tensor object), else a rounded copy."""
    if getattr(t, "_dgmr_tf32", False):
        return t
    r = getattr(t, "_dgmr_rounded", None)
    if r is not None:                      # a producer already wrote the rounded copy (BatchNorm branch node)
        return r
    if getattr(t, "_dgmr_conv_only", False):
        _be().round_tf32(t)
        t._dgmr_tf32 = True
        return t
    r = torch.empty_like(t)
    _be().round_tf32(t, r)
    r._dgmr_tf32 = True
    return r


class _ConvOperand(Function):
    """Identity in autograd; forward hands out the tf32-rounded copy that several convs of the same input can share
    (e.g. the read- and update-gate convs of one ConvGRU step both consume h)."""

    @staticmethod
    def forward(ctx, x):
        if not _rounding_on() or getattr(x, "_dgmr_tf32", False):     # already rounded by its producer's epilogue: pass through
            return x.view_as(x)
        return _round_(_c(x).detach())

    @staticmethod
    def backward(ctx, g):
        return g


def conv_operand(x):
    y = _ConvOperand.apply(x)
    if getattr(x, "_dgmr_tf32", False):
        y._dgmr_tf32 = True
    return y


def _rounding_on() -> bool:
    """Are conv operands rounded to tf32 at all (1xTF32 tensor-core mode on the CUDA library)?"""
    return config.round_tf32 and config.conv_algo != ALGO_SIMT and config.precision == PREC_TF32 and _be().name == "cuda"


def _tc_fwd(n, d, h, w, cin, cout, kd, kh, kw) -> bool:
    """Will dgmr_conv_fwd serve this shape on the tensor cores in 1xTF32 mode (and should operands therefore be tf32-rounded)?"""
    return (config.round_tf32 and config.precision == PREC_TF32 and config.conv_algo != ALGO_SIMT
            and _be().conv_umma_supported(n, d, h, w, cin, cout, kd, kh, kw))


def _tc_wgrad(n, d, h, w, cin, cout, kd, kh, kw) -> bool:
    return (config.round_tf32 and config.precision == PREC_TF32 and config.wgrad_algo != ALGO_SIMT
            and _be().wgrad_umma_supported(n, d, h, w, cin, cout, kd, kh, kw))


def _x3_fwd(n, d, h, w, cin, cout, kd, kh, kw) -> bool:
    """Parity mode and the tcgen05 path serves the shape: operands go in as 3xTF32 (hi, lo) pairs."""
    return (config.precision == PREC_3XTF32 and config.conv_algo != ALGO_SIMT and _be().name == "cuda"
            and _be().conv_umma_supported(n, d, h, w, cin, cout, kd, kh, kw))


def _x3_wgrad(n, d, h, w, cin, cout, kd, kh, kw) -> bool:
    return (config.precision == PREC_3XTF32 and config.wgrad_algo != ALGO_SIMT and _be().name == "cuda"
            and _be().wgrad_umma_supported(n, d, h, w, cin, cout, kd, kh, kw))


def _split(t: torch.Tensor):
    hl = _new((2,) + tuple(t.shape), t)
    _be().split_tf32(t, hl[0], hl[1])
    return hl[0], hl[1]


def _use_split_taps(n, d, h, w, cin, cout, taps, has_bias, act) -> bool:
    """Tap-split accumulate mode pays when the plain tiling leaves most SMs idle: few 128-pixel x 256-channel tiles, many taps."""
    if not config.split_taps or taps == 1 or has_bias or act != ACT_NONE or config.conv_algo == ALGO_SIMT:
        return False
    tiles = ((n * d * h * w + 127) // 128) * ((cout + 255) // 256)
    return tiles <= 32 and cin >= 32 and _be().name == "cuda" and _be().conv_umma_supported(n, d, h, w, cin, cout, 1, 3, 3)   # measured crossover (tests/time_gru_conv.py)


def _pack_slot(w: torch.Tensor):
    """The per-Parameter cache of packed copies.  It lives ON the Parameter object (so it dies with it: a new model whose
    storage lands on a freed model's addresses can never see the old packs) and each entry remembers the storage it was
    packed from (data pointer, device) and the parameter's version counter (moved by the optimiser step)."""
    if not isinstance(w, torch.nn.Parameter):
        # temporaries (e.g. the concatenated gate weights of a ConvGRU) are not cached: they can die and hand their
        # address + version 0 to the next temporary
        return None
    slot = w.__dict__.get("_dgmr_packs")
    if slot is None:
        slot = w.__dict__["_dgmr_packs"] = {}
        k = id(w)
        _packed_params[k] = weakref.ref(w, lambda _r, k=k: _packed_params.pop(k, None))
    return slot


def _pack_lookup(slot, w, key):
    if slot is None:
        return None
    hit = slot.get(key)
    if hit is not None and hit[0] == (w._version, w.data_ptr(), str(w.device)):
        return hit[1]
    return None


def _pack_store(slot, w, key, p):
    if slot is not None:
        slot[key] = ((w._version, w.data_ptr(), str(w.device)), p)


def packed_weight(w: torch.Tensor, ci0: int, cin: int, mode: int) -> torch.Tensor:
    """[tap][Cout][Cin] (mode 0) / flipped-transposed dgrad pack (mode 1) of the OIHW weight slice
    [:, ci0:ci0+cin]; cached on the Parameter until its version counter (or storage) moves.
    mode | FLAG_ROUND_TF32: tf32-rounded."""
    slot = _pack_slot(w)
    key = (ci0, cin, mode)
    hit = _pack_lookup(slot, w, key)
    if hit is not None:
        return hit
    cout, cintot = w.shape[0], w.shape[1]
    taps = w.numel() // (cout * cintot)
    p = _new((taps * cout * cin,), w)
    _be().pack_weight(_c(w.detach()), p, cout, cintot, ci0, cin, taps, mode & ~(FLAG_SPLIT | (FLAG_ROUND_TF32 if mode & FLAG_SPLIT else 0)))
    if mode & FLAG_SPLIT:   # parity mode: [2, n] = (hi, lo) of the unrounded pack
        p = torch.stack(_split(p))
    _pack_store(slot, w, key, p)
    return p


def packed_weight_padded(w: torch.Tensor, ci0: int, cin: int, cin_p: int, mode: int) -> torch.Tensor:
    """Like packed_weight but with the input-channel axis zero-padded to cin_p (the 4-channel space-to-depth inputs
    are carried as 8 channels so that the tensor-core path, whose K step is 8 tf32, can serve them)."""
    slot = _pack_slot(w)
    key = (ci0, cin, ("pad", cin_p, mode))
    hit = _pack_lookup(slot, w, key)
    if hit is not None:
        return hit
    cout, cintot = w.shape[0], w.shape[1]
    taps = w.numel() // (cout * cintot)
    p = _zeros((taps * cout * cin_p,), w)     # the pad rows / columns stay zero: the pack kernel writes the [cin] window only
    split = mode & FLAG_SPLIT
    kmode = mode & ~(FLAG_SPLIT | (FLAG_ROUND_TF32 if split else 0))
    _be().pack_weight_multi([dict(w=_c(w.detach()), packed=p, Cout=cout, CinTot=cintot, ci0=ci0, Cin=cin, taps=taps, mode=kmode,
                                  CinPad=cin_p, co0=0, CoutTot=cout)])
    if split:
        p = torch.stack(_split(p))
    _pack_store(slot, w, key, p)
    return p


def refresh_packs(params) -> int:
    """Re-pack, IN PLACE and in one launch per 64 packs, every cached packed copy of `params` that an optimiser step made stale
    (the optimiser calls this right after its update): from the second step on a network's ~100-200 packs cost a couple of
    launches instead of one launch each at first use.  Parity-mode (hi, lo) pairs are simply dropped and rebuilt on demand.
    In the 1xTF32 mode every pack keeps its address across optimiser steps (inference.GraphedGenerator(train_mode=True) relies on it)."""
    items, touched = [], []
    for w in params:
        slot = w.__dict__.get("_dgmr_packs")
        if not slot:
            continue
        tag = (w._version, w.data_ptr(), str(w.device))
        cout, cintot = w.shape[0], w.shape[1]
        taps = w.numel() // (cout * cintot)
        for key in list(slot):
            if slot[key][0] == tag:
                continue
            ci0, cin, m = key
            pad = cin
            if isinstance(m, tuple) and m[0] == "sub":   # pre-summed sub-pixel tiles: their own kernel (8 small launches per step), also in place --
                _be().pack_weight_subpix(_c(w.detach()), slot[key][1], cout, cintot, 0, cin, m[1])   # a captured CUDA graph keeps reading this buffer
                slot[key] = (tag, slot[key][1])
                continue
            if isinstance(m, tuple):
                _, pad, m = m
            if m & FLAG_SPLIT:
                del slot[key]
                continue
            items.append(dict(w=_c(w.detach()), packed=slot[key][1], Cout=cout, CinTot=cintot, ci0=ci0, Cin=cin, taps=taps, mode=m,
                              CinPad=pad, co0=0, CoutTot=cout))
            touched.append((slot, key, tag))
    if items:
        _be().pack_weight_multi(items)
        for slot, key, tag in touched:
            slot[key] = (tag, slot[key][1])
    return len(items)


def clear_pack_cache():
    for r in list(_packed_params.values()):
        w = r()
        if w is not None:
            w.__dict__.pop("_dgmr_packs", None)
    _packed_params.clear()


def _takes_split_taps(n, d, h, wd, c, cout, kd, kh, kw, has_bias, act, has_lo) -> bool:
    """Whether `_conv_launch` serves this call in the tap-split accumulate mode (callers that pre-zero the output ask first)."""
    return _use_split_taps(n, d, h, wd, c, cout, kd * kh * kw, has_bias, act) and _be().conv_umma_supported(n, d, h, wd, c, cout, kd, kh, kw) \
        and (config.precision == PREC_TF32 or has_lo)   # (any epilogue flag in `act` makes act != ACT_NONE: no tap split)


def _conv_launch(x, wp, bias, scale, res, y, n, d, h, wd, c, cout, kd, kh, kw, G, act, y_is_zero=False):
    """y = act(conv(x, wp) * scale + bias + res) through the C ABI; picks the tap-split accumulate mode for launches that
    would otherwise leave most SMs idle.  `res` may alias `y` (each element is read, then written, by the same thread).
    wp of shape [2, n] is a 3xTF32 (hi, lo) pair (parity mode): x is split the same way here.
    y_is_zero: the caller zeroed `y` (one fill for a whole sequence of calls) after `_takes_split_taps` said the accumulate mode applies."""
    be = _be()
    x_lo = wp_lo = None
    if wp.dim() == 2:
        wp, wp_lo = wp[0], wp[1]
        x, x_lo = _split(x)
    split = _takes_split_taps(n, d, h, wd, c, cout, kd, kh, kw, bias is not None, act, x_lo is not None)
    if y_is_zero and not (split and res is None):
        raise RuntimeError("dgmr_b200: _conv_launch(y_is_zero=True) outside the tap-split accumulate mode")
    if split:
        if y_is_zero:
            pass
        elif res is None:
            be.fill(y, 0.0)
        elif res.data_ptr() != y.data_ptr():
            be.axpby(1.0, res, 0.0, None, y)   # y starts as the residual, the taps accumulate on top
        be.conv_fwd(x, wp, None, scale, None, y, n, d, h, wd, c, cout, kd, kh, kw, G, ACT_NONE | FLAG_ACCUMULATE,
                    config.conv_algo, config.precision, x_lo=x_lo, wp_lo=wp_lo)
    else:
        be.conv_fwd(x, wp, bias, scale, res, y, n, d, h, wd, c, cout, kd, kh, kw, G, act, config.conv_algo, config.precision,
                    x_lo=x_lo, wp_lo=wp_lo)


def _wgrad_launch(x, dz, dwp, n, d, h, wd, cin, cout, kd, kh, kw):
    """dwp = wgrad(x, dz) through the C ABI; parity mode splits both operands into 3xTF32 pairs when the tcgen05 path takes the shape."""
    be = _be()
    if _x3_wgrad(n, d, h, wd, cin, cout, kd, kh, kw) and (dwp.data_ptr() & 15) == 0:
        xh, xl = _split(x)
        zh, zl = _split(dz)
        be.conv_wgrad(xh, zh, dwp, n, d, h, wd, cin, cout, kd, kh, kw, config.wgrad_algo, config.precision, x_lo=xl, dz_lo=zl)
    else:
        be.conv_wgrad(x, dz, dwp, n, d, h, wd, cin, cout, kd, kh, kw, config.wgrad_algo, config.precision)


class _Conv(Function):
    """y = act( conv(x, w[:, ci0:ci0+cin]) * scale[g, co] + bias + res ).  Kernel extents 1 or 3, same padding.
    res_up2: `res` is a half-resolution tensor added nearest-upsampled (read at (h/2, w/2) in the conv epilogue; its gradient is the
    2x2 sum-pool of the full-resolution one).  round_out: the output feeds tensor-core convolutions only and is written tf32-rounded
    by the epilogue (no separate rounding pass); ignored unless the 1xTF32 tensor-core mode is on."""

    @staticmethod
    def forward(ctx, x, w, bias, scale, res, ci0, cin, G, act, exact_dscale=False, res_up2=False, round_out=False, pool=None):
        """pool = (pd, ph, pw): the result is average-pooled (floor) and the POOLED tensor is returned (DBlock: conv -> AvgPool, ref:
        dgmr/common.py:234-236); fusing the two nodes lets the backward prologue read the pooled gradient directly (no upsample pass)."""
        x = _c(x)
        n, d, h, wd, c = x.shape
        assert c == cin or (c > cin and c == (cin + 7) // 8 * 8), (c, cin)   # c > cin: zero-padded input channels
        cout = w.shape[0]
        ks = tuple(w.shape[2:])
        kd, kh, kw = (1,) * (3 - len(ks)) + ks
        rnd = FLAG_ROUND_TF32 if _tc_fwd(n, d, h, wd, c, cout, kd, kh, kw) else 0
        if rnd and config._dbg_round_act:
            x = _round_(x)
        if not config._dbg_round_w:
            rnd = 0
        if _x3_fwd(n, d, h, wd, c, cout, kd, kh, kw):
            rnd = FLAG_SPLIT
        wp = packed_weight(w, ci0, cin, rnd) if c == cin else packed_weight_padded(w, ci0, cin, c, rnd)
        y = _new((n, d, h, wd, cout), x)
        res_c, scale_c, bias_c = _c(res), _c(scale), _c(bias)
        res_up2 = bool(res_up2 and res is not None)
        round_out = bool(round_out and _rounding_on())
        _conv_launch(x, wp, bias_c, scale_c, res_c, y, n, d, h, wd, c, cout, kd, kh, kw, G,
                     act | (FLAG_RES_UP2 if res_up2 else 0) | (FLAG_ROUND_OUT if round_out else 0))
        if round_out:
            y._dgmr_tf32 = True
        need_s = scale is not None and scale.requires_grad
        # one sigma for the whole batch (G = 1): the scale gradient comes from the weight gradient, <dW[co], W[co]> / s[co], instead of a
        # reduction over the activations -- y (and the residual) need not be kept or re-read for it
        wdot = bool(need_s and G == 1 and w.requires_grad and not exact_dscale and config.dscale_from_wgrad)
        need_y = act == ACT_RELU or (need_s and not wdot)
        ctx.save_for_backward(x, w, bias_c, scale_c, res_c if (need_s and not wdot) else None, y if need_y else None)
        ctx.meta = (ci0, cin, G, act, (kd, kh, kw), res is not None, exact_dscale, res_up2, pool, wdot)
        if pool:
            pd, ph, pw = pool
            yp = _new((n, d // pd, h // ph, wd // pw, cout), x)
            _be().pool_sum(y, yp, n, d, h, wd, cout, pd, ph, pw, 1.0 / (pd * ph * pw))
            return yp
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, bias, scale, res, y = ctx.saved_tensors
        ci0, cin, G, act, (kd, kh, kw), has_res, exact_dscale, res_up2, pool, wdot = ctx.meta
        be = _be()
        dy = _c(dy)
        n, d, h, wd, cp = x.shape   # cp > cin: zero-padded input channels
        cout = w.shape[0]
        rows = (n // G) * d * h * wd
        full_shape = (n, d, h, wd, cout)
        if pool and not (act == ACT_RELU or scale is not None or (ctx.needs_input_grad[2] and bias is not None)):
            # no prologue will run: undo the pooling explicitly
            g_full = _new(full_shape, dy)
            be.upsample(dy, g_full, n, d // pool[0], h // pool[1], wd // pool[2], cout, pool[0], pool[1], pool[2], d, h, wd, 1.0 / (pool[0] * pool[1] * pool[2]))
            dy, pool = g_full, None
        need_x, need_w, need_b, need_s, need_r = (ctx.needs_input_grad[i] for i in range(5))
        need_b = need_b and bias is not None
        need_s = need_s and scale is not None
        need_r = need_r and has_res
        wdot = wdot and need_s
        need_w = need_w or wdot
        dz, dpre, dbias, dscale = dy, dy, None, None
        if act == ACT_RELU or scale is not None or need_b:
            need_dz = need_x or need_w
            dz = _new(full_shape, dy) if (need_dz and (act == ACT_RELU or scale is not None or pool)) else None
            dpre = _new(full_shape, dy) if (need_r and (act == ACT_RELU or pool)) else None
            dbias = _new((cout,), dy) if need_b else None
            dscale = _new((G, cout), dy) if need_s else None
            tc_bwd = (need_x and _tc_fwd(n, d, h, wd, cout, cp, kd, kh, kw)) or (need_w and _tc_wgrad(n, d, h, wd, cp, cout, kd, kh, kw))
            be.conv_bwd_prep(dy, y, res if (need_s and not wdot) else None, bias, scale, dz, dpre, dbias, None if wdot else dscale, rows, G, cout,
                             act | (FLAG_ROUND_TF32 if (tc_bwd and dz is not None and config._dbg_round_dz) else 0),
                             up_hw=((h, wd) if (res_up2 and need_s and not wdot and res is not None) else (0, 0)),
                             pool=((pool[0], pool[1], pool[2], d, h, wd) if pool else None))
            if need_s and exact_dscale:
                # the <dY, Y-b-res>/scale identity divides by the scale, which may be exactly 0 (attention gamma starts at 0,
                # ref: dgmr/layers/Attention.py:69): recompute the raw conv output and reduce <dpre, z> directly
                assert act == ACT_NONE
                z = _new(dy.shape, dy)
                _conv_launch(x, packed_weight(w, ci0, cin, FLAG_SPLIT if _x3_fwd(n, d, h, wd, cin, cout, kd, kh, kw) else 0), None, None, None, z,
                             n, d, h, wd, cin, cout, kd, kh, kw, 1, ACT_NONE)
                ones = torch.ones((G, cout), device=dy.device, dtype=dy.dtype)
                be.conv_bwd_prep(dy, z, None, None, ones, None, None, None, dscale, rows, G, cout, ACT_NONE,
                                 pool=((pool[0], pool[1], pool[2], d, h, wd) if pool else None))
            if dz is None:
                dz = dy
            elif tc_bwd:
                dz._dgmr_tf32 = True
            if dpre is None:
                dpre = dy
        dx = dw = None
        if (need_x and _tc_fwd(n, d, h, wd, cout, cp, kd, kh, kw)) or (need_w and _tc_wgrad(n, d, h, wd, cp, cout, kd, kh, kw)):
            if config._dbg_round_dz and not getattr(dz, "_dgmr_tf32", False):
                # dz == dy straight from autograd (no prologue ran): it may be shared with other backward nodes -> private copy
                dz = _round_(dz)
        if need_x:
            rnd = FLAG_ROUND_TF32 if (_tc_fwd(n, d, h, wd, cout, cp, kd, kh, kw) and config._dbg_round_w) else 0
            if _x3_fwd(n, d, h, wd, cout, cp, kd, kh, kw):
                rnd = FLAG_SPLIT
            wpt = packed_weight(w, ci0, cin, 1 | rnd) if cp == cin else packed_weight_padded(w, ci0, cin, cp, 1 | rnd)
            dx = _new(x.shape, x)
            _conv_launch(dz, wpt, None, None, None, dx, n, d, h, wd, cout, cp, kd, kh, kw, 1, ACT_NONE)
        if need_w:
            taps = kd * kh * kw
            cintot = w.shape[1]
            dw = _new(w.shape, x) if cin == cintot else _zeros(w.shape, x)
            if kd == 3 and kh == 3 and kw == 3 and cp == cin and 3 * cin <= 160 and cout <= 128 and d >= 3 and _tc_wgrad(n, d, h, wd, 3 * cin, cout, 1, 3, 3) \
                    and wd % 32 == 0 and config.fold_depth_wgrad:
                # 3x3x3 weight gradient of a narrow layer (temporal discriminator, 48 -> 48): with M = Cout and N = Cin both far below the
                # 128-row tensor-core tile every MMA sits at the pipe's ~60-cycle floor, so the count of MMAs is what costs.  Folding the three
                # depth taps into the channel axis (x' = [x(d-1) | x(d) | x(d+1)], 3*Cin channels) turns 9 (kd, kh) filter rows of N = Cin
                # into 3 rows of N = 3*Cin: 2.25x fewer MMAs for the same products.  dW'[(kh,kw)][co][kd*Cin + ci] scatters back onto dW.
                xf = _FoldDepth3.apply(x.detach(), cin)                     # [N, D, H, W, 3*Cin] (pad8(3*cin) == 3*cin: cin % 8 == 0)
                cf = xf.shape[-1]
                dwp = _new((9 * cout * cf,), x)
                _wgrad_launch(xf, dz, dwp, n, d, h, wd, cf, cout, 1, 3, 3)
                # dw[co][ci0 + ci][kd][kh][kw] = dwp[kh*3 + kw][co][kd*cin + ci]
                be.permute(dwp, dw, (9, cout, 3, cin), (cout * cf, cf, cin, 1), (1, cintot * 27, 9, 27), False, 0, ci0 * 27)
            else:
                dwp = _new((taps * cout * cp,), x)
                _wgrad_launch(x, dz, dwp, n, d, h, wd, cp, cout, kd, kh, kw)
                if cp == cin:
                    be.unpack_wgrad(dwp, dw, cout, cintot, ci0, cin, taps, False)
                else:  # drop the padded channels: dw[co][ci0+ci][tap] = dwp[tap][co][ci], ci < cin
                    be.permute(dwp, dw, (taps, cout, cin), (cout * cp, cp, 1), (1, cintot * taps, taps), False, 0, ci0 * taps)
        if wdot:
            taps = kd * kh * kw
            be.rowdot_div(dw, w, scale, dscale, cout, cin * taps, w.shape[1] * taps, ci0 * taps)
            if not ctx.needs_input_grad[1]:
                dw = None
        dres = None
        if need_r:
            dres = dpre
            if res_up2:   # gradient of the half-resolution residual: 2x2 sum-pool of the full-resolution one
                dres = _new((n, d, h // 2, wd // 2, cout), dy)
                be.pool_sum(_c(dpre), dres, n, d, h, wd, cout, 1, 2, 2, 1.0)
        return dx, dw, dbias, dscale, dres, None, None, None, None, None, None, None, None


def conv(x, w, bias=None, scale=None, res=None, ci0=0, cin=None, G=1, act=ACT_NONE, exact_dscale=False, res_up2=False, round_out=False,
         pool=None):
    if cin is None:
        cin = w.shape[1]
    return _Conv.apply(x, w, bias, scale, res, ci0, cin, G, act, exact_dscale, res_up2, round_out, pool)


# ----------------------------------------------------------------------------- BatchNorm
class _BatchNorm(Function):
    """y = act(BN(x)) with per-group batch statistics (training) or running statistics (eval),
    optional fused ReLU and nearest x2 upsample of the output.  Running stats are updated in place,
    sequentially over the G groups, exactly as G separate reference calls would
    (ref: dgmr/common.py:74-82,145-153; generators.py:176)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, rmean, rvar, G, training, relu_, up2, eps, momentum, conv_only=False, branch=False):
        be = _be()
        x = _c(x)
        n, d, h, w, c = x.shape
        rows = (n // G) * d * h * w
        sums = _new((G, c, 2), x, torch.float64)
        if training:
            if rows <= 1:
                raise ValueError("Expected more than 1 value per channel when training")
            be.bn_stats(x, sums, rows, G, c)
        mean, invstd, a, b = (_new((G, c), x) for _ in range(4))
        be.bn_finalize(sums, gamma, beta, rmean, rvar, rows, G, c, eps, momentum, training, mean, invstd, a, b)
        y = _new((n, d, 2 * h, 2 * w, c) if up2 else (n, d, h, w, c), x)
        rnd = conv_only and _rounding_on()
        # branch: the shortcut convolution wants x tf32-rounded (a private copy: this BatchNorm must see the unrounded values) -- written by
        # this pass, which reads x anyway, instead of by a rounding pass of its own
        xr = _new(x.shape, x) if (branch and _rounding_on() and not up2 and not getattr(x, "_dgmr_tf32", False)) else None
        be.bn_apply(x, a, b, y, rows, G, c, int(relu_) | (FLAG_ROUND_TF32 if rnd else 0), up2, h, w, x_rounded=xr)
        if rnd:
            y._dgmr_tf32 = True
        ctx.save_for_backward(x, gamma, a, b, mean, invstd)
        ctx.meta = (G, training, relu_, up2)
        if branch:
            # second output: the input itself, for its OTHER consumer (the residual shortcut).  Routing that use through this node means
            # the two gradients of x meet in backward(), where dgmr_bn_bwd_apply adds the shortcut's while it writes dx -- instead of
            # autograd accumulating them in a separate read-read-write pass over the activation.
            if xr is not None:
                ctx.mark_non_differentiable(xr)
                return y, x.view_as(x), xr
            return y, x.view_as(x)
        return y

    @staticmethod
    def backward(ctx, dy, dskip=None, _dxr=None):
        x, gamma, a, b, mean, invstd = ctx.saved_tensors
        G, training, relu_, up2 = ctx.meta
        be = _be()
        dy = _c(dy)
        n, d, h, w, c = x.shape
        rows = (n // G) * d * h * w
        red = _new((G, c, 2), x, torch.float64)
        be.bn_bwd_reduce(dy, x, a, b, mean, invstd, red, rows, G, c, relu_, up2, h, w)
        dx = _new(x.shape, x) if ctx.needs_input_grad[0] else None
        dgamma = _new((c,), x) if (gamma is not None and ctx.needs_input_grad[1]) else None
        dbeta = _new((c,), x) if (gamma is not None and ctx.needs_input_grad[2]) else None
        if dy is None:      # only the shortcut carried a gradient
            return (_c(dskip) if ctx.needs_input_grad[0] else None), None, None, None, None, None, None, None, None, None, None, None, None
        be.bn_bwd_apply(dy, x, a, b, mean, invstd, None, red, dx, dgamma, dbeta, False, rows, G, c, relu_, up2, h, w, training,
                        dx_add=(_c(dskip) if (dskip is not None and dx is not None) else None))
        return dx, dgamma, dbeta, None, None, None, None, None, None, None, None, None, None


def batch_norm(x, gamma, beta, rmean, rvar, G, training, relu_=False, up2=False, eps=1e-5, momentum=0.1, conv_only=False, branch=False):
    """conv_only: the result is consumed by convolutions only, so it may be emitted tf32-rounded straight away.
    branch: returns (y, x_skip) -- x_skip is the input, to be handed to its other consumer (see _BatchNorm.forward)."""
    out = _BatchNorm.apply(x, gamma, beta, rmean, rvar, G, training, relu_, up2, eps, momentum, conv_only, branch)
    if branch and len(out) == 3:
        y, skip, xr = out
        xr._dgmr_tf32 = True
        skip._dgmr_rounded = xr          # picked up by _round_ when the shortcut convolution asks for its operand
        return y, skip
    return out


# ----------------------------------------------------------------------------- nearest x2 -> 3x3 conv, sub-pixel form
def upconv_available(n, h, w, cin, cout) -> bool:
    """Do the sub-pixel tensor-core kernels (forward, dgrad, wgrad) serve this up-convolution in the current mode?"""
    if not config.upconv:
        return False
    if config._force_upconv:
        return True
    return _rounding_on() and _be().upconv_supported(n, h, w, cin, cout)


def packed_weight_subpix(w: torch.Tensor, cin: int, mode: int) -> torch.Tensor:
    """The 16 pre-summed [Cout][Cin] tiles (mode 0) / their transposes (mode 1) of a 3x3 weight (dgmr_pack_weight_subpix), cached on the
    Parameter like the ordinary packs."""
    slot = _pack_slot(w)
    key = (0, cin, ("sub", mode))
    hit = _pack_lookup(slot, w, key)
    if hit is not None:
        return hit
    cout = w.shape[0]
    p = _new((16 * cout * cin,), w)
    _be().pack_weight_subpix(_c(w.detach()), p, cout, w.shape[1], 0, cin, mode)
    _pack_store(slot, w, key, p)
    return p


def _upconv_fwd(x, w, bias, scale, res, G, act):
    """x: [N,1,H,W,Cin] LOW resolution (tf32-rounded if rounding is on) -> y [N,1,2H,2W,Cout] = act(conv3x3(up2(x), w) * scale + bias + res)."""
    n, d, h, wd, c = x.shape
    assert d == 1 and tuple(w.shape[2:]) == (3, 3) and w.shape[1] == c, (x.shape, w.shape)
    cout = w.shape[0]
    wsp = packed_weight_subpix(w, c, FLAG_ROUND_TF32 if _rounding_on() else 0)
    y = _new((n, 1, 2 * h, 2 * wd, cout), x)
    _be().upconv_fwd(x, wsp, bias, scale, res, y, n, h, wd, c, cout, G, act)
    return y


def _upconv_bwd(x, w, dz, need_x, need_w):
    """dz: [N,1,2H,2W,Cout] (scaled, rounded) -> (dx [N,1,H,W,Cin], dw like w)."""
    be = _be()
    n, d, h, wd, c = x.shape
    cout = w.shape[0]
    dx = dw = None
    if need_x:
        wspt = packed_weight_subpix(w, c, 1 | (FLAG_ROUND_TF32 if _rounding_on() else 0))
        dx = _new(x.shape, x)
        be.upconv_dgrad(dz, wspt, dx, n, h, wd, c, cout)
    if need_w:
        dwsp = _new((16 * cout * c,), x)
        be.upconv_wgrad(x, dz, dwsp, n, h, wd, c, cout)
        dw = _new(w.shape, x)
        be.unpack_wgrad_subpix(dwsp, dw, cout, w.shape[1], 0, c, False)
    return dx, dw


class _UpConv(Function):
    """y = act(conv3x3(nearest_up2(x), w) * scale[g, co] + bias) computed on the LOW-resolution x in sub-pixel form (ref: UpsampleGBlock,
    dgmr/common.py:146-149): 2.25x fewer MACs, no upsampled tensor.  Caller checks upconv_available()."""

    @staticmethod
    def forward(ctx, x, w, bias, scale, G, act, round_out):
        x = _c(x)
        if _rounding_on() and config._dbg_round_act:
            x = _round_(x)
        scale_c, bias_c = _c(scale), _c(bias)
        round_out = bool(round_out and _rounding_on())
        y = _upconv_fwd(x, w, bias_c, scale_c, None, G, act | (FLAG_ROUND_OUT if round_out else 0))
        if round_out:
            y._dgmr_tf32 = True
        need_s = scale is not None and scale.requires_grad
        ctx.save_for_backward(x, w, bias_c, scale_c, y if (act == ACT_RELU or need_s) else None)
        ctx.meta = (G, act)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, bias, scale, y = ctx.saved_tensors
        G, act = ctx.meta
        be = _be()
        dy = _c(dy)
        n, d, h, wd, c = x.shape
        cout = w.shape[0]
        rows = (n // G) * 4 * h * wd
        need_x, need_w, need_b, need_s = (ctx.needs_input_grad[i] for i in range(4))
        need_b = need_b and bias is not None
        need_s = need_s and scale is not None
        dz = _new(dy.shape, dy)
        dbias = _new((cout,), dy) if need_b else None
        dscale = _new((G, cout), dy) if need_s else None
        be.conv_bwd_prep(dy, y, None, bias, scale, dz, None, dbias, dscale, rows, G, cout,
                         act | (FLAG_ROUND_TF32 if (_rounding_on() and config._dbg_round_dz) else 0))
        dx, dw = _upconv_bwd(x, w, dz, need_x, need_w)
        return dx, dw, dbias, dscale, None, None, None


def upconv(x, w, bias=None, scale=None, G=1, act=ACT_NONE, round_out=False):
    """conv3x3(nearest_up2(x)): sub-pixel kernels where available, else the materialised upsample + ordinary convolution."""
    n, d, h, wd, c = x.shape
    if d == 1 and tuple(w.shape[2:]) == (3, 3) and upconv_available(n, h, wd, c, w.shape[0]):
        return _UpConv.apply(x, w, bias, scale, G, act, round_out)
    return conv(mark_conv_only(upsample2(x)), w, bias, scale, None, 0, c, G, act, round_out=round_out)


class _ConvBNRelu(Function):
    """relu(BN_train(conv(x, w) * scale[g] + bias)) as ONE autograd node (GBlock / UpsampleGBlock: first_conv_3x3 -> bn2 -> ReLU,
    ref: dgmr/common.py:76-80, 146-151), train mode only.

    Fusing the two nodes is what makes the backward cheap: under batch-statistics BatchNorm the loss cannot depend on a per-channel
    scale or shift of the BatchNorm input, so the convolution's bias and spectral-norm-scale gradients are IDENTICALLY zero (the
    reference computes rounding noise there) and its output gradient is the BatchNorm input gradient -- which dgmr_bn_bwd_apply
    writes already multiplied by scale[g] and tf32-rounded, i.e. as the operand of dgrad / wgrad.  No conv_bwd_prep pass, no
    <dY, Y - b> reduction, and the conv output is saved once (as the BatchNorm input) instead of twice."""

    @staticmethod
    def forward(ctx, x, w, bias, scale, gamma, beta, rmean, rvar, cin, G, eps, momentum, conv_only, up2=False):
        """up2: x is the LOW-resolution tensor and the convolution runs on its nearest x2 upsampling, in sub-pixel form (the caller
        checked upconv_available)."""
        be = _be()
        x = _c(x)
        n, d, h, wd, c = x.shape
        assert c == cin
        cout = w.shape[0]
        ks = tuple(w.shape[2:])
        kd, kh, kw = (1,) * (3 - len(ks)) + ks
        scale_c, bias_c = _c(scale), _c(bias)
        if up2:
            if _rounding_on() and config._dbg_round_act:
                x = _round_(x)
            z = _upconv_fwd(x, w, bias_c, scale_c, None, G, ACT_NONE)
            h, wd = 2 * h, 2 * wd           # BatchNorm geometry = the convolution's output
        else:
            rnd = FLAG_ROUND_TF32 if _tc_fwd(n, d, h, wd, c, cout, kd, kh, kw) else 0
            if rnd and config._dbg_round_act:
                x = _round_(x)
            if _x3_fwd(n, d, h, wd, c, cout, kd, kh, kw):
                rnd = FLAG_SPLIT
            wp = packed_weight(w, 0, cin, rnd)
            z = _new((n, d, h, wd, cout), x)
            _conv_launch(x, wp, bias_c, scale_c, None, z, n, d, h, wd, c, cout, kd, kh, kw, G, ACT_NONE)
        rows = (n // G) * d * h * wd
        if rows <= 1:
            raise ValueError("Expected more than 1 value per channel when training")
        sums = _new((G, cout, 2), x, torch.float64)
        be.bn_stats(z, sums, rows, G, cout)
        mean, invstd, a, b = (_new((G, cout), x) for _ in range(4))
        be.bn_finalize(sums, gamma, beta, rmean, rvar, rows, G, cout, eps, momentum, True, mean, invstd, a, b)
        y = _new(z.shape, x)
        out_rnd = conv_only and _rounding_on()
        be.bn_apply(z, a, b, y, rows, G, cout, 1 | (FLAG_ROUND_TF32 if out_rnd else 0), False, h, wd)
        if out_rnd:
            y._dgmr_tf32 = True
        ctx.save_for_backward(x, w, scale_c, z, gamma, a, b, mean, invstd)
        ctx.meta = (cin, G, (kd, kh, kw), bool(up2))
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, scale, z, gamma, a, b, mean, invstd = ctx.saved_tensors
        cin, G, (kd, kh, kw), up2 = ctx.meta
        be = _be()
        dy = _c(dy)
        n, d, h, wd, c = x.shape
        cout = w.shape[0]
        if up2:
            h, wd = 2 * h, 2 * wd
        rows = (n // G) * d * h * wd
        need_x, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        red = _new((G, cout, 2), x, torch.float64)
        be.bn_bwd_reduce(dy, z, a, b, mean, invstd, red, rows, G, cout, True, False, h, wd)
        tc_bwd = up2 and _rounding_on() or \
            (need_x and _tc_fwd(n, d, h, wd, cout, c, kd, kh, kw)) or (need_w and _tc_wgrad(n, d, h, wd, c, cout, kd, kh, kw))
        dz = _new(z.shape, x) if (need_x or need_w) else None       # = dL/dz * scale[g], tf32-rounded: the dgrad / wgrad operand
        dgamma = _new((cout,), x) if ctx.needs_input_grad[4] else None
        dbeta = _new((cout,), x) if ctx.needs_input_grad[5] else None
        be.bn_bwd_apply(dy, z, a, b, mean, invstd, scale, red, dz, dgamma, dbeta, False, rows, G, cout,
                        1 | (FLAG_ROUND_TF32 if (tc_bwd and config._dbg_round_dz) else 0), False, h, wd, True)
        dx = dw = None
        if up2:
            dx, dw = _upconv_bwd(x, w, dz, need_x, need_w)
            return dx, dw, None, None, dgamma, dbeta, None, None, None, None, None, None, None, None
        if need_x:
            rnd = FLAG_ROUND_TF32 if (_tc_fwd(n, d, h, wd, cout, c, kd, kh, kw) and config._dbg_round_w) else 0
            if _x3_fwd(n, d, h, wd, cout, c, kd, kh, kw):
                rnd = FLAG_SPLIT
            dx = _new(x.shape, x)
            _conv_launch(dz, packed_weight(w, 0, cin, 1 | rnd), None, None, None, dx, n, d, h, wd, cout, c, kd, kh, kw, 1, ACT_NONE)
        if need_w:
            taps = kd * kh * kw
            dwp = _new((taps * cout * c,), x)
            _wgrad_launch(x, dz, dwp, n, d, h, wd, c, cout, kd, kh, kw)
            dw = _new(w.shape, x)
            be.unpack_wgrad(dwp, dw, cout, w.shape[1], 0, cin, taps, False)
        # bias and scale gradients: identically zero (None = zero for autograd; the flat gradient buffers keep their zeros)
        return dx, dw, None, None, dgamma, dbeta, None, None, None, None, None, None, None, None


def conv_bn_relu(x, w, bias, scale, gamma, beta, rmean, rvar, G, eps=1e-5, momentum=0.1, conv_only=False, up2=False):
    """up2: the convolution runs on the nearest x2 upsampling of x -- in sub-pixel form when available, else on the materialised upsample."""
    if up2:
        n, d, h, wd, c = x.shape
        if not (d == 1 and tuple(w.shape[2:]) == (3, 3) and upconv_available(n, h, wd, c, w.shape[0])):
            x, up2 = mark_conv_only(upsample2(x)), False
    return _ConvBNRelu.apply(x, w, bias, scale, gamma, beta, rmean, rvar, w.shape[1], G, eps, momentum, conv_only, up2)


# ----------------------------------------------------------------------------- ConvGRU gate arithmetic
class _GruGate(Function):
    """rh = sigmoid(pre_r) * h   (ref: dgmr/layers/ConvGRU.py:72,78)."""

    @staticmethod
    def forward(ctx, pre_r, h):
        pre_r, h = _c(pre_r), _c(h)
        ch = h.shape[-1]
        rows = h.numel() // ch
        rh = torch.empty_like(h)
        _be().gru_gate_fwd(pre_r, ch, h, rh, rows, ch, 0)
        ctx.save_for_backward(pre_r, h)
        return rh

    @staticmethod
    def backward(ctx, g):
        pre_r, h = ctx.saved_tensors
        g = _c(g)
        ch = h.shape[-1]
        rows = h.numel() // ch
        dpre, dh = torch.empty_like(pre_r), torch.empty_like(h)
        _be().gru_gate_bwd(g, pre_r, ch, h, dpre, ch, dh, False, rows, ch)
        return dpre, dh


class _GruBlend(Function):
    """h' = u*h + (1-u)*c, u = sigmoid(pre_u)   (ref: dgmr/layers/ConvGRU.py:75,82)."""

    @staticmethod
    def forward(ctx, pre_u, h, c, relu_c):
        pre_u, h, c = _c(pre_u), _c(h), _c(c)
        ch = h.shape[-1]
        rows = h.numel() // ch
        hn = torch.empty_like(h)
        _be().gru_blend_fwd(pre_u, ch, h, c, hn, None, rows, ch, relu_c)
        ctx.save_for_backward(pre_u, h, c)
        ctx.relu_c = relu_c
        return hn

    @staticmethod
    def backward(ctx, g):
        pre_u, h, c = ctx.saved_tensors
        g = _c(g)
        ch = h.shape[-1]
        rows = h.numel() // ch
        dpre, dh, dc = torch.empty_like(pre_u), torch.empty_like(h), torch.empty_like(c)
        _be().gru_blend_bwd(g, pre_u, ch, h, c, dpre, ch, dc, dh, False, rows, ch, ctx.relu_c)
        return dpre, dh, dc, None


def gru_gate(pre_r, h):
    return _GruGate.apply(pre_r, h)


def gru_blend(pre_u, h, c, relu_c=False):
    """relu_c: `c` is the candidate PRE-activation and the ReLU of ConvGRU.py:81 is applied inside the blend kernel."""
    return _GruBlend.apply(pre_u, h, c, relu_c)


class _GruSequence(Function):
    """All T steps of one ConvGRU (ref: dgmr/layers/ConvGRU.py:63-84 called T times by :103-110) as ONE autograd node.

    Inputs are the input-dependent parts of the gate pre-activations (already scaled, bias added): xru [T*B,1,H,W,2Ch]
    (read | update side by side) and xc [T*B,1,H,W,Ch]; the h-dependent parts stay on the serial path:
        pre_ru_t = conv(h_{t-1}, W_ru[:, cx:]) * s_ru[t] + xru_t        (one conv for both gates)
        rh_t     = sigmoid(pre_r_t) * h_{t-1}
        c_t      = conv(rh_t, W_c[:, cx:]) * s_c[t] + xc_t
        h_t      = u_t * h_{t-1} + (1 - u_t) * relu(c_t)
    Backward walks the steps in reverse with the data gradients only; the two weight gradients are ONE wgrad launch each
    over all T*B images (the conv operands and the scaled output gradients of every step sit in contiguous buffers)."""

    @staticmethod
    def forward(ctx, xru, xc, h0, w_ru, w_c, s_ru, s_c, T, cx):
        be = _be()
        xru, xc, h0, s_ru, s_c = _c(xru), _c(xc), _c(h0), _c(s_ru), _c(s_c)
        B, d, H, W, ch = h0.shape
        assert d == 1 and xru.shape == (T * B, 1, H, W, 2 * ch) and xc.shape == (T * B, 1, H, W, ch), (xru.shape, xc.shape, h0.shape)
        rows = B * H * W
        rnd_ru = FLAG_ROUND_TF32 if _tc_fwd(B, 1, H, W, ch, 2 * ch, 1, 3, 3) else 0
        rnd_c = FLAG_ROUND_TF32 if _tc_fwd(B, 1, H, W, ch, ch, 1, 3, 3) else 0
        x3 = _x3_fwd(B, 1, H, W, ch, 2 * ch, 1, 3, 3) and _x3_fwd(B, 1, H, W, ch, ch, 1, 3, 3)
        wp_ru = packed_weight(w_ru, cx, ch, FLAG_SPLIT if x3 else rnd_ru)
        wp_c = packed_weight(w_c, cx, ch, FLAG_SPLIT if x3 else rnd_c)
        out = _new((T * B, 1, H, W, ch), h0)
        # tap-split accumulate mode (the small levels): the convolutions add into pre-zeroed buffers (ONE fill per sequence) and the gate kernels add
        # the x parts and write the complete pre-activations back -- instead of one copy of the x part per convolution and step
        defer_ru = config.gru_defer_x and _takes_split_taps(B, 1, H, W, ch, 2 * ch, 1, 3, 3, False, ACT_NONE, x3)
        defer_c = config.gru_defer_x and _takes_split_taps(B, 1, H, W, ch, ch, 1, 3, 3, False, ACT_NONE, x3)
        pru = (_zeros if defer_ru else _new)((T * B, 1, H, W, 2 * ch), h0)
        cp = (_zeros if defer_c else _new)((T * B, 1, H, W, ch), h0)
        rh = _new((T * B, 1, H, W, ch), h0)
        # conv operand of step t = h_{t-1}; when the tensor-core path rounds operands it reads a rounded private copy (the gate
        # arithmetic must see the unrounded state), written by the previous step's blend kernel
        # (T+1 slots: slot t+1 = tf32(h_t), so hop[B:] is also the rounded copy of ALL outputs that the next layer's conv consumes --
        # `out` itself stays unrounded: the gate backward reads it as h_prev)
        hop = _new(((T + 1) * B, 1, H, W, ch), h0) if rnd_ru else None
        if rnd_ru:
            be.round_tf32(h0, hop[0:B])
        pru_flat, xru_flat = pru.view(-1), xru.view(-1)
        for t in range(T):
            sl = slice(t * B, (t + 1) * B)
            h_prev = h0 if t == 0 else out[(t - 1) * B:t * B]
            a = hop[sl] if rnd_ru else h_prev
            off_u = t * rows * 2 * ch + ch
            _conv_launch(a, wp_ru, None, s_ru[t:t + 1], None if defer_ru else xru[sl], pru[sl], B, 1, H, W, ch, 2 * ch, 1, 3, 3, 1, ACT_NONE, y_is_zero=defer_ru)
            be.gru_gate_fwd(pru[sl], 2 * ch, h_prev, rh[sl], rows, ch, rnd_c, x_r=xru[sl] if defer_ru else None)
            _conv_launch(rh[sl], wp_c, None, s_c[t:t + 1], None if defer_c else xc[sl], cp[sl], B, 1, H, W, ch, ch, 1, 3, 3, 1, ACT_NONE, y_is_zero=defer_c)
            nxt = hop[(t + 1) * B:(t + 2) * B] if rnd_ru else None
            be.gru_blend_fwd(pru_flat[off_u:], 2 * ch, h_prev, cp[sl], out[sl], nxt, rows, ch, True,
                             x_u=xru_flat[off_u:] if defer_ru else None, x_c=xc[sl] if defer_c else None)
        ctx.save_for_backward(xru, xc, h0, w_ru, w_c, s_ru, s_c, out, pru, cp, rh, hop)
        ctx.meta = (T, cx, bool(rnd_c))
        if rnd_ru:
            out_r = hop[B:]
            out_r._dgmr_tf32 = True
            return out, out_r
        return out, out.view_as(out)

    @staticmethod
    def backward(ctx, dout, dout_r):
        xru, xc, h0, w_ru, w_c, s_ru, s_c, out, pru, cp, rh, hop = ctx.saved_tensors
        T, cx, rh_rounded = ctx.meta
        be = _be()
        B, _, H, W, ch = h0.shape
        rows = B * H * W
        tc_dg_ru = _tc_fwd(B, 1, H, W, 2 * ch, ch, 1, 3, 3)
        tc_dg_c = _tc_fwd(B, 1, H, W, ch, ch, 1, 3, 3)
        tc_wg_ru = _tc_wgrad(T * B, 1, H, W, ch, 2 * ch, 1, 3, 3)
        tc_wg_c = _tc_wgrad(T * B, 1, H, W, ch, ch, 1, 3, 3)
        x3 = _x3_fwd(B, 1, H, W, 2 * ch, ch, 1, 3, 3) and _x3_fwd(B, 1, H, W, ch, ch, 1, 3, 3)
        wpt_ru = packed_weight(w_ru, cx, ch, 1 | (FLAG_SPLIT if x3 else FLAG_ROUND_TF32 if tc_dg_ru else 0))
        wpt_c = packed_weight(w_c, cx, ch, 1 | (FLAG_SPLIT if x3 else FLAG_ROUND_TF32 if tc_dg_c else 0))
        # running dL/dh_t: starts as the output gradient (of both views of the output), steps add their carry
        if dout is None:
            gh = _c(dout_r).clone()
        else:
            gh = _c(dout).clone()
            if dout_r is not None:
                be.axpby(1.0, gh, 1.0, _c(dout_r), gh)
        dh0 = _new(h0.shape, h0)
        dxru, dzru = torch.empty_like(pru), torch.empty_like(pru)
        dxc, dzc = torch.empty_like(cp), torch.empty_like(cp)
        ds_ru, ds_c = _new((T, 2 * ch), h0), _new((T, ch), h0)
        # d(r h) of each step: in the tap-split accumulate mode one pre-zeroed buffer for all steps (ONE fill), else a single reused slot
        defer_rh = config.gru_defer_x and _takes_split_taps(B, 1, H, W, ch, ch, 1, 3, 3, False, ACT_NONE, x3)
        drh_all = _zeros((T * B, 1, H, W, ch), h0) if defer_rh else _new(h0.shape, h0)
        pru_flat, dxru_flat = pru.view(-1), dxru.view(-1)
        rnd_ru = rnd_c = bool(tc_dg_ru or tc_wg_ru or tc_dg_c or tc_wg_c)     # (both convolutions have Ch input channels: served alike)
        dzru_flat = dzru.view(-1)
        for t in range(T - 1, -1, -1):
            sl = slice(t * B, (t + 1) * B)
            h_prev = h0 if t == 0 else out[(t - 1) * B:t * B]
            tgt = dh0 if t == 0 else gh[(t - 1) * B:t * B]
            off = t * rows * 2 * ch
            # h_t = u h + (1-u) relu(c):  d pre_u -> dxru[:, ch:], d c_pre -> dxc, u * dh_t -> tgt.  The gate kernels also emit the scaled (and
            # rounded) operands dzru / dzc of the recurrent convolutions' backward: no prologue pass per step (the per-step scale gradients are
            # reduced in ONE grouped pass per weight after the loop)
            be.gru_blend_bwd(gh[sl], pru_flat[off + ch:], 2 * ch, h_prev, cp[sl], dxru_flat[off + ch:], 2 * ch, dxc[sl], tgt, t > 0, rows, ch, True,
                             dz_u_scale=s_ru[t, ch:], dz_u=dzru_flat[off + ch:], dz_c_scale=s_c[t], dz_c=dzc[sl], dz_round=rnd_c)
            drh = drh_all[sl] if defer_rh else drh_all
            _conv_launch(dzc[sl], wpt_c, None, None, None, drh, B, 1, H, W, ch, ch, 1, 3, 3, 1, ACT_NONE, y_is_zero=defer_rh)
            # rh = r h:  d pre_r -> dxru[:, :ch], r * drh added to tgt
            be.gru_gate_bwd(drh, pru[sl], 2 * ch, h_prev, dxru[sl], 2 * ch, tgt, True, rows, ch, dz_scale=s_ru[t, :ch], dz=dzru[sl], dz_round=rnd_ru)
            _conv_launch(dzru[sl], wpt_ru, None, None, tgt, tgt, B, 1, H, W, 2 * ch, ch, 1, 3, 3, 1, ACT_NONE)
        # d s[t, co] = <d pre_t[co], pre_t[co] - x_t[co]> / s[t, co]: one grouped reduction (G = T) per weight
        be.conv_bwd_prep(dxc, cp, xc, None, s_c, None, None, None, ds_c, rows, T, ch, ACT_NONE)
        be.conv_bwd_prep(dxru, pru, xru, None, s_ru, None, None, None, ds_ru, rows, T, 2 * ch, ACT_NONE)
        # weight gradients: one launch per weight over all T*B images
        xop = hop[:T * B] if hop is not None else torch.cat([h0, out[:(T - 1) * B]], dim=0)
        dws = []
        for wt, x_all, dz_all, co in ((w_ru, xop, dzru, 2 * ch), (w_c, rh, dzc, ch)):
            dwp = _new((9 * co * ch,), h0)
            _wgrad_launch(x_all, dz_all, dwp, T * B, 1, H, W, ch, co, 1, 3, 3)
            dw = _zeros(wt.shape, h0)
            be.unpack_wgrad(dwp, dw, co, wt.shape[1], cx, ch, 9, False)
            dws.append(dw)
        return dxru, dxc, dh0, dws[0], dws[1], ds_ru, ds_c, None, None


def gru_sequence(xru, xc, h0, w_ru, w_c, s_ru, s_c, T, cx, rounded_out=False):
    """rounded_out: return the tf32-rounded copy of the outputs (what a convolution-only consumer wants) instead of the outputs."""
    out, out_r = _GruSequence.apply(xru, xc, h0, w_ru, w_c, s_ru, s_c, T, cx)
    return out_r if rounded_out else out


# ----------------------------------------------------------------------------- discriminator head
class _SumpoolRelu(Function):
    """[N,1,H,W,C] -> [N,C]: sum over H,W of relu(x)  (ref: dgmr/discriminators.py:129,209)."""

    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        n, d, h, w, c = x.shape
        y = _new((n, c), x)
        _be().sumpool_relu_fwd(x, y, n, d * h * w, c)
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        n, d, h, w, c = x.shape
        dx = torch.empty_like(x)
        _be().sumpool_relu_bwd(_c(g), x, dx, n, d * h * w, c)
        return dx


def sumpool_relu(x):
    return _SumpoolRelu.apply(x)


# ----------------------------------------------------------------------------- attention
class _Attention(Function):
    """ref: dgmr/layers/Attention.py:9-20 (with the reference's [C,H,W]-as-"h w c" axis convention)."""

    @staticmethod
    def forward(ctx, q, k, v):
        q, k, v = _c(q), _c(k), _c(v)
        b, d, h, w, c = q.shape
        L = c * h
        out = torch.empty_like(v)
        beta = _new((b, L, L), q)
        _be().attention_fwd(q, k, v, out, beta, b, h, w, c)
        ctx.save_for_backward(q, k, v, beta)
        return out

    @staticmethod
    def backward(ctx, g):
        q, k, v, beta = ctx.saved_tensors
        b, d, h, w, c = q.shape
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        ws = torch.empty_like(beta)
        _be().attention_bwd(_c(g), q, k, v, beta, dq, dk, dv, ws, b, h, w, c)
        return dq, dk, dv


def attention(q, k, v):
    return _Attention.apply(q, k, v)


# ----------------------------------------------------------------------------- losses
class _HingeDisc(Function):
    """ref: dgmr/losses.py:307-313 applied to the spatial and temporal columns and summed (dgmr/dgmr.py:166-168).
    scores: [2B, 2, 1]: real rows first, then generated."""

    @staticmethod
    def forward(ctx, scores):
        scores = _c(scores)
        b = scores.shape[0] // 2
        cols = scores.numel() // (2 * b)
        loss = _new((), scores)
        ds = torch.empty_like(scores)
        _be().hinge_disc(scores, b, cols, loss, ds)
        ctx.save_for_backward(ds)
        return loss

    @staticmethod
    def backward(ctx, g):
        (ds,) = ctx.saved_tensors
        return ds * g


class _HingeGen(Function):
    """ref: dgmr/losses.py:316-319."""

    @staticmethod
    def forward(ctx, scores):
        scores = _c(scores)
        loss = _new((), scores)
        ds = torch.empty_like(scores)
        _be().hinge_gen(scores, scores.numel(), loss, ds)
        ctx.save_for_backward(ds)
        return loss

    @staticmethod
    def backward(ctx, g):
        (ds,) = ctx.saved_tensors
        return ds * g


class _GridCell(Function):
    """ref: dgmr/losses.py:172-192 + weight_fn dgmr/dgmr.py:20-33 (max(y+1, cap); `/T*H*W` precedence)."""

    @staticmethod
    def forward(ctx, gen, target, cap):
        gen, target = _c(gen), _c(target)
        coef = float(target.size(3) * target.size(4)) / float(target.size(1))
        loss = _new((), gen)
        acc = _new((1,), gen, torch.float64)
        _be().grid_cell_fwd(gen, target, cap, coef, loss, acc)
        ctx.save_for_backward(gen, target)
        ctx.meta = (cap, coef)
        return loss

    @staticmethod
    def backward(ctx, g):
        gen, target = ctx.saved_tensors
        cap, coef = ctx.meta
        dgen = torch.empty_like(gen)
        _be().grid_cell_bwd(gen, target, cap, coef, _c(g), dgen)
        return dgen, None, None


def hinge_disc(scores):
    return _HingeDisc.apply(scores)


def hinge_gen(scores):
    return _HingeGen.apply(scores)


def grid_cell(gen, target, cap):
    return _GridCell.apply(gen, target, cap)


class _MeanK(Function):
    """mean over a list of equally shaped tensors (ref: torch.stack(predictions).mean(0), dgmr/dgmr.py:180)."""

    @staticmethod
    def forward(ctx, *xs):
        k = len(xs)
        out = torch.empty_like(xs[0])
        _be().axpby(1.0 / k, _c(xs[0]), 0.0, None, out)
        for x in xs[1:]:
            _be().axpby(1.0, out, 1.0 / k, _c(x), out)
        ctx.k = k
        return out

    @staticmethod
    def backward(ctx, g):
        g = _c(g)
        gi = torch.empty_like(g)
        _be().axpby(1.0 / ctx.k, g, 0.0, None, gi)
        return tuple(gi for _ in range(ctx.k))


class _Add(Function):
    @staticmethod
    def forward(ctx, a, b):
        a, b = _c(a), _c(b)
        out = torch.empty_like(a)
        _be().axpby(1.0, a, 1.0, b, out)
        return out

    @staticmethod
    def backward(ctx, g):
        return g, g


def add(a, b):
    return _Add.apply(a, b)


def mean_k(xs):
    return xs[0] if len(xs) == 1 else _MeanK.apply(*xs)
