"""Generator building blocks and the two conditioning stacks on the B200 path.

Public constructors / forward signatures / state-dict keys follow the reference's dgmr/common.py
(GBlock :17, UpsampleGBlock :87, DBlock :158, LBlock :241, ContextConditioningStack :303,
LatentConditioningStack :427).  Every `forward` takes and returns NCHW tensors like the reference;
internally each block has a channels-last `run(x, G)` used when blocks are chained, where G is the
number of reference calls folded into the batch dimension (per-call BatchNorm statistics and
spectral-norm sigmas become per-group quantities).
"""
from __future__ import annotations

from typing import Tuple

import torch
import torch.nn as nn
from .hub import HubMixin as PyTorchModelHubMixin   # same API; saves compact copies (see hub.py)

from . import ops
from .layers.Attention import AttentionLayer
from .layers.core import BatchNorm, PlainConv, SNConv, prefetch_sigmas
from .ops import ACT_NONE, ACT_RELU


def _kernel(conv_type: str, k: int):
    if conv_type == "standard":
        return (k, k)
    if conv_type == "3d":
        return (k, k, k)
    if conv_type == "coord":
        raise NotImplementedError("conv_type='coord' (CoordConv) is outside the B200 hot path (SURVEY.md 2, row 8)")
    raise ValueError(f"{conv_type} is not a recognized Conv method")


def _conv_bn_relu_eval(conv: SNConv, bn: BatchNorm, x, G: int, up2: bool = False):
    """Eval mode: relu(bn(conv(x))) as ONE convolution launch.  With running statistics BatchNorm is a per-channel affine map
    y = a*z + b (a = gamma / sqrt(running_var + eps), b = beta - a * running_mean), so it folds into the conv epilogue's per-group scale
    and bias -- scale'[g, co] = a[co] / sigma_g, bias'[co] = a[co] * bias[co] + b[co] -- followed by the fused ReLU: no BatchNorm pass over
    the activation at all (SURVEY.md 8f-2).  The [G, C]-sized folding arithmetic is plain differentiable tensor algebra on parameters."""
    a = bn.weight * torch.rsqrt(bn.running_var + bn.eps)
    b = bn.bias - a * bn.running_mean
    scale = conv.inv_sigma(G).view(G, 1) * a.view(1, -1)
    if up2:   # the convolution runs on the nearest x2 upsampling of x (sub-pixel form where available)
        return ops.upconv(x, conv.weight_orig, conv.bias * a + b, scale.contiguous(), G, ACT_RELU, round_out=True)
    return ops.conv(x, conv.weight_orig, conv.bias * a + b, scale.contiguous(), None, 0, conv.in_channels, G, ACT_RELU)


def _conv_bn_relu_train(conv: SNConv, bn: BatchNorm, x, G: int, up2: bool = False):
    """Train mode: relu(bn(conv(x))) as one autograd node (ops._ConvBNRelu): the BatchNorm backward hands the convolution its scaled,
    rounded output gradient directly."""
    bn.num_batches_tracked += G
    scale = conv.scale_of(conv.inv_sigma(G))
    return ops.conv_bn_relu(x, conv.weight_orig, conv.bias, scale, bn.weight, bn.bias, bn.running_mean, bn.running_var, G,
                            bn.eps, bn.momentum, conv_only=True, up2=up2)


class GBlock(nn.Module):
    """Residual generator block without upsampling (ref: dgmr/common.py:17-84)."""

    def __init__(self, input_channels: int = 12, output_channels: int = 12, conv_type: str = "standard",
                 spectral_normalized_eps=0.0001):
        super().__init__()
        self.input_channels, self.output_channels = input_channels, output_channels
        self.bn1 = BatchNorm(input_channels)
        self.bn2 = BatchNorm(input_channels)
        e = spectral_normalized_eps
        self.conv_1x1 = SNConv(input_channels, output_channels, _kernel(conv_type, 1), eps=e)
        self.first_conv_3x3 = SNConv(input_channels, input_channels, _kernel(conv_type, 3), eps=e)
        self.last_conv_3x3 = SNConv(input_channels, output_channels, _kernel(conv_type, 3), eps=e)

    def sn_calls(self, G: int = 1):
        """The spectrally normalised layers `run` will evaluate (conv_1x1 only when it projects, like the reference :71-74)."""
        proj = [(self.conv_1x1, G)] if self.input_channels != self.output_channels else []
        return proj + [(self.first_conv_3x3, G), (self.last_conv_3x3, G)]

    def run(self, x, G: int = 1):
        y, xs = self.bn1.run(x, G, relu=True, conv_only=True, branch=True)   # xs: x again, for the shortcut (gradients meet in the BN backward)
        y = ops.mark_conv_only(y)
        sc = xs if x.shape[-1] == self.output_channels else self.conv_1x1.run(xs, G)
        if self.training:
            y = ops.mark_conv_only(_conv_bn_relu_train(self.first_conv_3x3, self.bn2, y, G))
        else:
            y = ops.mark_conv_only(_conv_bn_relu_eval(self.first_conv_3x3, self.bn2, y, G))
        return self.last_conv_3x3.run(y, G, res=sc)  # residual add fused in the conv epilogue

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return ops.cl_to_nchw(self.run(ops.nchw_to_cl(x)))


class UpsampleGBlock(nn.Module):
    """Residual generator block with nearest x2 upsampling (ref: dgmr/common.py:87-155)."""

    def __init__(self, input_channels: int = 12, output_channels: int = 12, conv_type: str = "standard",
                 spectral_normalized_eps=0.0001):
        super().__init__()
        self.input_channels, self.output_channels = input_channels, output_channels
        self.bn1 = BatchNorm(input_channels)
        self.bn2 = BatchNorm(input_channels)
        e = spectral_normalized_eps
        self.conv_1x1 = SNConv(input_channels, output_channels, _kernel(conv_type, 1), eps=e)
        self.first_conv_3x3 = SNConv(input_channels, input_channels, _kernel(conv_type, 3), eps=e)
        self.last_conv_3x3 = SNConv(input_channels, output_channels, _kernel(conv_type, 3), eps=e)

    def sn_calls(self, G: int = 1):
        return [(self.conv_1x1, G), (self.first_conv_3x3, G), (self.last_conv_3x3, G)]

    def run(self, x, G: int = 1, round_out: bool = False):
        """round_out: the block output is read by tensor-core convolutions only (the next sampler level's gate convolutions) and is written tf32-rounded
        by last_conv_3x3's epilogue -- no rounding pass into a private copy.  (Its own backward then reduces <dY, Y - b - res> over the rounded Y: 2^-12
        relative noise on a sum of millions of terms, far below the 1xTF32 operand rounding of every product in that sum.)"""
        # conv1x1(up2(x)) == up2(conv1x1(x)) bit-for-bit (pointwise conv commutes with replication): 4x fewer MACs, and the
        # upsampled shortcut is never materialised: last_conv_3x3's epilogue reads it at (h/2, w/2)
        # BN -> ReLU at LOW resolution; the nearest x2 upsampling (ref :148) is folded into first_conv_3x3's sub-pixel form (ops.upconv:
        # 2.25x fewer MACs, the upsampled activation is never written); xs: x again, for the shortcut
        y, xs = self.bn1.run(x, G, relu=True, conv_only=True, branch=True)
        y = ops.mark_conv_only(y)
        sc = self.conv_1x1.run(xs, G)  # x also feeds BatchNorm: the conv rounds a private copy
        if self.training:
            y = ops.mark_conv_only(_conv_bn_relu_train(self.first_conv_3x3, self.bn2, y, G, up2=True))
        else:
            y = ops.mark_conv_only(_conv_bn_relu_eval(self.first_conv_3x3, self.bn2, y, G, up2=True))
        return self.last_conv_3x3.run(y, G, res=sc, res_up2=True, round_out=round_out)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return ops.cl_to_nchw(self.run(ops.nchw_to_cl(x)))


class DBlock(nn.Module):
    """Residual down block, 2-D or 3-D (ref: dgmr/common.py:158-238)."""

    def __init__(self, input_channels: int = 12, output_channels: int = 12, conv_type: str = "standard",
                 first_relu: bool = True, keep_same_output: bool = False):
        super().__init__()
        self.input_channels, self.output_channels = input_channels, output_channels
        self.first_relu, self.keep_same_output, self.conv_type = first_relu, keep_same_output, conv_type
        self.conv_1x1 = SNConv(input_channels, output_channels, _kernel(conv_type, 1))
        self.first_conv_3x3 = SNConv(input_channels, output_channels, _kernel(conv_type, 3))
        self.last_conv_3x3 = SNConv(output_channels, output_channels, _kernel(conv_type, 3))

    def _pool(self, x):
        return ops.avg_pool(x, 2, 2, 2) if self.conv_type == "3d" else ops.avg_pool(x, 1, 2, 2)

    def sn_calls(self, G: int = 1):
        proj = [(self.conv_1x1, G)] if self.input_channels != self.output_channels else []
        return proj + [(self.first_conv_3x3, G), (self.last_conv_3x3, G)]

    def _first_conv_depth_folded(self, x, G):
        """3x3x3 convolution over a few-channel input (first temporal-discriminator block, 4 channels carried as 8) with its three
        depth taps folded into the channel axis: x' = [x(d-1) | x(d) | x(d+1)] (12 real channels in 16), weight [Cout, kd*Cin + ci, kh, kw],
        a 1x3x3 convolution with K = 9*16 instead of 27*8 half-empty -- same products, same sums; 1.5x fewer forward MMAs and 3x
        fewer weight-gradient MMAs (its weight gradient ran at 24 TF/s)."""
        conv, cin = self.first_conv_3x3, self.input_channels
        w = conv.weight_orig                                               # [Cout, Cin, 3, 3, 3]
        wf = w.permute(0, 2, 1, 3, 4).reshape(w.shape[0], 3 * cin, 3, 3)   # [Cout, kd*Cin + ci, kh, kw] (differentiable view algebra)
        xf = ops.mark_conv_only(ops.fold_depth3(x, cin))
        scale = conv.scale_of(conv.inv_sigma(G))
        return ops.conv(xf, wf, conv.bias, scale, None, 0, 3 * cin, G, ACT_RELU, round_out=True)

    def run(self, x, G: int = 1):
        if self.input_channels != self.output_channels:
            if self.keep_same_output:
                x1 = self.conv_1x1.run(x, G)
            else:
                # avgpool(conv1x1(x)) == conv1x1(avgpool(x)) (both linear, the bias passes through the mean; SURVEY.md section 7, diff 6e-7):
                # 4x (2-D) / 8x (3-D) fewer MACs and no full-resolution shortcut tensor.  The pool is launched before anything rounds x
                # in place, so it averages the unrounded values.
                x1 = self.conv_1x1.run(ops.mark_conv_only(self._pool(x)), G)
            # x is otherwise read by convolutions and by ReLU only (ReLU commutes with tf32 rounding): rounding in place is exact
            ops.mark_conv_only(x)
        else:
            x1 = x
        y = ops.mark_conv_only(ops.relu(x)) if self.first_relu else x
        # the ReLU between the convs is fused, and the result (read by last_conv_3x3 only) leaves the epilogue tf32-rounded
        if self.conv_type == "3d" and self.input_channels <= 8 and x.shape[-1] == ops.pad8(self.input_channels) and x.shape[1] >= 3:
            y = ops.mark_conv_only(self._first_conv_depth_folded(y, G))
        else:
            y = ops.mark_conv_only(self.first_conv_3x3.run(y, G, act=ACT_RELU, round_out=True))
        if self.keep_same_output:
            return self.last_conv_3x3.run(y, G, res=x1)
        # conv -> AvgPool as one node: the backward prologue reads the pooled gradient directly (no upsample pass)
        y = self.last_conv_3x3.run(y, G, pool=((2, 2, 2) if self.conv_type == "3d" else (1, 2, 2)))
        return ops.add(x1, y)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return ops.cl_to_nchw(self.run(ops.nchw_to_cl(x)))


class LBlock(nn.Module):
    """Residual block of the latent stack, plain convolutions (ref: dgmr/common.py:241-300)."""

    def __init__(self, input_channels: int = 12, output_channels: int = 12, kernel_size: int = 3, conv_type: str = "standard"):
        super().__init__()
        self.input_channels, self.output_channels = input_channels, output_channels
        self.conv_1x1 = PlainConv(input_channels, output_channels - input_channels, _kernel(conv_type, 1))
        self.first_conv_3x3 = PlainConv(input_channels, output_channels, _kernel(conv_type, kernel_size))
        self.last_conv_3x3 = PlainConv(output_channels, output_channels, _kernel(conv_type, kernel_size))

    def run(self, x):
        if self.input_channels < self.output_channels:
            sc = ops.concat_channels(x, self.conv_1x1.run(x))
        else:
            sc = x
        y = ops.mark_conv_only(self.first_conv_3x3.run(ops.mark_conv_only(ops.relu(x)), act=ACT_RELU, round_out=True))
        return self.last_conv_3x3.run(y, res=sc)

    def forward(self, x) -> torch.Tensor:
        return ops.cl_to_nchw(self.run(ops.nchw_to_cl(x)))


class ContextConditioningStack(nn.Module, PyTorchModelHubMixin):
    """ref: dgmr/common.py:303-424.  The 4 context frames run as 4 groups of one launch."""

    def __init__(self, input_channels: int = 1, output_channels: int = 768, num_context_steps: int = 4,
                 conv_type: str = "standard"):
        super().__init__()
        self.input_channels, self.num_context_steps = input_channels, num_context_steps
        oc, ic, t = output_channels, input_channels, num_context_steps
        self.d1 = DBlock(4 * ic, ((oc // 4) * ic) // t, conv_type=conv_type)
        self.d2 = DBlock(((oc // 4) * ic) // t, ((oc // 2) * ic) // t, conv_type=conv_type)
        self.d3 = DBlock(((oc // 2) * ic) // t, (oc * ic) // t, conv_type=conv_type)
        self.d4 = DBlock((oc * ic) // t, (oc * 2 * ic) // t, conv_type=conv_type)
        k3 = _kernel(conv_type, 3)
        self.conv1 = SNConv((oc // 4) * ic, (oc // 8) * ic, k3)
        self.conv2 = SNConv((oc // 2) * ic, (oc // 4) * ic, k3)
        self.conv3 = SNConv(oc * ic, (oc // 2) * ic, k3)
        self.conv4 = SNConv(oc * 2 * ic, oc * ic, k3)

    def run(self, x: torch.Tensor):
        """x: [B,T,C,H,W] (reference layout) -> 4 channels-last states [B,1,h,w,c], largest first."""
        x = x.contiguous()
        b, t, c, h, w = x.shape
        h2, w2 = h // 2, w // 2
        # every spectral norm of the stack in one launch: the DBlocks are called once per context frame, the mixers once
        prefetch_sigmas([c_ for blk in (self.d1, self.d2, self.d3, self.d4) for c_ in blk.sn_calls(t)]
                        + [(m, 1) for m in (self.conv1, self.conv2, self.conv3, self.conv4)])
        # space-to-depth (PixelUnshuffle(2), :393) and regrouping to timestep-major in ONE permute:
        # dst[t, b, h2, w2, c*4 + i*2 + j] = x[b, t, c, 2*h2+i, 2*w2+j]
        cpad = ops.pad8(4 * c)  # 4 -> 8 zero-padded channels: lets the tcgen05 path (K step 8) take the first DBlock
        ds = ops.contig_strides((t, b, h2, w2, cpad))
        s = ops.permute(x, (t * b, 1, h2, w2, cpad), (b, t, c, h2, w2, 2, 2),
                        (t * c * h * w, c * h * w, h * w, 2 * w, 2, w, 1),
                        (ds[1], ds[0], 4, ds[2], ds[3], 2, 1))
        outs = []
        for blk, mix in ((self.d1, self.conv1), (self.d2, self.conv2), (self.d3, self.conv3), (self.d4, self.conv4)):
            s = blk.run(s, G=t)
            _, _, hh, ww, cc = s.shape
            # "b t c h w -> b (c t) h w" (:423): mixed[b, h, w, c*T + t] = s[t, b, h, w, c]
            mixed = ops.permute(s, (b, 1, hh, ww, cc * t), (t, b, hh * ww, cc),
                                (b * hh * ww * cc, hh * ww * cc, cc, 1), (1, hh * ww * cc * t, cc * t, t))
            outs.append(mix.run(ops.mark_conv_only(mixed), 1, act=ACT_RELU))   # (feeds the ConvGRU as h0: gate arithmetic reads it unrounded)
        return tuple(outs)

    def forward(self, x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
        return tuple(ops.cl_to_nchw(s) for s in self.run(x))


class LatentConditioningStack(nn.Module, PyTorchModelHubMixin):
    """ref: dgmr/common.py:427-497.  Batch is always 1; z is drawn on the CPU default generator exactly
    like the reference's `Normal(0,1).sample(shape)` so seeds reproduce."""

    def __init__(self, shape: (int, int, int) = (8, 8, 8), output_channels: int = 768, use_attention: bool = True):
        super().__init__()
        self.shape = tuple(shape)
        self.use_attention = use_attention
        self.conv_3x3 = SNConv(shape[0], shape[0], (3, 3))
        self.l_block1 = LBlock(shape[0], output_channels // 32)
        self.l_block2 = LBlock(output_channels // 32, output_channels // 16)
        self.l_block3 = LBlock(output_channels // 16, output_channels // 4)
        if self.use_attention:
            self.att_block = AttentionLayer(output_channels // 4, output_channels // 4)
        self.l_block4 = LBlock(output_channels // 4, output_channels)

    def sample_z(self, like: torch.Tensor, k: int = 1) -> torch.Tensor:
        """k successive draws (k reference calls' worth, in call order) as channels-last [k,1,H,W,C] on like's device."""
        s = tuple(self.shape) + (1,)
        zs = [torch.normal(torch.zeros(s), torch.ones(s)) for _ in range(k)]  # == distribution.sample(self.shape), CPU RNG (:481)
        # [C,H,W,1] -> channels-last [1,1,H,W,C]
        z = torch.stack(zs).squeeze(-1).permute(0, 2, 3, 1).contiguous().unsqueeze(1)
        return z.to(device=like.device, dtype=like.dtype)

    def run(self, x: torch.Tensor, members: int = 1):
        """-> channels-last [members,1,h,w,c]: one latent per ensemble member (batch 1 in the reference)."""
        z = self.sample_z(x, members)
        z = self.conv_3x3.run(z, 1)
        z = self.l_block1.run(z)
        z = self.l_block2.run(z)
        z = self.l_block3.run(z)
        if self.use_attention:
            z = self.att_block.run(z)
        return self.l_block4.run(z)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return ops.cl_to_nchw(self.run(x))
