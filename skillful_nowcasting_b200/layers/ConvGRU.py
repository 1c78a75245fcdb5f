"""ConvGRU on the B200 path (API of the reference's dgmr/layers/ConvGRU.py:8-111).

Restructuring that keeps the reference's results (SURVEY.md section 7, identities verified there):
conv(cat[x, h]) = conv_x(x) + conv_h(h), so the input-dependent two thirds of every gate
convolution are computed for ALL T timesteps in one launch (one group per timestep, each with its own
spectral-norm sigma_t), and only the h-dependent third stays on the serial path.  The T power
iterations a weight sees during one forward run inside a single spectral-norm launch.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Union

import torch
import torch.nn as nn

from .. import ops
from ..ops import ACT_NONE, ACT_RELU
from .core import SNConv


class ConvGRUCell(nn.Module):
    """ref: dgmr/layers/ConvGRU.py:8-85 (three spectrally normalised 3x3 convs, eps 1e-4)."""

    def __init__(self, input_channels: int, output_channels: int, kernel_size: int = 3, sn_eps: float = 0.0001):
        super().__init__()
        self._kernel_size = kernel_size
        self._sn_eps = sn_eps
        self.input_channels, self.output_channels = input_channels, output_channels
        k = (kernel_size, kernel_size)
        self.read_gate_conv = SNConv(input_channels, output_channels, k, eps=sn_eps)
        self.update_gate_conv = SNConv(input_channels, output_channels, k, eps=sn_eps)
        self.output_conv = SNConv(input_channels, output_channels, k, eps=sn_eps)

    # ---- channels-last multi-step engine -------------------------------------------------
    def run_sequence(self, xs: torch.Tensor, h0: torch.Tensor, T: int, shared_input: bool = False,
                     rounded_out: bool = False) -> torch.Tensor:
        """xs: [T*B,1,H,W,Cx] timestep-major (or [M,1,H,W,Cx] with shared_input=True: the same input at every step, one per
        member m for the B/M consecutive batch elements of that member, as at the sampler's first level, ref: generators.py:146-149,
        where M = 1); h0: [B,1,H,W,Ch].  Returns [T*B,1,H,W,Ch].  rounded_out: the caller feeds the result to convolutions only and
        accepts the tf32-rounded copy the recurrence writes anyway (fused path on the tensor cores)."""
        ch = self.output_channels
        cx = self.input_channels - ch
        B = h0.shape[0]
        gates = (self.read_gate_conv, self.update_gate_conv, self.output_conv)
        # one launch per weight: the T power iterations of this forward (ref: per-call parametrization)
        scales = [g.scale_of(g.inv_sigma(T)) for g in gates]  # [T, Ch] each
        if ops.config.gru_sequence:
            return self._run_fused(xs, h0, T, shared_input, scales, rounded_out)
        xparts = []
        for g, sc in zip(gates, scales):
            xparts.append(self._x_part(xs, g.weight_orig, g.bias, sc, T, B, cx, shared_input).unbind(0))
        srows = [sc.reshape(T, 1, ch).unbind(0) for sc in scales]
        h = h0
        outs = []
        wr, wu, wc = (g.weight_orig for g in gates)
        for t in range(T):
            hop = ops.conv_operand(h)  # h also feeds the gate arithmetic: both gate convs share one tf32-rounded copy
            pre_r = ops.conv(hop, wr, None, srows[0][t], xparts[0][t], cx, ch, 1, ACT_NONE)
            pre_u = ops.conv(hop, wu, None, srows[1][t], xparts[1][t], cx, ch, 1, ACT_NONE)
            rh = ops.mark_conv_only(ops.gru_gate(pre_r, h))
            c = ops.conv(rh, wc, None, srows[2][t], xparts[2][t], cx, ch, 1, ACT_NONE)  # candidate pre-activation
            h = ops.gru_blend(pre_u, h, c, relu_c=True)                                  # ReLU fused into the blend
            outs.append(h)
        return torch.cat(outs, dim=0)

    @staticmethod
    def _x_part(xs, w, bias, sc, T, B, cx, shared_input):
        """Input-dependent part of a gate pre-activation for all T steps: [T, B, 1, H, W, Cout] (bias and sigma_t applied).
        shared_input: xs [M,1,H,W,Cx] holds one input per member; the convolution runs on the T*M distinct images and its result is
        broadcast over each member's B/M batch elements."""
        if shared_input:
            m = xs.shape[0]
            p = xs.numel()
            x_rep = ops.mark_conv_only(ops.repeat_mid(xs.reshape(1, p), T).reshape((T * m,) + tuple(xs.shape[1:])))
            xp = ops.conv(x_rep, w, bias, sc, None, 0, cx, T, ACT_NONE)  # [T*M,1,H,W,Cout]
            q = xp.numel() // (T * m)
            return ops.repeat_mid(xp.reshape(T * m, q), B // m).reshape((T, B) + tuple(xp.shape[1:]))
        xp = ops.conv(xs, w, bias, sc, None, 0, cx, T, ACT_NONE)
        return xp.reshape((T, B) + tuple(xp.shape[1:]))

    def _run_fused(self, xs, h0, T, shared_input, scales, rounded_out=False):
        """Read and update gates as ONE convolution (their weights, biases and per-step sigmas side by side along Cout), and the
        whole recurrence as one autograd node (ops.gru_sequence): 2 serial convs per step instead of 3, weight gradients of all
        steps in one launch."""
        ch = self.output_channels
        cx = self.input_channels - ch
        B = h0.shape[0]
        gr, gu, gc = self.read_gate_conv, self.update_gate_conv, self.output_conv
        w_ru = torch.cat([gr.weight_orig, gu.weight_orig], dim=0)
        b_ru = torch.cat([gr.bias, gu.bias], dim=0)
        s_ru = torch.cat([scales[0], scales[1]], dim=1)                     # [T, 2Ch]
        xru = self._x_part(xs, w_ru, b_ru, s_ru, T, B, cx, shared_input)
        xc = self._x_part(xs, gc.weight_orig, gc.bias, scales[2], T, B, cx, shared_input)
        xru = xru.reshape((T * B,) + tuple(xru.shape[2:]))
        xc = xc.reshape((T * B,) + tuple(xc.shape[2:]))
        return ops.gru_sequence(xru, xc, h0, w_ru, gc.weight_orig, s_ru, scales[2], T, cx, rounded_out)

    def forward(self, x: torch.Tensor, prev_state: torch.Tensor):
        """NCHW in/out: (x [B,Cx,H,W], prev_state [B,Ch,H,W]) -> (out, new_state)."""
        out = self.run_sequence(ops.nchw_to_cl(x), ops.nchw_to_cl(prev_state), 1)
        out = ops.cl_to_nchw(out)
        return out, out


class ConvGRU(nn.Module):
    """ref: dgmr/layers/ConvGRU.py:88-111."""

    def __init__(self, input_channels: int, output_channels: int, kernel_size: int = 3, sn_eps=0.0001):
        super().__init__()
        self.cell = ConvGRUCell(input_channels, output_channels, kernel_size, sn_eps)

    def forward(self, x: Union[torch.Tensor, Sequence[torch.Tensor]], hidden_state=None) -> torch.Tensor:
        """x: list of T tensors [B,Cx,H,W] (or a tensor [T,B,Cx,H,W]); returns [T,B,Ch,H,W]."""
        T = len(x)
        xs = torch.cat([ops.nchw_to_cl(x[t]) for t in range(T)], dim=0)
        out = self.cell.run_sequence(xs, ops.nchw_to_cl(hidden_state), T)
        B = hidden_state.shape[0]
        out = ops.cl_to_nchw(out)
        return out.reshape((T, B) + tuple(out.shape[1:]))
