"""Sampler and Generator on the B200 path (API of the reference's dgmr/generators.py:20-212).

The reference runs every block once per forecast step through Python list comprehensions
(generators.py:152-178).  Here the T steps of each non-recurrent block are ONE launch over a
timestep-major batch [T*B, ...] with T groups: BatchNorm batch statistics, running-stat updates and
spectral-norm power iterations stay per timestep (SURVEY.md Appendix B 3-4), so results are those of
the reference's per-step calls.  Only the ConvGRU recurrence is sequential.
"""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.nn as nn
from .hub import HubMixin as PyTorchModelHubMixin   # same API; saves compact copies (see hub.py)

from . import ops
from .common import GBlock, UpsampleGBlock
from .layers.ConvGRU import ConvGRU
from .layers.core import BatchNorm, SNConv, prefetch_sigmas


class Sampler(nn.Module, PyTorchModelHubMixin):
    """ref: dgmr/generators.py:20-182."""

    def __init__(self, forecast_steps: int = 18, latent_channels: int = 768, context_channels: int = 384,
                 output_channels: int = 1):
        super().__init__()
        self.forecast_steps = forecast_steps
        lc, cc = latent_channels, context_channels
        self.convGRU1 = ConvGRU(lc + cc, cc, 3)
        self.gru_conv_1x1 = SNConv(cc, lc, (1, 1))
        self.g1 = GBlock(lc, lc)
        self.up_g1 = UpsampleGBlock(lc, lc // 2)
        self.convGRU2 = ConvGRU(lc // 2 + cc // 2, cc // 2, 3)
        self.gru_conv_1x1_2 = SNConv(cc // 2, lc // 2, (1, 1))
        self.g2 = GBlock(lc // 2, lc // 2)
        self.up_g2 = UpsampleGBlock(lc // 2, lc // 4)
        self.convGRU3 = ConvGRU(lc // 4 + cc // 4, cc // 4, 3)
        self.gru_conv_1x1_3 = SNConv(cc // 4, lc // 4, (1, 1))
        self.g3 = GBlock(lc // 4, lc // 4)
        self.up_g3 = UpsampleGBlock(lc // 4, lc // 8)
        self.convGRU4 = ConvGRU(lc // 8 + cc // 8, cc // 8, 3)
        self.gru_conv_1x1_4 = SNConv(cc // 8, lc // 8, (1, 1))
        self.g4 = GBlock(lc // 8, lc // 8)
        self.up_g4 = UpsampleGBlock(lc // 8, lc // 16)
        self.bn = BatchNorm(lc // 16)
        self.conv_1x1 = SNConv(lc // 16, 4 * output_channels, (1, 1))
        self.output_channels = output_channels

    def max_image_elements(self, h: int, w: int) -> int:
        """Elements of the largest per-image activation of one forecast step for an h x w latent grid: the widest tensor of every level
        (gate pre-activations, blocks, and the up-block's first convolution at twice the resolution), for sizing batched launches."""
        n = 0
        for lvl, (gru, g, ug) in enumerate(((self.convGRU1, self.g1, self.up_g1), (self.convGRU2, self.g2, self.up_g2),
                                            (self.convGRU3, self.g3, self.up_g3), (self.convGRU4, self.g4, self.up_g4))):
            hw = (h << lvl) * (w << lvl)
            cell = gru.cell
            n = max(n, hw * max(cell.input_channels, 2 * cell.output_channels), hw * g.output_channels,
                    4 * hw * max(ug.input_channels, ug.output_channels))
        return n

    def members_per_pass(self, batch: int, h: int, w: int) -> int:
        """Largest member count M whose sampler pass (T*M*batch images per launch) keeps every tensor below 2^31 elements: the tensor-core
        convolutions address with 32-bit offsets (N*H*W*Cout < 2^32, N*H*W < 2^31) and refuse larger launches."""
        per_member = self.forecast_steps * batch * self.max_image_elements(h, w)
        return max(1, ((1 << 31) - 1) // per_member)

    def run(self, init_states: List[torch.Tensor], latent: torch.Tensor, out: Optional[torch.Tensor] = None, member0: int = 0) -> torch.Tensor:
        """init_states: channels-last [B,1,h,w,c], largest first; latent: channels-last [M,1,h,w,c], one per ensemble member.
        Returns forecasts [B,T,C_out,H,W] (reference layout) for M = 1, else [B,M,T,C_out,H,W].
        The M members run as one batch of M*B images per step, ordered [T, M, B]; their conditioning states are the same.
        out: write the members into out[:, member0:member0 + M] of an existing [B,K,T,C_out,H,W] tensor instead (no autograd)."""
        T = self.forecast_steps
        B = init_states[0].shape[0]
        M = latent.shape[0]
        if M > 1:
            if self.training:
                raise RuntimeError("Sampler.run: several members per pass are eval-mode only (train-mode statistics are per reference call)")
            init_states = [ops.repeat_mid(s.reshape(1, s.numel()), M).reshape((M * B,) + tuple(s.shape[1:])) for s in init_states]
        levels = ((self.convGRU1, self.gru_conv_1x1, self.g1, self.up_g1),
                  (self.convGRU2, self.gru_conv_1x1_2, self.g2, self.up_g2),
                  (self.convGRU3, self.gru_conv_1x1_3, self.g3, self.up_g3),
                  (self.convGRU4, self.gru_conv_1x1_4, self.g4, self.up_g4))
        # all 37 spectral norms of the sampler (T power iterations each) in one launch
        calls = [(self.conv_1x1, T)]
        for gru, c11, g, ug in levels:
            cell = gru.cell
            calls += [(cell.read_gate_conv, T), (cell.update_gate_conv, T), (cell.output_conv, T), (c11, T)] + g.sn_calls(T) + ug.sn_calls(T)
        prefetch_sigmas(calls)
        hs = latent
        for lvl, (gru, c11, g, ug) in enumerate(levels):
            # level 0: identical latent input at every step and for every sample of a member (generators.py:146-149)
            # The level input is read by convolutions only: above level 0 it is the previous up-block's output, written tf32-rounded by that
            # block's last epilogue (conv_operand passes it through; unrounded tensors get one private rounded copy that both gate convs share).
            # The recurrence hands back the tf32-rounded copy of its outputs, which the 1x1 conv consumes as is.
            xin = ops.mark_conv_only(hs) if lvl == 0 else ops.conv_operand(hs)
            hs = gru.cell.run_sequence(xin, init_states[3 - lvl], T, shared_input=(lvl == 0), rounded_out=True)
            hs = c11.run(hs if getattr(hs, "_dgmr_tf32", False) else ops.mark_conv_only(hs), T)
            hs = g.run(hs, T)
            hs = ug.run(hs, T, round_out=(lvl < 3))      # levels 0-2: read by the next level's gate convolutions only
        hs = ops.mark_conv_only(self.bn.run(hs, T, relu=True, conv_only=True))
        hs = self.conv_1x1.run(hs, T)  # [T*M*B,1,h,w,4*Co]
        _, _, h, w, c4 = hs.shape
        co = c4 // 4
        F = co * 4 * h * w                                  # one output frame
        K = M if out is None else out.shape[1]
        # PixelShuffle(2) + stack on dim 1 (:178,181) in one permute:
        # out[b, member0 + m, t, co, 2h+i, 2w+j] = hs[(t*M + m)*B + b, h, w, co*4 + i*2 + j]
        shape = [T, M, B, h, w, co, 2, 2]
        sstr = [M * B * h * w * c4, B * h * w * c4, h * w * c4, w * c4, c4, 4, 2, 1]
        dstr = [F, T * F, K * T * F, 4 * w, 2, 4 * h * w, 2 * w, 1]
        if M == 1:                                          # no member axis: the reference's [B,T,...] permute
            del shape[1], sstr[1], dstr[1]
        if out is not None:
            ops.permute_into(hs, out, shape, sstr, dstr, member0 * T * F)
            return out
        return ops.permute(hs, (B, T, co, 2 * h, 2 * w) if M == 1 else (B, M, T, co, 2 * h, 2 * w), shape, sstr, dstr)

    def forward(self, conditioning_states: List[torch.Tensor], latent_dim: torch.Tensor) -> torch.Tensor:
        """NCHW conditioning states (largest first) + latent [1,C,h,w] -> [B,T,C_out,H,W]."""
        return self.run([ops.nchw_to_cl(s) for s in conditioning_states], ops.nchw_to_cl(latent_dim))


class Generator(nn.Module, PyTorchModelHubMixin):
    """ref: dgmr/generators.py:185-212."""

    def __init__(self, conditioning_stack: nn.Module, latent_stack: nn.Module, sampler: nn.Module):
        super().__init__()
        self.conditioning_stack = conditioning_stack
        self.latent_stack = latent_stack
        self.sampler = sampler

    def sample(self, x: torch.Tensor, num_samples: int, members_per_pass: Optional[int] = None) -> torch.Tensor:
        """An ensemble of `num_samples` eval-mode forecasts of the same context frames: x [B,T_in,C,H,W] -> [B,K,T,C_out,H,W].

        Equals torch.stack([self(x) for _ in range(K)], dim=1) from the same CPU seed, drawing the K latents in the same order (the CPU RNG
        ends in the same state), but runs the context stack once, the latent stack once at batch K and the sampler at M*B images per
        launch for passes of M members.  M is the largest count whose tensors stay addressable by the tensor-core kernels
        (Sampler.members_per_pass); `members_per_pass` can only lower it.  Eval mode only: in train mode every call advances the
        spectral-norm vectors and BatchNorm statistics in call order."""
        if self.training:
            raise RuntimeError("Generator.sample is eval-mode only (call .eval() first)")
        K = int(num_samples)
        if K < 1:
            raise RuntimeError(f"Generator.sample: num_samples must be >= 1, got {num_samples}")
        if not all(hasattr(m, "run") for m in (self.conditioning_stack, self.latent_stack, self.sampler)):
            raise RuntimeError("Generator.sample needs the package's own conditioning stacks and sampler")
        B, H, W = x.shape[0], x.shape[-2], x.shape[-1]
        lh, lw = self.latent_stack.shape[1], self.latent_stack.shape[2]
        M = self.sampler.members_per_pass(B, lh, lw)
        if members_per_pass is not None:
            if members_per_pass < 1:
                raise RuntimeError(f"Generator.sample: members_per_pass must be >= 1, got {members_per_pass}")
            M = min(M, int(members_per_pass))
        with torch.no_grad():
            cond = list(self.conditioning_stack.run(x))     # no RNG and no batch statistics in eval mode: the same for every member
            lat = self.latent_stack.run(x, K)               # [K,1,h,w,c]: the K draws in the sequential calls' order
            out = torch.empty((B, K, self.sampler.forecast_steps, self.sampler.output_channels, H, W), device=x.device, dtype=torch.float32)
            for k0 in range(0, K, M):
                self.sampler.run(cond, lat[k0:k0 + M], out=out, member0=k0)
        return out

    def forward(self, x: torch.Tensor):
        """x: [B,T_in,C,H,W] -> [B,T,C_out,H,W]; context stack, then latent stack, then sampler (RNG order)."""
        if all(hasattr(m, "run") for m in (self.conditioning_stack, self.latent_stack, self.sampler)):
            cond = self.conditioning_stack.run(x)   # stays channels-last between the stacks
            lat = self.latent_stack.run(x)
            return self.sampler.run(list(cond), lat)
        cond = self.conditioning_stack(x)
        lat = self.latent_stack(x)
        return self.sampler(cond, lat)
