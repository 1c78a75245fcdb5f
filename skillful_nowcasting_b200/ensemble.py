"""Ensemble statistics of K-member nowcasts (Generator.sample) on the device: mean, exceedance probabilities and CRPS at the pooling
scales of the DGMR paper's evaluation, in one pass over the ensemble (csrc/ensemble.cu, include/dgmr_b200.h: dgmr_ensemble_stats).

A verification and product path, not a loss: nothing here is differentiable."""
from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import _lib

CRPS_SCALES = ("1", "avg4", "max4", "avg16", "max16")   # last axis of `crps`


def summarize(ens: torch.Tensor, thresholds: Sequence[float] = (), target: Optional[torch.Tensor] = None) -> dict:
    """ens: [B, K, T, C, H, W] float32 CUDA (what Generator.sample returns); thresholds: up to 8 values; target: [B, T, C, H, W] or None.

    Returns dict(mean=[B, T, C, H, W],
                 prob=[n_thr, B, T, C, H, W] (fraction of members >= each threshold) or None without thresholds,
                 crps=[B, T, C, 5] (ensemble CRPS averaged over the cells of each frame, scales CRPS_SCALES) or None without a target).
    CRPS needs H and W multiples of 16; 1 <= K <= 64."""
    if not isinstance(ens, torch.Tensor) or not ens.is_cuda:
        raise RuntimeError("ensemble.summarize needs a CUDA tensor (there is no CPU path)")
    if ens.dim() != 6 or ens.dtype != torch.float32:
        raise RuntimeError(f"ensemble.summarize: ens must be float32 [B, K, T, C, H, W], got {ens.dtype} {tuple(ens.shape)}")
    B, K, T, C, H, W = ens.shape
    if target is not None:
        if not isinstance(target, torch.Tensor) or not target.is_cuda or target.device != ens.device:
            raise RuntimeError("ensemble.summarize: target must be a CUDA tensor on the ensemble's device")
        if tuple(target.shape) != (B, T, C, H, W) or target.dtype != torch.float32:
            raise RuntimeError(f"ensemble.summarize: target must be float32 {(B, T, C, H, W)}, got {target.dtype} {tuple(target.shape)}")
        target = target.contiguous()
    ens = ens.contiguous()
    thr = torch.tensor([float(v) for v in thresholds], dtype=torch.float32, device=ens.device) if len(thresholds) else None
    n_thr = 0 if thr is None else thr.numel()
    mean = torch.empty((B, T, C, H, W), dtype=torch.float32, device=ens.device)
    prob = torch.empty((n_thr, B, T, C, H, W), dtype=torch.float32, device=ens.device) if n_thr else None
    crps = ws = None
    if target is not None:
        crps = torch.empty((B, T, C, 5), dtype=torch.float32, device=ens.device)
        ws = torch.empty((B * T * C * max(H // 16, 1) * 5,), dtype=torch.float64, device=ens.device)
    _lib.backend().ensemble_stats(ens, target, thr, mean, prob, crps, ws, B, K, T, C, H, W)
    return dict(mean=mean, prob=prob, crps=crps)
