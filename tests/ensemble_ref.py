"""Plain-torch reference of the ensemble statistics (skillful_nowcasting_b200.ensemble.summarize), in float64, that the GPU tests compare
the kernel against.  The pairwise CRPS form is the definition; the sorted-order identity is the cheap equivalent used on large ensembles
(tests/test_ensemble_cpu.py checks that the two agree)."""
import torch
import torch.nn.functional as F


def crps_pairwise(ens, y):
    """ens [N, K], y [N] -> [N]: (1/K) sum_k |x_k - y| - (1/(2K^2)) sum_{j,k} |x_j - x_k|."""
    K = ens.shape[1]
    a = (ens - y[:, None]).abs().mean(1)
    pair = (ens[:, :, None] - ens[:, None, :]).abs().sum((1, 2))
    return a - pair / (2 * K * K)


def crps_sorted(ens, y):
    """Same value through sum_{j,k} |x_j - x_k| = 2 sum_i (2i - K + 1) x_(i) (0-based ascending order)."""
    K = ens.shape[1]
    a = (ens - y[:, None]).abs().mean(1)
    xs = ens.sort(dim=1).values
    w = (2 * torch.arange(K, dtype=ens.dtype, device=ens.device) - K + 1)
    return a - (xs * w).sum(1) / (K * K)


def _pool(x, s, kind):
    """x [..., H, W] -> [..., H/s, W/s] (non-overlapping windows)."""
    lead, (h, w) = x.shape[:-2], x.shape[-2:]
    y = x.reshape(-1, 1, h, w)
    y = F.avg_pool2d(y, s) if kind == "avg" else F.max_pool2d(y, s)
    return y.reshape(lead + y.shape[-2:])


def summarize_ref(ens, thresholds=(), target=None):
    """ens [B, K, T, C, H, W], target [B, T, C, H, W] -> dict(mean, prob, crps) with the layouts of ensemble.summarize."""
    B, K, T, C, H, W = ens.shape
    mean = ens.double().mean(1)
    # count / K correctly rounded (torch's CUDA division by a scalar multiplies by its reciprocal: up to 1 ulp off)
    prob = torch.stack([((ens >= t).sum(1).double() / K).float() for t in thresholds]) if len(thresholds) else None
    crps = None
    if target is not None:
        e, y = ens.double(), target.double()
        cols = []
        for s, kind in ((1, None), (4, "avg"), (4, "max"), (16, "avg"), (16, "max")):
            ep, yp = (e, y) if s == 1 else (_pool(e, s, kind), _pool(y, s, kind))
            cells = yp.shape[-2] * yp.shape[-1]
            flat_e = ep.permute(0, 2, 3, 4, 5, 1).reshape(-1, K)          # [B*T*C*cells, K]
            c = crps_sorted(flat_e, yp.reshape(-1))
            cols.append(c.reshape(B, T, C, cells).mean(-1))
        crps = torch.stack(cols, -1)
    return dict(mean=mean, prob=prob, crps=crps)
