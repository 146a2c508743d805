"""Post-path metrics on the device (SURVEY.md 8f N2): utils/utils.py:208-209 (acc), :225-235 (geodesic distances)."""
from __future__ import annotations

import torch

from . import _cabi


def min_geodesic_distance_rotmats(r1s: torch.Tensor, r2s: torch.Tensor) -> torch.Tensor:
    """r1s [n,3,3] (estimates), r2s [n,k,3,3] (ground-truth sets) -> [n] angle to the closest one (utils/utils.py:231-235)."""
    if not r1s.is_cuda:
        raise RuntimeError("rotationnormflow_b200 runs on a B200 only: tensors must be CUDA tensors (there is no CPU fallback)")
    n = r1s.shape[0]
    r2s = r2s.reshape(n, -1, 3, 3)
    est = r1s.reshape(n, 9).to(torch.float32).contiguous()
    gt = r2s.to(r1s.device, torch.float32).contiguous()
    out = torch.empty((n,), device=r1s.device, dtype=torch.float32)
    _cabi.launch("rnf_min_geodesic", r1s.device, est, gt, n, gt.shape[1], out)
    return out


def geodesic_distance_rotmats(r1s: torch.Tensor, r2s: torch.Tensor) -> torch.Tensor:
    """utils/utils.py:225-228."""
    return min_geodesic_distance_rotmats(r1s, r2s[:, None])


def acc(x: torch.Tensor, thres) -> torch.Tensor:
    """utils/utils.py:208-209."""
    return (x <= thres).sum() / len(x)


def mode_recall(modes: torch.Tensor, valid: torch.Tensor, gt: torch.Tensor, threshold) -> torch.Tensor:
    """Per image, the fraction of the K ground-truth equivalents gt [B,K,3,3] that have a valid mode (modes [B,M,3,3], valid [B,M],
    as returned by evalpath.estimate_rotation_modes) within ``threshold`` radians: [B] float32.  An image without a valid mode
    scores 0."""
    if not modes.is_cuda:
        raise RuntimeError("rotationnormflow_b200 runs on a B200 only: tensors must be CUDA tensors (there is no CPU fallback)")
    m = modes.to(torch.float32)
    g = gt.to(m.device, torch.float32)
    # angle(G_k, R_m) from the trace of G_k^T R_m, [B,K,M]
    tr = torch.einsum("bkij,bmij->bkm", g, m)
    ang = torch.arccos(((tr - 1) / 2).clamp(-1.0, 1.0))
    hit = ((ang <= threshold) & valid.to(m.device)[:, None, :]).any(-1)
    return hit.to(torch.float32).mean(-1)
