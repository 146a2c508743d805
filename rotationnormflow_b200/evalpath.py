"""The two evaluation call sites of the path (SURVEY.md 8f, N1), as single calls on [B,F] features.

    estimate_rotation_grid      eval.py:437-462  (gradient(): grid log-pdf + arg-max per image)
    estimate_rotation_sampling  agent.py:238-266 (eval_acc: inverse-flow samples + arg-max per image), uniform base
    refine_rotation             eval.py:464-480  (nll_grad: Adam on a quaternion per row, climbing log p; one fused launch per step)

Both avoid the reference's `feature.repeat` (4 GB per 500 000-row chunk at F = 2080, eval.py:450) and its per-image
Python loop; all per-rotation arithmetic runs in the fused kernels.
"""
from __future__ import annotations

import torch

from . import grid as rgrid


def _random_rotation(device, generator=None):
    q = torch.randn(4, generator=generator, device="cpu").to(device)
    q = q / torch.copysign(q.norm(), q[0])
    r, i, j, k = q.unbind(-1)
    two_s = 2.0 / (q * q).sum()
    return torch.stack((1 - two_s * (j * j + k * k), two_s * (i * j - k * r), two_s * (i * k + j * r),
                        two_s * (i * j + k * r), 1 - two_s * (i * i + k * k), two_s * (j * k - i * r),
                        two_s * (i * k - j * r), two_s * (j * k + i * r), 1 - two_s * (i * i + j * j))).reshape(3, 3)


@torch.no_grad()
def estimate_rotation_grid(flow, feature, number_queries, fisher_A=None, offset=None, generator=None, mlp_mode=None,
                           gt_rotations=None, refine_steps=0, refine_lr=None):
    """Returns (est_rotation [B,3,3], dict(max, argmax, sumexp[, spread])).  One random right-offset per batch
    (eval.py:439-440).  gt_rotations [B,K,3,3] adds the probability-weighted angular error (spread) of the same pass.
    refine_steps > 0 chains ``refine_rotation`` (lr = refine_lr) after the arg-max: the returned estimate is the refined one and
    the dict gains ``refined_logp`` [B] (the spread stays the grid's)."""
    dev = feature.device
    grid = rgrid.get_closest_available_grid(number_queries, dev)
    if offset is None:
        offset = _random_rotation(dev, generator)
    out = flow.grid_log_prob(grid, feature, offset=offset, fisher_A=fisher_A, mlp_mode=mlp_mode, gt_rotations=gt_rotations)
    est = grid[out["argmax"]] @ offset.to(dev)
    if refine_steps > 0:
        if refine_lr is None:
            raise ValueError("refine_steps > 0 needs refine_lr")
        est, out["refined_logp"] = refine_rotation(flow, feature, est, lr=refine_lr, steps=refine_steps, fisher_A=fisher_A)
    return est, out


@torch.no_grad()
def estimate_rotation_sampling(flow, feature, number_queries, base_samples=None, base_ll=None, mlp_mode=None,
                               fisher_A=None, seed=None):
    """agent.py:238-266: base rotations pushed through Flow.inverse; arg-max of -ldj + base_ll per image.

    Uniform base (default): the same `number_queries` rotations for every image (sd.generate_queries + repeat,
    agent.py:253-256).  ``fisher_A`` [B,3,3] (config.pretrain_fisher, agent.py:247-251): per-image samples from
    MatrixFisherN(A) drawn on the device, with their base log-likelihood.
    Returns (est_rotation [B,3,3], samples [B,Q,3,3], log_prob [B,Q])."""
    dev = feature.device
    B = feature.shape[0]
    if fisher_A is not None:
        from .fisher import MatrixFisherN
        pre = MatrixFisherN(fisher_A.to(dev))
        base = pre._sample(number_queries, seed=seed)                  # [B,Q,3,3]
        Q = base.shape[1]
        rows = base.reshape(-1, 3, 3)
        base_ll = pre._log_prob(rows).reshape(B, Q)
        idx = torch.arange(B, device=dev, dtype=torch.int32).repeat_interleave(Q)
        samples, ldj = flow.inverse(rows, feature, feature_index=idx, mlp_mode=mlp_mode)
        log_prob = -ldj.reshape(B, Q) + base_ll
        best = torch.argmax(log_prob, dim=-1)
        samples = samples.reshape(B, Q, 3, 3)
        return samples[torch.arange(B, device=dev), best], samples, log_prob
    if base_samples is None:
        base_samples = rgrid.generate_queries(number_queries, "random", dev)
    Q = base_samples.shape[0]
    rows = base_samples[None].expand(B, Q, 3, 3).reshape(-1, 3, 3)
    idx = torch.arange(B, device=dev, dtype=torch.int32).repeat_interleave(Q)
    samples, ldj = flow.inverse(rows, feature, feature_index=idx, mlp_mode=mlp_mode)
    log_prob = -ldj.reshape(B, Q)
    if base_ll is not None:
        log_prob = log_prob + base_ll
    best = torch.argmax(log_prob, dim=-1)
    samples = samples.reshape(B, Q, 3, 3)
    est = samples[torch.arange(B, device=dev), best]
    return est, samples, log_prob


def matrix_to_quaternion(R: torch.Tensor) -> torch.Tensor:
    """[...,3,3] -> unit quaternions [...,4] (real first) from the best-conditioned of the four candidate rows (the public
    pytorch3d construction); the sign is arbitrary, which quaternion_to_matrix does not see."""
    m = R.reshape(-1, 9)
    m00, m01, m02, m10, m11, m12, m20, m21, m22 = m.unbind(-1)
    q_abs = torch.sqrt(torch.clamp(torch.stack([1 + m00 + m11 + m22, 1 + m00 - m11 - m22, 1 - m00 + m11 - m22,
                                                1 - m00 - m11 + m22], dim=-1), min=0))
    cand = torch.stack([torch.stack([q_abs[:, 0] ** 2, m21 - m12, m02 - m20, m10 - m01], dim=-1),
                        torch.stack([m21 - m12, q_abs[:, 1] ** 2, m10 + m01, m02 + m20], dim=-1),
                        torch.stack([m02 - m20, m10 + m01, q_abs[:, 2] ** 2, m12 + m21], dim=-1),
                        torch.stack([m10 - m01, m20 + m02, m21 + m12, q_abs[:, 3] ** 2], dim=-1)], dim=-2)
    cand = cand / (2.0 * q_abs.clamp(min=0.1))[..., None]
    best = q_abs.argmax(dim=-1)
    q = cand[torch.arange(m.shape[0], device=R.device), best]
    return (q / q.norm(dim=-1, keepdim=True)).reshape(R.shape[:-2] + (4,))


def quaternion_to_matrix(q: torch.Tensor) -> torch.Tensor:
    """[...,4] (real first) -> [...,3,3], two_s = 2/|q|^2 as in the public pytorch3d definition (differentiable torch ops)."""
    r, i, j, k = q.unbind(-1)
    two_s = 2.0 / (q * q).sum(-1)
    o = torch.stack((1 - two_s * (j * j + k * k), two_s * (i * j - k * r), two_s * (i * k + j * r),
                     two_s * (i * j + k * r), 1 - two_s * (i * i + k * k), two_s * (j * k - i * r),
                     two_s * (i * k - j * r), two_s * (j * k + i * r), 1 - two_s * (i * i + j * j)), -1)
    return o.reshape(q.shape[:-1] + (3, 3))


def refine_rotation(flow, feature, rotation, *, lr, steps=100, fisher_A=None):
    """The nll_grad refinement of eval.py:464-480: ``steps`` Adam steps (learning rate ``lr``) on a real-first quaternion per row,
    maximising log p(R | image).

    rotation [B,3,3], or [B,M,3,3] for M seeds per image; feature [B,F] (None for an unconditional flow); fisher_A [B,3,3] adds the
    matrix-Fisher base term.  Per step the flow runs once, in one launch (Flow.log_prob_grad), and its tangential gradient is pulled
    back to the quaternion through R = quaternion_to_matrix(q / |q|).  Returns (R_refined, logp) shaped like rotation / rotation[..., 0, 0]."""
    if rotation.dim() not in (3, 4) or tuple(rotation.shape[-2:]) != (3, 3):
        raise ValueError(f"rotation must be [B,3,3] or [B,M,3,3], got {tuple(rotation.shape)}")
    shape = rotation.shape
    feat = feature.detach() if feature is not None else None
    q = matrix_to_quaternion(rotation.detach().to(torch.float32).reshape(-1, 3, 3))
    with torch.enable_grad():
        q = q.clone().requires_grad_(True)
        opt = torch.optim.Adam([q], lr=lr)
        for _ in range(int(steps)):
            R = quaternion_to_matrix(q / q.norm(dim=-1, keepdim=True))
            _, G = flow.log_prob_grad(R.detach(), feat, fisher_A=fisher_A)
            opt.zero_grad()
            R.backward(-G)                                     # ascend log p
            opt.step()
    with torch.no_grad():
        R = quaternion_to_matrix(q / q.norm(dim=-1, keepdim=True))
        logp, _ = flow.log_prob_grad(R, feat, fisher_A=fisher_A)
    return R.reshape(shape), logp.reshape(shape[:-2])
