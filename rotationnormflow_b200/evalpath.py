"""The two evaluation call sites of the path (SURVEY.md 8f, N1), as single calls on [B,F] features.

    estimate_rotation_grid      eval.py:437-462  (gradient(): grid log-pdf + arg-max per image)
    estimate_rotation_sampling  agent.py:238-266 (eval_acc: inverse-flow samples + arg-max per image), uniform base
    refine_rotation             eval.py:464-480  (nll_grad: Adam on a quaternion per row, climbing log p; one fused launch per step)
    estimate_rotation_modes     (no reference counterpart) the M best separated modes per image from one grid pass, optionally refined
    estimate_rotation_hierarchical  (no reference counterpart) the grid arg-max of a fine level from a coarse grid pass and a beam of
                                child cells per level

Both avoid the reference's `feature.repeat` (4 GB per 500 000-row chunk at F = 2080, eval.py:450) and its per-image
Python loop; all per-rotation arithmetic runs in the fused kernels.
"""
from __future__ import annotations

import math

import torch

from . import grid as rgrid
from .modes import rotation_modes

# Default neighbour_radius of estimate_rotation_modes per grid level: 1.5x the largest nearest-neighbour angle of the level-l HEALPix
# grid, measured once on the CPU by tools/grid_spacing.py (DESIGN 4.7).  From level 2 on the measured angle halves exactly per level
# (pi / 12 at level 2), so levels past 5 continue the halving.
NEIGHBOUR_RADIUS = (1.570796, 0.778990, 0.392699, 0.196350, 0.098175, 0.049087)
# estimate_rotation_modes evaluates the grid in image chunks whose [chunk, G] float32 log-density stays under this many bytes
# (a level-6 grid is 151 MB per image)
MODES_LOGP_BYTES = 1 << 30
# estimate_rotation_hierarchical scores flows the fused kernels cannot run in pieces of at most this many bytes of per-row state
# (a feature row per rotation, F = 2080: about 112 000 rotations)
HIER_LAYERWISE_BYTES = 1 << 30


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
def default_neighbour_radius(level: int) -> float:
    """1.5x the largest nearest-neighbour angle (radians) of the level-``level`` HEALPix grid (NEIGHBOUR_RADIUS)."""
    if level < len(NEIGHBOUR_RADIUS):
        return NEIGHBOUR_RADIUS[level]
    return NEIGHBOUR_RADIUS[-1] / 2 ** (level - len(NEIGHBOUR_RADIUS) + 1)


def _modes_radius(level, min_separation, neighbour_radius, refine_steps, refine_lr) -> float:
    """The checks of the mode-estimation arguments; returns neighbour_radius (default: default_neighbour_radius(level))."""
    rho = default_neighbour_radius(level) if neighbour_radius is None else float(neighbour_radius)
    if float(min_separation) < rho:
        raise ValueError(f"min_separation={min_separation} is below neighbour_radius={rho}: a mode's neighbourhood would reach past its "
                         "own ball")
    if refine_steps > 0 and refine_lr is None:
        raise ValueError("refine_steps > 0 needs refine_lr")
    return rho


def _image_chunks(flow, feature, fisher_A, G):
    """(feature, fisher_A, images) of consecutive image chunks whose [images, G] float32 log-density stays under MODES_LOGP_BYTES.
    An unconditional flow is one image, its feature passed on as given."""
    conditional = feature is not None and flow.condition
    B = feature.shape[0] if conditional else 1
    chunk = max(1, MODES_LOGP_BYTES // (G * 4))
    for s in range(0, B, chunk):
        yield (feature[s:s + chunk] if conditional else feature, fisher_A[s:s + chunk] if fisher_A is not None else None,
               min(chunk, B - s))


def _finish_modes(flow, feature, fisher_A, md, rows, offset, rho, refine_steps, refine_lr):
    """What follows ``rotation_modes`` in estimate_rotation_modes and dist.sharded_estimate_rotation_modes.  ``md`` holds index, value,
    local_max and mass [B,M] of the greedy picks, ``rows`` [B,M,3,3] their rotations before the ``offset`` [3,3] (None: no offset).
    Drops the shoulders, keeping the greedy order (non-increasing value) of the local maxima; refine_steps > 0 refines all modes and
    merges those within ``rho``.  Returns (rotations [B,M,3,3], dict(logp, mass, valid, count, grid_index)), padded with NaN, -inf,
    0 and -1."""
    valid = md["local_max"]
    order = torch.sort((~valid).to(torch.int8), dim=1, stable=True).indices
    valid = torch.gather(valid, 1, order)
    index = torch.where(valid, torch.gather(md["index"], 1, order), -1)
    logp = torch.where(valid, torch.gather(md["value"], 1, order), -math.inf)
    mass = torch.where(valid, torch.gather(md["mass"], 1, order), 0.0)
    rot = torch.gather(rows, 1, order[..., None, None].expand(-1, -1, 3, 3))
    if offset is not None:
        rot = rot @ offset
    if refine_steps > 0:
        mode0 = rows[:, 0] if offset is None else rows[:, 0] @ offset
        seeds = torch.where(valid[..., None, None], rot, mode0[:, None])          # padding: mode 0 of the grid
        rot, lp = refine_rotation(flow, feature, seeds, lr=refine_lr, steps=refine_steps, fisher_A=fisher_A)
        rot, logp, mass, valid, index = _merge_modes(rot, torch.where(valid, lp, -math.inf), mass, valid, index, rho)
    rot = torch.where(valid[..., None, None], rot, math.nan)
    return rot, dict(logp=logp, mass=mass, valid=valid, count=valid.sum(1), grid_index=index)


@torch.no_grad()
def estimate_rotation_modes(flow, feature, number_queries, num_modes, *, min_separation, neighbour_radius=None, fisher_A=None, offset=None,
                            generator=None, mlp_mode=None, refine_steps=0, refine_lr=None):
    """The ``num_modes`` best separated posterior modes per image from one grid pass (the grid and offset of
    ``estimate_rotation_grid``): ``modes.rotation_modes`` on the grid log-density with angles ``min_separation`` and
    ``neighbour_radius`` (default ``default_neighbour_radius(level)``; radians), keeping the local maxima only.

    refine_steps > 0 runs one ``refine_rotation`` (lr = refine_lr) on all [B,M] modes at once, then merges refined modes closer than
    ``neighbour_radius`` greedily by refined log p (the masses of merged modes add up).

    Returns (rotations [B,M,3,3], dict(logp [B,M], mass [B,M], valid [B,M] bool, count [B], grid_index [B,M] int64, max [B], argmax [B],
    sumexp [B])): modes sorted by log p (the refined one after refinement), valid ones first; padded entries have NaN rotations, logp
    -inf, mass 0 and grid_index -1.  ``max`` / ``argmax`` / ``sumexp`` are those of ``Flow.grid_log_prob``; mode 0 of the grid pass is
    its arg-max.  The grid is evaluated in image chunks of at most MODES_LOGP_BYTES of log-density."""
    rho = _modes_radius(rgrid.closest_grid_level(number_queries), min_separation, neighbour_radius, refine_steps, refine_lr)
    dev = feature.device if feature is not None else torch.device("cuda", torch.cuda.current_device())
    grid = rgrid.get_closest_available_grid(number_queries, dev)
    if offset is None:
        offset = _random_rotation(dev, generator)
    offset = offset.to(dev, torch.float32)
    parts = []
    for f, A, _ in _image_chunks(flow, feature, fisher_A, grid.shape[0]):
        out = flow.grid_log_prob(grid, f, offset=offset, fisher_A=A, return_logp=True, mlp_mode=mlp_mode)
        md = rotation_modes(out.pop("logp"), grid, int(num_modes), min_separation, rho)
        parts.append((out, md))
    out = {k: torch.cat([p[0][k] for p in parts]) for k in ("max", "argmax", "sumexp")}
    md = {k: torch.cat([p[1][k] for p in parts]) for k in ("index", "value", "local_max", "mass")}
    rot, modes = _finish_modes(flow, feature, fisher_A, md, grid[md["index"].clamp(min=0)], offset, rho, refine_steps, refine_lr)
    out.update(modes)
    return rot, out


def _score_rows(flow, rows, feature, per_image, fisher_A, mlp_mode):
    """log p of image-major ``rows`` [B*per_image,3,3] (or [per_image,3,3], the same rows for every image) through Flow.forward, plus
    the matrix-Fisher term of ``fisher_A`` [B,3,3]: ldj + (tr(A_b R') - c_b), the arithmetic of the grid kernels' epilogue.
    Returns [B, per_image].

    Flows the fused kernels run go in one launch.  The others (segments != 64, ConditionLU) run the per-layer operators, which build a
    feature row per rotation: they go one image at a time, in pieces of at most HIER_LAYERWISE_BYTES of per-row state, so memory does not
    grow with the number of images, and ConditionLU (batch-coupled: rows 0..3 of a launch decide its diagonal) sees one image's feature
    in every row of a launch, the reference's own calling convention (eval.py:450)."""
    from .fisher import MatrixFisherN
    from .flow import fused_kernels_run
    conditional = feature is not None and flow.condition
    B = feature.shape[0] if conditional else (fisher_A.shape[0] if fisher_A is not None else 1)
    shared = rows.shape[0] == per_image and B > 1
    if fused_kernels_run(flow.layers):
        R = rows.unsqueeze(0).expand(B, -1, -1, -1).reshape(-1, 3, 3) if shared else rows
        idx = torch.arange(B * per_image, device=rows.device, dtype=torch.int32) // per_image if conditional else None
        R_out, ldj = flow.forward(R, feature, feature_index=idx, mlp_mode=mlp_mode)
        if fisher_A is not None:
            ldj = ldj + MatrixFisherN(fisher_A)._log_prob(R_out)
        return ldj.reshape(B, per_image)
    K = max([l.K for l in flow.layers if l.kind == "mobius"] + [1])
    per_row = 4 * (flow.feature_dim + 19 + 4 * K + 2 * 64)          # feature row, R and R', ldj, one conditioner's output and hidden
    piece = max(1, HIER_LAYERWISE_BYTES // per_row)
    out = torch.empty((B, per_image), device=rows.device, dtype=torch.float32)
    for b in range(B):
        fb = feature[b:b + 1] if conditional else None
        fisher = MatrixFisherN(fisher_A[b:b + 1]) if fisher_A is not None else None
        for s in range(0, per_image, piece):
            n = min(piece, per_image - s)
            r = rows[s:s + n] if shared or B == 1 else rows[b * per_image + s:b * per_image + s + n]
            idx = torch.zeros(n, device=rows.device, dtype=torch.int32) if conditional else None
            R_out, ldj = flow.forward(r, fb, feature_index=idx, mlp_mode=mlp_mode)
            if fisher is not None:
                ldj = ldj + fisher._log_prob(R_out)
            out[b, s:s + n] = ldj
    return out


@torch.no_grad()
def estimate_rotation_hierarchical(flow, feature, number_queries, *, start_level=3, beam=64, fisher_A=None, offset=None, generator=None,
                                   mlp_mode=None):
    """The arg-max of log p over the level-L HEALPix grid (L = closest_grid_level(number_queries), as estimate_rotation_grid) by a
    coarse-to-fine search, per image (DESIGN 4.8):

    1. score the full level-``start_level`` grid (Flow.grid_log_prob) and keep the ``beam`` best indices in the order of the grid
       arg-max (NaN first, then the larger value, then the lower index; grid.top_k);
    2. for each finer level up to L: expand the kept indices to their 8 children each (grid.healpix_children), score them with
       Flow.forward at exactly the rotation the grid pass scores at that index (grid rotation times the offset, plus the matrix-Fisher
       term with ``fisher_A``), and keep the ``beam`` best;
    3. report the best candidate of level L.

    Every candidate is a member of the level-L grid; with beam >= 72 * 8^(L-1) the search scores every level-L rotation.  A peak
    narrower than the coarse spacing can be missed.  Flow.forward and Flow.grid_log_prob do not round a rotation's log p bit for bit
    alike (DESIGN 4.8: up to 6e-5 relative measured), so the reported log p can exceed the full grid's maximum by that difference, and
    an exhaustive search can pick another index whose full-grid log p is within it of the maximum.  A wider beam usually does at least
    as well, but not always: it can drop the branch a narrower beam follows.

    Flow.forward runs every layer kind (ablation layers, ConditionLU, segments != 64).  Flow.grid_log_prob refuses the last two, so for
    them the coarse pass scores the level-``start_level`` grid as the children of the level below, through Flow.forward, one image at
    a time (_score_rows): they need start_level >= 1 and a final level >= 1.  ``offset`` / ``generator`` as in estimate_rotation_grid.
    start_level >= L is the plain grid arg-max of level L.  Images are searched in chunks whose coarse [chunk, G0] log-density stays
    under MODES_LOGP_BYTES.

    Returns (est [B,3,3], dict(logp [B], index [B] int64 level-L grid index, level = L, top_logp [B,beam], top_index [B,beam] (the final
    beam, best first; (-inf, -1) where the level has fewer than beam rotations), evaluated = rotations scored per image))."""
    L = rgrid.closest_grid_level(number_queries)
    if isinstance(beam, bool) or int(beam) != beam or not 1 <= int(beam) <= rgrid.MAX_TOP_K:
        raise ValueError(f"beam must be an integer in 1..{rgrid.MAX_TOP_K}, got {beam}")
    if isinstance(start_level, bool) or int(start_level) != start_level or not 0 <= int(start_level) <= 8:
        raise ValueError(f"start_level must be an integer in 0..8, got {start_level}")
    beam, l0 = int(beam), min(int(start_level), L)
    from .flow import fused_kernels_run
    fused = fused_kernels_run(flow.layers)
    if not fused and l0 == 0:
        raise ValueError(f"a flow Flow.grid_log_prob cannot run (segments != 64 or ConditionLU) scores its coarse level as the children "
                         f"of the level below: it needs start_level >= 1 and a final level >= 1, got start_level={start_level}, final "
                         f"level {L} (number_queries={number_queries})")
    dev = feature.device if feature is not None else torch.device("cuda", torch.cuda.current_device())
    if offset is None:
        offset = _random_rotation(dev, generator)
    offset = offset.to(dev, torch.float32)
    G0 = rgrid.GRID_SIZES[l0]
    parts = []
    for f, A, nb in _image_chunks(flow, feature, fisher_A, G0):
        if fused:
            grid0 = rgrid.get_closest_available_grid(G0, dev)
            lp = flow.grid_log_prob(grid0, f, offset=offset, fisher_A=A, return_logp=True, mlp_mode=mlp_mode)["logp"]
            idx0 = None
        else:
            idx0, rot0 = rgrid.healpix_children(l0 - 1, torch.arange(G0 // 8, device=dev), offset)
            lp = _score_rows(flow, rot0.reshape(G0, 3, 3), f, G0, A, mlp_mode)
            idx0 = idx0.reshape(1, G0).expand(nb, G0)
        k = beam if l0 == L else min(beam, G0)
        top_v, top_i = rgrid.top_k(lp, idx0, k)
        if l0 == L:     # the plain grid arg-max: the grid pass's own rotation (estimate_rotation_grid)
            est = rgrid.get_closest_available_grid(G0, dev)[top_i[:, 0].clamp(min=0)] @ offset
        for level in range(l0 + 1, L + 1):
            child, rot = rgrid.healpix_children(level - 1, top_i.reshape(-1), offset)       # [nb*k, 8], [nb*k, 8, 3, 3]
            n = 8 * top_i.shape[1]
            lp = _score_rows(flow, rot.reshape(-1, 3, 3), f, n, A, mlp_mode)
            child = child.reshape(nb, n)
            top_v, top_i = rgrid.top_k(lp, child, beam if level == L else min(beam, rgrid.GRID_SIZES[level]))
            if level == L:
                pos = (child == top_i[:, :1]).to(torch.int8).argmax(1)
                est = rot.reshape(nb, n, 3, 3)[torch.arange(nb, device=dev), pos]
        parts.append((est, top_v, top_i))
    est = torch.cat([p[0] for p in parts])
    top_v = torch.cat([p[1] for p in parts])
    top_i = torch.cat([p[2] for p in parts])
    evaluated = G0 + sum(8 * min(beam, rgrid.GRID_SIZES[l - 1]) for l in range(l0 + 1, L + 1))
    return est, dict(logp=top_v[:, 0], index=top_i[:, 0], level=L, top_logp=top_v, top_index=top_i, evaluated=evaluated)


def _merge_modes(rot, logp, mass, valid, index, radius):
    """Greedy merge of refined modes by log p: a mode within ``radius`` of a better one that is kept adds its mass to the best such
    one and is dropped.  Returns the kept modes first, sorted by log p, padded as estimate_rotation_modes pads."""
    B, M = logp.shape
    order = torch.sort(logp, dim=1, descending=True, stable=True).indices
    rot = torch.gather(rot, 1, order[..., None, None].expand(B, M, 3, 3))
    logp, mass, valid, index = (torch.gather(t, 1, order) for t in (logp, mass, valid, index))
    q = matrix_to_quaternion(rot)
    close = (q @ q.transpose(1, 2)).abs() >= math.cos(radius / 2)            # [B,M,M], angle <= radius
    kept = torch.zeros_like(valid)
    target = torch.arange(M, device=rot.device).expand(B, M).clone()
    for i in range(M):
        near = close[:, i, :i] & kept[:, :i]
        merged = near.any(1)
        kept[:, i] = valid[:, i] & ~merged
        if i > 0:
            target[:, i] = torch.where(valid[:, i] & merged, near.to(torch.int8).argmax(1), i)
    mass = torch.zeros_like(mass).scatter_add_(1, target, torch.where(valid, mass, 0.0))
    order = torch.sort((~kept).to(torch.int8), dim=1, stable=True).indices
    rot = torch.gather(rot, 1, order[..., None, None].expand(B, M, 3, 3))
    logp, mass, kept, index = (torch.gather(t, 1, order) for t in (logp, mass, kept, index))
    return rot, torch.where(kept, logp, -math.inf), torch.where(kept, mass, 0.0), kept, torch.where(kept, index, -1)


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
