"""Grid-sharded evaluation across the GPUs of one box: one process per GPU, ``torch.distributed`` plumbing.

The reference evaluates the grid on a single GPU in 500 000-rotation chunks (eval.py:444-462) and only ever uses
``nn.DataParallel`` (agent.py:22).  Here every rank scores a contiguous slice ``[begin,end)`` of the grid for all B
images with the fused kernel and keeps, per image, (max log p, first arg-max index, sum exp(log p - max)); ONE
all-gather of ``[B,3]`` float64 (24 B per image per rank) merges them.  There is no other data-path collective: the
per-(rotation, image) evaluations are independent.

Separated modes over a sharded grid (``sharded_rotation_modes``, ``sharded_estimate_rotation_modes``; DESIGN 4.7 "Sharded") are the
exception: greedy picking needs each image's global best unlabelled point once per mode, so they make M + 1 all-gathers of an
80-byte record per image per rank, and return on every rank what the single-GPU call returns on the whole grid.
"""
from __future__ import annotations

import math

import torch
import torch.distributed as dist

from .modes import rotation_modes_rank


def shard_range(G: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous slice of ``range(G)`` owned by ``rank`` (sizes differ by at most one, earlier ranks larger)."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError(f"bad rank/world {rank}/{world}")
    base, rem = divmod(G, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def merge_partials(mx: torch.Tensor, am: torch.Tensor, se: torch.Tensor, sn: torch.Tensor | None = None):
    """Merge per-shard partials stacked on dim 0: mx/am/se are [W,B] -> (max [B], argmax [B], sumexp [B]).

    Ties on the maximum resolve to the smallest global index (torch.argmax / first-index semantics of
    agent.py:264, eval.py:461).  Shards holding no rotations carry max = -inf and sumexp = 0.
    ``sn`` [W,B] (spread numerators, relative to each shard's max) is rescaled and summed like sumexp and returned fourth."""
    m = mx.max(dim=0).values
    cand = torch.where(mx == m[None, :], am, torch.full_like(am, torch.iinfo(torch.int64).max))
    idx = cand.min(dim=0).values
    scale = torch.where(torch.isfinite(mx), torch.exp(mx.double() - m.double()[None, :]), torch.zeros_like(mx, dtype=torch.float64))
    s = (se.double() * scale).sum(dim=0)
    if sn is not None:
        return m, idx, s.to(se.dtype), (sn.double() * scale).sum(dim=0).to(sn.dtype)
    return m, idx, s.to(se.dtype)


def _world_size(group) -> int:
    return dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1


def _gather(t: torch.Tensor, group) -> torch.Tensor:
    """[n, ...] -> [W, n, ...], rank-major: one all_gather_into_tensor (the identity on one rank)."""
    world = _world_size(group)
    if world == 1:
        return t[None]
    flat = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(flat, t.contiguous(), group=group)
    return flat.view(world, *t.shape)


def all_merge(mx: torch.Tensor, am: torch.Tensor, se: torch.Tensor, group=None, sn: torch.Tensor | None = None):
    """One all-gather of the packed partials ([B,3] float64, [B,4] with spread numerators), then ``merge_partials`` on every rank."""
    if _world_size(group) == 1:
        return (mx, am, se) if sn is None else (mx, am, se, sn)
    cols = [mx.double(), am.double(), se.double()] + ([] if sn is None else [sn.double()])   # indices < 2^53 are exact
    gathered = _gather(torch.stack(cols, dim=1), group)
    return merge_partials(gathered[:, :, 0].to(mx.dtype), gathered[:, :, 1].to(torch.int64), gathered[:, :, 2].to(se.dtype),
                          None if sn is None else gathered[:, :, 3].to(sn.dtype))


def log_normaliser(mx: torch.Tensor, se: torch.Tensor, G_total: int) -> torch.Tensor:
    """log mean_g exp(logp)  (the ``exp(logp).mean()`` sanity value of eval.py:103-104), from (max, sumexp)."""
    return mx + torch.log(se) - math.log(G_total)


def sharded_grid_log_prob(flow, grid_shard: torch.Tensor, g_index0: int, G_total: int, feature=None, offset=None,
                          fisher_A=None, group=None, mlp_mode=None, gt_rotations=None):
    """Per-image (max, argmax, log-normaliser[, spread]) over a grid whose slices live on different ranks."""
    out = flow.grid_log_prob(grid_shard, feature, offset=offset, fisher_A=fisher_A, g_index0=g_index0, mlp_mode=mlp_mode,
                             gt_rotations=gt_rotations)
    if gt_rotations is not None:
        mx, am, se, sn = all_merge(out["max"], out["argmax"], out["sumexp"], group, sn=out["spread_num"])
        return dict(max=mx, argmax=am, sumexp=se, log_norm=log_normaliser(mx, se, G_total), spread=sn / se)
    mx, am, se = all_merge(out["max"], out["argmax"], out["sumexp"], group)
    return dict(max=mx, argmax=am, sumexp=se, log_norm=log_normaliser(mx, se, G_total))


def _record_gather(group):
    """[B, RECORD_BYTES] -> [W, B, RECORD_BYTES], rank-major: one all_gather_into_tensor (the identity on one rank)."""
    return lambda rec: _gather(rec, group)


def sharded_rotation_modes(values_shard: torch.Tensor, grid_shard: torch.Tensor, g_index0: int, G_total: int, num_modes: int,
                           min_separation: float, neighbour_radius: float, group=None) -> dict:
    """``modes.rotation_modes`` over a grid whose contiguous slices live on different ranks: this rank holds ``values_shard``
    [B,G_r] and ``grid_shard`` [G_r,3,3], the global slice [g_index0, g_index0 + G_r) of a G_total-point grid (``shard_range``).
    Every rank returns the same dict: index (global), value, local_max, mass, count, valid and ``rotations`` [B,M,3,3], each mode's
    ``grid_shard`` row as held by the rank that owns it (carried in the record, so any rotation set works; NaN padding).  It equals
    ``rotation_modes`` on the whole grid: index, value, local_max, count and valid bit for bit, mass up to the order of its sums.
    M + 1 all-gathers of [B, 80] bytes and nothing else; an empty slice (G_r = 0) takes part in each.  No host synchronisation."""
    G_r = grid_shard.shape[0]
    if not (0 <= g_index0 and g_index0 + G_r <= G_total):
        raise ValueError(f"slice [{g_index0}, {g_index0 + G_r}) is not inside the {G_total}-point grid")
    return rotation_modes_rank(values_shard, grid_shard, g_index0, num_modes, min_separation, neighbour_radius, _record_gather(group))


@torch.no_grad()
def sharded_estimate_rotation_modes(flow, grid_shard: torch.Tensor, g_index0: int, G_total: int, feature, num_modes: int, *,
                                    min_separation: float, neighbour_radius=None, fisher_A=None, offset=None, refine_steps: int = 0,
                                    refine_lr=None, group=None):
    """``evalpath.estimate_rotation_modes`` on a HEALPix grid of G_total points split across ranks: every rank scores its slice
    (``grid_shard``, starting at global index ``g_index0``) for all images, the modes are ``sharded_rotation_modes`` of the slices,
    and every rank returns (rotations [B,M,3,3], dict(logp, mass, valid, count, grid_index)) as the single-GPU call returns them for
    the same grid and offset.  ``offset`` (the same [3,3] on every rank; None = no offset) right-multiplies the grid.  With
    refine_steps > 0 every rank runs the same ``refine_rotation`` call on all modes (per-row arithmetic, so the ranks stay
    identical) and the same merge of refined modes.  ``neighbour_radius`` defaults to ``evalpath.default_neighbour_radius`` of the
    grid's level.  The images go in chunks whose log-density on the largest slice stays under ``evalpath.MODES_LOGP_BYTES``; the
    chunking depends on G_total and the world size only, so all ranks make the same collectives."""
    from . import evalpath
    from . import grid as rgrid
    rho = evalpath._modes_radius(rgrid.closest_grid_level(G_total), min_separation, neighbour_radius, refine_steps, refine_lr)
    dev = grid_shard.device
    G_r = grid_shard.shape[0]
    off = None if offset is None else offset.to(dev, torch.float32)
    parts = []
    for f, A, n in evalpath._image_chunks(flow, feature, fisher_A, -(-G_total // _world_size(group))):
        if G_r > 0:
            lp = flow.grid_log_prob(grid_shard, f, offset=off, fisher_A=A, return_logp=True, g_index0=g_index0)["logp"]
        else:
            lp = torch.empty((n, 0), device=dev, dtype=torch.float32)
        parts.append(sharded_rotation_modes(lp, grid_shard, g_index0, G_total, int(num_modes), min_separation, rho, group))
    md = {k: torch.cat([p[k] for p in parts]) for k in ("index", "value", "local_max", "mass", "rotations")}
    return evalpath._finish_modes(flow, feature, fisher_A, md, md["rotations"], off, rho, refine_steps, refine_lr)
