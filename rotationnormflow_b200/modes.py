"""Separated posterior modes of a grid log-density (csrc/modes.cu, rnf_rotation_modes; DESIGN 4.7).

One call finds, per image, the M best *separated* points of a log-density evaluated on a rotation set, says which of them are
local maxima and how much of the probability each one carries: greedy non-maximum suppression on SO(3), on the device.
"""
from __future__ import annotations

import math

import torch

from . import _cabi

MAX_MODES = 256
RECORD_BYTES = 80          # RNF_MODES_RECORD_BYTES: one rank's per-image record of a sharded round


def _inputs(values, rotations, num_modes, min_separation, neighbour_radius):
    """The checked arguments of rotation_modes, values as float32 [B,G], rotations as float32 [G,3,3] on the values' device, and the
    output dict: (M, theta, rho, squeeze, values, rotations, out)."""
    M = int(num_modes)
    theta, rho = float(min_separation), float(neighbour_radius)
    if not 1 <= M <= MAX_MODES:
        raise ValueError(f"num_modes must be in 1..{MAX_MODES}, got {num_modes}")
    if not (0.0 < rho <= theta <= math.pi):
        raise ValueError(f"need 0 < neighbour_radius <= min_separation <= pi, got neighbour_radius={rho}, min_separation={theta}")
    if values.dim() not in (1, 2):
        raise ValueError(f"values must be [B,G] or [G], got {tuple(values.shape)}")
    if rotations.dim() != 3 or tuple(rotations.shape[1:]) != (3, 3) or rotations.shape[0] != values.shape[-1]:
        raise ValueError(f"rotations must be [G,3,3] with G = values.shape[-1], got {tuple(rotations.shape)} for {tuple(values.shape)}")
    if not (values.is_cuda and rotations.is_cuda):
        raise RuntimeError("rotationnormflow_b200 runs on a B200 only: tensors must be CUDA tensors (there is no CPU fallback)")
    squeeze = values.dim() == 1
    v = (values[None] if squeeze else values).to(torch.float32).contiguous()      # (a reshape to [-1, G] is ambiguous when G == 0)
    B, dev = v.shape[0], v.device
    out = dict(index=torch.empty((B, M), device=dev, dtype=torch.int64), value=torch.empty((B, M), device=dev, dtype=torch.float32),
               local_max=torch.empty((B, M), device=dev, dtype=torch.bool), mass=torch.empty((B, M), device=dev, dtype=torch.float32),
               count=torch.empty((B,), device=dev, dtype=torch.int32))
    return M, theta, rho, squeeze, v, rotations.to(dev, torch.float32).contiguous(), out


def rotation_modes(values: torch.Tensor, rotations: torch.Tensor, num_modes: int, min_separation: float, neighbour_radius: float,
                   g_index0: int = 0) -> dict:
    """Greedy modes of ``values`` [B,G] (or [G]) over ``rotations`` [G,3,3].  Per image, for m = 0 .. num_modes-1:

    * the mode is the best point not yet labelled: NaN first, then the larger value, then the lower index (the order of the grid
      arg-max of ``Flow.grid_log_prob``);
    * ``local_max`` is False if a point within ``neighbour_radius`` of it has a larger value (a NaN mode is never a local maximum);
    * every unlabelled point closer than ``min_separation`` to it joins it, and ``mass`` is the share of sum_g exp(values) they
      carry (relative to all G points; the points no mode took make up the remainder 1 - sum(mass)).

    Angles are geodesic (radians) and tested on quaternions of the fp32 matrices; the angle is right-invariant, so a grid and the
    same grid times an offset give the same labels.  ``0 < neighbour_radius <= min_separation <= pi``, ``1 <= num_modes <= 256``.

    Returns dict(index [B,M] int64 (``g_index0`` + local index), value [B,M], local_max [B,M] bool, mass [B,M], count [B] int32),
    without the leading dimension for a [G] input.  Entries at or after ``count`` are padding: index -1, value -inf, local_max False,
    mass 0.  No host synchronisation; the outputs are bitwise reproducible and the call can be captured in a CUDA graph.

    A pick that is not a local maximum is a "shoulder": the rim of an earlier mode's ball.  On a continuous ridge of equal density
    (the cone and cylinder of SYMSOL) the picks sample the ridge about every ``min_separation``, and their ``local_max`` flags are
    decided by fp32 noise along it."""
    M, theta, rho, squeeze, v, rot, out = _inputs(values, rotations, num_modes, min_separation, neighbour_radius)
    B, G = v.shape
    if B > 0:
        nbytes = int(_cabi.load().rnf_rotation_modes_workspace_bytes(G, B, M))
        ws = torch.empty((nbytes,), device=v.device, dtype=torch.uint8)
        _cabi.launch("rnf_rotation_modes", v.device, v, B, G, int(g_index0), rot, M, theta, rho, ws, nbytes, out["index"], out["value"],
                     out["local_max"], out["mass"], out["count"])
    if squeeze:
        out = {k: t[0] for k, t in out.items()}
    return out


class RankModes:
    """One rank's part of ``rotation_modes`` over a grid split across ranks (rnf_rotation_modes_shard_*; DESIGN 4.7 "Sharded").

    The rank holds ``values`` [B,G_r] (or [G_r]) and ``rotations`` [G_r,3,3] of the contiguous global slice starting at ``g_index0``.
    For r = 0 .. num_modes, ``propose(r)`` returns this rank's records of round r ([B, RECORD_BYTES] uint8); the records of all W
    ranks, stacked rank-major to [W, B, RECORD_BYTES], go to ``merge(r, gathered)`` on every rank.  After the last merge ``result()``
    on every rank equals ``rotation_modes`` on the concatenated grid (index, value, local_max, count bit for bit; mass up to the
    order of its sums).  ``rotation_modes_rank`` runs the loop with a gather function; this class is the step-wise form, for callers
    that drive several simulated ranks in one process or capture a round in a CUDA graph.  No host synchronisation."""

    def __init__(self, values, rotations, g_index0, num_modes, min_separation, neighbour_radius):
        if int(g_index0) < 0:
            raise ValueError(f"g_index0 must be >= 0, got {g_index0}")
        M, self.theta, self.rho, self.squeeze, self.v, self.rot, self.out = _inputs(values, rotations, num_modes, min_separation,
                                                                                    neighbour_radius)
        self.M, self.g_index0 = M, int(g_index0)
        self.B, self.G = self.v.shape
        B, dev = self.B, self.v.device
        self.device = dev
        self.out["rotations"] = torch.empty((B, M, 3, 3), device=dev, dtype=torch.float32)
        self.record = torch.empty((B, RECORD_BYTES), device=dev, dtype=torch.uint8)
        self.nbytes = int(_cabi.load().rnf_rotation_modes_shard_workspace_bytes(self.G, B))
        self.ws = torch.empty((self.nbytes,), device=dev, dtype=torch.uint8)
        _cabi.launch("rnf_rotation_modes_shard_setup", dev, self.rot, self.G, B, self.ws, self.nbytes)

    def propose(self, r: int) -> torch.Tensor:
        """Round r on this rank's slice: labels mode r-1's points, tests it, proposes mode r.  Returns the record buffer (reused by
        the next round: gather it before proposing again)."""
        _cabi.launch("rnf_rotation_modes_shard_round", self.device, self.v, self.B, self.G, self.g_index0, self.rot, int(r), self.M, self.theta,
                     self.rho, self.ws, self.nbytes, self.record)
        return self.record

    def merge(self, r: int, gathered: torch.Tensor) -> None:
        """Folds the records of round r of every rank, ``gathered`` [W, B, RECORD_BYTES] uint8 in rank order."""
        if gathered.dim() != 3 or gathered.dtype != torch.uint8 or tuple(gathered.shape[1:]) != (self.B, RECORD_BYTES):
            raise ValueError(f"gathered records must be uint8 [W,{self.B},{RECORD_BYTES}], got {gathered.dtype} {tuple(gathered.shape)}")
        g = gathered.to(self.device).contiguous()
        o = self.out
        _cabi.launch("rnf_rotation_modes_shard_merge", self.device, g, g.shape[0], self.B, int(r), self.M, self.ws, self.nbytes, o["index"],
                     o["value"], o["local_max"], o["mass"], o["count"], o["rotations"])

    def result(self) -> dict:
        """The outputs of ``rotation_modes`` plus ``rotations`` [B,M,3,3] (the owning rank's matrix of each mode, NaN padding) and
        ``valid`` [B,M] (entry < count)."""
        out = dict(self.out)
        out["valid"] = torch.arange(self.M, device=self.device)[None, :] < out["count"][:, None]
        if self.squeeze:
            out = {k: t[0] for k, t in out.items()}
        return out


def rotation_modes_rank(values: torch.Tensor, rotations: torch.Tensor, g_index0: int, num_modes: int, min_separation: float,
                        neighbour_radius: float, gather) -> dict:
    """This rank's call of ``rotation_modes`` over a grid split across W ranks (``RankModes``): M + 1 rounds, each one call of
    ``gather`` ([B, RECORD_BYTES] uint8 -> [W, B, RECORD_BYTES], rank-major; ``torch.distributed.all_gather_into_tensor`` across
    processes, ``torch.stack`` over simulated ranks).  Every rank returns the dict of ``RankModes.result``."""
    rm = RankModes(values, rotations, g_index0, num_modes, min_separation, neighbour_radius)
    for r in range(rm.M + 1):
        rm.merge(r, gather(rm.propose(r)))
    return rm.result()
