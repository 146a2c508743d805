"""Separated posterior modes of a grid log-density (csrc/modes.cu, rnf_rotation_modes; DESIGN 4.7).

One call finds, per image, the M best *separated* points of a log-density evaluated on a rotation set, says which of them are
local maxima and how much of the probability each one carries: greedy non-maximum suppression on SO(3), on the device.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _cabi

MAX_MODES = 256


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
    B, G = v.shape
    dev = v.device
    rot = rotations.to(dev, torch.float32).contiguous()
    lib = _cabi.load()
    out = dict(index=torch.empty((B, M), device=dev, dtype=torch.int64), value=torch.empty((B, M), device=dev, dtype=torch.float32),
               local_max=torch.empty((B, M), device=dev, dtype=torch.bool), mass=torch.empty((B, M), device=dev, dtype=torch.float32),
               count=torch.empty((B,), device=dev, dtype=torch.int32))
    if B > 0:
        nbytes = int(lib.rnf_rotation_modes_workspace_bytes(G, B, M))
        ws = torch.empty((nbytes,), device=dev, dtype=torch.uint8)

        def p(t):
            return C.c_void_p(t.data_ptr())
        with torch.cuda.device(dev):
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(lib.rnf_rotation_modes(p(v), B, G, int(g_index0), p(rot), M, theta, rho, p(ws), nbytes, p(out["index"]),
                                               p(out["value"]), p(out["local_max"]), p(out["mass"]), p(out["count"]), st))
    if squeeze:
        out = {k: t[0] for k, t in out.items()}
    return out
