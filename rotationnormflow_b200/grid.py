"""HEALPix SO(3) query grids generated on the device (utils/sd.py:11-82)."""
from __future__ import annotations

import math

import torch

from . import _cabi

GRID_SIZES = tuple(72 * 8 ** l for l in range(9))          # utils/sd.py:32
_grids: dict = {}


def closest_grid_level(num_queries: int) -> int:
    """get_closest_available_grid (utils/sd.py:31-34): the level whose size is nearest in log space."""
    best, arg = None, 0
    for l, s in enumerate(GRID_SIZES):
        d = abs(math.log(num_queries) - math.log(s))
        if best is None or d < best:
            best, arg = d, l
    return arg


def healpix_grid(level: int, begin: int = 0, end: int | None = None, device=None) -> torch.Tensor:
    """Rotations [begin,end) of the level-`level` grid as float32 [n,3,3] on `device` (rnf_healpix_grid)."""
    total = 72 * 8 ** level
    end = total if end is None else end
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("healpix_grid generates the grid on a B200; there is no CPU path")
    out = torch.empty((max(end - begin, 0), 3, 3), device=device, dtype=torch.float32)
    _cabi.launch("rnf_healpix_grid", device, int(level), int(begin), int(end), out)
    return out


def generate_healpix_grid(recursion_level=None, size=None, device=None) -> torch.Tensor:
    """Signature of utils/sd.py:48 (returns a CUDA tensor instead of a CPU one)."""
    assert not (recursion_level is None and size is None)
    if size:
        recursion_level = max(int(round(math.log(size / 72.0) / math.log(8.0))), 0)
    return healpix_grid(recursion_level, device=device)


def get_closest_available_grid(num_queries: int, device=None) -> torch.Tensor:
    level = closest_grid_level(num_queries)
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    key = (level, dev.index)
    if key not in _grids:
        _grids[key] = healpix_grid(level, device=dev)
    return _grids[key]


def generate_queries(number_queries: int, mode: str = "random", device=None) -> torch.Tensor:
    """utils/sd.py:11-25.  'random': Haar-uniform rotations from normalised Gaussian quaternions (the public
    pytorch3d.random_rotations definition); 'grid': the closest HEALPix grid."""
    if mode == "grid":
        return get_closest_available_grid(number_queries, device)
    if mode != "random":
        raise ValueError(mode)
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    q = torch.randn((number_queries, 4), device=dev)
    q = q / torch.copysign(q.norm(dim=1), q[:, 0])[:, None]
    r, i, j, k = q.unbind(-1)
    two_s = 2.0 / (q * q).sum(-1)
    m = torch.stack((1 - two_s * (j * j + k * k), two_s * (i * j - k * r), two_s * (i * k + j * r),
                     two_s * (i * j + k * r), 1 - two_s * (i * i + k * k), two_s * (j * k - i * r),
                     two_s * (i * k - j * r), two_s * (j * k + i * r), 1 - two_s * (i * i + j * j)), -1)
    return m.reshape(-1, 3, 3)


# ---- coarse-to-fine search (csrc/hgrid.cu; DESIGN 4.8) ------------------------------------------------------------------------------
MAX_TOP_K = 4096


def healpix_children(level: int, index: torch.Tensor, offset: torch.Tensor | None = None):
    """The 8 level-(level+1) children of level-``level`` grid indices ``index`` [n] (rnf_healpix_children; 0 <= level <= 7).

    For idx = t * npix + p (nside = 2^level, npix = 12 nside^2, p the RING pixel) child k = 4 dt + j is the index t' * 4 npix + p' with
    t' = 2 t + dt and p' = nest2ring(2 nside, 4 ring2nest(nside, p) + j): the children of all level-l indices partition the
    level-(l+1) grid.  Returns (child [n,8] int64, rotations [n,8,3,3] float32): ``healpix_grid(level + 1)[child]`` times ``offset``
    [3,3] by the arithmetic of ``Flow.grid_log_prob``, bit for bit the rotation the grid pass scores at that index.  A parent outside
    the level's grid (padding -1) gives children -1 and NaN rotations.  No host synchronisation."""
    level = int(level)
    if not 0 <= level <= 7:
        raise ValueError(f"level must be in 0..7 (children at levels 1..8), got {level}")
    if not index.is_cuda:
        raise RuntimeError("healpix_children runs on a B200 only: `index` must be a CUDA tensor (there is no CPU fallback)")
    idx = index.reshape(-1).to(torch.int64).contiguous()
    dev = idx.device
    n = idx.shape[0]
    child = torch.empty((n, 8), device=dev, dtype=torch.int64)
    rot = torch.empty((n, 8, 3, 3), device=dev, dtype=torch.float32)
    off = None if offset is None else offset.to(dev, torch.float32).reshape(3, 3).contiguous()
    _cabi.launch("rnf_healpix_children", dev, level, idx, n, off, child, rot)
    return child, rot


def top_k(values: torch.Tensor, index: torch.Tensor | None, k: int):
    """Per image the ``k`` best of ``values`` [B,C] (or [C]) under the order of the grid arg-max: NaN first, then the larger value,
    then the lower index; best first (rnf_topk, 1 <= k <= 4096).  ``index`` (same shape, int64) gives each entry's index, None the
    column number; an entry with a negative index is padding and ranks after every other one.  Returns (values [B,k], index [B,k]
    int64); places without a real entry (k > C, or padding) are (-inf, -1).  No host synchronisation; bitwise reproducible."""
    k = int(k)
    if not 1 <= k <= MAX_TOP_K:
        raise ValueError(f"k must be in 1..{MAX_TOP_K}, got {k}")
    if values.dim() not in (1, 2):
        raise ValueError(f"values must be [B,C] or [C], got {tuple(values.shape)}")
    if index is not None and tuple(index.shape) != tuple(values.shape):
        raise ValueError(f"index must have the shape of values {tuple(values.shape)}, got {tuple(index.shape)}")
    if not values.is_cuda:
        raise RuntimeError("top_k runs on a B200 only: `values` must be a CUDA tensor (there is no CPU fallback)")
    squeeze = values.dim() == 1
    v = (values[None] if squeeze else values).to(torch.float32).contiguous()
    B, Cn = v.shape
    dev = v.device
    ix = None if index is None else (index[None] if squeeze else index).to(dev, torch.int64).contiguous()
    out_v = torch.empty((B, k), device=dev, dtype=torch.float32)
    out_i = torch.empty((B, k), device=dev, dtype=torch.int64)
    if B > 0:
        nbytes = int(_cabi.load().rnf_topk_workspace_bytes(B, Cn, k))
        ws = torch.empty((max(nbytes, 1),), device=dev, dtype=torch.uint8)
        _cabi.launch("rnf_topk", dev, v, ix, B, Cn, k, ws, nbytes, out_v, out_i)
    if squeeze:
        return out_v[0], out_i[0]
    return out_v, out_i
