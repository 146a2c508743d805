"""Coarse-to-fine search on the HEALPix grids (grid.healpix_children / rnf_healpix_children, grid.top_k / rnf_topk,
evalpath.estimate_rotation_hierarchical; DESIGN 4.8).

CPU: an integer restatement of RING <-> NESTED and of the children map (the partition of each finer grid, each child within the
parent's cell), a numpy restatement of the top-K order (NaN first, then the larger value, then the lower index; negative indices are
padding), and the argument errors of the C ABI and of the Python entry point.
GPU: the kernels bit for bit against the restatements and against healpix_grid; candidate log p from Flow.forward against
Flow.grid_log_prob at the same index; the exhaustive search against the full grid; a unimodal density; the invariants of the search
on a seeded flow and a sharpened stress model; determinism, no host synchronisation, CUDA-graph replay."""
import ctypes
import functools
import math

import numpy as np
import pytest
import torch

from conftest import golden, record_error, seeded_product_flow
from oracle import rnf_oracle as orc
import rotationnormflow_b200 as rnf
from rotationnormflow_b200 import _cabi, evalpath
from rotationnormflow_b200 import grid as rgrid

RNF_EINVAL = -1
# Flow.forward (rows) and Flow.grid_log_prob (grid) score the same rotation with the same weights, but not bit for bit: the two
# launch shapes of the forward kernel round the per-image conditioner term differently.  Candidate log p is held to
# |a - b| <= LOGP_TOL * max(1, |b|), several times the largest difference measured on a B200 (profiles/r10_hier_error_table.json),
# and the exact properties of the search (never above the full maximum, exhaustive = full arg-max) hold within it.
LOGP_TOL = 2e-4


def _close(a, b):
    return ((a - b).abs() <= LOGP_TOL * b.abs().clamp(min=1.0)).all().item()


# ---- integer restatement of the HEALPix pixel orderings (public HEALPix ring2xyf / xyf2nest / nest2xyf / xyf2ring) -------------------
JRLL = np.array([2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4], np.int64)
JPLL = np.array([1, 3, 5, 7, 0, 2, 4, 6, 1, 3, 5, 7], np.int64)


def _isqrt(v):
    r = np.floor(np.sqrt(v.astype(np.float64))).astype(np.int64)
    r = np.where(r * r > v, r - 1, r)
    return np.where((r + 1) * (r + 1) <= v, r + 1, r)


def _spread(v):
    out = np.zeros_like(v)
    for b in range(30):
        out |= ((v >> b) & 1) << (2 * b)
    return out


def _compress(v):
    out = np.zeros_like(v)
    for b in range(30):
        out |= ((v >> (2 * b)) & 1) << b
    return out


def ring2nest(nside, pix):
    pix = np.asarray(pix, np.int64)
    nl2, ncap, npix = 2 * nside, 2 * nside * (nside - 1), 12 * nside * nside
    iring, iphi, kshift, nr, face = (np.zeros_like(pix) for _ in range(5))
    north, south = pix < ncap, pix >= npix - ncap
    belt = ~north & ~south
    p = pix[north]
    i = (1 + _isqrt(1 + 2 * p)) >> 1
    iring[north], iphi[north], nr[north] = i, p + 1 - 2 * i * (i - 1), i
    face[north] = (iphi[north] - 1) // i
    ip = pix[belt] - ncap
    tmp = ip // (4 * nside)
    iring[belt] = tmp + nside
    iphi[belt] = ip - tmp * 4 * nside + 1
    kshift[belt] = (iring[belt] + nside) & 1
    nr[belt] = nside
    ire, irm = tmp + 1, nl2 + 2 - (tmp + 1)
    ifm = (iphi[belt] - (ire >> 1) + nside - 1) // nside
    ifp = (iphi[belt] - (irm >> 1) + nside - 1) // nside
    face[belt] = np.where(ifp == ifm, ifp | 4, np.where(ifp < ifm, ifp, ifm + 8))
    ip = npix - pix[south]
    i = (1 + _isqrt(2 * ip - 1)) >> 1
    iphi[south] = 4 * i + 1 - (ip - 2 * i * (i - 1))
    nr[south] = i
    iring[south] = 2 * nl2 - i
    face[south] = 8 + (iphi[south] - 1) // i
    irt = iring - JRLL[face] * nside + 1
    ipt = 2 * iphi - JPLL[face] * nr - kshift - 1
    ipt = np.where(ipt >= nl2, ipt - 8 * nside, ipt)
    ix, iy = (ipt - irt) >> 1, (-ipt - irt) >> 1
    return face * nside * nside + _spread(ix) + (_spread(iy) << 1)


def nest2ring(nside, pix):
    pix = np.asarray(pix, np.int64)
    npface = nside * nside
    npix, ncap, nl4 = 12 * npface, 2 * nside * (nside - 1), 4 * nside
    face, sub = pix // npface, pix % npface
    ix, iy = _compress(sub), _compress(sub >> 1)
    jr = JRLL[face] * nside - ix - iy - 1
    nr = np.where(jr < nside, jr, np.where(jr > 3 * nside, nl4 - jr, nside))
    n_before = np.where(jr < nside, 2 * nr * (nr - 1), np.where(jr > 3 * nside, npix - 2 * (nr + 1) * nr, ncap + (jr - nside) * nl4))
    kshift = np.where((jr < nside) | (jr > 3 * nside), 0, (jr - nside) & 1)
    jp = (JPLL[face] * nr + ix - iy + 1 + kshift) // 2
    jp = np.where(jp > nl4, jp - nl4, np.where(jp < 1, jp + nl4, jp))
    return n_before + jp - 1


def children(level, idx):
    """[n] level-`level` indices -> [n,8] level-(level+1) indices, child k = 4 dt + j (padding -1 for indices outside the grid)."""
    idx = np.asarray(idx, np.int64)
    nside = 2 ** level
    npix = 12 * nside * nside
    ok = (idx >= 0) & (idx < 72 * 8 ** level)
    safe = np.where(ok, idx, 0)
    t, p = safe // npix, safe % npix
    nest = ring2nest(nside, p)
    out = np.empty((idx.shape[0], 8), np.int64)
    for k in range(8):
        pc = nest2ring(2 * nside, 4 * nest + (k & 3))
        out[:, k] = (2 * t + (k >> 2)) * 4 * npix + pc
    return np.where(ok[:, None], out, -1)


def _angles(A, B):
    """Geodesic angles between fp64 rotation stacks A, B [n,3,3]."""
    tr = np.einsum("nij,nij->n", np.asarray(A, np.float64), np.asarray(B, np.float64))
    return np.arccos(np.clip((tr - 1) / 2, -1, 1))


# ---- top-K restatement ----------------------------------------------------------------------------------------------------------------
def _before(a, b):
    """a = (value, index) ranks before b: padding (index < 0) never; NaN first; then the larger value; then the lower index."""
    (av, ai), (bv, bi) = a, b
    if ai < 0:
        return False
    if bi < 0:
        return True
    an, bn = math.isnan(av), math.isnan(bv)
    if an or bn:
        return an and (not bn or ai < bi)
    return av > bv or (av == bv and ai < bi)


def ref_topk(values, index, k):
    """values [B,C] float32, index [B,C] int64 or None (column numbers) -> (values [B,k], index [B,k]) with (-inf, -1) padding."""
    v = np.atleast_2d(np.asarray(values, np.float32))
    B, C = v.shape
    ix = np.broadcast_to(np.arange(C, dtype=np.int64), (B, C)) if index is None else np.atleast_2d(np.asarray(index, np.int64))
    ov, oi = np.full((B, k), -np.inf, np.float32), np.full((B, k), -1, np.int64)
    cmp = functools.cmp_to_key(lambda a, b: -1 if _before(a, b) else (1 if _before(b, a) else 0))
    for b in range(B):
        vals = v[b]
        real = ix[b] >= 0
        # vectorised order of the real entries: NaN first (by index), then value descending, then index ascending
        nan = np.isnan(vals) & real
        fin = ~np.isnan(vals) & real
        o_nan = np.nonzero(nan)[0][np.argsort(ix[b][nan], kind="stable")]
        f = np.nonzero(fin)[0]
        o_fin = f[np.lexsort((ix[b][f], -vals[f].astype(np.float64)))]
        order = np.concatenate([o_nan, o_fin])[:k]
        if C <= 64:            # small rows: the comparator itself, as a check of the vectorised order
            ents = sorted([(float(vals[c]), int(ix[b][c])) for c in range(C)], key=cmp)
            ents = [e for e in ents if e[1] >= 0][:k]
            assert [e[1] for e in ents] == ix[b][order].tolist()
        ov[b, :order.size], oi[b, :order.size] = vals[order], ix[b][order]
    return ov, oi


# ============================================================ CPU ===============================================================
@pytest.mark.parametrize("level", range(6))
def test_ring_nest_are_inverse_permutations(level):
    nside = 2 ** level
    p = np.arange(12 * nside * nside)
    n = ring2nest(nside, p)
    assert np.array_equal(np.sort(n), p)
    assert np.array_equal(nest2ring(nside, n), p)


def test_ring_nest_known_values():
    # nside = 1: both orders number the 12 base pixels alike
    assert np.array_equal(ring2nest(1, np.arange(12)), np.arange(12))
    # nside = 2, RING pixel 0 is the north-most pixel of base pixel 0: its NESTED number is the last sub-pixel (3) of face 0
    assert ring2nest(2, np.array([0]))[0] == 3
    # and the south-most RING pixel is the first sub-pixel of face 11
    assert ring2nest(2, np.array([47]))[0] == 44


@pytest.mark.parametrize("level", range(4))
def test_children_partition_the_next_level(level):
    ch = children(level, np.arange(72 * 8 ** level))
    flat = np.sort(ch.ravel())
    assert np.array_equal(flat, np.arange(72 * 8 ** (level + 1)))


def test_children_of_padding_are_padding():
    ch = children(1, np.array([-1, 72 * 8, 5]))
    assert (ch[:2] == -1).all() and (ch[2] >= 0).all()


# The grid rotation is R = Rx(az) Rz(polar) Rx(tilt): its first column R e_x is the HEALPix pixel centre (the tilt turns about x), and
# the tilt index of a child is 2t or 2t + 1.  The cell of a parent is its pixel times its tilt step, so a child lies in it when its
# pixel centre is within the pixel radius of the parent's (measured: 0.423, 0.458, 0.487, 0.497 of the largest nearest-neighbour
# spacing of the level's pixel centres, levels 0-3).  In the SO(3) metric a child of a polar-cap pixel can be far from its parent
# (up to 0.46 rad at every level): at polar -> 0 the azimuth turns about the same axis as the tilt, so pixel centres that are close
# on the sphere carry rotations that differ by their azimuth (DESIGN 4.8, limits).
@pytest.mark.parametrize("level", range(4))
def test_children_lie_within_the_parent_cell(level):
    G, npix = 72 * 8 ** level, 12 * 4 ** level
    parent = orc.healpix_grid(level).double().numpy()
    child = orc.healpix_grid(level + 1).double().numpy()
    pts = parent[:npix, :, 0]
    d = np.arccos(np.clip(pts @ pts.T, -1, 1))
    np.fill_diagonal(d, np.inf)
    radius = 0.5 * d.min(1).max()
    ch = children(level, np.arange(G))
    ang = np.arccos(np.clip((np.repeat(parent[:, :, 0], 8, 0) * child[ch.ravel()][:, :, 0]).sum(1), -1, 1))
    record_error(test="children_cell_radius", level=level, max_pixel_angle=float(ang.max()), radius=float(radius))
    assert ang.max() <= radius
    t = np.arange(G) // npix
    assert np.array_equal(ch // (4 * npix), np.stack([2 * t] * 4 + [2 * t + 1] * 4, 1))
    # the map without the NESTED subdivision (RING pixel 4p + j) leaves the cell
    wrong = 4 * (np.arange(G) % npix)[:, None] + np.arange(4)
    ang_w = np.arccos(np.clip((np.repeat(parent[:, :, 0], 4, 0) * child[wrong.ravel()][:, :, 0]).sum(1), -1, 1))
    assert ang_w.max() > radius


def test_topk_restatement_order():
    nan, inf = float("nan"), float("inf")
    v = np.array([[1.0, 3.0, 3.0, nan, -inf, 2.0, nan, -inf]], np.float32)
    i = np.array([[7, 5, 2, 9, 0, -1, 4, 3]], np.int64)
    ov, oi = ref_topk(v, i, 10)
    assert oi[0].tolist() == [4, 9, 2, 5, 7, 0, 3, -1, -1, -1]           # NaN by index, 3 by index, 1, -inf by index; -1 is padding
    assert np.isnan(ov[0, :2]).all() and ov[0, 2:7].tolist() == [3.0, 3.0, 1.0, -inf, -inf] and (ov[0, 7:] == -inf).all()
    ov, oi = ref_topk(np.array([[0.5, 0.5, 0.5]], np.float32), None, 2)
    assert oi[0].tolist() == [0, 1]
    ov, oi = ref_topk(np.zeros((2, 0), np.float32), None, 3)
    assert (oi == -1).all() and (ov == -np.inf).all()


def test_cabi_argument_errors_without_gpu():
    lib = _cabi.load()
    buf = (ctypes.c_char * 4096)()
    P = ctypes.cast(buf, ctypes.c_void_p)
    for lvl in (-1, 8):
        assert lib.rnf_healpix_children(lvl, P, 1, None, P, P, None) == RNF_EINVAL and b"child level" in lib.rnf_last_error()
    assert lib.rnf_healpix_children(2, P, -1, None, P, P, None) == RNF_EINVAL
    assert lib.rnf_healpix_children(2, None, 1, None, P, P, None) == RNF_EINVAL
    assert lib.rnf_healpix_children(2, P, 1, None, None, P, None) == RNF_EINVAL
    assert lib.rnf_healpix_children(2, P, 1, None, P, None, None) == RNF_EINVAL
    assert lib.rnf_healpix_children(0, None, 0, None, None, None, None) == 0          # n = 0 does nothing
    assert lib.rnf_healpix_children(7, None, 0, None, None, None, None) == 0
    for K in (0, 4097, -3):
        assert lib.rnf_topk(P, None, 1, 10, K, P, 1 << 20, P, P, None) == RNF_EINVAL and b"K=" in lib.rnf_last_error()
    assert lib.rnf_topk(P, None, -1, 10, 4, P, 1 << 20, P, P, None) == RNF_EINVAL
    assert lib.rnf_topk(None, None, 1, 10, 4, P, 1 << 20, P, P, None) == RNF_EINVAL
    assert lib.rnf_topk(P, None, 1, 10, 4, P, 1 << 20, None, P, None) == RNF_EINVAL
    assert lib.rnf_topk(P, None, 1, 10, 4, P, 1 << 20, P, None, None) == RNF_EINVAL
    assert lib.rnf_topk(P, None, 2, 100000, 4, None, 0, P, P, None) == RNF_EINVAL       # needs a workspace
    assert lib.rnf_topk(P, None, 2, 100000, 4, P, 16, P, P, None) == RNF_EINVAL         # too small
    assert lib.rnf_topk(None, None, 0, 10, 4, None, 0, None, None, None) == 0           # B = 0 does nothing
    assert lib.rnf_topk(P, None, 1, 65536 * 4096, 4, P, 1 << 20, P, P, None) == RNF_EINVAL
    # workspace sizes: one slice needs none; otherwise B * S * Kp (4-byte values, 256-aligned, then 8-byte indices)
    assert lib.rnf_topk_workspace_bytes(3, 4096, 64) == 0
    assert lib.rnf_topk_workspace_bytes(3, 4097, 64) == 3 * 2 * 64 * 12
    assert lib.rnf_topk_workspace_bytes(1, 72 * 8 ** 5, 4096) == 288 * 4096 * 12
    assert lib.rnf_topk_workspace_bytes(1, 10, 0) == 0 and lib.rnf_topk_workspace_bytes(0, 10, 4) == 0


@pytest.mark.parametrize("kw", [dict(beam=0), dict(beam=4097), dict(beam=2.5), dict(beam=True), dict(start_level=-1), dict(start_level=9),
                                dict(start_level=1.5)])
def test_hierarchical_argument_errors(kw):
    with pytest.raises(ValueError):
        evalpath.estimate_rotation_hierarchical(None, None, 72 * 8 ** 3, **kw)


def test_python_argument_errors():
    with pytest.raises(ValueError):
        rgrid.healpix_children(8, torch.zeros(1, dtype=torch.int64))
    with pytest.raises(ValueError):
        rgrid.top_k(torch.zeros(2, 3), None, 0)
    with pytest.raises(ValueError):
        rgrid.top_k(torch.zeros(2, 3), torch.zeros(3, dtype=torch.int64), 1)


# ============================================================ GPU ===============================================================
def _fmaf(a, b, c):
    """float32 fmaf(a, b, c) = round(a * b + c) once: the product is exact in float64, the sum's rounding error comes from TwoSum, and a
    float64 sum that lands exactly between two float32 values is resolved by the sign of that error."""
    a, b, c = (np.asarray(x, np.float32).astype(np.float64) for x in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    e = (p - (s - bb)) + (c - bb)
    r = s.astype(np.float32)
    up = np.nextafter(r, np.float32(np.inf))
    dn = np.nextafter(r, np.float32(-np.inf))
    other = np.where(s > r.astype(np.float64), up, dn)
    tie = (s == (r.astype(np.float64) + other.astype(np.float64)) / 2) & (e != 0)
    pick = np.where(e > 0, np.maximum(r, other), np.minimum(r, other))
    return np.where(tie, pick, r)


def offset_product(G, O):
    """grid @ offset by the fmaf chain of the grid kernels (flow_t4.cu), in float32: [n,3,3] x [3,3]."""
    G = np.asarray(G, np.float32)
    O = np.asarray(O, np.float32)
    out = np.empty_like(G)
    for i in range(3):
        for j in range(3):
            x = (G[:, i, 0].astype(np.float64) * O[0, j]).astype(np.float32)
            out[:, i, j] = _fmaf(G[:, i, 2], O[2, j], _fmaf(G[:, i, 1], O[1, j], x))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("level", range(4))
def test_children_kernel_matches_grid_bit_for_bit(level):
    G = 72 * 8 ** level
    parents = np.concatenate([np.arange(G), [-1, G, -5]])
    ch, rot = rgrid.healpix_children(level, torch.from_numpy(parents).cuda())
    ref = children(level, parents)
    assert np.array_equal(ch.cpu().numpy(), ref)
    fine = rgrid.healpix_grid(level + 1)
    real = ch[:G].reshape(-1)
    assert torch.equal(rot[:G].reshape(-1, 3, 3), fine[real])
    assert torch.isnan(rot[G:]).all() and (ch[G:] == -1).all()
    off = orc.random_rotations(1, torch.Generator().manual_seed(level))[0]
    ch2, rot2 = rgrid.healpix_children(level, torch.from_numpy(parents).cuda(), off.cuda())
    assert torch.equal(ch2, ch)
    want = offset_product(fine[real].cpu().numpy(), off.numpy())
    assert np.array_equal(rot2[:G].reshape(-1, 3, 3).cpu().numpy(), want)
    assert torch.isnan(rot2[G:]).all()


@pytest.mark.gpu
def test_children_kernel_empty_and_levels_5_to_8():
    ch, rot = rgrid.healpix_children(3, torch.empty(0, dtype=torch.int64, device="cuda"))
    assert ch.shape == (0, 8) and rot.shape == (0, 8, 3, 3)
    gen = np.random.default_rng(3)
    for level in range(4, 8):
        G = 72 * 8 ** level
        parents = np.concatenate([gen.integers(0, G, 512), [0, G - 1]])
        ch, rot = rgrid.healpix_children(level, torch.from_numpy(parents).cuda())
        assert np.array_equal(ch.cpu().numpy(), children(level, parents))
        for c, r in zip(ch.reshape(-1)[::97].tolist(), rot.reshape(-1, 3, 3)[::97]):
            assert torch.equal(rgrid.healpix_grid(level + 1, c, c + 1)[0], r)


def _check_topk(v, ix, k):
    vd = torch.from_numpy(v).cuda()
    idd = None if ix is None else torch.from_numpy(ix).cuda()
    ov, oi = rgrid.top_k(vd, idd, k)
    rv, ri = ref_topk(v, ix, k)
    assert np.array_equal(oi.cpu().numpy(), ri)
    assert np.array_equal(ov.cpu().numpy(), rv, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("C,k", [(1, 1), (10, 3), (72, 576), (4096, 64), (4097, 64), (4608, 1), (4608, 100), (36864, 16), (36864, 576),
                                 (36864, 4096), (300000, 4096), (9000, 2049)])
def test_topk_matches_restatement(C, k):
    gen = np.random.default_rng(C + k)
    B = 3
    v = np.round(gen.standard_normal((B, C)) * 4).astype(np.float32)          # few distinct values: many ties
    v[gen.random((B, C)) < 0.01] = np.nan
    v[gen.random((B, C)) < 0.02] = -np.inf
    v[gen.random((B, C)) < 0.01] = np.inf
    _check_topk(v, None, k)
    ix = np.stack([gen.permutation(10 * C)[:C] for _ in range(B)]).astype(np.int64)
    ix[gen.random((B, C)) < 0.05] = -1                                         # padding entries
    _check_topk(v, ix, k)


@pytest.mark.gpu
def test_topk_shapes_and_coarse_pass_sizes():
    # B = 0, C = 0, K > C
    ov, oi = rgrid.top_k(torch.empty(0, 50, device="cuda"), None, 8)
    assert ov.shape == (0, 8) and oi.shape == (0, 8)
    ov, oi = rgrid.top_k(torch.empty(2, 0, device="cuda"), None, 8)
    assert (oi == -1).all() and (ov == -math.inf).all()
    _check_topk(np.array([[1.0, np.nan, 2.0]], np.float32), None, 4096)
    ov, oi = rgrid.top_k(torch.tensor([3.0, 1.0, 2.0], device="cuda"), None, 2)
    assert oi.tolist() == [0, 2] and ov.tolist() == [3.0, 2.0]
    # the level-5 coarse pass: 2.36 M entries per image
    gen = np.random.default_rng(11)
    C = 72 * 8 ** 5
    v = (gen.standard_normal((2, C)) * 8).astype(np.float16).astype(np.float32)   # fp16-rounded: ties
    v[0, gen.integers(0, C, 5)] = np.nan
    for k in (1, 64, 576, 4096):
        _check_topk(v, None, k)
    # nested: the top-k of one row is a prefix of its top-k' for k < k'
    vd = torch.from_numpy(v).cuda()
    a, b = rgrid.top_k(vd, None, 100), rgrid.top_k(vd, None, 1000)
    assert torch.equal(a[1], b[1][:, :100])


# ---- flows -------------------------------------------------------------------------------------------------------------------------
def _golden_flow(tag):
    g = golden(tag)
    m = seeded_product_flow(g.cfg, g.seed)
    m.load_state_dict(g.state_dict())
    feat = g.feat.cuda() if g.feat is not None else None
    A = torch.from_numpy(g.z["fisher_A"]).cuda() if "fisher_A" in g.z.files else None
    return m.cuda().eval(), feat, A


def _symsol_flow():
    cfg = rnf.load_config("symsol")
    m = seeded_product_flow(cfg, 4).cuda().eval()
    feat = torch.relu(torch.randn(4, m.feature_dim, generator=torch.Generator().manual_seed(6))).cuda()
    return m, feat


def _offset(seed):
    return orc.random_rotations(1, torch.Generator().manual_seed(seed))[0].cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["symsol", "s_modelnet_fisher", "modelnet_fisher"])
def test_forward_scores_equal_grid_log_prob(case):
    """Candidate log p through Flow.forward (+ the Fisher term) against Flow.grid_log_prob at the same level-(l+1) index."""
    if case == "symsol":
        m, feat = _symsol_flow()
        A = None
    elif case == "s_modelnet_fisher":
        m, feat, A = _golden_flow("s_modelnet")
    else:
        m, feat, _ = _golden_flow("modelnet")
        A = (4.0 * orc.random_rotations(feat.shape[0], torch.Generator().manual_seed(5))).cuda()
    B, off = feat.shape[0], _offset(1)
    for level in (2, 3):
        full = m.grid_log_prob(rgrid.healpix_grid(level + 1), feat, offset=off, fisher_A=A, return_logp=True)["logp"]
        coarse = m.grid_log_prob(rgrid.healpix_grid(level), feat, offset=off, fisher_A=A, return_logp=True)["logp"]
        _, top = rgrid.top_k(coarse, None, 64)
        ch, rot = rgrid.healpix_children(level, top.reshape(-1), off)
        with torch.no_grad():
            lp = evalpath._score_rows(m, rot.reshape(-1, 3, 3), feat, 8 * 64, A, None)
        want = torch.gather(full, 1, ch.reshape(B, -1))
        diff = (lp - want).abs().max().item()
        rel = ((lp - want).abs() / want.abs().clamp(min=1.0)).max().item()
        record_error(test="forward_vs_grid_log_prob", case=case, level=level + 1, max_abs_diff=diff, max_rel_diff=rel,
                     bitwise=bool(torch.equal(lp, want)), tol=LOGP_TOL)
        assert _close(lp, want), (diff, rel)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["s_symsol", "s_modelnet", "s_smith9c", "s_uncond"])
def test_exhaustive_search_equals_full_grid(tag):
    m, feat, A = _golden_flow(tag)
    off = _offset(2)
    Q = 72 * 8 ** 2
    est, out = evalpath.estimate_rotation_hierarchical(m, feat, Q, start_level=0, beam=576, fisher_A=A, offset=off)
    full = m.grid_log_prob(rgrid.healpix_grid(2), feat, offset=off, fisher_A=A, return_logp=True)
    assert out["level"] == 2 and out["evaluated"] == 72 + 576 + 8 * 576
    # every level-2 rotation was scored: the final beam is the full grid's top 576 up to the scoring difference
    lp = full["logp"]
    assert _close(out["logp"], full["max"]) and _close(out["top_logp"], torch.gather(lp, 1, out["top_index"]))
    top = out["top_index"].sort(1).values
    assert (top >= 0).all() and (top < 4608).all() and (top[:, 1:] > top[:, :-1]).all()
    at_best = torch.gather(lp, 1, out["index"][:, None])[:, 0]
    assert torch.equal(out["index"], full["argmax"]) or _close(at_best, full["max"])
    record_error(test="exhaustive", case=tag, argmax_equal=bool(torch.equal(out["index"], full["argmax"])),
                 logp_bitwise=bool(torch.equal(out["logp"], full["max"])), max_abs_diff=(out["logp"] - full["max"]).abs().max().item())
    # (a) the estimate is the grid rotation at the reported index, times the offset (fmaf chain)
    want = offset_product(rgrid.healpix_grid(2)[out["index"]].cpu().numpy(), off.cpu().numpy())
    assert np.array_equal(est.cpu().numpy(), want)


def test_layerwise_flow_needs_levels_of_at_least_one():
    """A flow Flow.grid_log_prob refuses (ConditionLU here) scores its coarse level as children of the level below: start_level 0 or
    a level-0 final grid is refused with a ValueError before anything runs (no GPU needed)."""
    g = golden("s_clu")
    m = seeded_product_flow(g.cfg, g.seed)
    for q, l0 in ((72 * 8 ** 2, 0), (72, 0), (72, 3)):
        with pytest.raises(ValueError, match="start_level >= 1 and a final level >= 1"):
            evalpath.estimate_rotation_hierarchical(m, None, q, start_level=l0, beam=4)


@pytest.mark.gpu
def test_exhaustive_search_on_a_conditionlu_flow(monkeypatch):
    """s_clu (ConditionLU: Flow.grid_log_prob refuses it; Flow.forward runs the per-layer operators).  Levels 1 -> 2 with beam 576 score
    every level-2 rotation; the reference is Flow.forward on the full level-2 grid, one image per call (the reference's convention for
    this batch-coupled layer).  The piece size of the per-image scoring does not change the result."""
    m, feat, _ = _golden_flow("s_clu")
    off = _offset(12)
    B = feat.shape[0]
    ch, rot = rgrid.healpix_children(1, torch.arange(576, device="cuda"), off)
    full = torch.empty(B, 4608, device="cuda")
    with torch.no_grad():
        for b in range(B):
            _, ldj = m(rot.reshape(-1, 3, 3), feat[b:b + 1], feature_index=torch.zeros(4608, dtype=torch.int32, device="cuda"))
            full[b, ch.reshape(-1)] = ldj
    mx, am = full.max(1)
    est, out = evalpath.estimate_rotation_hierarchical(m, feat, 72 * 8 ** 2, start_level=1, beam=576, offset=off)
    assert out["level"] == 2 and out["evaluated"] == 576 + 8 * 576
    assert _close(out["logp"], mx) and _close(out["top_logp"], torch.gather(full, 1, out["top_index"]))
    assert torch.equal(out["index"], am) or _close(torch.gather(full, 1, out["index"][:, None])[:, 0], mx)
    record_error(test="exhaustive", case="s_clu", argmax_equal=bool(torch.equal(out["index"], am)),
                 max_abs_diff=(out["logp"] - mx).abs().max().item())
    monkeypatch.setattr(evalpath, "HIER_LAYERWISE_BYTES", 1000 * 4 * (m.feature_dim + 19 + 4 * 64 + 128))   # 1000-row pieces
    est2, out2 = evalpath.estimate_rotation_hierarchical(m, feat, 72 * 8 ** 2, start_level=1, beam=576, offset=off)
    assert _close(out2["top_logp"], out["top_logp"])


@pytest.mark.gpu
def test_unimodal_fisher_density_is_found_from_level_2():
    """dist=noflow: one unconditional affine layer, so log p is the (concentrated) matrix-Fisher term plus a slowly varying affine
    log-det: one peak.  Levels 2 -> 5 with beam 16 find the full level-5 arg-max."""
    cfg = orc.simple_config(layers=1, dist="noflow")
    m = seeded_product_flow(cfg, 3).cuda().eval()
    grid5 = rgrid.healpix_grid(5)
    for s in range(6):
        A = (40.0 * orc.random_rotations(1, torch.Generator().manual_seed(100 + s))).cuda()
        off = _offset(200 + s)
        full = m.grid_log_prob(grid5, None, offset=off, fisher_A=A)
        est, out = evalpath.estimate_rotation_hierarchical(m, None, 72 * 8 ** 5, start_level=2, beam=16, fisher_A=A, offset=off)
        assert out["level"] == 5 and out["evaluated"] == 72 * 64 + 3 * 128
        assert torch.equal(out["index"], full["argmax"]) and _close(out["logp"], full["max"])


def _sharp12_flow():
    from test_weight_scales import sharp
    g = golden("s_symsol")
    m = seeded_product_flow(g.cfg, g.seed)
    m.load_state_dict(sharp(g.cfg, g.state_dict(), 12.0))
    return m.cuda().eval(), g.feat.cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["symsol", "sharp12"])
def test_search_invariants(case):
    """(b) never above the full level-5 maximum; the reported log p is the full grid's at the reported index; the agreement with the
    full arg-max and the beam monotonicity are recorded (not pass thresholds: a beam can drop the branch a narrower beam follows)."""
    m, feat = _symsol_flow() if case == "symsol" else _sharp12_flow()
    off = _offset(7)
    with torch.no_grad():
        full = m.grid_log_prob(rgrid.healpix_grid(5), feat, offset=off, return_logp=True)
    prev = None
    for beam in (1, 4, 16, 64, 256):
        est, out = evalpath.estimate_rotation_hierarchical(m, feat, 72 * 8 ** 5, start_level=3, beam=beam, offset=off)
        assert (out["logp"] <= full["max"] + LOGP_TOL * full["max"].abs().clamp(min=1.0)).all()
        assert _close(out["top_logp"], torch.gather(full["logp"], 1, out["top_index"]))
        assert (out["top_logp"][:, :-1] >= out["top_logp"][:, 1:]).all()
        agree = (out["index"] == full["argmax"]).float().mean().item()
        gap = (full["max"] - out["logp"]).max().item()
        mono = None if prev is None else bool((out["logp"] >= prev).all())
        record_error(test="search_invariants", case=case, beam=beam, agreement_with_full_argmax=agree, max_logp_gap=gap,
                     non_decreasing_from_previous_beam=mono)
        prev = out["logp"]


@pytest.mark.gpu
def test_start_level_at_or_above_final_is_the_grid_argmax():
    m, feat = _symsol_flow()
    off = _offset(8)
    est, out = evalpath.estimate_rotation_hierarchical(m, feat, 72 * 8 ** 3, start_level=5, beam=8, offset=off)
    e2, o2 = evalpath.estimate_rotation_grid(m, feat, 72 * 8 ** 3, offset=off)
    assert out["level"] == 3 and out["evaluated"] == 72 * 8 ** 3
    assert torch.equal(out["index"], o2["argmax"]) and torch.equal(out["logp"], o2["max"]) and torch.equal(est, e2)


@pytest.mark.gpu
def test_search_chunks_images(monkeypatch):
    m, feat = _symsol_flow()
    off = _offset(9)
    a = evalpath.estimate_rotation_hierarchical(m, feat, 72 * 8 ** 4, start_level=2, beam=32, offset=off)
    monkeypatch.setattr(evalpath, "MODES_LOGP_BYTES", 4608 * 4 * 3)          # three images per chunk
    b = evalpath.estimate_rotation_hierarchical(m, feat, 72 * 8 ** 4, start_level=2, beam=32, offset=off)
    assert torch.equal(a[0], b[0])
    for k in ("logp", "index", "top_logp", "top_index"):
        assert torch.equal(a[1][k], b[1][k]), k


@pytest.mark.gpu
def test_deterministic_without_sync_and_graph_capturable():
    m, feat = _symsol_flow()
    off = _offset(10)
    args = (m, feat, 72 * 8 ** 5)
    kw = dict(start_level=3, beam=64, offset=off)
    a = evalpath.estimate_rotation_hierarchical(*args, **kw)
    torch.cuda.set_sync_debug_mode("error")
    try:
        b = evalpath.estimate_rotation_hierarchical(*args, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.equal(a[0], b[0])
    for k in ("logp", "index", "top_logp", "top_index"):
        assert torch.equal(a[1][k], b[1][k]), k
    # one expand / score / select level in a CUDA graph
    top = a[1]["top_index"].clone()

    @torch.no_grad()
    def level():
        ch, rot = rgrid.healpix_children(5, top.reshape(-1), off)
        lp = evalpath._score_rows(m, rot.reshape(-1, 3, 3), feat, 8 * 64, None, None)
        return rgrid.top_k(lp, ch.reshape(feat.shape[0], -1), 64)
    ref = level()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        level()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = level()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[0], ref[0]) and torch.equal(out[1], ref[1])
