"""Separated modes over a grid split across ranks (modes.RankModes / rotation_modes_rank, rnf_rotation_modes_shard_*,
dist.sharded_rotation_modes, dist.sharded_estimate_rotation_modes; DESIGN 4.7 "Sharded").

The claim under test: every rank returns what ``modes.rotation_modes`` returns on the concatenated grid, with index, value,
local_max, count and valid bit for bit and mass within 1e-5 relative.  On the CPU, an fp64 restatement of the sharded algorithm
(per-rank proposals merged in the record order) against ``ref_modes`` of tests/test_modes.py, and the ABI's argument errors.  On one
GPU, W simulated ranks in one process (``torch.stack`` as the gather) against ``rotation_modes``; on two or more GPUs, NCCL ranks
against the single-GPU ``evalpath.estimate_rotation_modes``."""
import math
import os
import socket
import threading

import numpy as np
import pytest
import torch

from oracle import rnf_oracle as orc
from rotationnormflow_b200 import _cabi, evalpath
from rotationnormflow_b200 import dist as rdist
from rotationnormflow_b200 import grid as rgrid
from rotationnormflow_b200.modes import RECORD_BYTES, RankModes, rotation_modes, rotation_modes_rank
from test_modes import quaternions, ref_modes, symmetric_case

RNF_EINVAL = -1


# ---- CPU: the sharded algorithm restated in fp64, against the single-grid definition ------------------------------------------------
def record_better(ov, oi, bv, bi):
    """The order of the record merge (grid_red_better): NaN first, then the larger value, then the lower global index."""
    on, bn = math.isnan(ov), math.isnan(bv)
    return (not bn or oi < bi) if on else (not bn and (ov > bv or (ov == bv and oi < bi)))


def merge_records(recs):
    """recs: per rank, in rank order, (best_v, best_i, mass, total, disq) with best_i None for "no point".  Returns the merged
    (best_v, best_i, mass, total, disq): the best proposal in the record order, sums in rank order, OR of the flags."""
    bv, bi, mass, total, disq = -math.inf, None, 0.0, 0.0, False
    for v, i, m, t, d in recs:
        if i is not None and (bi is None or record_better(v, i, bv, bi)):
            bv, bi = v, i
        mass, total, disq = mass + m, total + t, disq or d
    return bv, bi, mass, total, disq


def sharded_ref(values, R, M, theta, rho, bounds):
    """The sharded rounds in fp64 torch: per rank, the slice's labels, partial sums and best unlabelled point; per round one merge of
    the rank records.  bounds: [0 = b_0 <= b_1 <= ... <= b_W = G] (empty slices allowed)."""
    v_all = torch.from_numpy(np.atleast_2d(np.asarray(values, np.float32)).astype(np.float64))
    B, G = v_all.shape
    q = torch.from_numpy(quaternions(R)) if G else torch.zeros(0, 4, dtype=torch.float64)
    cs, cn = math.cos(theta / 2), math.cos(rho / 2)
    out = dict(index=np.full((B, M), -1, np.int64), local_max=np.zeros((B, M), bool), mass=np.zeros((B, M)), count=np.zeros(B, np.int64))
    shards = [(bounds[k], bounds[k + 1]) for k in range(len(bounds) - 1)]
    for b in range(B):
        v = v_all[b]
        unl = torch.ones(G, dtype=torch.bool)
        c = None                              # (global index, value, quaternion) of the last mode, as the merged state holds it
        v0 = total = None
        for r in range(M + 1):
            recs = []
            for lo, hi in shards:
                mass_r, tot_r, disq = 0.0, 0.0, False
                g = torch.arange(lo, hi)
                if c is not None:
                    ci, cv, cq = c
                    d = (q[lo:hi] @ cq).abs()
                    w = torch.exp(v[lo:hi] - v0)
                    if r == 1:
                        tot_r = float(w.sum())
                    lab = unl[lo:hi] & ((d > cs) | (g == ci))
                    mass_r = float(w[lab].sum())
                    disq = bool(((v[lo:hi] > cv) & (g != ci) & (d >= cn)).any())
                    unl[lo:hi] &= ~lab
                best_v, best_i = -math.inf, None
                if r < M:
                    for i in g[unl[lo:hi]].tolist():
                        if best_i is None or record_better(float(v[i]), i, best_v, best_i):
                            best_v, best_i = float(v[i]), i
                recs.append((best_v, best_i, mass_r, tot_r, disq))
            bv, bi, mass, tot, disq = merge_records(recs)
            if c is not None:
                if r == 1:
                    total = tot
                out["mass"][b, r - 1] = mass / total if total else math.nan
                out["local_max"][b, r - 1] = not disq and not math.isnan(c[1])
            if r == M or bi is None:
                break
            if r == 0:
                v0 = bv
            c = (bi, bv, q[bi])
            out["index"][b, r] = bi
            out["count"][b] = r + 1
    return out


def even_bounds(G, W):
    return [rdist.shard_range(G, k, W)[0] for k in range(W)] + [G]


def _bounds_cases(G, W, rng):
    """W slices: the even shard_range split and, for W > 1, an uneven one whose second slice is empty."""
    out = [even_bounds(G, W)]
    if W > 1:
        cuts = sorted(rng.choice(np.arange(1, G), W - 2, replace=False).tolist()) if W > 2 else []
        b = [0] + cuts + [G]
        out.append(b[:1] + [b[1]] + b[1:])
    return out


def _line_rotations(angles):
    from test_modes import _axis_angle
    return np.stack([_axis_angle([0, 0, 1], a) for a in angles]).astype(np.float32)


def _check_sharded_ref(values, R, M, theta, rho, bounds):
    ref, _ = ref_modes(values, R, M, theta, rho)
    got = sharded_ref(values, R, M, theta, rho, bounds)
    for k in ("index", "local_max", "count"):
        assert np.array_equal(got[k], ref[k]), (k, bounds, got[k], ref[k])
    finite = np.isfinite(ref["mass"])
    assert np.array_equal(np.isfinite(got["mass"]), finite)
    assert np.allclose(got["mass"][finite], ref["mass"][finite], rtol=1e-12, atol=0)


def test_record_merge_order():
    assert record_better(math.nan, 9, 5.0, 1) and not record_better(5.0, 1, math.nan, 9)         # NaN first
    assert record_better(math.nan, 2, math.nan, 9) and not record_better(math.nan, 9, math.nan, 2)
    assert record_better(3.0, 9, 2.0, 1) and record_better(3.0, 1, 3.0, 9) and not record_better(3.0, 9, 3.0, 1)
    assert record_better(-math.inf, 7, -math.inf, 8)
    # rank order only sums; the winner does not depend on it
    recs = [(2.0, 40, 0.5, 1.0, False), (2.0, 12, 0.25, 2.0, True), (1.0, 3, 0.0, 0.0, False), (-math.inf, None, 0.0, 0.0, False)]
    assert merge_records(recs) == (2.0, 12, 0.75, 3.0, True)
    assert merge_records(recs[::-1])[:2] == (2.0, 12)


@pytest.mark.parametrize("W", [1, 2, 3, 8])
def test_sharded_restatement_matches_definition(W):
    rng = np.random.default_rng(W)
    R = orc.healpix_grid(1).numpy()
    G = R.shape[0]
    v = rng.integers(-3, 3, (4, G)).astype(np.float32)          # many exact ties, also across shard boundaries
    v[1, 100] = np.nan
    v[2, [7, 300]] = np.nan
    v[3] = -np.inf
    for bounds in _bounds_cases(G, W, rng):
        _check_sharded_ref(v, R, 10, 0.9, 0.6, bounds)


def test_sharded_restatement_hand_cases():
    R = _line_rotations([0.0, 1.0, 2.0, 3.0])
    for bounds in ([0, 1, 4], [0, 2, 4], [0, 2, 2, 4], [0, 0, 4], [0, 1, 2, 3, 4]):
        _check_sharded_ref(np.array([1.0, 3.0, 3.0, 0.0]), R, 4, 0.5, 0.5, bounds)      # equal values on two ranks: index 1 first
        _check_sharded_ref(np.array([1.0, 3.0, 3.0, 0.0]), R, 4, 1.2, 1.2, bounds)
        _check_sharded_ref(np.array([5.0, np.nan, 1.0, 2.0]), R, 3, 0.5, 0.2, bounds)
        _check_sharded_ref(np.full(4, -np.inf), R, 6, 0.5, 0.5, bounds)                 # M > G
    R = _line_rotations([0.0, 0.2, 0.3, 2.0])                                             # the shoulder, split between its points
    for bounds in ([0, 1, 4], [0, 2, 4], [0, 3, 4]):
        _check_sharded_ref(np.array([3.0, 2.5, 2.0, 1.0]), R, 3, 0.25, 0.25, bounds)


# ---- CPU: argument errors of the entry points ---------------------------------------------------------------------------------------
def test_cabi_shard_argument_errors_without_gpu():
    lib = _cabi.load()
    P = 0x1000                                    # never dereferenced: every call below fails (or returns) before any device work

    def setup(G=10, B=2, ptr=P, ws=1 << 20):
        return lib.rnf_rotation_modes_shard_setup(ptr, G, B, ptr, ws, None)

    def rnd(B=2, G=10, g0=0, r=0, M=4, theta=0.5, rho=0.2, ptr=P, rec=P, ws=1 << 20):
        return lib.rnf_rotation_modes_shard_round(ptr, B, G, g0, ptr, r, M, theta, rho, ptr, ws, rec, None)

    def merge(recs=P, W=2, B=2, r=0, M=4, ptr=P, ws=1 << 20):
        return lib.rnf_rotation_modes_shard_merge(recs, W, B, r, M, ptr, ws, ptr, ptr, ptr, ptr, ptr, ptr, None)

    cases = [(setup, dict(ptr=None), b"null"), (setup, dict(G=-1), b"negative"), (setup, dict(B=-1), b"negative"),
             (setup, dict(ws=0), b"workspace"),
             (rnd, dict(ptr=None), b"null"), (rnd, dict(rec=None), b"null"), (rnd, dict(B=-1), b"negative"), (rnd, dict(G=-1), b"negative"),
             (rnd, dict(g0=-1), b"g_index0"), (rnd, dict(M=0), b"outside"), (rnd, dict(M=257), b"outside"), (rnd, dict(r=-1), b"round"),
             (rnd, dict(r=5), b"round"), (rnd, dict(rho=0.0), b"radius"), (rnd, dict(rho=0.6), b"radius"),
             (rnd, dict(theta=3.2, rho=0.2), b"radius"), (rnd, dict(ws=0), b"workspace"), (rnd, dict(rec=P + 8), b"aligned"),
             (merge, dict(recs=None), b"null"), (merge, dict(ptr=None), b"null"), (merge, dict(W=0), b"ranks"), (merge, dict(B=-1), b"negative"),
             (merge, dict(M=0), b"outside"), (merge, dict(r=5), b"round"), (merge, dict(recs=P + 4), b"aligned"), (merge, dict(ws=0), b"workspace")]
    for fn, kw, what in cases:
        assert fn(**kw) == RNF_EINVAL, (fn.__name__, kw)
        assert what in lib.rnf_last_error(), (fn.__name__, kw, lib.rnf_last_error())
    # B == 0 does nothing; an empty slice needs no rotations for the set-up and no values or rotations for a round
    assert setup(B=0, ptr=None, ws=0) == 0 and setup(G=0, ptr=None, ws=0) == 0
    assert rnd(B=0, ptr=None, rec=None, ws=0) == 0 and merge(B=0, recs=None, ptr=None, ws=0) == 0
    # state 2 x 48 B, quaternions 4608 x 16 B, labels 2 x 4608 B, partials 2 x 2 slices x 24 B, each section 256-byte aligned
    assert lib.rnf_rotation_modes_shard_workspace_bytes(4608, 2) == 256 + 73728 + 9216 + 256
    assert lib.rnf_rotation_modes_shard_workspace_bytes(0, 3) == 256
    assert lib.rnf_rotation_modes_shard_workspace_bytes(10, 0) == 0
    assert RECORD_BYTES == 80
    with pytest.raises(_cabi.RnfError):
        _cabi.check(rnd(M=0))


def test_python_argument_errors():
    v, R = torch.zeros(2, 10), torch.eye(3).expand(10, 3, 3)
    with pytest.raises(ValueError, match="neighbour_radius"):
        RankModes(v, R, 0, 4, 0.2, 0.5)
    with pytest.raises(ValueError, match="g_index0"):
        RankModes(v, R, -1, 4, 0.5, 0.2)
    with pytest.raises(RuntimeError, match="CUDA"):
        RankModes(v, R, 0, 4, 0.5, 0.2)
    with pytest.raises(ValueError, match="inside"):
        rdist.sharded_rotation_modes(v, R, 5, 12, 4, 0.5, 0.2)
    with pytest.raises(ValueError, match="min_separation"):
        rdist.sharded_estimate_rotation_modes(None, R, 0, 4608, None, 4, min_separation=0.1, neighbour_radius=0.2)


# ---- GPU: simulated ranks in one process ---------------------------------------------------------------------------------------------
def simulate(values, R, M, theta, rho, bounds):
    """W ranks in one process: one RankModes per slice, each round's records stacked rank-major and merged on every rank."""
    ranks = [RankModes(values[..., lo:hi], R[lo:hi], lo, M, theta, rho) for lo, hi in zip(bounds[:-1], bounds[1:])]
    for r in range(M + 1):
        gathered = torch.stack([k.propose(r) for k in ranks])
        for k in ranks:
            k.merge(r, gathered)
    return [k.result() for k in ranks]


def same_bits(a, b):
    """Bitwise equality (NaN values included) of two tensors."""
    if a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)
    return a.shape == b.shape and torch.equal(a, b)


def assert_same_as_single(values, R, M, theta, rho, bounds):
    want = rotation_modes(values, R, M, theta, rho)
    valid = torch.arange(M, device=values.device) < want["count"][..., None]
    outs = simulate(values, R, M, theta, rho, bounds)
    for k, got in enumerate(outs):
        for key in ("index", "value", "local_max", "count"):
            assert same_bits(got[key], want[key]), (key, k, bounds)
        assert torch.equal(got["valid"], valid)
        m, w = got["mass"].double(), want["mass"].double()
        assert torch.equal(torch.isnan(m), torch.isnan(w))
        ok = ~torch.isnan(w)
        rel = ((m - w).abs() / w.abs().clamp(min=1e-30))[ok]
        assert rel.numel() == 0 or rel.max().item() <= 1e-5, rel.max().item()
        rows = R[got["index"].clamp(min=0)]
        assert torch.equal(got["rotations"][valid], rows[valid])
        assert torch.isnan(got["rotations"][~valid]).all()
        if k > 0:                                                              # every rank holds the same bytes
            for key in got:
                assert same_bits(got[key], outs[0][key]), key
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("W", [1, 2, 3, 8])
@pytest.mark.parametrize("level", [2, 3, 4])
def test_sharded_matches_single_random_values(W, level):
    R = rgrid.healpix_grid(level)
    G = R.shape[0]
    rng = np.random.default_rng(level * 10 + W)
    v = torch.from_numpy((2.0 * rng.standard_normal((3, G))).astype(np.float32))
    v[1, torch.from_numpy(rng.integers(0, G, 50))] = v[1].max()         # exact ties, across the shard boundaries too
    v = v.cuda()
    for bounds in _bounds_cases(G, W, rng):
        assert_same_as_single(v, R, 12, 0.45, evalpath.default_neighbour_radius(level), bounds)


@pytest.mark.gpu
@pytest.mark.parametrize("W", [1, 2, 3, 8])
@pytest.mark.parametrize("name", ["tet", "oct", "ico"])
def test_sharded_matches_single_symmetric_densities(W, name):
    Rn, v, centres = symmetric_case(name, 4, seed=3)
    R, v = torch.from_numpy(Rn).cuda(), torch.from_numpy(v).cuda()
    M = len(centres) + 8
    for bounds in _bounds_cases(R.shape[0], W, np.random.default_rng(W)):
        want = assert_same_as_single(v[None], R, M, 0.5, evalpath.default_neighbour_radius(4), bounds)
        assert want["local_max"].sum() == len(centres)


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 8])
def test_sharded_boundary_inside_a_mode_and_ties_across_ranks(W):
    R = rgrid.healpix_grid(3)
    G = R.shape[0]
    rng = np.random.default_rng(30 + W)
    v = (2.0 * rng.standard_normal((2, G))).astype(np.float32)
    theta, rho = 0.45, evalpath.default_neighbour_radius(3)
    # image 0: its best point starts slice 1, and its separation disc holds points of slice 0 too
    c = G // 3 + 7
    v[0, c] = v[0].max() + 1.0
    q = quaternions(R.cpu().numpy())
    disc = np.abs(q @ q[c]) > math.cos(theta / 2)
    assert disc[:c].any() and disc[c + 1:].any()
    bounds = [0] + sorted(set(np.linspace(c, G, W - 1, endpoint=False).astype(int).tolist())) + [G]
    assert bounds[1] == c
    # image 1: equal maxima at points of different ranks; the lower global index must win
    hi = v[1].max() + 1.0
    ties = [bounds[-2] + 3, bounds[1] + 5, 2]
    v[1, ties] = hi
    want = assert_same_as_single(torch.from_numpy(v).cuda(), R, 16, theta, rho, bounds)
    assert want["index"][0, 0].item() == c and want["index"][1, 0].item() == 2


@pytest.mark.gpu
@pytest.mark.parametrize("W", [1, 2, 3, 8])
def test_sharded_matches_single_shapes_nan_inf(W):
    R = rgrid.healpix_grid(2)
    G = R.shape[0]
    rng = np.random.default_rng(5 + W)
    for B in (0, 1, 7):
        v = torch.from_numpy(rng.standard_normal((B, G)).astype(np.float32)).cuda()
        for bounds in _bounds_cases(G, W, rng):
            assert_same_as_single(v, R, 9, 0.5, 0.3, bounds)
    v = rng.standard_normal((3, G)).astype(np.float32)
    v[0, 17] = np.nan
    v[1, [40, 3000]] = np.nan
    v[2] = -np.inf
    for bounds in _bounds_cases(G, W, rng):
        assert_same_as_single(torch.from_numpy(v).cuda(), R, 4, 0.5, 0.3, bounds)
    R0 = rgrid.healpix_grid(0)                                                  # M > G
    v = torch.from_numpy(rng.standard_normal((2, 72)).astype(np.float32)).cuda()
    for bounds in _bounds_cases(72, W, rng):
        assert_same_as_single(v, R0, 256, 2.0, 1.1, bounds)
    # [G] input, and a grid of no points at all
    assert_same_as_single(v[0], R0, 5, 0.5, 0.3, even_bounds(72, W))
    outs = simulate(torch.empty(3, 0, device="cuda"), torch.empty(0, 3, 3, device="cuda"), 4, 0.5, 0.3, [0] * (W + 1))
    for o in outs:
        assert (o["count"] == 0).all() and (o["index"] == -1).all() and not o["valid"].any() and (o["mass"] == 0).all()


@pytest.mark.gpu
def test_rotation_modes_rank_with_a_gather_function():
    """rotation_modes_rank as each rank calls it: three simulated ranks in three threads, the gather a barrier and torch.stack."""
    R = rgrid.healpix_grid(3)
    G, W = R.shape[0], 3
    v = 2.0 * torch.randn(4, G, generator=torch.Generator().manual_seed(4)).cuda()
    bounds = even_bounds(G, W)
    slots, res = [None] * W, [None] * W
    barrier = threading.Barrier(W)

    def run(k):
        def gather(rec):
            slots[k] = rec.clone()
            barrier.wait()
            out = torch.stack(slots)
            barrier.wait()                                   # nobody overwrites a slot before all have stacked
            return out
        res[k] = rotation_modes_rank(v[:, bounds[k]:bounds[k + 1]], R[bounds[k]:bounds[k + 1]], bounds[k], 10, 0.4, 0.2, gather)

    threads = [threading.Thread(target=run, args=(k,)) for k in range(W)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    torch.cuda.synchronize()
    want = rotation_modes(v, R, 10, 0.4, 0.2)
    for got in res:
        for key in ("index", "value", "local_max", "count"):
            assert torch.equal(got[key], want[key]), key
        assert torch.allclose(got["mass"], want["mass"], rtol=1e-5, atol=0)
    # one rank alone: the identity gather is rotation_modes
    one = rdist.sharded_rotation_modes(v, R, 0, G, 10, 0.4, 0.2)
    for key in ("index", "value", "local_max", "count"):
        assert torch.equal(one[key], want[key]), key


@pytest.mark.gpu
def test_sharded_is_deterministic_without_sync_and_graph_capturable():
    R = rgrid.healpix_grid(4)
    v = 2.0 * torch.randn(5, R.shape[0], generator=torch.Generator().manual_seed(2)).cuda()
    bounds = even_bounds(R.shape[0], 3)
    args = (v, R, 16, 0.4, 0.1, bounds)
    a = simulate(*args)
    torch.cuda.set_sync_debug_mode("error")
    try:
        b = simulate(*args)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    for x, y in zip(a, b):
        for k in x:
            assert same_bits(x[k], y[k]), k
    # one round + merge of every rank, captured and replayed
    ranks = [RankModes(v[:, lo:hi], R[lo:hi], lo, 16, 0.4, 0.1) for lo, hi in zip(bounds[:-1], bounds[1:])]
    for r in range(3):                                           # rounds 0..2 eagerly
        g = torch.stack([k.propose(r) for k in ranks])
        for k in ranks:
            k.merge(r, g)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g = torch.stack([k.propose(3) for k in ranks])
        for k in ranks:
            k.merge(3, g)
    graph.replay()                                               # round 3
    for r in range(4, 17):
        g = torch.stack([k.propose(r) for k in ranks])
        for k in ranks:
            k.merge(r, g)
    torch.cuda.synchronize()
    for k, x in zip(ranks, a):
        got = k.result()
        for key in x:
            assert same_bits(got[key], x[key]), key


# ---- several GPUs: NCCL ranks ------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, q):
    try:
        q.put((rank, _nccl_body(rank, world, port)))
    except Exception as e:  # surface failures instead of letting the parent wait for its timeout
        q.put((rank, repr(e)))


def _nccl_body(rank, world, port):
    import torch.distributed as dist
    import rotationnormflow_b200 as rnf
    from conftest import seeded_product_flow
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        m = seeded_product_flow(rnf.load_config("symsol"), 4).to(dev).eval()
        feat = torch.relu(torch.randn(4, m.feature_dim, generator=torch.Generator().manual_seed(6))).to(dev)
        level, M, theta = 3, 8, 0.6
        G = 72 * 8 ** level
        rho = evalpath.default_neighbour_radius(level)
        offset = evalpath._random_rotation(dev, torch.Generator().manual_seed(7))
        lo, hi = rdist.shard_range(G, rank, world)
        shard = rgrid.healpix_grid(level, lo, hi, device=dev)
        if not torch.equal(shard, rgrid.healpix_grid(level, device=dev)[lo:hi]):
            return "grid slice differs from the full grid's rows"
        for steps in (0, 40):
            kw = dict(min_separation=theta, neighbour_radius=rho, offset=offset, refine_steps=steps, refine_lr=1e-3 if steps else None)
            rot, md = rdist.sharded_estimate_rotation_modes(m, shard, lo, G, feat, M, **kw)
            want_rot, want = evalpath.estimate_rotation_modes(m, feat, G, M, **kw)
            for k in ("valid", "count", "grid_index"):
                if not torch.equal(md[k], want[k]):
                    return f"{k} differs (refine_steps={steps})"
            v = want["valid"]
            if steps == 0:
                if not (torch.equal(md["logp"], want["logp"]) and torch.equal(rot[v], want_rot[v]) and torch.isnan(rot[~v]).all()):
                    return "unrefined modes differ"
            elif not (torch.allclose(rot[v], want_rot[v], atol=1e-6) and torch.allclose(md["logp"][v], want["logp"][v], atol=1e-5)):
                return "refined modes differ"
            if not torch.allclose(md["mass"], want["mass"], rtol=1e-5, atol=0):
                return f"mass differs (refine_steps={steps})"
            # every rank holds the same result
            got = torch.cat([md["grid_index"].double().flatten(), md["logp"].double().flatten(), rot.double().flatten()]).nan_to_num()
            all_ = torch.empty((world, got.numel()), dtype=got.dtype, device=dev)
            dist.all_gather_into_tensor(all_, got)
            if not all(torch.equal(all_[0], all_[k]) for k in range(world)):
                return "ranks disagree"
        return True
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
@pytest.mark.parametrize("world", sorted({2, max(2, torch.cuda.device_count())}))
def test_sharded_estimate_on_nccl_ranks(world):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = [q.get(timeout=600) for _ in procs]
    finally:
        for p in procs:
            p.join(timeout=120)
            if p.is_alive():
                p.terminate()
                p.join()
    assert sorted(res) == [(r, True) for r in range(world)], res
