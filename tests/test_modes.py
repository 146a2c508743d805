"""Separated posterior modes (modes.rotation_modes / rnf_rotation_modes, evalpath.estimate_rotation_modes, metrics.mode_recall).

The reference is `ref_modes`, a vectorised fp64 numpy restatement of the definition (DESIGN 4.7): per image, M greedy rounds of
  c_m = best unlabelled point (NaN first, then larger value, then lower index)
  local_max = no g != c_m with |q_g . q_c| >= cos(rho / 2) has v_g > v_c (NaN never higher; a NaN mode is no local max)
  label m = unlabelled g with g == c_m or |q_g . q_c| > cos(theta / 2)
  mass = sum_{label m} exp(v - v_c0) / sum_all exp(v - v_c0)
Data of the kernel comparisons keeps every dot product that decides a label or a local maximum at least 1e-6 away from its
threshold, so the fp32 kernel and the fp64 reference cannot disagree on a label."""
import importlib.util
import math
import os

import numpy as np
import pytest
import torch

from conftest import ROOT, seeded_product_flow
from oracle import rnf_oracle as orc
import rotationnormflow_b200 as rnf
from rotationnormflow_b200 import _cabi, evalpath, metrics
from rotationnormflow_b200 import grid as rgrid
from rotationnormflow_b200.modes import rotation_modes

RNF_EINVAL = -1
MARGIN = 1e-6


# ---- the fp64 reference ------------------------------------------------------------------------------------------------------------
def quaternions(R):
    """[N,3,3] -> unit quaternions [N,4] (fp64), best-conditioned of the four candidate rows (as the kernel)."""
    m = np.asarray(R, dtype=np.float64).reshape(-1, 9)
    m00, m01, m02, m10, m11, m12, m20, m21, m22 = m.T
    a = np.sqrt(np.maximum(np.stack([1 + m00 + m11 + m22, 1 + m00 - m11 - m22, 1 - m00 + m11 - m22, 1 - m00 - m11 + m22], -1), 0))
    cand = np.stack([np.stack([a[:, 0] ** 2, m21 - m12, m02 - m20, m10 - m01], -1),
                     np.stack([m21 - m12, a[:, 1] ** 2, m10 + m01, m02 + m20], -1),
                     np.stack([m02 - m20, m10 + m01, a[:, 2] ** 2, m12 + m21], -1),
                     np.stack([m10 - m01, m20 + m02, m21 + m12, a[:, 3] ** 2], -1)], -2)
    q = cand[np.arange(m.shape[0]), a.argmax(-1)]
    return q / np.linalg.norm(q, axis=-1, keepdims=True)


def ref_modes(values, rotations, M, theta, rho, g_index0=0):
    """Returns (dict(index, value, local_max, mass, count) as numpy arrays [B,M] / [B], margin): margin = the smallest distance of a
    deciding dot product from its threshold."""
    v_all = np.atleast_2d(np.asarray(values, dtype=np.float32)).astype(np.float64)
    B, G = v_all.shape
    q = quaternions(rotations) if G else np.zeros((0, 4))
    cs, cn = math.cos(theta / 2), math.cos(rho / 2)
    out = dict(index=np.full((B, M), -1, np.int64), value=np.full((B, M), -np.inf, np.float64), local_max=np.zeros((B, M), bool),
               mass=np.zeros((B, M), np.float64), count=np.zeros(B, np.int64))
    margin = np.inf
    ar = np.arange(G)
    for b in range(B):
        v = v_all[b]
        unl = np.ones(G, bool)
        nan = np.isnan(v)
        c0 = None
        with np.errstate(invalid="ignore", over="ignore"):
            for m in range(M):
                cand = ar[unl]
                if cand.size == 0:
                    break
                cn_ = cand[nan[cand]]
                c = int(cn_[0]) if cn_.size else int(cand[np.argmax(v[cand])])   # argmax: first of the ties = lowest index
                if c0 is None:
                    c0 = c
                d = np.abs(q @ q[c])
                higher = v > v[c]
                higher[c] = False
                out["local_max"][b, m] = not np.isnan(v[c]) and not (higher & (d >= cn)).any()
                lab = unl & ((d > cs) | (ar == c))
                w = np.exp(v - v[c0])
                out["mass"][b, m] = w[lab].sum() / w.sum()
                out["index"][b, m] = c + g_index0
                out["value"][b, m] = v[c]
                out["count"][b] = m + 1
                near_s = np.abs(d[unl & (ar != c)] - cs)
                near_n = np.abs(d[higher] - cn)
                margin = min([margin] + [x.min() for x in (near_s, near_n) if x.size])
                unl &= ~lab
    return out, margin


# ---- test densities ----------------------------------------------------------------------------------------------------------------
def _axis_angle(axis, angle):
    a = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + math.sin(angle) * K + (1 - math.cos(angle)) * K @ K


def symmetry_group(name):
    """The rotation groups of the SYMSOL solids by closure of two generators: tetrahedron 12, cube 24, icosahedron 60 elements."""
    phi = (1 + 5 ** 0.5) / 2
    gens = {"tet": [_axis_angle([0, 0, 1], math.pi), _axis_angle([1, 1, 1], 2 * math.pi / 3)],
            "oct": [_axis_angle([0, 0, 1], math.pi / 2), _axis_angle([1, 1, 1], 2 * math.pi / 3)],
            "ico": [_axis_angle([0, 1, phi], 2 * math.pi / 5), _axis_angle([1, 1, 1], 2 * math.pi / 3)]}[name]
    elems = [np.eye(3)]
    keys = {tuple(np.round(np.eye(3), 6).ravel())}
    i = 0
    while i < len(elems):
        for g in gens:
            x = g @ elems[i]
            k = tuple(np.round(x, 6).ravel())
            if k not in keys:
                keys.add(k)
                elems.append(x)
        i += 1
    return np.stack(elems)


def symmetric_density(R, centres, kappa):
    """v(R) = log sum_k exp(kappa tr(R_k^T R)) in fp64, returned as float32."""
    R = np.asarray(R, np.float64)
    tr = np.einsum("kij,gij->gk", centres, R)
    mx = tr.max(1, keepdims=True)
    return (kappa * mx[:, 0] + np.log(np.exp(kappa * (tr - mx)).sum(1))).astype(np.float32)


def symmetric_case(name, level, kappa=20.0, seed=0):
    Q = orc.random_rotations(1, torch.Generator().manual_seed(seed), torch.float64)[0].numpy()
    centres = Q @ symmetry_group(name)
    R = orc.healpix_grid(level).numpy()
    return R, symmetric_density(R, centres, kappa), centres


def _angle(A, B):
    return float(np.arccos(np.clip((np.trace(A.T @ B) - 1) / 2, -1, 1)))


def safe_thresholds(values, R, M, theta, rho, g_index0=0):
    """theta and rho nudged (by < 1 %) until no deciding dot product lies within MARGIN of its threshold; the reference result."""
    for _ in range(40):
        ref, margin = ref_modes(values, R, M, theta, rho, g_index0)
        if margin >= MARGIN:
            return theta, rho, ref
        theta *= 1.000317
        rho *= 1.000529
    raise AssertionError("no threshold pair with a 1e-6 margin")


# ---- CPU: the reference on hand-checkable cases ---------------------------------------------------------------------------------------
def _line_rotations(angles):
    return np.stack([_axis_angle([0, 0, 1], a) for a in angles]).astype(np.float32)


def test_reference_ties_go_to_the_lower_index():
    R = _line_rotations([0.0, 1.0, 2.0, 3.0])
    ref, _ = ref_modes(np.array([1.0, 3.0, 3.0, 0.0]), R, 4, 0.5, 0.5)
    assert ref["index"][0].tolist() == [1, 2, 0, 3]
    assert ref["local_max"][0].all()
    ref, _ = ref_modes(np.array([1.0, 3.0, 3.0, 0.0]), R, 4, 1.2, 1.2)     # 1 takes 0 and its tie 2; 3 sees 2 (higher) 1 rad away
    assert ref["index"][0].tolist() == [1, 3, -1, -1] and ref["count"][0] == 2
    assert ref["local_max"][0].tolist() == [True, False, False, False]


def test_reference_nan_ranks_first_and_is_never_a_local_max():
    R = _line_rotations([0.0, 0.1, 1.0, 2.0])
    ref, _ = ref_modes(np.array([5.0, np.nan, 1.0, 2.0]), R, 3, 0.5, 0.2)
    assert ref["index"][0].tolist() == [1, 3, 2]                          # the NaN, then 3 (0 went into the NaN's ball)
    assert ref["local_max"][0].tolist() == [False, True, True]
    assert np.isnan(ref["mass"][0]).all()                                 # NaN propagates through the normaliser


def test_reference_all_minus_inf_and_more_modes_than_points():
    R = _line_rotations([0.0, 1.0, 2.0])
    ref, _ = ref_modes(np.full(3, -np.inf), R, 5, 0.5, 0.5)
    assert ref["count"][0] == 3 and ref["index"][0].tolist() == [0, 1, 2, -1, -1]
    assert np.isnan(ref["mass"][0, :3]).all() and (ref["mass"][0, 3:] == 0).all()          # 0 / 0
    assert ref["local_max"][0].tolist() == [True, True, True, False, False]
    assert (ref["value"][0, 3:] == -np.inf).all()
    ref, _ = ref_modes(np.array([0.0, 1.0, 2.0]), R, 5, 0.5, 0.5)
    assert ref["count"][0] == 3 and ref["index"][0].tolist() == [2, 1, 0, -1, -1]
    assert abs(ref["mass"][0, :3].sum() - 1) < 1e-12


def test_reference_shoulder_is_not_a_local_max():
    # mode 0 at 0 takes the point 0.2 rad away; the next pick, 0.3 rad from the peak, sees that labelled point (higher, 0.1 rad
    # away) within the neighbour radius: a shoulder
    R = _line_rotations([0.0, 0.2, 0.3, 2.0])
    ref, _ = ref_modes(np.array([3.0, 2.5, 2.0, 1.0]), R, 3, 0.25, 0.25)
    assert ref["index"][0].tolist() == [0, 2, 3]
    assert ref["local_max"][0].tolist() == [True, False, True]            # 2 sees 1 (0.1 rad away, higher, already labelled 0)
    w = np.exp(np.array([3.0, 2.5, 2.0, 1.0]) - 3.0)
    assert np.allclose(ref["mass"][0], [w[:2].sum() / w.sum(), w[2] / w.sum(), w[3] / w.sum()])


def test_reference_tetrahedral_density_level3():
    R, v, centres = symmetric_case("tet", 3)
    assert len(centres) == 12
    M = 24
    ref, _ = ref_modes(v, R, M, 0.9, evalpath.default_neighbour_radius(3))
    lm = ref["local_max"][0]
    assert lm.sum() == 12 and lm[:12].all()
    spacing = 0.1309                                      # largest nearest-neighbour angle of the level-3 grid (tools/grid_spacing.py)
    found = R[ref["index"][0, :12]].astype(np.float64)
    for c in centres:
        assert min(_angle(c, f) for f in found) <= spacing
    assert np.allclose(ref["mass"][0, :12], 1 / 12, atol=2e-3), ref["mass"][0, :12]


def test_symmetry_groups_have_their_orders():
    assert [len(symmetry_group(n)) for n in ("tet", "oct", "ico")] == [12, 24, 60]


def test_default_neighbour_radius_is_measured():
    spec = importlib.util.spec_from_file_location("grid_spacing", os.path.join(ROOT, "tools", "grid_spacing.py"))
    gs = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gs)
    for level in range(4):
        assert abs(evalpath.default_neighbour_radius(level) - 1.5 * gs.largest_nn_angle(level)) < 1e-6
    assert evalpath.default_neighbour_radius(6) == evalpath.default_neighbour_radius(5) / 2


# ---- CPU: argument errors ---------------------------------------------------------------------------------------------------------
def test_cabi_modes_argument_errors_without_gpu():
    lib = _cabi.load()
    P = 0x1000                                    # never dereferenced: every call below fails before any device work

    def call(B=1, G=10, M=4, theta=0.5, rho=0.2, ptr=P, ws=1 << 20):
        return lib.rnf_rotation_modes(ptr, B, G, 0, ptr, M, theta, rho, ptr, ws, ptr, ptr, ptr, ptr, ptr, None)

    assert call(ptr=None) == RNF_EINVAL and b"null" in lib.rnf_last_error()
    for kw, what in ((dict(B=-1), b"negative"), (dict(G=-1), b"negative"), (dict(M=0), b"outside"), (dict(M=257), b"outside"),
                     (dict(rho=0.0), b"radius"), (dict(rho=0.6), b"radius"), (dict(theta=3.2, rho=0.2), b"radius"),
                     (dict(ws=0), b"workspace")):
        assert call(**kw) == RNF_EINVAL, kw
        assert what in lib.rnf_last_error(), (kw, lib.rnf_last_error())
    assert call(B=0, ptr=None, ws=0) == 0                               # B == 0 does nothing
    # quaternions 4608 x 16 B, labels 2 x 4608 B, partials 2 x 2 slices x 24 B, state 2 x 24 B, each section 256-byte aligned
    assert lib.rnf_rotation_modes_workspace_bytes(4608, 2, 12) == 73728 + 9216 + 256 + 256
    assert lib.rnf_rotation_modes_workspace_bytes(10, 0, 4) == 0
    with pytest.raises(_cabi.RnfError):
        _cabi.check(call(M=0))


def test_python_argument_errors():
    v, R = torch.zeros(2, 10), torch.eye(3).expand(10, 3, 3)
    with pytest.raises(ValueError, match="neighbour_radius"):
        rotation_modes(v, R, 4, 0.2, 0.5)                 # rho > theta
    with pytest.raises(ValueError, match="num_modes"):
        rotation_modes(v, R, 0, 0.5, 0.2)
    with pytest.raises(ValueError, match="min_separation"):
        evalpath.estimate_rotation_modes(None, torch.zeros(1, 8), 4608, 4, min_separation=0.1, neighbour_radius=0.2)
    with pytest.raises(RuntimeError, match="CUDA"):
        rotation_modes(v, R, 4, 0.5, 0.2)


# ---- GPU: the kernel against the reference ---------------------------------------------------------------------------------------------
def _check_against_reference(values, R, M, theta, rho, g_index0=0):
    theta, rho, ref = safe_thresholds(values, R, M, theta, rho, g_index0)
    out = rotation_modes(torch.from_numpy(np.asarray(values, np.float32)).cuda(), torch.from_numpy(np.asarray(R, np.float32)).cuda(), M,
                         theta, rho, g_index0=g_index0)
    out = {k: t.cpu().numpy() for k, t in out.items()}
    if np.asarray(values).ndim == 1:
        ref = {k: t[0] for k, t in ref.items()}
    assert np.array_equal(out["count"], ref["count"])
    assert np.array_equal(out["index"], ref["index"])
    assert np.array_equal(out["local_max"], ref["local_max"])
    assert np.array_equal(out["value"], ref["value"].astype(np.float32), equal_nan=True)
    rel = np.abs(out["mass"] - ref["mass"]) / np.maximum(np.abs(ref["mass"]), 1e-30)
    assert np.nanmax(rel, initial=0.0) <= 1e-5, np.nanmax(rel)
    assert np.array_equal(np.isnan(out["mass"]), np.isnan(ref["mass"]))
    return out, ref


@pytest.mark.gpu
@pytest.mark.parametrize("level", [2, 3, 4])
def test_kernel_matches_reference_random_values(level):
    R = orc.healpix_grid(level).numpy()
    rng = np.random.default_rng(level)
    v = (2.0 * rng.standard_normal((3, R.shape[0]))).astype(np.float32)
    v[1, rng.integers(0, R.shape[0], 50)] = v[1].max()       # exact ties
    _check_against_reference(v, R, 12, 0.45, evalpath.default_neighbour_radius(level))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tet", "oct", "ico"])
def test_kernel_matches_reference_symmetric_densities(name):
    R, v, centres = symmetric_case(name, 4, seed=3)
    M = len(centres) + 8
    out, ref = _check_against_reference(v, R, M, 0.5, evalpath.default_neighbour_radius(4))
    assert out["local_max"].sum() == len(centres)


@pytest.mark.gpu
def test_kernel_matches_reference_shapes_and_index_offset():
    R = orc.healpix_grid(2).numpy()
    rng = np.random.default_rng(5)
    for B in (1, 7):
        v = rng.standard_normal((B, R.shape[0])).astype(np.float32)
        _check_against_reference(v, R, 9, 0.5, 0.3)
    v = rng.standard_normal(R.shape[0]).astype(np.float32)                   # [G] input
    _check_against_reference(v, R, 5, 0.5, 0.3, g_index0=123456789)
    _check_against_reference(rng.standard_normal((2, R.shape[0])).astype(np.float32), R, 6, 0.5, 0.3, g_index0=4608 * 3)
    # the NaN and all -inf cases of the reference, on the device
    v = rng.standard_normal((3, R.shape[0])).astype(np.float32)
    v[0, 17] = np.nan
    v[2] = -np.inf
    _check_against_reference(v, R, 4, 0.5, 0.3)
    # M > G
    _check_against_reference(rng.standard_normal((2, 72)).astype(np.float32), orc.healpix_grid(0).numpy(), 256, 2.0, 1.1)
    # B = 0 and G = 0
    out = rotation_modes(torch.empty(0, 4608, device="cuda"), torch.from_numpy(R).cuda(), 4, 0.5, 0.3)
    assert out["index"].shape == (0, 4) and out["count"].shape == (0,)
    out = rotation_modes(torch.empty(3, 0, device="cuda"), torch.empty(0, 3, 3, device="cuda"), 4, 0.5, 0.3)
    assert (out["count"] == 0).all() and (out["index"] == -1).all() and (out["value"] == -math.inf).all()
    assert not out["local_max"].any() and (out["mass"] == 0).all()


@pytest.mark.gpu
def test_kernel_is_deterministic_without_sync_and_graph_capturable():
    R = rgrid.healpix_grid(4)
    v = 2.0 * torch.randn(5, R.shape[0], generator=torch.Generator().manual_seed(2)).cuda()
    args = (v, R, 16, 0.4, 0.1)
    a = rotation_modes(*args)
    torch.cuda.set_sync_debug_mode("error")
    try:
        b = rotation_modes(*args)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        rotation_modes(*args)                                                 # warm-up off the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = rotation_modes(*args)
    g.replay()
    torch.cuda.synchronize()
    for k in a:
        assert torch.equal(a[k], c[k]), k


@pytest.mark.gpu
def test_mode_recall_tetrahedral():
    R, v, centres = symmetric_case("tet", 4, seed=1)
    Rd = torch.from_numpy(R).cuda()
    out = rotation_modes(torch.from_numpy(v).cuda(), Rd, 20, 0.9, evalpath.default_neighbour_radius(4))
    modes = Rd[out["index"].clamp(min=0)][None]
    gt = torch.from_numpy(centres).float()[None]
    rec = metrics.mode_recall(modes, out["local_max"][None], gt, 0.0655)     # one level-4 grid spacing
    assert rec.shape == (1,) and rec.item() == 1.0
    assert metrics.mode_recall(modes, torch.zeros_like(out["local_max"])[None], gt, 0.0655).item() == 0.0


# ---- GPU: end to end on a seeded flow ------------------------------------------------------------------------------------------------
def _symsol_flow():
    cfg = rnf.load_config("symsol")
    m = seeded_product_flow(cfg, 4).cuda().eval()
    feat = torch.relu(torch.randn(4, m.feature_dim, generator=torch.Generator().manual_seed(6))).cuda()
    return m, feat


@pytest.mark.gpu
def test_estimate_rotation_modes_end_to_end():
    m, feat = _symsol_flow()
    Q, M, theta = 72 * 8 ** 3, 8, 0.6
    rho = evalpath.default_neighbour_radius(3)
    est, og = evalpath.estimate_rotation_grid(m, feat, Q, generator=torch.Generator().manual_seed(7))
    # thresholds with a 1e-6 margin on this log-density, so that the reference and the kernel agree label for label
    grid = rgrid.get_closest_available_grid(Q)
    offset = evalpath._random_rotation(feat.device, torch.Generator().manual_seed(7))
    lp = m.grid_log_prob(grid, feat, offset=offset, return_logp=True)["logp"]
    theta, rho, ref = safe_thresholds(lp.cpu().numpy(), grid.cpu().numpy(), M, theta, rho)
    raw = rotation_modes(lp, grid, M, theta, rho)
    assert np.array_equal(raw["index"].cpu().numpy(), ref["index"])
    assert np.array_equal(raw["local_max"].cpu().numpy(), ref["local_max"])
    rot, md = evalpath.estimate_rotation_modes(m, feat, Q, M, min_separation=theta, neighbour_radius=rho,
                                               generator=torch.Generator().manual_seed(7))
    assert rot.shape == (4, M, 3, 3) and md["valid"][:, 0].all()
    assert torch.equal(md["grid_index"][:, 0], og["argmax"])
    assert torch.allclose(rot[:, 0], est, atol=1e-6)
    for k in ("max", "argmax", "sumexp"):
        assert torch.equal(md[k], og[k]), k
    # the values are the grid log-density at the returned indices; the modes are the reference's local maxima, in order
    valid, gi = md["valid"], md["grid_index"]
    assert torch.equal(md["logp"][valid], torch.gather(lp, 1, gi.clamp(min=0))[valid])
    assert torch.isnan(rot[~valid]).all() and (gi[~valid] == -1).all() and (md["count"] == valid.sum(1)).all()
    for b in range(4):
        assert gi[b][valid[b]].cpu().numpy().tolist() == ref["index"][b][ref["local_max"][b]].tolist()
    # refinement: no refined mode falls below its grid log p, and the refined grid arg-max is estimate_rotation_grid's refinement
    rr, mr = evalpath.estimate_rotation_modes(m, feat, Q, M, min_separation=theta, neighbour_radius=rho,
                                              generator=torch.Generator().manual_seed(7), refine_steps=100, refine_lr=1e-3)
    est2, og2 = evalpath.estimate_rotation_grid(m, feat, Q, generator=torch.Generator().manual_seed(7), refine_steps=100, refine_lr=1e-3)
    v2 = mr["valid"]
    grid_lp = torch.gather(lp, 1, mr["grid_index"].clamp(min=0))
    assert (mr["logp"][v2] >= grid_lp[v2] - 1e-3).all()
    assert (mr["logp"][:, :-1] >= mr["logp"][:, 1:]).all()                  # sorted by refined log p, padding (-inf) last
    assert torch.allclose(mr["mass"].sum(1), md["mass"].sum(1), rtol=1e-5)   # merging moves mass, never loses it
    survived = 0
    for b in range(4):
        hit = (mr["grid_index"][b] == og["argmax"][b]) & v2[b]
        if hit.any():
            j = int(hit.nonzero()[0])
            assert torch.allclose(rr[b, j], est2[b], atol=1e-6)
            assert torch.allclose(mr["logp"][b, j], og2["refined_logp"][b], atol=1e-5)
            survived += 1
        else:       # merged into a better refined mode within the neighbour radius
            q = evalpath.matrix_to_quaternion(torch.cat([rr[b][v2[b]], est2[b][None]]))
            near = (q[:-1] @ q[-1]).abs() >= math.cos(rho / 2)
            assert (near & (mr["logp"][b][v2[b]] >= og2["refined_logp"][b] - 1e-5)).any()
    assert survived >= 1


@pytest.mark.gpu
def test_estimate_rotation_modes_with_fisher_base():
    m, feat = _symsol_flow()
    Q = 72 * 8 ** 2
    A = (3.0 * orc.random_rotations(4, torch.Generator().manual_seed(9))).cuda()
    rot, md = evalpath.estimate_rotation_modes(m, feat, Q, 6, min_separation=0.8, fisher_A=A, generator=torch.Generator().manual_seed(3))
    grid = rgrid.get_closest_available_grid(Q)
    offset = evalpath._random_rotation(feat.device, torch.Generator().manual_seed(3))
    lpA = m.grid_log_prob(grid, feat, offset=offset, fisher_A=A, return_logp=True)["logp"]
    lp0 = m.grid_log_prob(grid, feat, offset=offset, return_logp=True)["logp"]
    v, gi = md["valid"], md["grid_index"].clamp(min=0)
    assert torch.equal(md["logp"][v], torch.gather(lpA, 1, gi)[v])
    assert not torch.equal(md["logp"][v], torch.gather(lp0, 1, gi)[v])
    assert torch.equal(md["argmax"], lpA.argmax(1))


@pytest.mark.gpu
def test_estimate_rotation_modes_chunks_images(monkeypatch):
    m, feat = _symsol_flow()
    Q = 72 * 8 ** 2
    a = evalpath.estimate_rotation_modes(m, feat, Q, 5, min_separation=0.8, generator=torch.Generator().manual_seed(3))
    monkeypatch.setattr(evalpath, "MODES_LOGP_BYTES", 4608 * 4 * 3)         # three images per chunk
    b = evalpath.estimate_rotation_modes(m, feat, Q, 5, min_separation=0.8, generator=torch.Generator().manual_seed(3))
    assert torch.equal(a[0].nan_to_num(), b[0].nan_to_num())
    for k in a[1]:
        assert torch.equal(a[1][k], b[1][k]), k
