"""The flow kernels at trained-model weight scales, against the fp64 oracle.

Every other test runs random-initialisation weights: hidden activations of 0.01 - 1, O(1) mixture logits, centres well inside
the 0.7 disk.  Trained checkpoints leave that regime, and several fast paths are only right inside a numeric range:
  - the tensor-core GEMMs (modes tc, tc_row) split each activation into fp16 hi / lo planes (flow_t4.cu relu_split_pair,
    flow_row.cu store_a32): exact to 22 bits for 0.125 <= x < 65536, 2^-25 absolute below, +Inf from 65536 on;
  - the fast-path mixture weights (mobius_pair.cuh mixture_pairs) use ex2.approx.ftz and switch
    branches at 2^t = 2^-7 (a = -4.852) and t = 28.85 (a = 20); a row whose logits are all below -87.3 has no weight left;
  - the inverse's Newton + replay root search was justified for F' in [0.17, 5.7].
The stress models are transforms of golden weights whose effect is known exactly:
  rescale(k)   fc_first.{weight,bias}, layers.{1,3,5}.bias x 2^k, fc_last.weight x 2^-k of every Mobius conditioner: by ReLU
               homogeneity the flow is unchanged and every hidden pre-activation (the per-image feature term included) is x 2^k;
  sharp(c)     fc_last.{weight,bias} x c: peaky mixtures, centres at |w'| -> 0.7;
  logits_at    logit biases of fc_last set so that every row's logits straddle the branch points.
CPU tests check that each transform reaches its regime, the oracle's invariance and its own fp32 error, and an fp32 / fp16
emulation of the split; GPU tests hold every mode to the fp64 oracle (inside the limits) or to "right or non-finite" (outside)."""
import contextlib
import ctypes
import math

import numpy as np
import pytest
import torch

from conftest import golden, record_error, seeded_product_flow
from oracle import rnf_oracle as orc
import rotationnormflow_b200 as rnf

K = 64
FP16_MAX = 65504.0
SPLIT_LIMIT = 65536.0                           # tc / tc_row: activations from here on turn the row into Inf / NaN
SERIES_SWITCH = -7.0 * math.log(2.0)            # a where 2^t = 2^-7: the softplus series branch of the fast paths
OWN_ERROR_FACTOR = {"tc": 2.0, "tc_row": 2.0, "fp32": 4.0}    # as tests/test_gpu_parity.py
MODES = ["fp32", "tc", "tc_row"]
FAMILIES = ["s_symsol", "s_modelnet", "s_uncond", "s_lu"]

# rescale targets: (name, statistic, log2 of the target) -- statistic "p10" is the 10th percentile of the positive hidden
# pre-activations (the smallest significant ones), "max" the largest; "init" is a fixed k (activations 2^k of random init)
RESCALES = [("init_2^-6", "init", -6.0), ("p10_2^-14", "p10", -14.0), ("p10_2^-16", "p10", -16.0), ("p10_2^-18", "p10", -18.0),
            ("max_1", "max", 0.0), ("max_2^10", "max", 10.0), ("max_6e4", "max", math.log2(6e4)),
            ("max_1.1e5", "max", math.log2(1.1e5)), ("max_3e5", "max", math.log2(3e5))]
SHARP = [("sharp3", 3.0), ("sharp12", 12.0), ("sharp100", 100.0)]
CASES = [r[0] for r in RESCALES] + [s[0] for s in SHARP] + ["logits", "logits_below_88"]
FULL_CASES = ["max_6e4", "max_1.1e5", "sharp100", "logits"]      # symsol2048: one point per transform
OUTSIDE = {"max_1.1e5", "max_3e5"}              # hidden activations >= SPLIT_LIMIT: tc / tc_row rows must be non-finite or ...
# ... within the bounds below, which is all the tc modes reach once the rescale moves the fp16 planes of the activations (k < -9)
# or of the fc_last weights (k > 9, weights x 2^-k) into the fp16 subnormals: measured on a B200 and held to about twice that,
# (forward max|dR|, forward rel dldj, grid rel dlogp, inverse worst row).  A build with the saturating split fails these
# bounds on max_1.1e5 / max_3e5 (finite rows up to 2e-2 off); the split's own limits come from the emulation below.
PRECISION = {"p10_2^-16": (3e-5, 5e-5, 3e-4, 1e-3), "p10_2^-18": (1.5e-4, 2.5e-4, 8e-4, 1e-3),
             "max_2^10": (3e-5, 5e-5, 2e-4, 1e-3), "max_6e4": (6e-3, 1e-2, 1e-2, 1e-2)}
PRECISION.update({c: PRECISION["max_6e4"] for c in OUTSIDE})


def _all_cases():
    return [(t, c) for t in FAMILIES for c in CASES] + [("symsol2048", c) for c in FULL_CASES]


# ---- stress models --------------------------------------------------------------------------------------------------------------
def _mobius_prefixes(cfg):
    return [f"layers.{i}.conditioner." for i, k in enumerate(orc.layer_plan(cfg)) if k == "mobius"]


def rescale(cfg, sd, k):
    s = 2.0 ** k
    out = {n: v.clone() for n, v in sd.items()}
    for p in _mobius_prefixes(cfg):
        for n in ("fc_first.weight", "fc_first.bias", "layers.1.bias", "layers.3.bias", "layers.5.bias"):
            out[p + n] *= s
        out[p + "fc_last.weight"] *= 1.0 / s
    return out


def sharp(cfg, sd, c):
    """fc_last x c.  The golden weights need c = 100 to bring max |w'| above 0.69 (c = 40 reaches 0.677 - 0.683)."""
    out = {n: v.clone() for n, v in sd.items()}
    for p in _mobius_prefixes(cfg):
        out[p + "fc_last.weight"] *= c
        out[p + "fc_last.bias"] *= c
    return out


def _logit_pattern(j):
    """Logit biases of the j-th Mobius layer: even layers straddle a = 20 (+-1e-3) and sit at a = -60 next to O(1) logits; odd
    layers straddle the series switch a = -4.852 and fill the band where the series / log2 choice matters (-5.5 .. -1.5)."""
    b = np.empty(K)
    pm = np.where(np.arange(16) % 2 == 0, 1e-3, -1e-3)
    if j % 2 == 0:
        b[:16] = 20.0 + pm
        b[16:24] = -60.0 + np.linspace(-0.5, 0.5, 8)
        b[24:] = np.linspace(-2.0, 2.0, 40)
    else:
        b[:16] = SERIES_SWITCH + pm
        b[16:] = np.linspace(-5.5, -1.5, 48)
    return torch.from_numpy(b).float()


def logits_at(cfg, sd, below_88=False):
    """fc_last logit rows scaled by 1e-4 (a row's logits vary by ~1e-5 around their biases), biases set to _logit_pattern;
    below_88: every logit at -90 (outside the fast paths' range: all weights flush to zero)."""
    out = {n: v.clone() for n, v in sd.items()}
    for j, p in enumerate(_mobius_prefixes(cfg)):
        out[p + "fc_last.weight"][:K] *= 1e-4
        out[p + "fc_last.bias"][:K] = -90.0 + torch.linspace(-0.5, 0.5, K) if below_88 else _logit_pattern(j)
    return out


def stress_inputs(n=512, seed=0):
    """n Haar rotations, the identity, the 24 rotations with entries in {0, +-1}, 16 rotations by pi about random axes (quaternion
    real part 0: ties between the candidates of matrix_to_quaternion) and the same 16 perturbed by one fp32 ulp."""
    gen = torch.Generator().manual_seed(seed)
    haar = orc.random_rotations(n, gen, torch.float64)
    perms = []
    for p in ((0, 1, 2), (1, 2, 0), (2, 0, 1), (0, 2, 1), (2, 1, 0), (1, 0, 2)):
        for s in range(8):
            M = torch.zeros(3, 3, dtype=torch.float64)
            for i in range(3):
                M[i, p[i]] = -1.0 if (s >> i) & 1 else 1.0
            if torch.linalg.det(M) > 0:
                perms.append(M)
    ax = torch.randn(16, 3, generator=gen, dtype=torch.float64)
    ax = ax / ax.norm(dim=1, keepdim=True)
    pi_rot = 2.0 * ax[:, :, None] * ax[:, None, :] - torch.eye(3, dtype=torch.float64)
    R = torch.cat([haar, torch.eye(3, dtype=torch.float64)[None], torch.stack(perms), pi_rot]).float()
    bumped = torch.nextafter(pi_rot.float(), torch.full_like(pi_rot.float(), 2.0))
    assert len(perms) == 24
    return torch.cat([R, bumped])


_base_cache, _case_cache = {}, {}


def _base(tag):
    if tag not in _base_cache:
        g = golden(tag)
        R = stress_inputs()
        N = R.shape[0]
        d = dict(g=g, cfg=g.cfg, sd=g.state_dict(), R=R, feat=g.feat, fi=None, rows=None, A=None)
        if g.feat is not None:
            d["fi"] = torch.arange(N) % g.feat.shape[0]
            d["rows"] = g.feat[d["fi"]]
        if "fisher_A" in g.z.files:
            d["A"] = torch.from_numpy(g.z["fisher_A"])
        gen = torch.Generator().manual_seed(21)
        d["grid"] = orc.healpix_grid(2, 1000, 2500)                    # ragged level-2 slice, global index 1000
        d["off"] = orc.random_rotations(1, gen)[0]
        d["stats"] = activation_stats(g.cfg, d["sd"], R, d["rows"], d["feat"], d["grid"] @ d["off"] if tag != "symsol2048" else None)
        _base_cache[tag] = d
    return _base_cache[tag]


@contextlib.contextmanager
def _recording(cfg):
    """Records, for every Mobius conditioner the fp64 oracle evaluates, the inputs of the four ReLU + fp16 splits (h0, h1, h3,
    h0 + h5: the same arithmetic as orc.conditioner), the logits, the squashed centres w' and the Jacobians f_k."""
    prefixes = set(_mobius_prefixes(cfg))
    rec = dict(acts=[], logits=[], wn=[], f=[])
    cond, prep, mh = orc.conditioner, orc._mobius_prep, orc._mobius_h

    def conditioner(sd, prefix, x):
        out = cond(sd, prefix, x)
        if prefix in prefixes:
            lin = torch.nn.functional.linear
            h0 = lin(x, sd[prefix + "fc_first.weight"], sd[prefix + "fc_first.bias"])
            h, acts = h0, [h0]
            for j in (1, 3, 5):
                h = lin(torch.relu(h), sd[f"{prefix}layers.{j}.weight"], sd[f"{prefix}layers.{j}.bias"])
                acts.append(h if j != 5 else h0 + h)
            rec["acts"].append(torch.cat([a.reshape(-1) for a in acts]))
            rec["logits"].append(out[:, :K].reshape(-1))
        return out

    def mobius_prep(*a):
        r, v, pi, w = prep(*a)
        rec["wn"].append(w.norm(dim=-1).reshape(-1))
        return r, v, pi, w

    def mobius_h(z, w):
        h, f = mh(z, w)
        rec["f"].append(f.reshape(-1))
        return h, f

    orc.conditioner, orc._mobius_prep, orc._mobius_h = conditioner, mobius_prep, mobius_h
    try:
        yield rec
    finally:
        orc.conditioner, orc._mobius_prep, orc._mobius_h = cond, prep, mh


def activation_stats(cfg, sd, R, rows, feat, grid_samples=None):
    """fp64: hidden pre-activations over the forward and inverse passes of R (and the forward pass of every image's grid rows)."""
    o = orc.OracleFlow(cfg, sd, torch.float64)
    with _recording(cfg) as rec:
        o.forward(R, rows)
        o.inverse(R, rows)
        if grid_samples is not None:
            B = 1 if feat is None else feat.shape[0]
            o.forward(grid_samples.repeat(B, 1, 1), None if feat is None else feat.repeat_interleave(grid_samples.shape[0], 0))
    a = torch.cat(rec["acts"]).numpy()
    pos = a[a > 0]
    lg = torch.cat(rec["logits"]).numpy()
    f = torch.cat(rec["f"]).numpy()
    return dict(max=float(pos.max()), p10=float(np.percentile(pos, 10)), logits=lg,
                wn_max=float(torch.cat(rec["wn"]).max()), f_min=float(f.min()), f_max=float(f.max()))


def _rescale_k(stats, stat, log2_target):
    if stat == "init":
        return int(log2_target)
    v = math.log2(stats[stat])
    if log2_target == math.log2(6e4):
        return math.floor(math.log2(6e4) - v)                     # just inside 65504 (and SPLIT_LIMIT)
    if log2_target == math.log2(1.1e5):
        return math.ceil(math.log2(SPLIT_LIMIT) - v)              # in [65536, 131072): between 65504 and 2 x 65504
    if log2_target == math.log2(3e5):
        return math.ceil(math.log2(2 * 131008.0) - v)             # beyond both
    return round(log2_target - v)


def stress_case(tag, case):
    """(state dict, k or None) of one stress model, built from the golden weights of ``tag``."""
    key = (tag, case)
    if key not in _case_cache:
        b = _base(tag)
        cfg, sd, k = b["cfg"], b["sd"], None
        resc = {r[0]: r for r in RESCALES}
        if case in resc:
            _, stat, t = resc[case]
            k = _rescale_k(b["stats"], stat, t)
            sd = rescale(cfg, sd, k)
        elif case.startswith("sharp"):
            sd = sharp(cfg, sd, dict(SHARP)[case])
        else:
            sd = logits_at(cfg, sd, below_88=case == "logits_below_88")
        _case_cache[key] = (sd, k)
    return _case_cache[key]


_oracle_cache = {}


def oracle_outputs(tag, case):
    """fp64 and fp32 oracle on the stress inputs: forward and inverse (R, ldj)."""
    key = (tag, case)
    if key not in _oracle_cache:
        b = _base(tag)
        sd, _ = stress_case(tag, case)
        out = {}
        for dt in (torch.float64, torch.float32):
            o = orc.OracleFlow(b["cfg"], sd, dt)
            out[("fwd", dt)] = o.forward(b["R"], b["rows"])
            out[("inv", dt)] = o.inverse(b["R"], b["rows"])
        _oracle_cache[key] = out
    return _oracle_cache[key]


def _row_err(R, ldj, R64, l64):
    dR = (R.double() - R64).abs().amax(dim=(1, 2))
    dl = (ldj.double() - l64).abs() / l64.abs().clamp(min=1.0)
    return dR, dl


def own_error(tag, case, direction="fwd"):
    o = oracle_outputs(tag, case)
    dR, dl = _row_err(*o[(direction, torch.float32)], *o[(direction, torch.float64)])
    return dR, dl


def tolerances(tag, case, mode):
    dR, dl = own_error(tag, case)
    k = OWN_ERROR_FACTOR[mode]
    own_R, own_l = dR.max().item(), dl.max().item()
    return max(1e-5, k * own_R), max(1e-4, k * own_l)


# ---- split emulation (fp32 / fp16, numpy) ---------------------------------------------------------------------------------------
def _f16_rz(x):
    h = x.astype(np.float16)
    over = np.abs(h.astype(np.float32)) > np.abs(x)
    h[over] = np.nextafter(h[over], np.float16(0))
    return h


def split_emulation(x, variant):
    """hi, lo planes (fp16) of non-negative fp32 activations x as the kernels build them.
    'mask':     the kernels' variant: m = x with its low 13 mantissa bits cleared, hi = cvt.rn(m) (no satfinite),
                lo = cvt.rn.satfinite(x - m)
    'mask_sat': the same with hi = cvt.rz.satfinite(x) (the variant before overflow was made loud)
    'convert':  hi = cvt.rz.satfinite(x), lo = cvt.rn.satfinite(x - float(hi))   (the convert-back variant, removed from
                tc_common.cuh; its code is in commit d73682a)"""
    x = np.asarray(x, dtype=np.float32)
    sat = lambda v: np.clip(v, -FP16_MAX, FP16_MAX)
    m = (x.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        if variant == "mask":
            hi = m.astype(np.float16)
            lo = sat(x - m).astype(np.float16)
        elif variant == "mask_sat":
            hi = _f16_rz(sat(x))
            lo = sat(x - m).astype(np.float16)
        else:
            hi = _f16_rz(sat(x))
            lo = sat(x - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def _split_value(x, variant):
    hi, lo = split_emulation(x, variant)
    with np.errstate(invalid="ignore"):
        return hi.astype(np.float64) + lo.astype(np.float64)


# ================================================= CPU ============================================================================
def test_split_emulation_limits():
    """Where hi + lo stops being x to the split's 22 bits, for the three split variants: these are the limits stated in
    DESIGN section 4.1 and in the kernel comments."""
    x = np.concatenate([np.geomspace(2.0 ** -30, 4e5, 400001), np.linspace(65000.0, 140000.0, 150001)]).astype(np.float32)
    x = np.unique(x)
    rel_bound = 2.0 ** -22
    for variant in ("mask", "mask_sat", "convert"):
        v = _split_value(x, variant)
        err = np.abs(v - x) / x
        good = np.isfinite(v) & (err <= rel_bound)
        first_bad_above_1 = x[(x > 1.0) & ~good].min()
        last_bad_below_1 = x[(x < 1.0) & ~good].max()
        # lower end, every variant: lo reaches the fp16 subnormals once x - hi < 2^-14, i.e. for x below 2^-3: hi + lo is then
        # within 2^-25 absolute of x, and within 2^-24 for the mask variants where x < 2^-14 makes hi itself subnormal
        assert 2.0 ** -4 < last_bad_below_1 < 2.0 ** -3, (variant, last_bad_below_1)
        small, tiny = x < 2.0 ** -3, x < 2.0 ** -14
        assert (np.abs(v[small & ~tiny] - x[small & ~tiny]) <= 2.0 ** -25).all(), variant
        assert (np.abs(v[tiny] - x[tiny]) <= (2.0 ** -25 if variant == "convert" else 2.0 ** -24)).all(), variant
        if variant == "mask":
            # exact to the split's precision up to 65536, +Inf from there on: never finite and wrong
            assert first_bad_above_1 == np.float32(65536.0)
            assert np.isinf(v[x >= 65536.0]).all() and np.isfinite(v[x < 65536.0]).all()
        elif variant == "mask_sat":
            # silently clipped: finite and wrong from 65536 on (hi stays 65504, lo is the residual against the unclipped mask)
            assert first_bad_above_1 == np.float32(65536.0)
            big = x >= 65536.0
            assert np.isfinite(v[big]).all() and (v[big] < 65504.0 + x[big] * 2.0 ** -10).all()
        else:
            # full precision up to 65536 only: past it lo = x - 65504 is rounded to 11 bits (relative error up to 1.2e-4 at
            # 131008), and from 131024 on lo saturates too: clipped at 2 x 65504, finite and wrong
            assert 65536.0 <= first_bad_above_1 < 65600.0, first_bad_above_1
            mid = (x >= 65536.0) & (x < 131008.0)
            assert (err[mid] < 2.0 ** -12).all() and err[mid].max() > 2.0 ** -13
            assert np.isfinite(v).all() and v.max() == 2 * FP16_MAX
    record_error(test="split_emulation", rel_bound=rel_bound, mask_exact_below=65536.0, mask_inf_from=65536.0,
                 convert_full_precision_below=float(first_bad_above_1), lo_subnormal_below=0.125)


@pytest.mark.parametrize("tag,case", _all_cases())
def test_transform_reaches_its_regime(tag, case):
    """No stress case is vacuous: the measured activations / centres / logits are where the case name says."""
    b = _base(tag)
    sd, k = stress_case(tag, case)
    st = activation_stats(b["cfg"], sd, b["R"], b["rows"], b["feat"], None)
    resc = {r[0]: r for r in RESCALES}
    if case in resc:
        _, stat, t = resc[case]
        got = math.log2(st[stat]) if stat != "init" else math.log2(st["max"] / b["stats"]["max"])
        record_error(test="regime", case=tag, stress=case, k=k, act_max=st["max"], act_p10=st["p10"])
        assert abs(got - t) <= 1.0, (case, got, t)
        if case == "max_6e4":
            assert _base(tag)["stats"]["max"] * 2.0 ** k < 6e4
        if case in OUTSIDE:
            assert st["max"] >= SPLIT_LIMIT
    elif case == "sharp100":
        assert st["wn_max"] > 0.69
        assert st["f_min"] < 0.25 and st["f_max"] > 4.0, (st["f_min"], st["f_max"])
    elif case == "logits":
        lg = st["logits"]
        for point in (20.0, SERIES_SWITCH):
            assert ((lg > point) & (lg < point + 2e-3)).any() and ((lg < point) & (lg > point - 2e-3)).any(), point
        assert ((lg > -61) & (lg < -59)).any()
        assert ((lg > -4.5) & (lg < -2.5)).any()                   # the band where the series / log2 choice matters
    elif case == "logits_below_88":
        assert st["logits"].max() < -88.0


@pytest.mark.parametrize("tag", FAMILIES + ["symsol2048"])
def test_oracle_invariant_under_rescale(tag):
    """ReLU homogeneity: the fp64 oracle gives the same flow for every rescale(2^k) used here."""
    b = _base(tag)
    ref = oracle_outputs(tag, "max_1")
    for case in [r[0] for r in RESCALES] if tag != "symsol2048" else ["max_6e4", "max_1.1e5"]:
        o = oracle_outputs(tag, case)
        for d in ("fwd", "inv"):
            R, l = o[(d, torch.float64)]
            R0, l0 = ref[(d, torch.float64)]
            assert ((R - R0).abs().max() / R0.abs().max()).item() <= 1e-12, (case, d)
            assert ((l - l0).abs() / l0.abs().clamp(min=1e-300)).max().item() <= 1e-12 or (l - l0).abs().max().item() <= 1e-12, (case, d)


@pytest.mark.parametrize("tag,case", _all_cases())
def test_oracle_own_fp32_error(tag, case):
    """The oracle's own fp32-vs-fp64 error on each stress model: the yardstick of the GPU tolerances (recorded)."""
    dR, dl = own_error(tag, case)
    dRi, _ = own_error(tag, case, "inv")
    record_error(test="oracle_fp32_vs_fp64", case=tag, stress=case, dR=dR.max().item(), dldj=dl.max().item(),
                 inv_rows_within_1e5=(dRi <= 1e-5).float().mean().item())
    assert torch.isfinite(dR).all() and torch.isfinite(dl).all()
    assert dR.max().item() < 1e-3 and dl.max().item() < 1e-3


# ================================================= GPU ============================================================================
def _product(tag, case):
    b = _base(tag)
    sd, _ = stress_case(tag, case)
    m = seeded_product_flow(b["cfg"], 0)
    m.load_state_dict(sd)
    return m.cuda().eval()


def _call(m, fn, R, b, mode):
    f = None if b["feat"] is None else b["feat"].cuda()
    fi = None if b["fi"] is None else b["fi"][:R.shape[0]].cuda()
    with torch.no_grad():
        return getattr(m, fn)(R.cuda(), f, feature_index=fi, mlp_mode=mode)


def _check_rows(tag, case, mode, direction, R, ldj):
    o = oracle_outputs(tag, case)
    R64, l64 = o[(direction, torch.float64)]
    R, ldj = R.cpu(), ldj.cpu()
    dR, dl = _row_err(R, ldj, R64, l64)
    finite = torch.isfinite(R).all(dim=2).all(dim=1) & torch.isfinite(ldj)
    return dR, dl, finite


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("tag,case", _all_cases())
def test_forward_rows(tag, case, mode):
    b = _base(tag)
    m = _product(tag, case)
    R, ldj = _call(m, "forward", b["R"], b, mode)
    dR, dl, finite = _check_rows(tag, case, mode, "fwd", R, ldj)
    tol_R, tol_l = tolerances(tag, case, mode)
    ok = (dR <= tol_R) & (dl <= tol_l)
    fin = finite.all().item()
    record_error(test="ws_forward", case=tag, stress=case, mode=mode, max_abs_dR=dR[finite].max().item() if finite.any() else None,
                 rel_dldj=dl[finite].max().item() if finite.any() else None, nonfinite_rows=int((~finite).sum()),
                 wrong_finite_rows=int((finite & ~ok).sum()), tol_dR=tol_R, tol_dldj=tol_l)
    if case == "logits_below_88" and mode != "fp32":
        assert not finite.any()                                   # all weights flush to zero: NaN, never finite and wrong
    elif case in PRECISION and mode != "fp32":
        bR, bl = PRECISION[case][:2]
        assert case in OUTSIDE or finite.all()
        assert (((dR <= bR) & (dl <= bl)) | ~finite).all()
    else:
        assert fin and ok.all(), (dR.max().item(), dl.max().item(), tol_R, tol_l)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("tag,case", _all_cases())
def test_inverse_rows(tag, case, mode):
    """The inverse's dyadic root: as test_gpu_parity.test_inverse_parity -- as many rows within 1e-5 as the oracle's own fp32 run
    (minus slack), no row further than the flip bound -- on the finite rows; plus ldj on the rows that are within 1e-5."""
    b = _base(tag)
    m = _product(tag, case)
    R, ldj = _call(m, "inverse", b["R"], b, mode)
    dR, dl, finite = _check_rows(tag, case, mode, "inv", R, ldj)
    own, _ = own_error(tag, case, "inv")
    nmob = len(_mobius_prefixes(b["cfg"]))
    frac = (dR[finite] <= 1e-5).float().mean().item() if finite.any() else 1.0
    frac_own = (own <= 1e-5).float().mean().item()
    record_error(test="ws_inverse", case=tag, stress=case, mode=mode, rows_within_1e5=frac, own_rows_within_1e5=frac_own,
                 worst_row=dR[finite].max().item() if finite.any() else None, nonfinite_rows=int((~finite).sum()))
    if case == "logits_below_88" and mode != "fp32":
        assert not finite.any()
        return
    if not (case in OUTSIDE and mode != "fp32"):
        assert finite.all()
    if case in PRECISION and mode != "fp32":
        assert not finite.any() or dR[finite].max().item() <= PRECISION[case][3]
        return
    flip = max(2e-4 * nmob, 1e-5)
    assert frac >= min(frac_own, 0.97) - 0.05
    assert dR[finite].max().item() <= flip
    exact = finite & (dR <= 1e-5)
    if exact.any():
        assert dl[exact].max().item() <= 2e-4


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("tag,case", [(t, c) for t in FAMILIES for c in CASES])
def test_grid_log_prob(tag, case, mode):
    """logp on a ragged level-2 slice (offset, global index 1000), arg-max, max and sumexp per image; Fisher term for s_modelnet.
    An image with a non-finite row must get non-finite reductions, never a maximum taken over its remaining rows."""
    b = _base(tag)
    m = _product(tag, case)
    sd, _ = stress_case(tag, case)
    feat = None if b["feat"] is None else b["feat"].cuda()
    A = b["A"]
    with torch.no_grad():
        out = m.grid_log_prob(b["grid"].cuda(), feat, offset=b["off"].cuda(), fisher_A=None if A is None else A.cuda(),
                              return_logp=True, g_index0=1000, mlp_mode=mode)
    s64 = b["grid"].double() @ b["off"].double()
    G, B = s64.shape[0], 1 if feat is None else feat.shape[0]
    lp = []
    for dt in (torch.float64, torch.float32):
        o = orc.OracleFlow(b["cfg"], sd, dt)
        Rb, l = o.forward(s64.to(dt).repeat(B, 1, 1), None if feat is None else b["feat"].to(dt).repeat_interleave(G, 0))
        if A is not None:
            l = l + orc.fisher_log_prob(A.to(dt), Rb)
        lp.append(l.reshape(B, G).double())
    lp64, lp32 = lp
    own = ((lp32 - lp64).abs() / lp64.abs().clamp(min=1.0)).max().item()
    tol = max(1e-4, OWN_ERROR_FACTOR[mode] * own)
    got = out["logp"].cpu().double()
    err = (got - lp64).abs() / lp64.abs().clamp(min=1.0)
    finite = torch.isfinite(got)
    record_error(test="ws_grid", case=tag, stress=case, mode=mode, rel_dlogp=err[finite].max().item() if finite.any() else None,
                 own_fp32=own, tol=tol, nonfinite=int((~finite).sum()))
    if case == "logits_below_88" and mode != "fp32":
        assert not finite.any()
    elif case in PRECISION and mode != "fp32":
        assert case in OUTSIDE or finite.all()
        tol = PRECISION[case][2]
        assert ((err <= tol) | ~finite).all()
    else:
        assert finite.all() and err.max().item() <= tol, (err.max().item(), tol)
    for bi in range(B):
        k = int(out["argmax"][bi]) - 1000
        assert 0 <= k < G
        if not finite[bi].all():
            # a non-finite log-density reaches the reductions: NaN max and sumexp, arg-max at the first such row
            assert not math.isfinite(float(out["max"][bi])) and not math.isfinite(float(out["sumexp"][bi]))
            assert k == int((~finite[bi]).nonzero()[0])
            continue
        assert k == int(got[bi].argmax())
        assert float(lp64[bi].max() - lp64[bi, k]) <= 2 * tol * max(1.0, float(lp64[bi].abs().max()))
        assert float(out["max"][bi]) == float(out["logp"][bi].max())
        lse = float(out["max"][bi]) + math.log(float(out["sumexp"][bi]))
        ref = float(torch.logsumexp(lp64[bi], 0))
        assert abs(lse - ref) <= tol * max(1.0, abs(ref))
    record_error(test="ws_grid_reductions", case=tag, stress=case, mode=mode, images_with_nonfinite_rows=int((~finite.all(dim=1)).sum()),
                 nonfinite_max=int((~torch.isfinite(out["max"].cpu())).sum()))


def _vee(R, G):
    H = R.transpose(1, 2) @ G
    return torch.stack([H[:, 2, 1] - H[:, 1, 2], H[:, 0, 2] - H[:, 2, 0], H[:, 1, 0] - H[:, 0, 1]], dim=1)


def _rel_to_max(a, ref):
    a, ref = a.detach().cpu().double(), ref.detach().cpu().double()
    return (a - ref).abs().max().item() / max(ref.abs().max().item(), 1e-6)


NG = 128                                        # rows of the gradient tests


def _oracle_grads(tag, case, dt, c, Rg, with_params=True):
    """Autograd through the oracle in dtype dt: logp = ldj [+ Fisher], gradients of sum c_n logp_n."""
    b = _base(tag)
    sd, _ = stress_case(tag, case)
    cfg = b["cfg"]
    o = orc.OracleFlow(cfg, sd, dt)
    names = [n for n, _ in seeded_product_flow(cfg, 0).named_parameters()] if with_params else []
    for n in names:
        o.sd[n] = o.sd[n].clone().requires_grad_(True)
    R2 = Rg.to(dt).clone().requires_grad_(True)
    fi = None if b["fi"] is None else b["fi"][:NG]
    f2 = None if b["feat"] is None else b["feat"].to(dt).clone().requires_grad_(True)
    A2 = None if b["A"] is None else b["A"].to(dt).clone().requires_grad_(True)
    Ro, lp = o.with_grad(R2, None if f2 is None else f2[fi])
    if A2 is not None:
        U, S, V = torch.svd(A2)
        S2 = S[:, 2] * torch.det(U) * torch.det(V)
        S0, S1 = S[:, 0], S[:, 1]
        cst = S0 + S1 + S2 - 0.5 * torch.log(8 * np.pi * (S0 + S1) * (S2 + S1) * (S0 + S2))
        lp = lp + (A2[fi] * Ro).sum(dim=(1, 2)) - cst[fi]
    (c.to(dt) * lp).sum().backward()
    grads = {n: o.sd[n].grad for n in names}
    return lp.detach(), grads, None if f2 is None else f2.grad, _vee(Rg.double(), R2.grad.double()), None if A2 is None else A2.grad


@pytest.mark.gpu
@pytest.mark.parametrize("tag,case", [(t, c) for t, c in _all_cases() if c != "logits_below_88"])
def test_log_prob_grad(tag, case):
    """Flow.log_prob_grad (fp32 CUDA-core kernel) against autograd through the fp64 oracle; tolerance 1e-4 or 4 x the oracle's
    own fp32 error, whichever is larger."""
    b = _base(tag)
    m = _product(tag, case)
    Rg = b["R"][:NG]
    ones = torch.ones(NG, dtype=torch.float64)
    fi = None if b["fi"] is None else b["fi"][:NG].cuda()
    lp, G = m.log_prob_grad(Rg.cuda(), None if b["feat"] is None else b["feat"].cuda(), feature_index=fi,
                            fisher_A=None if b["A"] is None else b["A"].cuda())
    ref = _oracle_grads(tag, case, torch.float64, ones, Rg, with_params=False)
    r32 = _oracle_grads(tag, case, torch.float32, ones, Rg, with_params=False)
    rel_lp = lambda a, r: ((a.cpu().double() - r.double()).abs() / r.double().abs().clamp(min=1.0)).max().item()
    own_lp, own_g = rel_lp(r32[0], ref[0]), _rel_to_max(r32[3], ref[3])
    dl, dg = rel_lp(lp, ref[0]), _rel_to_max(_vee(Rg.double(), G.cpu().double()), ref[3])
    record_error(test="ws_log_prob_grad", case=tag, stress=case, logp_err=dl, grad_rel_err=dg, own_logp=own_lp, own_grad=own_g)
    assert dl <= max(1e-4, 4 * own_lp) and dg <= max(1e-4, 4 * own_g), (dl, dg, own_lp, own_g)


def _fused(m, Rg, b, c):
    m.zero_grad(set_to_none=True)
    R = Rg.clone().cuda().requires_grad_(True)
    f = None if b["feat"] is None else b["feat"].clone().cuda().requires_grad_(True)
    A = None if b["A"] is None else b["A"].clone().cuda().float().requires_grad_(True)
    fi = None if b["fi"] is None else b["fi"][:NG].cuda()
    lp = m.log_prob(R, f, feature_index=fi, fisher_A=A)
    (c.cuda().float() * lp).sum().backward()
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
    return lp.detach(), grads, None if f is None else f.grad, _vee(Rg.cuda().float(), R.grad), None if A is None else A.grad


@pytest.mark.gpu
@pytest.mark.parametrize("tag,case", [(t, c) for t in FAMILIES for c in CASES if c != "logits_below_88"])
def test_log_prob_gradients(tag, case):
    """Flow.log_prob forward + backward (fused training kernels): parameter, feature, fisher_A and rotation gradients against the
    fp64 oracle, each relative to its largest component."""
    b = _base(tag)
    m = _product(tag, case).train()
    Rg = b["R"][:NG]
    c = torch.randn(NG, generator=torch.Generator().manual_seed(77), dtype=torch.float64)
    got = _fused(m, Rg, b, c)
    ref = _oracle_grads(tag, case, torch.float64, c, Rg)
    r32 = _oracle_grads(tag, case, torch.float32, c, Rg)
    worst, where, tol_at = 0.0, "", 0.0
    items = [(n, got[1].get(n), ref[1][n], r32[1][n]) for n in ref[1]]
    items += [(n, a, r, q) for n, a, r, q in (("feature", got[2], ref[2], r32[2]), ("rotation", got[3], ref[3], r32[3]),
                                              ("fisher_A", got[4], ref[4], r32[4])) if r is not None]
    for n, a, r, q in items:
        if r is None or r.abs().max() == 0:
            continue
        assert a is not None, f"no gradient reached {n}"
        e, own = _rel_to_max(a, r), _rel_to_max(q, r)
        tol = max(1e-4, 4 * own)
        if e / tol > worst / max(tol_at, 1e-30):
            worst, where, tol_at = e, n, tol
    dl = ((got[0].cpu().double() - ref[0]).abs() / ref[0].abs().clamp(min=1.0)).max().item()
    own_l = ((r32[0].double() - ref[0]).abs() / ref[0].abs().clamp(min=1.0)).max().item()
    record_error(test="ws_log_prob", case=tag, stress=case, logp_err=dl, grad_rel_err=worst, worst_at=where, tol=tol_at)
    assert dl <= max(1e-4, 4 * own_l)
    assert worst <= tol_at, (where, worst, tol_at)


@pytest.mark.gpu
@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("tag,case", [(t, c) for t in FAMILIES for c in ("max_1", "max_6e4", "sharp100", "logits")])
def test_composed_operators(tag, case, inverse, request):
    """The per-layer differentiable operators (train.composed_run: Flow.forward / Flow.inverse under autograd) against autograd
    through the fp64 oracle, as tests/test_gpu_train.py: values, then parameter / feature / tangential rotation gradients."""
    if (tag, case, inverse) == ("s_symsol", "logits", False):
        # measured on a B200: the layers.3 fc_first.weight gradient is 4.9e-3 from the fp64 oracle (bound 2e-3).  One first-layer
        # pre-activation of that conditioner (row 41, unit 1) is -1.2e-7 in the fp64 oracle and positive in the fp32 forward, so the
        # two take different sides of the ReLU kink, where the gradient is discontinuous.  With the oracle's ReLU branches, the G_out
        # the Mobius kernel returns reproduces the oracle's gradient to 1e-6 (tests/test_train_ops.py
        # test_composed_symsol_logits_localised; DESIGN 4.1).  No bound fits a discontinuity, so this case stays an expected failure.
        request.applymarker(pytest.mark.xfail(strict=True, reason="s_symsol/logits: a layers.3 fc_first pre-activation -1.2e-7 "
                                                                  "from zero takes the other ReLU branch in fp32 (gradient 4.9e-3 off)"))
    b = _base(tag)
    sd, _ = stress_case(tag, case)
    cfg = b["cfg"]
    n = 96
    gen = torch.Generator().manual_seed(77)
    Aw = torch.randn(n, 3, 3, generator=gen, dtype=torch.float64)
    c = torch.randn(n, generator=gen, dtype=torch.float64)
    m = _product(tag, case).train()
    rows = None if b["rows"] is None else b["rows"][:n]
    R = b["R"][:n].clone().cuda().requires_grad_(True)
    f = None if rows is None else rows.clone().cuda().requires_grad_(True)
    out, ldj = (m.inverse if inverse else m)(R, f)
    ((Aw.cuda().float() * out).sum() + (c.cuda().float() * ldj).sum()).backward()
    res = {}
    for dt in (torch.float64, torch.float32):
        o = orc.OracleFlow(cfg, sd, dt)
        names = [k for k, _ in m.named_parameters()]
        for k in names:
            o.sd[k] = o.sd[k].clone().requires_grad_(True)
        R2 = b["R"][:n].to(dt).clone().requires_grad_(True)
        f2 = None if rows is None else rows.to(dt).clone().requires_grad_(True)
        Ro, lo = o.with_grad(R2, f2, inverse=inverse)
        ((Aw.to(dt) * Ro).sum() + (c.to(dt) * lo).sum()).backward()
        res[dt] = (Ro.detach(), {k: o.sd[k].grad for k in names}, None if f2 is None else f2.grad, _vee(b["R"][:n].double(), R2.grad.double()))
    ref, r32 = res[torch.float64], res[torch.float32]
    dR = (out.detach().cpu().double() - ref[0]).abs().amax(dim=(1, 2))
    assert (dR <= 1e-5).float().mean() > (0.9 if inverse else 0.999) and dR.max() < 2e-3
    got = dict(m.named_parameters())
    worst = 0.0
    pairs = [(k, got[k].grad, ref[1][k], r32[1][k]) for k in ref[1] if ref[1][k] is not None]
    pairs += [("feature", None if f is None else f.grad, ref[2], r32[2]), ("rotation", _vee(b["R"][:n].cuda().float(), R.grad), ref[3], r32[3])]
    for k, a, r, q in pairs:
        if r is None or r.abs().max() == 0:
            continue
        assert a is not None, k
        e = _rel_to_max(a, r)
        tol = max(2e-3, 4 * _rel_to_max(q, r))
        worst = max(worst, e / tol)
        assert e <= tol, (k, e, tol)
    record_error(test="ws_composed", case=tag, stress=case, inverse=inverse, worst_err_over_tol=worst)


# ---- exact checks: power-of-two rescaling commutes with fp32 rounding ------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tag", FAMILIES)
def test_fp32_mode_bit_identical_under_rescale(tag):
    """fp32 mode, Flow.log_prob_grad and Flow.log_prob's gradients under rescale(2^k): the flow is bit-identical; the gradients of
    the scaled weights are the unscaled ones x 2^-k (fc_first, biases of layers 1/3/5) or x 2^k (fc_last.weight), bit for bit.
    Conditional flows: the gradients that pass through per-image sums (feature, fisher_A, and the parameters fed by the per-image
    term: fc_first's feature columns, the conditional affine networks) are summed with index_add_, whose atomic adds run in a
    different order on every call; those agree to 1e-6 of their largest component instead of bit for bit."""
    b = _base(tag)
    m0 = _product(tag, "max_1")
    fwd0, inv0 = _call(m0, "forward", b["R"], b, "fp32"), _call(m0, "inverse", b["R"], b, "fp32")
    Rg = b["R"][:NG]
    c = torch.randn(NG, generator=torch.Generator().manual_seed(77), dtype=torch.float64)
    fi = None if b["fi"] is None else b["fi"][:NG].cuda()
    feat = None if b["feat"] is None else b["feat"].cuda()
    A = None if b["A"] is None else b["A"].cuda()
    lpg0 = m0.log_prob_grad(Rg.cuda(), feat, feature_index=fi, fisher_A=A)
    g0 = _fused(m0.train(), Rg, b, c)
    _, k0 = stress_case(tag, "max_1")
    prefixes = _mobius_prefixes(b["cfg"])
    for case in [r[0] for r in RESCALES]:
        m = _product(tag, case)
        _, k = stress_case(tag, case)
        d = k - k0
        for fn, ref in (("forward", fwd0), ("inverse", inv0)):
            out = _call(m, fn, b["R"], b, "fp32")
            assert torch.equal(out[0], ref[0]) and torch.equal(out[1], ref[1]), (case, fn)
        lpg = m.log_prob_grad(Rg.cuda(), feat, feature_index=fi, fisher_A=A)
        assert torch.equal(lpg[0], lpg0[0]) and torch.equal(lpg[1], lpg0[1]), case
        g = _fused(m.train(), Rg, b, c)
        assert torch.equal(g[0], g0[0]) and torch.equal(g[3], g0[3]), case
        near = lambda a, r: _rel_to_max(a, r) <= 1e-6
        for other in (2, 4):
            assert (g[other] is None) or near(g[other], g0[other]), case
        for n, v in g[1].items():
            p = next((p for p in prefixes if n.startswith(p)), None)
            scale = 1.0
            if p is not None:
                tail = n[len(p):]
                if tail in ("fc_first.weight", "fc_first.bias", "layers.1.bias", "layers.3.bias", "layers.5.bias"):
                    scale = 2.0 ** -d
                elif tail == "fc_last.weight":
                    scale = 2.0 ** d
            per_image = b["feat"] is not None and (p is None or n.endswith("fc_first.weight"))
            assert (near if per_image else torch.equal)(v, g0[1][n] * scale), (case, n)


# ---- the inverse's root search on hard mixtures ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tag,case", [(t, c) for t in ("s_symsol", "symsol2048") for c in ("sharp100", "logits_below_88")])
def test_inverse_evaluation_counts(tag, case):
    """Evaluations of the mixture map per row and Mobius layer in the tc_row inverse (the rnf_debug_set_probe_counter hook).  A
    warp whose Newton iteration has not converged in 10 steps falls back to the 15-probe bisection (10 + 15 evaluations): NaN
    rows (every logit below -88) always take it.  For finite sharp mixtures only the mean is recorded: it does not show whether
    any single warp took the fallback, which therefore remains uncovered for finite rows."""
    from rotationnormflow_b200 import _cabi
    _cabi.load()
    lib = ctypes.CDLL(_cabi.library_path())
    lib.rnf_debug_set_probe_counter.argtypes = [ctypes.c_void_p]
    lib.rnf_debug_set_probe_counter.restype = None
    b = _base(tag)
    m = _product(tag, case)
    R = b["R"][:512]                    # whole pairs of 128-row tiles: no padded rows run the root search
    _call(m, "inverse", R, b, "tc_row")
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    lib.rnf_debug_set_probe_counter(ctypes.c_void_p(counter.data_ptr()))
    try:
        _call(m, "inverse", R, b, "tc_row")
        torch.cuda.synchronize()
    finally:
        lib.rnf_debug_set_probe_counter(ctypes.c_void_p(0))
    nmob = len(_mobius_prefixes(b["cfg"]))
    ev = counter.item() / (R.shape[0] * nmob)
    record_error(test="ws_inverse_evaluations", case=tag, stress=case, evaluations_per_row_layer=ev)
    if case == "logits_below_88":
        assert ev == 25.0                                          # every warp: 10 Newton steps, then the 15 probes
    else:
        assert 2.0 <= ev < 25.0
