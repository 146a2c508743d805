"""The differentiable per-layer operators of csrc/train_ops.cu, one at a time, against autograd through the fp64 oracle.

These operators run whenever autograd is on (training through Flow.forward / Flow.inverse, nll_grad, segments != 64, aff_clu):
  MobiusMixture   rnf_train_mobius_forward / _backward, both directions, any K in 1..256, moving column p0 in {0, 1, 2};
  QuatAffine      rnf_train_affine_forward / _backward;
  AblationLayer   rnf_train_ablation_forward / _backward, five kinds.
The flow-level tests bound a gradient against the largest entry of a whole parameter tensor, where a wrong term weighted by one
mixture weight pi_k ~ 1/K can hide.  Here every operator gets fp32 inputs, the reference the same inputs cast to fp64, and every row
of every output and gradient is held to a bound relative to that row's own magnitude:
    bound = max(floor, OWN_ERROR_FACTOR x the fp32 oracle's own error on that row)
with floors of 1e-5 (values) and 1e-4 (gradients).  Each case runs three losses -- on R' only, on the log-det only, on both -- so
that a wrong sign in one cotangent's path cannot hide behind the other.  A gradient row's magnitude is its largest reference entry
under any of the three losses (for the conditioner output: over the whole row, logit and w parts), because under one loss a row
can be zero by structure (the logits of K = 1, the log-length of an orthogonal W, the log-det of M = I) or by a cotangent that
happens to cancel (the mixture sees only the e_p1 component of vee(R'^T G')), and its fp32 rounding noise is no yardstick.  Compared: R', ldj, the tangential rotation gradient
vee(R^T G_R), and the gradient of the operator's other input (the conditioner output's logit and w parts separately, W, M).
The inverse Mobius direction is checked in two parts, so that no fp32 / fp64 bisection flip has to be tolerated: the kernel's root
must be within the final bisection half-width pi/2^15 (plus fp32 slack) of the fp64 root, and values and gradients are compared with
the reference evaluated at the kernel's own root (BinFind.backward's implicit-function gradient there).
Invariants on every case: R' orthonormal with det +1, and R^T G_R antisymmetric (the operators return tangential gradients only).

Without a GPU: the oracle's per-operator references against its flow-level functions, the reachability of the bounds by the fp32
oracle itself, and the C ABI's argument checks."""
import math

import numpy as np
import pytest
import torch

from conftest import golden, record_error
from oracle import rnf_oracle as orc
from oracle.stubs import matrix_to_quaternion
from rotationnormflow_b200 import _cabi, engine, train

OWN_ERROR_FACTOR = 4.0                          # as the fp32 mode in tests/test_weight_scales.py
VALUE_FLOOR, GRAD_FLOOR = 1e-5, 1e-4
# A row whose reference is below this in every entry is all fp32 subnormals (logits at -100: softplus 3.7e-44) and carries nothing;
# its error is taken against this magnitude instead of its own.
TINY = 1e-30
ROOT_HALF_WIDTH = math.pi / 2 ** 15             # the 15-halving bisection's last midpoint is this close to the bracketed root
ROOT_SLACK = 2e-5                               # fp32 evaluation of Theta near the root (checked against the fp32 oracle on the CPU)
ORTHO_TOL, ANTISYM_TOL = 2e-6, 1e-6
# Bounds widened from measurement (one B200, 1000 W power limit): case -> (own-error factor, gradient floor), each with its reason.
PRECISION = {
    # theta = sum_k sp_k theta_k / S is summed in sequence over K components in fp32 (the oracle sums pairwise): R' carries those
    # rounding errors, and a gradient row whose contraction of the cotangent with R' cancels inherits them.  Measured: 1.3e-4 of
    # the row at K = 255, forward (K <= 128: within 1e-4).
    "mobius_K>128": (OWN_ERROR_FACTOR, 2e-4),
    # |W q| = 1e-3 is the cancellation of O(1) terms: the rounding of the fp32 quaternion (the kernel's and the oracle's extraction
    # formulas round differently) is amplified 1e3 x into R'.  Measured: R' 4.8 x the fp32 oracle's own error.
    "quat_affine_near_kernel": (8.0, GRAD_FLOOR),
    # 6 x 6 M, then the log-det of the tangent frame through two normalisations: measured 5.5 x the fp32 oracle's own ldj error and
    # 5 x on its gradients (singular values 1e-3 apart, and repeated).
    "smith36": (8.0, GRAD_FLOOR),
}

KS = [1, 2, 3, 63, 64, 65, 128, 255, 256]
NS = [1, 127, 128, 129, 1000]
OUTS = ["random", "w_zero", "w_parallel_y", "w_1e4", "logits_equal", "straddle_20", "straddle_series", "one_at_30"]
SERIES_SWITCH = -7.0 * math.log(2.0)            # the softplus series branch of the fused kernels' fast paths (a = -4.852)


def stress_inputs(n=512, seed=0):
    """n Haar rotations, the identity, the 24 rotations with entries in {0, +-1}, 16 rotations by pi about random axes (quaternion
    real part 0: ties between the candidates of matrix_to_quaternion) and the same 16 perturbed by one fp32 ulp.  (A copy of the
    helper in tests/test_weight_scales.py.)"""
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


N_SPECIAL = 57                                  # the rows of stress_inputs after the Haar ones


def rotations(N):
    """N rows of stress_inputs, the special rotations last: every N >= 57 contains all of them."""
    return stress_inputs(max(N - N_SPECIAL, 0))[-N:] if N > 0 else torch.empty(0, 3, 3)


def _logit_pattern(j, K=64):
    """As tests/test_weight_scales.py _logit_pattern: j = 0 straddles a = 20 (+-1e-3) and sits at -60 next to O(1) logits, j = 1
    straddles the series switch -4.852 and fills -5.5 .. -1.5."""
    b = np.empty(K)
    pm = np.where(np.arange(16) % 2 == 0, 1e-3, -1e-3)
    if j == 0:
        b[:16] = 20.0 + pm
        b[16:24] = -60.0 + np.linspace(-0.5, 0.5, 8)
        b[24:] = np.linspace(-2.0, 2.0, 40)
    else:
        b[:16] = SERIES_SWITCH + pm
        b[16:] = np.linspace(-5.5, -1.5, 48)
    return torch.from_numpy(b)


def make_out(kind, R, p0, K, seed=0):
    """Conditioner output [N,4K] (logits, then w_k at K + 3k) in fp32: random O(1) values with the named edge on component 0 (or on
    the logits)."""
    N = R.shape[0]
    gen = torch.Generator().manual_seed(1000 + seed)
    a = torch.randn(N, K, generator=gen, dtype=torch.float64)
    w = torch.randn(N, K, 3, generator=gen, dtype=torch.float64)
    y = R.double()[:, :, (p0 + 1) % 3]
    if kind == "w_zero":
        w[:, 0] = 0.0                                           # the n > 1e-30 guard of the squash Jacobian
    elif kind == "w_parallel_y":
        w[:, 0] = 1.5 * y                                       # projects to (almost) zero in the plane orthogonal to y
    elif kind == "w_1e4":
        w[:, 0] = 1e4 * w[:, 0] / w[:, 0].norm(dim=-1, keepdim=True)   # w' -> 0.7 |w| / (1 + |w|): f_k up to 5.7
    elif kind == "logits_equal":
        a[:] = 0.3
    elif kind in ("straddle_20", "straddle_series"):
        assert K == 64
        a = _logit_pattern(0 if kind == "straddle_20" else 1)[None].expand(N, K) + 1e-5 * a
    elif kind == "one_at_30":
        a[:] = -100.0                                           # softplus(-100) = 3.7e-44: an fp32 subnormal
        a[:, 0] = 30.0
    return torch.cat([a, w.reshape(N, 3 * K)], dim=1).float()


# ---- comparisons ----------------------------------------------------------------------------------------------------------------
def _vee(R, G):
    H = R.transpose(1, 2) @ G
    return torch.stack([H[:, 2, 1] - H[:, 1, 2], H[:, 0, 2] - H[:, 2, 0], H[:, 1, 0] - H[:, 0, 1]], dim=1)


def row_ratio(got, r64, r32, floor, scale=None, factor=OWN_ERROR_FACTOR):
    """Per row: error against the fp64 reference over max(floor, factor x the fp32 oracle's error), both relative to the row's
    magnitude (largest reference entry of the row, or ``scale``)."""
    got, r64, r32 = (t.detach().cpu().double().reshape(t.shape[0], -1) for t in (got, r64, r32))
    s = r64.abs().amax(1) if scale is None else scale
    s = s.clamp(min=TINY)
    err = (got - r64).abs().amax(1) / s
    own = (r32 - r64).abs().amax(1) / s
    bound = (factor * own).clamp(min=floor)
    return torch.where(torch.isfinite(err), err / bound, torch.full_like(err, math.inf)), err, bound


class Report:
    """Worst err / bound per compared quantity of one case; fails on any row over its bound."""

    def __init__(self, **case):
        self.case, self.rows = case, {}

    def add(self, name, got, r64, r32, floor, scale=None, factor=OWN_ERROR_FACTOR):
        if got.shape[0] == 0:
            return
        ratio, err, bound = row_ratio(got, r64, r32, floor, scale, factor)
        i = int(torch.argmax(torch.nan_to_num(ratio, nan=math.inf)))
        self.rows[name] = (float(ratio[i]), float(err[i]), float(bound[i]), i)

    def check(self):
        record_error(test="train_ops", **self.case, worst=self.rows)
        bad = {k: v for k, v in self.rows.items() if not v[0] <= 1.0}
        assert not bad, f"{self.case}: (err/bound, err, bound, row) {bad}"


def check_invariants(R, R_out, G_R, what):
    """R' orthonormal with det +1; R^T G_R antisymmetric (a purely tangential rotation gradient)."""
    Ro = R_out.detach().cpu().double()
    if Ro.shape[0] == 0:
        return
    eye = torch.eye(3, dtype=torch.float64)
    assert ((Ro.transpose(1, 2) @ Ro - eye).abs().amax(dim=(1, 2)) <= ORTHO_TOL).all(), what
    assert ((torch.linalg.det(Ro) - 1.0).abs() <= ORTHO_TOL).all(), what
    H = R.detach().cpu().double().transpose(1, 2) @ G_R.detach().cpu().double()
    sym = 0.5 * (H + H.transpose(1, 2))
    hn = H.flatten(1).norm(dim=1)
    assert (sym.flatten(1).norm(dim=1) <= ANTISYM_TOL * hn + TINY).all(), what


def loss_scale(ref, idx, cols=None):
    """Per row: the largest entry of gradient ``idx`` of a _reference result over all losses (columns ``cols`` of it)."""
    g = [v[idx] for v in ref[2].values()]
    return torch.stack([t.reshape(t.shape[0], -1)[:, cols or slice(None)].abs().amax(1) for t in g]).amax(0)


def _cotangents(N, seed):
    gen = torch.Generator().manual_seed(seed)
    A = torch.randn(N, 3, 3, generator=gen, dtype=torch.float64)
    c = torch.randn(N, generator=gen, dtype=torch.float64)
    z3, z = torch.zeros_like(A), torch.zeros_like(c)
    return {"R": (A, z), "ldj": (z3, c), "both": (A, c)}


def _grads(outs, ins, A, c):
    """d/d ins of <A, R'> + <c, ldj> (zeros where the loss does not depend on an input)."""
    R_out, ldj = outs
    loss = (A.to(R_out.device, R_out.dtype) * R_out).sum() + (c.to(ldj.device, ldj.dtype) * ldj).sum()
    if not loss.requires_grad:
        return [torch.zeros_like(t) for t in ins]
    g = torch.autograd.grad(loss, ins, retain_graph=True, allow_unused=True)
    return [torch.zeros_like(t) if gi is None else gi for t, gi in zip(ins, g)]


def _reference(fn, R, X, losses, dtypes=(torch.float64, torch.float32)):
    """Autograd through the oracle's operator fn(R, X) -> (R', ldj) on the fp32 inputs cast to each dtype: values and, per loss,
    the tangential rotation gradient and the gradient of X."""
    res = {}
    for dt in dtypes:
        R2 = R.to(dt).clone().requires_grad_(True)
        X2 = X.to(dt).clone().requires_grad_(True)
        Ro, l = fn(R2, X2)
        g = {}
        for name, (A, c) in losses.items():
            GR, GX = _grads((Ro, l), (R2, X2), A, c)
            g[name] = (_vee(R.double(), GR.double()), GX)
        res[dt] = (Ro.detach(), l.detach(), g)
    return res


# ---- Mobius mixture -------------------------------------------------------------------------------------------------------------
def _root64(R, out, p0, K, halvings=60):
    """The fp64 root of Theta(x) = y* in BinFind's bracket [pi/2, 3 pi/2], bisected to fp64 resolution with BinFind's update."""
    p = orc.PERMUTE_TABLE[p0]
    R, out = R.double(), out.double()
    x, y = R[:, :, p[0]], R[:, :, p[1]]
    r, v, pi, w = orc.mobius_params(out, x, y, K)
    tt = orc._target_angle(x, r, v)
    a = torch.full_like(tt, math.pi / 2)
    b = torch.full_like(tt, 1.5 * math.pi)
    for _ in range(halvings):
        x0 = (a + b) / 2
        lower = orc._theta_of(x0, r, v, pi, w) - tt < 0
        a, b = torch.where(lower, x0, a), torch.where(lower, b, x0)
    return ((a + b) / 2)[:, 0]


def mobius_layer_fn(p0, K, inverse, root=None):
    return lambda R, out: orc.mobius_layer(R, out, p0, K, inverse, root=root)


def run_mobius(R, out, p0, K, inverse, cotangents=None, seed=7):
    """MobiusMixture (train.py) on the device at fp32 inputs, against autograd through orc.mobius_layer in fp64 (and fp32 for the
    bounds) on the same inputs; the inverse at the kernel's own root, which must bracket the fp64 root.  ``cotangents``: {loss:
    (G_R', g_ldj)} applied as given instead of the three random losses."""
    N = R.shape[0]
    losses = _cotangents(N, seed) if cotangents is None else cotangents
    Rd = R.cuda().requires_grad_(True)
    od = out.cuda().requires_grad_(True)
    R_out, ldj = train.MobiusMixture.apply(Rd, od, p0, inverse, K)
    theta = ldj.grad_fn.saved_tensors[2].cpu()                 # the root (inverse) / mixture angle (forward) the backward uses
    got = {name: _grads((R_out, ldj), (Rd, od), A, c) for name, (A, c) in losses.items()}
    rep = Report(op="mobius", direction="inverse" if inverse else "forward", K=K, N=N, p0=p0)
    factor, gfloor = PRECISION["mobius_K>128"] if K > 128 else (OWN_ERROR_FACTOR, GRAD_FLOOR)
    root = None
    if inverse:
        root = theta.double()
        if N:
            dist = (root - _root64(R, out, p0, K)).abs()
            rep.rows["root"] = (float(dist.max() / (ROOT_HALF_WIDTH + ROOT_SLACK)), float(dist.max()), ROOT_HALF_WIDTH + ROOT_SLACK,
                                int(dist.argmax()))
    ref = _reference(mobius_layer_fn(p0, K, inverse, root), R, out, losses)
    r64, r32 = ref[torch.float64], ref[torch.float32]
    rep.add("R'", R_out, r64[0], r32[0], VALUE_FLOOR, scale=torch.ones(N, dtype=torch.float64))
    rep.add("ldj", ldj, r64[1], r32[1], VALUE_FLOOR, scale=r64[1].abs().clamp(min=1.0))
    s_rot, s_out = loss_scale(r64, 0), loss_scale(r64, 1)
    for name in losses:
        GR, Go = got[name]
        check_invariants(R, R_out, GR, (rep.case, name))
        g64, g32 = r64[2][name], r32[2][name]
        rep.add(f"{name}:vee(R^T G_R)", _vee(R.double(), GR.cpu().double()), g64[0], g32[0], gfloor, s_rot, factor)
        rep.add(f"{name}:G_logit", Go[:, :K], g64[1][:, :K], g32[1][:, :K], gfloor, s_out, factor)
        rep.add(f"{name}:G_w", Go[:, K:], g64[1][:, K:], g32[1][:, K:], gfloor, s_out, factor)
    rep.check()
    return dict(R_out=R_out.detach(), ldj=ldj.detach(), theta=theta, got=got, ref=ref, report=rep)


# ================================================= CPU ============================================================================
def _golden_layer(tag, i):
    g = golden(tag)
    sd = {k: v.double() for k, v in g.state_dict().items()}
    p = orc.PERMUTE_TABLE[orc.permute_rows(g.cfg, orc.layer_plan(g.cfg))[i]]
    return g, sd, p


@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("tag", ["s_symsol", "s_uncond"])
def test_mobius_layer_is_the_flow_layer(tag, inverse):
    """orc.mobius_layer on the conditioner's output is orc.mobius_forward / mobius_inverse of that layer, bit for bit, gradients
    included; and its inverse at a given root equals the bisection's when given the bisection's root."""
    g, sd, _ = _golden_layer(tag, 0)
    i = orc.layer_plan(g.cfg).index("mobius")
    p = orc.PERMUTE_TABLE[orc.permute_rows(g.cfg, orc.layer_plan(g.cfg))[i]]
    assert p in orc.PERMUTE_TABLE[:3]
    p0 = orc.PERMUTE_TABLE.index(p)
    K = g.cfg.segments
    R = g.R[:40].double()
    feat = None if g.rows is None else g.rows[:40].double()
    fn = orc.mobius_inverse if inverse else orc.mobius_forward
    gen = torch.Generator().manual_seed(3)
    A, c = torch.randn(40, 3, 3, generator=gen, dtype=torch.float64), torch.randn(40, generator=gen, dtype=torch.float64)
    R1 = R.clone().requires_grad_(True)
    Ro1, l1 = fn(sd, f"layers.{i}.", R1, p, feat, K)
    ((A * Ro1).sum() + (c * l1).sum()).backward()
    R2 = R.clone().requires_grad_(True)
    inp = R2[:, :, p[1]] if feat is None else torch.cat((R2[:, :, p[1]], feat), -1)
    out = orc.conditioner(sd, f"layers.{i}.conditioner.", inp)
    Ro2, l2 = orc.mobius_layer(R2, out, p0, K, inverse)
    ((A * Ro2).sum() + (c * l2).sum()).backward()
    assert torch.equal(Ro1, Ro2) and torch.equal(l1, l2)
    assert torch.equal(R1.grad, R2.grad)
    if inverse:
        x, y = R[:, :, p[0]], R[:, :, p[1]]
        r, v, pi, w = orc.mobius_params(out.detach(), x, y, K)
        root = orc.bisect(orc._target_angle(x, r, v), r, v, pi, w)[:, 0]
        R3 = R.clone().requires_grad_(True)
        out3 = out.detach().clone().requires_grad_(True)
        Ro3, l3 = orc.mobius_layer(R3, out3, p0, K, True, root=root)
        ((A * Ro3).sum() + (c * l3).sum()).backward()
        assert torch.equal(Ro3, Ro2) and torch.equal(l3, l2)
        out4 = out.detach().clone().requires_grad_(True)
        Ro4, l4 = orc.mobius_layer(R.clone().requires_grad_(True), out4, p0, K, True)
        ((A * Ro4).sum() + (c * l4).sum()).backward()
        assert torch.equal(out3.grad, out4.grad)


@pytest.mark.parametrize("kind", ["random", "straddle_20", "w_1e4", "one_at_30"])
@pytest.mark.parametrize("p0", [0, 1, 2])
def test_fp32_oracle_meets_the_root_bound(p0, kind):
    """The root part of the inverse check is attainable: the fp32 oracle's own 15-halving bisection lands within pi/2^15 + the fp32
    slack of the fp64 root on the stress rotations."""
    R = rotations(300)
    K = 64
    out = make_out(kind, R, p0, K)
    p = orc.PERMUTE_TABLE[p0]
    x, y = R[:, :, p[0]], R[:, :, p[1]]
    r, v, pi, w = orc.mobius_params(out, x, y, K)
    th32 = orc.bisect(orc._target_angle(x, r, v), r, v, pi, w)[:, 0].double()
    dist = (th32 - _root64(R, out, p0, K)).abs()
    assert dist.max().item() <= ROOT_HALF_WIDTH + ROOT_SLACK, dist.max().item()


def test_make_out_reaches_its_edges():
    """The conditioner outputs of the cases are where their names say (fp64, on the stress rotations)."""
    R = rotations(200)
    for p0 in (0, 1, 2):
        y = R.double()[:, :, (p0 + 1) % 3]
        for kind in OUTS:
            out = make_out(kind, R, p0, 64).double()
            a, w = out[:, :64], out[:, 64:].reshape(-1, 64, 3)
            wp = w - (w * y[:, None]).sum(-1, keepdim=True) * y[:, None]
            if kind == "w_zero":
                assert (w[:, 0] == 0).all()
            elif kind == "w_parallel_y":
                assert (wp[:, 0].norm(dim=-1) < 1e-6).all()
            elif kind == "w_1e4":
                assert (0.69 < 0.7 * wp[:, 0].norm(dim=-1) / (1 + wp[:, 0].norm(dim=-1))).all()
            elif kind == "straddle_20":
                assert ((a > 20) & (a < 20.002)).any(1).all() and ((a < 20) & (a > 19.998)).any(1).all()
                assert ((a > -61) & (a < -59)).any(1).all()
            elif kind == "straddle_series":
                assert ((a > SERIES_SWITCH) & (a < SERIES_SWITCH + 2e-3)).any(1).all()
                assert ((a < SERIES_SWITCH) & (a > SERIES_SWITCH - 2e-3)).any(1).all()
            elif kind == "one_at_30":
                sp = torch.nn.functional.softplus(a.float())
                assert (sp[:, 1:] < 1e-38).all() and (sp[:, 1:] > 0).all()       # fp32 subnormal weights


def test_train_abi_argument_errors_without_gpu():
    """rnf_train_mobius_* / rnf_train_affine_*: K, perm and N are checked before the device, so a bad call is reported as such on
    any host."""
    lib = _cabi.load()
    assert lib.rnf_train_max_components() == 256
    RNF_EINVAL, RNF_ESHAPE = -1, -2
    fwd = lambda N, K, perm: lib.rnf_train_mobius_forward(None, None, N, K, perm, 0, None, None, None, None)
    bwd = lambda N, K, perm: lib.rnf_train_mobius_backward(None, None, N, K, perm, 1, None, None, None, None, None, None, None)
    for call in (fwd, bwd):
        for K in (0, 257, -1):
            assert call(4, K, 0) == RNF_ESHAPE, K
            assert b"mixture components" in lib.rnf_last_error()
        for perm in (3, -1):
            assert call(4, 64, perm) == RNF_EINVAL, perm
            assert b"perm" in lib.rnf_last_error()
        assert call(-1, 64, 0) == RNF_EINVAL
        assert b"negative N" in lib.rnf_last_error()
    assert lib.rnf_train_affine_forward(None, None, -1, None, None, None) == RNF_EINVAL
    assert lib.rnf_train_affine_backward(None, None, -1, None, None, None, None, None, None) == RNF_EINVAL
    assert b"negative N" in lib.rnf_last_error()


# ================================================= GPU: Mobius ====================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("p0", [0, 1, 2])
@pytest.mark.parametrize("K", KS)
def test_mobius_components(K, p0, inverse):
    """K from 1 to the kMaxK bound of 256 (local arrays of the inverse), across 2 blocks (129 rows) of stress rotations."""
    R = rotations(129)
    run_mobius(R, make_out("random", R, p0, K, seed=K), p0, K, inverse)


@pytest.mark.gpu
@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("N", NS)
def test_mobius_rows(N, inverse):
    """1 row, a block but one, one block, a block and one row, and 7 full blocks followed by a partial one."""
    p0 = N % 3
    R = rotations(N)
    run_mobius(R, make_out("random", R, p0, 64, seed=N), p0, 64, inverse)


@pytest.mark.gpu
@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("p0", [0, 1, 2])
@pytest.mark.parametrize("kind", OUTS)
def test_mobius_edges(kind, p0, inverse):
    """Conditioner outputs at the edges of the mixture math (w = 0, w parallel to y, |w| = 1e4, equal logits, logits across the
    softplus threshold 20 and the series switch, one logit at 30 and the others at -100) on all stress rotations."""
    R = rotations(585)
    run_mobius(R, make_out(kind, R, p0, 64), p0, 64, inverse)


@pytest.mark.gpu
def test_empty_and_null_buffers():
    """N = 0 is a no-op returning empty tensors (all three operators, both directions); a null buffer with N > 0 is RNF_EINVAL."""
    R0 = torch.empty(0, 3, 3, device="cuda", requires_grad=True)
    for inverse in (False, True):
        o = torch.empty(0, 4 * 5, device="cuda", requires_grad=True)
        Ro, l = train.MobiusMixture.apply(R0, o, 1, inverse, 5)
        assert Ro.shape == (0, 3, 3) and l.shape == (0,)
        (Ro.sum() + l.sum()).backward()
    W = torch.empty(0, 4, 4, device="cuda", requires_grad=True)
    Ro, l = train.QuatAffine.apply(R0, W)
    assert Ro.shape == (0, 3, 3) and l.shape == (0,)
    (Ro.sum() + l.sum()).backward()
    for kind, n in ((_cabi.RNF_LAYER_SMITH9, 3), (_cabi.RNF_LAYER_SMITH36, 6), (_cabi.RNF_LAYER_POLAR9R, 3)):
        M = torch.empty(0, n, n, device="cuda", requires_grad=True)
        Ro, l = train.AblationLayer.apply(R0, M, kind)
        assert Ro.shape == (0, 3, 3) and l.shape == (0,)
        (Ro.sum() + l.sum()).backward()
    lib = _cabi.load()
    buf = torch.zeros(4 * 9 * 64, device="cuda")
    p = buf.data_ptr()
    assert lib.rnf_train_mobius_forward(p, None, 4, 16, 0, 0, p, p, p, None) == -1
    assert lib.rnf_train_mobius_backward(p, p, 4, 16, 0, 1, p, p, p, p, None, p, None) == -1
    assert lib.rnf_train_affine_forward(p, p, 4, None, p, None) == -1
    assert lib.rnf_train_affine_backward(p, p, 4, p, p, p, p, None, None) == -1
    assert b"null buffer" in lib.rnf_last_error()
    torch.cuda.synchronize()


# ================================================= GPU: quaternion affine ========================================================
def _rand_orth(n, dim, gen):
    Q, Rr = torch.linalg.qr(torch.randn(n, dim, dim, generator=gen, dtype=torch.float64))
    Q = Q * torch.sign(torch.diagonal(Rr, dim1=-2, dim2=-1))[:, None, :]
    flip = torch.linalg.det(Q) < 0
    Q[flip, :, 0] *= -1.0
    return Q


def affine_W(kind, R, seed=0):
    N = R.shape[0]
    gen = torch.Generator().manual_seed(2000 + seed)
    eye = torch.eye(4, dtype=torch.float64)
    if kind == "identity":
        W = eye.expand(N, 4, 4)
    elif kind == "orthogonal":
        W = _rand_orth(1, 4, gen).expand(N, 4, 4)
    elif kind == "cond1e3":
        U, V = _rand_orth(1, 4, gen), _rand_orth(1, 4, gen)
        W = (U @ torch.diag(torch.tensor([1.0, 0.3, 0.03, 1e-3], dtype=torch.float64)) @ V.transpose(1, 2)).expand(N, 4, 4)
    elif kind == "near_kernel":
        # W_n = O (I - (1 - 1e-3) q q^T) with q the row's quaternion: |W q| = 1e-3, the other directions unchanged
        q = matrix_to_quaternion(R.double())
        O = _rand_orth(1, 4, gen)
        W = O @ (eye - (1.0 - 1e-3) * q[:, :, None] * q[:, None, :])
    else:                                                      # "per_row"
        W = eye + 0.5 * torch.randn(N, 4, 4, generator=gen, dtype=torch.float64)
    return W.contiguous().float()


def quat_affine_loglen(R, W):
    """orc.quat_affine with the log-length instead of the log-det: (R', log|W q|) = (R', (log|det W| - ldj) / 4)."""
    Rt, ldj = orc.quat_affine(W, R)
    return Rt, (orc.det4(W).abs().log() - ldj) / 4.0


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["identity", "orthogonal", "cond1e3", "near_kernel", "per_row"])
def test_quat_affine(kind):
    R = rotations(585)
    N = R.shape[0]
    W = affine_W(kind, R)
    losses = _cotangents(N, 11)
    Rd, Wd = R.cuda().requires_grad_(True), W.cuda().requires_grad_(True)
    R_out, loglen = train.QuatAffine.apply(Rd, Wd)
    ref = _reference(quat_affine_loglen, R, W, losses)
    r64, r32 = ref[torch.float64], ref[torch.float32]
    rep = Report(op="quat_affine", case=kind, N=N)
    factor, gfloor = PRECISION.get(f"quat_affine_{kind}", (OWN_ERROR_FACTOR, GRAD_FLOOR))
    rep.add("R'", R_out, r64[0], r32[0], VALUE_FLOOR, torch.ones(N, dtype=torch.float64), factor)
    rep.add("loglen", loglen, r64[1], r32[1], VALUE_FLOOR, r64[1].abs().clamp(min=1.0), factor)
    s_rot, s_W = loss_scale(r64, 0), loss_scale(r64, 1)
    for name, (A, c) in losses.items():
        GR, GW = _grads((R_out, loglen), (Rd, Wd), A, c)
        check_invariants(R, R_out, GR, (kind, name))
        rep.add(f"{name}:vee(R^T G_R)", _vee(R.double(), GR.cpu().double()), r64[2][name][0], r32[2][name][0], gfloor, s_rot, factor)
        rep.add(f"{name}:G_W", GW, r64[2][name][1], r32[2][name][1], gfloor, s_W, factor)
    rep.check()


# ================================================= GPU: ablation layers ==========================================================
ABL = {"smith9": (_cabi.RNF_LAYER_SMITH9, 3), "smith36": (_cabi.RNF_LAYER_SMITH36, 6), "polar9l": (_cabi.RNF_LAYER_POLAR9L, 3),
       "polar9r": (_cabi.RNF_LAYER_POLAR9R, 3), "right9": (_cabi.RNF_LAYER_RIGHT9, 3)}


def ablation_reference(kind):
    """The oracle's layer for the matrix the operator receives (train._ablation_matrix): right9 gets the Gram-Schmidt factor Q
    itself, so its operator is R Q."""
    if kind == "smith9":
        return orc.smith9
    if kind == "smith36":
        return orc.smith36
    if kind in ("polar9l", "polar9r"):
        return lambda M, R: orc.polar9(M, R, kind == "polar9l")
    return lambda M, R: (R @ M, torch.zeros(R.shape[0], dtype=R.dtype))


def ablation_M(kind, case, N, seed=0):
    n = ABL[kind][1]
    gen = torch.Generator().manual_seed(3000 + seed)
    eye = torch.eye(n, dtype=torch.float64)
    if case == "identity":
        M = eye.expand(N, n, n).clone()
    elif case == "random":
        # 0.15 keeps the smallest singular value of every row above 0.1 (I + 0.5 randn reaches 1e-4: near singular, its own regime)
        M = eye + 0.15 * torch.randn(N, n, n, generator=gen, dtype=torch.float64)
        M[torch.linalg.det(M) < 0, :, 0] *= -1.0               # keep the polar factor proper
    else:                                                      # singular values 1e-3 apart, or exactly repeated
        s = torch.tensor([1.0, 1.0 + (1e-3 if case == "gap1e-3" else 0.0), 0.9, 0.8, 0.7, 0.6][:n], dtype=torch.float64)
        M = _rand_orth(N, n, gen) @ torch.diag(s) @ _rand_orth(N, n, gen).transpose(1, 2)
    if kind == "right9":
        M = engine.gram_schmidt_columns(M)
    return M.contiguous().float()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["identity", "random", "gap1e-3", "repeated"])
@pytest.mark.parametrize("kind", list(ABL))
def test_ablation_layer(kind, case):
    R = rotations(585)
    N = R.shape[0]
    M = ablation_M(kind, case, N)
    code = ABL[kind][0]
    losses = _cotangents(N, 13)
    Rd, Md = R.cuda().requires_grad_(True), M.cuda().requires_grad_(True)
    R_out, ldj = train.AblationLayer.apply(Rd, Md, code)
    got = {name: _grads((R_out, ldj), (Rd, Md), A, c) for name, (A, c) in losses.items()}
    for name, (GR, GM) in got.items():
        assert torch.isfinite(R_out).all() and torch.isfinite(ldj).all() and torch.isfinite(GR).all() and torch.isfinite(GM).all()
        check_invariants(R, R_out, GR, (kind, case, name))
    if case in ("identity", "repeated") and kind.startswith("polar"):
        return                         # a repeated singular value (M R of M = I is orthogonal): torch.svd's backward is NaN there
    ref = _reference(lambda R2, M2: ablation_reference(kind)(M2, R2), R, M, losses)
    r64, r32 = ref[torch.float64], ref[torch.float32]
    rep = Report(op="ablation", kind=kind, case=case, N=N)
    factor, gfloor = PRECISION.get(kind, (OWN_ERROR_FACTOR, GRAD_FLOOR))
    rep.add("R'", R_out, r64[0], r32[0], VALUE_FLOOR, torch.ones(N, dtype=torch.float64), factor)
    rep.add("ldj", ldj, r64[1], r32[1], VALUE_FLOOR, r64[1].abs().clamp(min=1.0), factor)
    s_rot, s_M = loss_scale(r64, 0), loss_scale(r64, 1)
    for name in losses:
        GR, GM = got[name]
        rep.add(f"{name}:vee(R^T G_R)", _vee(R.double(), GR.cpu().double()), r64[2][name][0], r32[2][name][0], gfloor, s_rot, factor)
        rep.add(f"{name}:G_M", GM, r64[2][name][1], r32[2][name][1], gfloor, s_M, factor)
    rep.check()


# ================================================= GPU: the composed path on the logit stress model ===============================
def _masked_conditioner(sd, prefix, x, masks):
    """orc.conditioner with each ReLU replaced by the given 0/1 mask (the branch the evaluation took)."""
    lin = torch.nn.functional.linear
    h0 = lin(x, sd[prefix + "fc_first.weight"], sd[prefix + "fc_first.bias"])
    h = h0
    for j, m in zip((1, 3, 5), masks[:3]):
        h = lin(h * m, sd[f"{prefix}layers.{j}.weight"], sd[f"{prefix}layers.{j}.bias"])
    return lin((h0 + h) * masks[3], sd[prefix + "fc_last.weight"], sd[prefix + "fc_last.bias"])


def _relu_masks(sd, prefix, x):
    """The four ReLU branches of orc.conditioner at x, and the pre-activations."""
    lin = torch.nn.functional.linear
    h0 = lin(x, sd[prefix + "fc_first.weight"], sd[prefix + "fc_first.bias"])
    pre, h = [h0], h0
    for j in (1, 3, 5):
        h = lin(torch.relu(h), sd[f"{prefix}layers.{j}.weight"], sd[f"{prefix}layers.{j}.bias"])
        pre.append(h if j != 5 else h0 + h)
    return [(p > 0).to(x.dtype) for p in pre], pre


@pytest.mark.gpu
def test_composed_symsol_logits_localised(monkeypatch):
    """The s_symsol / logits case of test_weight_scales.test_composed_operators (forward), layer by layer.
    1. Records each Mobius operator's inputs and the cotangents it receives in the composed run, and holds the operator to the
       per-row bounds at exactly those fp32 tensors.
    2. Pushes the G_out the kernel handed to each conditioner through the fp64 conditioner backward at the recorded fp32 inputs,
       once with the ReLU branches the device's fp32 forward took and once with those of the fp64 oracle at its own inputs.  With
       the device's branches it is the product's gradient; with the oracle's it is the oracle's within the composed bound.  So
       what separates the composed path from the oracle is which side of a ReLU kink a pre-activation next to zero falls on --
       the gradient is discontinuous there -- and neither the operators nor the torch conditioner backward."""
    import test_weight_scales as ws
    tag, case, n = "s_symsol", "logits", 96
    b = ws._base(tag)
    sd, _ = ws.stress_case(tag, case)
    gen = torch.Generator().manual_seed(77)
    Aw = torch.randn(n, 3, 3, generator=gen, dtype=torch.float64)
    c = torch.randn(n, generator=gen, dtype=torch.float64)
    m = ws._product(tag, case).train()
    mob = {id(l.conditioner): i for i, l in enumerate(m.layers) if l.kind == "mobius"}
    rec, inputs = [], {}
    real_apply, real_cond = train.MobiusMixture.apply, engine.conditioner_torch

    def conditioner(ct, x):
        out = real_cond(ct, x)
        if id(ct) in mob:
            inputs[id(out)] = (mob[id(ct)], x.detach().clone())
        return out

    class Recorder:
        @staticmethod
        def apply(R, out, p0, inverse, K):
            i, x = inputs[id(out)]
            r = dict(layer=i, R=R.detach().clone(), out=out.detach().clone(), p0=p0, K=K, x=x)
            out.register_hook(lambda g: r.__setitem__("G_out", g.detach().clone()))
            R_out, ldj = real_apply(R, out, p0, inverse, K)
            R_out.register_hook(lambda g: r.__setitem__("G_Rout", g.detach().clone()))
            ldj.register_hook(lambda g: r.__setitem__("g_ldj", g.detach().clone()))
            rec.append(r)
            return R_out, ldj

    monkeypatch.setattr(engine, "conditioner_torch", conditioner)
    monkeypatch.setattr(train, "MobiusMixture", Recorder)
    R = b["R"][:n].clone().cuda().requires_grad_(True)
    f = b["rows"][:n].clone().cuda().requires_grad_(True)
    out, ldj = m(R, f)
    ((Aw.cuda().float() * out).sum() + (c.cuda().float() * ldj).sum()).backward()
    monkeypatch.undo()
    assert [r["layer"] for r in rec] == [1, 3]

    # the fp64 oracle's parameter gradients of the whole flow, as test_composed_operators computes them, and the inputs of its
    # Mobius conditioners
    o = orc.OracleFlow(b["cfg"], sd, torch.float64)
    names = [k for k, _ in m.named_parameters()]
    for k in names:
        o.sd[k] = o.sd[k].clone().requires_grad_(True)
    oracle_x = {}
    real_orc_cond = orc.conditioner

    def orc_conditioner(sd_, prefix, x):
        oracle_x[prefix] = x.detach().clone()
        return real_orc_cond(sd_, prefix, x)

    monkeypatch.setattr(orc, "conditioner", orc_conditioner)
    Ro, lo = o.with_grad(b["R"][:n].double().clone(), b["rows"][:n].double().clone())
    monkeypatch.undo()
    ((Aw * Ro).sum() + (c * lo).sum()).backward()
    got = dict(m.named_parameters())
    sd64 = {k: v.detach().double() for k, v in sd.items()}
    rel = lambda a, r: (a.detach().cpu().double() - r).abs().max().item() / max(r.abs().max().item(), 1e-6)
    for r in rec:
        # 1. the operator at the recorded inputs, with the recorded cotangents
        cot = {"recorded": (r["G_Rout"].cpu().double(), r["g_ldj"].cpu().double())}
        res = run_mobius(r["R"].cpu(), r["out"].cpu(), r["p0"], r["K"], False, cotangents=cot)
        assert torch.equal(res["got"]["recorded"][1], r["G_out"]), "the operator's G_out is not the one the composed run used"
        # 2. the kernel's G_out through the fp64 conditioner backward, with the oracle's branches and with the device's
        prefix = f"layers.{r['layer']}.conditioner."
        masks_oracle, pre_oracle = _relu_masks(sd64, prefix, oracle_x[prefix])
        with torch.no_grad():
            masks_dev, _ = _relu_masks({k: v for k, v in m.state_dict().items() if k.startswith(prefix)}, prefix, r["x"])
        masks_dev = [mk.cpu().double() for mk in masks_dev]
        flips = [(a != d).nonzero().tolist() for a, d in zip(masks_oracle, masks_dev)]
        at = [[float(pre_oracle[i][j, u]) for j, u in fl] for i, fl in enumerate(flips)]
        worst = {}
        x64 = r["x"].cpu().double()
        for label, masks in (("oracle_branches", masks_oracle), ("device_branches", masks_dev)):
            w = {k: sd64[k].clone().requires_grad_(True) for k in sd64 if k.startswith(prefix)}
            _masked_conditioner(w, prefix, x64, masks).backward(r["G_out"].cpu().double())
            for k in w:
                worst[(label, k[len(prefix):])] = (rel(got[k].grad, w[k].grad), rel(w[k].grad, o.sd[k].grad))
        record_error(test="train_ops_composed_localised", layer=r["layer"], relu_flips=flips, oracle_preactivation_at_flips=at,
                     op_worst=res["report"].rows, product_vs_oracle={k: rel(got[prefix + k].grad, o.sd[prefix + k].grad)
                                                                     for k in [kk[len(prefix):] for kk in sd64 if kk.startswith(prefix)]},
                     **{f"{lab}:{k}": v for (lab, k), v in worst.items()})
        for (label, k), (vs_product, vs_oracle) in worst.items():
            if label == "device_branches":
                assert vs_product <= 1e-4, (r["layer"], k, vs_product)   # the product's conditioner backward, in fp64
            else:
                assert vs_oracle <= 2e-3, (r["layer"], k, vs_oracle)     # the oracle's, within the composed bound
