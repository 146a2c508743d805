"""The differentiable path of the ablation layers (36Trans, 9TransLSmith with and without lu, 9TransLSVD, 9TransRSVD, 9TransRSmith;
flow/affineflow.py:27-41,55-70): AblationLayer in rotationnormflow_b200/train.py over rnf_train_ablation_* (csrc/train_ops.cu).
Flow.forward / Flow.inverse run it when autograd is on, and for config.segments != 64.

Without a GPU: the fp64 prototype of the vector-Jacobian products (tools/proto/ablation_vjp.py) against autograd through the oracle,
the oracle's SVD-layer gradients against central differences, and the C ABI's argument checks.  On the GPU: gradients and values of
every ablation golden case against autograd through the fp64 oracle, agreement with the fused inference kernels, segments != 64,
and a few training steps."""
import importlib.util
import os

import pytest
import torch

from conftest import ABLATION_CASES, ROOT, golden, record_error, seeded_product_flow
from oracle import rnf_oracle as orc
import rotationnormflow_b200 as rnf
from rotationnormflow_b200 import _cabi


def _proto():
    spec = importlib.util.spec_from_file_location("ablation_vjp", os.path.join(ROOT, "tools", "proto", "ablation_vjp.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _vee(R, G):
    H = R.transpose(1, 2) @ G
    return torch.stack([H[:, 2, 1] - H[:, 1, 2], H[:, 0, 2] - H[:, 2, 0], H[:, 1, 0] - H[:, 0, 1]], dim=1)


# ---- without a GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale", [1e-3, 0.3])
def test_prototype_vjps_match_oracle_autograd(scale):
    """The formulas ablation_bwd_kernel implements, in fp64, for M = I + scale * randn (near identity as initialised, and well away
    from it): tangential rotation gradient and matrix gradient of all five kinds (right9 in both directions)."""
    errs = _proto().check(N=64, scale=scale, seed=3)
    assert set(errs) == {"smith9", "smith36", "polar9l", "polar9r", "right9", "right9_inv"}
    for kind, (eR, eM) in errs.items():
        assert eR < 1e-10 and eM < 1e-10, (kind, eR, eM)


def _polar_matrices(tag):
    g = golden(tag)
    sd = {k: v.double() for k, v in g.state_dict().items()}
    if g.cfg.condition:
        eye = torch.eye(3, dtype=torch.float64)
        return [orc.conditioner(sd, f"layers.{i}.net.", g.rows[:16].double()).reshape(-1, 3, 3) + eye for i in (1, 3)]
    return [sd[f"layers.{i}.mat"].expand(16, 3, 3) for i in (1, 3)]


@pytest.mark.parametrize("tag", ["s_polar9l", "s_polar9r", "s_polar9lc", "s_polar9rc"])
def test_oracle_polar_gradients_match_central_differences(tag):
    """The SVD layers' matrices are I + 1e-3 noise, whose singular values nearly coincide; torch.svd's backward divides by their
    gaps.  Its gradient of U V^T is still the reference for the GPU comparison: directional derivatives in M and along the rotation's
    tangent space agree with central differences of the fp64 forward."""
    gen = torch.Generator().manual_seed(5)
    R = orc.random_rotations(16, gen, torch.float64)
    A = torch.randn(16, 3, 3, generator=gen, dtype=torch.float64)
    left = tag.startswith("s_polar9l")
    for M in _polar_matrices(tag):
        for MM in (M, M.transpose(-1, -2)):                  # the forward and the inverse direction's matrix
            Mr, Rr = MM.clone().requires_grad_(True), R.clone().requires_grad_(True)
            (A * orc.polar9(Mr, Rr, left)[0]).sum().backward()
            dM = torch.randn(MM.shape, generator=gen, dtype=torch.float64)
            w = torch.randn(16, 3, generator=gen, dtype=torch.float64)
            loss = lambda M_, R_: float((A * orc.polar9(M_, R_, left)[0]).sum())
            h = 1e-6
            fd_M = (loss(MM + h * dM, R) - loss(MM - h * dM, R)) / (2 * h)
            rot = lambda s: R @ torch.linalg.matrix_exp(s * _proto().hat(w))
            fd_R = (loss(MM, rot(h)) - loss(MM, rot(-h))) / (2 * h)
            ad_M = float((Mr.grad * dM).sum())
            ad_R = float((_vee(R, Rr.grad) * w).sum())
            assert abs(ad_M - fd_M) < 1e-6 * max(1.0, abs(fd_M)), (ad_M, fd_M)
            assert abs(ad_R - fd_R) < 1e-6 * max(1.0, abs(fd_R)), (ad_R, fd_R)


def test_ablation_abi_argument_errors_without_gpu():
    lib = _cabi.load()
    assert lib.rnf_train_ablation_forward(None, None, 4, _cabi.RNF_LAYER_SMITH9, None, None, None) == -1
    assert b"null buffer" in lib.rnf_last_error()
    assert lib.rnf_train_ablation_forward(None, None, -1, _cabi.RNF_LAYER_SMITH9, None, None, None) == -1
    assert b"negative N" in lib.rnf_last_error()
    for kind in (_cabi.RNF_LAYER_AFFINE, _cabi.RNF_LAYER_RIGHT9 + 1):
        assert lib.rnf_train_ablation_backward(None, None, 4, kind, None, None, None, None, None, None) == -1
        assert b"not an ablation layer" in lib.rnf_last_error()
    assert lib.rnf_train_ablation_backward(None, None, 4, _cabi.RNF_LAYER_SMITH36, None, None, None, None, None, None) == -1
    assert b"null buffer" in lib.rnf_last_error()
    assert lib.rnf_train_ablation_forward(None, None, 0, _cabi.RNF_LAYER_POLAR9L, None, None, None) == 0
    assert lib.rnf_train_ablation_backward(None, None, 0, _cabi.RNF_LAYER_RIGHT9, None, None, None, None, None, None) == 0


# ---- on the GPU ----------------------------------------------------------------------------------------------------------------
def _loss(R, ldj, A, c):
    return (A * R).sum() + (c * ldj).sum()


def _compare(cfg, sd, R0, feat_rows, inverse, tol=2e-3):
    """Parameter / feature / (tangential) rotation gradients of the product against the fp64 oracle; returns the worst relative
    gradient error and the worst value error."""
    gen = torch.Generator().manual_seed(77)
    N = R0.shape[0]
    A = torch.randn(N, 3, 3, generator=gen, dtype=torch.float64)
    c = torch.randn(N, generator=gen, dtype=torch.float64)
    m = rnf.get_flow(cfg)
    m.load_state_dict(sd)
    m = m.cuda().train()
    R = R0.clone().cuda().requires_grad_(True)
    f = None if feat_rows is None else feat_rows.clone().cuda().requires_grad_(True)
    out, ldj = (m.inverse if inverse else m)(R, f)
    assert out.requires_grad and ldj.requires_grad
    _loss(out, ldj, A.cuda().float(), c.cuda().float()).backward()
    o = orc.OracleFlow(cfg, sd, torch.float64)
    names = [k for k, _ in m.named_parameters()]
    for k in names:
        o.sd[k] = o.sd[k].clone().requires_grad_(True)
    R2 = R0.double().clone().requires_grad_(True)
    f2 = None if feat_rows is None else feat_rows.double().clone().requires_grad_(True)
    Ro, lo = o.with_grad(R2, f2, inverse=inverse)
    _loss(Ro, lo, A, c).backward()
    # values first (fp32 vs fp64; the inverse direction returns a dyadic angle: allow the flip bound on a few rows)
    dR = (out.detach().cpu().double() - Ro.detach()).abs().amax(dim=(1, 2))
    assert (dR <= 1e-5).float().mean() > (0.9 if inverse else 0.999) and dR.max() < 2e-3
    worst = 0.0
    got = dict(m.named_parameters())
    for k in names:
        ref = o.sd[k].grad
        if ref is None:
            continue
        g = got[k].grad
        assert g is not None, f"no gradient reached {k}"
        err = (g.cpu().double() - ref).abs().max().item() / max(ref.abs().max().item(), 1e-6)
        worst = max(worst, err)
        assert err < tol, (k, err)
    if f is not None:
        err = (f.grad.cpu().double() - f2.grad).abs().max().item() / max(f2.grad.abs().max().item(), 1e-6)
        worst = max(worst, err)
        assert err < tol, ("feature", err)
    tR = _vee(R0.double(), R.grad.cpu().double())
    tref = _vee(R0.double(), R2.grad)
    err = (tR - tref).abs().max().item() / max(tref.abs().max().item(), 1e-6)
    assert err < tol, ("rotation (tangential)", err)
    return max(worst, err), dR.max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("tag", ABLATION_CASES)
def test_ablation_gradients_match_oracle_autograd(tag, inverse):
    g = golden(tag)
    n = 96
    worst, dR = _compare(g.cfg, g.state_dict(), g.R[:n], None if g.rows is None else g.rows[:n], inverse)
    direction = "inverse" if inverse else "forward"
    record_error(test="ablation_gradients", case=tag, direction=direction, rows=n, worst_rel_grad_err=worst, max_abs_R_err=dR,
                 reference="autograd through the fp64 oracle")
    print(f"\n[{tag} {direction}] worst relative gradient error {worst:.2e}, max |dR| {dR:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ABLATION_CASES)
def test_autograd_path_matches_fused_path(tag):
    """With autograd on, Flow.forward of an ablation flow runs the per-layer operators; the values are those of the fused kernels."""
    g = golden(tag)
    m = rnf.get_flow(g.cfg)
    m.load_state_dict(g.state_dict())
    m = m.cuda()
    R = g.R.cuda()
    rows = None if g.rows is None else g.rows.cuda()
    with torch.no_grad():
        Rf, lf = m(R, rows)
    Rc, lc = m(R, rows)
    assert lc.requires_grad and not lf.requires_grad
    assert (Rc.detach() - Rf).abs().max() < 1e-5 and (lc.detach() - lf).abs().max() < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("rot", ["9TransLSmith", "36Trans"])
def test_ablation_with_other_segment_count(rot):
    """segments != 64 always runs the per-layer operators, under no_grad too: values and gradients against the oracle."""
    cfg = rnf.load_config("symsol", layers=2, feature_dim=12, segments=32, rot=rot)
    m = seeded_product_flow(cfg, 6)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    gen = torch.Generator().manual_seed(32)
    R = orc.random_rotations(64, gen)
    rows = torch.relu(torch.randn(4, 12, generator=gen))[torch.arange(64) // 16]
    o = orc.OracleFlow(cfg, sd, torch.float64)
    mc = m.cuda().eval()
    with torch.no_grad():
        for inv in (False, True):
            Rp, lp = (mc.inverse if inv else mc)(R.cuda(), rows.cuda())
            Ro, lo = (o.inverse if inv else o.forward)(R, rows)
            d = (Rp.cpu().double() - Ro).abs().amax(dim=(1, 2))
            assert (d <= 1e-5).float().mean() > (0.9 if inv else 0.999) and d.max() < 1e-3
            if not inv:
                assert (lp.cpu().double() - lo).abs().max() < 1e-4
    for inv in (False, True):
        _compare(cfg, sd, R, rows, inv)


@pytest.mark.gpu
@pytest.mark.parametrize("overrides", [dict(rot="36Trans"), dict(rot="9TransLSmith", lu=1, condition=0)], ids=["36Trans_cond", "9TransLSmith_lu"])
def test_ablation_training_reduces_the_nll(overrides):
    """Twelve Adam steps on the NLL of a fixed batch (agent.py:60-87): the loss goes down, every parameter moves (the LU factors and
    the conditioner weights included), and the fused inference path then sees the trained weights."""
    cfg = rnf.load_config("symsol", layers=3, feature_dim=16, **overrides)
    m = seeded_product_flow(cfg, 9).cuda().train()
    gen = torch.Generator().manual_seed(10)
    R = orc.random_rotations(128, gen).cuda()
    feat = torch.relu(torch.randn(128, 16, generator=gen)).cuda() if cfg.condition else None
    before = {k: p.detach().clone() for k, p in m.named_parameters()}
    assert any(".mat.w_" in k for k in before) or any(".net." in k for k in before)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    losses = []
    for _ in range(12):
        _, ldj = m(R, feat)
        loss = -ldj.mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert losses[-1] < losses[0] - 1e-3, losses
    assert all((p.detach() - before[k]).abs().max() > 0 for k, p in m.named_parameters())
    with torch.no_grad():
        _, l2 = m(R, feat)
    assert abs(float(-l2.mean()) - float(-m(R, feat)[1].mean())) < 1e-4
