"""Flow.log_prob_grad (csrc/flow_grad.cu through rnf_flow_logprob_grad) and evalpath.refine_rotation, the nll_grad refinement of
eval.py:464-480.  Gradients are compared in the tangent space of SO(3): vee(R^T G), the part of d logp / dR that a rotation can feel."""
import pytest
import torch

from conftest import golden, record_error, seeded_product_flow
from oracle import rnf_oracle as orc
import rotationnormflow_b200 as rnf
from rotationnormflow_b200 import _cabi, evalpath

RNF_EINVAL = -1


def _vee(R, G):
    H = R.transpose(1, 2) @ G
    return torch.stack([H[:, 2, 1] - H[:, 1, 2], H[:, 0, 2] - H[:, 2, 0], H[:, 1, 0] - H[:, 0, 1]], dim=1)


def _flow(g):
    m = rnf.get_flow(g.cfg)
    m.load_state_dict(g.state_dict())
    return m.cuda().eval()


def _oracle_logp_grad(cfg, sd, R0, feat, fi, A=None):
    """fp64 oracle: logp = ldj [+ Fisher term of image fi[n]] and d logp / dR0 by autograd."""
    o = orc.OracleFlow(cfg, sd, torch.float64)
    R2 = R0.double().clone().requires_grad_(True)
    rows = None if feat is None else feat.double()[fi]
    Ro, lp = o.with_grad(R2, rows)
    if A is not None:
        sumS, logc = orc.fisher_constants(A.double())
        lp = lp + (A.double()[fi] * Ro).sum(dim=(1, 2)) - sumS[fi] - logc[fi]
    lp.sum().backward()
    return lp.detach(), R2.grad


def _check_against(tag, R0, lp, G, lp_ref, G_ref, lp_tol, g_tol):
    dl = ((lp.cpu().double() - lp_ref).abs() / lp_ref.abs().clamp(min=1)).max().item()
    t, tref = _vee(R0.double(), G.cpu().double()), _vee(R0.double(), G_ref)
    dg = (t - tref).abs().max().item() / max(tref.abs().max().item(), 1e-6)
    record_error(test="log_prob_grad", case=tag, logp_err=dl, grad_rel_err=dg)
    print(f"\n[{tag}] logp |d|/max(1,|ref|) {dl:.2e}, tangent max|d|/max|ref| {dg:.2e}")
    assert dl <= lp_tol and dg <= g_tol, (tag, dl, dg)


# ---- 1. parity with the fp64 oracle, every golden row ----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["s_uncond", "s_symsol", "s_modelnet", "s_pascal", "s_lu", "s_mobonly"])
def test_log_prob_grad_matches_oracle(tag):
    g = golden(tag)
    m = _flow(g)
    fi = g.feat_index
    lp, G = m.log_prob_grad(g.R.cuda(), None if g.feat is None else g.feat.cuda(),
                            feature_index=None if fi is None else fi.cuda())
    lp_ref, G_ref = _oracle_logp_grad(g.cfg, g.state_dict(), g.R, g.feat, fi)
    _check_against(tag, g.R, lp, G, lp_ref, G_ref, 1e-4, 1e-4)


@pytest.mark.gpu
def test_log_prob_grad_with_fisher_base_matches_oracle():
    g = golden("s_modelnet")
    m = _flow(g)
    gen = torch.Generator().manual_seed(3)
    A = 3.0 * torch.randn(g.feat.shape[0], 3, 3, generator=gen)
    lp, G = m.log_prob_grad(g.R.cuda(), g.feat.cuda(), feature_index=g.feat_index.cuda(), fisher_A=A.cuda())
    lp_ref, G_ref = _oracle_logp_grad(g.cfg, g.state_dict(), g.R, g.feat, g.feat_index, A)
    _check_against("s_modelnet+fisher", g.R, lp, G, lp_ref, G_ref, 1e-4, 1e-4)


# ---- 2. full-size configurations ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tag,fisher", [("symsol2048", False), ("modelnet", True)])
def test_log_prob_grad_full_size(tag, fisher):
    g = golden(tag)
    m = _flow(g)
    gen = torch.Generator().manual_seed(11)
    B = g.feat.shape[0]
    R0 = orc.random_rotations(512, gen)
    fi = torch.arange(512) % B
    A = 3.0 * torch.randn(B, 3, 3, generator=gen) if fisher else None
    lp, G = m.log_prob_grad(R0.cuda(), g.feat.cuda(), feature_index=fi.cuda(), fisher_A=None if A is None else A.cuda())
    lp_ref, G_ref = _oracle_logp_grad(g.cfg, g.state_dict(), R0, g.feat, fi, A)
    _check_against(tag, R0, lp, G, lp_ref, G_ref, 1e-4, 1e-3)


# ---- 3. rotation layers: against the composed path's autograd on the GPU --------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["s_rot", "s_rotc", "s_unrot"])
def test_log_prob_grad_rotation_layers_match_composed_path(tag):
    # (torch.svd of the nearly degenerate I + 1e-3 noise makes fp32 and fp64 differ by 7e-3: see test_gpu_train.py)
    g = golden(tag)
    m = _flow(g)
    R0 = g.R.cuda()
    feat = None if g.feat is None else g.feat.cuda()
    fi = None if g.feat_index is None else g.feat_index.cuda()
    lp, G = m.log_prob_grad(R0, feat, feature_index=fi)
    R = R0.clone().requires_grad_(True)
    _, ldj = m(R, None if feat is None else feat[fi])          # autograd on -> the per-layer operators of train.py
    ldj.sum().backward()
    dl = (lp - ldj.detach()).abs().max().item()
    t, tref = _vee(R0.double(), G.double()), _vee(R0.double(), R.grad.double())
    dg = (t - tref).abs().max().item() / max(tref.abs().max().item(), 1e-6)
    record_error(test="log_prob_grad_vs_composed", case=tag, logp_err=dl, grad_rel_err=dg)
    assert dl <= 1e-4 and dg <= 1e-3, (dl, dg)


# ---- 4. consistency -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_log_prob_grad_consistency():
    g = golden("s_symsol")
    m = _flow(g)
    R, feat, fi = g.R.cuda(), g.feat.cuda(), g.feat_index.cuda()
    lp, G = m.log_prob_grad(R, feat, feature_index=fi)
    with torch.no_grad():
        _, ldj = m(R, feat[fi], mlp_mode="fp32")
    assert (lp - ldj).abs().max().item() <= 2e-5
    H = R.transpose(1, 2) @ G
    assert (H + H.transpose(1, 2)).abs().max().item() / 2 <= 1e-6 * H.abs().max().item()
    # image-major rows: feature_index and the implicit mapping give identical results
    B = feat.shape[0]
    Rm = orc.random_rotations(B * 40, torch.Generator().manual_seed(5)).cuda()
    a = m.log_prob_grad(Rm, feat)
    b = m.log_prob_grad(Rm, feat, feature_index=torch.arange(B * 40, device="cuda") // 40)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
@pytest.mark.parametrize("N", [0, 1, 33, 1000])
def test_log_prob_grad_sizes(N):
    g = golden("s_symsol")
    m = _flow(g)
    gen = torch.Generator().manual_seed(N + 1)
    R = orc.random_rotations(1000, gen).cuda()
    fi = torch.randint(0, g.feat.shape[0], (1000,), generator=gen).cuda()
    feat = g.feat.cuda()
    full = m.log_prob_grad(R, feat, feature_index=fi)
    lp, G = m.log_prob_grad(R[:N], feat, feature_index=fi[:N])
    assert lp.shape == (N,) and G.shape == (N, 3, 3)
    assert torch.equal(lp, full[0][:N]) and torch.equal(G, full[1][:N])      # a row's result does not depend on the batch
    if N:
        with torch.no_grad():
            _, ldj = m(R[:N], feat[fi[:N]], mlp_mode="fp32")
        assert (lp - ldj).abs().max().item() <= 2e-5


@pytest.mark.gpu
def test_log_prob_grad_cuda_graph_replay():
    g = golden("s_symsol")
    m = _flow(g)
    feat, fi = g.feat.cuda(), g.feat_index.cuda().int()
    R = g.R.cuda().clone()
    R2 = orc.random_rotations(R.shape[0], torch.Generator().manual_seed(8)).cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.log_prob_grad(R, feat, feature_index=fi)                # warm-up: packs the program, sets the kernel attributes
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        lp, G = m.log_prob_grad(R, feat, feature_index=fi)
    R.copy_(R2)
    graph.replay()
    torch.cuda.synchronize()
    ref = m.log_prob_grad(R2, feat, feature_index=fi)
    assert torch.equal(lp, ref[0]) and torch.equal(G, ref[1])


# ---- 5. fallbacks and refusals --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_log_prob_grad_other_segment_count_uses_composed_path():
    cfg = rnf.load_config("symsol", layers=2, feature_dim=12, segments=32)
    m = seeded_product_flow(cfg, 5)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    gen = torch.Generator().manual_seed(32)
    R0 = orc.random_rotations(64, gen)
    feat = torch.relu(torch.randn(4, 12, generator=gen))
    fi = torch.arange(64) // 16
    lp, G = m.cuda().eval().log_prob_grad(R0.cuda(), feat.cuda(), feature_index=fi.cuda())
    lp_ref, G_ref = _oracle_logp_grad(cfg, sd, R0, feat, fi)
    _check_against("segments=32", R0, lp, G, lp_ref, G_ref, 1e-4, 2e-3)


def test_log_prob_grad_refuses_ablation_layers():
    g = golden("s_smith9")
    m = rnf.get_flow(g.cfg)
    with pytest.raises(NotImplementedError):
        m.log_prob_grad(g.R)


def test_log_prob_grad_cpu_tensors_fail_loudly():
    g = golden("s_symsol")
    m = rnf.get_flow(g.cfg)
    with pytest.raises(RuntimeError, match="CUDA"):
        m.log_prob_grad(g.R, g.feat, feature_index=g.feat_index)


def test_cabi_logprob_grad_argument_errors_without_gpu():
    lib = _cabi.load()
    assert lib.rnf_flow_logprob_grad(None, None, 1, None, 0, None, 0, None, None, None, None, None) == RNF_EINVAL
    assert b"null handle" in lib.rnf_last_error()
    with pytest.raises(_cabi.RnfError):
        _cabi.check(lib.rnf_flow_logprob_grad(None, None, -1, None, 0, None, 0, None, None, None, None, None))



# ---- 6. refinement ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refine_rotation_equals_composed_autograd_loop():
    g = golden("s_symsol")
    m = _flow(g)
    feat = g.feat.cuda()
    B = feat.shape[0]
    R0 = orc.random_rotations(B * 3, torch.Generator().manual_seed(21)).cuda().reshape(B, 3, 3, 3)
    Rf, lpf = evalpath.refine_rotation(m, feat, R0, lr=1e-3, steps=10)
    # the same Adam loop with the gradient from autograd through the per-layer operators
    q = evalpath.matrix_to_quaternion(R0.reshape(-1, 3, 3)).clone().requires_grad_(True)
    opt = torch.optim.Adam([q], lr=1e-3)
    rows = feat.repeat_interleave(3, dim=0)
    for _ in range(10):
        R = evalpath.quaternion_to_matrix(q / q.norm(dim=-1, keepdim=True))
        _, ldj = m(R, rows)
        opt.zero_grad()
        (-ldj.sum()).backward()
        opt.step()
    Rc = evalpath.quaternion_to_matrix(q / q.norm(dim=-1, keepdim=True)).detach().reshape(B, 3, 3, 3)
    assert Rf.shape == R0.shape and lpf.shape == (B, 3)
    assert (Rf - Rc).abs().max().item() <= 1e-3


@pytest.mark.gpu
def test_refinement_after_the_grid_climbs_log_p():
    cfg = rnf.load_config("symsol")
    m = seeded_product_flow(cfg, 4).cuda().eval()
    F = m.feature_dim
    feat = torch.relu(torch.randn(16, F, generator=torch.Generator().manual_seed(6))).cuda()
    est, _ = evalpath.estimate_rotation_grid(m, feat, 72 * 8 ** 3, generator=torch.Generator().manual_seed(7))
    lp0, _ = m.log_prob_grad(est, feat)
    Rr, lp1 = evalpath.refine_rotation(m, feat, est, lr=1e-3, steps=100)
    print(f"\nmean log p: grid {lp0.mean().item():.4f} -> refined {lp1.mean().item():.4f}")
    assert lp1.mean().item() > lp0.mean().item()
    assert (lp1 - lp0).min().item() >= -1e-3
    est2, out = evalpath.estimate_rotation_grid(m, feat, 72 * 8 ** 3, generator=torch.Generator().manual_seed(7), refine_steps=100,
                                                refine_lr=1e-3)
    assert torch.allclose(est2, Rr, atol=1e-6) and torch.allclose(out["refined_logp"], lp1, atol=1e-5)
