"""Flow.log_prob, the differentiable log-density of training (agent.py:49-87) in the fused kernels: forward and backward of
csrc/flow_grad.cu through rnf_flow_train_forward / rnf_flow_train_backward, weights packed on the device (engine.mobius_images,
engine.affine_blocks, engine.condition_torch), weight gradients as batched GEMMs over the kernel's training records.
Rotation gradients are compared in the tangent space of SO(3): vee(R^T G)."""
import numpy as np
import pytest
import torch

from conftest import golden, record_error, seeded_product_flow
from oracle import rnf_oracle as orc
import rotationnormflow_b200 as rnf
from rotationnormflow_b200 import _cabi, engine

RNF_EINVAL = -1


def _vee(R, G):
    H = R.transpose(1, 2) @ G
    return torch.stack([H[:, 2, 1] - H[:, 1, 2], H[:, 0, 2] - H[:, 2, 0], H[:, 1, 0] - H[:, 0, 1]], dim=1)


def _cpu_flow(g):
    m = rnf.get_flow(g.cfg)
    m.load_state_dict(g.state_dict())
    return m


# ---- 1. packing on the device equals the host packing (CPU tensors, no GPU needed) -----------------------------------------------
@pytest.mark.parametrize("tag", ["s_symsol", "s_mobonly", "s_modelnet"])
def test_mobius_images_equal_pack_mobius(tag):
    m = _cpu_flow(golden(tag))
    mob = [l for l in m.layers if l.kind == "mobius"]
    imgs = engine.mobius_images([engine.conditioner_tensors(l.conditioner) for l in mob])
    assert imgs.shape == (len(mob), engine.MOB_FLOATS)
    for i, l in enumerate(mob):
        ref, _ = engine.pack_mobius(engine.conditioner_tensors(l.conditioner), m.feature_dim if l.condition else 0)
        assert np.array_equal(imgs[i].detach().numpy(), ref)


@pytest.mark.parametrize("tag", ["s_symsol", "s_uncond", "s_lu", "s_rot", "s_unrot"])
def test_affine_blocks_equal_pack_affine_matrix(tag):
    m = _cpu_flow(golden(tag))
    aff = [l for l in m.layers if l.kind in ("aff_u", "aff_lu", "rot_u")]
    assert aff
    blk = engine.affine_blocks(aff).detach().numpy()
    for i, l in enumerate(aff):
        ref = engine.pack_affine_matrix(l.matrix(), is_rot=(l.kind == "rot_u"))
        assert np.array_equal(blk[i], ref[:17]), (l.kind, blk[i], ref[:17])


@pytest.mark.parametrize("tag", ["s_symsol", "s_modelnet", "s_rotc"])
def test_condition_torch_layout(tag):
    g = golden(tag)
    m = _cpu_flow(g)
    layers = list(m.layers)
    cond = engine.condition_torch(layers, g.feat).detach()
    mob = [l for l in layers if l.kind == "mobius" and l.condition]
    aff = [l for l in layers if l.kind in ("aff_c", "rot_c")]
    B = g.feat.shape[0]
    assert cond.shape == (B, len(mob) * engine.HIDDEN + len(aff) * (engine.AFF_FLOATS + engine.HIDDEN))
    for s, l in enumerate(mob):
        ref = g.feat @ l.conditioner.fc_first.weight[:, 3:].detach().t()
        assert torch.allclose(cond[:, s * 64:(s + 1) * 64], ref, rtol=1e-5, atol=1e-6)
    base = len(mob) * engine.HIDDEN
    for s, l in enumerate(aff):
        blk = cond[:, base + s * engine.AFF_FLOATS: base + (s + 1) * engine.AFF_FLOATS]
        assert (blk[:, 17:] == 0).all()
        W = blk[:, :16].reshape(B, 4, 4).double()
        if l.kind == "rot_c":
            assert torch.allclose(W @ W.transpose(1, 2), torch.eye(4, dtype=W.dtype).expand(B, 4, 4), atol=1e-5)
        else:
            assert torch.allclose(blk[:, 16].double(), torch.linalg.slogdet(W)[1], atol=1e-5)
    assert (cond[:, base + len(aff) * engine.AFF_FLOATS:] == 0).all()


def test_cabi_train_argument_errors_without_gpu():
    lib = _cabi.load()
    assert lib.rnf_flow_train_forward(None, None, None, 1, None, 0, None, 0, None, None, None) == RNF_EINVAL
    assert b"null handle" in lib.rnf_last_error()
    assert lib.rnf_flow_train_backward(None, None, None, 1, None, 0, None, 0, None, None, None, None, 0, None) == RNF_EINVAL
    assert b"null handle" in lib.rnf_last_error()
    assert lib.rnf_flow_train_workspace_floats(None, 10) == 0
    with pytest.raises(_cabi.RnfError):
        _cabi.check(lib.rnf_flow_train_backward(None, None, None, -1, None, 0, None, 0, None, None, None, None, 0, None))


def test_log_prob_refuses_ablation_layers():
    g = golden("s_smith9")
    m = rnf.get_flow(g.cfg)
    with pytest.raises(NotImplementedError):
        m.log_prob(g.R)


def test_log_prob_cpu_tensors_fail_loudly():
    g = golden("s_symsol")
    m = rnf.get_flow(g.cfg)
    with pytest.raises(RuntimeError, match="CUDA"):
        m.log_prob(g.R, g.feat, feature_index=g.feat_index)


# ---- 2. gradients against autograd through the fp64 oracle ------------------------------------------------------------------------
def _flow(cfg, sd):
    m = rnf.get_flow(cfg)
    m.load_state_dict(sd)
    return m.cuda().train()


def _fused_grads(m, R0, feat, fi, c, A=None):
    """Gradients of sum_n c_n logp_n through Flow.log_prob: (logp, {param: grad}, feature grad, tangential R grad, A grad)."""
    m.zero_grad(set_to_none=True)
    R = R0.clone().cuda().requires_grad_(True)
    f = None if feat is None else feat.clone().cuda().requires_grad_(True)
    Ag = None if A is None else A.clone().cuda().float().requires_grad_(True)
    lp = m.log_prob(R, f, feature_index=None if fi is None else fi.cuda(), fisher_A=Ag)
    (c.cuda().float() * lp).sum().backward()
    grads = {k: p.grad.detach().clone() if p.grad is not None else None for k, p in m.named_parameters()}
    return lp.detach(), grads, None if f is None else f.grad, _vee(R0.cuda().float(), R.grad), None if Ag is None else Ag.grad


def _composed_grads(m, R0, feat, fi, c, A=None):
    """The same through the per-layer operators (Flow.forward with autograd on, train.composed_run)."""
    from rotationnormflow_b200.fisher import fisher_constants
    m.zero_grad(set_to_none=True)
    R = R0.clone().cuda().requires_grad_(True)
    f = None if feat is None else feat.clone().cuda().requires_grad_(True)
    Ag = None if A is None else A.clone().cuda().float().requires_grad_(True)
    img = None if fi is None else fi.cuda()
    Ro, lp = m(R, None if f is None else f[img])
    if Ag is not None:
        A9, cc = fisher_constants(Ag)
        lp = lp + (A9[img].reshape(-1, 3, 3) * Ro).sum(dim=(1, 2)) - cc[img]
    (c.cuda().float() * lp).sum().backward()
    grads = {k: p.grad.detach().clone() if p.grad is not None else None for k, p in m.named_parameters()}
    return lp.detach(), grads, None if f is None else f.grad, _vee(R0.cuda().float(), R.grad), None if Ag is None else Ag.grad


def _oracle_grads(cfg, sd, R0, feat, fi, c, A=None):
    o = orc.OracleFlow(cfg, sd, torch.float64)
    for k in [k for k, _ in _cpu_flow_of(cfg, sd).named_parameters()]:
        o.sd[k] = o.sd[k].clone().requires_grad_(True)
    R2 = R0.double().clone().requires_grad_(True)
    f2 = None if feat is None else feat.double().clone().requires_grad_(True)
    A2 = None if A is None else A.double().clone().requires_grad_(True)
    Ro, lp = o.with_grad(R2, None if f2 is None else f2[fi])
    if A2 is not None:
        lp = lp + (A2[fi] * Ro).sum(dim=(1, 2)) - _fisher_c64(A2)[fi]
    (c.double() * lp).sum().backward()
    grads = {k: v.grad for k, v in o.sd.items() if torch.is_tensor(v) and v.requires_grad}
    return lp.detach(), grads, None if f2 is None else f2.grad, _vee(R0.double(), R2.grad), None if A2 is None else A2.grad


def _fisher_c64(A):
    """sum of the proper singular values + log of the type-1 normaliser (utils/fisher.py:67-97), fp64 and differentiable in A."""
    U, S, V = torch.svd(A)
    S2 = S[:, 2] * torch.det(U) * torch.det(V)
    S0, S1 = S[:, 0], S[:, 1]
    return S0 + S1 + S2 - 0.5 * torch.log(8 * np.pi * (S0 + S1) * (S2 + S1) * (S0 + S2))


def _cpu_flow_of(cfg, sd):
    m = seeded_product_flow(cfg, 0)
    m.load_state_dict(sd)
    return m


def _rel(a, ref):
    a, ref = a.detach().cpu().double(), ref.detach().cpu().double()
    return (a - ref).abs().max().item() / max(ref.abs().max().item(), 1e-6)


def _compare(tag, got, ref, tol, test):
    lp, gp, gf, gr, ga = got
    lr, rp, rf, rr, ra = ref
    worst, where = 0.0, ""
    for k, g in gp.items():
        if k not in rp or rp[k] is None:
            continue
        assert g is not None, f"no gradient reached {k}"
        e = _rel(g, rp[k])
        if e > worst:
            worst, where = e, k
    for name, a, b in (("feature", gf, rf), ("rotation (tangential)", gr, rr), ("fisher_A", ga, ra)):
        if b is not None:
            assert a is not None, name
            e = _rel(a, b)
            if e > worst:
                worst, where = e, name
    dl = ((lp.cpu().double() - lr.cpu().double()).abs() / lr.cpu().double().abs().clamp(min=1)).max().item()
    record_error(test=test, case=tag, logp_err=dl, grad_rel_err=worst, worst_at=where)
    print(f"\n[{tag}] logp {dl:.2e}, worst gradient {worst:.2e} ({where})")
    assert dl <= 1e-4 and worst <= tol, (tag, dl, worst, where)


def _coeffs(N, seed=77):
    return torch.randn(N, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["s_uncond", "s_symsol", "s_modelnet", "s_pascal", "s_lu", "s_mobonly"])
def test_log_prob_gradients_match_oracle(tag):
    g = golden(tag)
    sd = g.state_dict()
    c = _coeffs(g.R.shape[0])
    got = _fused_grads(_flow(g.cfg, sd), g.R, g.feat, g.feat_index, c)
    ref = _oracle_grads(g.cfg, sd, g.R, g.feat, g.feat_index, c)
    _compare(tag, got, ref, 1e-4, "log_prob_vs_oracle")


@pytest.mark.gpu
def test_log_prob_with_fisher_base_matches_oracle():
    g = golden("s_modelnet")
    sd = g.state_dict()
    A = 3.0 * torch.randn(g.feat.shape[0], 3, 3, generator=torch.Generator().manual_seed(3))
    c = _coeffs(g.R.shape[0])
    got = _fused_grads(_flow(g.cfg, sd), g.R, g.feat, g.feat_index, c, A)
    ref = _oracle_grads(g.cfg, sd, g.R, g.feat, g.feat_index, c, A)
    _compare("s_modelnet+fisher", got, ref, 1e-4, "log_prob_vs_oracle")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["s_rot", "s_rotc", "s_unrot"])
def test_log_prob_rotation_layers_match_composed_path(tag):
    # (torch.svd of the nearly degenerate I + 1e-3 noise makes fp32 and fp64 differ by 7e-3: see test_gpu_train.py)
    g = golden(tag)
    m = _flow(g.cfg, g.state_dict())
    c = _coeffs(g.R.shape[0])
    _compare(tag, _fused_grads(m, g.R, g.feat, g.feat_index, c), _composed_grads(m, g.R, g.feat, g.feat_index, c), 1e-3,
             "log_prob_vs_composed")


@pytest.mark.gpu
@pytest.mark.parametrize("tag,fisher", [("symsol2048", False), ("modelnet", True)])
def test_log_prob_full_size_matches_composed_path(tag, fisher):
    g = golden(tag)
    m = _flow(g.cfg, g.state_dict())
    gen = torch.Generator().manual_seed(11)
    B = g.feat.shape[0]
    R0 = orc.random_rotations(512, gen)
    fi = torch.arange(512) % B
    A = 3.0 * torch.randn(B, 3, 3, generator=gen) if fisher else None
    c = _coeffs(512)
    _compare(tag, _fused_grads(m, R0, g.feat, fi, c, A), _composed_grads(m, R0, g.feat, fi, c, A), 1e-3, "log_prob_vs_composed")


# ---- 3. values, batch sizes, chunking ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["s_uncond", "s_symsol", "s_modelnet", "s_pascal", "s_lu", "s_mobonly"])
def test_log_prob_values(tag):
    g = golden(tag)
    m = _flow(g.cfg, g.state_dict())
    feat = None if g.feat is None else g.feat.cuda()
    fi = None if g.feat_index is None else g.feat_index.cuda()
    lp = m.log_prob(g.R.cuda(), feat, feature_index=fi)
    with torch.no_grad():
        _, ldj = m(g.R.cuda(), None if feat is None else feat[fi], mlp_mode="fp32")
    assert (lp.detach() - ldj).abs().max().item() <= 2e-5
    assert (lp.detach().cpu().double() - g.out("fwd", "ldj", "f64").double()).abs().max().item() <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("N", [0, 1, 33])
def test_log_prob_batch_sizes(N):
    g = golden("s_symsol")
    m = _flow(g.cfg, g.state_dict())
    gen = torch.Generator().manual_seed(N + 1)
    R = orc.random_rotations(max(N, 1), gen)[:N]
    fi = torch.randint(0, g.feat.shape[0], (max(N, 1),), generator=gen)[:N]
    c = _coeffs(N)
    got = _fused_grads(m, R, g.feat, fi, c)
    assert got[0].shape == (N,)
    if N == 0:
        assert all(v is None or v.abs().max().item() == 0 for v in got[1].values())
        return
    _compare(f"N={N}", got, _composed_grads(m, R, g.feat, fi, c), 1e-3, "log_prob_vs_composed")


@pytest.mark.gpu
def test_log_prob_chunked_rows_and_unsorted_feature_index(monkeypatch):
    """SYMSOL-style rows (several ground truths per image, rows in no particular image order) over several workspace chunks."""
    g = golden("s_symsol")
    m = _flow(g.cfg, g.state_dict())
    B = g.feat.shape[0]
    gen = torch.Generator().manual_seed(19)
    N = 1500
    R = orc.random_rotations(N, gen)
    fi = torch.randperm(N, generator=gen) % B                  # non-monotone row -> image map
    c = _coeffs(N)
    whole = _fused_grads(m, R, g.feat, fi, c)
    tp = next(iter(m.__dict__["_rnf_train_programs"].values()))
    per_row = 4 * (tp.n_mob * engine.TRAIN_RECORD_FLOATS + tp.n_aff * 16)
    monkeypatch.setattr(engine, "TRAIN_WORKSPACE_BYTES", per_row * 400)      # 4 chunks of rows
    chunked = _fused_grads(m, R, g.feat, fi, c)
    assert torch.equal(whole[0], chunked[0]) and torch.equal(whole[3], chunked[3])
    _compare("chunked vs whole", chunked, whole, 1e-5, "log_prob_chunks")
    _compare("chunked vs composed", chunked, _composed_grads(m, R, g.feat, fi, c), 1e-3, "log_prob_vs_composed")


# ---- 4. training --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_training_steps_fused_match_composed():
    cfg = rnf.load_config("symsol", layers=3, feature_dim=16)
    gen = torch.Generator().manual_seed(10)
    R = orc.random_rotations(256, gen).cuda()
    feat = torch.relu(torch.randn(32, 16, generator=gen)).cuda()
    fi = (torch.arange(256) % 32).cuda()
    runs = []
    for fused in (True, False):
        m = seeded_product_flow(cfg, 9).cuda().train()
        before = {k: p.detach().clone() for k, p in m.named_parameters()}
        opt = torch.optim.Adam(m.parameters(), lr=1e-3)
        losses = []
        for _ in range(12):
            if fused:
                loss = -m.log_prob(R, feat, feature_index=fi).mean()
            else:
                loss = -m(R, feat[fi])[1].mean()
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses.append(float(loss.detach()))
        runs.append((m, losses, before))
    (mf, lf, bf), (_, lc, _) = runs
    print(f"\nfused losses {lf[0]:.5f} -> {lf[-1]:.5f}, composed {lc[0]:.5f} -> {lc[-1]:.5f}")
    for a, b in zip(lf, lc):
        assert abs(a - b) <= 1e-4 * max(1.0, abs(b)), (lf, lc)
    assert lf[-1] < lf[0] - 1e-3
    assert all((p.detach() - bf[k]).abs().max() > 0 for k, p in mf.named_parameters())
    with torch.no_grad():                                      # the fused inference path sees the trained weights
        _, ldj = mf(R, feat[fi])
    assert abs(float(-ldj.mean()) - float(-mf.log_prob(R, feat, feature_index=fi).mean())) < 1e-4


@pytest.mark.gpu
def test_log_prob_forward_and_backward_do_not_synchronise():
    cfg = rnf.load_config("symsol", layers=4, feature_dim=64)
    m = seeded_product_flow(cfg, 2).cuda().train()
    gen = torch.Generator().manual_seed(4)
    R = orc.random_rotations(512, gen).cuda()
    feat = torch.relu(torch.randn(64, 64, generator=gen)).cuda().requires_grad_(True)
    fi = (torch.arange(512) % 64).cuda()
    (-m.log_prob(R, feat, feature_index=fi).mean()).backward()      # warm-up: builds the structural program (host packing, once)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        (-m.log_prob(R, feat, feature_index=fi).mean()).backward()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()


# ---- 5. fallbacks ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["segments=32", "s_clu"])
def test_log_prob_fallbacks_give_composed_numbers(case):
    if case == "s_clu":
        g = golden("s_clu")
        cfg, sd, R, feat, fi = g.cfg, g.state_dict(), g.R, g.feat, g.feat_index
    else:
        cfg = rnf.load_config("symsol", layers=2, feature_dim=12, segments=32)
        sd = {k: v.clone() for k, v in seeded_product_flow(cfg, 5).state_dict().items()}
        gen = torch.Generator().manual_seed(32)
        R = orc.random_rotations(64, gen)
        feat = torch.relu(torch.randn(4, 12, generator=gen))
        fi = torch.arange(64) // 16
    m = _flow(cfg, sd)
    c = _coeffs(R.shape[0])
    got = _fused_grads(m, R, feat, fi, c)
    ref = _composed_grads(m, R, feat, fi, c)
    # the same operators in the same order: equal up to the order of atomic sums in the backward of the row gather
    _compare(case, got, ref, 1e-6, "log_prob_fallback")
