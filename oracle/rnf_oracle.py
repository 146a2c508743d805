"""TEST INFRASTRUCTURE ONLY -- CPU restatement (the "oracle") of the reference hot path.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this file.  The product package
(``rotationnormflow_b200``) never does: it fails loudly when its CUDA library is
missing.

What is restated (reference file:line, all relative to /root/reference):
  flow/flow.py:13-15,36-51,53-92      layer stack, permutation table, fwd / inverse order
  flow/condition.py:9-30              4-layer residual ReLU MLP
  flow/mobiusflow.py:17-24,46-125     Mobius coupling forward (+ analytic Jacobian)
  flow/mobiusflow.py:127-245          Mobius inverse, 15-step bisection (BinFind.forward)
  flow/squeezetrans.py:10-38          quaternion affine  q -> Wq/|Wq|,  ldj = log|det W| - 4 log|Wq|
  flow/squeezetrans.py:41-91,147-174  Condition16Trans / UnconditionLU / Uncondition16Trans(LU)
  flow/rottrans.py:8-66               UnconditionRot / ConditionRot  (W = U^T V from torch.svd)
  flow/affineflow.py:5-73             config -> affine layer class
  utils/sd.py:31-82                   HEALPix SO(3) grid
  utils/fisher.py:67-97,209-232       matrix-Fisher log-prob (type-1 normaliser)
  agent.py:263-266, eval.py:460-462   arg-max,  eval.py:103  normaliser exp(logp).mean()

Third-party arithmetic that is NOT under /root/reference (pytorch3d 0.7.5 "tested on",
README.md:29; healpy / scipy unpinned) is restated in ``oracle/stubs.py`` from the
public definitions.

PARITY PINNING: the reference has no tests / golden vectors for this path
(SURVEY.md section 4).  This restatement is pinned instead against outputs of the
reference itself run in the build container (``oracle/make_golden.py`` ->
``tests/golden/*.npz``; ``tests/test_oracle.py`` re-runs the comparison live when
/root/reference is present).  The pytorch3d / healpy boundaries remain "parity
unpinned" in the strict sense (public formulas + known-answer values only).

The code is dtype-generic: run it in float32 for "what the reference computes"
and in float64 for "what the reference means".
"""
from __future__ import annotations

import math
import types

import numpy as np
import torch

from .stubs import matrix_to_quaternion, quaternion_to_matrix, pix2zphi  # public third-party formulas

PERMUTE_TABLE = ((0, 1, 2), (1, 2, 0), (2, 0, 1), (0, 1, 2), (1, 2, 0), (2, 0, 1))  # flow/flow.py:13-15


# ----------------------------------------------------------------------------------------------
# config -> layer plan            (flow/flow.py:24-51, flow/affineflow.py:5-73, flow/mobiusflow.py:7-14)
# ----------------------------------------------------------------------------------------------
def feature_dim_of(cfg) -> int:
    if not cfg.condition:
        return 0
    f = 32 if cfg.feature_dim is None else cfg.feature_dim
    if cfg.embedding:
        f += cfg.embedding_dim
    return f


def _affine_kind(cfg, first_layer_condition=False):
    """Returns one of None, 'aff_u','aff_c','aff_lu','aff_clu','rot_u','rot_c', an ablation kind
    ('smith9|smith36|polar9l|polar9r|right9' + '_u'|'_c', 'smith9_lu') or 'unsupported:<what>'."""
    rot, lu = cfg.rot, bool(cfg.lu)
    if first_layer_condition:
        if rot == "16UnTrans":
            return "aff_clu" if lu else "aff_c"
        if rot == "16UnRot":
            return "rot_c"
    if cfg.condition:
        table = {"16Trans": "aff_clu" if lu else "aff_c", "16UnTrans": "aff_lu" if lu else "aff_u",
                 "16Rot": "rot_c", "16UnRot": "rot_u"}
    else:
        table = {"16Trans": "aff_lu" if lu else "aff_u", "16Rot": "rot_u"}
    if rot in table:
        return table[rot]
    # ablation replacements of the affine layer (flow/affineflow.py:27-41,55-70)
    ablation = {"36Trans": "smith36", "9TransLSVD": "polar9l", "9TransRSVD": "polar9r", "9TransRSmith": "right9",
                "9TransLSmith": "smith9"}
    if rot in ablation:
        if rot == "9TransLSmith" and lu:
            return "unsupported:Condition9TransLU" if cfg.condition else "smith9_lu"
        return ablation[rot] + ("_c" if cfg.condition else "_u")
    return None


def layer_plan(cfg):
    """List of layer kinds in module order (index i == ``layers.{i}`` in the state dict)."""
    plan = []
    if cfg.last_affine:
        plan.append(_affine_kind(cfg, first_layer_condition=True))
    for i in range(cfg.layers):
        if cfg.dist != "noflow":
            plan.append("mobius")
        k = _affine_kind(cfg)
        if k is not None and (i != cfg.layers - 1 or cfg.first_affine):
            plan.append(k)
    return plan


def permute_rows(cfg, plan, inverse=False):
    """Permutation-table row handed to every layer (flow/flow.py:58-70 fwd, :78-88 inverse)."""
    rows = [0] * len(plan)
    if not inverse:
        c = 0
        for i, k in enumerate(plan):
            rows[i] = c % 6
            if k == "mobius" or cfg.frequent_permute:
                c += 1
    else:
        c = len(plan) if cfg.frequent_permute else cfg.layers
        for i in range(len(plan) - 1, -1, -1):
            if plan[i] == "mobius" or cfg.frequent_permute:
                c -= 1
            rows[i] = c % 6
    return rows


# ----------------------------------------------------------------------------------------------
# conditioner                                                           (flow/condition.py:24-30)
# ----------------------------------------------------------------------------------------------
def conditioner(sd, prefix, x):
    lin = torch.nn.functional.linear
    h0 = lin(x, sd[prefix + "fc_first.weight"], sd[prefix + "fc_first.bias"])
    h = h0
    for j in (1, 3, 5):
        h = lin(torch.relu(h), sd[f"{prefix}layers.{j}.weight"], sd[f"{prefix}layers.{j}.bias"])
    return lin(torch.relu(h0 + h), sd[prefix + "fc_last.weight"], sd[prefix + "fc_last.bias"])


# ----------------------------------------------------------------------------------------------
# Mobius coupling                                                     (flow/mobiusflow.py:17-245)
# ----------------------------------------------------------------------------------------------
def _mobius_h(z, w):
    """h_w(z) = (1-|w|^2)/|z-w|^2 (z-w) - w          (flow/mobiusflow.py:17-24)."""
    d = z[:, None, :] - w
    f = (1 - (w * w).sum(-1, keepdim=True)) / (d * d).sum(-1, keepdim=True)
    return f * d - w, f[..., 0]


def _wrapped_angles(h, r, v):
    th = torch.atan2((h * v[:, None, :]).sum(-1), (h * r[:, None, :]).sum(-1))
    return torch.where(th >= 0, th, th + 2 * math.pi)                     # :94-99


def _mobius_prep(sd, prefix, x, y, feature, K):
    """(flow/mobiusflow.py:52-72): MLP, then mobius_params of its output."""
    inp = y if feature is None else torch.cat((y, feature), -1)
    return mobius_params(conditioner(sd, prefix + "conditioner.", inp), x, y, K)


def mobius_params(out, x, y, K):
    """(flow/mobiusflow.py:58-72): conditioner output out [N,4K] -> frame r, v [N,3], mixture weights pi [N,K] and squashed centres
    w' [N,K,3]: split, project w onto the plane orthogonal to y, frame, softplus weights, squash."""
    a, w = out[:, :K], out[:, K:].reshape(-1, K, 3)
    w = w - (w * y[:, None, :]).sum(-1, keepdim=True) * y[:, None, :]     # (I - y y^T) w
    r = -x
    r = r / r.norm(dim=-1, keepdim=True)
    v = torch.linalg.cross(y, r, dim=-1)
    v = v / v.norm(dim=-1, keepdim=True)
    sp = torch.nn.functional.softplus(a)
    pi = sp / sp.sum(-1, keepdim=True)
    w = 0.7 / (1 + w.norm(dim=-1, keepdim=True)) * w
    return r, v, pi, w


def _explicit_ldj(x, r, v, pi, w):
    """The reference's literal Jacobian construction (flow/mobiusflow.py:104-125); equals log sum pi_k f_k."""
    eye = torch.eye(3, dtype=x.dtype, device=x.device)
    z_w = x[:, None, :] - w
    n = z_w.norm(dim=-1)
    u = z_w / n[..., None]
    th = torch.atan2((x * v).sum(-1), (x * r).sum(-1)).reshape(-1, 1)
    dz = -torch.sin(th) * r + torch.cos(th) * v
    dh_dz = ((1 - w.norm(dim=-1) ** 2)[..., None, None]
             * (eye[None, None] - 2 * torch.einsum("nki,nkj->nkij", u, u)) / (n[..., None, None] ** 2))
    dh = torch.einsum("nkpq,nq->nkp", dh_dz, dz)
    return torch.log((dh.norm(dim=-1) * pi).sum(1))


def _assemble(p, c0, c1, c2):
    out = torch.empty((c0.shape[0], 3, 3), dtype=c0.dtype, device=c0.device)
    out[:, :, p[0]] = c0
    out[:, :, p[1]] = c1
    out[:, :, p[2]] = c2
    return out


def mobius_forward(sd, prefix, R, p, feature, K, explicit_jacobian=False):
    x, y = R[:, :, p[0]], R[:, :, p[1]]
    return _mobius_forward(x, y, p, *_mobius_prep(sd, prefix, x, y, feature, K), explicit_jacobian)


def _mobius_forward(x, y, p, r, v, pi, w, explicit_jacobian=False):
    h, f = _mobius_h(x, w)
    th = (pi * _wrapped_angles(h, r, v)).sum(1, keepdim=True)             # :100
    tx = r * torch.cos(th) + v * torch.sin(th)                            # :102
    ldj = _explicit_ldj(x, r, v, pi, w) if explicit_jacobian else torch.log((pi * f).sum(1))
    tz = torch.linalg.cross(tx, y, dim=-1)                                # cyclic perms only -> this branch (:75-76)
    tz = tz / tz.norm(dim=-1, keepdim=True)
    return _assemble(p, tx, y, tz), ldj


def bisect(ystar, r, v, pi, w):
    """BinFind.forward (flow/mobiusflow.py:191-224): same bracket, same update arithmetic, returns last x0."""
    one = torch.ones_like(ystar)
    a = one * math.pi / 2
    b = one * 3 / 2 * math.pi
    x0 = None
    it = 1
    while abs(torch.max(b - a)) >= 1e-4:
        x0 = (a + b) / 2
        z = r * torch.cos(x0) + v * torch.sin(x0)
        h, _ = _mobius_h(z, w)
        fx0 = (pi * _wrapped_angles(h, r, v)).sum(1, keepdim=True) - ystar
        if it > 100:
            break
        bigger = fx0 < 0
        lesser = fx0 >= 0
        a = a + (b - a) / 2 * bigger
        b = b - (b - a) / 2 * lesser
        it += 1
    return x0


def _theta_of(x0, r, v, pi, w):
    """BinFind._forward_theta (flow/mobiusflow.py:230-245)."""
    z = r * torch.cos(x0) + v * torch.sin(x0)
    h, _ = _mobius_h(z, w)
    return (pi * _wrapped_angles(h, r, v)).sum(1, keepdim=True)


class BinFindWithGrad(torch.autograd.Function):
    """BinFind (flow/mobiusflow.py:189-273) including its backward: the implicit-function gradient at the returned root."""

    @staticmethod
    def forward(ctx, y, r, v, pi, w, root=None):
        """``root`` [N,1]: return it instead of bisecting, so that the implicit-function gradient is evaluated at a given point (the
        root another implementation returned)."""
        x0 = bisect(y, r, v, pi, w) if root is None else root.detach().to(y.dtype)
        ctx.save_for_backward(x0.detach(), r.detach(), v.detach(), pi.detach(), w.detach())
        return x0

    @staticmethod
    def backward(ctx, x_grad):
        x, r, v, pi, w = (t.clone().requires_grad_(True) for t in ctx.saved_tensors)
        with torch.enable_grad():
            gx, gr, gv, gpi, gw = torch.autograd.grad(_theta_of(x, r, v, pi, w), (x, r, v, pi, w), torch.ones_like(x_grad))
        ok = gx != 0                                                         # :262-272
        y_grad = torch.where(ok, 1 / gx, torch.zeros_like(gx)) * x_grad
        r_grad = torch.where(ok, -gr / gx, torch.zeros_like(gr)) * x_grad
        v_grad = torch.where(ok, -gv / gx, torch.zeros_like(gv)) * x_grad
        w_grad = torch.where(ok.unsqueeze(-1), -gw / gx.unsqueeze(-1), torch.zeros_like(gw)) * x_grad.unsqueeze(-1)
        pi_grad = torch.where(ok, -gpi / gx, torch.zeros_like(gpi)) * x_grad
        return y_grad, r_grad, v_grad, pi_grad, w_grad, None


def mobius_inverse(sd, prefix, R, p, feature, K, explicit_jacobian=False):
    tx, ty = R[:, :, p[0]], R[:, :, p[1]]
    return _mobius_inverse(tx, ty, p, *_mobius_prep(sd, prefix, tx, ty, feature, K), explicit_jacobian)


def _target_angle(tx, r, v):
    """The angle of the given column in its own frame, wrapped to [0, 2 pi) with 2 pi - 1e-4 .. 2 pi mapped to 0 (:157-167)."""
    tt = torch.atan2((tx * v).sum(-1), (tx * r).sum(-1)).reshape(-1, 1)
    tt = torch.where(tt >= 0, tt, tt + 2 * math.pi)
    return torch.where(abs(tt - 2 * math.pi) < 1e-4, torch.zeros_like(tt), tt)   # :163-167


def _mobius_inverse(tx, ty, p, r, v, pi, w, explicit_jacobian=False, root=None):
    tt = _target_angle(tx, r, v)
    if torch.is_grad_enabled() or root is not None:
        th = BinFindWithGrad.apply(tt, r, v, pi, w, root)
    else:
        th = bisect(tt, r, v, pi, w)
    x = r * torch.cos(th) + v * torch.sin(th)
    if explicit_jacobian:
        ldj = _explicit_ldj(x, r, v, pi, w)
    else:
        _, f = _mobius_h(x, w)
        ldj = torch.log((pi * f).sum(1))
    z = torch.linalg.cross(x, ty, dim=-1)
    z = z / z.norm(dim=-1, keepdim=True)
    return _assemble(p, x, ty, z), -ldj


def mobius_layer(R, out, p0, K, inverse, root=None):
    """One Mobius layer after its conditioner: (R [N,3,3], out [N,4K]) -> (R', ldj), the moving column p0 (the cyclic rows 0-2 of
    PERMUTE_TABLE).  Inverse direction: ``root`` [N] evaluates the layer and BinFind's implicit-function gradient at that angle
    instead of the bisection's."""
    p = PERMUTE_TABLE[p0]
    x, y = R[:, :, p[0]], R[:, :, p[1]]
    prm = mobius_params(out, x, y, K)
    if not inverse:
        return _mobius_forward(x, y, p, *prm)
    return _mobius_inverse(x, y, p, *prm, root=None if root is None else root.reshape(-1, 1))


# ----------------------------------------------------------------------------------------------
# quaternion affine / rotation layers                      (flow/squeezetrans.py, flow/rottrans.py)
# ----------------------------------------------------------------------------------------------
def det3(A):
    d00 = A[..., 1, 1] * A[..., 2, 2] - A[..., 1, 2] * A[..., 2, 1]
    d01 = A[..., 1, 2] * A[..., 2, 0] - A[..., 1, 0] * A[..., 2, 2]
    d02 = A[..., 1, 0] * A[..., 2, 1] - A[..., 1, 1] * A[..., 2, 0]
    return d00 * A[..., 0, 0] + d01 * A[..., 0, 1] + d02 * A[..., 0, 2]


def det4(A):
    """cofactor expansion along row 0 (flow/squeezetrans.py:10-22)."""
    s = A[..., 1:, :]
    return (A[..., 0, 0] * det3(s[..., [1, 2, 3]]) - A[..., 0, 1] * det3(s[..., [0, 2, 3]])
            + A[..., 0, 2] * det3(s[..., [0, 1, 3]]) - A[..., 0, 3] * det3(s[..., [0, 1, 2]]))


def quat_affine(W, R, with_ldj=True):
    """calculate_16 (flow/squeezetrans.py:33-38).  W: [1,4,4] or [N,4,4]."""
    q = matrix_to_quaternion(R)
    q = W @ q.reshape(-1, 4, 1)
    length = q.norm(dim=-2, keepdim=True)
    Rt = quaternion_to_matrix((q / length).reshape(-1, 4))
    if not with_ldj:
        return Rt, torch.zeros(R.shape[0], dtype=R.dtype, device=R.device)
    return Rt, det4(W).abs().log() - 4 * length.reshape(-1).log()


def lu_weight(sd, prefix):
    """UnconditionLU.forward (flow/squeezetrans.py:85-91)."""
    g = lambda n: sd[prefix + n]
    W = g("w_p") @ (g("w_l") * g("l_mask") + g("l_eye")) @ (
        g("w_u") * g("u_mask") + torch.diag(g("s_sign") * torch.exp(g("w_s"))))
    return W.unsqueeze(0)


def rot_weight(M):
    """rot = U^T V with (U,S,V) = torch.svd(M)  (flow/rottrans.py:15-16) -- note V, not V^T."""
    U, _, V = torch.svd(M)
    return U.transpose(-1, -2) @ V


def affine_matrix(sd, prefix, kind, feature, inverse):
    """The 4x4 matrix a layer applies in the requested direction, and whether it carries a log-det."""
    eye = torch.eye(4, dtype=next(iter(sd.values())).dtype, device=next(iter(sd.values())).device).unsqueeze(0)
    if kind == "aff_u":
        W = sd[prefix + "mat"]
    elif kind == "aff_lu":
        W = lu_weight(sd, prefix + "mat.")
    elif kind == "aff_c":
        W = conditioner(sd, prefix + "net.", feature).reshape(-1, 4, 4) + eye
    elif kind == "aff_clu":
        # ConditionLU.forward as written (flow/squeezetrans.py:121-128): torch.diag of the [N,4] tensor is the batch's diagonal
        g = lambda n: sd[prefix + "net." + n]
        low = conditioner(sd, prefix + "net.w_l_net.", feature).reshape(-1, 4, 4) * g("l_mask") + g("l_eye")
        up = conditioner(sd, prefix + "net.w_u_net.", feature).reshape(-1, 4, 4) * g("u_mask") + torch.diag(
            g("s_sign") * torch.exp(conditioner(sd, prefix + "net.w_s_net.", feature)))
        W = torch.einsum("ab,nbc,ncd->nad", g("w_p"), low, up)
    elif kind == "rot_u":
        W = rot_weight(sd[prefix + "rot"])
        return (W.transpose(-1, -2) if inverse else W), False
    elif kind == "rot_c":
        W = rot_weight(conditioner(sd, prefix + "net.", feature).reshape(-1, 4, 4) + eye)
        return (W.transpose(-1, -2) if inverse else W), False
    else:
        raise NotImplementedError(kind)
    return (torch.linalg.inv(W) if inverse else W), True


# ----------------------------------------------------------------------------------------------
# ablation layers                                (flow/squeezetrans.py:177-361, flow/rottrans.py:69-181)
# ----------------------------------------------------------------------------------------------
_GENERATORS = ((0, 1), (0, 2), (1, 2))          # G_k = e_ab - e_ba for (a, b) in this order  (squeezetrans.py:198-199)


def _generators(dtype, device):
    G = torch.zeros(3, 3, 3, dtype=dtype, device=device)
    for k, (a, b) in enumerate(_GENERATORS):
        G[k, a, b], G[k, b, a] = 1.0, -1.0
    return G


def _normalize_t(v, dv):
    """accp_normalize (squeezetrans.py:177-188): v [N,3], tangents dv [3,N,3]."""
    n = v.norm(dim=-1, keepdim=True)
    dn = (dv * v).sum(-1, keepdim=True) / n
    return v / n, dv / n - v * dn / n ** 2


def _smith_tail(c0, dc0, c1, dc1):
    """Gram-Schmidt with tangent propagation and the log-det of squeezetrans.py:209-232 (shared by calculate_9 / calculate_36)."""
    t0, dt0 = _normalize_t(c0, dc0)
    dot = (t0 * c1).sum(-1, keepdim=True)
    ddot = (dt0 * c1 + t0 * dc1).sum(-1, keepdim=True)
    t1, dt1 = _normalize_t(c1 - dot * t0, dc1 - (ddot * t0 + dot * dt0))
    t2 = torch.linalg.cross(t0, t1, dim=-1)
    dt2 = torch.linalg.cross(t0.expand_as(dt1), dt1, dim=-1) + torch.linalg.cross(dt0, t1.expand_as(dt0), dim=-1)
    T = torch.stack([t0, t1, t2], dim=-1)                       # [N,3,3], columns
    dT = torch.stack([dt0, dt1, dt2], dim=-1)                   # [3,N,3,3]
    delta = dT @ T.transpose(-1, -2)
    vec = torch.stack([delta[..., 0, 1], delta[..., 0, 2], delta[..., 1, 2]], dim=-1)    # [3(k),N,3]
    return T, det3(vec.transpose(0, 1)).abs().log()


def smith9(M, R):
    """calculate_9 (squeezetrans.py:197-232): A = M R, tangents A G_k."""
    A = M.reshape(-1, 3, 3) @ R
    dA = torch.einsum("nab,kbc->knac", A, _generators(R.dtype, R.device))
    return _smith_tail(A[..., 0], dA[..., 0], A[..., 1], dA[..., 1])


def smith36(M, R):
    """calculate_36 (squeezetrans.py:291-331): 6-D vector (R[:,0], R[:,1]) and its tangents under G_k R, mapped by the 6x6 M."""
    M = M.reshape(-1, 6, 6)
    dR = torch.einsum("kab,nbc->knac", _generators(R.dtype, R.device), R)
    v = torch.cat([R[..., 0], R[..., 1]], dim=-1)
    dv = torch.cat([dR[..., 0], dR[..., 1]], dim=-1)
    t = torch.einsum("nab,nb->na", M.expand(R.shape[0], 6, 6), v)
    dt = torch.einsum("nab,knb->kna", M.expand(R.shape[0], 6, 6), dv)
    return _smith_tail(t[..., :3], dt[..., :3], t[..., 3:], dt[..., 3:])


def polar9(M, R, left):
    """calculate_9_l / calculate_9_r (rottrans.py:69-78): U V^T of svd(M R) / svd(R M); log-det 0."""
    A = (M.reshape(-1, 3, 3) @ R) if left else (R @ M.reshape(-1, 3, 3))
    U, _, V = torch.svd(A)
    return U @ V.transpose(-1, -2), torch.zeros(R.shape[0], dtype=R.dtype, device=R.device)


def right9(M, R, inverse):
    """calculate_9_r_smith (rottrans.py:81-91)."""
    M = M.reshape(-1, 3, 3)
    m0 = M[..., 0] / M[..., 0].norm(dim=-1, keepdim=True)
    m1 = M[..., 1] - (m0 * M[..., 1]).sum(dim=-1, keepdim=True) * m0
    m1 = m1 / m1.norm(dim=-1, keepdim=True)
    Q = torch.stack([m0, m1, torch.linalg.cross(m0, m1, dim=-1)], dim=-1)
    if inverse:
        Q = Q.transpose(-1, -2)
    return R @ Q, torch.zeros(R.shape[0], dtype=R.dtype, device=R.device)


def ablation_layer(sd, prefix, kind, R, feature, inverse):
    """One ablation layer in the requested direction: the module classes of squeezetrans.py:235-361 / rottrans.py:94-181."""
    base = kind.split("_")[0]
    n = 6 if base == "smith36" else 3
    if kind.endswith("_c"):
        M = conditioner(sd, prefix + "net.", feature).reshape(-1, n, n) + torch.eye(n, dtype=R.dtype, device=R.device)
    elif kind == "smith9_lu":
        M = lu_weight(sd, prefix + "mat.")
    else:
        M = sd[prefix + "mat"].unsqueeze(0)
    if base in ("smith9", "smith36"):
        if inverse:
            M = torch.linalg.inv(M)
        return smith9(M, R) if base == "smith9" else smith36(M, R)
    if base in ("polar9l", "polar9r"):
        return polar9(M.transpose(-1, -2) if inverse else M, R, base == "polar9l")
    return right9(M, R, inverse)


# ----------------------------------------------------------------------------------------------
# the composed flow                                                       (flow/flow.py:53-92)
# ----------------------------------------------------------------------------------------------
class OracleFlow:
    """``OracleFlow(cfg, state_dict)``; ``forward/inverse(rotation[N,3,3], feature[N,F]|None) -> (rotation, ldj)``."""

    def __init__(self, cfg, state_dict, dtype=torch.float32, explicit_jacobian=False, device="cpu"):
        """``device``: "cpu" (the oracle proper).  bench.py's incumbent leg passes a CUDA device to time the same eager
        torch op sequence the reference would run on the GPU (SURVEY.md 8d) -- a baseline, never the product path."""
        self.cfg = cfg
        self.dtype = dtype
        self.device = torch.device(device)
        self.K = cfg.segments
        self.plan = layer_plan(cfg)
        for k in self.plan:
            if k is None or str(k).startswith("unsupported"):
                raise NotImplementedError(f"layer kind {k!r} is outside the hot-path scope (SURVEY.md section 2 rows 5,7)")
        self.sd = {k: torch.as_tensor(v).detach().to(self.device).to(dtype if torch.as_tensor(v).is_floating_point() else torch.as_tensor(v).dtype)
                   for k, v in state_dict.items()}
        self.explicit = explicit_jacobian

    def _run(self, R, feature, inverse):
        R = R.detach().to(self.device, self.dtype)
        feature = None if (feature is None or not self.cfg.condition) else feature.detach().to(self.device, self.dtype)
        return self._run_graph(R, feature, inverse)

    def _run_graph(self, R, feature, inverse):
        cfg = self.cfg
        rows = permute_rows(cfg, self.plan, inverse)
        ldjs = torch.zeros(R.shape[0], dtype=self.dtype, device=self.device)
        order = range(len(self.plan) - 1, -1, -1) if inverse else range(len(self.plan))
        for i in order:
            kind, pre, p = self.plan[i], f"layers.{i}.", PERMUTE_TABLE[rows[i]]
            if kind == "mobius":
                fn = mobius_inverse if inverse else mobius_forward
                R, ldj = fn(self.sd, pre, R, p, feature, self.K, self.explicit)
            elif kind.split("_")[0] in ("smith9", "smith36", "polar9l", "polar9r", "right9"):
                R, ldj = ablation_layer(self.sd, pre, kind, R, feature, inverse)
            else:
                W, has_ldj = affine_matrix(self.sd, pre, kind, feature, inverse)
                R, ldj = quat_affine(W, R, has_ldj)
            ldjs = ldjs + ldj
        return R, ldjs

    def forward(self, R, feature=None):
        with torch.no_grad():
            return self._run(R, feature, False)

    def with_grad(self, R, feature=None, inverse=False):
        """The same evaluation with autograd on (what the reference does outside torch.no_grad(): training at agent.py:87, the
        nll_grad evaluation at eval.py:468-477); make entries of ``self.sd`` / ``feature`` require grad before calling."""
        with torch.enable_grad():
            R = R.to(self.device, self.dtype)
            feature = None if (feature is None or not self.cfg.condition) else feature.to(self.device, self.dtype)
            return self._run_graph(R, feature, inverse)

    def inverse(self, R, feature=None):
        with torch.no_grad():
            return self._run(R, feature, True)

    __call__ = forward


# ----------------------------------------------------------------------------------------------
# HEALPix SO(3) grid                                                        (utils/sd.py:31-82)
# ----------------------------------------------------------------------------------------------
GRID_SIZES = tuple(72 * 8 ** l for l in range(9))


def closest_grid_level(num_queries: int) -> int:
    """get_closest_available_grid (utils/sd.py:31-34): nearest 72*8^l in log space."""
    sizes = np.asarray(GRID_SIZES, dtype=np.float64)
    return int(np.argmin(np.abs(np.log(num_queries) - np.log(sizes))))


def healpix_grid(level: int, begin: int = 0, end: int | None = None) -> torch.Tensor:
    """generate_healpix_grid (utils/sd.py:48-82): R[t*npix+b] = Rx(az_b) Rz(polar_b) Rx(tilt_t); fp64 -> fp32."""
    nside = 2 ** level
    npix = 12 * nside * nside
    ntilt = 6 * nside
    end = npix * ntilt if end is None else end
    idx = np.arange(begin, end, dtype=np.int64)
    t, b = idx // npix, idx % npix
    z, phi = pix2zphi(nside, b)
    st = np.sqrt((1 - z) * (1 + z))
    az = np.arctan2(st * np.sin(phi), st * np.cos(phi))                    # utils/sd.py:73
    polar = np.arccos(z)                                                   # :74
    tilt = np.linspace(0, 2 * np.pi, ntilt, endpoint=False)[t]            # :75

    def rx(a):
        c, s, o, l = np.cos(a), np.sin(a), np.zeros_like(a), np.ones_like(a)
        return np.stack([l, o, o, o, c, -s, o, s, c], -1).reshape(-1, 3, 3)

    def rz(a):
        c, s, o, l = np.cos(a), np.sin(a), np.zeros_like(a), np.ones_like(a)
        return np.stack([c, -s, o, s, c, o, o, o, l], -1).reshape(-1, 3, 3)

    Rs = rx(az) @ rz(polar) @ rx(tilt)
    return torch.from_numpy(Rs).to(torch.float32)                          # torch.Tensor(Rs) -> fp32 (:82)


# ----------------------------------------------------------------------------------------------
# matrix-Fisher base log-prob                                      (utils/fisher.py:67-97,209-232)
# ----------------------------------------------------------------------------------------------
def fisher_constants(A: torch.Tensor):
    """Per image: (sum of proper singular values, log c) with the type-1 normaliser (utils/fisher.py:87-91)."""
    U, S, V = torch.svd(A)
    S = S.clone()
    S[:, 2] = S[:, 2] * torch.det(U) * torch.det(V)
    c = 1.0 / torch.sqrt(8 * math.pi * (S[:, 0] + S[:, 1]) * (S[:, 2] + S[:, 1]) * (S[:, 0] + S[:, 2]))
    return S.sum(-1), c.log()


def fisher_log_prob(A: torch.Tensor, R: torch.Tensor) -> torch.Tensor:
    """MatrixFisherN._log_prob (utils/fisher.py:217-232); R is image-major [B*G,3,3] -> [B*G]."""
    B = A.shape[0]
    sumS, logc = fisher_constants(A)
    tr = (R.reshape(B, -1, 3, 3) * A.reshape(B, 1, 3, 3)).sum(-1).sum(-1)
    return ((tr - sumS.reshape(-1, 1)) - logc.reshape(-1, 1)).reshape(-1)


# ----------------------------------------------------------------------------------------------
# grid reductions                                    (agent.py:263-266, eval.py:460-462, eval.py:103)
# ----------------------------------------------------------------------------------------------
def grid_reduce(logp: torch.Tensor):
    """logp [B,G] -> (argmax int64 [B] (first index on ties), max [B], log mean exp [B])."""
    idx = torch.argmax(logp, dim=-1)
    mx = logp.gather(-1, idx[:, None])[:, 0]
    lme = torch.logsumexp(logp.double(), dim=-1) - math.log(logp.shape[-1])
    return idx, mx, lme.to(logp.dtype)


def min_geodesic_distance_rotmats(r1s: torch.Tensor, r2s: torch.Tensor) -> torch.Tensor:
    """utils/utils.py:231-235: r1s [n,3,3], r2s [n,k,3,3] -> angle to the closest rotation of each set."""
    prod = torch.einsum("nij,nkij->nk", r1s, r2s)
    return torch.acos(torch.clip((prod.max(-1).values - 1.0) / 2.0, -1.0, 1.0))


def sample_matrix_fisher(A: torch.Tensor, num_samples: int, generator: torch.Generator | None = None, b: float = 1.5,
                         oversampling_ratio: int = 8) -> torch.Tensor:
    """utils/fisher.py:117-207 (sample_bingham + sample_matrix_fisher) for ONE image, float64: batched rejection from the
    ACG envelope, first ``num_samples`` accepted candidates, R = U quat_to_rotmat(q) V^T with the proper SVD (:48-64)."""
    A = A.double()
    U, S, Vh = torch.linalg.svd(A)
    V = Vh.T.clone(); U = U.clone(); S = S.clone()
    dU, dV = torch.linalg.det(U), torch.linalg.det(V)
    U[:, 2] *= dU; V[:, 2] *= dV; S[2] *= dU * dV
    lam = torch.stack([torch.zeros((), dtype=torch.float64), 2 * (S[1] + S[2]), 2 * (S[0] + S[2]), 2 * (S[0] + S[1])])
    omega = 1.0 + 2.0 * lam / b
    std = omega ** -0.5
    m_star = math.exp(-(4 - b) / 2) * (4 / b) ** 2
    while True:
        eps = torch.randn(num_samples * oversampling_ratio, 4, generator=generator, dtype=torch.float64)
        y = std * eps
        q = y / y.norm(dim=1, keepdim=True)
        p_bing = torch.exp(-(q * lam * q).sum(-1))
        p_acg = (q * omega * q).sum(-1) ** -2
        w = torch.rand(num_samples * oversampling_ratio, generator=generator, dtype=torch.float64)
        acc = w < p_bing / (m_star * p_acg)
        if int(acc.sum()) >= num_samples:
            q = q[acc][:num_samples]
            break
    return U @ quaternion_to_matrix(q) @ V.T


def spread(logp: torch.Tensor, samples: torch.Tensor, gt: torch.Tensor) -> torch.Tensor:
    """Spread of the north star (IPDF-style; the reference has no implementation, SURVEY.md 8f N2): per image
    sum_g p_g d(R_g, R_gt) / sum_g p_g with p_g = exp(logp[b,g]) and d = min_geodesic_distance_rotmats (utils/utils.py:231-235).
    logp [B,G], samples [G,3,3] (the evaluation points grid @ offset), gt [B,K,3,3] -> [B] radians (float64)."""
    w = torch.softmax(logp.double(), dim=-1)
    prod = torch.einsum("gij,bkij->bgk", samples.double(), gt.double())
    d = torch.acos(torch.clip((prod.max(-1).values - 1.0) / 2.0, -1.0, 1.0))
    return (w * d).sum(-1)


def random_rotations(n: int, generator: torch.Generator | None = None, dtype=torch.float32) -> torch.Tensor:
    """Haar-uniform rotations from normalised Gaussian quaternions (public pytorch3d definition)."""
    o = torch.randn((n, 4), generator=generator, dtype=torch.float64)
    o = o / torch.copysign(o.norm(dim=1), o[:, 0])[:, None]
    return quaternion_to_matrix(o).to(dtype)


def simple_config(**kw) -> types.SimpleNamespace:
    base = dict(dist="mobiusflow", condition=0, layers=24, segments=64, rot="16Trans", lu=0,
                feature_dim=512, embedding=0, embedding_dim=512, last_affine=0, first_affine=1,
                frequent_permute=0)
    base.update(kw)
    return types.SimpleNamespace(**base)
