"""Prototype (float64, CPU) of the vector-Jacobian products of the ablation layers (csrc/ablation_layers.cuh), checked against
autograd through the oracle restatement of the reference (oracle/rnf_oracle.py smith9 / smith36 / polar9 / right9).  Not product
code: ablation_bwd_kernel in csrc/train_ops.cu implements exactly these formulas, in the same order.

Shapes follow the kernel: one row per rotation, tangents indexed [row, k, i] for the three generators k.  Every function takes the
upstream G' = dL/dR' and g = dL/dldj and returns the MATRIX gradient with respect to R (the kernel then keeps its tangential part)
and the gradient with respect to the layer's matrix M in this direction."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from oracle import rnf_oracle as orc


def vee(R, G):
    """tangent (body-frame) vector of a matrix gradient G at R: g_i = <G, R [e_i]x>"""
    H = R.transpose(1, 2) @ G
    return torch.stack([H[:, 2, 1] - H[:, 1, 2], H[:, 0, 2] - H[:, 2, 0], H[:, 1, 0] - H[:, 0, 1]], dim=1)


def hat(g):
    Z = torch.zeros_like(g[:, 0])
    return torch.stack([torch.stack([Z, -g[:, 2], g[:, 1]], 1), torch.stack([g[:, 2], Z, -g[:, 0]], 1), torch.stack([-g[:, 1], g[:, 0], Z], 1)], 1)


def dot(a, b):
    return (a * b).sum(-1, keepdim=True)


def cross(a, b):
    return torch.linalg.cross(*torch.broadcast_tensors(a, b), dim=-1)


# ---- forward pieces (the arithmetic of ablation_layers.cuh) ------------------------------------------------------------------
def normalize_t(v, d):
    """t = v/|v|, dt_k = d_k/|v| - v (v.d_k)/|v|^3;  v [N,3], d [N,3,3]"""
    inv = 1.0 / v.norm(dim=-1, keepdim=True)
    s = (d * v[:, None]).sum(-1, keepdim=True)                       # [N,3,1]
    return inv * v, inv[:, None] * d - (inv ** 3)[:, None] * s * v[:, None]


def smith_tail_fwd(c0, dc0, c1, dc1):
    t0, dt0 = normalize_t(c0, dc0)
    dt = dot(t0, c1)
    ddot = (dt0 * c1[:, None]).sum(-1, keepdim=True) + (t0[:, None] * dc1).sum(-1, keepdim=True)
    raw1, draw1 = c1 - dt * t0, dc1 - (ddot * t0[:, None] + dt[:, None] * dt0)
    t1, dt1 = normalize_t(raw1, draw1)
    t2 = cross(t0, t1)
    dt2 = cross(t0[:, None].expand_as(dt1), dt1) + cross(dt0, t1[:, None].expand_as(dt0))
    T = torch.stack([t0, t1, t2], -1)
    dT = torch.stack([dt0, dt1, dt2], -1)                            # [N,k,3(a),3(c)]
    delta = dT @ T[:, None].transpose(-1, -2)
    V = torch.stack([delta[..., 0, 1], delta[..., 0, 2], delta[..., 1, 2]], -1)   # [N,k,3]
    return T, torch.linalg.det(V).abs().log(), dict(t0=t0, dt0=dt0, dot=dt, ddot=ddot, raw1=raw1, draw1=draw1, t1=t1, dt1=dt1,
                                                    t2=t2, dt2=dt2, V=V)


# ---- reverse sweep ----------------------------------------------------------------------------------------------------------
def normalize_bwd(v, d, Gt, Gdt):
    """VJP of normalize_t: (v [N,3], d [N,3,3]) <- (G_t [N,3], G_dt [N,3,3]).  dt_k = i d_k - i^3 s_k v, i = 1/|v|, s_k = v.d_k;
    the second-order terms (dt_k depends on v through i, i^3 and s_k) feed the log-det gradient."""
    i = 1.0 / v.norm(dim=-1, keepdim=True)                           # [N,1]
    s = (d * v[:, None]).sum(-1)                                     # [N,3]  s_k = v.d_k
    a = (Gdt * d).sum(-1)                                            # [N,3]  G_dt_k . d_k
    b = (Gdt * v[:, None]).sum(-1)                                   # [N,3]  G_dt_k . v
    Gd = i[:, None] * Gdt - (i ** 3)[:, None] * b[..., None] * v[:, None]
    i3, i5 = i ** 3, i ** 5
    Gv = i * Gt - i3 * dot(v, Gt) * v
    Gv = Gv + (-i3 * a.sum(-1, keepdim=True) + 3 * i5 * (s * b).sum(-1, keepdim=True)) * v \
        - i3 * (b[..., None] * d).sum(1) - i3 * (s[..., None] * Gdt).sum(1)
    return Gv, Gd


def smith_tail_bwd(c0, dc0, c1, dc1, GT, gL):
    """VJP of the Gram-Schmidt with tangents and log|det V|: (c0, dc0, c1, dc1) <- (G_T [N,3,3], g_ldj [N])."""
    _, _, f = smith_tail_fwd(c0, dc0, c1, dc1)
    t0, dt0, t1, dt1, t2, dt2, V = f["t0"], f["dt0"], f["t1"], f["dt1"], f["t2"], f["dt2"], f["V"]
    GV = gL[:, None, None] * torch.linalg.inv(V).transpose(-1, -2)   # d log|det V| = V^{-T}
    # delta_k[a][b] = sum_c dt_c,k[a] t_c[b];  E_k carries G_V into entries (0,1), (0,2), (1,2)
    E = torch.zeros(V.shape[0], 3, 3, 3, dtype=V.dtype)
    E[:, :, 0, 1], E[:, :, 0, 2], E[:, :, 1, 2] = GV[..., 0], GV[..., 1], GV[..., 2]
    ts, dts = (t0, t1, t2), (dt0, dt1, dt2)
    Gt = [GT[:, :, c].clone() for c in range(3)]
    Gdt = [(E @ ts[c][:, None, :, None])[..., 0] for c in range(3)]                  # E_k t_c
    for c in range(3):
        Gt[c] = Gt[c] + (E.transpose(-1, -2) @ dts[c][..., None])[..., 0].sum(1)    # sum_k E_k^T dt_c,k
    # dt2_k = t0 x dt1_k + dt0_k x t1 ; t2 = t0 x t1      (z = a x b: G_a = b x G_z, G_b = G_z x a)
    Gt[0] = Gt[0] + cross(dt1, Gdt[2]).sum(1) + cross(t1, Gt[2])
    Gt[1] = Gt[1] + cross(Gdt[2], dt0).sum(1) + cross(Gt[2], t0)
    Gdt[1] = Gdt[1] + cross(Gdt[2], t0[:, None].expand_as(Gdt[2]))
    Gdt[0] = Gdt[0] + cross(t1[:, None].expand_as(Gdt[2]), Gdt[2])
    Graw1, Gdraw1 = normalize_bwd(f["raw1"], f["draw1"], Gt[1], Gdt[1])
    # draw1_k = dc1_k - ddot_k t0 - dot dt0_k ; ddot_k = dt0_k.c1 + t0.dc1_k ; raw1 = c1 - dot t0 ; dot = t0.c1
    d_, dd = f["dot"], f["ddot"]                                     # [N,1], [N,3,1]
    Gdc1 = Gdraw1.clone()
    Gddot = -(Gdraw1 * t0[:, None]).sum(-1, keepdim=True)            # [N,3,1]
    G_t0 = Gt[0] - (dd * Gdraw1).sum(1)
    Gdot = -(Gdraw1 * dt0).sum(-1).sum(-1, keepdim=True)
    Gdt0 = Gdt[0] - d_[:, None] * Gdraw1
    Gdt0 = Gdt0 + Gddot * c1[:, None]
    Gc1 = (Gddot * dt0).sum(1)
    G_t0 = G_t0 + (Gddot * dc1).sum(1)
    Gdc1 = Gdc1 + Gddot * t0[:, None]
    Gc1 = Gc1 + Graw1
    Gdot = Gdot - dot(Graw1, t0)
    G_t0 = G_t0 - d_ * Graw1
    G_t0 = G_t0 + Gdot * c1
    Gc1 = Gc1 + Gdot * t0
    Gc0, Gdc0 = normalize_bwd(c0, dc0, G_t0, Gdt0)
    return Gc0, Gdc0, Gc1, Gdc1


def smith9_vjp(M, R, G, gL):
    """calculate_9: A = M R, c0 = a0, c1 = a1, dc0 = (-a1, -a2, 0), dc1 = (a0, 0, -a2)."""
    A = M @ R
    a0, a1, a2 = A[..., 0], A[..., 1], A[..., 2]
    z = torch.zeros_like(a0)
    dc0, dc1 = torch.stack([-a1, -a2, z], 1), torch.stack([a0, z, -a2], 1)
    Gc0, Gdc0, Gc1, Gdc1 = smith_tail_bwd(a0, dc0, a1, dc1, G, gL)
    GA = torch.stack([Gc0 + Gdc1[:, 0], Gc1 - Gdc0[:, 0], -Gdc0[:, 1] - Gdc1[:, 2]], -1)
    return M.transpose(-1, -2) @ GA, GA @ R.transpose(-1, -2)


def _gen_tangents(u):
    """G_k u for G_0 = e01 - e10, G_1 = e02 - e20, G_2 = e12 - e21:  (u1, -u0, 0), (u2, 0, -u0), (0, u2, -u1)"""
    z = torch.zeros_like(u[:, 0])
    return torch.stack([torch.stack([u[:, 1], -u[:, 0], z], -1), torch.stack([u[:, 2], z, -u[:, 0]], -1),
                        torch.stack([z, u[:, 2], -u[:, 1]], -1)], 1)


def smith36_vjp(M6, R, G, gL):
    """calculate_36: v = (r0, r1), dv_k = (G_k r0, G_k r1), t = M6 v, dt_k = M6 dv_k."""
    r0, r1 = R[..., 0], R[..., 1]
    v = torch.cat([r0, r1], -1)
    dv = torch.cat([_gen_tangents(r0), _gen_tangents(r1)], -1)       # [N,3,6]
    t = (M6 @ v[..., None])[..., 0]
    dt = dv @ M6.transpose(-1, -2)
    Gc0, Gdc0, Gc1, Gdc1 = smith_tail_bwd(t[:, :3], dt[..., :3], t[:, 3:], dt[..., 3:], G, gL)
    Gt, Gdt = torch.cat([Gc0, Gc1], -1), torch.cat([Gdc0, Gdc1], -1)
    GM = Gt[..., None] * v[:, None] + Gdt.transpose(1, 2) @ dv      # G_t v^T + sum_k G_dt_k dv_k^T
    Gv = (M6.transpose(-1, -2) @ Gt[..., None])[..., 0]
    Gdv = Gdt @ M6                                                   # [N,k,6]: M6^T G_dt_k
    GR = torch.zeros_like(R)
    for h in range(2):
        g, gd = Gv[:, 3 * h:3 * h + 3].clone(), Gdv[..., 3 * h:3 * h + 3]
        g[:, 0] += -gd[:, 0, 1] - gd[:, 1, 2]
        g[:, 1] += gd[:, 0, 0] - gd[:, 2, 2]
        g[:, 2] += gd[:, 1, 0] + gd[:, 2, 1]
        GR[..., h] = g
    return GR, GM


def polar_fwd(A):
    U, _, V = torch.svd(A)
    return U @ V.transpose(-1, -2)


def polar_vjp(M, R, G, left):
    """R' = polar(A), A = M R (left) or R M: H = R'^T A, X = R'^T G', x = vee(X - X^T), y = ((tr H) I - H)^{-1} x, G_A = R' [y]x."""
    A = M @ R if left else R @ M
    Q = polar_fwd(A)
    H = Q.transpose(-1, -2) @ A
    X = Q.transpose(-1, -2) @ G
    x = torch.stack([X[:, 2, 1] - X[:, 1, 2], X[:, 0, 2] - X[:, 2, 0], X[:, 1, 0] - X[:, 0, 1]], 1)
    K = H.diagonal(dim1=-2, dim2=-1).sum(-1)[:, None, None] * torch.eye(3, dtype=H.dtype) - H
    y = torch.linalg.solve(K, x[..., None])[..., 0]
    GA = Q @ hat(y)
    if left:
        return M.transpose(-1, -2) @ GA, GA @ R.transpose(-1, -2)
    return GA @ M.transpose(-1, -2), R.transpose(-1, -2) @ GA


def right9_vjp(Q, R, G):
    """R' = R Q:  G_R = G' Q^T, G_Q = R^T G'."""
    return G @ Q.transpose(-1, -2), R.transpose(-1, -2) @ G


# ---- checks ------------------------------------------------------------------------------------------------------------------
def _errors(ref_R, ref_M, R, GR, GM):
    tr, tp = vee(R, ref_R), vee(R, GR)
    return ((tp - tr).abs().max() / tr.abs().max()).item(), ((GM - ref_M).abs().max() / ref_M.abs().max()).item()


def check(N: int = 64, scale: float = 0.3, seed: int = 1) -> dict:
    """Worst relative errors (tangential rotation gradient, matrix gradient) of each prototype VJP against oracle autograd,
    loss = <A, R'> + c . ldj, with per-row matrices M = I + scale * randn."""
    g = torch.Generator().manual_seed(seed)
    R = orc.random_rotations(N, g, torch.float64)
    A = torch.randn(N, 3, 3, generator=g, dtype=torch.float64)
    c = torch.randn(N, generator=g, dtype=torch.float64)
    out = {}

    def ref(fn, M):
        Rr, Mr = R.clone().requires_grad_(True), M.clone().requires_grad_(True)
        Ro, lo = fn(Mr, Rr)
        ((A * Ro).sum() + (c * lo).sum()).backward()
        return Rr.grad, Mr.grad

    M3 = torch.eye(3, dtype=torch.float64) + scale * torch.randn(N, 3, 3, generator=g, dtype=torch.float64)
    M6 = torch.eye(6, dtype=torch.float64) + scale * torch.randn(N, 6, 6, generator=g, dtype=torch.float64)
    T, _, _ = smith_tail_fwd(*_smith9_inputs(M3, R))
    assert (T - orc.smith9(M3, R)[0]).abs().max() < 1e-12
    out["smith9"] = _errors(*ref(orc.smith9, M3), R, *smith9_vjp(M3, R, A, c))
    out["smith36"] = _errors(*ref(orc.smith36, M6), R, *smith36_vjp(M6, R, A, c))
    for left, name in ((True, "polar9l"), (False, "polar9r")):
        out[name] = _errors(*ref(lambda M, Rr: orc.polar9(M, Rr, left), M3), R, *polar_vjp(M3, R, A, left))
    # right9: only G_R = G' Q^T and G_Q = R^T G' are hand-written (exact products, hence errors of 0); torch autograd carries G_Q
    # through the Gram-Schmidt to M, as train.py does.  This checks that composition and the Q / Q^T choice of both directions.
    for inverse in (False, True):
        Mr = M3.clone().requires_grad_(True)
        Q = orc.right9(Mr, torch.eye(3, dtype=torch.float64).expand(N, 3, 3), inverse)[0]
        GR, GQ = right9_vjp(Q.detach(), R, A)
        GM, = torch.autograd.grad(Q, Mr, GQ)
        out["right9" + ("_inv" if inverse else "")] = _errors(*ref(lambda M, Rr: orc.right9(M, Rr, inverse), M3), R, GR, GM)
    return out


def _smith9_inputs(M, R):
    A = M @ R
    a0, a1, a2 = A[..., 0], A[..., 1], A[..., 2]
    z = torch.zeros_like(a0)
    return a0, torch.stack([-a1, -a2, z], 1), a1, torch.stack([a0, z, -a2], 1)


if __name__ == "__main__":
    for scale in (1e-3, 0.3):
        for k, (eR, eM) in check(scale=scale).items():
            print(f"M = I + {scale:g} randn  {k:10s} tangent dR err {eR:.2e}  dM err {eM:.2e}")
