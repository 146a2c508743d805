"""Differentiable evaluation of the flow (training, agent.py:87 ``loss.backward()``; eval.py:468-477 ``nll_grad``) and the general
``config.segments`` path.

The fused tcgen05 kernels of the inference path keep nothing for a backward pass.  With autograd on, ``Flow.forward`` /
``Flow.inverse`` run layer by layer instead, like the reference does (flow/flow.py:53-92):
  * the conditioner MLP (flow/condition.py:24-30) as library GEMMs -- torch autograd supplies its backward, weight gradients included;
  * everything after it in hand-written CUDA operators with hand-written vector-Jacobian products (csrc/train_ops.cu through the C
    ABI ``rnf_train_*``): the Mobius mixture with its frame, log-det and, in the inverse direction, the 15-halving bisection and the
    implicit-function gradient of BinFind.backward (flow/mobiusflow.py:248-273); the quaternion affine map calculate_16; and the
    ablation layers (36Trans, 9Trans*: csrc/ablation_layers.cuh) with their log-det.
Rotation gradients are carried in the tangent space of SO(3) (see csrc/train_ops.cu): parameter and feature gradients equal the
reference's; ``rotation.grad`` of the input is the tangential part of the reference's (the normal part of a gradient with respect to
a rotation matrix has no meaning on the manifold)."""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from . import _cabi, engine


class MobiusMixture(torch.autograd.Function):
    """(R [N,3,3], out [N,4K]) -> (R' [N,3,3], ldj [N]) for one Mobius layer in either direction (rnf_train_mobius_*)."""

    @staticmethod
    def forward(ctx, R, out, perm: int, inverse: bool, K: int):
        R, out = R.contiguous().float(), out.contiguous().float()
        N = R.shape[0]
        R_out, ldj, theta = torch.empty_like(R), R.new_empty(N), R.new_empty(N)
        _cabi.launch("rnf_train_mobius_forward", R.device, R, out, N, K, perm, int(inverse), R_out, ldj, theta)
        ctx.save_for_backward(R, out, theta, R_out)
        ctx.meta = (perm, inverse, K)
        return R_out, ldj

    @staticmethod
    @once_differentiable
    def backward(ctx, G_Rout, g_ldj):
        R, out, theta, R_out = ctx.saved_tensors
        perm, inverse, K = ctx.meta
        N = R.shape[0]
        G_Rout = torch.zeros_like(R) if G_Rout is None else G_Rout.contiguous().float()
        g_ldj = R.new_zeros(N) if g_ldj is None else g_ldj.contiguous().float()
        G_R, G_out = torch.empty_like(R), torch.empty_like(out)
        _cabi.launch("rnf_train_mobius_backward", R.device, R, out, N, K, perm, int(inverse), theta, R_out, G_Rout, g_ldj, G_R, G_out)
        return G_R, G_out, None, None, None


class QuatAffine(torch.autograd.Function):
    """(R [N,3,3], W [N,4,4]) -> (R' = q2m(W q / |W q|), log|W q|)   (calculate_16, flow/squeezetrans.py:33-38; rnf_train_affine_*)."""

    @staticmethod
    def forward(ctx, R, W):
        R, W = R.contiguous().float(), W.contiguous().float()
        N = R.shape[0]
        R_out, loglen = torch.empty_like(R), R.new_empty(N)
        _cabi.launch("rnf_train_affine_forward", R.device, R, W, N, R_out, loglen)
        ctx.save_for_backward(R, W, R_out)
        return R_out, loglen

    @staticmethod
    @once_differentiable
    def backward(ctx, G_Rout, g_loglen):
        R, W, R_out = ctx.saved_tensors
        N = R.shape[0]
        G_Rout = torch.zeros_like(R) if G_Rout is None else G_Rout.contiguous().float()
        g_loglen = R.new_zeros(N) if g_loglen is None else g_loglen.contiguous().float()
        G_R, G_W = torch.empty_like(R), torch.empty_like(W)
        _cabi.launch("rnf_train_affine_backward", R.device, R, W, N, R_out, G_Rout, g_loglen, G_R, G_W)
        return G_R, G_W


class AblationLayer(torch.autograd.Function):
    """(R [N,3,3], M [N,n,n], kind) -> (R', ldj) for one ablation layer (csrc/ablation_layers.cuh; rnf_train_ablation_*).  M is the
    matrix the layer applies in this direction; ldj is the Smith layers' log-det by tangent propagation (0 for the others)."""

    @staticmethod
    def forward(ctx, R, M, kind: int):
        R, M = R.contiguous().float(), M.contiguous().float()
        N = R.shape[0]
        R_out, ldj = torch.empty_like(R), R.new_empty(N)
        _cabi.launch("rnf_train_ablation_forward", R.device, R, M, N, kind, R_out, ldj)
        ctx.save_for_backward(R, M, R_out)
        ctx.kind = kind
        return R_out, ldj

    @staticmethod
    @once_differentiable
    def backward(ctx, G_Rout, g_ldj):
        R, M, R_out = ctx.saved_tensors
        N = R.shape[0]
        G_Rout = torch.zeros_like(R) if G_Rout is None else G_Rout.contiguous().float()
        g_ldj = R.new_zeros(N) if g_ldj is None else g_ldj.contiguous().float()
        G_R, G_M = torch.empty_like(R), torch.empty_like(M)
        _cabi.launch("rnf_train_ablation_backward", R.device, R, M, N, ctx.kind, R_out, G_Rout, g_ldj, G_R, G_M)
        return G_R, G_M, None


class FusedLogDensity(torch.autograd.Function):
    """(R [N,3,3], Mobius images, unconditional affine blocks, per-image constants) -> (R' [N,3,3], ldj [N]) of the forward direction
    in the fused training kernels (csrc/flow_grad.cu through rnf_flow_train_forward / rnf_flow_train_backward).  The gradients it
    returns are with respect to the packed image and constants of engine.TrainProgram; autograd through the packing
    (engine.mobius_images, engine.affine_blocks, engine.condition_torch) carries them to the parameters and the features."""

    @staticmethod
    def forward(ctx, tp, R, idx32, B: int, mob, aff, cond):
        weights = tp.weights(mob, aff)
        R_out, ldj = tp.forward(weights, R, cond, B, idx32)
        ctx.tp, ctx.B, ctx.idx32, ctx.weights = tp, B, idx32, weights
        ctx.save_for_backward(R, cond)
        return R_out, ldj

    @staticmethod
    @once_differentiable
    def backward(ctx, G_Rout, g_ldj):
        R, cond = ctx.saved_tensors
        G_Rout = None if G_Rout is None else G_Rout.contiguous().float()
        g_ldj = R.new_zeros(R.shape[0]) if g_ldj is None else g_ldj.contiguous().float()
        G_R, g_mob, g_aff, g_cond = ctx.tp.backward(ctx.weights, R, cond, ctx.B, ctx.idx32, G_Rout, g_ldj)
        return None, G_R, None, None, g_mob, g_aff, g_cond


def fused_run(tp, layers, R, feature, idx32, B: int):
    """(R', ldj) of the forward direction through FusedLogDensity; feature [B,F] one row per image (None if unconditional),
    idx32 [N] row -> image."""
    mob, aff = tp.images()
    cond = engine.condition_torch(layers, feature) if tp.cond_floats else None
    return FusedLogDensity.apply(tp, R, idx32, B, mob, aff, cond)


def _affine_matrix(layer, rows, inverse: bool):
    """The 4x4 a layer applies in this direction ([1,4,4] or [N,4,4], differentiable torch algebra) and whether it has a log-det."""
    eye = None
    kind = layer.kind
    if kind == "aff_u":
        W = layer.mat
    elif kind == "aff_lu":
        W = layer.mat()
    elif kind in ("aff_c", "rot_c"):
        eye = torch.eye(4, device=rows.device, dtype=rows.dtype)
        W = engine.conditioner_torch(layer.net, rows).reshape(-1, 4, 4) + eye
    elif kind == "aff_clu":
        W = layer.net.weight(rows)                            # batch-coupled in the reference; reproduced as written
    elif kind == "rot_u":
        W = layer.rot
    else:
        raise NotImplementedError(f"layer kind {kind!r} has no differentiable / general-segments path")
    if kind.startswith("rot"):
        U, _, V = torch.svd(W)                                # flow/rottrans.py:15-16 (note V, not V^T)
        W = U.transpose(-1, -2) @ V
        return (W.transpose(-1, -2) if inverse else W), False
    return (torch.linalg.inv(W) if inverse else W), True


def _ablation_matrix(layer, base: str, rows, inverse: bool):
    """The n x n matrix an ablation layer applies in this direction ([1,n,n] or [N,n,n], differentiable torch algebra), as
    engine.ablation_blocks packs it for the fused kernels: inv(M) of the Smith layers and M^T of the SVD layers in the inverse
    direction, the Gram-Schmidt Q (Q^T inverse) of calculate_9_r_smith."""
    if layer.kind.endswith("_c"):
        n = layer.n
        M = engine.conditioner_torch(layer.net, rows).reshape(-1, n, n) + torch.eye(n, device=rows.device, dtype=rows.dtype)
    elif isinstance(layer.mat, torch.nn.Module):
        M = layer.mat()                                       # Uncondition9TransLU: UnconditionLU.forward, [1,3,3]
    else:
        M = layer.mat.unsqueeze(0)
    if base in ("smith9", "smith36"):
        return torch.linalg.inv(M) if inverse else M
    if base in ("polar9l", "polar9r"):
        return M.transpose(-1, -2) if inverse else M
    Q = engine.gram_schmidt_columns(M)
    return Q.transpose(-1, -2) if inverse else Q


def composed_run(layers, perms, rotation, feature_rows, inverse: bool):
    """flow/flow.py:53-92 layer by layer with the differentiable operators.  ``feature_rows`` [N,F] row-aligned (or None)."""
    R = rotation.to(torch.float32)
    N = R.shape[0]
    ldjs = R.new_zeros(N)
    order = range(len(layers) - 1, -1, -1) if inverse else range(len(layers))
    for i in order:
        layer, p0 = layers[i], int(perms[i]) % 3
        if layer.kind == "mobius":
            y = R[:, :, (p0 + 1) % 3]
            inp = torch.cat((y, feature_rows), dim=-1) if layer.condition else y          # flow/mobiusflow.py:52-56
            out = engine.conditioner_torch(layer.conditioner, inp)
            R, ldj = MobiusMixture.apply(R, out, p0, inverse, layer.K)
        elif layer.kind.split("_")[0] in engine.ABLATION_KINDS:
            base = layer.kind.split("_")[0]
            M = _ablation_matrix(layer, base, feature_rows, inverse)
            R, ldj = AblationLayer.apply(R, M.expand(N, M.shape[-2], M.shape[-1]), engine.ABLATION_KINDS[base])
        else:
            W, has_ldj = _affine_matrix(layer, feature_rows, inverse)
            R, loglen = QuatAffine.apply(R, W.expand(N, 4, 4))
            ldj = (torch.linalg.slogdet(W)[1] - 4.0 * loglen) if has_ldj else torch.zeros_like(loglen)
        ldjs = ldjs + ldj
    return R, ldjs
