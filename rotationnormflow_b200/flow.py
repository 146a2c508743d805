"""Drop-in replacement for the reference's ``flow/flow.py`` (and the layer classes it instantiates).

Same public surface, same constructor semantics, same ``state_dict`` keys -- checkpoints written by
``Agent.save_ckpt`` (agent.py:111-153, key ``flow_state_dict``) load with ``load_state_dict``:

    get_flow(config) -> Flow                                             flow/flow.py:9-10
    Flow.forward(rotation, feature=None, inverse=False, draw=False)      flow/flow.py:53-72
    Flow.inverse(rotation, feature=None, draw=False)                     flow/flow.py:74-92
    layer(rotation, permute, feature) / layer.inverse(...)               per-layer protocol of flow/*.py

but every call runs as ONE fused CUDA kernel over the whole layer stack (csrc/flow_v1.cu, csrc/flow_t4.cu, csrc/flow_row.cu)
instead of ~6.5 k (forward) / ~22 k (inverse) ATen launches.  The modules below only hold parameters; they
contain no per-rotation PyTorch arithmetic and there is no CPU path: tensors must live on a B200.

Additions that the reference does not have (N1 in SURVEY.md section 8f):
    Flow.forward(..., feature_index=idx)   features given once per image [B,F] plus a row->image index
    Flow.grid_log_prob(grid, feature, ...) fused log-prob / arg-max / normaliser over a rotation grid
"""
from __future__ import annotations

import numpy as np
import torch
from torch import nn

from . import engine

_PERMUTE_ROWS = ((0, 1, 2), (1, 2, 0), (2, 0, 1), (0, 1, 2), (1, 2, 0), (2, 0, 1))   # flow/flow.py:13-15


def get_flow(config):
    return Flow(config)


class _NoProgramState:
    """Mixin: the packed-program cache holds device pointers and a ctypes handle; it is rebuilt on demand and must not travel
    through copy.deepcopy / pickle / torch.save of the module."""

    _CACHES = ("_rnf_programs", "_rnf_train_programs")      # set by _program and _train_program

    def invalidate_cache(self):
        """Forget the packed weights (needed only after writes that bypass autograd versioning, e.g. ``p.data.copy_()``)."""
        for k in self._CACHES:
            self.__dict__.pop(k, None)

    def __getstate__(self):
        return {k: v for k, v in self.__dict__.items() if k not in self._CACHES}


# ------------------------------------------------------------------------------------------------------
# parameter containers (state-dict compatible with the reference modules)
# ------------------------------------------------------------------------------------------------------
class ConditionalTransform(nn.Module):
    """Parameters of the 4-layer residual ReLU MLP of flow/condition.py:4-30 (Ni -> 64 -> 64 -> 64 -> 64 -> No).

    Keys: fc_first.{weight,bias}, layers.{1,3,5}.{weight,bias}, fc_last.{weight,bias}.  Creation order matches the
    reference so that a seeded construction draws identical initial weights."""

    def __init__(self, Ni: int, No: int, Nh: int = 64):
        super().__init__()
        self.fc_first = nn.Linear(Ni, Nh)
        hidden = []
        for _ in range(3):
            hidden += [nn.ReLU(), nn.Linear(Nh, Nh)]
        self.relu_last = nn.ReLU()
        self.fc_last = nn.Linear(Nh, No)
        self.layers = nn.ModuleList(hidden)

    def forward(self, x):  # pragma: no cover - deliberately not a compute path
        raise RuntimeError("ConditionalTransform is evaluated inside the fused CUDA kernels; call the owning layer / Flow")


class _FusedLayer(_NoProgramState, nn.Module):
    """Common per-layer protocol: ``layer(rotation, permute, feature)`` and ``layer.inverse(...)``."""

    kind = ""
    uses_feature = False

    def _feature_dim(self) -> int:
        return 0

    def forward(self, rotation, permute=None, feature=None):
        return _run([self], [_perm_row(permute, self)], self._feature_dim(), self, rotation, feature, False)

    def inverse(self, rotation, permute=None, feature=None):
        return _run([self], [_perm_row(permute, self)], self._feature_dim(), self, rotation, feature, True)


class MobiusFlow(_FusedLayer):
    """flow/mobiusflow.py:27-183.  ``conditioner`` = ConditionalTransform(D + feature_dim, 4K)."""

    kind = "mobius"

    def __init__(self, D, K, condition=0, feature_dim=None):
        super().__init__()
        if D != 3:
            raise ValueError("MobiusFlow acts on columns of a 3x3 rotation: D must be 3")
        if K < 1:
            raise ValueError("MobiusFlow needs at least one mixture component")
        # K = 64 (every settings/*.yml) runs in the fused tcgen05 kernels; any other K in the per-layer operators of train.py
        self.D, self.K = D, K
        self.condition = condition
        self.feature_dim = feature_dim
        self.uses_feature = bool(condition)
        self.conditioner = ConditionalTransform(D + (feature_dim if condition else 0), 4 * K)

    def _feature_dim(self):
        return self.feature_dim if self.condition else 0

    def forward(self, rotation, permute=None, feature=None):
        assert permute is not None, "The permuting function is needed in this module"
        if self.condition:
            assert feature is not None, "The input feature is needed in this module"
        return super().forward(rotation, permute, feature if self.condition else None)

    def inverse(self, rotation, permute=None, feature=None):
        assert permute is not None, "The permuting function is needed in this module"
        if self.condition:
            assert feature is not None, "feature input is needed in this module"
        return super().inverse(rotation, permute, feature if self.condition else None)


class Uncondition16Trans(_FusedLayer):
    """flow/squeezetrans.py:161-174: a free 4x4 matrix acting on the quaternion."""

    kind = "aff_u"

    def __init__(self):
        super().__init__()
        self.mat = nn.Parameter(torch.eye(4).unsqueeze(0) + torch.randn(1, 4, 4) * 1e-3)

    def matrix(self):
        return self.mat


class UnconditionLU(nn.Module):
    """flow/squeezetrans.py:58-91: PLU parameterisation W = P (L*lmask + I) (U*umask + diag(sign*exp(s)))."""

    def __init__(self, in_channel: int):
        super().__init__()
        from scipy import linalg as la
        w0 = 1e-3 * np.random.randn(in_channel, in_channel) + np.eye(in_channel)
        q, _ = la.qr(w0)
        p, l, u = la.lu(q.astype(np.float32))
        s = np.diag(u)
        u = np.triu(u, 1)
        um = np.triu(np.ones_like(u), 1)
        self.register_buffer("w_p", torch.from_numpy(p))
        self.register_buffer("u_mask", torch.from_numpy(um))
        self.register_buffer("l_mask", torch.from_numpy(um.T.copy()))
        s_t = torch.from_numpy(np.copy(s))
        self.register_buffer("s_sign", torch.sign(s_t))
        self.register_buffer("l_eye", torch.eye(in_channel))
        self.w_l = nn.Parameter(torch.from_numpy(l))
        self.w_s = nn.Parameter(s_t.abs().log())
        self.w_u = nn.Parameter(torch.from_numpy(u))

    def forward(self):
        """Parameter algebra on one 4x4 (not a per-rotation path): returns W [1,4,4]."""
        low = self.w_l * self.l_mask + self.l_eye
        up = self.w_u * self.u_mask + torch.diag(self.s_sign * torch.exp(self.w_s))
        return (self.w_p @ low @ up).unsqueeze(0)


class Uncondition16TransLU(_FusedLayer):
    """flow/squeezetrans.py:147-158."""

    kind = "aff_lu"

    def __init__(self):
        super().__init__()
        self.mat = UnconditionLU(4)

    def matrix(self):
        with torch.no_grad():
            return self.mat()


class ConditionLU(nn.Module):
    """flow/squeezetrans.py:94-129: the feature-conditioned PLU parameterisation, reproduced as written.  NOTE the reference applies
    ``torch.diag`` to the [N,n] output of ``w_s_net``: that returns the DIAGONAL of the batch (entry j of row j, j < n) and broadcasts
    it over the columns of every row's U factor -- the layer is batch-coupled (rows 0..n-1 of the feature batch decide ``d`` for all
    rows).  With the reference's own calling convention (one image's feature repeated, eval.py:450) it is well defined per image."""

    def __init__(self, in_channel: int, feature_dim: int):
        super().__init__()
        from scipy import linalg as la
        self.in_channel = in_channel
        q, _ = la.qr(np.random.randn(in_channel, in_channel))
        p, l, u = la.lu(q.astype(np.float32))
        s = np.diag(u)
        um = np.triu(np.ones_like(np.triu(u, 1)), 1)
        self.register_buffer("w_p", torch.from_numpy(p))
        self.register_buffer("u_mask", torch.from_numpy(um))
        self.register_buffer("l_mask", torch.from_numpy(um.T.copy()))
        self.register_buffer("s_sign", torch.sign(torch.from_numpy(np.copy(s))))
        self.register_buffer("l_eye", torch.eye(in_channel))
        self.w_l_net = ConditionalTransform(feature_dim, in_channel * in_channel)
        self.w_u_net = ConditionalTransform(feature_dim, in_channel * in_channel)
        self.w_s_net = ConditionalTransform(feature_dim, in_channel)

    def weight(self, feature):
        """[N,n,n], the expression of flow/squeezetrans.py:121-128 (library GEMMs on the feature rows; differentiable)."""
        n = self.in_channel
        low = engine.conditioner_torch(self.w_l_net, feature).reshape(-1, n, n) * self.l_mask + self.l_eye
        up = engine.conditioner_torch(self.w_u_net, feature).reshape(-1, n, n) * self.u_mask \
            + torch.diag(self.s_sign * torch.exp(engine.conditioner_torch(self.w_s_net, feature)))
        return torch.einsum("ab,nbc,ncd->nad", self.w_p, low, up)


class Condition16TransLU(_FusedLayer):
    """flow/squeezetrans.py:132-144.  Batch-coupled (see ConditionLU): always evaluated by the per-layer operators of train.py."""

    kind = "aff_clu"
    uses_feature = True

    def __init__(self, feature_dim):
        super().__init__()
        self.feature_dim = feature_dim
        self.net = ConditionLU(4, feature_dim)

    def _feature_dim(self):
        return self.feature_dim


class Condition16Trans(_FusedLayer):
    """flow/squeezetrans.py:41-55: W = MLP(feature).reshape(4,4) + I, evaluated once per image on device."""

    kind = "aff_c"
    uses_feature = True

    def __init__(self, feature_dim):
        super().__init__()
        self.feature_dim = feature_dim
        self.net = ConditionalTransform(feature_dim, 16)

    def _feature_dim(self):
        return self.feature_dim


class UnconditionRot(_FusedLayer):
    """flow/rottrans.py:8-35: 4-D rotation U^T V from torch.svd of a free 4x4; log-det 0."""

    kind = "rot_u"

    def __init__(self):
        super().__init__()
        self.rot = nn.Parameter(torch.randn((1, 4, 4)) * 1e-3 + torch.eye(4).unsqueeze(0))

    def matrix(self):
        # U^T V depends on the sign convention of the SVD routine (engine.Program._polar_factor): evaluated where the reference
        # would evaluate it -- on the parameter's own device -- unless RNF_SVD_BACKEND=cpu asks for the LAPACK convention
        with torch.no_grad():
            M = self.rot.detach()
            U, _, V = torch.svd(M.to("cpu") if engine.svd_backend() == "cpu" else M)
            return U.transpose(-1, -2) @ V


class ConditionRot(_FusedLayer):
    """flow/rottrans.py:38-66."""

    kind = "rot_c"
    uses_feature = True

    def __init__(self, feature_dim):
        super().__init__()
        self.feature_dim = feature_dim
        self.net = ConditionalTransform(feature_dim, 16)

    def _feature_dim(self):
        return self.feature_dim


class _AblationUncond(_FusedLayer):
    """Unconditional ablation layer: a free n x n matrix ``mat`` (init I + 1e-3 randn), reference state-dict key ``mat``."""

    n = 3

    def __init__(self):
        super().__init__()
        self.mat = nn.Parameter(torch.eye(self.n) + torch.randn(self.n, self.n) * 1e-3)

    def matrix(self):
        return self.mat


class _AblationCond(_FusedLayer):
    """Conditional ablation layer: ``net`` = ConditionalTransform(feature_dim, n*n); M = net(feature).reshape(n,n) + I per image."""

    n = 3
    uses_feature = True

    def __init__(self, feature_dim):
        super().__init__()
        self.feature_dim = feature_dim
        self.net = ConditionalTransform(feature_dim, self.n * self.n)

    def _feature_dim(self):
        return self.feature_dim


class Uncondition9Trans(_AblationUncond):
    """flow/squeezetrans.py:250-262 (calculate_9: Gram-Schmidt of M R with its log-det)."""
    kind = "smith9_u"


class Condition9Trans(_AblationCond):
    """flow/squeezetrans.py:235-247."""
    kind = "smith9_c"


class Uncondition9TransLU(_FusedLayer):
    """flow/squeezetrans.py:279-291: calculate_9 with the PLU-parameterised 3x3."""
    kind = "smith9_u"

    def __init__(self):
        super().__init__()
        self.mat = UnconditionLU(3)

    def matrix(self):
        with torch.no_grad():
            return self.mat()


class Uncondition36Trans(_AblationUncond):
    """flow/squeezetrans.py:350-361 (calculate_36: 6x6 matrix on the 6-D representation)."""
    kind, n = "smith36_u", 6


class Condition36Trans(_AblationCond):
    """flow/squeezetrans.py:334-347."""
    kind, n = "smith36_c", 6


class Uncondition9RotL(_AblationUncond):
    """flow/rottrans.py:94-105 (calculate_9_l: polar factor of M R; the inverse direction uses M^T, as the reference does)."""
    kind = "polar9l_u"


class Condition9RotL(_AblationCond):
    """flow/rottrans.py:107-121."""
    kind = "polar9l_c"


class Uncondition9RotR(_AblationUncond):
    """flow/rottrans.py:124-135 (calculate_9_r: polar factor of R M)."""
    kind = "polar9r_u"


class Condition9RotR(_AblationCond):
    """flow/rottrans.py:138-151."""
    kind = "polar9r_c"


class Uncondition9RotRSmith(_AblationUncond):
    """flow/rottrans.py:154-165 (calculate_9_r_smith: R Q, Q = Gram-Schmidt of M)."""
    kind = "right9_u"


class Condition9RotRSmith(_AblationCond):
    """flow/rottrans.py:168-181."""
    kind = "right9_c"


def get_mobius(config, feature_dim):
    """flow/mobiusflow.py:7-14."""
    if config.dist == "noflow":
        return None
    return MobiusFlow(3, config.segments, condition=config.condition, feature_dim=feature_dim)


def get_affine(config, feature_dim, first_layer_condition=False):
    """Dispatch table of flow/affineflow.py:5-73."""
    rot, lu = config.rot, bool(getattr(config, "lu", 0))

    def lu_conditional(n):
        if n == 4:
            return Condition16TransLU(feature_dim)
        raise NotImplementedError(
            "Condition9TransLU (flow/squeezetrans.py:265-277): calculate_9 with the batch-coupled ConditionLU(3) has no per-image "
            "parameter block for the fused kernels and no differentiable operator here")

    if first_layer_condition:
        if rot == "16UnTrans":
            return lu_conditional(4) if lu else Condition16Trans(feature_dim)
        if rot == "16UnRot":
            return ConditionRot(feature_dim)
    if config.condition:
        if rot == "16Trans":
            return lu_conditional(4) if lu else Condition16Trans(feature_dim)
        if rot == "16UnTrans":
            return Uncondition16TransLU() if lu else Uncondition16Trans()
        if rot == "36Trans":
            return Condition36Trans(feature_dim)
        if rot == "9TransLSVD":
            return Condition9RotL(feature_dim)
        if rot == "9TransRSVD":
            return Condition9RotR(feature_dim)
        if rot == "9TransLSmith":
            return lu_conditional(3) if lu else Condition9Trans(feature_dim)
        if rot == "9TransRSmith":
            return Condition9RotRSmith(feature_dim)
        if rot == "16Rot":
            return ConditionRot(feature_dim)
        if rot == "16UnRot":
            return UnconditionRot()
        return None
    if rot == "16Trans":
        return Uncondition16TransLU() if lu else Uncondition16Trans()
    if rot == "36Trans":
        return Uncondition36Trans()
    if rot == "9TransLSVD":
        return Uncondition9RotL()
    if rot == "9TransRSVD":
        return Uncondition9RotR()
    if rot == "9TransLSmith":
        return Uncondition9TransLU() if lu else Uncondition9Trans()
    if rot == "9TransRSmith":
        return Uncondition9RotRSmith()
    if rot == "16Rot":
        return UnconditionRot()
    return None


# ------------------------------------------------------------------------------------------------------
# execution plumbing
# ------------------------------------------------------------------------------------------------------
def _perm_row(permute, layer) -> int:
    if permute is None:
        return 0
    p = [int(v) for v in (permute.tolist() if torch.is_tensor(permute) else permute)]
    if len(p) != 3 or sorted(p) != [0, 1, 2] or (p[1] - p[0]) % 3 != 1 or (p[2] - p[1]) % 3 != 1:
        raise NotImplementedError(f"permute={p}: only the cyclic rows of flow/flow.py:13-15 exist in the reference")
    return p[0]


def _signature(layers) -> tuple:
    sig = [engine.svd_backend()]
    for l in layers:
        for t in engine.layer_tensors(l):
            sig.append((t.data_ptr(), t._version))
    return tuple(sig)


def _program(owner, layers, perms, F, device) -> engine.Program:
    """The packed program of (layers, perms) on ``device``, cached on the owning module.

    The cache is keyed on (data_ptr, _version) of every weight tensor: optimizer steps, ``load_state_dict`` and any other in-place
    write through the tensor itself are picked up.  Writes through ``.data`` (``p.data.copy_()``, some EMA / clipping code) do not
    bump ``_version``: call ``Flow.invalidate_cache()`` after those."""
    cache = owner.__dict__.setdefault("_rnf_programs", {})
    key = (device.index if device.index is not None else torch.cuda.current_device(), tuple(perms))
    sig = _signature(layers)
    hit = cache.get(key)
    if hit is not None and hit[0] == sig:
        return hit[1]
    specs = [engine.LayerSpec(l.kind, p, l) for l, p in zip(layers, perms)]
    prog = engine.Program(specs, F, torch.device("cuda", key[0]))
    cache[key] = (sig, prog)
    return prog


def _train_program(owner, layers, perms, F, device) -> engine.TrainProgram:
    """The training path's program, cached on the owning module and keyed on structure only (device, layer modules and kinds, perms,
    F): it is packed once, and every call brings the current weights as a device image, so optimiser steps cost no re-pack."""
    cache = owner.__dict__.setdefault("_rnf_train_programs", {})
    dev = device.index if device.index is not None else torch.cuda.current_device()
    key = (dev, tuple(perms), tuple((id(l), l.kind) for l in layers), int(F))
    tp = cache.get(key)
    if tp is None:
        tp = cache[key] = engine.TrainProgram(layers, perms, F, torch.device("cuda", dev))
    return tp


def _wants_grad(layers, rotation, feature) -> bool:
    if not torch.is_grad_enabled():
        return False
    if rotation.requires_grad or (torch.is_tensor(feature) and feature.requires_grad):
        return True
    return any(t.requires_grad for l in layers for t in engine.layer_tensors(l))


_GRAD_MESSAGE = (
    "Flow.grid_log_prob is the fused grid evaluation (arg-max / normaliser reduced on the fly) and keeps nothing for a backward pass; "
    "this call runs with autograd enabled and {what} requires grad.  Wrap it in torch.no_grad() (as eval.py:539 / agent.py:102 do), or "
    "call Flow.forward / Flow.inverse, which run the differentiable per-layer operators (rotationnormflow_b200/train.py) in that case.")


def _check_rotation(rotation):
    if not torch.is_tensor(rotation) or rotation.dim() != 3 or tuple(rotation.shape[1:]) != (3, 3):
        raise ValueError(f"rotation must be a [N,3,3] tensor, got {tuple(getattr(rotation, 'shape', ()))}")
    if not rotation.is_cuda:
        raise RuntimeError("rotationnormflow_b200 runs on a B200 only: `rotation` must be a CUDA tensor (there is no CPU fallback)")
    return rotation.to(torch.float32).contiguous()


def _refuse_ablation(layers, what: str) -> None:
    ablation = [l.kind for l in layers if l.kind.split("_")[0] in engine.ABLATION_KINDS]
    if ablation:
        raise NotImplementedError(f"{what} the ablation layers {sorted(set(ablation))}")


def _per_image(conditional, feature, fisher_A, dev, N=None, feature_index=None):
    """The per-image arguments of a call on N rotations (Flow.log_prob_grad, Flow.log_prob) or on a grid (Flow.grid_log_prob, N None):
    (feature [B,F] float32 on ``dev`` or None, B, idx int32 [N] or None, rows per image, A9, c).  B is the number of feature rows, else
    (not on a grid) of fisher_A's matrices, else 1.  Rows reach their image through ``feature_index``, else image-major, N % B == 0."""
    from .fisher import fisher_constants
    B = 1
    if conditional:
        if feature is None:
            raise AssertionError("The input feature is needed in this module")
        feature = feature.to(dev, torch.float32)
        if N is not None and feature.dim() != 2:
            raise ValueError(f"feature must be [B,F] with one row per image, got {tuple(feature.shape)}")
        B = feature.shape[0]
    else:
        feature = None
        if N is not None and fisher_A is not None:
            B = fisher_A.shape[0]
    idx, rpi = None, 1
    if feature_index is not None:
        idx = feature_index.to(dev, torch.int32).contiguous()
        if idx.shape != (N,):
            raise ValueError("feature_index must have one entry per rotation")
    elif N is not None and (conditional or fisher_A is not None):
        if B <= 0 or N % B != 0:
            raise ValueError(f"{N} rotations do not split image-major over B={B} images: pass feature_index")
        rpi = N // B
    A9 = c = None
    if fisher_A is not None:
        A9, c = fisher_constants(fisher_A.to(dev))
        if A9.shape[0] != B:
            raise ValueError("fisher_A must have one 3x3 matrix per image")
    return feature, B, idx, rpi, A9, c


def fused_kernels_run(layers) -> bool:
    """True when the fused kernels evaluate this layer stack: they are specialised for Mobius layers of K_SEGMENTS components and have
    no ConditionLU (batch-coupled in the reference), which run in the per-layer operators of train.py instead."""
    return not any((l.kind == "mobius" and l.K != engine.K_SEGMENTS) or l.kind == "aff_clu" for l in layers)


def _needs_composed(layers, rotation, feature) -> bool:
    """True when the call must run layer by layer in the differentiable operators of train.py: autograd is on and something
    requires grad (the reference builds a graph there: training at agent.py:87, eval.py:468-477), or a Mobius layer has a number of
    mixture components other than the 64 the fused kernels are specialised for."""
    if not fused_kernels_run(layers):
        return True
    return _wants_grad(layers, rotation, feature)


def _run_composed(layers, perms, rotation, feature, inverse, feature_index):
    from . import train
    R = _check_rotation(rotation)
    conditional = any(getattr(l, "uses_feature", False) or (l.kind == "mobius" and l.condition) for l in layers)
    rows = None
    if conditional:
        if feature is None:
            raise AssertionError("The input feature is needed in this module")
        rows = feature.to(R.device, torch.float32)
        if feature_index is not None:
            rows = rows[feature_index.to(R.device).long()]
        if rows.shape[0] != R.shape[0]:
            raise ValueError(f"feature has {rows.shape[0]} rows for {R.shape[0]} rotations (the reference asserts equality, agent.py:211,259)")
    return train.composed_run(layers, perms, R, rows, inverse)


def _run(layers, perms, F, owner, rotation, feature, inverse, feature_index=None, mode=None):
    if _needs_composed(layers, rotation, feature):
        return _run_composed(layers, perms, rotation, feature, inverse, feature_index)
    R = _check_rotation(rotation)
    prog = _program(owner, layers, perms, F, R.device)
    mode = mode or engine.default_mlp_mode()
    N = R.shape[0]
    conditional = prog.cond_floats != 0
    if conditional and feature is None:
        raise AssertionError("The input feature is needed in this module")
    if conditional and feature_index is None and feature.shape[0] != N:
        raise ValueError(f"feature has {feature.shape[0]} rows for {N} rotations (the reference asserts equality, agent.py:211,259)")
    if not conditional:
        return prog.run(R, None, 0, None, 1, inverse, mode)
    feature = feature.to(R.device)
    if feature_index is not None:
        idx = feature_index.to(R.device, torch.int32).contiguous()
        if idx.shape[0] != N:
            raise ValueError("feature_index must have one entry per rotation")
        return prog.run(R, prog.condition(feature), feature.shape[0], idx, 0, inverse, mode)
    if N == 0:
        return prog.run(R, None, 0, None, 1, inverse, mode)
    # ---- the reference's convention: one feature row per rotation (built by .repeat, agent.py:240-244 / eval.py:450) ----
    if feature.stride(0) == 0 or N == 1:                         # an expanded view: one image, nothing to read
        return prog.run(R, prog.condition(feature[:1]), 1, None, N, inverse, mode)
    feat = feature.to(torch.float32).contiguous()
    capturing = torch.cuda.is_current_stream_capturing()
    cap = min(N, engine.DEDUP_CAP)
    idx, first, count = engine.dedup_rows(feat, cap)             # device side, asynchronous
    if N > cap and not capturing:
        # more rows than the optimistic capacity: the run count decides (one 4-byte read; the reference itself synchronises
        # 15 times per Mobius layer in this direction of use).  Under stream capture the capacity is a documented
        # precondition, enforced by rnf_poison_if_overflow below.
        B = int(count.item())
        if B > cap:
            max_rows = max(1, (1 << 28) // max(1, prog.cond_floats))    # bound the per-image constant buffer
            if B > max_rows:
                outs = [_run(layers, perms, F, owner, R[s:s + max_rows], feat[s:s + max_rows], inverse, None, mode) for s in range(0, N, max_rows)]
                return torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs])
            cap = B
            idx, first, count = engine.dedup_rows(feat, cap)
    out = prog.run(R, prog.condition_runs(feat, first, count, cap), cap, idx, 0, inverse, mode)
    if N > cap and capturing:
        prog.poison_if_overflow(count, cap, out[1])
    return out


class Flow(_NoProgramState, nn.Module):
    """flow/flow.py:18-92."""

    def __init__(self, config):
        super().__init__()
        self.config = config
        self.condition = config.condition
        self._permute = torch.tensor(_PERMUTE_ROWS, dtype=torch.long)
        if self.condition:
            self.feature_dim = 32 if config.feature_dim is None else config.feature_dim
            if config.embedding:
                self.feature_dim += config.embedding_dim
        else:
            self.feature_dim = 0
        n = config.layers
        stack = []
        if getattr(config, "last_affine", 0):
            stack.append(get_affine(config, self.feature_dim, first_layer_condition=True))
        for i in range(n):
            m = get_mobius(config, self.feature_dim)
            if m is not None:
                stack.append(m)
            a = get_affine(config, self.feature_dim)
            if a is not None and (i != n - 1 or getattr(config, "first_affine", 1)):
                stack.append(a)
        print("total layers of flow: ", len(stack))
        self.layers = nn.ModuleList(stack)

    # permutation row handed to layer i in either direction (flow/flow.py:58-70 and :78-88 agree layer by layer)
    def _perm_rows(self):
        rows, c = [], 0
        freq = bool(getattr(self.config, "frequent_permute", 0))
        for l in self.layers:
            rows.append(_PERMUTE_ROWS[c % 6][0])
            if isinstance(l, MobiusFlow) or freq:
                c += 1
        return rows

    def forward(self, rotation, feature=None, inverse=False, draw=False, feature_index=None, mlp_mode=None):
        if not self.condition:
            feature = None
        return _run(list(self.layers), self._perm_rows(), self.feature_dim, self, rotation, feature, bool(inverse),
                    feature_index, mlp_mode)

    def inverse(self, rotation, feature=None, draw=False, feature_index=None, mlp_mode=None):
        return self.forward(rotation, feature, True, draw, feature_index, mlp_mode)

    # ---- the score d log p / dR of the forward direction (eval.py:464-480 nll_grad) as one call ---------------
    def log_prob_grad(self, rotation, feature=None, feature_index=None, fisher_A=None):
        """(logp [N], grad [N,3,3]): log p(R | image) = ldj [+ matrix-Fisher base term] and its tangential gradient R [g]x / 2 with
        respect to R (what ``rotation.grad`` holds after ``logp.sum().backward()``, projected on the tangent space of SO(3)).

        feature [B,F] one row per image (None for an unconditional flow); row -> image from ``feature_index`` [N], else image-major
        with N % B == 0.  fisher_A [B,3,3] adds log p of MatrixFisherN(A_b) at the flow's output (utils/fisher.py:217-232).
        One launch of csrc/flow_grad.cu; the outputs are plain tensors, not autograd graphs.  Flows with segments != 64 or
        ConditionLU layers run autograd through the per-layer operators of train.py instead (same numbers)."""
        layers = list(self.layers)
        _refuse_ablation(layers, "Flow.log_prob_grad: no rotation gradient for")
        R = _check_rotation(rotation).detach()
        N = R.shape[0]
        dev = R.device
        feature, B, idx, rpi, A9, c = _per_image(bool(self.condition), None if feature is None else feature.detach(),
                                                 None if fisher_A is None else fisher_A.detach(), dev, N, feature_index)
        if N == 0:
            return R.new_empty((0,)), R.new_empty((0, 3, 3))
        if not fused_kernels_run(layers):
            return self._log_prob_grad_composed(R, feature, idx, rpi, A9, c)
        prog = _program(self, layers, self._perm_rows(), self.feature_dim, dev)
        cond = prog.condition(feature) if prog.cond_floats else None
        return prog.logprob_grad(R, cond, B, idx, 0 if idx is not None else rpi, A9, c)

    # ---- training: differentiable log p in the fused kernels (agent.py:49-87) ------------------------------------------------
    def log_prob(self, rotation, feature=None, feature_index=None, fisher_A=None):
        """log p(R | image) [N] = ldj [+ sum(A_b * R') - c_b with a matrix-Fisher base A_b], differentiable by autograd with respect to
        every flow parameter, ``feature``, ``fisher_A`` and ``rotation`` (tangential gradient, as the per-layer operators give).

        feature [B,F] one row per image (None for an unconditional flow); row -> image from ``feature_index`` [N], else image-major
        with N % B == 0.  Forward and backward each run as one kernel launch over the whole stack (csrc/flow_grad.cu) plus batched
        GEMMs for the weight gradients; the weights reach the kernels as a device-side image built by torch ops, so an optimiser step
        costs no re-pack and nothing synchronises with the host.  Flows with segments != 64 or ConditionLU run train.composed_run
        instead (same numbers); ablation layers raise NotImplementedError.

        The loss of agent.py:54-73 (``rotation, ldjs = flow(gt, feature)``, then the Fisher log-prob of ``rotation``) becomes::

            logp = flow.log_prob(gt, feature, feature_index=idx, fisher_A=A)     # A [B,3,3] or None (uniform base)
            loss = -logp.mean()
        """
        from . import train
        layers = list(self.layers)
        _refuse_ablation(layers, "Flow.log_prob: no differentiable path for")
        R = _check_rotation(rotation)
        N, dev = R.shape[0], R.device
        conditional = bool(self.condition)
        feature, B, idx, rpi, A9, c = _per_image(conditional, feature, fisher_A, dev, N, feature_index)
        if idx is None and (conditional or fisher_A is not None):
            idx = torch.arange(N, device=dev, dtype=torch.int32) // rpi
        perms = self._perm_rows()
        if not fused_kernels_run(layers):
            rows = feature[idx.long()] if feature is not None else None
            R_out, logp = train.composed_run(layers, perms, R, rows, False)
        else:
            tp = _train_program(self, layers, perms, self.feature_dim, dev)
            R_out, logp = train.fused_run(tp, layers, R, feature, idx if conditional else None, B)
        if fisher_A is not None:
            img = idx.long()
            logp = logp + (A9[img].reshape(N, 3, 3) * R_out).sum(dim=(1, 2)) - c[img]
        return logp

    def _log_prob_grad_composed(self, R, feature, idx, rpi, A9, c):
        """log_prob_grad by autograd through the differentiable per-layer operators (train.composed_run)."""
        from . import train
        N = R.shape[0]
        img = idx.long() if idx is not None else torch.arange(N, device=R.device) // rpi
        rows = feature[img] if feature is not None else None
        with torch.enable_grad():
            Rg = R.clone().requires_grad_(True)
            Rout, logp = train.composed_run(list(self.layers), self._perm_rows(), Rg, rows, False)
            if A9 is not None:
                logp = logp + (A9[img].reshape(N, 3, 3) * Rout).sum(dim=(1, 2)) - c[img]
            (G,) = torch.autograd.grad(logp.sum(), Rg)
        H = R.transpose(1, 2) @ G                      # tangential part R (H - H^T) / 2, the convention of the fused kernel
        return logp.detach(), R @ (H - H.transpose(1, 2)) / 2

    # ---- N1 (SURVEY.md 8f): the loops of eval.py:444-462 / agent.py:246-266 as one call -------------------
    def grid_log_prob(self, grid, feature=None, offset=None, fisher_A=None, return_logp=False, g_index0=0, mlp_mode=None,
                      gt_rotations=None):
        """log p(grid[g] @ offset | image b) for all b, g, reduced per image on the fly.

        grid [G,3,3] (this rank's slice; ``g_index0`` = global index of grid[0]); feature [B,F] one row per image
        (None for an unconditional flow -> B = 1); fisher_A [B,3,3] adds the matrix-Fisher base term
        (utils/fisher.py:217-232, image-major as at agent.py:246-251).
        gt_rotations [B,K,3,3] (K >= 1 equivalent ground truths per image) adds the spread metric
        sum_g p_g d(grid[g] @ offset, R_gt) / sum_g p_g, d = angle to the closest ground truth (utils/utils.py:231-235),
        fused into the same pass: ``spread`` [B] in radians over THIS slice and ``spread_num`` [B] for merging slices.
        Returns dict(max [B], argmax [B] int64 global grid index (first on ties), sumexp [B] = sum_g exp(logp - max),
        logp [B,G] if requested)."""
        G_ = _check_rotation(grid)
        if torch.is_grad_enabled() and torch.is_tensor(feature) and feature.requires_grad:
            raise NotImplementedError(_GRAD_MESSAGE.format(what="the feature"))
        if not fused_kernels_run(self.layers):
            raise NotImplementedError(f"Flow.grid_log_prob runs in the fused kernels, which are specialised for segments={engine.K_SEGMENTS} and "
                                      "per-image conditional affines; use Flow.forward on the grid rotations for other segment counts / ConditionLU")
        prog = _program(self, list(self.layers), self._perm_rows(), self.feature_dim, G_.device)
        feature, B, _, _, A9, c = _per_image(prog.cond_floats != 0, feature, fisher_A, G_.device)
        cond = prog.condition(feature) if feature is not None else None
        off = None if offset is None else offset.to(G_.device, torch.float32).contiguous()
        mode = mlp_mode or engine.default_mlp_mode()
        if gt_rotations is not None:
            if gt_rotations.shape[0] != B or tuple(gt_rotations.shape[-2:]) != (3, 3):
                raise ValueError("gt_rotations must be [B,K,3,3] with one set of ground truths per image")
            mx, am, se, logp, sn = prog.grid_logprob(G_, g_index0, off, cond, B, A9, c, return_logp, mode, gt=gt_rotations)
            out = dict(max=mx, argmax=am, sumexp=se, spread_num=sn, spread=sn / se)
        else:
            mx, am, se, logp = prog.grid_logprob(G_, g_index0, off, cond, B, A9, c, return_logp, mode)
            out = dict(max=mx, argmax=am, sumexp=se)
        if return_logp:
            out["logp"] = logp
        return out
