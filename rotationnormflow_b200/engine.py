"""Host side of the fused flow kernels: weight packing, handle management and launches.

PyTorch is used here only as plumbing (device memory, the current CUDA stream, ``torch.svd`` / LU algebra on
4x4 parameter matrices exactly where the reference calls them).  All per-rotation arithmetic runs inside
``librnf_b200.so``; there is no CPU or eager-PyTorch path -- CPU tensors raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _cabi

K_SEGMENTS = 64   # kernels are specialised for the value every settings/*.yml uses
HIDDEN = 64       # flow/condition.py:9 (Nh)

# float sizes of the packed blocks; must mirror csrc/rnf_common.cuh
MOB_FLOATS = 64 * 4 + 3 * (64 * 64 + 64) + 64 * 256 + 256
AFF_FLOATS = 80          # RNF_AFFINE_BLOCK_FLOATS: forward block [0,40), inverse-direction block [40,80)
AFF_INV = 40
CAFF_FLOATS = 64 + 3 * (64 * 64 + 64) + 16 * 64 + 16

TC_AVAILABLE = True    # csrc/flow_t4.cu (forward, grid) + csrc/flow_row.cu (inverse): tcgen05 conditioner
TC_WEIGHT_SCALE = 1.0    # fp16 hi/lo weight planes are stored unscaled (biases ride along as a K=16 block, see pack_mobius_tc)
MOB_TC_FLOATS = (3 * (2 * 8192 + 64 * 32) + (2 * 32768 + 256 * 32) + 1024 + 64 * 32) // 4   # kTcImageBytes / 4 in csrc/tc_common.cuh

LOG2E = 1.4426950408889634
CENTRE_SCALE = 0.7       # folded into the centre rows of fc_last in the tensor-core image (pack_mobius_tc)

_MODES = {"fp32": _cabi.RNF_MLP_FP32, "tc": _cabi.RNF_MLP_TC, "tc_row": _cabi.RNF_MLP_TC_ROW}


def default_mlp_mode() -> str:
    """"tc" (tcgen05 conditioner, the product path) unless RNF_MLP_MODE=fp32 selects the exact-FP32 CUDA-core kernels."""
    return os.environ.get("RNF_MLP_MODE", "tc")


def _np(t: torch.Tensor) -> np.ndarray:
    return t.detach().to("cpu", torch.float32).contiguous().numpy()


def _last_layer_perm(K: int) -> np.ndarray:
    """Output permutation of fc_last: component c gets columns 4c..4c+3 = (logit_c, w_c.x, w_c.y, w_c.z).

    The reference splits the 4K outputs as [K logits | K x 3 centres] (flow/mobiusflow.py:58-61)."""
    perm = np.empty(4 * K, dtype=np.int64)
    for c in range(K):
        perm[4 * c] = c
        perm[4 * c + 1: 4 * c + 4] = K + 3 * c + np.arange(3)
    return perm


def _last_layer_perm_pairs(K: int) -> np.ndarray:
    """Output permutation of fc_last for the tensor-core kernels: components are laid out in pairs (a, b) = (2p, 2p+1),
    8 columns per pair: (logit_a, logit_b, w_a.x, w_b.x, w_a.y, w_b.y, w_a.z, w_b.z), so that a tcgen05.ld vector delivers
    the operands of the packed f32x2 arithmetic as aligned register pairs (csrc/mobius_pair.cuh)."""
    perm = np.empty(4 * K, dtype=np.int64)
    for c in range(K):
        base = 8 * (c // 2) + (c % 2)
        perm[base] = c
        for q in range(3):
            perm[base + 2 * (q + 1)] = K + 3 * c + q
    return perm


def pack_mobius(cond_sd: dict, F: int) -> tuple[np.ndarray, np.ndarray | None]:
    """ConditionalTransform(3+F, 4K) -> (FP32 kernel image [MOB_FLOATS] (mobius_images), W_f [64,F] or None)."""
    W0 = _np(cond_sd["fc_first.weight"])
    if W0.shape != (HIDDEN, 3 + F):
        raise ValueError(f"fc_first.weight has shape {W0.shape}, expected {(HIDDEN, 3 + F)}")
    W4_shape = tuple(cond_sd["fc_last.weight"].shape)
    if W4_shape != (4 * K_SEGMENTS, HIDDEN):
        raise ValueError(f"fc_last.weight has shape {W4_shape}; kernels are built for segments={K_SEGMENTS}")
    blk = mobius_images([{k: t.detach().to("cpu", torch.float32) for k, t in cond_sd.items()}])[0].numpy()
    return blk, (np.ascontiguousarray(W0[:, 3:]) if F > 0 else None)


def _umma_k_major_sw128(W: np.ndarray) -> np.ndarray:
    """[N,64] fp16 -> bytes of the UMMA canonical K-major SWIZZLE_128B tile (N multiple of 8): element (n,k) at
    (n/8)*1024 + (n%8)*128 + ((k/8) ^ (n%8))*16 + (k%8)*2   (cute::UMMA::Layout_K_SW128_Atom)."""
    N, K = W.shape
    assert K == 64 and N % 8 == 0 and W.dtype == np.float16
    n = np.arange(N)[:, None]
    k = np.arange(K)[None, :]
    off = (n // 8) * 1024 + (n % 8) * 128 + (((k // 8) ^ (n % 8)) * 16) + (k % 8) * 2      # byte offsets
    out = np.zeros(N * 64, dtype=np.float16)
    out[(off // 2).reshape(-1)] = W.reshape(-1)
    return out


def _split_fp16(W: np.ndarray):
    Ws = W.astype(np.float32) * np.float32(TC_WEIGHT_SCALE)
    hi = Ws.astype(np.float16)
    lo = (Ws - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def _hi_lo(x: np.ndarray):
    hi = x.astype(np.float16)
    return hi, (x - hi.astype(np.float32)).astype(np.float16)


def _bias_block(b: np.ndarray, W0: np.ndarray | None = None, b0: np.ndarray | None = None, b0_slot: int = 11) -> np.ndarray:
    """[N x 16] fp16 B-operand block in the no-swizzle K-major UMMA layout: element (n, k) at
    (n/8)*256 + (k/8)*128 + (n%8)*16 + (k%8)*2 bytes.  K slots per output unit n:
        0, 1   : (b_hi, b_lo)                                  -- bias of the layer
        2 .. 10: (W0hi[n,:3], W0hi[n,:3], W0lo[n,:3])           -- fc_first columns acting on the conditioning column y
        b0_slot, b0_slot + 1 : (b0_hi, b0_lo)                   -- fc_first bias (for the residual x0 + x3)
    The kernels multiply it by a per-rotation [128 x 16] A block.  csrc/flow_row.cu uses a constant block with
    ones in slots 0, 1 (bias only); csrc/flow_t4.cu uses (1, 1, y_hi, y_lo, y_hi, 1, 1, 0, 0, 0), which makes the tensor core
    evaluate fc_first (flow/condition.py:25) and re-create x0 inside the last hidden GEMM (flow/condition.py:29)."""
    N = b.shape[0]
    slots = np.zeros((N, 16), dtype=np.float16)
    slots[:, 0], slots[:, 1] = _hi_lo(b.astype(np.float32))
    if W0 is not None:
        whi, wlo = _hi_lo(W0.astype(np.float32))
        slots[:, 2:5], slots[:, 5:8], slots[:, 8:11] = whi, whi, wlo
    if b0 is not None:
        slots[:, b0_slot], slots[:, b0_slot + 1] = _hi_lo(b0.astype(np.float32))
    n = np.arange(N)[:, None]
    k = np.arange(16)[None, :]
    off = ((n // 8) * 256 + (k // 8) * 128 + (n % 8) * 16 + (k % 8) * 2) // 2
    out = np.zeros(N * 16, dtype=np.float16)
    out[off.reshape(-1)] = slots.reshape(-1)
    return out


def pack_mobius_tc(cond_sd: dict) -> np.ndarray:
    """Tensor-core image of one Mobius conditioner = the exact shared-memory pieces of the tcgen05 kernels:
    3 x [hi 64x64 | lo 64x64 fp16 SW128 | bias block 64x16] | [hi 256x64 | lo 256x64 SW128 | bias block 256x16]
    | aux: first[64][4] fp32 (flow_row: fc_first on the CUDA cores), fc_first block 64x16 (flow_t4: on the tensor core)
    returned as float32 words (MOB_TC_FLOATS of them).  The block of the last hidden layer also carries fc_first (residual)."""
    W0, b0 = _np(cond_sd["fc_first.weight"]), _np(cond_sd["fc_first.bias"])
    W0y = np.ascontiguousarray(W0[:, :3])
    parts = []
    for j in (1, 3, 5):
        hi, lo = _split_fp16(_np(cond_sd[f"layers.{j}.weight"]))          # nn.Linear weight is [out=N, in=K]: K-major
        b = _np(cond_sd[f"layers.{j}.bias"])
        blk = _bias_block(b, W0y, b0) if j == 5 else _bias_block(b)
        parts += [_umma_k_major_sw128(hi).view(np.float32), _umma_k_major_sw128(lo).view(np.float32), blk.view(np.float32)]
    # fc_last: pair layout; the logit rows carry the factor log2(e) so that the kernels feed them to ex2 directly (the
    # mixture weights then come out in units of ln 2, a common factor that cancels in every ratio the flow uses)
    W4, b4 = _np(cond_sd["fc_last.weight"]).copy(), _np(cond_sd["fc_last.bias"]).copy()
    W4[:K_SEGMENTS] *= np.float32(LOG2E)
    b4[:K_SEGMENTS] *= np.float32(LOG2E)
    # ... and the centre rows the factor 0.7 of flow/mobiusflow.py:72 (w <- 0.7 w / (1 + |w|)): the kernels work with
    # (a', b') = 0.7 (w.r, w.v) and u = 1 + |(a', b')| / 0.7, which saves the forward direction a reciprocal (mobius_pair.cuh)
    W4[K_SEGMENTS:] *= np.float32(CENTRE_SCALE)
    b4[K_SEGMENTS:] *= np.float32(CENTRE_SCALE)
    perm = _last_layer_perm_pairs(K_SEGMENTS)
    hi, lo = _split_fp16(W4[perm])
    parts += [_umma_k_major_sw128(hi).view(np.float32), _umma_k_major_sw128(lo).view(np.float32),
              _bias_block(b4[perm]).view(np.float32)]
    parts.append(np.concatenate([W0y, b0[:, None]], axis=1).astype(np.float32).reshape(-1))
    parts.append(_bias_block(b0, W0y).view(np.float32))
    blk = np.concatenate(parts).astype(np.float32, copy=False)
    assert blk.size == MOB_TC_FLOATS
    return blk


def pack_affine_matrix(W: torch.Tensor, is_rot: bool) -> np.ndarray:
    """One unconditional 4x4 layer -> [W16, log|det W|, pad3, Winv16, log|det Winv|, pad3].

    Forward uses W (flow/squeezetrans.py:167-169); inverse uses torch.linalg.inv(W) (:171-174) and, for rotation
    layers, the transpose (flow/rottrans.py:26).  Determinants are evaluated in float64 and rounded once."""
    W64 = W.detach().to("cpu", torch.float64).reshape(4, 4)
    blk = np.zeros(AFF_FLOATS, dtype=np.float32)
    blk[:16] = W64.to(torch.float32).reshape(-1).numpy()
    if is_rot:
        blk[AFF_INV:AFF_INV + 16] = W64.t().to(torch.float32).reshape(-1).numpy()
        return blk
    Winv = torch.linalg.inv(W64)
    blk[16] = float(torch.linalg.det(W64).abs().log())
    Winv32 = Winv.to(torch.float32)
    blk[AFF_INV:AFF_INV + 16] = Winv32.reshape(-1).numpy()
    blk[AFF_INV + 16] = float(torch.linalg.det(Winv32.double()).abs().log())
    return blk


ABLATION_KINDS = {"smith9": _cabi.RNF_LAYER_SMITH9, "smith36": _cabi.RNF_LAYER_SMITH36, "polar9l": _cabi.RNF_LAYER_POLAR9L,
                  "polar9r": _cabi.RNF_LAYER_POLAR9R, "right9": _cabi.RNF_LAYER_RIGHT9}


def gram_schmidt_columns(M: torch.Tensor) -> torch.Tensor:
    """Q of calculate_9_r_smith (flow/rottrans.py:82-88): Gram-Schmidt of the first two columns of M [...,3,3], third = cross."""
    c0 = M[..., 0] / M[..., 0].norm(dim=-1, keepdim=True)
    c1 = M[..., 1] - (c0 * M[..., 1]).sum(dim=-1, keepdim=True) * c0
    c1 = c1 / c1.norm(dim=-1, keepdim=True)
    return torch.stack([c0, c1, torch.linalg.cross(c0, c1, dim=-1)], dim=-1)


def ablation_blocks(kind: str, M: torch.Tensor) -> torch.Tensor:
    """Matrices M [B,n,n] of an ablation layer -> parameter blocks [B, AFF_FLOATS]: what the layer applies in the forward direction
    at [0, n*n) and in the inverse direction at [AFF_INV, AFF_INV + n*n) -- torch.linalg.inv(M) for the Smith layers
    (flow/squeezetrans.py:245,260,347,360), M^T for the SVD layers (flow/rottrans.py:103,119), Q / Q^T of the Gram-Schmidt
    for the right-multiplied rotation (flow/rottrans.py:81-91).  Per-layer / per-image parameter algebra, not a per-rotation path."""
    B, n = M.shape[0], M.shape[-1]
    if kind in ("smith9", "smith36"):
        fwd, inv = M, torch.linalg.inv(M)
    elif kind in ("polar9l", "polar9r"):
        fwd, inv = M, M.transpose(-1, -2)
    else:
        fwd = gram_schmidt_columns(M)
        inv = fwd.transpose(-1, -2)
    blk = torch.zeros((B, AFF_FLOATS), dtype=torch.float32, device=M.device)
    blk[:, :n * n] = fwd.reshape(B, -1).to(torch.float32)
    blk[:, AFF_INV:AFF_INV + n * n] = inv.reshape(B, -1).to(torch.float32)
    return blk


def conditioner_torch(ct, x: torch.Tensor) -> torch.Tensor:
    """ConditionalTransform.forward (flow/condition.py:24-30) on PER-IMAGE inputs x [B,Ni], as plain library GEMMs (the ablation
    layers' 3x3 / 6x6 matrix networks: B rows, never the per-rotation path)."""
    lin = torch.nn.functional.linear
    h0 = lin(x, ct.fc_first.weight, ct.fc_first.bias)
    h = h0
    for j in (1, 3, 5):
        h = lin(torch.relu(h), ct.layers[j].weight, ct.layers[j].bias)
    return lin(torch.relu(h0 + h), ct.fc_last.weight, ct.fc_last.bias)


def pack_cond_affine(net_sd: dict, F: int) -> tuple[np.ndarray, np.ndarray]:
    """ConditionalTransform(F, 16) -> (tail block [CAFF_FLOATS], W_f [64,F])."""
    W0, b0 = _np(net_sd["fc_first.weight"]), _np(net_sd["fc_first.bias"])
    if W0.shape != (HIDDEN, F):
        raise ValueError(f"net.fc_first.weight has shape {W0.shape}, expected {(HIDDEN, F)}")
    parts = [b0]
    for j in (1, 3, 5):
        parts += [_np(net_sd[f"layers.{j}.weight"]).reshape(-1), _np(net_sd[f"layers.{j}.bias"])]
    parts += [_np(net_sd["fc_last.weight"]).reshape(-1), _np(net_sd["fc_last.bias"])]
    blk = np.concatenate(parts).astype(np.float32)
    assert blk.size == CAFF_FLOATS
    return blk, W0


class LayerSpec:
    """What the packer needs to know about one layer (produced by the nn.Modules in flow.py)."""

    __slots__ = ("kind", "perm", "module")

    def __init__(self, kind: str, perm: int, module):
        self.kind = kind      # 'mobius' | 'aff_u' | 'aff_lu' | 'aff_c' | 'rot_u' | 'rot_c'
        self.perm = perm
        self.module = module


def conditioner_tensors(ct) -> dict:
    """ConditionalTransform -> {state-dict key: tensor}, read through ATTRIBUTES: nn.DataParallel replicas (agent.py:22) carry
    their weights as plain attributes, not as registered parameters, so state_dict() is empty there."""
    out = {"fc_first.weight": ct.fc_first.weight, "fc_first.bias": ct.fc_first.bias,
           "fc_last.weight": ct.fc_last.weight, "fc_last.bias": ct.fc_last.bias}
    for j in (1, 3, 5):
        out[f"layers.{j}.weight"], out[f"layers.{j}.bias"] = ct.layers[j].weight, ct.layers[j].bias
    return out


def layer_tensors(layer) -> list:
    """Every tensor a layer's packed image depends on (attribute access, see conditioner_tensors)."""
    if layer.kind == "mobius":
        return list(conditioner_tensors(layer.conditioner).values())
    if layer.kind in ("aff_c", "rot_c"):
        return list(conditioner_tensors(layer.net).values())
    if layer.kind == "aff_u":
        return [layer.mat]
    if layer.kind == "rot_u":
        return [layer.rot]
    if layer.kind == "aff_lu" or (layer.kind.endswith("_u") and isinstance(getattr(layer, "mat", None), torch.nn.Module)):
        m = layer.mat
        return [m.w_p, m.u_mask, m.l_mask, m.s_sign, m.l_eye, m.w_l, m.w_s, m.w_u]
    if layer.kind == "aff_clu":
        n = layer.net
        return [t for ct in (n.w_l_net, n.w_u_net, n.w_s_net) for t in conditioner_tensors(ct).values()]
    if layer.kind.split("_")[0] in ABLATION_KINDS:
        return list(conditioner_tensors(layer.net).values()) if layer.kind.endswith("_c") else [layer.mat]
    return [t for t in list(layer.parameters()) + list(layer.buffers())]


class Program:
    """A packed layer list bound to one CUDA device (weights + C handle)."""

    def __init__(self, specs: list[LayerSpec], F: int, device: torch.device):
        self.lib = _cabi.load()
        self.F = int(F)
        self.device = device
        self.n_layers = len(specs)
        blocks: list[np.ndarray] = []
        off = 0

        def push(a: np.ndarray) -> int:
            nonlocal off
            a = np.ascontiguousarray(a, dtype=np.float32).reshape(-1)
            pad = (-a.size) % 4
            if pad:
                a = np.concatenate([a, np.zeros(pad, np.float32)])
            blocks.append(a)
            o = off
            off += a.size
            return o

        descs = (_cabi.LayerDesc * max(1, len(specs)))()
        wf_mob, wf_aff, caff = [], [], []
        self.rot_slots: list = []          # modules of conditional rotation layers, slot order
        self.ablation_slots: list = []     # (kind, module) of conditional ablation layers, slot order
        n_mob = n_aff = 0
        cond_kinds = set()
        for i, s in enumerate(specs):
            d = descs[i]
            d.perm = int(s.perm) % 3
            d.cond_slot = -1
            d.has_ldj = 0
            d.w_off = 0
            d.w_off_tc = -1
            if s.kind == "mobius":
                d.kind = _cabi.RNF_LAYER_MOBIUS
                csd = conditioner_tensors(s.module.conditioner)
                blk, wf = pack_mobius(csd, self.F if s.module.condition else 0)
                d.w_off = push(blk)
                d.w_off_tc = push(pack_mobius_tc(csd))
                if wf is not None:
                    d.cond_slot = n_mob
                    n_mob += 1
                    wf_mob.append(wf)
            elif s.kind.split("_")[0] in ABLATION_KINDS:
                base_kind = s.kind.split("_")[0]
                d.kind = ABLATION_KINDS[base_kind]
                d.has_ldj = 1 if base_kind.startswith("smith") else 0
                if s.kind.endswith("_c"):
                    cond_kinds.add("ablation")
                    d.cond_slot = n_aff
                    n_aff += 1
                    self.ablation_slots.append((base_kind, s.module))
                else:
                    with torch.no_grad():
                        M = s.module.matrix().detach().to("cpu", torch.float64)
                        d.w_off = push(ablation_blocks(base_kind, M.reshape(1, M.shape[-1], M.shape[-1])).numpy())
            else:
                d.kind = _cabi.RNF_LAYER_AFFINE
                d.has_ldj = 0 if s.kind.startswith("rot") else 1
                if s.kind in ("aff_c", "rot_c"):
                    cond_kinds.add(s.kind)
                    blk, wf = pack_cond_affine(conditioner_tensors(s.module.net), self.F)
                    d.cond_slot = n_aff
                    n_aff += 1
                    wf_aff.append(wf)
                    caff.append(blk)
                    if s.kind == "rot_c":
                        self.rot_slots.append(s.module)
                else:
                    d.w_off = push(pack_affine_matrix(s.module.matrix(), is_rot=(s.kind == "rot_u")))
        if len(cond_kinds) > 1:
            raise NotImplementedError("mixing different families of conditional affine layers in one flow")
        model = _cabi.ModelDesc()
        model.abi_version = _cabi.ABI_VERSION
        model.n_layers = len(specs)
        model.K, model.H, model.F = K_SEGMENTS, HIDDEN, self.F
        model.n_mobius_slots, model.n_affine_slots = n_mob, n_aff
        model.affine_is_rot = 1 if "rot_c" in cond_kinds else (2 if "ablation" in cond_kinds else 0)
        model.wf_off = push(np.concatenate([w.reshape(-1) for w in wf_mob + wf_aff])) if (wf_mob or wf_aff) else 0
        model.caff_off = push(np.concatenate(caff)) if caff else 0
        if not blocks:
            blocks.append(np.zeros(4, np.float32))
            off = 4
        model.n_floats = off
        self.model = model
        self.descs = descs
        self.n_mob, self.n_aff = n_mob, n_aff
        with torch.cuda.device(device):
            self.weights = torch.from_numpy(np.concatenate(blocks)).to(device)
            handle = C.c_void_p()
            _cabi.check(self.lib.rnf_flow_create(C.byref(model), descs, C.c_void_p(self.weights.data_ptr()), C.byref(handle)))
        self.handle = handle
        self.cond_floats = int(self.lib.rnf_flow_cond_floats(handle))

    def __del__(self):
        h = getattr(self, "handle", None)
        if h is not None and h.value:
            try:
                self.lib.rnf_flow_destroy(h)
            except Exception:
                pass
            self.handle = None

    # ------------------------------------------------------------------------------------------
    def condition(self, feat: torch.Tensor) -> torch.Tensor:
        """feat [B,F] -> per-image constants [B, cond_floats] (rnf_flow_condition)."""
        B = feat.shape[0]
        feat = feat.to(self.device, torch.float32).contiguous()
        if feat.dim() != 2 or feat.shape[1] != self.F:
            raise ValueError(f"feature must be [B,{self.F}], got {tuple(feat.shape)}")
        cond = torch.empty((B, self.cond_floats), device=self.device, dtype=torch.float32)
        _cabi.launch("rnf_flow_condition", self.device, self.handle, feat, B, cond)
        if self.rot_slots:
            self._polar_factor(cond, B)
        if self.ablation_slots:
            self._fill_ablation_slots(cond, feat)
        return cond

    def _fill_ablation_slots(self, cond: torch.Tensor, feat_rows: torch.Tensor) -> None:
        """Conditional ablation layers (Condition9Trans, Condition36Trans, Condition9Rot*; flow/squeezetrans.py:235-247,334-347,
        flow/rottrans.py:107-181): M = MLP(feature).reshape(n,n) + I per IMAGE, written into the slots' parameter blocks."""
        base = self.n_mob * HIDDEN
        B = cond.shape[0]
        blk = cond[:, base: base + self.n_aff * AFF_FLOATS].view(B, self.n_aff, AFF_FLOATS)
        with torch.no_grad():
            for slot, (kind, module) in enumerate(self.ablation_slots):
                n = 6 if kind == "smith36" else 3
                M = conditioner_torch(module.net, feat_rows).reshape(B, n, n) + torch.eye(n, device=cond.device)
                blk[:, slot] = ablation_blocks(kind, M)

    def _polar_factor(self, cond: torch.Tensor, B: int) -> None:
        """ConditionRot (flow/rottrans.py:43-46,55-58): rot = U^T V with (U,S,V) = torch.svd(MLP(feature)+I), in place.

        U^T V is NOT invariant under the sign freedom of an SVD (U -> U D, V -> V D maps it to D U^T V D), so the layer is
        defined by the SVD routine the reference calls.  ``svd_backend()``: "device" (default) = torch.svd on the CUDA tensor, the
        very call the reference makes when it runs on a GPU (cuSOLVER; asynchronous, no host round trip); "cpu" = LAPACK through
        a host round trip, the convention of a reference run on the CPU (the golden vectors of tests/golden were minted there)."""
        base = self.n_mob * HIDDEN
        blk = cond[:, base: base + self.n_aff * AFF_FLOATS].view(B, self.n_aff, AFF_FLOATS)
        M = blk[:, :, :16].reshape(B, self.n_aff, 4, 4)
        if svd_backend() == "cpu":
            U, _, V = torch.svd(M.cpu())
            rot = (U.transpose(-1, -2) @ V).to(M.device)
        else:
            U, _, V = torch.svd(M)
            rot = U.transpose(-1, -2) @ V
        blk[:, :, :16] = rot.reshape(B, self.n_aff, 16)
        blk[:, :, AFF_INV:AFF_INV + 16] = rot.transpose(-1, -2).reshape(B, self.n_aff, 16)

    def condition_runs(self, feat: torch.Tensor, first: torch.Tensor, count: torch.Tensor, cap: int) -> torch.Tensor:
        """Per-image constants for the runs found by ``dedup_rows`` (rnf_flow_condition_runs): image b < count reads feature
        row first[b]; rows b >= count of the returned [cap, cond_floats] buffer are left untouched (never indexed)."""
        # capacity rows beyond the run count are never indexed; for ConditionRot they still go through the batched SVD: keep them 0
        alloc = torch.zeros if self.rot_slots else torch.empty
        cond = alloc((cap, self.cond_floats), device=self.device, dtype=torch.float32)
        _cabi.launch("rnf_flow_condition_runs", self.device, self.handle, feat, first, count, cap, cond)
        if self.rot_slots:
            self._polar_factor(cond, cap)
        if self.ablation_slots:
            self._fill_ablation_slots(cond, feat[first.long()])      # rows beyond the run count read row 0: never indexed
        return cond

    def poison_if_overflow(self, count: torch.Tensor, cap: int, ldj: torch.Tensor) -> None:
        _cabi.launch("rnf_poison_if_overflow", self.device, count, cap, ldj, ldj.numel())

    def run(self, R: torch.Tensor, cond, B: int, feat_index, rows_per_image: int, inverse: bool, mode: str):
        N = R.shape[0]
        R_out = torch.empty((N, 3, 3), device=self.device, dtype=torch.float32)
        ldj = torch.empty((N,), device=self.device, dtype=torch.float32)
        if N == 0:
            return R_out, ldj
        if inverse:
            ns = int(self.lib.rnf_flow_inverse_scratch_floats(self.handle, N))
            scratch = torch.empty((max(ns, 1),), device=self.device, dtype=torch.float32)
            _cabi.launch("rnf_flow_inverse", self.device, self.handle, R, N, cond, B, feat_index, rows_per_image, R_out, ldj, scratch,
                         _MODES[mode])
        else:
            _cabi.launch("rnf_flow_forward", self.device, self.handle, R, N, cond, B, feat_index, rows_per_image, R_out, ldj, _MODES[mode])
        return R_out, ldj

    def logprob_grad(self, R: torch.Tensor, cond, B: int, feat_index, rows_per_image: int, A9=None, c=None):
        """(logp [N], G [N,3,3]) of the forward direction in one launch (rnf_flow_logprob_grad): logp = ldj [+ sum(A_b R') - c_b],
        G = R [g]x / 2 the tangential gradient of logp with respect to R."""
        N = R.shape[0]
        logp = torch.empty((N,), device=self.device, dtype=torch.float32)
        G = torch.empty((N, 3, 3), device=self.device, dtype=torch.float32)
        if N == 0:
            return logp, G
        _cabi.launch("rnf_flow_logprob_grad", self.device, self.handle, R, N, cond, B, feat_index, rows_per_image, A9, c, logp, G)
        return logp, G

    def grid_logprob(self, grid: torch.Tensor, g_index0: int, offset, cond, B: int, fisher_A, fisher_c,
                     want_logp: bool, mode: str, gt: torch.Tensor | None = None):
        """-> (max [B], argmax [B], sumexp [B], logp [B,G] | None[, spread_num [B] when gt [B,K,3,3] is given])."""
        G = grid.shape[0]
        dev = self.device
        mx = torch.empty((B,), device=dev, dtype=torch.float32)
        am = torch.empty((B,), device=dev, dtype=torch.int64)
        se = torch.empty((B,), device=dev, dtype=torch.float32)
        logp = torch.empty((B, G), device=dev, dtype=torch.float32) if want_logp else None
        part = torch.empty((max(1, int(self.lib.rnf_grid_partial_floats(G, B))),), device=dev, dtype=torch.float32)
        sn = None
        if gt is not None:
            gt = gt.to(dev, torch.float32).reshape(B, -1, 9).contiguous()
            sn = torch.empty((B,), device=dev, dtype=torch.float32)
        _cabi.launch("rnf_grid_logprob_spread", dev, self.handle, grid, G, int(g_index0), offset, cond, B, fisher_A, fisher_c, gt,
                     0 if gt is None else int(gt.shape[1]), logp, part, mx, am, se, sn, _MODES[mode])
        return (mx, am, se, logp) if gt is None else (mx, am, se, logp, sn)


DEDUP_CAP = 8192      # optimistic image capacity of the sync-free drop-in path (44 MB of per-image constants at most)


def svd_backend() -> str:
    """"device" (default) or "cpu": where ConditionRot / UnconditionRot evaluate torch.svd (RNF_SVD_BACKEND); see Program._polar_factor."""
    v = os.environ.get("RNF_SVD_BACKEND", "device")
    if v not in ("device", "cpu"):
        raise ValueError(f"RNF_SVD_BACKEND={v!r}: expected 'device' or 'cpu'")
    return v


def dedup_rows(feature: torch.Tensor, cap: int):
    """Row-aligned ``feature [N,F]`` (float32, contiguous, CUDA; built by ``.repeat`` at agent.py:240-244 / eval.py:450) ->
    (idx int32 [N] row -> run number, first int32 [cap] first row of every run, count int32 [1] number of runs), all on the
    device and asynchronous (rnf_dedup_rows: one streaming pass over the N x F floats, a scan, a scatter)."""
    lib = _cabi.load()
    N, F = feature.shape
    dev = feature.device
    idx = torch.empty((N,), dtype=torch.int32, device=dev)
    first = torch.empty((cap,), dtype=torch.int32, device=dev)
    count = torch.empty((1,), dtype=torch.int32, device=dev)
    nbytes = int(lib.rnf_dedup_workspace_bytes(N))
    ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=dev)
    _cabi.launch("rnf_dedup_rows", dev, feature, N, F, idx, first, cap, count, ws, nbytes)
    return idx, first, count


# ------------------------------------------------------------------------------------------------------
# training path: the FP32 image and the per-image constants built by differentiable torch ops on the parameters' device
# (csrc/flow_grad.cu, flow_train_kernel).  The kernel returns gradients with respect to this image and these constants; autograd
# through the packing below carries them to the parameters, the features and the SVDs.
# ------------------------------------------------------------------------------------------------------
TRAIN_RECORD_FLOATS = 772                  # kTwsFloats in csrc/flow_grad.cu: training record of one (Mobius layer, row)
TRAIN_WORKSPACE_BYTES = 512 << 20          # bound of the backward's training records; larger batches run in chunks of rows
_PERM_CACHE: dict = {}


def _last_layer_perm_on(device) -> torch.Tensor:
    key = str(device)
    if key not in _PERM_CACHE:
        _PERM_CACHE[key] = torch.from_numpy(_last_layer_perm(K_SEGMENTS)).to(device)
    return _PERM_CACHE[key]


def mobius_images(conds: list) -> torch.Tensor:
    """Conditioner tensors (conditioner_tensors) of Lm Mobius layers -> [Lm, MOB_FLOATS]: the images of pack_mobius, stacked."""
    Lm = len(conds)
    st = lambda k: torch.stack([c[k] for c in conds]).to(torch.float32)
    W0 = st("fc_first.weight")
    perm = _last_layer_perm_on(W0.device)
    parts = [torch.cat([W0[:, :, :3], st("fc_first.bias")[:, :, None]], dim=2).reshape(Lm, 4 * HIDDEN)]
    for j in (1, 3, 5):
        parts += [st(f"layers.{j}.weight").transpose(1, 2).reshape(Lm, HIDDEN * HIDDEN), st(f"layers.{j}.bias")]
    parts += [st("fc_last.weight")[:, perm].transpose(1, 2).reshape(Lm, -1), st("fc_last.bias")[:, perm]]
    return torch.cat(parts, dim=1)


def logabsdet4(W: torch.Tensor) -> torch.Tensor:
    """log|det W| of [...,4,4] by the expansion in 2x2 minors, evaluated in float64 and rounded to float32 (as pack_affine_matrix).
    Differentiable, batched, and free of the LU factorisation's pivoting and info checks."""
    a = W.to(torch.float64)
    e = [[a[..., i, j] for j in range(4)] for i in range(4)]
    m = lambda r0, r1, c0, c1: e[r0][c0] * e[r1][c1] - e[r1][c0] * e[r0][c1]
    det = (m(0, 1, 0, 1) * m(2, 3, 2, 3) - m(0, 1, 0, 2) * m(2, 3, 1, 3) + m(0, 1, 0, 3) * m(2, 3, 1, 2)
           + m(0, 1, 1, 2) * m(2, 3, 0, 3) - m(0, 1, 1, 3) * m(2, 3, 0, 2) + m(0, 1, 2, 3) * m(2, 3, 0, 1))
    return det.abs().log().to(torch.float32)


def affine_blocks(layers: list) -> torch.Tensor:
    """Unconditional affine layers -> [La, 17]: the forward block (W, log|det W|) of pack_affine_matrix; U^T V and 0 for rot_u."""
    from . import train
    Ws, has = [], []
    for l in layers:
        W, h = train._affine_matrix(l, None, False)
        Ws.append(W.reshape(4, 4))
        has.append(h)
    W = torch.stack(Ws).to(torch.float32)
    ld = logabsdet4(W)
    if not all(has):
        ld = torch.stack([x if h else torch.zeros_like(x) for x, h in zip(ld.unbind(0), has)])
    return torch.cat([W.reshape(-1, 16), ld[:, None]], dim=1)


def _conditioners_stacked(cts: list, x: torch.Tensor) -> torch.Tensor:
    """conditioner_torch of S conditioners on the same per-image input x [B,Ni] -> [S,B,No], as batched GEMMs."""
    sd = [conditioner_tensors(ct) for ct in cts]
    st = lambda k: torch.stack([d[k] for d in sd])
    h0 = torch.baddbmm(st("fc_first.bias")[:, None, :], x.expand(len(cts), -1, -1), st("fc_first.weight").transpose(1, 2))
    h = h0
    for j in (1, 3, 5):
        h = torch.baddbmm(st(f"layers.{j}.bias")[:, None, :], torch.relu(h), st(f"layers.{j}.weight").transpose(1, 2))
    return torch.baddbmm(st("fc_last.bias")[:, None, :], torch.relu(h0 + h), st("fc_last.weight").transpose(1, 2))


def condition_torch(layers: list, feature: torch.Tensor) -> torch.Tensor:
    """feature [B,F] -> [B, cond_floats]: the per-image constants rnf_flow_condition writes (+ the polar factor of ConditionRot),
    differentiable.  Sections: W_f . feature per conditional Mobius slot; the forward block (W_b, log|det W_b|) per conditional affine
    slot (U^T V and 0 for rot_c); zeros where the forward kernels read nothing (inverse blocks, first-layer scratch)."""
    feat = feature.to(torch.float32)
    B = feat.shape[0]
    mob = [l for l in layers if l.kind == "mobius" and l.condition]
    aff = [l for l in layers if l.kind in ("aff_c", "rot_c")]
    parts = []
    if mob:
        Wf = torch.cat([conditioner_tensors(l.conditioner)["fc_first.weight"][:, 3:] for l in mob])     # [Lc*64, F]
        parts.append(feat @ Wf.t())
    if aff:
        S = len(aff)
        if len({l.kind for l in aff}) > 1:
            raise NotImplementedError("mixing different families of conditional affine layers in one flow")
        W = _conditioners_stacked([l.net for l in aff], feat).reshape(S, B, 4, 4) + torch.eye(4, device=feat.device)
        if aff[0].kind == "rot_c":
            U, _, V = torch.svd(W)                                  # flow/rottrans.py:43-46 (V, not V^T)
            W = U.transpose(-1, -2) @ V
            ld = W.new_zeros((S, B))
        else:
            ld = logabsdet4(W)
        blk = torch.cat([W.reshape(S, B, 16), ld[..., None], W.new_zeros((S, B, AFF_FLOATS - 17))], dim=2)
        parts += [blk.transpose(0, 1).reshape(B, S * AFF_FLOATS), feat.new_zeros((B, S * HIDDEN))]
    return torch.cat(parts, dim=1)


class TrainProgram:
    """The training path's Program: packed once for a layer structure (kinds, perms, F, device) and reused whatever the weights are --
    every call brings its own image (``image``) and per-image constants.  Holds what the gradient reductions need."""

    def __init__(self, layers: list, perms: list, F: int, device: torch.device):
        self.prog = Program([LayerSpec(l.kind, p, l) for l, p in zip(layers, perms)], F, device)
        self.device = device
        descs = self.prog.descs
        self.mob_layers, mob_off, self.mob_cond = [], [], []
        self.aff_u_layers, aff_u_off, self.aff_u, self.aff_c = [], [], [], []
        self.aff_c_has_ldj = False
        n_aff = 0
        for i, l in enumerate(layers):
            d = descs[i]
            if d.kind == _cabi.RNF_LAYER_MOBIUS:
                if d.cond_slot >= 0:
                    self.mob_cond.append(len(self.mob_layers))
                self.mob_layers.append(l)
                mob_off.append(d.w_off)
            elif d.kind == _cabi.RNF_LAYER_AFFINE:
                if d.cond_slot >= 0:
                    self.aff_c.append(n_aff)
                    self.aff_c_has_ldj = bool(d.has_ldj)
                else:
                    self.aff_u.append(n_aff)
                    self.aff_u_layers.append(l)
                    aff_u_off.append(d.w_off)
                n_aff += 1
            else:
                raise NotImplementedError(f"layer kind {l.kind!r} (ablation) has no differentiable path")
        self.aff_u_has_ldj = [not l.kind.startswith("rot") for l in self.aff_u_layers]
        self.n_mob, self.n_aff = len(self.mob_layers), n_aff
        self.cond_floats = self.prog.cond_floats
        self.n_mob_slots, self.n_aff_slots = self.prog.n_mob, self.prog.n_aff
        idx = [torch.arange(o, o + MOB_FLOATS) for o in mob_off] + [torch.arange(o, o + 17) for o in aff_u_off]
        self.image_index = torch.cat(idx).to(device) if idx else torch.zeros(0, dtype=torch.int64, device=device)
        self.aff_c_t = torch.tensor(self.aff_c, dtype=torch.int64, device=device)
        self.aff_u_t = torch.tensor(self.aff_u, dtype=torch.int64, device=device)
        self.mob_cond_t = torch.tensor(self.mob_cond, dtype=torch.int64, device=device)
        self.ldj_mask_u = torch.tensor(self.aff_u_has_ldj, dtype=torch.float32, device=device)

    def images(self):
        """(mob [Lm, MOB_FLOATS], aff [Lu, 17]): the FP32 image sections the kernels read, differentiable in the parameters."""
        mob = mobius_images([conditioner_tensors(l.conditioner) for l in self.mob_layers]) if self.mob_layers else None
        aff = affine_blocks(self.aff_u_layers) if self.aff_u_layers else None
        return mob, aff

    def weights(self, mob, aff) -> torch.Tensor:
        """A fresh weight buffer with the image sections at the Program's offsets (the tensor-core sections are left unwritten:
        the FP32 training kernels do not read them)."""
        buf = torch.empty((int(self.prog.model.n_floats),), device=self.device, dtype=torch.float32)
        src = [t.reshape(-1) for t in (mob, aff) if t is not None]
        if src:
            buf.index_copy_(0, self.image_index, torch.cat(src).detach())
        return buf

    def forward(self, weights, R, cond, B: int, idx32):
        N = R.shape[0]
        R_out = torch.empty((N, 3, 3), device=self.device, dtype=torch.float32)
        ldj = torch.empty((N,), device=self.device, dtype=torch.float32)
        if N:
            _cabi.launch("rnf_flow_train_forward", self.device, self.prog.handle, weights, R, N, cond, B, idx32, 0, R_out, ldj)
        return R_out, ldj

    def backward(self, weights, R, cond, B: int, idx32, G_Rout, g_ldj):
        """-> (G_R [N,3,3] tangential, g_mob [Lm, MOB_FLOATS] | None, g_aff [Lu,17] | None, g_cond [B, cond_floats] | None).

        The kernel writes per row the training records (rnf_abi.h); the weight gradients are FP32 GEMMs over rows batched across
        layers, the per-image sums are index_add over rows.  Rows run in chunks so that the records stay within
        TRAIN_WORKSPACE_BYTES; the sums accumulate across chunks."""
        N, dev = R.shape[0], self.device
        Lm, La, H = self.n_mob, self.n_aff, HIDDEN
        TF = TRAIN_RECORD_FLOATS
        G_R = torch.empty((N, 3, 3), device=dev, dtype=torch.float32)
        g_mob = torch.zeros((Lm, MOB_FLOATS), device=dev, dtype=torch.float32) if Lm else None
        g_aff = torch.zeros((len(self.aff_u), 17), device=dev, dtype=torch.float32) if self.aff_u else None
        g_cmob = torch.zeros((B, len(self.mob_cond) * H), device=dev, dtype=torch.float32) if cond is not None and self.mob_cond else None
        g_caff = torch.zeros((B, len(self.aff_c), 16), device=dev, dtype=torch.float32) if cond is not None and self.aff_c else None
        img = idx32.long() if idx32 is not None else None
        per_row = Lm * TF + La * 16
        chunk = max(1, min(N, TRAIN_WORKSPACE_BYTES // (4 * max(per_row, 1))))
        ws = torch.empty((max(1, chunk * per_row),), device=dev, dtype=torch.float32)
        for s in range(0, N, chunk):
            n = min(chunk, N - s)
            sl = lambda t: None if t is None else t[s:s + n]
            _cabi.launch("rnf_flow_train_backward", dev, self.prog.handle, weights, R[s:s + n], n, cond, B, sl(idx32), 0, sl(G_Rout), sl(g_ldj),
                         G_R[s:s + n], ws, int(ws.numel()))
            wm = ws[:Lm * n * TF].view(Lm, n, TF)
            wa = ws[Lm * n * TF: Lm * n * TF + La * n * 16].view(La, n, 16)
            if Lm:
                act = lambda i: wm[:, :, 4 + H * i: 4 + H * (i + 1)]
                grad = lambda i: wm[:, :, 4 + 4 * H + H * i: 4 + 4 * H + H * (i + 1)]
                gout = wm[:, :, 4 + 8 * H:]
                bsum = wm[:, :, 4 + 5 * H:].sum(dim=1)                      # biases of layers.1/3/5 and fc_last
                parts = [torch.bmm(grad(0).transpose(1, 2), wm[:, :, 0:4]).reshape(Lm, 4 * H)]
                for i in range(3):
                    parts += [torch.bmm(act(i).transpose(1, 2), grad(i + 1)).reshape(Lm, H * H), bsum[:, H * i: H * (i + 1)]]
                parts += [torch.bmm(act(3).transpose(1, 2), gout).reshape(Lm, -1), bsum[:, 3 * H:]]
                g_mob += torch.cat(parts, dim=1)
                if g_cmob is not None:
                    gh0 = grad(0) if len(self.mob_cond) == Lm else grad(0).index_select(0, self.mob_cond_t)
                    g_cmob.index_add_(0, img[s:s + n], gh0.transpose(0, 1).reshape(n, -1))
            if g_aff is not None:
                g_aff[:, :16] += wa.index_select(0, self.aff_u_t).sum(dim=1)
            if g_caff is not None:
                g_caff.index_add_(0, img[s:s + n], wa.index_select(0, self.aff_c_t).transpose(0, 1))
        # log-det slots: d ldj / d log|det W| = 1 on every row the block acts on
        gl = g_ldj if g_ldj is not None else torch.ones((N,), device=dev, dtype=torch.float32)
        if g_aff is not None:
            g_aff[:, 16] = gl.sum() * self.ldj_mask_u
        g_cond = None
        if cond is not None:
            parts = [] if g_cmob is None else [g_cmob]
            if g_caff is not None:
                Sc = len(self.aff_c)
                ld = torch.zeros((B,), device=dev, dtype=torch.float32)
                if self.aff_c_has_ldj:
                    ld.index_add_(0, img, gl)
                parts += [torch.cat([g_caff, ld[:, None, None].expand(B, Sc, 1), g_caff.new_zeros((B, Sc, AFF_FLOATS - 17))], dim=2).reshape(B, -1),
                          g_caff.new_zeros((B, Sc * H))]
            g_cond = torch.cat(parts, dim=1)
        return G_R, g_mob, g_aff, g_cond
