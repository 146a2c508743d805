"""ctypes binding of ``librnf_b200.so`` (C ABI declared in ``include/rnf_abi.h``).

There is no CPU fallback and no alternative backend: if the library cannot be loaded (or built with
nvcc for sm_100a) importing the compute path raises, and every call checks the C return code.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

from . import build as _build

ABI_VERSION = 15

RNF_LAYER_MOBIUS = 0
RNF_LAYER_AFFINE = 1
RNF_LAYER_SMITH9, RNF_LAYER_SMITH36, RNF_LAYER_POLAR9L, RNF_LAYER_POLAR9R, RNF_LAYER_RIGHT9 = 2, 3, 4, 5, 6
RNF_MLP_FP32 = 0
RNF_MLP_TC = 1
RNF_MLP_TC_ROW = 2


class LayerDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("perm", C.c_int32),
        ("cond_slot", C.c_int32),
        ("has_ldj", C.c_int32),
        ("w_off", C.c_int64),
        ("w_off_tc", C.c_int64),
    ]


class ModelDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("n_layers", C.c_int32),
        ("K", C.c_int32),
        ("H", C.c_int32),
        ("F", C.c_int32),
        ("n_mobius_slots", C.c_int32),
        ("n_affine_slots", C.c_int32),
        ("affine_is_rot", C.c_int32),
        ("wf_off", C.c_int64),
        ("caff_off", C.c_int64),
        ("n_floats", C.c_int64),
    ]


class RnfError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"librnf_b200 error {code}: {msg}")
        self.code = code


_P = C.c_void_p
_I64 = C.c_int64
_SIGNATURES = {
    # name: (restype, argtypes)            -- must list every symbol declared in include/rnf_abi.h
    "rnf_abi_version": (C.c_int, []),
    "rnf_last_error": (C.c_char_p, []),
    "rnf_device_check": (C.c_int, [C.POINTER(C.c_int)]),
    "rnf_flow_create": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(LayerDesc), _P, C.POINTER(_P)]),
    "rnf_flow_destroy": (None, [_P]),
    "rnf_flow_cond_floats": (_I64, [_P]),
    "rnf_flow_condition": (C.c_int, [_P, _P, _I64, _P, _P]),
    "rnf_dedup_workspace_bytes": (_I64, [_I64]),
    "rnf_dedup_rows": (C.c_int, [_P, _I64, _I64, _P, _P, _I64, _P, _P, _I64, _P]),
    "rnf_flow_condition_runs": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P]),
    "rnf_poison_if_overflow": (C.c_int, [_P, _I64, _P, _I64, _P]),
    "rnf_train_max_components": (C.c_int, []),
    "rnf_train_mobius_forward": (C.c_int, [_P, _P, _I64, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "rnf_train_mobius_backward": (C.c_int, [_P, _P, _I64, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P]),
    "rnf_train_affine_forward": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "rnf_train_affine_backward": (C.c_int, [_P, _P, _I64, _P, _P, _P, _P, _P, _P]),
    "rnf_train_ablation_forward": (C.c_int, [_P, _P, _I64, C.c_int, _P, _P, _P]),
    "rnf_train_ablation_backward": (C.c_int, [_P, _P, _I64, C.c_int, _P, _P, _P, _P, _P, _P]),
    "rnf_flow_forward": (C.c_int, [_P, _P, _I64, _P, _I64, _P, _I64, _P, _P, C.c_int, _P]),
    "rnf_flow_inverse_scratch_floats": (_I64, [_P, _I64]),
    "rnf_flow_inverse": (C.c_int, [_P, _P, _I64, _P, _I64, _P, _I64, _P, _P, _P, C.c_int, _P]),
    "rnf_flow_logprob_grad": (C.c_int, [_P, _P, _I64, _P, _I64, _P, _I64, _P, _P, _P, _P, _P]),
    "rnf_flow_train_workspace_floats": (_I64, [_P, _I64]),
    "rnf_flow_train_forward": (C.c_int, [_P, _P, _P, _I64, _P, _I64, _P, _I64, _P, _P, _P]),
    "rnf_flow_train_backward": (C.c_int, [_P, _P, _P, _I64, _P, _I64, _P, _I64, _P, _P, _P, _P, _I64, _P]),
    "rnf_grid_partial_floats": (_I64, [_I64, _I64]),
    "rnf_grid_logprob": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _I64, _P, _P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "rnf_fisher_sample": (C.c_int, [_P, _I64, _I64, C.c_uint64, _P, _P]),
    "rnf_grid_logprob_spread": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _I64, _P, _P, _P, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "rnf_healpix_grid": (C.c_int, [C.c_int, _I64, _I64, _P, _P]),
    "rnf_fisher_log_prob": (C.c_int, [_P, _P, _I64, _P, _I64, _P, _P]),
    "rnf_min_geodesic": (C.c_int, [_P, _P, _I64, _I64, _P, _P]),
    "rnf_rotation_modes_workspace_bytes": (_I64, [_I64, _I64, C.c_int]),
    "rnf_rotation_modes": (C.c_int, [_P, _I64, _I64, _I64, _P, C.c_int, C.c_float, C.c_float, _P, _I64, _P, _P, _P, _P, _P, _P]),
    "rnf_rotation_modes_shard_workspace_bytes": (_I64, [_I64, _I64]),
    "rnf_rotation_modes_shard_setup": (C.c_int, [_P, _I64, _I64, _P, _I64, _P]),
    "rnf_rotation_modes_shard_round": (C.c_int, [_P, _I64, _I64, _I64, _P, C.c_int, C.c_int, C.c_float, C.c_float, _P, _I64, _P, _P]),
    "rnf_rotation_modes_shard_merge": (C.c_int, [_P, C.c_int, _I64, C.c_int, C.c_int, _P, _I64, _P, _P, _P, _P, _P, _P, _P]),
    "rnf_healpix_children": (C.c_int, [C.c_int, _P, _I64, _P, _P, _P, _P]),
    "rnf_topk_workspace_bytes": (_I64, [_I64, _I64, C.c_int]),
    "rnf_topk": (C.c_int, [_P, _P, _I64, _I64, C.c_int, _P, _I64, _P, _P, _P]),
}

_lib = None
_lock = threading.Lock()


def library_path() -> str:
    return _build.LIB


def load(build_if_needed: bool = True):
    """Load (building first when the sources changed) and type the library.  Raises on any failure."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if build_if_needed and not _build.up_to_date():
            _build.build_library()
        if not os.path.exists(_build.LIB):
            raise ImportError(
                f"{_build.LIB} is missing: the CUDA extension has not been built (python -m rotationnormflow_b200.build). "
                "rotationnormflow_b200 has no CPU or PyTorch fallback."
            )
        lib = C.CDLL(_build.LIB)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        got = lib.rnf_abi_version()
        if got != ABI_VERSION:
            raise ImportError(f"librnf_b200.so reports ABI {got}, python binding expects {ABI_VERSION}: rebuild")
        _lib = lib
    return _lib


def check(code: int) -> None:
    if code != 0:
        msg = load().rnf_last_error()
        raise RnfError(code, msg.decode() if msg else "?")


def launch(name: str, device, *args) -> None:
    """Calls the streamed entry point ``name`` on ``device``: tensors become their data pointers (None a null pointer), other
    arguments pass through, the device's current stream goes last, and the return code is checked."""
    fn = getattr(load(), name)
    with torch.cuda.device(device):
        ptrs = [C.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a for a in args]
        check(fn(*ptrs, C.c_void_p(torch.cuda.current_stream(device).cuda_stream)))


def exported_symbols() -> list[str]:
    return list(_SIGNATURES)
