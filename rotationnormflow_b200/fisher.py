"""Matrix-Fisher base distribution: per-image constants for the fused log-prob epilogue.

Follows utils/fisher.py:67-97 (proper_svd_N, matrix_fisher_norm_N type 1) and :217-232 (_log_prob):
    log p(R) = sum_ij A_ij R_ij - (S0+S1+S2) - log c,   c = 1/sqrt(8 pi (S0+S1)(S1+S2)(S0+S2))
with S the *proper* singular values (S2 multiplied by det(U) det(V)).  The 3x3 SVD is the same library call the
reference makes, once per image; the per-rotation term sum(A*R) is evaluated inside the flow kernel.
"""
from __future__ import annotations

import math

import torch


def fisher_constants(A: torch.Tensor):
    """A [B,3,3] -> (A9 [B,9] float32 contiguous, c [B] = sum(S) + log c_norm) on A's device."""
    if A.dim() != 3 or tuple(A.shape[1:]) != (3, 3):
        raise ValueError(f"A must be [B,3,3], got {tuple(A.shape)}")
    A = A.to(torch.float32)
    U, S, V = torch.svd(A)
    S2 = S[:, 2] * torch.det(U) * torch.det(V)
    S0, S1 = S[:, 0], S[:, 1]
    log_norm = -0.5 * torch.log(8 * math.pi * (S0 + S1) * (S2 + S1) * (S0 + S2))
    c = (S0 + S1 + S2) + log_norm
    return A.reshape(-1, 9).contiguous(), c.contiguous()


class MatrixFisherN(torch.nn.Module):
    """Drop-in for the log-prob side of utils/fisher.py:209-232 (``MatrixFisherN(A)._log_prob(inputs)``), type-1 normaliser.

    ``inputs`` [B*Q,3,3] (or anything reshapable to (B,-1,3,3), image-major) on the device of ``A``; returns [B*Q].
    ``_sample`` draws on the device (csrc/fisher_sample.cu; utils/fisher.py:117-207,234-243 restated per output sample)."""

    def __init__(self, A, norm_type=1, approx_num=None):
        super().__init__()
        if norm_type != 1:
            raise NotImplementedError("only the type-1 (high concentration) normaliser is on the hot path (utils/fisher.py:87-91)")
        self.A = A
        self._A9, self._c = fisher_constants(A)

    def _log_prob(self, inputs, context=9):
        from . import _cabi
        if not inputs.is_cuda:
            raise RuntimeError("rotationnormflow_b200 runs on a B200 only: `inputs` must be a CUDA tensor (there is no CPU fallback)")
        if inputs.shape[-1] != 3 or inputs.shape[-2] != 3:
            raise NotImplementedError("quaternion inputs: convert with quaternion_to_matrix first (utils/fisher.py:219-220)")
        dev = inputs.device
        if self._A9.device != dev:
            self._A9, self._c = self._A9.to(dev), self._c.to(dev)
        R = inputs.reshape(-1, 3, 3).to(torch.float32).contiguous()
        out = torch.empty((R.shape[0],), device=dev, dtype=torch.float32)
        _cabi.launch("rnf_fisher_log_prob", dev, self._A9, self._c, self._A9.shape[0], R, R.shape[0], out)
        return out

    log_prob = _log_prob

    def _sample(self, num_samples, context=9, seed=None):
        """[B, num_samples, 3, 3] rotations R ~ exp(tr(A_b^T R)) on the device of ``A`` (utils/fisher.py:234-243).

        ``seed`` (default: drawn from torch's global generator, so ``torch.manual_seed`` makes it reproducible) selects the
        Philox stream of the kernel; the streams differ from the reference's torch.randn / torch.rand draws, the
        distribution is the same."""
        import ctypes as C
        from . import _cabi
        if context != 9:
            raise NotImplementedError("quaternion output: convert with matrix_to_quaternion (utils/fisher.py:244-245)")
        if not self.A.is_cuda:
            raise RuntimeError("rotationnormflow_b200 runs on a B200 only: `A` must be a CUDA tensor (there is no CPU fallback)")
        dev = self.A.device
        usv = proper_svd_packed(self.A).to(dev)
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        B = usv.shape[0]
        out = torch.empty((B, int(num_samples), 3, 3), device=dev, dtype=torch.float32)
        _cabi.launch("rnf_fisher_sample", dev, usv, B, int(num_samples), C.c_uint64(seed), out)
        return out

    sample = _sample


def proper_svd_packed(A: torch.Tensor) -> torch.Tensor:
    """A [B,3,3] -> [B,24] float32 (U row-major, proper S, V row-major, 3 pad): proper_svd of utils/fisher.py:48-64
    (third columns of U, V and S2 flipped so that det U = det V = +1), evaluated once per image in float64 on the host."""
    A64 = A.detach().to("cpu", torch.float64)
    U, S, Vh = torch.linalg.svd(A64)
    V = Vh.transpose(-1, -2)
    dU, dV = torch.linalg.det(U), torch.linalg.det(V)
    U = U.clone(); V = V.clone(); S = S.clone()
    U[:, :, 2] *= dU[:, None]
    V[:, :, 2] *= dV[:, None]
    S[:, 2] *= dU * dV
    out = torch.zeros((A64.shape[0], 24), dtype=torch.float64)
    out[:, 0:9] = U.reshape(-1, 9)
    out[:, 9:12] = S
    out[:, 12:21] = V.reshape(-1, 9)
    return out.to(torch.float32).contiguous()
