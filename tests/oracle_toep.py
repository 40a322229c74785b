"""Float64 restatement of the Toeplitz-embedded NUFFT normal operator (TEST INFRASTRUCTURE, like oracle/).

[RECALL] torchkbnufft calc_toeplitz_kernel / ToepNufft: the point-spread function
    p[r0, r1] = s * sum_m w_m exp(i (omega0_m r0 + omega1_m r1)),  |r0| < N0, |r1| < N1,
is taken from two adjoint transforms of the weights with n_shift = 0 -- q1 (omega) = p[a, b] and q2 (omega0 negated)
= p[-a, b] -- laid out circulantly on the 2 N0 x 2 N1 grid (p[-a, -b] = conj p[a, b] for real weights; row N0 and
column N1 zero) and transformed with an unnormalised FFT.  The apply is ifft2(kernel * fft2(zero_pad(x))) cropped
to N0 x N1."""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from oracle.nufft import NufftSpec, _as_omega, ndft_adjoint, nufft_adjoint


def circulant_psf(q1: torch.Tensor, q2: torch.Tensor) -> torch.Tensor:
    """q1, q2 [..., N0, N1] -> p_circ [..., 2 N0, 2 N1] (the quadrant table of calc_toeplitz_kernel)."""
    N0, N1 = q1.shape[-2:]
    out = torch.zeros(q1.shape[:-2] + (2 * N0, 2 * N1), dtype=torch.complex128)
    out[..., :N0, :N1] = q1
    out[..., N0 + 1:, :N1] = q2[..., 1:, :].flip(-2)                        # i0 > N0: q2[L0 - i0, i1]
    out[..., :N0, N1 + 1:] = q2[..., :, 1:].flip(-1).conj()                 # i1 > N1: conj q2[i0, L1 - i1]
    out[..., N0 + 1:, N1 + 1:] = q1[..., 1:, 1:].flip(-2).flip(-1).conj()   # both: conj q1[L0 - i0, L1 - i1]
    return out


def toeplitz_kernel(omega, spec: NufftSpec, weights=None, norm: Optional[str] = None, exact: bool = False) -> torch.Tensor:
    """complex128 [2 N0, 2 N1].  exact=False: the PSF from the Kaiser-Bessel adjoint (oracle.nufft_adjoint) at the
    spec's grid / table; exact=True: from the exact non-uniform DFT (ndft_adjoint)."""
    s = spec.resolved()
    spec0 = NufftSpec(s.im_size, s.grid_size, s.numpoints, (0, 0), s.table_oversamp, s.kbwidth, s.order)
    om = _as_omega(omega)
    M = om.shape[1]
    w = torch.ones(M, dtype=torch.float64) if weights is None else torch.as_tensor(np.asarray(weights)).reshape(-1)
    data = w.to(torch.complex128).reshape(1, 1, M)
    scale = 1.0 / (s.grid_size[0] * s.grid_size[1]) if norm == "ortho" else 1.0
    adj = (lambda d, o: ndft_adjoint(d, o, spec0)) if exact else (lambda d, o: nufft_adjoint(d, o, spec0))
    om_neg = om.copy()
    om_neg[0] = -om_neg[0]
    q1 = adj(data, om)[0, 0]
    q2 = adj(data, om_neg)[0, 0]
    return torch.fft.fft2(circulant_psf(q1, q2) * scale)


def toep_apply(image, kernel, smaps=None) -> torch.Tensor:
    """image [B, C, N0, N1]; kernel [2 N0, 2 N1] or [1 or B, 2 N0, 2 N1]; smaps [1 or B, coils, N0, N1] (image then
    [B, 1, N0, N1]) -> complex128, the same shape as the image."""
    x = torch.as_tensor(image).to(torch.complex128)
    k = torch.as_tensor(kernel).to(torch.complex128)
    if k.dim() == 2:
        k = k[None]
    N0, N1 = x.shape[-2:]
    if smaps is not None:
        sm = torch.as_tensor(smaps).to(torch.complex128)
        x = x * sm
    y = torch.fft.ifft2(k[:, None] * torch.fft.fft2(x, s=(2 * N0, 2 * N1)))[..., :N0, :N1]
    if smaps is not None:
        y = (y * sm.conj()).sum(1, keepdim=True)
    return y
