"""Float64 restatement of toep_cg (TEST INFRASTRUCTURE, like oracle/): conjugate gradient on T + lam I with
T = oracle_toep.toep_apply, the freeze rules of include/pdu.h included.  Per system (a plane; a batch element with
smaps):
    r = b - (T + lam) x0 (r = b without x0);  p = r;  rho = ||r||^2;  bb = ||b||^2
    repeat max_iter times:
        q = (T + lam) p;  pi = Re<p, q>
        if frozen or rho == 0 or pi <= 0:  freeze (x, r stay)
        alpha = rho / pi;  x += alpha p;  r -= alpha q;  rho' = ||r||^2
        if rho' <= tol^2 bb:  freeze
        p = r + (rho' / rho) p;  rho = rho'"""
from __future__ import annotations

import numpy as np
import torch

from oracle_toep import toep_apply


def _lam_b(lam, B):
    lam = torch.as_tensor(np.asarray(lam, dtype=np.float64)).reshape(-1)
    if lam.numel() == 1:
        lam = lam.expand(B)
    return lam.reshape(B, 1, 1, 1).to(torch.complex128)


def toep_cg(b, kernel, smaps=None, lam=0.0, x0=None, max_iter=10, tol=0.0, conj=False) -> torch.Tensor:
    """b [B, C, N0, N1] (with smaps [1 or B, coils, N0, N1]: C = 1); lam a number or 1 / B values; conj solves with
    conj(kernel).  complex128, the shape of b."""
    b = torch.as_tensor(b).to(torch.complex128)
    k = torch.as_tensor(kernel).to(torch.complex128)
    if conj:
        k = k.conj()
    lam_b = _lam_b(lam, b.shape[0])

    def op(v):
        return toep_apply(v, k, smaps) + lam_b * v

    def dot(u, v):                                     # Re<u, v> per system, [B, C, 1, 1]
        return (u.conj() * v).real.sum(dim=(-2, -1), keepdim=True)

    x = torch.zeros_like(b) if x0 is None else torch.as_tensor(x0).to(torch.complex128).clone()
    r = b - op(x) if x0 is not None else b.clone()
    p = r.clone()
    rho = dot(r, r)
    bb = dot(b, b)
    frozen = torch.zeros_like(rho, dtype=torch.bool)
    for _ in range(max_iter):
        q = op(p)
        pi = dot(p, q)
        stop = frozen | (rho == 0) | ~(pi > 0)
        alpha = torch.where(stop, torch.zeros_like(rho), rho / torch.where(stop, torch.ones_like(pi), pi))
        x = torch.where(stop, x, x + alpha * p)
        r = torch.where(stop, r, r - alpha * q)
        rho_new = dot(r, r)
        frozen = stop | (rho_new <= tol * tol * bb)
        beta = torch.where(frozen, torch.zeros_like(rho), rho_new / torch.where(frozen, torch.ones_like(rho), rho))
        p = torch.where(frozen, p, r + beta * p)
        rho = torch.where(frozen, rho, rho_new)
    return x


def dense_operator(kernel, shape, smaps=None, lam=0.0) -> np.ndarray:
    """The matrix of T + lam I on one system of `shape` [1, C, N0, N1], built column by column from toep_apply."""
    n = int(np.prod(shape))
    cols = []
    for i in range(n):
        e = torch.zeros(n, dtype=torch.complex128)
        e[i] = 1.0
        cols.append(toep_apply(e.reshape(shape), kernel, smaps).reshape(-1).numpy())
    return np.stack(cols, axis=1) + lam * np.eye(n)
