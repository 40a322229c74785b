"""The float64 CG restatement (tests/oracle_cg.py) against a direct solve of the dense T + lam I, its freeze rules,
and the argument checks of pdu_toep_cg_* on a host without a device."""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from oracle_cg import dense_operator, toep_cg
from oracle_toep import toep_apply, toeplitz_kernel
from util import rel_l2, seeded

IM = (12, 12)                                          # 2 N = 24 = 2^3 3: a generic size


def _kernel(weighted=True):
    om = oracle.radial_trajectory(5, 24)
    w = (0.5 + torch.rand(om.shape[1], generator=torch.Generator().manual_seed(5), dtype=torch.float64)).numpy() \
        if weighted else None
    return toeplitz_kernel(om, oracle.NufftSpec(IM), weights=w, exact=True)


@pytest.mark.parametrize("smaps", [False, True])
@pytest.mark.parametrize("warm", [False, True])
def test_oracle_reaches_the_direct_solution(smaps, warm):
    k = _kernel()
    sm = seeded((1, 3) + IM, 2, complex_=True).to(torch.complex128) if smaps else None
    b = seeded((2, 1) + IM, 3, complex_=True).to(torch.complex128)
    lam = [0.05 * float(k.abs().max()), 0.2 * float(k.abs().max())]
    x0 = seeded((2, 1) + IM, 4, complex_=True) if warm else None
    x = toep_cg(b, k, smaps=sm, lam=lam, x0=x0, max_iter=300)
    for i in range(2):
        M = dense_operator(k, (1, 1) + IM, smaps=sm, lam=lam[i])
        assert np.allclose(M, M.conj().T, atol=1e-9 * np.abs(M).max())       # Hermitian: real weights
        want = np.linalg.solve(M, b[i].reshape(-1).numpy())
        assert rel_l2(x[i].reshape(-1), torch.from_numpy(want)) <= 1e-9
    # the residual the iteration reports agrees with the operator
    res = toep_apply(x, k, sm) + torch.tensor(lam, dtype=torch.float64).reshape(2, 1, 1, 1) * x - b
    assert float(res.norm() / b.norm()) <= 1e-9


def test_planes_are_independent_systems_without_smaps():
    k = _kernel()
    b = seeded((1, 3) + IM, 6, complex_=True)
    x = toep_cg(b, k, lam=1.0, max_iter=7)
    for c in range(3):
        assert torch.equal(x[:, c:c + 1], toep_cg(b[:, c:c + 1], k, lam=1.0, max_iter=7))


def test_zero_rhs_gives_zero_and_a_zero_operator_gives_x0():
    k = _kernel()
    x = toep_cg(torch.zeros((1, 1) + IM, dtype=torch.complex64), k, lam=0.5, max_iter=5)
    assert torch.count_nonzero(x) == 0
    x0 = seeded((1, 1) + IM, 7, complex_=True)
    b = seeded((1, 1) + IM, 8, complex_=True)
    x = toep_cg(b, torch.zeros_like(k), lam=0.0, x0=x0, max_iter=5)
    assert torch.equal(x, x0.to(torch.complex128))
    assert bool(torch.isfinite(x).all())


def test_tol_freezes_a_system_while_another_goes_on():
    k = _kernel()
    big = float(k.abs().max())
    b = seeded((2, 1) + IM, 9, complex_=True)
    lam = [100.0 * big, 1e-3 * big]                    # well conditioned vs. ill conditioned
    xs = [toep_cg(b, k, lam=lam, max_iter=m, tol=1e-4) for m in (3, 8, 20)]
    assert torch.equal(xs[1][0], xs[2][0])             # converged early and frozen
    assert not torch.equal(xs[1][1], xs[2][1])         # still iterating
    assert float(toep_cg(b[:1], k, lam=lam[0], max_iter=3, tol=0.0).sub(xs[0][0:1]).abs().max()) < 1e-6 * float(xs[0].abs().max())


def test_max_iter_zero_returns_x0_or_zero():
    k = _kernel()
    b = seeded((1, 1) + IM, 10, complex_=True)
    assert torch.count_nonzero(toep_cg(b, k, lam=1.0, max_iter=0)) == 0
    x0 = seeded((1, 1) + IM, 11, complex_=True)
    assert torch.equal(toep_cg(b, k, lam=1.0, x0=x0, max_iter=0), x0.to(torch.complex128))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    from pd_unet_b200 import _lib
    return _lib.lib()


def test_cg_entry_points_reject_bad_arguments_without_a_device(lib):
    assert lib.pdu_toep_cg_workspace_bytes(None, 1, 1, 0) == 0
    assert lib.pdu_toep_cg_c64(None, None, None, None, None, 1, None, 1, 1, 1, None, 1, 1, 0.0, 0, None, 0, None) == -1
    assert b"plan is null" in lib.pdu_last_error()
    assert lib.pdu_last_kernel(b"cg") == b""
