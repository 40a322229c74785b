"""The float64 Toeplitz restatement (tests/oracle_toep.py) against first principles, and the argument checks of the
pdu_toep_* entry points on a host without a device."""
import ctypes

import pytest
import torch

import oracle
from oracle_toep import toep_apply, toeplitz_kernel
from util import rel_l2, seeded


def _normal_ndft(x, om, spec, w):
    y = oracle.ndft_forward(x, om, spec)
    if w is not None:
        y = y * torch.as_tensor(w, dtype=torch.float64)
    return oracle.ndft_adjoint(y, om, spec)


@pytest.mark.parametrize("im", [(24, 24), (20, 28)])
@pytest.mark.parametrize("weighted", [False, True])
def test_exact_psf_embedding_is_the_normal_operator(im, weighted):
    spec = oracle.NufftSpec(im)
    om = oracle.radial_trajectory(6, 2 * max(im))
    w = (0.5 + torch.rand(om.shape[1], generator=torch.Generator().manual_seed(3), dtype=torch.float64)).numpy() if weighted else None
    k = toeplitz_kernel(om, spec, weights=w, exact=True)
    assert k.shape == (2 * im[0], 2 * im[1])
    x = seeded((2, 3) + im, 11, complex_=True)
    want = _normal_ndft(x, om, spec, w)
    assert rel_l2(toep_apply(x, k), want) <= 1e-12
    # with coil maps: sum_c conj(S_c) T (S_c x)
    sm = seeded((1, 3) + im, 12, complex_=True).to(torch.complex128)
    x1 = x[:, :1].to(torch.complex128)
    want_s = (_normal_ndft(x1 * sm, om, spec, w) * sm.conj()).sum(1, keepdim=True)
    assert rel_l2(toep_apply(x1, k, smaps=sm), want_s) <= 1e-12


def test_exact_kernel_is_real_and_ortho_scales_it():
    im = (24, 24)
    spec = oracle.NufftSpec(im)
    om = oracle.radial_trajectory(6, 48)
    k = toeplitz_kernel(om, spec, exact=True)
    assert float(k.imag.abs().max()) <= 1e-12 * float(k.abs().max())
    ko = toeplitz_kernel(om, spec, exact=True, norm="ortho")
    assert rel_l2(ko * (48 * 48), k) <= 1e-14


@pytest.mark.parametrize("im", [(24, 24), (20, 28)])
def test_kaiser_bessel_kernel_is_close_to_the_exact_one(im):
    spec = oracle.NufftSpec(im)
    om = oracle.radial_trajectory(6, 2 * max(im))
    assert rel_l2(toeplitz_kernel(om, spec), toeplitz_kernel(om, spec, exact=True)) <= 2e-3   # J = 6 approximation


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    from pd_unet_b200 import _lib
    return _lib.lib()


def test_toep_entry_points_reject_bad_arguments_without_a_device(lib):
    p = ctypes.c_void_p()
    assert lib.pdu_toep_plan_create(None, 8, 8) == -1
    assert lib.pdu_toep_plan_create(ctypes.byref(p), 0, 8) == -1
    assert lib.pdu_toep_plan_create(ctypes.byref(p), 77, 77) == -4          # 154 = 2 * 7 * 11: no Toeplitz path
    assert b"2, 3, 5" in lib.pdu_last_error()
    assert lib.pdu_toep_workspace_bytes(None, 4) == 0
    assert lib.pdu_toep_kernel_c64(None, None, None, None, 1, 1.0, None, 0, None) == -1
    assert lib.pdu_toep_apply_c64(None, None, None, None, 1, None, 1, 1, 1, 0, None, 0, None) == -1
    assert lib.pdu_last_kernel(b"toep") == b""
