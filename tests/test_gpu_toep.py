"""The Toeplitz-embedded NUFFT normal operator (calc_toeplitz_kernel, ToepNufft) against the float64 restatement in
tests/oracle_toep.py, against the library's own NUFFT pair, and its autograd, reproducibility, graph capture and errors."""
import ctypes

import numpy as np
import pytest
import torch

import oracle
import pd_unet_b200 as pdu
from oracle_toep import toep_apply, toeplitz_kernel
from pd_unet_b200 import _lib
from pd_unet_b200 import nufft as nufft_mod
from pd_unet_b200.phantoms import coil_maps
from util import TOL, rel_l2, seeded

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FAST = {(128, 128), (256, 256), (320, 320), (512, 512), (1024, 1024)}


def _traj(n_spokes, n_readout):
    return oracle.radial_trajectory(n_spokes, n_readout)


def _dcf(omd, im):
    return pdu.calc_density_compensation_function(omd, im, num_iterations=4)     # complex64 [1, 1, M], zero imaginary part


@pytest.mark.parametrize("im,spokes,norm,dcf", [
    ((32, 32), 8, None, False), ((48, 40), 10, "ortho", True), ((96, 96), 12, None, True),
    ((128, 128), 12, "ortho", False), ((256, 256), 16, None, True), ((320, 320), 16, "ortho", True),
    ((512, 512), 16, None, False)])
def test_kernel_matches_oracle(im, spokes, norm, dcf):
    om = _traj(spokes, 2 * max(im))
    omd = torch.from_numpy(om).to(DEV)
    w = _dcf(omd, im) if dcf else None
    k = pdu.calc_toeplitz_kernel(omd, im, weights=w, norm=norm)
    assert k.shape == (2 * im[0], 2 * im[1]) and k.dtype == torch.complex64
    wn = w.real.reshape(-1).cpu().double().numpy() if dcf else None
    assert rel_l2(k, toeplitz_kernel(om, oracle.NufftSpec(im), weights=wn, norm=norm)) <= TOL


def test_batched_omega_gives_one_kernel_per_trajectory():
    im = (64, 64)
    oms = [_traj(8, 128), _traj(11, 128)[:, :8 * 128]]
    omd = torch.from_numpy(np.stack(oms)).to(DEV)
    w = torch.linspace(0.5, 1.5, 8 * 128, device=DEV)
    k = pdu.calc_toeplitz_kernel(omd, im, weights=w, norm="ortho", n_shift=(3, 5))
    assert k.shape == (2, 128, 128)
    for b in range(2):
        want = toeplitz_kernel(oms[b], oracle.NufftSpec(im), weights=w.cpu().double().numpy(), norm="ortho")
        assert rel_l2(k[b], want) <= TOL


# (im, B, channels or coils, smaps batch (0: no smaps), kernel batch)
APPLY_CASES = [((32, 32), 2, 3, 0, 1), ((48, 40), 2, 3, 2, 2), ((96, 96), 2, 3, 1, 1), ((128, 128), 2, 2, 0, 2),
               ((256, 256), 2, 4, 1, 2), ((320, 320), 2, 4, 2, 1), ((512, 512), 1, 2, 0, 1), ((1024, 1024), 1, 2, 0, 1)]


@pytest.mark.parametrize("im,B,C,sb,kb", APPLY_CASES)
def test_apply_matches_oracle(im, B, C, sb, kb):
    om = _traj(8, 2 * max(im))
    om2 = np.stack([om, _traj(9, 2 * max(im))[:, :om.shape[1]]])[:kb]
    omd = torch.from_numpy(om2 if kb > 1 else om).to(DEV)
    k = pdu.calc_toeplitz_kernel(omd, im, norm="ortho")
    sm = None
    if sb:
        sm = seeded((sb, C) + im, 21, complex_=True)
        x = seeded((B, 1) + im, 22, complex_=True)
    else:
        x = seeded((B, C) + im, 22, complex_=True)
    y = pdu.ToepNufft()(x.to(DEV), k, smaps=sm.to(DEV) if sm is not None else None, norm="ortho")
    assert y.shape == x.shape
    name = _lib.last_kernel("toep")
    assert ("tz_cols_kernel" in name) == (im in FAST) and ("tz_mul_kernel" in name) == (im not in FAST), name
    assert rel_l2(y, toep_apply(x, k.cpu(), smaps=sm)) <= TOL


def test_normal_operator_matches_the_nufft_pair_at_the_configs3_share():
    im, coils, B, spokes = (320, 320), 8, 8, 48
    omd = torch.from_numpy(_traj(spokes, 2 * im[0])).to(DEV)
    sm = coil_maps(coils, im[0])[None].to(DEV)
    w = _dcf(omd, im)
    x = seeded((B, 1) + im, 31, complex_=True).to(DEV)
    k = pdu.calc_toeplitz_kernel(omd, im, weights=w, norm="ortho")
    got = pdu.ToepNufft()(x, k, smaps=sm, norm="ortho")
    A, AH = pdu.KbNufft(im).to(DEV), pdu.KbNufftAdjoint(im).to(DEV)
    want = AH(A(x, omd, smaps=sm, norm="ortho") * w, omd, smaps=sm, norm="ortho")
    err = rel_l2(got, want)
    print(f"\nToeplitz vs KbNufftAdjoint(KbNufft(x) * w), 320^2 x 8 coils x 8, 48 spokes, ortho, DCF: rel-L2 {err:.3e}")
    assert err <= 2e-3


@pytest.mark.parametrize("im,smaps", [((256, 256), True), ((48, 40), False)])
def test_adjoint_and_autograd_with_a_non_hermitian_kernel(im, smaps):
    k = seeded((2 * im[0], 2 * im[1]), 41, complex_=True).to(DEV)            # not the transform of a Hermitian PSF
    sm = seeded((1, 3) + im, 42, complex_=True).to(DEV) if smaps else None
    shape = (2, 1) + im if smaps else (2, 3) + im
    x = seeded(shape, 43, complex_=True).to(DEV)
    y = seeded(shape, 44, complex_=True).to(DEV)
    op = pdu.ToepNufft()
    Tx = op(x, k, smaps=sm)
    THy = nufft_mod._toep_apply(y, k, sm, True)
    lhs, rhs = torch.vdot(Tx.flatten().cdouble(), y.flatten().cdouble()), torch.vdot(x.flatten().cdouble(), THy.flatten().cdouble())
    assert abs(complex(lhs - rhs)) <= 1e-5 * abs(complex(lhs))
    xr = x.clone().requires_grad_(True)
    op(xr, k, smaps=sm).backward(y)
    assert rel_l2(xr.grad, THy) <= 1e-6
    assert rel_l2(THy, toep_apply(y.cpu(), k.cpu().conj(), smaps=sm.cpu() if smaps else None)) <= TOL


@pytest.mark.parametrize("im", [(320, 320), (96, 96)])
def test_two_calls_are_bit_identical(im):
    omd = torch.from_numpy(_traj(12, 2 * im[0])).to(DEV)
    k = pdu.calc_toeplitz_kernel(omd, im)
    sm = coil_maps(4, im[0])[None].to(DEV)
    x = seeded((3, 1) + im, 51, complex_=True).to(DEV)
    a = pdu.ToepNufft()(x, k, smaps=sm)
    b = pdu.ToepNufft()(x, k, smaps=sm)
    assert torch.equal(a, b)
    assert ("fast path" if im[0] == 320 else "generic path") in _lib.last_kernel("toep")


def test_graph_capture_replays_the_eager_result():
    im = (320, 320)
    omd = torch.from_numpy(_traj(16, 640)).to(DEV)
    k = pdu.calc_toeplitz_kernel(omd, im, norm="ortho")
    sm = coil_maps(4, im[0])[None].to(DEV)
    x = seeded((2, 1) + im, 61, complex_=True).to(DEV)
    op = pdu.ToepNufft()
    eager = op(x, k, smaps=sm)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        op(x, k, smaps=sm)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = op(x, k, smaps=sm)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)


def test_a_toeplitz_plan_collected_during_capture_is_destroyed_later():
    import gc
    tp = nufft_mod._ToepPlan((64, 64))
    tp.handle(torch.device(DEV))
    a = torch.arange(256.0, device=DEV)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        del tp
        gc.collect()
        b = a + 1
    assert nufft_mod._DEFERRED_DESTROY
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(b, a + 1)
    other = nufft_mod._ToepPlan((64, 64))
    other.handle(torch.device(DEV))
    del other
    gc.collect()
    assert not nufft_mod._DEFERRED_DESTROY


def test_errors():
    im = (64, 64)
    omd = torch.from_numpy(_traj(8, 128)).to(DEV)
    k = pdu.calc_toeplitz_kernel(omd, im)
    x = seeded((1, 2) + im, 71, complex_=True).to(DEV)
    with pytest.raises(ValueError):
        pdu.ToepNufft()(x, k[:, :-2])
    with pytest.raises(ValueError):
        pdu.ToepNufft()(x, torch.stack([k, k, k]))                     # kernel batch 3 for an image batch of 1
    with pytest.raises(ValueError):
        pdu.ToepNufft()(x, k, norm="forward")
    with pytest.raises(pdu.PduError):
        pdu.ToepNufft()(x.cpu(), k.cpu())
    with pytest.raises(pdu.PduError):
        pdu.calc_toeplitz_kernel(omd.cpu(), im)
    bad = torch.complex(torch.ones(omd.shape[1]), torch.full((omd.shape[1],), 0.1)).to(DEV)
    with pytest.raises(ValueError):
        pdu.calc_toeplitz_kernel(omd, im, weights=bad)
    with pytest.raises(NotImplementedError):
        pdu.calc_toeplitz_kernel(torch.from_numpy(_traj(8, 154)).to(DEV), (77, 77))
    with pytest.raises(NotImplementedError):
        pdu.ToepNufft()(torch.zeros(1, 1, 77, 77, dtype=torch.complex64, device=DEV),
                        torch.zeros(154, 154, dtype=torch.complex64, device=DEV))


def test_toeplitz_and_kaiser_bessel_plans_are_not_interchangeable():
    L = _lib.lib()
    im = (64, 64)
    th = nufft_mod._toep_plan(im).handle(torch.device(DEV))
    kb = pdu.KbNufft(im)._plan.handle(torch.device(DEV))
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device=DEV)
    ptr = buf.data_ptr()
    st = _lib.stream_ptr()
    assert L.pdu_nufft_fwd_c64(th, ptr, ptr, ptr, None, 1, 1, 1, 16, 1.0, ptr, buf.numel(), st) == -1
    assert b"Toeplitz" in L.pdu_last_error()
    assert L.pdu_nufft_csr_build(th, ptr, 16, ptr, buf.numel(), st) == -1
    assert L.pdu_toep_apply_c64(kb, ptr, ptr, ptr, 1, None, 1, 1, 1, 0, ptr, buf.numel(), st) == -1
    assert L.pdu_toep_kernel_c64(kb, ptr, ptr, ptr, 1, 1.0, ptr, buf.numel(), st) == -1
    assert L.pdu_toep_workspace_bytes(kb, 4) == 0
    # 128-point grids are no FastFft size: the generic scratch, grid + intermediate + cropped plane
    assert L.pdu_toep_workspace_bytes(th, 4) == 4 * (128 * 128 + 64 * 128 + 64 * 64) * 8
