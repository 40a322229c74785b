"""toep_cg, conjugate gradient on the Toeplitz normal operator: iterates against the float64 restatement in
tests/oracle_cg.py, convergence, launch counts, the freeze rules, determinism (batch make-up, graph replay, no host
synchronisation), the implicit gradients, consistency with the NUFFT pair and the errors."""
import numpy as np
import pytest
import torch

import oracle
import pd_unet_b200 as pdu
from oracle_cg import toep_cg as cg_ref
from oracle_toep import toep_apply
from pd_unet_b200 import _lib
from pd_unet_b200 import nufft as nufft_mod
from pd_unet_b200.phantoms import coil_maps
from util import TOL, rel_l2, seeded

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FAST = {(128, 128), (256, 256), (320, 320), (512, 512), (1024, 1024)}
LAUNCHES_PER_ITER = {True: 5, False: 9}                 # fast path: 3 apply + update + direction; generic: 6 + 3
APPLY_LAUNCHES = {True: 3, False: 7}                    # the apply with the CG epilogue (set-up with x0)
# after 30 iterations with lam = 0.1 max|kernel| (condition number <= 11) exact CG is at ~1e-8; what remains is the
# float32 floor: each apply carries ~1e-6 relative error and the recursive residual drifts from the true one by a few
# times that, so the true residual settles in the 1e-6 .. 1e-5 range.  1e-4 leaves a margin of ten.
RESIDUAL_BOUND = 1e-4


def _kernel(im, kb, norm="ortho"):
    om = oracle.radial_trajectory(8, 2 * max(im))
    if kb > 1:
        om = np.stack([om, oracle.radial_trajectory(9, 2 * max(im))[:, :om.shape[1]]])[:kb]
    return pdu.calc_toeplitz_kernel(torch.from_numpy(om).to(DEV), im, norm=norm)


def _lam(kind, k, B):
    big = float(k.abs().max())
    if kind == "scalar":
        return 0.1 * big, 0.1 * big
    vals = [0.1 * big * (1 + i) for i in range(B)]
    return torch.tensor(vals, dtype=torch.float32, device=DEV), vals


def _problem(im, B, C, sb, seed):
    if sb:
        sm = seeded((sb, C) + im, seed, complex_=True)
        sm = sm / (sm.abs() ** 2).sum(1, keepdim=True).sqrt()         # sum_c |S_c|^2 = 1: ||operator|| <= max|kernel|
        b = seeded((B, 1) + im, seed + 1, complex_=True)
    else:
        sm, b = None, seeded((B, C) + im, seed + 1, complex_=True)
    return b, sm


# (im, B, channels or coils, smaps batch (0: no smaps), kernel batch, lam kind, warm start)
CASES = [((128, 128), 2, 2, 0, 1, "scalar", False), ((256, 256), 2, 3, 1, 2, "tensor", True),
         ((320, 320), 2, 4, 2, 1, "tensor", False), ((320, 320), 2, 2, 0, 2, "scalar", True),
         ((32, 32), 2, 3, 0, 2, "scalar", True), ((48, 40), 2, 3, 2, 2, "tensor", False),
         ((96, 96), 2, 2, 1, 1, "scalar", True), ((96, 96), 2, 2, 0, 1, "tensor", False)]


@pytest.mark.parametrize("im,B,C,sb,kb,lam_kind,warm", CASES)
def test_iterates_match_oracle(im, B, C, sb, kb, lam_kind, warm):
    k = _kernel(im, kb)
    b, sm = _problem(im, B, C, sb, 11)
    x0 = seeded(tuple(b.shape), 13, complex_=True) if warm else None
    lam, lam_ref = _lam(lam_kind, k, B)
    fast = im in FAST
    smd = sm.to(DEV) if sm is not None else None
    x0d = x0.to(DEV) if warm else None
    for m in (1, 3):
        pdu.launch_count(reset=True)
        x = pdu.toep_cg(b.to(DEV), k, smaps=smd, lam=lam, x0=x0d, max_iter=m)
        torch.cuda.synchronize()
        launches = pdu.launch_count()
        assert launches == (APPLY_LAUNCHES[fast] if warm else 0) + 1 + LAUNCHES_PER_ITER[fast] * m
        name = _lib.last_kernel("cg")
        assert ("tz_rows_out_kernel" in name and ",cg>" in name) == fast, name
        assert ("cg_lam_dot_kernel" in name) == (not fast), name
        want = cg_ref(b, k.cpu(), smaps=sm, lam=lam_ref, x0=x0, max_iter=m)
        assert rel_l2(x, want) <= TOL, (m, rel_l2(x, want))


@pytest.mark.parametrize("im,sb", [((320, 320), 1), ((96, 96), 0), ((48, 40), 2)])
def test_thirty_iterations_solve_the_system(im, sb):
    B, C = 2, 3
    k = _kernel(im, 1)
    b, sm = _problem(im, B, C, sb, 21)
    lam, lam_ref = _lam("tensor", k, B)
    x = pdu.toep_cg(b.to(DEV), k, smaps=sm.to(DEV) if sm is not None else None, lam=lam, max_iter=30)
    x64 = x.cpu().to(torch.complex128)
    lam_b = torch.tensor(lam_ref, dtype=torch.float64).reshape(B, 1, 1, 1)
    res = toep_apply(x64, k.cpu(), smaps=sm) + lam_b * x64 - b.to(torch.complex128)
    err = float(res.norm() / b.to(torch.complex128).norm())
    print(f"\n30 iterations, {im}, smaps batch {sb}: ||(T + lam) x - b|| / ||b|| = {err:.2e}")
    assert err <= RESIDUAL_BOUND
    assert bool(torch.isfinite(x).all())


def test_a_converged_system_freezes_while_a_harder_one_goes_on():
    im = (128, 128)
    k = _kernel(im, 1)
    big = float(k.abs().max())
    b = seeded((2, 1) + im, 31, complex_=True).to(DEV)
    lam = torch.tensor([100.0 * big, 2e-2 * big], dtype=torch.float32, device=DEV)
    xa = pdu.toep_cg(b, k, lam=lam, max_iter=8, tol=1e-3)
    xb = pdu.toep_cg(b, k, lam=lam, max_iter=13, tol=1e-3)
    assert torch.equal(xa[0], xb[0])
    assert not torch.equal(xa[1], xb[1])
    assert bool(torch.isfinite(xb).all())


@pytest.mark.parametrize("im", [(128, 128), (48, 40)])
def test_zero_rhs_and_zero_kernel(im):
    k = _kernel(im, 1)
    z = torch.zeros((2, 2) + im, dtype=torch.complex64, device=DEV)
    x = pdu.toep_cg(z, k, lam=1.0, max_iter=4)
    assert torch.count_nonzero(x) == 0
    b = seeded((2, 2) + im, 41, complex_=True).to(DEV)
    x0 = seeded((2, 2) + im, 42, complex_=True).to(DEV)
    x = pdu.toep_cg(b, torch.zeros_like(k), lam=0.0, x0=x0, max_iter=4)
    assert torch.equal(x, x0)
    x = pdu.toep_cg(b, torch.zeros_like(k), lam=0.0, max_iter=4)      # no x0: stays at zero
    assert torch.count_nonzero(x) == 0
    assert torch.equal(pdu.toep_cg(b, k, lam=1.0, x0=x0, max_iter=0), x0)
    assert torch.count_nonzero(pdu.toep_cg(b, k, lam=1.0, max_iter=0)) == 0


@pytest.mark.parametrize("im", [(320, 320), (96, 96)])
def test_two_calls_and_batch_make_up_are_bit_identical(im):
    k = _kernel(im, 1)
    big = float(k.abs().max())
    sm = coil_maps(4, im[0])[None].to(DEV)
    b = seeded((3, 1) + im, 51, complex_=True).to(DEV)
    lam = torch.tensor([0.05 * big, 0.1 * big, 0.2 * big], dtype=torch.float32, device=DEV)
    a = pdu.toep_cg(b, k, smaps=sm, lam=lam, max_iter=10)
    assert torch.equal(a, pdu.toep_cg(b, k, smaps=sm, lam=lam, max_iter=10))
    alone = pdu.toep_cg(b[1:2].clone(), k, smaps=sm, lam=lam[1:2].clone(), max_iter=10)
    assert torch.equal(alone[0], a[1])


def test_no_host_synchronisation():
    im = (320, 320)
    k = _kernel(im, 1)
    sm = coil_maps(4, im[0])[None].to(DEV)
    b = seeded((2, 1) + im, 61, complex_=True).to(DEV)
    lam_t = torch.tensor([1.0, 2.0], device=DEV)
    pdu.toep_cg(b, k, smaps=sm, lam=0.5, max_iter=3)
    pdu.toep_cg(b, k, smaps=sm, lam=lam_t, x0=b, max_iter=3)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        pdu.toep_cg(b, k, smaps=sm, lam=0.5, max_iter=3)
        pdu.toep_cg(b, k, smaps=sm, lam=lam_t, x0=b, max_iter=3, tol=1e-3)
    finally:
        torch.cuda.set_sync_debug_mode(0)


def test_graph_capture_replays_the_eager_result():
    im = (320, 320)
    k = _kernel(im, 1)
    sm = coil_maps(4, im[0])[None].to(DEV)
    b = seeded((2, 1) + im, 71, complex_=True).to(DEV)
    b2 = seeded((2, 1) + im, 72, complex_=True).to(DEV)
    lam = torch.tensor([0.5, 1.0], device=DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pdu.toep_cg(b, k, smaps=sm, lam=lam, max_iter=6, tol=1e-4)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = pdu.toep_cg(b, k, smaps=sm, lam=lam, max_iter=6, tol=1e-4)
    b.copy_(b2)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, pdu.toep_cg(b2, k, smaps=sm, lam=lam, max_iter=6, tol=1e-4))


@pytest.mark.parametrize("im,smaps,per_batch", [((256, 256), True, False), ((48, 40), False, True)])
def test_implicit_gradients(im, smaps, per_batch):
    B = 2
    k = _kernel(im, 1)
    big = float(k.abs().max())
    sm = _problem(im, B, 3, 1, 81)[1] if smaps else None
    b = seeded((B, 1 if smaps else 2) + im, 82, complex_=True)
    g = seeded(tuple(b.shape), 83, complex_=True)
    vals = [0.1 * big, 0.3 * big] if per_batch else [0.2 * big]
    lam = torch.tensor(vals if per_batch else vals[0], dtype=torch.float32, device=DEV).requires_grad_(True)
    bd = b.to(DEV).requires_grad_(True)
    x = pdu.toep_cg(bd, k, smaps=sm.to(DEV) if smaps else None, lam=lam, max_iter=40)
    x.backward(g.to(DEV))
    x64 = cg_ref(b, k.cpu(), smaps=sm, lam=vals, max_iter=80)
    gb64 = cg_ref(g, k.cpu(), smaps=sm, lam=vals, max_iter=80, conj=True)
    assert rel_l2(bd.grad, gb64) <= 1e-4
    prod = (gb64.conj() * x64).real
    want = -(prod.sum(dim=(1, 2, 3)) if per_batch else prod.sum())
    assert lam.grad.shape == lam.shape
    assert rel_l2(lam.grad.cpu().double(), want) <= 1e-4


def _power_norm(op, shape, iters=12):
    v = seeded(shape, 91, complex_=True).to(DEV)
    for _ in range(iters):
        v = op(v)
        v = v / v.norm()
    return float(op(v).norm())


def test_solution_satisfies_the_nufft_pair_normal_equation():
    im, coils, B, spokes = (320, 320), 8, 2, 48
    omd = torch.from_numpy(oracle.radial_trajectory(spokes, 2 * im[0])).to(DEV)
    sm = coil_maps(coils, im[0])[None].to(DEV)
    w = pdu.calc_density_compensation_function(omd, im, num_iterations=4)
    wr = w.real.reshape(-1).contiguous()
    A, AH = pdu.KbNufft(im).to(DEV), pdu.KbNufftAdjoint(im).to(DEV)
    y = A(seeded((B, 1) + im, 92, complex_=True).to(DEV), omd, smaps=sm, norm="ortho")
    b = AH(y, omd, smaps=sm, norm="ortho", kweight=wr)
    k = pdu.calc_toeplitz_kernel(omd, im, weights=w, norm="ortho")
    lam = 0.05 * _power_norm(lambda v: pdu.ToepNufft()(v, k, smaps=sm), (1, 1) + im)
    x = pdu.toep_cg(b, k, smaps=sm, lam=lam, max_iter=40)
    res = AH(A(x, omd, smaps=sm, norm="ortho"), omd, smaps=sm, norm="ortho", kweight=wr) + lam * x - b
    err = float(res.norm() / b.norm())
    print(f"\ntoep_cg, 320^2 x 8 coils x 2, 48 spokes, DCF, lam {lam:.3g}: NUFFT-pair residual {err:.3e}")
    assert err <= 2e-3


def test_errors():
    im = (64, 64)
    k = _kernel(im, 1)
    b = seeded((2, 2) + im, 95, complex_=True).to(DEV)
    with pytest.raises(ValueError):
        pdu.toep_cg(b[0], k)
    with pytest.raises(ValueError):
        pdu.toep_cg(b, k[:, :-2])
    with pytest.raises(ValueError):
        pdu.toep_cg(b, k, lam=-1.0)
    with pytest.raises(ValueError):
        pdu.toep_cg(b, k, tol=-1e-3)
    with pytest.raises(ValueError):
        pdu.toep_cg(b, k, max_iter=-1)
    with pytest.raises(ValueError):
        pdu.toep_cg(b, k, max_iter=3.0)
    with pytest.raises(ValueError):
        pdu.toep_cg(b, k, lam=torch.ones(3, device=DEV))
    with pytest.raises(ValueError):
        pdu.toep_cg(b, k, x0=b[:1])
    with pytest.raises(ValueError):
        pdu.toep_cg(b, k, smaps=torch.ones((1, 3) + im, dtype=torch.complex64, device=DEV))   # b has 2 channels
    with pytest.raises(pdu.PduError):
        pdu.toep_cg(b.cpu(), k.cpu())
    with pytest.raises(pdu.PduError):
        pdu.toep_cg(b, k, lam=torch.ones(1))
    with pytest.raises(NotImplementedError):
        pdu.toep_cg(torch.zeros(1, 1, 77, 77, dtype=torch.complex64, device=DEV),
                    torch.zeros(154, 154, dtype=torch.complex64, device=DEV))
    L = _lib.lib()
    kb = pdu.KbNufft(im)._plan.handle(torch.device(DEV))
    th = nufft_mod._toep_plan(im).handle(torch.device(DEV))
    buf = torch.zeros(64 << 20, dtype=torch.uint8, device=DEV)
    ptr, st = buf.data_ptr(), _lib.stream_ptr()
    assert L.pdu_toep_cg_c64(kb, ptr, None, ptr, ptr, 1, None, 1, 1, 1, None, 1, 1, 0.0, 0, ptr, buf.numel(), st) == -1
    assert b"Toeplitz" in L.pdu_last_error()
    assert L.pdu_toep_cg_workspace_bytes(kb, 1, 1, 0) == 0
    need = L.pdu_toep_cg_workspace_bytes(th, 1, 1, 0)
    assert 0 < need <= buf.numel()
    assert L.pdu_toep_cg_c64(th, ptr, None, ptr, ptr, 1, None, 1, 1, 1, None, 1, -1, 0.0, 0, ptr, buf.numel(), st) == -1
    assert L.pdu_toep_cg_c64(th, ptr, None, ptr, ptr, 1, None, 1, 1, 1, None, 1, 1, -1.0, 0, ptr, buf.numel(), st) == -1
    assert L.pdu_toep_cg_c64(th, ptr, None, ptr, ptr, 1, None, 1, 1, 1, None, 2, 1, 0.0, 0, ptr, buf.numel(), st) == -1
    assert L.pdu_toep_cg_c64(th, ptr, None, ptr, ptr, 1, None, 1, 1, 1, None, 1, 1, 0.0, 0, ptr, need - 1, st) == -1
    assert b"workspace" in L.pdu_last_error()
