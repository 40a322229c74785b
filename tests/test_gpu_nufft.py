"""Parity of the CUDA NUFFT (through the C ABI, via pd_unet_b200.nufft) with the CPU oracle."""
import numpy as np
import pytest
import torch

import oracle
import pd_unet_b200 as pdu
from pd_unet_b200.phantoms import coil_maps
from util import TOL, rel_l2, seeded

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _traj(n_spokes, n_readout):
    return oracle.radial_trajectory(n_spokes, n_readout)


@pytest.mark.parametrize("im,spokes", [((32, 32), 8), ((64, 48), 12), ((256, 256), 32), ((320, 320), 48)])
def test_forward_and_adjoint_match_oracle(im, spokes):
    spec = oracle.NufftSpec(im)
    om = _traj(spokes, 2 * im[0])
    omd = torch.from_numpy(om).to(DEV)
    B, C = (2, 3) if im[0] <= 64 else (1, 2)
    x = seeded((B, C) + im, 1, complex_=True)
    y = pdu.KbNufft(im)(x.to(DEV), omd)
    assert y.shape == (B, C, om.shape[1])
    assert rel_l2(y, oracle.nufft_forward(x, om, spec)) <= TOL
    k = seeded((B, C, om.shape[1]), 2, complex_=True)
    xa = pdu.KbNufftAdjoint(im)(k.to(DEV), omd)
    assert rel_l2(xa, oracle.nufft_adjoint(k, om, spec)) <= TOL


def test_ortho_norm_and_smaps():
    im, coils = (64, 64), 4
    spec = oracle.NufftSpec(im)
    om = _traj(16, 128)
    omd = torch.from_numpy(om).to(DEV)
    smaps = coil_maps(coils, 64)[None]
    x = seeded((2, 1) + im, 3, complex_=True)
    y = pdu.KbNufft(im)(x.to(DEV), omd, smaps=smaps.to(DEV), norm="ortho")
    assert y.shape == (2, coils, om.shape[1])
    assert rel_l2(y, oracle.nufft_forward(x, om, spec, smaps=smaps, norm="ortho")) <= TOL
    k = seeded((2, coils, om.shape[1]), 4, complex_=True)
    xa = pdu.KbNufftAdjoint(im)(k.to(DEV), omd, smaps=smaps.to(DEV), norm="ortho")
    assert xa.shape == (2, 1) + im
    assert rel_l2(xa, oracle.nufft_adjoint(k, om, spec, smaps=smaps, norm="ortho")) <= TOL
    # per-batch smaps
    sm2 = torch.cat([smaps, smaps.flip(1)], 0)
    y2 = pdu.KbNufft(im)(x.to(DEV), omd, smaps=sm2.to(DEV))
    assert rel_l2(y2, oracle.nufft_forward(x, om, spec, smaps=sm2)) <= TOL


def test_against_exact_ndft_small():
    im = (24, 24)
    spec = oracle.NufftSpec(im)
    om = _traj(6, 48)
    x = seeded((1, 1) + im, 5, complex_=True)
    y = pdu.KbNufft(im)(x.to(DEV), torch.from_numpy(om).to(DEV))
    assert rel_l2(y, oracle.ndft_forward(x, om, spec)) < 2e-3     # Kaiser-Bessel J=6 approximation error


def test_interp_pair_and_dcf():
    im = (48, 48)
    spec = oracle.NufftSpec(im)
    om = _traj(10, 96)
    omd = torch.from_numpy(om).to(DEV)
    grid = seeded((1, 2, 96, 96), 6, complex_=True)
    y = pdu.KbInterp(im)(grid.to(DEV), omd)
    assert rel_l2(y, oracle.interp_forward(grid, om, spec)) <= TOL
    k = seeded((1, 2, om.shape[1]), 7, complex_=True)
    ga = pdu.KbInterpAdjoint(im)(k.to(DEV), omd)
    assert rel_l2(ga, oracle.interp_adjoint(k, om, spec)) <= TOL
    w = pdu.calc_density_compensation_function(omd, im, num_iterations=6)
    assert w.shape == (1, 1, om.shape[1])
    assert rel_l2(w.real.reshape(-1), oracle.calc_dcf(om, spec, 6)) <= 5e-5   # six chained divisions


def test_adjointness_and_autograd():
    im = (64, 64)
    om = torch.from_numpy(_traj(12, 128)).to(DEV)
    A, AH = pdu.KbNufft(im), pdu.KbNufftAdjoint(im)
    x = seeded((1, 2) + im, 8, complex_=True).to(DEV)
    k = seeded((1, 2, om.shape[1]), 9, complex_=True).to(DEV)
    lhs = torch.vdot(k.reshape(-1).to(torch.complex128), A(x, om).reshape(-1).to(torch.complex128))
    rhs = torch.vdot(AH(k, om).reshape(-1).to(torch.complex128), x.reshape(-1).to(torch.complex128))
    assert abs(lhs - rhs) / abs(lhs) < 1e-5
    xr = x.clone().requires_grad_()
    (A(xr, om) * k.conj()).real.sum().backward()
    assert rel_l2(xr.grad, AH(k, om)) <= 1e-6


def test_batched_trajectory_empty_and_errors():
    im = (32, 32)
    om = torch.from_numpy(_traj(4, 64)).to(DEV)
    x = seeded((2, 1) + im, 10, complex_=True).to(DEV)
    A = pdu.KbNufft(im)
    both = A(x, torch.stack([om, -om]))
    assert torch.equal(both[0:1], A(x[0:1], om)) and torch.equal(both[1:2], A(x[1:2], -om))
    assert A(x[:0], om).shape == (0, 1, om.shape[1])
    with pytest.raises(pdu.PduError):
        A(x.cpu(), om.cpu())
    with pytest.raises(TypeError):
        A(x.real, om)
    with pytest.raises(NotImplementedError):
        A(x, om, interp_mats=(None, None))


def test_sorted_gather_adjoint_matches_scatter_and_is_reproducible():
    """The CSR (sorted gather) adjoint interpolator: same numbers as the atomic scatter and the oracle,
    bit-identical from call to call, rebuilt when the trajectory changes."""
    im = (64, 48)
    spec = oracle.NufftSpec(im)
    om = _traj(14, 128)
    omd = torch.from_numpy(om).to(DEV)
    k = seeded((2, 3, om.shape[1]), 21, complex_=True)
    adj = pdu.KbNufftAdjoint(im)
    adj._plan.use_csr = True                                     # "auto" would pick the scatter for 6 planes
    a1 = adj(k.to(DEV), omd)
    a2 = adj(k.to(DEV), omd)
    assert torch.equal(a1, a2)                                   # no atomics: reproducible
    assert rel_l2(a1, oracle.nufft_adjoint(k, om, spec)) <= TOL
    adj._plan.use_csr = False
    assert rel_l2(adj(k.to(DEV), omd), a1) <= 1e-6               # the scatter agrees
    adj._plan.use_csr = True
    # interp-only path and a modified trajectory (in-place change bumps the version -> rebuild)
    ia = pdu.KbInterpAdjoint(im)
    ia._plan.use_csr = True
    g1 = ia(k.to(DEV), omd)
    assert rel_l2(g1, oracle.interp_adjoint(k, om, spec)) <= TOL
    omd.mul_(0.5)
    assert rel_l2(adj(k.to(DEV), omd), oracle.nufft_adjoint(k, 0.5 * om, spec)) <= TOL
    # smaps + ortho through the same path
    sm = coil_maps(3, 64)[None][..., :48].contiguous()
    xa = adj(k.to(DEV), omd, smaps=sm.to(DEV), norm="ortho")
    assert rel_l2(xa, oracle.nufft_adjoint(k, 0.5 * om, spec, smaps=sm, norm="ortho")) <= TOL


@pytest.mark.parametrize("planes", [(1, 4), (1, 5), (1, 7), (2, 4), (3, 4), (1, 16), (3, 7), (2, 16), (1, 33), (4, 16)])
@pytest.mark.parametrize("dense", [False, True])
def test_sorted_gather_shapes_over_plane_counts(planes, dense):
    """Every instantiation of the sorted gather -- 2 lanes per cell (4 - 7 planes), 4 lanes x 8 planes (8 - 15, and dense
    trajectories), 4 lanes x 16 planes (sparse trajectories from 16 planes, everything from 64), plane counts that are
    not a multiple of the group size, and the long rows (k-space centre) inside the same launch -- against the oracle,
    against the atomic scatter, and bit-reproducible."""
    from pd_unet_b200 import _lib
    B, Cc = planes
    im = (40, 36)
    spec = oracle.NufftSpec(im)
    om = _traj(36 if dense else 7, 80)                # dense: 18 entries per cell and centre cells far above 32 entries
    omd = torch.from_numpy(om).to(DEV)
    k = seeded((B, Cc, om.shape[1]), 100 + B * Cc, complex_=True)
    adj = pdu.KbNufftAdjoint(im)
    adj._plan.use_csr, adj._plan.use_fused = True, False
    a1 = adj(k.to(DEV), omd)
    assert "interp_adj_csrT_kernel" in _lib.last_kernel("nufft_adj")
    assert torch.equal(a1, adj(k.to(DEV), omd))
    pick = [(0, 0), (B - 1, Cc - 1), (B // 2, Cc // 2)]
    for b, c in pick:
        assert rel_l2(a1[b:b + 1, c:c + 1], oracle.nufft_adjoint(k[b:b + 1, c:c + 1], om, spec)) <= TOL
    adj._plan.use_csr = False
    assert rel_l2(adj(k.to(DEV), omd), a1) <= 2e-6    # every plane agrees with the scatter


@pytest.mark.parametrize("traj", ["radial", "few", "cluster", "uniform"])
@pytest.mark.parametrize("planes", [(1, 8), (3, 4), (1, 17), (3, 11)])
def test_compact_gridded_samples_between_gather_and_row_pass(planes, traj):
    """On the grids with the register FFT a sparse trajectory's gridded samples stay compact (one value per non-empty
    cell) between the sorted gather and the row pass: radial spokes, a handful of samples (most grid rows entirely
    empty), a tight cluster (long rows only, a few cells) and uniform random samples, plane counts around the group
    sizes -- against the oracle on three planes, against the atomic scatter on all, and bit-reproducible."""
    from pd_unet_b200 import _lib
    B, Cc = planes
    im = (128, 128)
    spec = oracle.NufftSpec(im)
    rng = np.random.default_rng(7)
    if traj == "radial":
        om = _traj(12, 256)
    elif traj == "few":
        om = rng.uniform(-np.pi, np.pi, (2, 23))
    elif traj == "cluster":
        om = np.clip(rng.normal(0.3, 0.01, (2, 900)), -np.pi, np.pi)
    else:
        om = rng.uniform(-np.pi, np.pi, (2, 5000))
    om = om.astype(np.float32).astype(np.float64)
    omd = torch.from_numpy(om).to(DEV).float()
    k = seeded((B, Cc, om.shape[1]), 300 + B * Cc, complex_=True)
    adj = pdu.KbNufftAdjoint(im)
    adj._plan.use_csr, adj._plan.use_fused = True, False
    a1 = adj(k.to(DEV), omd)
    name = _lib.last_kernel("nufft_adj")
    assert "non-empty cells only" in name and "ff_rows_adj_compact_kernel" in name, name
    assert torch.equal(a1, adj(k.to(DEV), omd))
    for b, c in [(0, 0), (B - 1, Cc - 1), (B // 2, Cc // 2)]:
        assert rel_l2(a1[b:b + 1, c:c + 1], oracle.nufft_adjoint(k[b:b + 1, c:c + 1], om, spec)) <= TOL
    adj._plan.use_csr = False
    assert rel_l2(adj(k.to(DEV), omd), a1) <= 2e-6


@pytest.mark.parametrize("im", [(32, 32), (48, 40), (320, 320), (256, 256), (250, 250)])
def test_pruned_fft_and_cufft_paths_agree(im):
    """variant 1: the own pruned shared-memory FFT; variant 0 (default, currently faster): pad + cuFFT.  Same
    numbers, both within budget of the oracle.  250 -> grid 500 = 4 * 5^3 exercises the radix-5 passes."""
    spec = oracle.NufftSpec(im)
    om = _traj(9, 2 * im[0])
    omd = torch.from_numpy(om).to(DEV)
    x = seeded((1, 2) + im, 31, complex_=True)
    k = seeded((1, 2, om.shape[1]), 32, complex_=True)
    A, AH = pdu.KbNufft(im), pdu.KbNufftAdjoint(im)
    want_f, want_a = oracle.nufft_forward(x, om, spec), oracle.nufft_adjoint(k, om, spec)
    try:
        for v in (2, 1, 0):      # 2: register-resident pruned FFT (grids 512 / 640; other sizes fall back to 0)
            pdu.set_option("nufft_fwd_variant", v)
            pdu.set_option("nufft_adj_variant", v)
            assert rel_l2(A(x.to(DEV), omd), want_f) <= TOL, f"forward variant {v}"
            assert rel_l2(AH(k.to(DEV), omd), want_a) <= TOL, f"adjoint variant {v}"
    finally:
        pdu.set_option("nufft_fwd_variant", -1)
        pdu.set_option("nufft_adj_variant", -1)


@pytest.mark.parametrize("n,coils,batch,spokes", [(320, 8, 8, 48), (256, 1, 1, 32)])
def test_full_size_adjointness_and_linearity(n, coils, batch, spokes):
    """BASELINE configs[3] / configs[0] shapes (the register-resident pruned FFT and the sorted gather are the
    default paths there), checked through size-independent properties: <A x, y> = <x, A^H y> with coil maps and
    ortho norm, and A(a x1 + x2) = a A x1 + A x2."""
    im = (n, n)
    om = torch.from_numpy(_traj(spokes, 2 * n)).to(DEV)
    A, AH = pdu.KbNufft(im), pdu.KbNufftAdjoint(im)
    sm = coil_maps(coils, n)[None].to(DEV) if coils > 1 else None
    ci = 1 if coils > 1 else coils
    x = seeded((batch, ci) + im, 41, complex_=True).to(DEV)
    x2 = seeded((batch, ci) + im, 42, complex_=True).to(DEV)
    k = seeded((batch, coils, om.shape[1]), 43, complex_=True).to(DEV)
    Ax = A(x, om, smaps=sm, norm="ortho")
    AHk = AH(k, om, smaps=sm, norm="ortho")
    assert Ax.shape == k.shape and AHk.shape == x.shape
    c128 = torch.complex128
    lhs = torch.vdot(k.reshape(-1).to(c128), Ax.reshape(-1).to(c128))
    rhs = torch.vdot(AHk.reshape(-1).to(c128), x.reshape(-1).to(c128))
    assert abs(lhs - rhs) / abs(lhs) < 1e-5
    a = 0.37 - 1.2j
    assert rel_l2(A(a * x + x2, om, smaps=sm, norm="ortho"), a * Ax + A(x2, om, smaps=sm, norm="ortho")) <= 1e-6
    # the three FFT paths agree at full size
    try:
        outs = []
        for v in (2, 0):
            pdu.set_option("nufft_fwd_variant", v)
            pdu.set_option("nufft_adj_variant", v)
            outs.append((A(x, om, smaps=sm, norm="ortho"), AH(k, om, smaps=sm, norm="ortho")))
        assert rel_l2(outs[0][0], outs[1][0]) <= 2e-6 and rel_l2(outs[0][1], outs[1][1]) <= 2e-6
    finally:
        pdu.set_option("nufft_fwd_variant", -1)
        pdu.set_option("nufft_adj_variant", -1)


@pytest.mark.parametrize("numpoints", [4, 5, 8])
def test_non_default_numpoints(numpoints):
    """J != 6 takes the run-time-J instantiation of the gather / scatter kernels (J = 6 is compiled straight-line)."""
    im = (48, 40)
    spec = oracle.NufftSpec(im, numpoints=numpoints)
    om = _traj(10, 96)
    omd = torch.from_numpy(om).to(DEV)
    x = seeded((2, 2) + im, 51, complex_=True)
    k = seeded((2, 2, om.shape[1]), 52, complex_=True)
    A, AH = pdu.KbNufft(im, numpoints=numpoints), pdu.KbNufftAdjoint(im, numpoints=numpoints)
    assert rel_l2(A(x.to(DEV), omd), oracle.nufft_forward(x, om, spec)) <= TOL
    assert rel_l2(AH(k.to(DEV), omd), oracle.nufft_adjoint(k, om, spec)) <= TOL


def test_default_path_at_the_cfg4_share_matches_oracle():
    """VERDICT r01 weak #2: the DEFAULT kernels at BASELINE configs[3]'s per-GPU share (320^2, 8 coils, batch 8,
    48 spokes: 64 planes -> own FFT, sorted / binned gathers, fused coil combine) compared with the float64 oracle
    itself, not only through properties.  The oracle runs batch element 5 (all 8 coils) and, without coil maps, planes
    (0, 0) and (7, 7) of a 64-plane call: seconds on the CPU."""
    from pd_unet_b200 import _lib
    n, coils, batch, spokes = 320, 8, 8, 48
    im = (n, n)
    spec = oracle.NufftSpec(im)
    om = _traj(spokes, 2 * n)
    omd = torch.from_numpy(om).to(DEV)
    A, AH = pdu.KbNufft(im), pdu.KbNufftAdjoint(im)
    sm = coil_maps(coils, n)[None]
    x = seeded((batch, 1) + im, 61, complex_=True)
    k = seeded((batch, coils, om.shape[1]), 62, complex_=True)
    y = A(x.to(DEV), omd, smaps=sm.to(DEV), norm="ortho")
    fwd_kernel = _lib.last_kernel("nufft_fwd")
    xa = AH(k.to(DEV), omd, smaps=sm.to(DEV), norm="ortho")
    adj_kernel = _lib.last_kernel("nufft_adj")
    assert "cufft" not in fwd_kernel.lower() and "cufft" not in adj_kernel.lower(), (fwd_kernel, adj_kernel)
    assert "fz_rows_fwd_kernel" in fwd_kernel and "ff_rows_adj_" in adj_kernel       # the measured-fastest pair at 64 planes
    b = 5
    assert rel_l2(y[b:b + 1], oracle.nufft_forward(x[b:b + 1], om, spec, smaps=sm, norm="ortho")) <= TOL
    assert rel_l2(xa[b:b + 1], oracle.nufft_adjoint(k[b:b + 1], om, spec, smaps=sm, norm="ortho")) <= TOL
    # no coil maps: 64 independent planes in one call
    x64 = seeded((batch, coils) + im, 63, complex_=True)
    y64 = A(x64.to(DEV), omd)
    xa64 = AH(k.to(DEV), omd)
    for bb, cc in ((0, 0), (7, 7)):
        assert rel_l2(y64[bb, cc], oracle.nufft_forward(x64[bb:bb + 1, cc:cc + 1], om, spec)[0, 0]) <= TOL
        assert rel_l2(xa64[bb, cc], oracle.nufft_adjoint(k[bb:bb + 1, cc:cc + 1], om, spec)[0, 0]) <= TOL
    # the adjoint of a fixed trajectory is bit-reproducible (no atomics on the default path)
    assert torch.equal(AH(k.to(DEV), omd, smaps=sm.to(DEV), norm="ortho"), xa)


@pytest.mark.parametrize("n,planes,spokes", [(128, 3, 24), (256, 9, 20), (320, 2, 17), (512, 3, 12), (1024, 2, 6)])
def test_fused_path_every_grid_size(n, planes, spokes):
    """csrc/nufft_fused.cu on each grid it is compiled for (256, 512, 640, 1024, 2048), with plane counts that are
    not multiples of the CTA's plane group, against the float64 oracle -- and against the generic path."""
    from pd_unet_b200 import _lib
    im = (n, n)
    spec = oracle.NufftSpec(im)
    om = _traj(spokes, 2 * n)
    omd = torch.from_numpy(om).to(DEV)
    A, AH = pdu.KbNufft(im), pdu.KbNufftAdjoint(im)
    A._plan.use_fused = AH._plan.use_fused = True          # "auto" keeps small plane counts on the generic path
    x = seeded((1, planes) + im, 71, complex_=True)
    k = seeded((1, planes, om.shape[1]), 72, complex_=True)
    y, xa = A(x.to(DEV), omd), AH(k.to(DEV), omd)
    assert "fz_rows_fwd_kernel" in _lib.last_kernel("nufft_fwd") and "fz_rows_adj_kernel" in _lib.last_kernel("nufft_adj")
    check = [0, planes - 1]
    assert rel_l2(y[:, check], oracle.nufft_forward(x[:, check], om, spec)) <= TOL
    assert rel_l2(xa[:, check], oracle.nufft_adjoint(k[:, check], om, spec)) <= TOL
    A._plan.use_fused = AH._plan.use_fused = False
    assert rel_l2(A(x.to(DEV), omd), y) <= 2e-6 and rel_l2(AH(k.to(DEV), omd), xa) <= 2e-6
    assert "fz_" not in _lib.last_kernel("nufft_fwd")


def test_split_layout_and_density_weights():
    """The (re, im)-as-channels layout and the fused density compensation give the same numbers as the complex API
    followed by the layout passes -- with and without coil maps, on the fused path and on the generic one."""
    for n, coils, fused in ((256, 1, True), (320, 4, True), (320, 4, "auto"), (48, 3, "auto")):
        im = (n, n)
        om = torch.from_numpy(_traj(11, 2 * n)).to(DEV)
        M = om.shape[1]
        A, AH = pdu.KbNufft(im), pdu.KbNufftAdjoint(im)
        A._plan.use_fused = AH._plan.use_fused = fused
        sm = coil_maps(coils, n)[None].to(DEV) if coils > 1 else None
        x = seeded((2, 1) + im, 81, complex_=True).to(DEV)
        k = seeded((2, coils, M), 82, complex_=True).to(DEV)
        w = torch.rand(M, generator=torch.Generator().manual_seed(3)).to(DEV) + 0.5
        xs = torch.stack([x.real, x.imag], 2).reshape(2, 2, n, n).contiguous()
        ks = torch.stack([k.real, k.imag], 2).reshape(2, 2 * coils, M).contiguous()
        y = A(x, om, smaps=sm, norm="ortho")
        ys = A(xs, om, smaps=sm, norm="ortho", split=True)
        assert ys.shape == (2, 2 * coils, M) and ys.dtype == torch.float32
        assert rel_l2(torch.complex(ys.reshape(2, coils, 2, M)[:, :, 0], ys.reshape(2, coils, 2, M)[:, :, 1]), y) <= 1e-6
        xa = AH(k * w, om, smaps=sm, norm="ortho")
        xas = AH(ks, om, smaps=sm, norm="ortho", split=True, kweight=w)
        co = xa.shape[1]
        assert xas.shape == (2, 2 * co, n, n)
        assert rel_l2(torch.complex(xas.reshape(2, co, 2, n, n)[:, :, 0], xas.reshape(2, co, 2, n, n)[:, :, 1]), xa) <= 1e-6
        # gradients flow through the split / weighted forms: <A^H(w k), x> differentiated in k is w A x
        ksr = ks.clone().requires_grad_()
        (AH(ksr, om, smaps=sm, norm="ortho", split=True, kweight=w) * xs[:, :2 * co]).sum().backward()
        want = A(xs, om, smaps=sm, norm="ortho", split=True) * w
        assert rel_l2(ksr.grad, want) <= 1e-5


def test_a_plan_collected_during_graph_capture_leaves_the_capture_intact():
    """An MRI model refers to itself through its operator closures, so the cyclic garbage collector may free it, and its
    NUFFT plans, inside another CUDA-graph capture.  Releasing a plan's device memory there would invalidate that
    capture; it is released with the next plan collected outside a capture instead."""
    import gc
    from pd_unet_b200 import nufft as nufft_mod
    im = (128, 128)
    omd = torch.from_numpy(_traj(12, 256)).to(DEV)
    x = seeded((1, 1) + im, 91, complex_=True).to(DEV)
    cycle = [pdu.KbNufft(im)]
    cycle.append(cycle)
    cycle[0]._plan.use_fused = True                  # builds the trajectory's row bins (device buffer + CUDA event)
    cycle[0](x, omd)
    a = torch.arange(1024.0, device=DEV)
    gc.collect()                                     # only this test's plan is left to collect inside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        del cycle
        gc.collect()
        b = a * 2
    assert nufft_mod._DEFERRED_DESTROY
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(b, a * 2)
    op = pdu.KbNufft(im)
    op(x, omd)
    del op
    gc.collect()
    assert not nufft_mod._DEFERRED_DESTROY
