"""Coil-map gradients of KbNufft, KbNufftAdjoint, ToepNufft and toep_cg against autograd through the float64 oracles
(tests/test_oracle_smaps_grad.py pins those to finite differences), on every adjoint path the dispatcher can choose, with
the unchanged-behaviour, determinism and graph-capture checks."""
import numpy as np
import pytest
import torch
from torch import nn

import oracle
import pd_unet_b200 as pdu
from oracle_toep import toep_apply
from pd_unet_b200 import _lib
from pd_unet_b200.model import PrimalDualUNetMRI
from pd_unet_b200.phantoms import coil_maps
from util import TOL, rel_l2, seeded

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _c(shape, seed):
    return seeded(shape, seed, complex_=True)


def _split(z):            # [B, C, ...] complex -> [B, 2 C, ...] float32, (re, im) neighbouring channels
    return torch.view_as_real(z).movedim(-1, 2).reshape(z.shape[0], 2 * z.shape[1], *z.shape[2:]).contiguous()


def _ref_grad(fn, S, G):
    S = S.detach().cpu().to(torch.complex128).requires_grad_(True)
    (g,) = torch.autograd.grad(fn(S), S, G.detach().cpu().to(torch.complex128))
    return g


PATH_SEEN = []


def _lib_grad(fn, S, G, split=False):
    """S.grad of fn(S) for G; PATH_SEEN[-1] is pdu_last_kernel("smaps_grad") read in the thread that ran the backward
    (the record is per thread, and autograd runs CUDA backward functions in its own thread)."""
    S = S.detach().clone().to(DEV).requires_grad_(True)
    S.register_hook(lambda g: PATH_SEEN.append(_lib.last_kernel("smaps_grad")))
    out = fn(S)
    out.backward(_split(G).to(DEV) if split else G.to(DEV))
    return S.grad


# (im, spokes, readout, B, coils, path substring): the fused row-binned path (640 grid, >= 8 planes, sparse), the
# register-FFT generic path (< 8 planes), the pfft path (96 = 2^5 3), the cuFFT path (112 = 2^4 7)
PATHS = [((320, 320), 48, 640, 2, 8, "fz_rows_adj_kernel"), ((128, 128), 8, 256, 2, 3, "ff_rows_adj"),
         ((48, 48), 8, 96, 2, 3, "pfft_rows_adj_kernel"), ((56, 56), 8, 112, 2, 3, "cuFFT")]
LAYOUTS = [(1, False, None), ("B", True, "ortho"), (3, False, "ortho")]      # smaps batch (3: 3-D maps), split, norm


@pytest.mark.parametrize("im,spokes,readout,B,coils,path", PATHS)
@pytest.mark.parametrize("sb,split,norm", LAYOUTS)
def test_kbnufft_smaps_grad(im, spokes, readout, B, coils, path, sb, split, norm):
    spec = oracle.NufftSpec(im)
    om = oracle.radial_trajectory(spokes, readout)
    omd = torch.from_numpy(om).to(DEV)
    shape = (coils,) + im if sb == 3 else ((1 if sb == 1 else B), coils) + im
    S, x, G = _c(shape, 1), _c((B, 1) + im, 2), _c((B, coils, om.shape[1]), 3)
    op = pdu.KbNufft(im).to(DEV)
    xin = (_split(x) if split else x).to(DEV)
    got = _lib_grad(lambda s: op(xin, omd, smaps=s, norm=norm, split=split), S, G, split)
    assert path in PATH_SEEN[-1]
    want = _ref_grad(lambda s: oracle.nufft_forward(x.to(torch.complex128), om, spec, smaps=s, norm=norm), S, G)
    assert got.shape == S.shape and rel_l2(got, want) <= TOL


@pytest.mark.parametrize("im,spokes,readout,B,coils,path", PATHS)
@pytest.mark.parametrize("sb,split,norm", LAYOUTS)
def test_kbnufft_adjoint_smaps_grad(im, spokes, readout, B, coils, path, sb, split, norm):
    spec = oracle.NufftSpec(im)
    om = oracle.radial_trajectory(spokes, readout)
    omd = torch.from_numpy(om).to(DEV)
    M = om.shape[1]
    shape = (coils,) + im if sb == 3 else ((1 if sb == 1 else B), coils) + im
    S, y, G = _c(shape, 4), _c((B, coils, M), 5), _c((B, 1) + im, 6)
    w = torch.linspace(0.5, 1.5, M)
    op = pdu.KbNufftAdjoint(im).to(DEV)
    yin = (_split(y) if split else y).to(DEV)
    got = _lib_grad(lambda s: op(yin, omd, smaps=s, norm=norm, split=split, kweight=w.to(DEV)), S, G, split)
    assert path in PATH_SEEN[-1]
    yw = y.to(torch.complex128) * w.double()
    want = _ref_grad(lambda s: oracle.nufft_adjoint(yw, om, spec, smaps=s, norm=norm), S, G)
    assert got.shape == S.shape and rel_l2(got, want) <= TOL


@pytest.mark.parametrize("adjoint", [False, True])
def test_batched_omega_shared_maps(adjoint):
    im, coils, B = (128, 128), 8, 2                       # 8 planes per trajectory, sparse: the fused path
    spec = oracle.NufftSpec(im)
    oms = [oracle.radial_trajectory(24, 256), oracle.radial_trajectory(25, 256)[:, :24 * 256]]
    omd = torch.from_numpy(np.stack(oms)).to(DEV)
    S = _c((1, coils) + im, 7)
    if adjoint:
        y, G = _c((B, coils, oms[0].shape[1]), 8), _c((B, 1) + im, 9)
        got = _lib_grad(lambda s: pdu.KbNufftAdjoint(im)(y.to(DEV), omd, smaps=s), S, G)
        ref = lambda s: torch.cat([oracle.nufft_adjoint(y[b:b + 1].to(torch.complex128), oms[b], spec, smaps=s)  # noqa: E731
                                   for b in range(B)])
    else:
        x, G = _c((B, 1) + im, 8), _c((B, coils, oms[0].shape[1]), 9)
        got = _lib_grad(lambda s: pdu.KbNufft(im)(x.to(DEV), omd, smaps=s), S, G)
        ref = lambda s: torch.cat([oracle.nufft_forward(x[b:b + 1].to(torch.complex128), oms[b], spec, smaps=s)  # noqa: E731
                                   for b in range(B)])
    assert "fz_rows_adj_kernel" in PATH_SEEN[-1]
    assert rel_l2(got, _ref_grad(ref, S, G)) <= TOL


def _toep_kernel(im, B, seed):
    # a non-Hermitian kernel, one per batch element: T^H differs from T
    return _c((B, 2 * im[0], 2 * im[1]), seed)


@pytest.mark.parametrize("im,path", [((128, 128), "tz_rows_out_kernel"), ((60, 60), "smaps_grad_kernel")])
@pytest.mark.parametrize("sb", [1, "B", 3])
def test_toep_smaps_grad(im, path, sb):
    B, coils = 3, 4
    k = _toep_kernel(im, B, 10)
    shape = (coils,) + im if sb == 3 else ((1 if sb == 1 else B), coils) + im
    S, x, G = _c(shape, 11), _c((B, 1) + im, 12), _c((B, 1) + im, 13)
    got = _lib_grad(lambda s: pdu.ToepNufft()(x.to(DEV), k.to(DEV), smaps=s), S, G)
    assert path in PATH_SEEN[-1]
    want = _ref_grad(lambda s: toep_apply(x, k, s), S, G)
    assert got.shape == S.shape and rel_l2(got, want) <= TOL


@pytest.mark.parametrize("im", [(128, 128), (32, 32)])
@pytest.mark.parametrize("sb", [1, 2])
def test_toep_cg_smaps_grad(im, sb):
    B, coils = 2, 3
    om = oracle.radial_trajectory(16, 2 * im[0])
    omd = torch.from_numpy(om).to(DEV)
    k = pdu.calc_toeplitz_kernel(omd, im, norm="ortho")
    lam = 0.1 * float(k.abs().max())
    S = coil_maps(coils, im[0])[None].repeat(sb, 1, 1, 1) * (1.0 + 0.1 * _c((sb, coils) + im, 14))
    b, G = _c((B, 1) + im, 15), _c((B, 1) + im, 16)
    got = _lib_grad(lambda s: pdu.toep_cg(b.to(DEV), k, smaps=s, lam=lam, max_iter=60), S, G)
    # reference: -G(x, v) with x = M^-1 b and v = M^-H g from the float64 restatement, G the ToepNufft map gradient
    from oracle_cg import toep_cg as cg_ref
    kc = k.cpu().to(torch.complex128)
    Sd = S.to(torch.complex128)
    x = cg_ref(b.to(torch.complex128), kc, smaps=Sd, lam=lam, max_iter=200)
    v = cg_ref(G.to(torch.complex128), kc, smaps=Sd, lam=lam, max_iter=200, conj=True)
    want = -_ref_grad(lambda s: toep_apply(x, kc, s), S, v)
    assert rel_l2(got, want) <= 1e-4


def test_kbnufft_matches_aten_composition():
    # reduced configs[3] share: 320^2, 8 coils, 48 spokes, DCF; the no-smaps operators with an ATen multiply
    im, coils, B = (320, 320), 8, 2
    om = torch.from_numpy(oracle.radial_trajectory(48, 640)).to(DEV)
    w = pdu.calc_density_compensation_function(om, im, num_iterations=4).real.reshape(-1).contiguous()
    S0 = coil_maps(coils, 320)[None].to(DEV)
    x, y = _c((B, 1) + im, 17).to(DEV), _c((B, coils, om.shape[1]), 18).to(DEV)
    gy, gx = _c((B, coils, om.shape[1]), 19).to(DEV), _c((B, 1) + im, 20).to(DEV)
    fwd, adj = pdu.KbNufft(im).to(DEV), pdu.KbNufftAdjoint(im).to(DEV)
    for lib_fn, aten_fn, G in [
            (lambda s: fwd(x, om, smaps=s, norm="ortho"), lambda s: fwd(x * s, om, norm="ortho"), gy),
            (lambda s: adj(y, om, smaps=s, norm="ortho", kweight=w),
             lambda s: (adj(y, om, norm="ortho", kweight=w) * s.conj()).sum(1, keepdim=True), gx)]:
        a, b = S0.clone().requires_grad_(True), S0.clone().requires_grad_(True)
        lib_fn(a).backward(G)
        aten_fn(b).backward(G)
        assert rel_l2(a.grad, b.grad) <= TOL


def _backward_counts(fn, S, G, inp):
    """(launches of the backward, image gradient) for maps with and without requires_grad."""
    out = {}
    for need in (False, True):
        s = S.clone().requires_grad_(need)
        i = inp.clone().requires_grad_(True)
        y = fn(i, s)
        torch.cuda.synchronize()
        _lib.launch_count(reset=True)
        y.backward(G)
        torch.cuda.synchronize()
        out[need] = (_lib.launch_count(), i.grad.clone(), y.detach().clone())
    return out


def test_unchanged_without_map_gradient():
    im, coils, B = (128, 128), 8, 2          # 16 planes: the fused path both ways, no atomics in the data gradient
    om = torch.from_numpy(oracle.radial_trajectory(8, 256)).to(DEV)
    S = _c((1, coils) + im, 21).to(DEV)
    x, y = _c((B, 1) + im, 22).to(DEV), _c((B, coils, om.shape[1]), 23).to(DEV)
    k = _toep_kernel(im, 1, 24)[0].to(DEV)
    cases = [
        (lambda i, s: pdu.KbNufft(im)(i, om, smaps=s), x, _c((B, coils, om.shape[1]), 25).to(DEV), 1),
        (lambda i, s: pdu.KbNufftAdjoint(im)(i, om, smaps=s), y, _c((B, 1) + im, 26).to(DEV), 1),
        (lambda i, s: pdu.ToepNufft()(i, k, smaps=s), x, _c((B, 1) + im, 27).to(DEV), 3),
    ]
    for fn, inp, G, extra_sets in cases:
        r = _backward_counts(fn, S, G, inp)
        # the same launches as the parent without the map gradient; the image / data gradient is bit-identical
        assert torch.equal(r[False][1], r[True][1]) and torch.equal(r[False][2], r[True][2])
        assert r[True][0] > r[False][0]
    # the parent's launch counts: the NUFFT backward is one transform; the Toeplitz backward one fast apply (3 launches)
    r = _backward_counts(cases[2][0], S, cases[2][2], x)
    assert r[False][0] == 3 and r[True][0] == 3 + 6


def test_deterministic_and_graph_capture():
    im, coils, B = (128, 128), 8, 2
    om = torch.from_numpy(oracle.radial_trajectory(24, 256)).to(DEV)
    k = pdu.calc_toeplitz_kernel(om, im)
    lam = 0.1 * float(k.abs().max())
    fwd, adj = pdu.KbNufft(im).to(DEV), pdu.KbNufftAdjoint(im).to(DEV)
    S = _c((1, coils) + im, 28).to(DEV).requires_grad_(True)
    x = _c((B, 1) + im, 29).to(DEV)
    G = _c((B, 1) + im, 30).to(DEV)

    def step():
        S.grad = None
        z = adj(fwd(x, om, smaps=S), om, smaps=S)
        u = pdu.toep_cg(z, k, smaps=S, lam=lam, max_iter=5)
        u.backward(G)
        return S.grad.clone()

    a, b = step(), step()
    assert torch.equal(a, b)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    S.grad = None
    with torch.cuda.graph(g):
        z = adj(fwd(x, om, smaps=S), om, smaps=S)
        u = pdu.toep_cg(z, k, smaps=S, lam=lam, max_iter=5)
        u.backward(G)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(S.grad, a)


class _MapNet(nn.Module):
    """A small conv net refining coil maps: [coils, N, N] complex -> complex, as an E2E-VarNet-style sensitivity
    network would."""

    def __init__(self, coils):
        super().__init__()
        self.conv = nn.Conv2d(2 * coils, 2 * coils, 3, padding=1)

    def forward(self, s):
        r = torch.view_as_real(s).permute(0, 3, 1, 2).reshape(1, -1, *s.shape[-2:])
        r = r + 0.1 * self.conv(r)
        r = r.reshape(s.shape[0], 2, *s.shape[-2:]).permute(0, 2, 3, 1).contiguous()
        return torch.view_as_complex(r)[None]


def test_map_network_trains_through_the_mri_model_and_cg():
    im, spokes, readout, coils = (32, 32), 8, 64, 2
    om = torch.from_numpy(oracle.radial_trajectory(spokes, readout)).to(DEV)
    maps0 = coil_maps(coils, 32).to(DEV)
    torch.manual_seed(3)
    net = _MapNet(coils).to(DEV)
    model = PrimalDualUNetMRI(im, spokes, readout, coils=coils, n_iter=2, n_primal=4, n_dual=2 * coils, unet_base=8,
                              unet_depth=2, dual_features=8).to(DEV)
    kdata = _c((1, coils, spokes * readout), 31).to(DEV)
    dcf = pdu.calc_density_compensation_function(om, im)
    out = model(kdata, om, net(maps0), dcf)
    out.abs().pow(2).mean().backward()
    for p in net.parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all() and p.grad.abs().sum() > 0
    # a toep_cg data-consistency step
    net.zero_grad()
    k = pdu.calc_toeplitz_kernel(om, im)
    b = _c((1, 1) + im, 32).to(DEV)
    x = pdu.toep_cg(b, k, smaps=net(maps0), lam=0.1 * float(k.abs().max()), max_iter=10)
    x.abs().pow(2).mean().backward()
    for p in net.parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all() and p.grad.abs().sum() > 0
