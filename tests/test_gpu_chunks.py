"""NUFFT, Toeplitz, CG and coil-map-gradient calls large enough to be cut into several batch chunks.

Every case derives its chunk size from the library's size rules (csrc/nufft.cu batch_chunk: 512 MB of scratch and at
most 65535 planes per chunk; nufft.py _Plan._binned_chunks: 1 GiB for the fused path), asserts at least two chunks
with a shorter last one, and checks that the chunked call
  - is bit-identical to the same wrapper called on each chunk's batch range (the atomic scatter: to 2e-6),
  - matches the float64 oracle on the batch elements next to every chunk boundary,
  - through the C ABI: writes every output element and nothing behind it, stays inside the workspace its size
    function asks for, and rejects one byte less."""
import math
import re

import pytest
import torch

import oracle
import pd_unet_b200 as pdu
from oracle_cg import toep_cg as cg_ref
from oracle_toep import toep_apply
from pd_unet_b200 import _lib
from pd_unet_b200 import nufft as nufft_mod
from util import TOL, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SCRATCH = 512 << 20          # csrc/nufft.cu batch_chunk: scratch per chunk of the generic NUFFT and Toeplitz paths
GRID_Y = 65535               # and planes per chunk (gridDim.y of the per-plane passes)
BINNED = 1 << 30             # pd_unet_b200/nufft.py _Plan._binned_chunks: scratch per chunk of the fused path
PDU_EINVAL, PDU_ENOMEM = -1, -3
GUARD = 1 << 20              # bytes of pattern behind a workspace
PATTERN = (torch.arange(GUARD) * 151 % 251).to(torch.uint8)
TAIL = 4096                  # NaN elements behind an output


# ----------------------------------------------------------------------------- chunk arithmetic
def _nufft_chunk(plan, coils):
    k0, k1 = plan.grid_size
    return max(1, min(SCRATCH // (k0 * k1 * 8), GRID_Y) // coils)


def _toep_chunk(h, coils):
    return max(1, min(SCRATCH // int(_lib.lib().pdu_toep_workspace_bytes(h, 1)), GRID_Y) // coils)


def _binned_chunk(h, coils, M):
    return max(1, BINNED // int(_lib.lib().pdu_nufft_binned_workspace_bytes(h, coils, M)))


def _chunks(B, cb):
    ch = [(b0, min(B, b0 + cb)) for b0 in range(0, B, cb)]
    assert len(ch) >= 2 and ch[-1][1] - ch[-1][0] < cb, (B, cb)
    return ch


def _edges(ch):
    """The batch elements next to a boundary: the last of every chunk and the first of every later one."""
    return sorted({b1 - 1 for _, b1 in ch} | {b0 for b0, _ in ch[1:]})


def _count(record):
    """The plane / system count a pdu_last_kernel record names: the last chunk's."""
    m = re.findall(r"(\d+) (?:planes|systems) of \d+x\d+", record)
    assert m, record
    return int(m[-1])


def _last_count(op):
    return _count(_lib.last_kernel(op))


def _backward(out, grad, S):
    """out.backward(grad) -> the smaps_grad record of the thread that ran it (autograd runs CUDA backward functions
    in its own thread, and the record is per thread)."""
    seen = []
    S.register_hook(lambda g: seen.append(_lib.last_kernel("smaps_grad")))
    out.backward(grad)
    return seen[-1]


# ----------------------------------------------------------------------------- data
def _rand(shape, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(shape, dtype=torch.complex64, device=DEV, generator=g)


def _traj(spokes, readout):
    om = oracle.radial_trajectory(spokes, readout)
    return om, torch.from_numpy(om).to(DEV)


def _bs(t, b0, b1):
    return nufft_mod._batch_slice(t, b0, b1)


def _at(t, e):
    """t at the batch elements e (all of t when its one entry is shared), float64 on the host."""
    if t is None:
        return None
    t = t.detach()
    return (t if t.shape[0] == 1 else t[e]).cpu().to(torch.complex128)


def _split(z):            # [B, C, ...] complex -> [B, 2 C, ...] float32, (re, im) neighbouring channels
    return torch.view_as_real(z).movedim(-1, 2).reshape(z.shape[0], 2 * z.shape[1], *z.shape[2:]).contiguous()


def _unsplit(t):
    B, C2 = t.shape[:2]
    return torch.view_as_complex(t.reshape(B, C2 // 2, 2, *t.shape[2:]).movedim(2, -1).contiguous())


def _cat(parts):
    return torch.cat([p.detach() for p in parts])


# ----------------------------------------------------------------------------- direct C-ABI calls
def _nan_out(shape, dtype=torch.complex64):
    """(buffer, output view): NaN everywhere, TAIL more elements behind the view."""
    buf = torch.full((math.prod(shape) + TAIL,), float("nan"), dtype=dtype, device=DEV)
    return buf, buf[:math.prod(shape)].view(shape)


def _written(buf, out):
    """Every element of out was written and none behind it."""
    n = out.numel()
    return not bool(torch.isnan(buf[:n]).any()) and bool(torch.isnan(buf[n:]).all())


def _abi(call, need, short_rc=PDU_ENOMEM):
    """call(ws_ptr, ws_bytes) -> rc.  One byte less than need is rejected with short_rc; with need bytes the call
    succeeds and leaves the pattern behind the workspace as it was."""
    ws = torch.empty(need + GUARD, dtype=torch.uint8, device=DEV)
    ws[need:] = PATTERN.to(DEV)
    assert call(ws.data_ptr(), need - 1) == short_rc
    _lib.check(call(ws.data_ptr(), need), "chunked call")
    torch.cuda.synchronize()
    assert torch.equal(ws[need:].cpu(), PATTERN)


def _nufft_ops(im, fused=False, csr=True):
    fwd, adj = pdu.KbNufft(im).to(DEV), pdu.KbNufftAdjoint(im).to(DEV)
    for op in (fwd, adj):
        op._plan.use_fused = fused
        op._plan.use_csr = csr
    return fwd, adj


def _abi_nufft_fwd(plan, x, omd, S, B, coils, M, scale, cb):
    L, h = _lib.lib(), plan.handle(torch.device(DEV))
    buf, out = _nan_out((B, coils, M))
    _abi(lambda ws, n: L.pdu_nufft_fwd_c64(h, x.data_ptr(), out.data_ptr(), omd.data_ptr(),
                                           S.data_ptr() if S is not None else None, B, coils,
                                           S.shape[0] if S is not None else 1, M, scale, ws, n, _lib.stream_ptr()),
         L.pdu_nufft_workspace_bytes(h, min(cb, B) * coils))
    assert _written(buf, out)
    return out


def _abi_nufft_adj(plan, y, omd, S, B, coils, M, scale, cb, im):
    L, h = _lib.lib(), plan.handle(torch.device(DEV))
    csr = plan._csr_for(omd)
    buf, out = _nan_out((B, 1 if S is not None else coils) + im)
    _abi(lambda ws, n: L.pdu_nufft_adj_csr_c64(h, y.data_ptr(), out.data_ptr(), omd.data_ptr(),
                                               S.data_ptr() if S is not None else None, B, coils,
                                               S.shape[0] if S is not None else 1, M, scale, csr.data_ptr(), ws, n,
                                               _lib.stream_ptr()),
         L.pdu_nufft_workspace_bytes(h, min(cb, B) * coils))
    assert _written(buf, out)
    return out


def _abi_nufft_smaps_grad(plan, y, omd, q, gs_shape, B, coils, M, scale, cb, accumulate=None):
    """gs of pdu_nufft_adj_smaps_grad_c64 on the generic path (sorted gather); accumulate: start from this gs."""
    L, h = _lib.lib(), plan.handle(torch.device(DEV))
    csr = plan._csr_for(omd)
    buf, gs = _nan_out(gs_shape)
    if accumulate is not None:
        gs.copy_(accumulate)
    _abi(lambda ws, n: L.pdu_nufft_adj_smaps_grad_c64(h, y.data_ptr(), q.data_ptr(), gs.data_ptr(), omd.data_ptr(),
                                                      csr.data_ptr(), None, None, B, coils, gs_shape[0], M, scale, 0,
                                                      0 if accumulate is None else 1, ws, n, _lib.stream_ptr()),
         L.pdu_nufft_workspace_bytes(h, min(cb, B) * coils))
    assert _written(buf, gs)
    return gs


# ----------------------------------------------------------------------------- generic NUFFT path (C-side cut)
def _check_nufft_fwd_adj(im, B, coils, sb, spokes, readout, norm, variant, seed):
    """KbNufft / KbNufftAdjoint on the generic path over the chunks of B batch elements; variant: the FFT the
    dispatcher names."""
    spec = oracle.NufftSpec(im)
    om, omd = _traj(spokes, readout)
    M = om.shape[1]
    fwd, adj = _nufft_ops(im)
    plan = fwd._plan
    scale = plan.scale(norm)
    cb = _nufft_chunk(plan, coils)
    ch = _chunks(B, cb)
    e = _edges(ch)
    last = (ch[-1][1] - ch[-1][0]) * coils
    S = None if sb is None else _rand(((B if sb == "B" else 1), coils) + im, seed)
    x = _rand((B, 1 if S is not None else coils) + im, seed + 1)
    y = _rand((B, coils, M), seed + 2)

    wrapped = fwd(x, omd, smaps=S, norm=norm)
    got = _abi_nufft_fwd(plan, x, omd, S, B, coils, M, scale, cb)
    assert _last_count("nufft_fwd") == last and variant in _lib.last_kernel("nufft_fwd")
    assert torch.equal(wrapped, got)
    assert torch.equal(_cat(fwd(x[b0:b1], omd, smaps=_bs(S, b0, b1), norm=norm) for b0, b1 in ch), got)
    assert rel_l2(got[e], oracle.nufft_forward(_at(x, e), om, spec, smaps=_at(S, e), norm=norm)) <= TOL

    wrapped = adj(y, omd, smaps=S, norm=norm)
    got = _abi_nufft_adj(adj._plan, y, omd, S, B, coils, M, scale, cb, im)
    assert _last_count("nufft_adj") == last and "sorted gather" in _lib.last_kernel("nufft_adj")
    assert torch.equal(wrapped, got)
    assert torch.equal(_cat(adj(y[b0:b1], omd, smaps=_bs(S, b0, b1), norm=norm) for b0, b1 in ch), got)
    want = oracle.nufft_adjoint(_at(y, e), om, spec, smaps=_at(S, e), norm=norm)
    assert rel_l2(got[e], want) <= TOL

    adj._plan.use_csr = False                           # the atomic scatter: not bit-reproducible
    got = adj(y, omd, smaps=S, norm=norm)
    assert _last_count("nufft_adj") == last and "float2 atomics" in _lib.last_kernel("nufft_adj")
    assert rel_l2(got, _cat(adj(y[b0:b1], omd, smaps=_bs(S, b0, b1), norm=norm) for b0, b1 in ch)) <= 2e-6
    assert rel_l2(got[e], want) <= TOL


@pytest.mark.parametrize("sb", ["B", 1])
def test_nufft_register_fft_two_chunks(sb):
    # 16 planes of 2048^2 per chunk: batch 3 x 8 coils -> [0, 2), [2, 3); per-batch maps move with the chunk
    _check_nufft_fwd_adj((1024, 1024), 3, 8, sb, 4, 2048, "ortho", "register-resident", 10)


def test_nufft_generic_pruned_fft_three_chunks():
    # 16384 planes of 64^2 per chunk; a short third chunk
    cb = _nufft_chunk(pdu.KbNufft((32, 32))._plan, 1)
    _check_nufft_fwd_adj((32, 32), 2 * cb + 232, 1, None, 4, 64, None, "generic pruned FFT", 20)


@pytest.mark.parametrize("im", [(16, 16), (8, 8)])
def test_nufft_more_planes_than_grid_y(im):
    """A grid of at most 1024 cells fits more than 65535 planes into the 512 MB scratch: the chunk is cut at 65535
    planes, the gridDim.y limit of the FFT passes."""
    plan = pdu.KbNufft(im)._plan
    k0, k1 = plan.grid_size
    assert SCRATCH // (k0 * k1 * 8) > GRID_Y
    _check_nufft_fwd_adj(im, GRID_Y + 465, 1, None, 2, 2 * im[0], "ortho", "generic pruned FFT", 30)


@pytest.mark.parametrize("im", [(16, 16), (8, 8)])
def test_nufft_smaps_grad_more_planes_than_grid_y(im):
    spec = oracle.NufftSpec(im)
    om, omd = _traj(2, 2 * im[0])
    M, B = om.shape[1], GRID_Y + 465
    plan = pdu.KbNufft(im)._plan
    plan.use_csr = True
    cb = _nufft_chunk(plan, 1)
    ch = _chunks(B, cb)
    e = _edges(ch)
    y, q = _rand((B, 1, M), 40), _rand((B, 1) + im, 41)
    # per-batch maps: gs[b] = A^H(y[b]) conj(q[b])
    wrapped = torch.empty((B, 1) + im, dtype=torch.complex64, device=DEV)
    plan.smaps_grad(y, omd, q, wrapped, None)
    gs = _abi_nufft_smaps_grad(plan, y, omd, q, (B, 1) + im, B, 1, M, 1.0, cb)
    assert _last_count("smaps_grad") == ch[-1][1] - ch[-1][0]
    assert torch.equal(wrapped, gs)
    assert torch.equal(_cat(_abi_nufft_smaps_grad(plan, y[b0:b1], omd, q[b0:b1], (b1 - b0, 1) + im, b1 - b0, 1, M, 1.0, cb)
                            for b0, b1 in ch), gs)
    assert rel_l2(gs[e], oracle.nufft_adjoint(_at(y, e), om, spec) * _at(q, e).conj()) <= TOL
    # a shared map: the sum carried from chunk 0 into chunk 1
    gs = _abi_nufft_smaps_grad(plan, y, omd, q, (1, 1) + im, B, 1, M, 1.0, cb)
    part = None
    for b0, b1 in ch:
        part = _abi_nufft_smaps_grad(plan, y[b0:b1], omd, q[b0:b1], (1, 1) + im, b1 - b0, 1, M, 1.0, cb, accumulate=part)
    assert torch.equal(part, gs)


@pytest.mark.parametrize("adjoint", [False, True])
@pytest.mark.parametrize("sb", ["B", 1])
def test_nufft_smaps_grad_carry(adjoint, sb):
    """The coil-map gradient of KbNufft / KbNufftAdjoint on the generic path: a shared map's sum is carried from
    chunk 0 into chunk 1 (accumulate)."""
    im, B, coils, norm = (1024, 1024), 3, 8, "ortho"
    spec = oracle.NufftSpec(im)
    om, omd = _traj(4, 2048)
    M = om.shape[1]
    fwd, adj = _nufft_ops(im)
    op = adj if adjoint else fwd
    plan = op._plan
    ch = _chunks(B, _nufft_chunk(plan, coils))
    S = _rand(((B if sb == "B" else 1), coils) + im, 50).requires_grad_(True)
    img, ks = _rand((B, 1) + im, 51), _rand((B, coils, M), 52)
    inp, G = (ks, img) if adjoint else (img, ks)
    assert _count(_backward(op(inp, omd, smaps=S, norm=norm), G, S)) == (ch[-1][1] - ch[-1][0]) * coils
    got = S.grad
    # the map gradient pairs the samples (data) with the image side (q)
    data, q = (ks, G) if adjoint else (G, img)
    gs = torch.empty_like(got)
    for b0, b1 in ch:
        plan.smaps_grad(data[b0:b1], omd, q[b0:b1], _bs(gs, b0, b1), norm, accumulate=sb == 1 and b0 > 0)
    assert torch.equal(gs, got)
    per = []
    for b in range(B):
        g1 = torch.empty((1, coils) + im, dtype=torch.complex64, device=DEV)
        plan.smaps_grad(data[b:b + 1], omd, q[b:b + 1], g1, norm)
        per.append(g1.cpu().to(torch.complex128))
    per = torch.cat(per)
    assert rel_l2(got, per.sum(0, keepdim=True) if sb == 1 else per) <= 1e-6
    e = list(range(B)) if sb == 1 else _edges(ch)
    want = oracle.nufft_adjoint(_at(data, e), om, spec, norm=norm) * _at(q, e).conj()
    if sb == 1:
        assert rel_l2(got, want.sum(0, keepdim=True)) <= TOL
    else:
        assert rel_l2(got[e], want) <= TOL


# ----------------------------------------------------------------------------- fused path (cut in Python)
@pytest.mark.parametrize("sb", ["B", 1])
def test_fused_path_chunks(sb):
    """The row-binned path in the split layout with density weights, cut at 1 GiB of scratch in nufft.py."""
    im, coils, norm = (1024, 1024), 8, "ortho"
    spec = oracle.NufftSpec(im)
    om, omd = _traj(4, 2048)
    M = om.shape[1]
    fwd, adj = _nufft_ops(im, fused=True)
    h = fwd._plan.handle(torch.device(DEV))
    cb = _binned_chunk(h, coils, M)
    B = cb + 1
    ch = _chunks(B, cb)
    e = _edges(ch)
    last = (ch[-1][1] - ch[-1][0]) * coils
    S = _rand(((B if sb == "B" else 1), coils) + im, 60)
    x, y, g = _rand((B, 1) + im, 61), _rand((B, coils, M), 62), _rand((B, 1) + im, 63)
    w = torch.linspace(0.5, 1.5, M, device=DEV)
    xs, ys, gsp = _split(x), _split(y), _split(g)

    got = fwd(xs, omd, smaps=S, norm=norm, split=True)
    assert "fz_rows_fwd_kernel" in _lib.last_kernel("nufft_fwd") and _last_count("nufft_fwd") == last
    assert torch.equal(_cat(fwd(xs[b0:b1], omd, smaps=_bs(S, b0, b1), norm=norm, split=True) for b0, b1 in ch), got)
    assert rel_l2(_unsplit(got[e]), oracle.nufft_forward(_at(x, e), om, spec, smaps=_at(S, e), norm=norm)) <= TOL

    Sg = S.clone().requires_grad_(True)
    got = adj(ys, omd, smaps=Sg, norm=norm, split=True, kweight=w)
    assert "fz_rows_adj_kernel" in _lib.last_kernel("nufft_adj") and _last_count("nufft_adj") == last
    assert torch.equal(_cat(adj(ys[b0:b1], omd, smaps=_bs(S, b0, b1), norm=norm, split=True, kweight=w) for b0, b1 in ch),
                       got)
    yw = _at(y, e) * w.cpu().double()
    assert rel_l2(_unsplit(got[e]), oracle.nufft_adjoint(yw, om, spec, smaps=_at(S, e), norm=norm)) <= TOL

    rec = _backward(got, gsp, Sg)                       # gS_c = sum_b A^H(w y[b, c]) conj(g_b)
    assert "fz_rows_adj_kernel" in rec and _count(rec) == last
    gs = torch.empty_like(S)
    for b0, b1 in ch:
        adj._plan.smaps_grad(ys[b0:b1], omd, gsp[b0:b1], _bs(gs, b0, b1), norm, split=True, kweight=w,
                             accumulate=sb == 1 and b0 > 0)
    assert torch.equal(gs, Sg.grad)
    if sb == 1:
        per = torch.empty((B, coils) + im, dtype=torch.complex64, device=DEV)
        for b in range(B):
            adj._plan.smaps_grad(ys[b:b + 1], omd, gsp[b:b + 1], per[b:b + 1], norm, split=True, kweight=w)
        assert rel_l2(Sg.grad, per.cpu().to(torch.complex128).sum(0, keepdim=True)) <= 1e-6
    else:
        want = oracle.nufft_adjoint(yw, om, spec, norm=norm) * _at(g, e).conj()
        assert rel_l2(Sg.grad[e], want) <= TOL


# ----------------------------------------------------------------------------- Toeplitz apply and map gradient
def _abi_toep_apply(h, x, k, S, B, coils, conj, cb):
    L = _lib.lib()
    buf, out = _nan_out(tuple(x.shape))
    _abi(lambda ws, n: L.pdu_toep_apply_c64(h, x.data_ptr(), out.data_ptr(), k.data_ptr(), k.shape[0],
                                            S.data_ptr() if S is not None else None, B, coils,
                                            S.shape[0] if S is not None else 1, conj, ws, n, _lib.stream_ptr()),
         L.pdu_toep_workspace_bytes(h, min(cb, B) * coils))
    assert _written(buf, out)
    return out


def _abi_toep_smaps_grad(h, x, g, k, S, B, coils, cb, accumulate=None):
    L = _lib.lib()
    buf, gs = _nan_out(tuple(S.shape))
    if accumulate is not None:
        gs.copy_(accumulate)
    _abi(lambda ws, n: L.pdu_toep_smaps_grad_c64(h, x.data_ptr(), g.data_ptr(), gs.data_ptr(), k.data_ptr(), k.shape[0],
                                                 S.data_ptr(), B, coils, S.shape[0], 0, 1.0,
                                                 0 if accumulate is None else 1, ws, n, _lib.stream_ptr()),
         L.pdu_toep_workspace_bytes(h, min(cb, B) * coils))
    assert _written(buf, gs)
    return gs


def _toep_smaps_grad_ref(x, g, k, S):
    """sum over the batch (shared map) or per element: T(S_c x_b) conj(g_b) + T^H(S_c g_b) conj(x_b), float64."""
    t = toep_apply(S * x, k) * g.conj() + toep_apply(S * g, k.conj()) * x.conj()
    return t.sum(0, keepdim=True) if S.shape[0] == 1 else t


# (im, coils, smaps batch (None: no maps), fast path); the batch is derived from the chunk
TOEP_CASES = [((1024, 1024), 8, "B", True), ((8, 8), 1, None, False), ((8, 8), 3, 1, False)]


@pytest.mark.parametrize("im,coils,sb,fast", TOEP_CASES)
def test_toep_chunks(im, coils, sb, fast):
    """ToepNufft forward, backward (conjugate kernel) and map gradient with one kernel per batch element: 32 planes of
    the 1024^2 fast path per chunk, and the 65535-plane cap of the 8 x 8 generic path (21845 batch elements with 3
    coils)."""
    tp = nufft_mod._toep_plan(im)
    h = tp.handle(torch.device(DEV))
    cb = _toep_chunk(h, coils)
    B = cb + max(1, cb // 10)
    ch = _chunks(B, cb)
    e = _edges(ch)
    N0, N1 = im
    k = _rand((B, 2 * N0, 2 * N1), 70)                 # non-Hermitian: T^H differs from T
    S = None if sb is None else _rand(((B if sb == "B" else 1), coils) + im, 71)
    C = 1 if S is not None else coils
    x, g = _rand((B, C) + im, 72), _rand((B, C) + im, 73)

    got = _abi_toep_apply(h, x, k, S, B, coils, 0, cb)
    assert _last_count("toep") == (ch[-1][1] - ch[-1][0]) * coils
    assert ("fast path" if fast else "generic path") in _lib.last_kernel("toep")
    back = _abi_toep_apply(h, g, k, S, B, coils, 1, cb)
    op = pdu.ToepNufft()

    def run(b0, b1):
        xr = x[b0:b1].clone().requires_grad_(True)
        Sr = None if S is None else _bs(S, b0, b1).clone().requires_grad_(sb == "B")
        out = op(xr, k[b0:b1], smaps=Sr)
        out.backward(g[b0:b1])
        return out, xr.grad, (Sr.grad if sb == "B" else None)

    full = run(0, B)
    parts = [run(b0, b1) for b0, b1 in ch]
    assert torch.equal(full[0], got) and torch.equal(full[1], back)
    assert torch.equal(_cat(p[0] for p in parts), got) and torch.equal(_cat(p[1] for p in parts), back)
    kd = _at(k, e)
    assert rel_l2(got[e], toep_apply(_at(x, e), kd, _at(S, e))) <= TOL
    assert rel_l2(back[e], toep_apply(_at(g, e), kd.conj(), _at(S, e))) <= TOL
    if S is None:
        return

    gs = _abi_toep_smaps_grad(h, x, g, k, S, B, coils, cb)
    assert _last_count("smaps_grad") == (ch[-1][1] - ch[-1][0]) * coils
    if sb == "B":
        assert torch.equal(full[2], gs) and torch.equal(_cat(p[2] for p in parts), gs)
        assert rel_l2(gs[e], _toep_smaps_grad_ref(_at(x, e), _at(g, e), kd, _at(S, e))) <= TOL
    else:
        # a shared map: the chunked sum equals chunk 0 followed by chunk 1 with accumulate
        part = None
        for b0, b1 in ch:
            part = _abi_toep_smaps_grad(h, x[b0:b1], g[b0:b1], k[b0:b1], S, b1 - b0, coils, cb, accumulate=part)
        assert torch.equal(part, gs)
        Sr = S.clone().requires_grad_(True)
        op(x, k, smaps=Sr).backward(g)
        assert torch.equal(Sr.grad, gs)
        all_ = list(range(B))
        assert rel_l2(gs, _toep_smaps_grad_ref(_at(x, all_), _at(g, all_), _at(k, all_), _at(S, all_))) <= TOL


# ----------------------------------------------------------------------------- toep_cg
@pytest.mark.parametrize("im,coils,sb,fast", TOEP_CASES)
def test_toep_cg_chunks(im, coils, sb, fast):
    """toep_cg with one kernel, one lam and one warm start per batch element: a system of the chunked call is
    bit-identical to toep_cg on that system alone, on both sides of every chunk boundary."""
    tp = nufft_mod._toep_plan(im)
    h = tp.handle(torch.device(DEV))
    cb = _toep_chunk(h, coils)
    B = cb + max(1, cb // 10)
    ch = _chunks(B, cb)
    e = _edges(ch)
    N0, N1 = im
    iters = 3
    # a real positive kernel: T is Hermitian positive semi-definite and every system runs all iterations
    k = (1.0 + torch.rand((B, 2 * N0, 2 * N1), device=DEV, generator=torch.Generator(device=DEV).manual_seed(80))).to(
        torch.complex64)
    S = None if sb is None else _rand(((B if sb == "B" else 1), coils) + im, 81)
    if S is not None:
        S = S / (S.abs() ** 2).sum(1, keepdim=True).sqrt()
    C = 1 if S is not None else coils
    b, x0 = _rand((B, C) + im, 82), _rand((B, C) + im, 83)
    lam = 0.1 + torch.arange(B, device=DEV, dtype=torch.float32) % 7 * 0.05
    L = _lib.lib()
    buf, x = _nan_out(tuple(b.shape))
    _abi(lambda ws, n: L.pdu_toep_cg_c64(h, b.data_ptr(), x0.data_ptr(), x.data_ptr(), k.data_ptr(), B,
                                         S.data_ptr() if S is not None else None, B, coils,
                                         S.shape[0] if S is not None else 1, lam.data_ptr(), B, iters, 0.0, 0, ws, n,
                                         _lib.stream_ptr()),
         L.pdu_toep_cg_workspace_bytes(h, B, coils, 1 if S is not None else 0), PDU_EINVAL)
    assert _written(buf, x)
    assert _last_count("cg") == (ch[-1][1] - ch[-1][0]) * (1 if S is not None else coils)
    assert ("fast path" if fast else "generic path") in _lib.last_kernel("cg")
    assert torch.equal(pdu.toep_cg(b, k, smaps=S, lam=lam, x0=x0, max_iter=iters), x)
    for i in e:
        xi = pdu.toep_cg(b[i:i + 1], k[i:i + 1], smaps=_bs(S, i, i + 1), lam=lam[i:i + 1], x0=x0[i:i + 1], max_iter=iters)
        assert torch.equal(xi, x[i:i + 1]), i
    i = ch[1][0]                                        # the first system of the second chunk
    want = cg_ref(_at(b, [i]), _at(k, [i]), smaps=_at(S, [i]), lam=[float(lam[i])], x0=_at(x0, [i]), max_iter=iters)
    assert rel_l2(x[i:i + 1], want) <= TOL
