"""The float64 coil-map gradients the GPU tests compare against: autograd through the complex128 oracle operators
(oracle.nufft_forward / nufft_adjoint, tests/oracle_toep.toep_apply, tests/oracle_cg.dense_operator), pinned to central
finite differences of a real loss along random map directions, and to the closed forms the library implements
(sum over b of P[b, c] conj(Q[b]), DESIGN.md section 3.4)."""
import numpy as np
import pytest
import torch

import oracle
from oracle_cg import dense_operator
from oracle_toep import toep_apply, toeplitz_kernel
from util import rel_l2, seeded

IM = (12, 12)
SPEC = oracle.NufftSpec(IM)
OM = oracle.radial_trajectory(5, 24)
M = OM.shape[1]


def _c128(shape, seed):
    return seeded(shape, seed, complex_=True).to(torch.complex128)


def _re_dot(a, b):
    return float((a.conj() * b).real.sum())


def _fd_check(loss, S, gS, seed, h=1e-4):
    """Re<gS, D> against (L(S + h D) - L(S - h D)) / 2h for two random directions D."""
    for k in range(2):
        D = _c128(S.shape, seed + k)
        fd = (loss(S + h * D) - loss(S - h * D)) / (2 * h)
        an = _re_dot(gS, D)
        assert abs(fd - an) <= 1e-7 * max(abs(an), 1e-30), (fd, an)


def _grad(fn, S, G):
    S = S.clone().requires_grad_(True)
    (g,) = torch.autograd.grad(fn(S), S, G)
    return g


@pytest.mark.parametrize("sb,norm", [(1, None), (2, "ortho")])
def test_kbnufft_smaps_gradient(sb, norm):
    x, S = _c128((2, 1) + IM, 1), _c128((sb, 3) + IM, 2)
    G = _c128((2, 3, M), 3)
    fwd = lambda s: oracle.nufft_forward(x, OM, SPEC, smaps=s, norm=norm)       # noqa: E731
    gS = _grad(fwd, S, G)
    _fd_check(lambda s: _re_dot(G, fwd(s)), S, gS, 10)
    # closed form: P[b, c] = A^H(g[b, c]) un-combined, Q[b] = x_b
    P = oracle.nufft_adjoint(G, OM, SPEC, norm=norm)
    want = (P * x.conj()).sum(0, keepdim=True) if sb == 1 else P * x.conj()
    assert rel_l2(gS, want) <= 1e-12


@pytest.mark.parametrize("sb,norm", [(1, "ortho"), (2, None)])
def test_kbnufft_adjoint_smaps_gradient(sb, norm):
    y, S = _c128((2, 3, M), 4), _c128((sb, 3) + IM, 5)
    w = torch.linspace(0.5, 1.5, M, dtype=torch.float64)
    G = _c128((2, 1) + IM, 6)
    adj = lambda s: oracle.nufft_adjoint(y * w, OM, SPEC, smaps=s, norm=norm)    # noqa: E731
    gS = _grad(adj, S, G)
    _fd_check(lambda s: _re_dot(G, adj(s)), S, gS, 20)
    P = oracle.nufft_adjoint(y * w, OM, SPEC, norm=norm)         # A^H(w y[b, c]), Q[b] = g_b
    want = (P * G.conj()).sum(0, keepdim=True) if sb == 1 else P * G.conj()
    assert rel_l2(gS, want) <= 1e-12


@pytest.mark.parametrize("sb", [1, 2])
def test_toep_smaps_gradient(sb):
    k = _c128((2 * IM[0], 2 * IM[1]), 7)                       # non-Hermitian: T^H differs from T
    x, S, G = _c128((2, 1) + IM, 8), _c128((sb, 3) + IM, 9), _c128((2, 1) + IM, 10)
    app = lambda s: toep_apply(x, k, s)                          # noqa: E731
    gS = _grad(app, S, G)
    _fd_check(lambda s: _re_dot(G, app(s)), S, gS, 30)
    # sum_b T(S_c x_b) conj(g_b) + T^H(S_c g_b) conj(x_b)
    terms = toep_apply(x * S, k) * G.conj() + toep_apply(G * S, k.conj()) * x.conj()
    want = terms.sum(0, keepdim=True) if sb == 1 else terms
    assert rel_l2(gS, want) <= 1e-12


def test_toep_cg_smaps_gradient_pinned_to_the_dense_solve():
    om = oracle.radial_trajectory(5, 24)
    w = (0.5 + torch.rand(om.shape[1], generator=torch.Generator().manual_seed(5), dtype=torch.float64)).numpy()
    k = toeplitz_kernel(om, SPEC, weights=w, exact=True)
    lam = 0.1 * float(k.abs().max())
    S, b, G = _c128((1, 3) + IM, 11), _c128((1, 1) + IM, 12), _c128((1, 1) + IM, 13)
    n = IM[0] * IM[1]
    T = torch.from_numpy(dense_operator(k, (1, 1) + IM))          # no maps: the plain T on one plane

    def solve_t(s):                                                # torch: differentiable in s
        sv = s.reshape(3, n)
        Mm = sum(torch.diag(sv[c].conj()) @ T @ torch.diag(sv[c]) for c in range(3)) + lam * torch.eye(n, dtype=T.dtype)
        return torch.linalg.solve(Mm, b.reshape(n)).reshape(b.shape)

    def solve_np(s):                                               # numpy, from the oracle's dense operator
        Mm = dense_operator(k, (1, 1) + IM, smaps=s, lam=lam)
        return torch.from_numpy(np.linalg.solve(Mm, b.reshape(-1).numpy())).reshape(b.shape)

    assert rel_l2(solve_t(S), solve_np(S)) <= 1e-10
    gS = _grad(solve_t, S, G)
    _fd_check(lambda s: _re_dot(G, solve_np(s)), S, gS, 40)
    # the library's form: -G(x, v), v = M^-H g, G the ToepNufft map gradient
    x = solve_np(S)
    v = torch.from_numpy(np.linalg.solve(dense_operator(k, (1, 1) + IM, smaps=S, lam=lam).conj().T, G.reshape(-1).numpy()))
    v = v.reshape(G.shape)
    want = -(toep_apply(x * S, k) * v.conj() + toep_apply(v * S, k.conj()) * x.conj())
    assert rel_l2(gS, want) <= 1e-9
