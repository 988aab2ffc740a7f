"""Single-kernel checks through the C ABI test hooks, against numpy.  GPU only."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _lib():
    from hydra_pspec_b200 import _lib
    return _lib


def crandn(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def rel(a, b):
    return np.max(np.abs(a - b)) / np.max(np.abs(b))


@pytest.mark.parametrize("M,N,K", [(64, 64, 16), (70, 45, 33), (7, 130, 5), (200, 136, 120)])
@pytest.mark.parametrize("tA,cA,tB,cB", [(0, 0, 0, 0), (1, 1, 0, 0), (0, 0, 1, 1), (1, 0, 1, 1)])
def test_zgemm(M, N, K, tA, cA, tB, cB):
    L = _lib()
    rng = np.random.default_rng(M * 1000 + N + K)
    A = crandn(rng, M, K)
    B = crandn(rng, K, N)
    dk = rng.random(K) + 0.5
    want = (A * dk[None, :]) @ B
    As = A.T if tA else A
    Bs = B.T if tB else B
    As = np.ascontiguousarray(As.conj() if cA else As)
    Bs = np.ascontiguousarray(Bs.conj() if cB else Bs)
    C = np.empty((M, N), dtype=np.complex128)
    L.check(L.lib().hp_test_zgemm(M, N, K, L.ptr(As), tA, cA, L.ptr(Bs), tB, cB, L.ptr(dk), L.ptr(C)))
    assert rel(C, want) < 1e-14


def test_fourier_operator_matches_reference_definition():
    from hydra_pspec_b200 import utils
    for n in (4, 5, 120, 384):
        i = np.arange(n) - n // 2
        want = np.exp(-2 * np.pi * 1j * (i.reshape(-1, 1) * i.reshape(1, -1) / n))  # utils.py:36-38
        got = utils.fourier_operator(n)
        assert np.max(np.abs(got - want)) < 5e-13  # the reference's own argument is only good to ~n*eps


@pytest.mark.parametrize("n,m,T", [(32, 0, 16), (20, 4, 5), (64, 8, 33), (120, 12, 24), (384, 32, 48),
                                   (500, 44, 20)])   # Np = 544: k_solve takes the resident systems k_solve3 cannot
def test_chol_solve(n, m, T):
    L = _lib()
    rng = np.random.default_rng(n + m + T)
    N = n + m
    Bm = crandn(rng, n + 8, N)
    G = Bm.conj().T @ Bm / (n + 8)
    G = (G + G.conj().T) / 2
    lam = np.concatenate([0.3 + rng.random(n), np.ones(m)])
    J = np.concatenate([np.ones(n), np.zeros(m)])
    Mmat = np.diag(J) + lam[:, None] * G * lam[None, :]
    Rfix = crandn(rng, T, N)
    wa = crandn(rng, T, n)
    R = Rfix * lam[None, :]
    R[:, :n] += wa
    Xw = np.linalg.solve(Mmat, R.T).T
    Lw = np.linalg.cholesky(Mmat)
    Ld = np.empty((N, N), dtype=np.complex128)
    X = np.empty((T, N), dtype=np.complex128)
    info = np.zeros(1, dtype=np.int32)
    G = np.ascontiguousarray(G)
    L.check(L.lib().hp_test_chol_solve(n, m, T, L.ptr(G), L.ptr(lam), L.ptr(Rfix), L.ptr(wa), 0, L.ptr(Ld), L.ptr(X),
                                       L.ptr(info)))
    assert info[0] == 0
    assert rel(Ld, Lw) < 1e-12
    assert rel(X, Xw) < 1e-11


def test_chol_reports_indefinite():
    L = _lib()
    m, T = 0, 4
    for n in (40, 20):   # two block columns; one block (the factorisation is k_chol_w's first launch only)
        G = -2.0 * np.eye(n, dtype=np.complex128)  # M = I - 2 I is negative definite
        lam = np.ones(n)
        Rfix = np.zeros((T, n), dtype=np.complex128)
        X = np.empty((T, n), dtype=np.complex128)
        info = np.zeros(1, dtype=np.int32)
        L.check(L.lib().hp_test_chol_solve(n, m, T, L.ptr(G), L.ptr(lam), L.ptr(Rfix), None, 0, None, L.ptr(X), L.ptr(info)))
        assert info[0] != 0, n


def test_arena_cache_and_deferred_setup_survive_engine_churn():
    """Engines of different sizes created and destroyed back to back (the drop-in functions do this once per
    baseline): the cached device arena must be reused / replaced correctly and results must not depend on it."""
    import os
    from hydra_pspec_b200 import _lib, pspec
    rng = np.random.default_rng(0)

    def run(nt, nf, nm, nch):
        F = np.linalg.qr(rng.standard_normal((nf, nm)) + 1j * rng.standard_normal((nf, nm)))[0]
        vis = rng.standard_normal((nt, nf)) + 1j * rng.standard_normal((nt, nf))
        eng = pspec.GibbsEngine(nch, nt, nf, nm, max_iters=3, rng="philox", keep=(), seed=5)
        for c in range(nch):
            eng.load_chain(c, vis * (c + 1), np.ones(nf, bool), F, np.ones(nf), np.ones(nf))
        eng.run(3)
        out = np.stack([eng.signal_ps(c) for c in range(nch)])
        eng.close()
        return vis, F, out

    np.random.seed(0)
    sizes = [(16, 32, 2, 3), (40, 96, 6, 5), (8, 16, 1, 1), (40, 96, 6, 5)]
    outs = []
    for s in sizes:
        rng = np.random.default_rng(sum(s))
        outs.append(run(*s)[2])
    assert np.array_equal(outs[1], outs[3])          # same problem, arena reused after a smaller engine
    _lib.lib().hp_release_cached_memory()
    rng = np.random.default_rng(sum(sizes[1]))
    assert np.array_equal(run(*sizes[1])[2], outs[1])  # and after the cache has been dropped
    assert all(np.all(np.isfinite(o)) for o in outs)


def test_two_devices_in_one_process():
    """The drop-in functions take `device=`: kernels with > 48 KB of dynamic shared memory need their attribute set on
    every device they run on (the launch wrappers cache it per device)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from hydra_pspec_b200 import pspec
    rng = np.random.default_rng(3)
    nt, nf, nm = 24, 96, 6
    F = np.linalg.qr(rng.standard_normal((nf, nm)) + 1j * rng.standard_normal((nf, nm)))[0]
    vis = rng.standard_normal((nt, nf)) + 1j * rng.standard_normal((nt, nf))
    flags = np.ones(nf, bool)
    flags[[5, 50]] = False
    prior = np.zeros((2, nf))
    a = pspec.gibbs_sample_with_fg(vis, flags, np.eye(nf), F, np.eye(nf) * 2.0, prior, Niter=3, seed=4, verbose=False, device=0)
    b = pspec.gibbs_sample_with_fg(vis, flags, np.eye(nf), F, np.eye(nf) * 2.0, prior, Niter=3, seed=4, verbose=False, device=1)
    fl2 = np.broadcast_to(flags, (nt, nf)).copy()
    fl2[3, 7] = False
    c = pspec.gibbs_sample_with_fg(vis, fl2, np.eye(nf), F, np.eye(nf) * 2.0, prior, Niter=2, seed=4, verbose=False, device=1)
    for x, y in zip(a[:6], b[:6]):
        assert np.array_equal(x, y)
    assert np.all(np.isfinite(c[2]))


@pytest.mark.parametrize("n,m,T,nsys,grid,use_wa,cg", [
    (32, 0, 16, 1, 0, False, 0),      # one block, one tile
    (20, 4, 5, 2, 1, True, 0),        # padded rows and times, two tiles on one persistent CTA
    (64, 8, 33, 3, 2, False, 0),      # 3 block rows, 9 tiles on 2 CTAs (mbarrier phases wrap)
    (120, 12, 24, 2, 1, True, 1),     # cg_compat through k_cg_scale
    (96, 8, 48, 4, 3, False, 0),      # 4 block rows, uneven tile split
    (384, 32, 48, 2, 4, False, 0),    # the headline system: 13 block rows
    (384, 32, 40, 1, 0, True, 1),
    (416, 32, 20, 1, 0, False, 0),    # Np = 448: the largest system k_solve3 takes (28 strips)
    (416, 32, 17, 2, 3, True, 1),     # Np = 448 with wa and cg_compat; the second tile holds one time
    (256, 16, 20, 2, 0, True, 0),     # N = 272: the trailing strip of pure padding is left out (272 rows in 288)
    (40, 0, 64, 5, 7, False, 0),      # no foreground modes; 20 tiles on 7 CTAs
    (200, 24, 48, 2, 5, False, 1),    # cg_compat with unscaled right-hand sides (Wf1 = W diag(lam))
    (300, 20, 16, 3, 1, True, 0),     # N = 320, whole blocks; three tiles on one CTA
    (64, 8, 1, 1, 0, False, 0),       # one time, 15 padded columns
    (352, 32, 40, 2, 2, False, 0),    # 12 block rows, 6 tiles on 2 CTAs
    (24, 8, 7, 3, 2, True, 0),        # one block, 3 partly filled tiles on 2 CTAs
    (180, 12, 64, 1, 3, True, 0),     # N = 192, 4 tiles on 3 CTAs
])
def test_solve3(n, m, T, nsys, grid, use_wa, cg):
    """k_solve3 (persistent solve, hp_solve3.cu) against numpy: X, and the sum_t |x|^2 sums."""
    from oracle import hydra_oracle as ho  # checker only
    L = _lib()
    rng = np.random.default_rng(7 * n + m + T + nsys)
    N = n + m
    Bm = crandn(rng, n + 8, N)
    G = Bm.conj().T @ Bm / (n + 8)
    G = np.ascontiguousarray((G + G.conj().T) / 2)
    lam = np.concatenate([0.3 + rng.random(n), np.ones(m)])
    J = np.concatenate([np.ones(n), np.zeros(m)])
    Mmat = np.diag(J) + lam[:, None] * G * lam[None, :]
    Rfix = crandn(rng, nsys, T, N)
    wa = crandn(rng, nsys, T, n) if use_wa else None
    R = Rfix * lam[None, None, :]
    if use_wa:
        R[:, :, :n] += wa
    Xw = np.linalg.solve(Mmat, R.reshape(-1, N).T).T.reshape(nsys, T, N)
    if cg:
        wgt = np.concatenate([lam[:n] ** 2, np.ones(m)])
        for s in range(nsys):
            for t in range(T):
                c = np.sum(wgt * R[s, t].conj() * Xw[s, t])
                b = np.sqrt(np.sum(wgt * np.abs(R[s, t]) ** 2))
                Xw[s, t] *= ho.cg_theta(c, b)
    X = np.empty((nsys, T, N), dtype=np.complex128)
    psum = np.empty((nsys, n))
    L.check(L.lib().hp_test_solve3(n, m, T, nsys, L.ptr(G), L.ptr(lam), L.ptr(np.ascontiguousarray(Rfix)),
                                   L.ptr(None if wa is None else np.ascontiguousarray(wa)), cg, grid, L.ptr(X), L.ptr(psum)))
    assert rel(X, Xw) < 1e-11
    if not cg:  # (with cg_compat the engine recomputes the sums after the scaling)
        assert rel(psum, np.sum(np.abs(Xw[:, :, :n]) ** 2, axis=1)) < 1e-11


@pytest.mark.parametrize("n,batch", [(5, 2), (33, 3), (120, 2), (384, 3)])
def test_device_eigh_batch(n, batch):
    """hp_eigh_batch (one-sided Jacobi, csrc/hp_eigh.cu) against numpy.linalg.eigh: eigenvalues, unitarity, reconstruction;
    a rank-deficient and a slightly indefinite matrix in the batch (signed Rayleigh quotients)."""
    from hydra_pspec_b200 import pspec
    rng = np.random.default_rng(10 * n + batch)
    mats = []
    for b in range(batch):
        X = crandn(rng, n, n if b != 1 else max(1, n // 2))          # b == 1: rank n / 2
        S = X @ X.conj().T * 10.0 ** rng.uniform(-3, 3)
        if b == 0:
            S = S - 1e-9 * np.trace(S).real / n * np.eye(n) * (n > 5)   # eigenvalues down to slightly negative values
        mats.append(0.5 * (S + S.conj().T))
    mats = np.stack(mats)
    w, V = pspec.device_eigh(mats)
    for b in range(batch):
        scale = np.abs(np.linalg.eigvalsh(mats[b])).max()
        assert np.max(np.abs(V[b].conj().T @ V[b] - np.eye(n))) < 1e-12
        assert np.max(np.abs((V[b] * w[b]) @ V[b].conj().T - mats[b])) < 1e-11 * scale
        assert np.max(np.abs(np.sort(w[b]) - np.linalg.eigvalsh(mats[b]))) < 1e-11 * scale
