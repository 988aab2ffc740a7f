"""Distribution of the device-RNG (Philox) GCR draws at multi-block shapes (VERDICT r1, parity item 1a).

With the spectrum held fixed, every `eng.gcr()` call draws a new constrained realisation x_t = [s_t ; f_t] for every
time of every chain.  Its distribution is Gaussian with

    Sigma = (diag(S^-1, 0) + [I|F]^H N^-1 [I|F])^-1,      E[x_t] = Sigma [I|F]^H N^-1 (w d_t)

(the reference's GCR, pspec.py:151-235, draws exactly this through omega_a / omega_b).  The tests pool >= 4000 draws:
the sample covariance must equal Sigma within Monte-Carlo error -- which exercises the Philox counter layout over block
rows / time tiles / chains of k_solve3, of the dense-product solve (k_add_noise) and of the per-time kernel -- and the
cross-time, cross-chain and cross-draw covariances must vanish (a wrong counter mapping gives correlated xi).  GPU only.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import hydra_oracle as ho  # noqa: E402  (checker only)


def crandn(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def posterior(ps, flags, F, ninv_diag):
    """Sigma and the map  d -> E[x]  of the GCR distribution for one flag vector."""
    n, m = F.shape
    fop = ho.fourier_operator(n)
    S = ho.covariance_from_pspec(ps / n ** 2, fop)
    P = np.concatenate([np.eye(n), F], axis=1)
    Ni = np.diag(flags.astype(float) * ninv_diag)
    prec = P.conj().T @ Ni @ P
    prec[:n, :n] += np.linalg.inv(S)
    Sigma = np.linalg.inv(prec)
    return Sigma, Sigma @ P.conj().T @ Ni


def nrm(C, Sigma):
    d = np.sqrt(np.real(np.diagonal(Sigma)))
    return np.max(np.abs(C) / np.outer(d, d))


@pytest.mark.parametrize("variant", ["solve3", "dense_solve", "time_flags", "time_flags_direct"])
def test_philox_gcr_covariance_multiblock(variant):
    from hydra_pspec_b200 import pspec
    nt, nf, nm, nch, ndraw = 48, 96, 8, 4, 4000          # N = 104: 4 block rows; 3 time tiles; 4 chains
    rng = np.random.default_rng(2024)
    F = np.linalg.qr(crandn(rng, nf, nm))[0]
    ps = nf * (0.5 + 2.0 * rng.random(nf))                # fixed spectrum: lam^2 = ps / nf in [0.5, 2.5]
    ninv_diag = 1.0 + rng.random(nf)
    vis = crandn(rng, nch, nt, nf) + (3 * crandn(rng, nch, nt, nm)) @ F.T
    per_time = variant.startswith("time_flags")
    if per_time:
        masks = np.ones((2, nf), dtype=bool)
        masks[0, [5, 40, 41]] = False
        masks[1, [17, 66]] = False
        flags = masks[np.arange(nt) % 2]                   # two masks alternating in time: no factor re-use
    else:
        masks = np.ones((1, nf), dtype=bool)
        masks[0, [5, 40, 41, 77]] = False
        flags = masks[0]
    # per-time flags: the low-rank form (k_solve3 + k_pt_lowrank with its own zeta draws; default) and, with
    # force_dense_solve, one factorisation per time (k_pt_cholsolve)
    eng = pspec.GibbsEngine(nch, nt, nf, nm, max_iters=1, rng="philox", refresh_omega=True, keep=(), seed=99,
                            time_flags=per_time, force_dense_solve=variant in ("dense_solve", "time_flags_direct"))
    for c in range(nch):
        eng.load_chain(c, vis[c] * flags, flags, F, ninv_diag, ps / nf)
    post = [posterior(ps, mk, F, ninv_diag) for mk in masks]
    tmask = (np.arange(nt) % 2) if per_time else np.zeros(nt, dtype=int)
    mean = np.empty((nch, nt, nf + nm), dtype=complex)
    for c in range(nch):
        for t in range(nt):
            mean[c, t] = post[tmask[t]][1] @ (vis[c, t] * masks[tmask[t]])
    N = nf + nm
    C0 = [np.zeros((N, N), dtype=complex) for _ in masks]  # same (draw, chain, time)
    Ct1 = np.zeros((N, N), dtype=complex)                  # time t vs t + 2 (same mask; neighbours in a tile)
    Ct16 = np.zeros((N, N), dtype=complex)                 # time t vs t + 16 (next tile)
    Cch = np.zeros((N, N), dtype=complex)                  # chain c vs c + 1
    Cit = np.zeros((N, N), dtype=complex)                  # draw k vs k + 1
    prev = None
    for k in range(ndraw):
        eng.gcr()
        E = np.stack([eng.last_gcr(c) for c in range(nch)]) - mean       # (nch, nt, N)
        for im in range(len(masks)):
            e2 = E[:, tmask == im].reshape(-1, N)
            C0[im] += e2.T @ e2.conj()
        Ct1 += E[:, :-2].reshape(-1, N).T @ E[:, 2:].reshape(-1, N).conj()
        Ct16 += E[:, :-16].reshape(-1, N).T @ E[:, 16:].reshape(-1, N).conj()
        Cch += E[:-1].reshape(-1, N).T @ E[1:].reshape(-1, N).conj()
        if prev is not None:
            Cit += prev.reshape(-1, N).T @ E.reshape(-1, N).conj()
        prev = E
    eng.close()
    Sig = post[0][0]
    for im in range(len(masks)):
        ns = ndraw * nch * int(np.sum(tmask == im))
        err = nrm(C0[im] / ns - post[im][0], post[im][0])
        assert err < 6.0 / np.sqrt(ns), (variant, im, err, 6.0 / np.sqrt(ns))
    for name, C, ns in (("time+2", Ct1, ndraw * nch * (nt - 2)), ("time+16", Ct16, ndraw * nch * (nt - 16)),
                        ("chain", Cch, ndraw * (nch - 1) * nt), ("draw", Cit, (ndraw - 1) * nch * nt)):
        err = nrm(C / ns, Sig)
        assert err < 6.0 / np.sqrt(ns), (variant, name, err, 6.0 / np.sqrt(ns))
