"""The dense-product GCR solve taken when Nfreqs + Nmodes exceeds k_solve's shared-memory resident
tile (BASELINE.json configs[4]: Nfreq=1024, Nfg=64, non-diagonal noise covariance).  GPU only."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import hydra_oracle as ho  # noqa: E402  (checker only)

TOL = 1e-10
KEYS = ["signal_cr", "signal_S", "signal_ps", "fg_amps", "chisq", "ln_post"]


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    return np.max(np.abs(a - b)) / np.max(np.abs(b))


def crandn(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def make_case(nt, nf, nm, nflag, seed, dense_noise):
    rng = np.random.default_rng(seed)
    F = np.linalg.qr(crandn(rng, nf, nm))[0]
    fop = ho.fourier_operator(nf)
    S0 = fop.conj().T @ np.diag((0.5 + rng.random(nf)) / nf ** 2) @ fop
    if dense_noise:
        # calc-vis-cov-matrices.py form: a sample covariance of noise-like visibilities, plus a white floor
        Xn = crandn(rng, nf, 2 * nf) * (0.3 + rng.random(nf))[:, None]
        Ncov = Xn @ Xn.conj().T / (2 * nf) + 0.05 * np.eye(nf)
        noise = crandn(rng, nt, nf) @ np.linalg.cholesky(Ncov).T
    else:
        sig = 0.3 + rng.random(nf)
        Ncov = np.diag(sig ** 2)
        noise = crandn(rng, nt, nf) * sig
    vis = noise + (5 * crandn(rng, nt, nm)) @ F.T + crandn(rng, nt, nf) @ np.linalg.cholesky(S0 + 1e-13 * np.eye(nf)).T
    flags = np.ones(nf, dtype=bool)
    flags[rng.choice(nf, nflag, replace=False)] = False
    prior = np.zeros((2, nf))
    prior[0, nf // 2 - 1:nf // 2 + 2] = 50.0
    prior[1, nf // 2 - 1:nf // 2 + 2] = 0.05
    return vis, flags, S0, F, np.linalg.inv(Ncov), prior


@pytest.mark.parametrize("dense_noise", [False, True])
@pytest.mark.parametrize("nt,nf,nm,nflag,seed", [(16, 32, 4, 0, 1), (21, 45, 5, 3, 2), (40, 120, 12, 5, 3), (9, 37, 3, 1, 5)])
def test_dense_product_solve_matches_oracle(nt, nf, nm, nflag, seed, dense_noise, monkeypatch):
    """The large-N path forced at sizes the oracle finishes quickly."""
    from hydra_pspec_b200 import pspec
    monkeypatch.setattr(pspec, "_FORCE_DENSE_SOLVE", True)
    vis, flags, S0, F, Ninv, prior = make_case(nt, nf, nm, nflag, seed, dense_noise)
    want = ho.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=3, seed=seed, solver="direct", symmetric_flags=True)
    got = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=3, seed=seed, verbose=False, solver="exact")
    for o, w, k in zip(got[:6], want, KEYS):
        assert rel(o, w) < TOL, k


def test_stress_shape_1024_64_dense_noise_matches_oracle():
    """configs[4] system size (N = 1088 > 576: no forcing needed), six times, one iteration."""
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, Ninv, prior = make_case(6, 1024, 64, 7, 77, True)  # 6 times: two k_post_fft<4> tiles, one partial
    want = ho.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=1, seed=3, solver="direct", symmetric_flags=True)
    got = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=1, seed=3, verbose=False, solver="exact")
    for o, w, k in zip(got[:6], want, KEYS):
        assert rel(o, w) < 1e-9, k


def test_large_n_philox_chain_and_reference_cg():
    """N = 656 > 576 (dense-product solve): a Philox chain runs, and the drop-in default (numpy draws + the scalar model
    of the reference's truncated CG, k_cg_scale) matches the oracle's theta-scaled solves (pspec.py:228)."""
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, Ninv, prior = make_case(24, 640, 16, 5, 9, False)
    out = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=4, seed=2, verbose=False, rng="philox")
    assert np.all(np.isfinite(out[2])) and np.all(out[2] > 0) and np.all(np.isfinite(out[5]))
    want = ho.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=2, seed=2, solver="theta")
    got = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=2, seed=2, verbose=False)  # default: reference-cg
    for o, w, k in zip(got[:6], want, KEYS):
        assert rel(o, w) < 1e-9, k


@pytest.mark.parametrize("nf,nm", [(448, 32), (500, 44)])
def test_resident_k_solve_chain_matches_oracle(nf, nm):
    """Np = 480 and 544 (past k_solve3's range, resident k_solve): two iterations with injected draws match the oracle in
    every output, signal_ps (the partial sums of |ytilde|^2) included, and a Philox chain runs."""
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, Ninv, prior = make_case(6, nf, nm, 4, nf, False)
    want = ho.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=2, seed=4, solver="direct", symmetric_flags=True)
    got = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=2, seed=4, verbose=False, solver="exact")
    for o, w, k in zip(got[:6], want, KEYS):
        assert rel(o, w) < 1e-9, k
    out = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=3, seed=4, verbose=False, rng="philox")
    assert np.all(np.isfinite(out[2])) and np.all(out[2] > 0) and np.all(np.isfinite(out[5]))


@pytest.mark.parametrize("nf,nm", [(448, 32), (512, 32), (544, 32), (560, 32)])
def test_resident_tile_boundary_residual(nf, nm):
    """Np = 480 and 544 are past k_solve3's range (Np <= 448) and take the resident k_solve; N = 576 is the largest system
    k_solve keeps resident in shared memory (Np = 576); N = 592 is the first that takes the dense-product solve.
    Size-independent property on both sides of each boundary: the solution satisfies the reference's A x = b for every
    time (map_estimate: no fluctuation terms), and the two paths agree on a common sub-problem through the chi^2 of the
    fit."""
    from hydra_pspec_b200 import pspec
    rng = np.random.default_rng(nf)
    nt = 20
    F = np.linalg.qr(crandn(rng, nf, nm))[0]
    fop = ho.fourier_operator(nf)
    p0 = 0.5 + rng.random(nf)
    S0 = fop.conj().T @ np.diag(p0 / nf ** 2) @ fop
    vis = crandn(rng, nt, nf) + (30 * crandn(rng, nt, nm)) @ F.T
    flags = np.ones(nf, dtype=bool)
    flags[[10, 11, 200]] = False
    ninv = 2.0
    cr, _, _, fg, _, _, _ = pspec.gibbs_sample_with_fg(vis, flags, S0, F, np.eye(nf) * ninv, None, Niter=1, verbose=False,
                                                       map_estimate=True, solver="exact")
    Ni = np.diag(flags * ninv).astype(complex)
    A = np.zeros((nf + nm, nf + nm), complex)
    A[:nf, :nf] = np.eye(nf) + S0 @ Ni
    A[:nf, nf:] = S0 @ Ni @ F
    A[nf:, :nf] = F.conj().T @ Ni
    A[nf:, nf:] = F.conj().T @ Ni @ F
    worst = 0.0
    for t in range(nt):
        z = Ni @ (flags * vis[t])
        b = np.concatenate([S0 @ z, F.conj().T @ z])
        x = np.concatenate([cr[0, t], fg[0, t]])
        worst = max(worst, np.linalg.norm(A @ x - b) / np.linalg.norm(b))
    assert worst < 1e-10
