"""Per-time diagonal noise (an inverse noise variance per time and channel).  GPU only.

Anchored on the per-time-noise oracle (tests/time_noise_oracle.py, exact solves) with the reference's injected draws, on
the 2-D paths it must reduce to (identical slices, weights equal to one diagonal), on the analytic GCR covariance of the
Philox draws, and on single-chain runs for a batch.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import hydra_oracle as ho  # noqa: E402  (checker only)
import time_noise_oracle as tno  # noqa: E402

TOL = 1e-10
KEYS = ["signal_cr", "signal_S", "signal_ps", "fg_amps", "chisq", "ln_post"]


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    if b.size == 0:
        return 0.0
    return np.max(np.abs(a - b)) / np.max(np.abs(b))


def crandn(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def make_case(nt, nf, nm, seed, weights, per_time_flags):
    """Inputs with per-time weights v_t = nsamples_t * diag(Ninv):
    piecewise: constant over runs of times (factor re-use); every: a new row every time; zeros: some cells weighted out;
    zero_time: additionally one time with all weights zero."""
    rng = np.random.default_rng(seed)
    F = np.linalg.qr(crandn(rng, nf, nm))[0] if nm else np.zeros((nf, 0), dtype=complex)
    fop = ho.fourier_operator(nf)
    p0 = 0.5 + rng.random(nf)
    S0 = fop.conj().T @ np.diag(p0 / nf ** 2) @ fop
    sig = 0.3 + rng.random(nf)
    vis = crandn(rng, nt, nf) * sig + (5 * crandn(rng, nt, nm)) @ F.T + crandn(rng, nt, nf) @ np.linalg.cholesky(
        S0 + 1e-12 * np.eye(nf)).T
    if "piecewise" in weights:
        rows = 1.0 + rng.integers(0, 4, size=(4, nf))
        nsamp = rows[np.minimum(np.arange(nt) // 10, 3)]
    else:
        nsamp = 0.5 + 3.0 * rng.random((nt, nf))
    if "zeros" in weights or "zero_time" in weights:
        nsamp = nsamp * (rng.random((nt, nf)) > 0.08)
    if "zero_time" in weights:
        nsamp[5] = 0.0
    ninv_t = nsamp / sig[None, :] ** 2
    if per_time_flags:
        flags = np.ones((nt, nf), dtype=bool)
        for t0 in range(0, nt, 10):        # flags change where the weights may change (piecewise rows keep re-use)
            flags[t0:t0 + 10, rng.choice(nf, 3, replace=False)] = False
        flags[:, 3] = False
    else:
        flags = rng.random(nf) > 0.05
    prior = np.zeros((2, nf))
    prior[0, nf // 2 - 1:nf // 2 + 2] = 40.0
    prior[1, nf // 2 - 1:nf // 2 + 2] = 0.2
    return vis, flags, S0, F, ninv_t, prior


# k_post_fft2 (128, 256, 384) and k_post_fft (96, 120); T = 37 ends in a partial time tile
@pytest.mark.parametrize("nf,nm,weights,per_time_flags", [
    (128, 8, "piecewise", False),
    (256, 0, "zero_time", True),
    (384, 8, "piecewise+zeros", True),
    (96, 8, "every+zeros", True),
    (120, 0, "every+zero_time", False),
    (120, 8, "piecewise", True),
    (512, 16, "piecewise", True),       # N = 528: k_pt_cholsolve at nblk = 17, k_post_fft2 at 512
])
def test_time_noise_chain_matches_oracle(nf, nm, weights, per_time_flags):
    from hydra_pspec_b200 import pspec
    nt, niter = 37, 3
    vis, flags, S0, F, ninv_t, prior = make_case(nt, nf, nm, nf + nm, weights, per_time_flags)
    Ninv = tno.diag_stack(ninv_t)
    ref = tno.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=niter, seed=17, solver="direct")
    out = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=niter, seed=17, verbose=False)
    for o, r, k in zip(out[:6], ref, KEYS):
        # chi^2 of near-zero residuals carries the cancellation of d - s - F f (as in test_gpu_pertime)
        assert rel(o, r) < (1e-8 if k == "chisq" else TOL), (k, rel(o, r))
    if "zero_time" in weights:
        # no data weight at time 5 and no foreground modes: the solution is the prior draw S^1/2 omega_a
        oma, _ = ho.reference_gcr_draws(nt, nf)
        x = ho.build_matrices(np.ones(nf, bool), S0, np.zeros((nf, nf)), F, need_pinv=False)["Sh"] @ oma[5]
        assert rel(out[0][0, 5], x) < TOL


def test_fully_weighted_out_time_with_modes_reports_singular_system():
    """With foreground modes a time without any data weight has a singular system, reported through info() as a fully
    flagged time is."""
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, ninv_t, prior = make_case(12, 64, 4, 3, "every", True)
    ninv_t[4] = 0.0
    eng = pspec.GibbsEngine(1, 12, 64, 4, max_iters=1, rng="philox", keep=(), time_flags=True)
    try:
        eng.load_chain(0, vis, flags, F, None, np.full(64, 1.0 / 64), ninv_t=ninv_t)
        eng.run(1)
        assert eng.info()[0] != 0
    finally:
        eng.close()


@pytest.mark.parametrize("rng_mode", ["philox", "numpy"])
def test_identical_slices_bit_identical_to_2d(rng_mode):
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, ninv_t, prior = make_case(20, 96, 8, 7, "every", False)
    Ninv = np.diag(ninv_t[0])
    a = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=3, seed=4, verbose=False, rng=rng_mode)
    b = pspec.gibbs_sample_with_fg(vis, flags, S0, F, np.stack([Ninv] * 20), prior, Niter=3, seed=4, verbose=False,
                                   rng=rng_mode)
    for x, y, k in zip(a[:6], b[:6], KEYS):
        assert np.array_equal(np.asarray(x), np.asarray(y)), k


def _run_engine(vis, flags, F, ninv, lam0sq, ninv_t, force_dense_solve, niter=3):
    from hydra_pspec_b200 import pspec
    T, n = vis.shape
    eng = pspec.GibbsEngine(1, T, n, F.shape[1], max_iters=niter, rng="philox", seed=11, time_flags=True,
                            force_dense_solve=force_dense_solve)
    try:
        eng.load_chain(0, vis, flags, F, ninv, lam0sq, ninv_t=ninv_t)
        eng.run(niter)
        return [eng.signal_cr(0), eng.signal_ps(0), eng.fg_amps(0), eng.chisq(0), eng.ln_post(0)]
    finally:
        eng.close()


def test_broadcast_weights_equal_per_time_flags_direct_form():
    vis, flags, S0, F, ninv_t, prior = make_case(37, 128, 8, 9, "every", True)
    ninv = ninv_t[0]
    lam0sq = np.full(128, 1.0 / 128)
    a = _run_engine(vis, flags, F, ninv, lam0sq, None, True)
    b = _run_engine(vis, flags, F, None, lam0sq, np.tile(ninv, (37, 1)), False)
    for x, y, k in zip(a, b, ["signal_cr", "signal_ps", "fg_amps", "chisq", "ln_post"]):
        assert rel(y, x) < 1e-12, (k, rel(y, x))


def test_philox_covariance_two_weight_rows():
    """Sample covariance of the Philox GCR draws at two times with different weights (and flags) equals the analytic
    M_t^-1; draws of different times -- also of a time that re-uses the factor of the time before -- are uncorrelated."""
    from hydra_pspec_b200 import pspec
    nt, nf, nm, nch, ndraw = 32, 96, 8, 2, 3000
    rng = np.random.default_rng(77)
    F = np.linalg.qr(crandn(rng, nf, nm))[0]
    ps = nf * (0.5 + 2.0 * rng.random(nf))
    rows = np.stack([1.0 + rng.random(nf), 0.2 + 3.0 * rng.random(nf)])
    rows[1, [9, 50]] = 0.0
    masks = np.ones((2, nf), dtype=bool)
    masks[0, [5, 40]] = False
    masks[1, [17]] = False
    tmask = (np.arange(nt) // 2) % 2                      # A A B B A A ...: every odd time re-uses the factor of t - 1
    flags = masks[tmask]
    ninv_t = rows[tmask]
    vis = crandn(rng, nch, nt, nf) + (3 * crandn(rng, nch, nt, nm)) @ F.T
    eng = pspec.GibbsEngine(nch, nt, nf, nm, max_iters=1, rng="philox", refresh_omega=True, keep=(), seed=5, time_flags=True)
    for c in range(nch):
        eng.load_chain(c, vis[c], flags, F, None, ps / nf, ninv_t=ninv_t)
    assert eng.pt_form()[0] == "direct"
    fop = ho.fourier_operator(nf)
    S = ho.covariance_from_pspec(ps / nf ** 2, fop)
    P = np.concatenate([np.eye(nf), F], axis=1)
    post = []
    for i in range(2):
        Ni = np.diag(masks[i] * rows[i])
        prec = P.conj().T @ Ni @ P
        prec[:nf, :nf] += np.linalg.inv(S)
        Sigma = np.linalg.inv(prec)
        post.append((Sigma, Sigma @ P.conj().T @ Ni))
    mean = np.stack([np.stack([post[tmask[t]][1] @ (vis[c, t] * masks[tmask[t]]) for t in range(nt)]) for c in range(nch)])
    N = nf + nm
    C0 = [np.zeros((N, N), dtype=complex) for _ in range(2)]
    Ct1 = np.zeros((N, N), dtype=complex)                  # t vs t + 1 for even t: same system, re-used factor
    Cit = np.zeros((N, N), dtype=complex)
    prev = None
    for k in range(ndraw):
        eng.gcr()
        E = np.stack([eng.last_gcr(c) for c in range(nch)]) - mean
        for i in range(2):
            e2 = E[:, tmask == i].reshape(-1, N)
            C0[i] += e2.T @ e2.conj()
        Ct1 += E[:, 0::2].reshape(-1, N).T @ E[:, 1::2].reshape(-1, N).conj()
        if prev is not None:
            Cit += prev.reshape(-1, N).T @ E.reshape(-1, N).conj()
        prev = E
    eng.close()

    def nrm(C, var):
        d = np.sqrt(var)
        return np.max(np.abs(C) / np.outer(d, d))

    for i in range(2):
        ns = ndraw * nch * int(np.sum(tmask == i))
        err = nrm(C0[i] / ns - post[i][0], np.real(np.diagonal(post[i][0])))
        assert err < 6.0 / np.sqrt(ns), (i, err)
    # the cross terms pool pairs of both systems: scaled by the larger of the two variances of each element
    env = np.maximum(np.real(np.diagonal(post[0][0])), np.real(np.diagonal(post[1][0])))
    for name, C, ns in (("time", Ct1, ndraw * nch * nt // 2), ("draw", Cit, (ndraw - 1) * nch * nt)):
        err = nrm(C / ns, env)
        assert err < 6.0 / np.sqrt(ns), (name, err)


def test_form_switching_and_refusals():
    from hydra_pspec_b200 import pspec, _lib
    nt, nf, nm = 20, 64, 4
    vis, flags, S0, F, ninv_t, prior = make_case(nt, nf, nm, 13, "every", True)
    lam0sq = np.full(nf, 1.0 / nf)
    eng = pspec.GibbsEngine(2, nt, nf, nm, max_iters=2, rng="philox", keep=(), time_flags=True)
    try:
        eng.load_chain(0, vis, flags, F, ninv_t[0], lam0sq)
        eng.load_chain(1, vis, flags, F, ninv_t[0], lam0sq)
        assert eng.pt_form()[0] == "low-rank"
        eng.load_chain(1, vis, flags, F, None, lam0sq, ninv_t=ninv_t)
        assert eng.pt_form()[0] == "direct"
        eng.run(1)
        assert np.all(eng.info() == 0)
        eng.load_chain(1, vis, flags, F, ninv_t[0], lam0sq)       # reloaded without per-time noise
        assert eng.pt_form()[0] == "low-rank"
        eng.rewind()
        eng.run(1)
        assert np.all(eng.info() == 0)
        for bad in (np.nan, np.inf, -1.0):
            w = ninv_t.copy()
            w[3, 7] = bad
            with pytest.raises(_lib.HydraLibError):
                eng.load_chain(0, vis, flags, F, None, lam0sq, ninv_t=w)
    finally:
        eng.close()
    # a general S_initial: the direct form takes a delay-diagonal one only
    eng = pspec.GibbsEngine(1, nt, nf, nm, max_iters=1, rng="philox", keep=(), time_flags=True, general_basis0=True)
    try:
        with pytest.raises(_lib.HydraLibError):
            eng.load_chain(0, vis, flags, F, None, lam0sq, basis0=np.eye(nf, dtype=complex), ninv_t=ninv_t)
    finally:
        eng.close()
    # an engine without per-time flags
    eng = pspec.GibbsEngine(1, nt, nf, nm, max_iters=1, rng="philox", keep=())
    try:
        with pytest.raises(ValueError):
            eng.load_chain(0, vis, flags[0], F, None, lam0sq, ninv_t=ninv_t)
    finally:
        eng.close()
    with pytest.raises(NotImplementedError):
        pspec.gibbs_sample_with_fg(vis, flags, S0, F, tno.diag_stack(ninv_t), prior, Niter=1, verbose=False,
                                   solver="reference-cg")


@pytest.mark.parametrize("force_direct", [True, False])
def test_batch_mixed_equals_single_chains(force_direct, monkeypatch):
    """A batch of baselines with and without per-time noise on 4 sub-streams gives the samples of single-chain runs with
    the same Philox chain ids: on the direct form from the start, and when the engine starts in the low-rank form and switches
    to the direct form as the per-time-noise baselines are loaded.  To round-off, not bit for bit: k_pt_cholsolve re-uses the
    factor of time t - 1 only when both times fall on the same persistent CTA, and which times do depends on the number of
    systems in the launch; a re-used factor is applied by a separate forward substitution instead of the one fused into the
    factorisation."""
    from hydra_pspec_b200 import pspec
    nt, nf, nm = 37, 96, 8
    bls = []
    for i in range(5):
        vis, flags, S0, F, ninv_t, prior = make_case(nt, nf, nm, 100 + i, "piecewise" if i % 2 else "every", True)
        b = dict(vis=vis, flags=flags, S_initial=S0, fgmodes=F, ps_prior=prior)
        b["Ninv"] = tno.diag_stack(ninv_t) if i in (0, 3) else np.diag(ninv_t[0])
        bls.append(b)
    bls[4]["ninv_t"] = ninv_t   # per-time noise in the compact (Ntimes, Nfreqs) form
    ids = np.arange(5) * 3 + 1
    single = []
    monkeypatch.setattr(pspec, "_FORCE_DENSE_SOLVE", True)
    for i, b in enumerate(bls):
        single.append(pspec.gibbs_sample_batch([b], Niter=3, seed=21, rng="philox", chain_ids=ids[i:i + 1]))
    monkeypatch.setattr(pspec, "_FORCE_DENSE_SOLVE", force_direct)
    batch = pspec.gibbs_sample_batch(bls, Niter=3, seed=21, rng="philox", chain_ids=ids, substreams=4)
    for i in range(5):
        for k, (x, y) in enumerate(zip(single[i][0][:6], batch[i][:6])):
            assert rel(y, x) < (1e-10 if KEYS[k] == "chisq" else 1e-12), (i, KEYS[k], rel(y, x))
