"""Per-time flags (BASELINE.json configs[2]: in-painting, one factorisation per time).  GPU only.

The reference has no per-time path (it asserts 1-D flags, pspec.py:428, and its driver collapses the
flags, run-hydra-pspec.py:520-526), so parity is anchored three ways:
  * a golden produced by the unmodified reference's `gcr_fgmodes_1d` called time by time with that
    time's flags and operators (tests/golden/make_golden_pertime.py);
  * the oracle's 2-D flag extension (the same per-time algebra) on fresh inputs, exact solves, 1e-10;
  * consistency: per-time flags that are equal at all times reproduce the shared-factorisation path.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import hydra_oracle as ho  # noqa: E402  (checker only)

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


def make_case(nt, nf, nm, frac, seed):
    rng = np.random.default_rng(seed)
    F = np.linalg.qr(crandn(rng, nf, nm))[0] if nm else np.zeros((nf, 0), dtype=complex)
    fop = ho.fourier_operator(nf)
    p0 = 0.5 + rng.random(nf)
    S0 = fop.conj().T @ np.diag(p0 / nf ** 2) @ fop
    sig = 0.3 + rng.random(nf)
    vis = crandn(rng, nt, nf) * sig + (5 * crandn(rng, nt, nm)) @ F.T + crandn(rng, nt, nf) @ np.linalg.cholesky(
        S0 + 1e-12 * np.eye(nf)).T
    flags = rng.random((nt, nf)) > frac
    flags[0] = True          # one time without flags
    flags[:, 3] = False      # one channel flagged at all times
    prior = np.zeros((2, nf))
    prior[0, nf // 2 - 1:nf // 2 + 2] = 40.0
    prior[1, nf // 2 - 1:nf // 2 + 2] = 0.2
    return vis, flags, S0, F, np.diag(1.0 / sig ** 2), prior


@pytest.fixture(params=["lowrank", "direct"])
def pt_form(request, monkeypatch):
    """Both forms of the per-time solve: the low-rank correction of one shared factorisation (hp_ptlow.cu, default) and
    one factorisation per time (hp_pertime.cu: the engine's force_dense_solve field)."""
    from hydra_pspec_b200 import pspec
    if request.param == "direct":
        monkeypatch.setattr(pspec, "_FORCE_DENSE_SOLVE", True)
    return request.param


@pytest.mark.parametrize("nt,nf,nm,frac,seed", [(6, 32, 4, 0.1, 1), (9, 45, 5, 0.2, 2), (12, 120, 12, 0.05, 3),
                                                (5, 64, 0, 0.3, 4), (7, 96, 33, 0.1, 5), (4, 256, 16, 0.1, 6)])
def test_per_time_chain_matches_oracle(nt, nf, nm, frac, seed, pt_form):
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, Ninv, prior = make_case(nt, nf, nm, frac, seed)
    niter = 3
    ref = ho.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=niter, seed=17, solver="direct")
    out = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=niter, seed=17, verbose=False)
    for o, r, k in zip(out[:6], ref, KEYS):
        assert rel(o, r) < (1e-8 if k == "chisq" else TOL), k


def test_constant_per_time_flags_equal_shared_factorisation():
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, Ninv, prior = make_case(10, 48, 6, 0.15, 11)
    w1 = flags[1]
    a = pspec.gibbs_sample_with_fg(vis, w1, S0, F, Ninv, prior, Niter=3, seed=5, verbose=False, solver="exact")
    b = pspec.gibbs_sample_with_fg(vis, np.broadcast_to(w1, vis.shape).copy(), S0, F, Ninv, prior, Niter=3, seed=5,
                                   verbose=False)
    for x, y, k in zip(a[:6], b[:6], KEYS):
        assert rel(y, x) < (1e-8 if k == "chisq" else TOL), k


def test_per_time_solution_solves_each_time_system(pt_form):
    """Size-independent property at the configs[2] system size (Nfreq=256, Nfg=16): residual of every
    per-time system M_t x = b_t, map_estimate (no fluctuation terms)."""
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, Ninv, _ = make_case(40, 256, 16, 0.1, 21)
    cr, _, _, fg, _, _, _ = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, None, Niter=1, verbose=False,
                                                       map_estimate=True)
    ni = np.real(np.diagonal(Ninv))
    Sinv = np.linalg.inv(S0)
    worst = 0.0
    for t in range(vis.shape[0]):
        w = flags[t].astype(float)
        Ni = np.diag(w * ni)
        s, f = cr[0, t], fg[0, t]
        top = Sinv @ s + Ni @ (s + F @ f) - Ni @ (w * vis[t])     # (S^-1 + Ni) s + Ni F f = Ni d
        bot = F.conj().T @ (Ni @ (s + F @ f - w * vis[t]))
        scale = np.linalg.norm(Ni @ (w * vis[t]))
        worst = max(worst, np.linalg.norm(top) / scale, np.linalg.norm(bot) / scale)
    assert worst < 1e-9


def test_per_time_reference_golden(golden_dir):
    """GCR solves of the unmodified reference (gcr_fgmodes_1d, one call per time with that time's
    operators); the reference's CG truncation is ~1e-8 relative, hence the tolerance."""
    from hydra_pspec_b200 import pspec
    g = np.load(golden_dir / "gcr_pertime.npz")
    eng = pspec._single_chain_engine(g["vis"] * g["flags"], g["flags"], g["S"], g["fgmodes"], g["Ninv"], None, 1, "numpy",
                                     None, False, (), None, 0)
    try:
        eng.gcr()
        out = eng.last_gcr(0)
    finally:
        eng.close()
    assert rel(out, g["cr"]) < 1e-7


def test_per_time_philox_batch_runs_and_is_reproducible():
    from hydra_pspec_b200 import pspec
    bls = []
    for s in range(3):
        vis, flags, S0, F, Ninv, prior = make_case(24, 64, 6, 0.1, 30 + s)
        bls.append(dict(vis=vis, flags=flags, S_initial=S0, fgmodes=F, Ninv=Ninv, ps_prior=prior))
    a = pspec.gibbs_sample_batch(bls, Niter=5, seed=3, rng="philox")
    b = pspec.gibbs_sample_batch(bls, Niter=5, seed=3, rng="philox")
    c = pspec.gibbs_sample_batch(bls, Niter=5, seed=4, rng="philox")
    for x, y, z in zip(a, b, c):
        assert np.all(np.isfinite(x[2])) and np.all(x[2] > 0)
        np.testing.assert_array_equal(x[2], y[2])
        assert not np.array_equal(x[2], z[2])


def test_per_time_unsupported_combinations_raise():
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, Ninv, prior = make_case(6, 32, 4, 0.1, 1)
    with pytest.raises(NotImplementedError):
        pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=1, verbose=False, solver="reference-cg")
    dense = Ninv + 0.01 * np.ones_like(Ninv)
    with pytest.raises(NotImplementedError):
        pspec.gibbs_sample_with_fg(vis, flags, S0, F, dense, prior, Niter=1, verbose=False)


@pytest.mark.parametrize("nt,nf,nm,frac,seed", [(7, 32, 4, 0.1, 81), (9, 96, 8, 0.15, 82), (5, 128, 0, 0.2, 83)])
def test_per_time_flags_with_general_S_initial(nt, nf, nm, frac, seed, monkeypatch):
    """A non-delay-diagonal S_initial (first iteration in its eigenbasis) together with per-time flags: taken by the low-rank
    form (any first basis; hp_ptlow.cu), refused by the direct form (force_dense_solve; k_pt_cholsolve relies on the
    circulant signal block)."""
    from hydra_pspec_b200 import pspec, _lib
    vis, flags, S0, F, Ninv, prior = make_case(nt, nf, nm, frac, seed)
    rng = np.random.default_rng(seed)
    G = crandn(rng, nf, nf)
    Sg = S0 + 0.3 * np.trace(S0).real / nf * (G @ G.conj().T) / nf          # Hermitian positive definite, not circulant
    ref = ho.gibbs_sample_with_fg(vis, flags, Sg, F, Ninv, prior, Niter=3, seed=5, solver="direct")
    out = pspec.gibbs_sample_with_fg(vis, flags, Sg, F, Ninv, prior, Niter=3, seed=5, verbose=False)
    for o, r, k in zip(out[:6], ref, KEYS):
        assert rel(o, r) < (1e-8 if k == "chisq" else 5e-10), k
    monkeypatch.setattr(pspec, "_FORCE_DENSE_SOLVE", True)
    with pytest.raises(_lib.HydraLibError):
        pspec.gibbs_sample_with_fg(vis, flags, Sg, F, Ninv, prior, Niter=1, seed=5, verbose=False)


@pytest.mark.parametrize("nt,nf,nm,seed", [(2, 8, 1, 1), (3, 12, 2, 2), (5, 16, 0, 3)])
def test_per_time_tiny_shapes(nt, nf, nm, seed, pt_form):
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, Ninv, _ = make_case(nt, nf, nm, 0.2, 50 + seed)
    prior = np.zeros((2, nf))
    ref = ho.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=2, seed=seed, solver="direct")
    out = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=2, seed=seed, verbose=False)
    for o, r, k in zip(out[:6], ref, KEYS):
        assert rel(o, r) < (1e-8 if k == "chisq" else TOL), k


def test_per_time_fully_flagged_integration_is_refused(pt_form):
    """An integration with every channel flagged leaves the (flat-prior) foreground amplitudes of that time
    unconstrained: the system is singular and the chain is refused with LinAlgError instead of returning NaNs."""
    from hydra_pspec_b200 import pspec
    vis, flags, S0, F, Ninv, prior = make_case(6, 32, 4, 0.1, 1)
    flags[2, :] = False
    with pytest.raises(np.linalg.LinAlgError):
        pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=2, seed=1, verbose=False)


@pytest.mark.parametrize("hold", [2, 5, 100])
def test_per_time_repeated_masks_reuse_the_factor(hold, pt_form):
    """Consecutive times with identical flag vectors re-use the factorisation held in the CTA's scratch slot
    (forward + backward substitution only): results must not depend on it."""
    from hydra_pspec_b200 import pspec
    nt = 23
    vis, flags, S0, F, Ninv, prior = make_case(nt, 64, 6, 0.15, 40 + hold)
    flags = np.repeat(flags[::hold], hold, axis=0)[:nt]     # every mask held for `hold` times (100: one mask for all)
    ref = ho.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=3, seed=7, solver="direct")
    out = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=3, seed=7, verbose=False)
    for o, r, k in zip(out[:6], ref, KEYS):
        assert rel(o, r) < (1e-8 if k == "chisq" else TOL), k
    # many chains in one engine: ranges of (chain, time) pairs per CTA straddle chain boundaries
    bls = [dict(vis=vis * (1 + 0.1 * c), flags=flags, S_initial=S0, fgmodes=F, Ninv=Ninv, ps_prior=prior) for c in range(7)]
    outs = pspec.gibbs_sample_batch(bls, Niter=2, seed=7, rng="numpy", solver="exact")
    one = pspec.gibbs_sample_with_fg(bls[3]["vis"], flags, S0, F, Ninv, prior, Niter=2, seed=7, verbose=False)
    for o, r, k in zip(outs[3][:6], one[:6], KEYS):
        assert rel(o, r) < (1e-8 if k == "chisq" else TOL), k


@pytest.mark.parametrize("nf,nm,frac,expect_lowrank", [
    pytest.param(256, 16, 0.2, True, id="0.2-True"),
    pytest.param(256, 16, 0.45, False, id="0.45-False"),
    pytest.param(384, 32, 0.1, True, id="384-32-0.1-True"),       # N = 416: k_pt_lowrank<14>, one time at rank 64
    pytest.param(384, 32, 0.45, False, id="384-32-0.45-False"),
    pytest.param(512, 16, 0.1, False, id="512-16-0.1-False"),     # N = 528: no k_solve3, so direct although every k_t <= 64
    pytest.param(1024, 64, 0.05, False, id="1024-64-0.05-False"),  # nblk = 34, k_post_fft2 at 1024 (4 times, 1 iteration)
])
def test_per_time_rank_limit_selects_the_form(nf, nm, frac, expect_lowrank):
    """Nfreq=256: 20 % per-time flags stay below the 64-channel limit of the low-rank form (ranks up to ~60); 45 % exceed it
    and the engine falls back to one factorisation per time.  At 384 + 32 the same two sides of the rank limit, at 512 + 16 and
    1024 + 64 the direct form because N > 448.  The form is asserted on an engine loaded with the same chain; both forms
    against the oracle."""
    from hydra_pspec_b200 import pspec
    nt, niter = (4, 1) if nf >= 1024 else (6, 2)
    vis, flags, S0, F, Ninv, prior = make_case(nt, nf, nm, frac, 61)
    if expect_lowrank:
        wbar = flags.any(axis=0)
        flags[1, np.flatnonzero(wbar)[:64]] = False       # one time at exactly the limit
        flags[1, np.flatnonzero(wbar)[64:]] = True
    kmax = int(np.max(np.sum(flags.any(axis=0)[None, :] & ~flags, axis=1)))
    if nf + nm <= 448:
        assert (kmax <= 64) == expect_lowrank
    eng = pspec.GibbsEngine(1, nt, nf, nm, max_iters=1, rng="numpy", keep=(), time_flags=True)
    try:
        eng.load_chain(0, vis, flags, F, np.real(np.diag(Ninv)), np.full(nf, 1.0 / nf))
        form, kcap = eng.pt_form()
    finally:
        eng.close()
    assert form == ("low-rank" if expect_lowrank else "direct")
    if expect_lowrank:
        assert kcap == kmax == 64
    ref = ho.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=niter, seed=9, solver="direct")
    out = pspec.gibbs_sample_with_fg(vis, flags, S0, F, Ninv, prior, Niter=niter, seed=9, verbose=False)
    for o, r, k in zip(out[:6], ref, KEYS):
        assert rel(o, r) < (1e-8 if k == "chisq" else TOL), k


def test_per_time_forms_agree_at_config2_shape(monkeypatch):
    """BASELINE.json configs[2] shape (Nfreq=256, Nfg=16, 5 % per-time flags on top of a 5 % all-times mask), 64 times, four
    chains in one engine: low-rank form == one factorisation per time (force_dense_solve) to round-off (injected draws, two
    iterations)."""
    from hydra_pspec_b200 import pspec
    bls = []
    for c in range(4):
        vis, flags, S0, F, Ninv, prior = make_case(64, 256, 16, 0.05, 70 + c)
        flags[:, np.random.default_rng(c).choice(256, 12, replace=False)] = False
        bls.append(dict(vis=vis, flags=flags, S_initial=S0, fgmodes=F, Ninv=Ninv, ps_prior=prior))
    low = pspec.gibbs_sample_batch(bls, Niter=2, seed=5, rng="numpy", solver="exact")
    monkeypatch.setattr(pspec, "_FORCE_DENSE_SOLVE", True)
    direct = pspec.gibbs_sample_batch(bls, Niter=2, seed=5, rng="numpy", solver="exact")
    for a, b in zip(low, direct):
        for x, y, k in zip(a[:6], b[:6], KEYS):
            assert rel(x, y) < (1e-8 if k == "chisq" else TOL), k


def test_per_time_fallback_after_low_rank_chains_were_loaded():
    """Two chains in one engine: the first stays within the rank limit (its direct-form operands are not built at load time),
    the second has times with more than 64 extra flags, which switches the whole engine to one factorisation per time: the
    operands of the first chain are then built lazily.  Both against the oracle."""
    from hydra_pspec_b200 import pspec
    a = make_case(5, 256, 8, 0.05, 91)
    b = make_case(5, 256, 8, 0.45, 92)
    bls = [dict(vis=c[0], flags=c[1], S_initial=c[2], fgmodes=c[3], Ninv=c[4], ps_prior=c[5]) for c in (a, b)]
    outs = pspec.gibbs_sample_batch(bls, Niter=2, seed=13, rng="numpy", solver="exact")
    for c, out in zip((a, b), outs):
        ref = ho.gibbs_sample_with_fg(c[0], c[1], c[2], c[3], c[4], c[5], Niter=2, seed=13, solver="direct")
        for o, r, k in zip(out[:6], ref, KEYS):
            assert rel(o, r) < (1e-8 if k == "chisq" else TOL), k
