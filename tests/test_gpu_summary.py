"""On-device posterior moments of signal_cr and fg_amps (hp_engine_set_summary / hp_engine_read_summary, k_moments).
GPU only.  The moments are compared with numpy's mean / var of the same chain's samples, read back from the device."""
import json
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

sys.path.insert(0, str(Path(__file__).resolve().parent / "golden"))
from make_golden_testdata import driver_argv  # noqa: E402
from testdata_fixture import materialize  # noqa: E402

TOL = 1e-10          # golden parity (test_gpu_parity.py)
MEAN_TOL = 1e-12     # moments against numpy on the same samples
VAR_TOL = 1e-11


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    if b.size == 0:
        return 0.0
    den = np.max(np.abs(b))
    return np.max(np.abs(a - b)) / den if den > 0 else np.max(np.abs(a))


def crandn(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def chain_inputs(seed, T, n, m, per_time=False, dense=False, general=False):
    """load_chain keyword arguments of one synthetic baseline."""
    rng = np.random.default_rng(seed)
    F = np.linalg.qr(crandn(rng, n, max(m, 1)))[0][:, :m]
    sig = 0.5 + 0.5 * rng.random(n)
    vis = crandn(rng, T, n) * (1.0 + sig) + (crandn(rng, T, m) * np.logspace(2, 0, m)) @ F.T
    flags = np.ones(n, dtype=bool)
    flags[rng.choice(n, max(1, n // 20), replace=False)] = False
    if per_time:
        flags = np.broadcast_to(flags, (T, n)) & (rng.random((T, n)) > 0.05)
    kw = dict(vis=vis, flags=flags, fgmodes=F, ninv_diag=1.0 / sig ** 2, lam0sq=0.5 + rng.random(n))
    if dense:
        X = crandn(rng, n, 2 * n)
        Ninv = np.linalg.inv(X @ X.conj().T / (2 * n) + 0.5 * np.eye(n))
        kw.update(ninv_dense=Ninv, ninv_diag=np.real(np.diagonal(Ninv)).copy())
    if general:
        Q = np.linalg.qr(crandn(rng, n, n))[0]
        kw.update(basis0=Q)
    return kw


def make_engine(C=5, T=40, n=96, m=8, niter=13, keep=("cr", "fg"), ring_iters=0, substreams=2, seed=7, per_time=False,
                dense=False, general=False, **kw):
    from hydra_pspec_b200 import pspec
    eng = pspec.GibbsEngine(C, T, n, m, niter, rng="philox", keep=keep, ring_iters=ring_iters, seed=seed, substreams=substreams,
                            time_flags=per_time, dense_noise=dense, general_basis0=general, **kw)
    for c in range(C):
        eng.load_chain(c, **chain_inputs(100 + c, T, n, m, per_time=per_time, dense=dense, general=general))
    return eng


def check_moments(eng, c, sel):
    """moments of chain c against numpy on its samples selected by `sel`"""
    got = eng.summary(c)
    for key, samples in (("signal_cr", eng.signal_cr(c)[sel]), ("fg_amps", eng.fg_amps(c)[sel])):
        assert got["count"] == samples.shape[0]
        assert rel(got[f"{key}_mean"], samples.mean(axis=0)) <= MEAN_TOL, key
        assert rel(got[f"{key}_var"], samples.var(axis=0)) <= VAR_TOL, key
    return got


CASES = {
    "fft_n96": dict(),
    "fft2_n128": dict(n=128),
    "fft2_n384": dict(n=384),
    "dense_transforms": dict(force_dense_transforms=True),
    "dense_solve": dict(force_dense_solve=True),
    "dense_noise": dict(dense=True),
    "per_time_lowrank": dict(per_time=True),
    "per_time_direct": dict(per_time=True, force_dense_solve=True),
    "general_basis0": dict(general=True),
    "no_fg_modes": dict(m=0),
    "odd_rows_prime_nfreqs": dict(T=41, n=37, m=3),   # odd T n and T m (padded accumulator rows); no FFT plan for 37
}


@pytest.mark.parametrize("case", list(CASES))
def test_moments_match_samples(case):
    """5 chains in 2 sub-batches, 13 iterations, burn_in 3, thin 2: the moments are those of samples [3::2]."""
    eng = make_engine(**CASES[case])
    try:
        if case.startswith("per_time"):
            assert eng.pt_form()[0] == ("direct" if case == "per_time_direct" else "low-rank")
        eng.set_summary(("cr", "fg"), burn_in=3, thin=2)
        eng.run(13)
        assert np.all(eng.info() == 0)
        for c in range(eng.nchains):
            got = check_moments(eng, c, slice(3, None, 2))
            assert got["count"] == 5
            if eng.nmodes == 0:
                assert got["fg_amps_mean"].shape == (eng.ntimes, 0)
    finally:
        eng.close()


def read_all(eng):
    return [eng.summary(c) for c in range(eng.nchains)]


def assert_identical(a, b):
    for x, y in zip(a, b):
        assert x.keys() == y.keys()
        for k in x:
            assert np.array_equal(x[k], y[k]), k


def test_splitting_does_not_change_the_moments():
    """run(13), run(4) + run(9), and run_to_host in chunks with read-ahead give bit-identical moments."""
    res = []
    eng = make_engine()
    eng.set_summary(burn_in=3, thin=2)
    eng.run(13)
    res.append(read_all(eng))
    eng.close()

    eng = make_engine()
    eng.set_summary(burn_in=3, thin=2)
    eng.run(4)
    eng.run(9)
    res.append(read_all(eng))
    eng.close()

    eng = make_engine(ring_iters=3)
    eng.set_summary(burn_in=3, thin=2)
    stage = eng.host_buffers(4, iter_major=True)
    done = 0
    while done < 13:
        c = min(4, 13 - done)
        last = done + c >= 13
        eng.run_to_host(c, stage, first_iter=done, iter_major=True, read_ahead=0 if last else 2)
        done += c
        if not last:
            from hydra_pspec_b200 import _lib
            with pytest.raises(_lib.HydraLibError, match="read-ahead"):
                eng.summary(0)   # the moments already include iterations that were not delivered
    res.append(read_all(eng))
    eng.close()
    assert res[0][0]["count"] == 5
    assert_identical(res[0], res[1])
    assert_identical(res[0], res[2])


def test_summary_does_not_change_the_chain():
    out = []
    for on in (False, True):
        eng = make_engine()
        if on:
            eng.set_summary(burn_in=1, thin=1)
        eng.run(13)
        out.append([(eng.signal_ps(c), eng.ln_post(c), eng.signal_cr(c)) for c in range(eng.nchains)])
        eng.close()
    for a, b in zip(*out):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    # signal_cr read from the Sf scratch (keep=()) and from the ring slot (keep cr): the same moments
    mom = []
    for keep in ((), ("cr", "fg")):
        eng = make_engine(keep=keep)
        eng.set_summary(burn_in=2, thin=3)
        eng.run(13)
        mom.append(read_all(eng))
        eng.close()
    assert_identical(*mom)


def test_reference_parity_golden(golden_dir):
    """numpy draws + reference CG on the golden chain B: the moments of the call's own samples, and the golden means."""
    from hydra_pspec_b200 import pspec
    g = np.load(golden_dir / "chain_B_defaults.npz", allow_pickle=True)
    out = pspec.gibbs_sample_with_fg(g["vis"], g["flags"], g["S_initial"], g["fgmodes"], g["Ninv"], g["ps_prior"],
                                     Niter=int(g["Niter"]), seed=int(g["seed"]), verbose=False, summary=dict(burn_in=1, thin=1))
    assert len(out) == 8
    mom = out[7]
    assert mom["count"] == int(g["Niter"]) - 1
    for key, samples, gold in (("signal_cr", out[0], g["signal_cr"]), ("fg_amps", out[3], g["fg_amps"])):
        assert rel(mom[f"{key}_mean"], samples[1:].mean(axis=0)) <= MEAN_TOL, key
        assert rel(mom[f"{key}_var"], samples[1:].var(axis=0)) <= VAR_TOL, key
        assert rel(mom[f"{key}_mean"], gold[1:].mean(axis=0)) < TOL, key
        # the reference re-uses its fluctuation draws: the spread between iterations can be tiny next to the mean
        assert np.max(np.abs(mom[f"{key}_var"] - gold[1:].var(axis=0))) <= TOL * np.max(np.abs(gold[1:])) ** 2, key


def test_refusals_and_empty_summary():
    from hydra_pspec_b200 import _lib
    L = _lib.lib()
    eng = make_engine(C=2, niter=4)
    try:
        assert L.hp_engine_set_summary(eng._h, _lib.HP_SUMMARY_CR, 0, 0) == -1   # HP_ERR_ARG
        assert L.hp_engine_set_summary(eng._h, _lib.HP_SUMMARY_CR, -1, 1) == -1
        assert L.hp_engine_set_summary(eng._h, 4, 0, 1) == -1
        with pytest.raises(ValueError):
            eng.summary(0)                       # nothing accumulated yet
        eng.set_summary(("cr",), burn_in=0, thin=1)
        mean = np.empty((eng.ntimes, eng.nmodes), np.complex128)
        var = np.empty((eng.ntimes, eng.nmodes))
        cnt = _lib.C.c_int(-1)
        assert L.hp_engine_read_summary(eng._h, 0, _lib.HP_SUMMARY_FG, _lib.ptr(mean), _lib.ptr(var), mean.nbytes,
                                        _lib.C.byref(cnt)) == -1   # fg_amps is not being accumulated
        small = np.empty((eng.ntimes, eng.nfreqs - 1), np.complex128)
        assert L.hp_engine_read_summary(eng._h, 0, _lib.HP_SUMMARY_CR, _lib.ptr(small), None, small.nbytes, None) == -1
        assert L.hp_engine_read_summary(eng._h, 2, _lib.HP_SUMMARY_CR, None, None, 0, None) == -1   # chain out of range
        assert L.hp_engine_read_summary(eng._h, 0, 3, None, None, 0, None) == -1                    # two quantities at once
        s = eng.summary(1)
        assert s["count"] == 0 and not np.any(s["signal_cr_mean"]) and not np.any(s["signal_cr_var"])
        eng.run(2)
        eng.gcr()                                # not a Gibbs iteration: not accumulated
        assert eng.summary(0)["count"] == 2
        eng.rewind()                             # keeps the accumulators
        assert eng.summary(0)["count"] == 2
        eng.set_summary(("cr", "fg"), burn_in=0, thin=1)   # restart: zeroed
        s = eng.summary(0)
        assert s["count"] == 0 and not np.any(s["signal_cr_mean"]) and not np.any(s["fg_amps_var"])
    finally:
        eng.close()


def test_batch_keep_nothing_returns_moments(monkeypatch):
    """keep=() with a summary needs neither an out_dir nor host memory for the samples; the moments equal those of the
    samples a keep-everything run of the same seed returns."""
    from hydra_pspec_b200 import pspec
    T, n, m = 24, 64, 4
    bls = []
    for c in range(3):
        kw = chain_inputs(200 + c, T, n, m)
        bls.append(dict(vis=kw["vis"], flags=kw["flags"], S_initial=np.eye(n), fgmodes=kw["fgmodes"], Ninv=np.diag(kw["ninv_diag"]),
                        ps_prior=None))
    full = pspec.gibbs_sample_batch(bls, Niter=9, seed=5, rng="philox")
    monkeypatch.setenv("HP_HOST_BUDGET_GB", "1e-9")
    res = pspec.gibbs_sample_batch(bls, Niter=9, seed=5, rng="philox", keep=(), summary=dict(burn_in=2, thin=3))
    assert len(res) == 3
    for r, f in zip(res, full):
        assert len(r) == 8 and r[0] is None and r[3] is None and r[4] is None
        assert np.array_equal(r[2], f[2]) and np.array_equal(r[5], f[5])
        mom = r[7]
        assert mom["count"] == 3
        for key, samples in (("signal_cr", f[0][2::3]), ("fg_amps", f[3][2::3])):
            assert rel(mom[f"{key}_mean"], samples.mean(axis=0)) <= MEAN_TOL, key
            assert rel(mom[f"{key}_var"], samples.var(axis=0)) <= VAR_TOL, key


@pytest.fixture(scope="module")
def td(tmp_path_factory):
    return materialize(tmp_path_factory.mktemp("testdata"))


def _set(argv, key, value):
    argv = list(argv)
    argv[argv.index(key) + 1] = value
    return argv


@pytest.mark.parametrize("rng", ["philox", "numpy"])
def test_driver_summary_files(td, tmp_path, rng):
    import run_hydra_pspec_b200 as drv
    base = _set(driver_argv(td, tmp_path), "--Niter", "8") + ["--rng", rng]
    assert drv.main(_set(base, "--dirname", "all")) == 0
    assert drv.main(_set(base, "--dirname", "summ") + ["--samples", "summary", "--burn_in", "2", "--thin", "3"]) == 0
    a, s = tmp_path / "all" / "0-1", tmp_path / "summ" / "0-1"
    for f in ("gcr-eor.npy", "fg-amps.npy", "chisq.npy"):
        assert not (s / f).exists(), f
    for f in ("cov-eor.npy", "dps-eor.npy", "ln-post.npy"):
        assert np.array_equal(np.load(s / f), np.load(a / f)), f
    assert (tmp_path / "summ" / "args.json").exists() and (tmp_path / "summ" / "timings.json").exists()
    meta = json.loads((s / "summary.json").read_text())
    assert meta == {"count": 2, "burn_in": 2, "thin": 3}
    for stem in ("gcr-eor", "fg-amps"):
        samples = np.load(a / f"{stem}.npy")[2::3]
        assert rel(np.load(s / f"{stem}-mean.npy"), samples.mean(axis=0)) <= MEAN_TOL, stem
        assert rel(np.load(s / f"{stem}-var.npy"), samples.var(axis=0)) <= VAR_TOL, stem
