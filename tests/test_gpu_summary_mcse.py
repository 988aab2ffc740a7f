"""Batch-means Monte-Carlo standard errors and effective sample sizes of the on-device posterior means
(hp_engine_set_summary_batched / hp_engine_read_summary_mcse, k_moments_batch).  GPU only.  The numbers are compared with
numpy's batch means of the same chain's samples, read back from the device."""
import json

import numpy as np
import pytest

import test_gpu_summary as tgs
from test_gpu_summary import CASES, chain_inputs, make_engine, rel

pytestmark = pytest.mark.gpu

MCSE_TOL = 1e-9


def batch_means_ref(samples, b):
    """mcse, ess, nb of the mean of samples [k, ...] over batches of b (the definition in hp_engine_read_summary_mcse)."""
    k = samples.shape[0]
    nb = k // b
    if nb < 2:
        nan = np.full(samples.shape[1:], np.nan)
        return nan, nan.copy(), nb
    Y = samples[:nb * b].reshape((nb, b) + samples.shape[1:]).mean(axis=1)
    s2 = np.sum(np.abs(Y - Y.mean(axis=0)) ** 2, axis=0) / (nb - 1)
    mcse = np.sqrt(b * s2 / k)
    return mcse, samples.var(axis=0) / mcse ** 2, nb


def check_against(got, key, samples, b):
    mcse, ess, nb = batch_means_ref(samples, b)
    assert got["nbatch"] == nb and got["batch"] == b
    for name, want in (("mcse", mcse), ("ess", ess)):
        g = got[f"{key}_{name}"]
        assert g.shape == want.shape and g.dtype == np.float64, (key, name)
        assert np.array_equal(np.isnan(g), np.isnan(want)), (key, name)
        fin = ~np.isnan(want)
        assert rel(g[fin], want[fin]) <= MCSE_TOL, (key, name)


@pytest.mark.parametrize("case", list(CASES))
def test_mcse_matches_numpy(case):
    """5 chains in 2 sub-batches, 40 iterations, burn_in 3, thin 2, batch 4: k = 19 samples [3::2], 4 complete batches and
    a partial batch of 3."""
    eng = make_engine(niter=40, **CASES[case])
    try:
        eng.set_summary(("cr", "fg"), burn_in=3, thin=2, batch=4)
        eng.run(40)
        assert np.all(eng.info() == 0)
        for c in range(eng.nchains):
            got = eng.summary(c)
            assert got["count"] == 19 and got["nbatch"] == 4
            check_against(got, "signal_cr", eng.signal_cr(c)[3::2], 4)
            check_against(got, "fg_amps", eng.fg_amps(c)[3::2], 4)
    finally:
        eng.close()


def test_batch_means_change_nothing_else():
    """batch 0 against batch 3: bit-identical mean, var, chain and launch count."""
    out = []
    for batch in (0, 3):
        eng = make_engine(niter=20)
        eng.set_summary(("cr", "fg"), burn_in=1, thin=1, batch=batch)
        eng.run(20)
        got = [eng.summary(c) for c in range(eng.nchains)]
        assert ("nbatch" in got[0]) == (batch > 0)
        if batch:
            assert got[0]["nbatch"] == 6
        out.append(dict(mom=got, launches=eng.launch_count,
                        chain=[(eng.signal_ps(c), eng.ln_post(c), eng.signal_cr(c)) for c in range(eng.nchains)]))
        eng.close()
    off, on = out
    assert off["launches"] == on["launches"]
    for a, b in zip(off["mom"], on["mom"]):
        for k in a:
            assert np.array_equal(a[k], b[k]), k
    for a, b in zip(off["chain"], on["chain"]):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


def mcse_all(eng):
    return [{k: v for k, v in eng.summary(c).items() if k.endswith(("_mcse", "_ess")) or k in ("nbatch", "count")}
            for c in range(eng.nchains)]


def test_splitting_does_not_change_mcse():
    """run(40), run(7) + run(33), and run_to_host in chunks with read-ahead: bit-identical mcse, ess and nbatch."""
    from hydra_pspec_b200 import _lib
    kw = dict(burn_in=3, thin=2, batch=4)
    res = []
    eng = make_engine(niter=40)
    eng.set_summary(**kw)
    eng.run(40)
    res.append(mcse_all(eng))
    eng.close()

    eng = make_engine(niter=40)
    eng.set_summary(**kw)
    eng.run(7)
    eng.run(33)
    res.append(mcse_all(eng))
    eng.close()

    eng = make_engine(niter=40, ring_iters=3)
    eng.set_summary(**kw)
    stage = eng.host_buffers(6, iter_major=True)
    done = 0
    while done < 40:
        c = min(6, 40 - done)
        last = done + c >= 40
        eng.run_to_host(c, stage, first_iter=done, iter_major=True, read_ahead=0 if last else 2)
        done += c
        if not last:
            with pytest.raises(_lib.HydraLibError, match="read-ahead"):
                eng.summary(0)
    res.append(mcse_all(eng))
    eng.close()
    assert res[0][0]["nbatch"] == 4 and np.all(np.isfinite(res[0][0]["signal_cr_mcse"]))
    for other in res[1:]:
        for a, b in zip(res[0], other):
            assert a.keys() == b.keys()
            for k in a:
                assert np.array_equal(a[k], b[k]), k


def _read_mcse(L, eng, chain, what, mcse, ess, nbytes, nb):
    from hydra_pspec_b200 import _lib
    return L.hp_engine_read_summary_mcse(eng._h, chain, what, None if mcse is None else _lib.ptr(mcse),
                                         None if ess is None else _lib.ptr(ess), nbytes, nb)


def test_edges_and_refusals():
    from hydra_pspec_b200 import _lib
    L = _lib.lib()
    eng = make_engine(C=2, niter=12)
    try:
        T, n, m = eng.ntimes, eng.nfreqs, eng.nmodes
        assert L.hp_engine_set_summary_batched(eng._h, _lib.HP_SUMMARY_CR, 0, 1, -1) == -1   # HP_ERR_ARG
        assert L.hp_engine_set_summary_batched(eng._h, _lib.HP_SUMMARY_CR, 0, 0, 2) == -1
        # batch means off: refused, and summary() has no mcse keys
        eng.set_summary(("cr", "fg"), burn_in=0, thin=1)
        buf = np.empty((T, n))
        nb = _lib.C.c_int(-1)
        assert _read_mcse(L, eng, 0, _lib.HP_SUMMARY_CR, buf, buf, buf.nbytes, _lib.C.byref(nb)) == -1
        assert not any(k.endswith(("_mcse", "_ess")) or k in ("batch", "nbatch") for k in eng.summary(0))

        eng.set_summary(("cr",), burn_in=0, thin=1, batch=3)
        s = eng.summary(1)                                   # count = 0: nbatch 0, NaN
        assert s["count"] == 0 and s["nbatch"] == 0
        assert np.all(np.isnan(s["signal_cr_mcse"])) and np.all(np.isnan(s["signal_cr_ess"]))
        fgbuf = np.empty((T, m))
        assert _read_mcse(L, eng, 0, _lib.HP_SUMMARY_FG, fgbuf, fgbuf, fgbuf.nbytes, None) == -1   # not accumulated
        assert _read_mcse(L, eng, 2, _lib.HP_SUMMARY_CR, buf, buf, buf.nbytes, None) == -1         # chain out of range
        assert _read_mcse(L, eng, -1, _lib.HP_SUMMARY_CR, buf, buf, buf.nbytes, None) == -1
        assert _read_mcse(L, eng, 0, 3, buf, buf, buf.nbytes, None) == -1                          # two quantities
        small = np.empty((T, n - 1))
        assert _read_mcse(L, eng, 0, _lib.HP_SUMMARY_CR, small, None, small.nbytes, None) == -1    # too small
        assert _read_mcse(L, eng, 0, _lib.HP_SUMMARY_CR, None, small, small.nbytes, None) == -1
        nb = _lib.C.c_int(-1)
        assert _read_mcse(L, eng, 0, _lib.HP_SUMMARY_CR, None, None, 0, _lib.C.byref(nb)) == 0 and nb.value == 0

        eng.run(5)                                           # k = 5, nb = 1: NaN
        s = eng.summary(0)
        assert (s["count"], s["nbatch"]) == (5, 1)
        assert np.all(np.isnan(s["signal_cr_mcse"])) and np.all(np.isnan(s["signal_cr_ess"]))
        eng.run(1)                                           # k = 6, nb = 2: numbers
        s = eng.summary(0)
        assert (s["count"], s["nbatch"]) == (6, 2)
        check_against(s, "signal_cr", eng.signal_cr(0), 3)

        eng.gcr()                                            # not a Gibbs iteration: not accumulated
        s2 = eng.summary(0)
        eng.rewind()                                         # keeps the state
        s3 = eng.summary(0)
        for k in s:
            assert np.array_equal(s[k], s2[k], equal_nan=True) and np.array_equal(s[k], s3[k], equal_nan=True), k

        eng.set_summary(("cr", "fg"), burn_in=0, thin=1, batch=3)   # restart
        s = eng.summary(0)
        assert (s["count"], s["nbatch"]) == (0, 0) and np.all(np.isnan(s["fg_amps_mcse"]))
    finally:
        eng.close()

    # pending read-ahead iterations are refused
    eng = make_engine(C=2, niter=12, ring_iters=3)
    try:
        eng.set_summary(burn_in=0, thin=1, batch=1)
        stage = eng.host_buffers(2, iter_major=True)
        eng.run_to_host(2, stage, first_iter=0, iter_major=True, read_ahead=2)
        assert _read_mcse(L, eng, 0, _lib.HP_SUMMARY_CR, buf, buf, buf.nbytes, None) == -1
        eng.run_to_host(2, stage, first_iter=2, iter_major=True, read_ahead=0)
        assert _read_mcse(L, eng, 0, _lib.HP_SUMMARY_CR, buf, buf, buf.nbytes, None) == 0
        assert eng.summary(0)["nbatch"] == 4
    finally:
        eng.close()


def test_restart_zeroes_the_batch_means():
    """After a restart the numbers are those of the samples since the restart, as on a fresh engine."""
    eng = make_engine(niter=24)
    try:
        eng.set_summary(burn_in=0, thin=1, batch=2)
        eng.run(9)
        eng.set_summary(burn_in=1, thin=1, batch=3)   # restart: iterations 9 .. 23 are seen, 10 .. 23 accumulated
        eng.run(15)
        for c in range(eng.nchains):
            got = eng.summary(c)
            assert (got["count"], got["nbatch"]) == (14, 4)
            check_against(got, "signal_cr", eng.signal_cr(c)[10:], 3)
            check_against(got, "fg_amps", eng.fg_amps(c)[10:], 3)
    finally:
        eng.close()


def test_mcse_is_the_spread_of_independent_chain_means():
    """16 Philox chains of one baseline: the variance of the 16 chain means over the chain-average mcse^2 is about 1."""
    from hydra_pspec_b200 import pspec
    C, T, n, m = 16, 40, 96, 8
    eng = pspec.GibbsEngine(C, T, n, m, 300, rng="philox", keep=(), seed=11, substreams=2)
    try:
        eng.set_chain_ids(np.arange(1000, 1000 + C, dtype=np.int32))
        kw = chain_inputs(123, T, n, m)
        for c in range(C):
            eng.load_chain(c, **kw)
        eng.set_summary(("cr", "fg"), burn_in=50, thin=1, batch=25)
        eng.run(300)
        assert np.all(eng.info() == 0)
        got = [eng.summary(c) for c in range(C)]
        assert got[0]["count"] == 250 and got[0]["nbatch"] == 10
        ratios = {}
        for key in ("signal_cr", "fg_amps"):
            means = np.stack([g[f"{key}_mean"] for g in got])
            spread = np.var(means.real, axis=0, ddof=1) + np.var(means.imag, axis=0, ddof=1)
            mcse2 = np.mean(np.stack([g[f"{key}_mcse"] for g in got]) ** 2, axis=0)
            ratios[key] = spread / mcse2
        ratio = float(np.mean(np.concatenate([r.ravel() for r in ratios.values()])))
        print(f"spread of chain means / mcse^2: {ratio:.3f} "
              f"(signal_cr {np.mean(ratios['signal_cr']):.3f}, fg_amps {np.mean(ratios['fg_amps']):.3f})")
        assert 0.5 <= ratio <= 2.0, ratio
    finally:
        eng.close()


def test_batch_keep_nothing_returns_mcse(monkeypatch):
    """gibbs_sample_batch(keep=(), summary=dict(..., batch=3)) against numpy on a keep-everything run of the same seed."""
    from hydra_pspec_b200 import pspec
    T, n, m = 24, 64, 4
    bls = []
    for c in range(3):
        kw = chain_inputs(200 + c, T, n, m)
        bls.append(dict(vis=kw["vis"], flags=kw["flags"], S_initial=np.eye(n), fgmodes=kw["fgmodes"],
                        Ninv=np.diag(kw["ninv_diag"]), ps_prior=None))
    full = pspec.gibbs_sample_batch(bls, Niter=14, seed=5, rng="philox")
    monkeypatch.setenv("HP_HOST_BUDGET_GB", "1e-9")
    res = pspec.gibbs_sample_batch(bls, Niter=14, seed=5, rng="philox", keep=(), summary=dict(burn_in=2, thin=1, batch=3))
    for r, f in zip(res, full):
        mom = r[7]
        assert (mom["count"], mom["batch"], mom["nbatch"]) == (12, 3, 4)
        check_against(mom, "signal_cr", f[0][2:], 3)
        check_against(mom, "fg_amps", f[3][2:], 3)


@pytest.fixture(scope="module")
def td(tmp_path_factory):
    return tgs.materialize(tmp_path_factory.mktemp("testdata"))


@pytest.mark.parametrize("rng", ["philox", "numpy"])
def test_driver_mcse_files(td, tmp_path, rng):
    import run_hydra_pspec_b200 as drv
    base = tgs._set(tgs.driver_argv(td, tmp_path), "--Niter", "8") + ["--rng", rng]
    assert drv.main(tgs._set(base, "--dirname", "all")) == 0
    assert drv.main(tgs._set(base, "--dirname", "summ") + ["--samples", "summary", "--burn_in", "2", "--batch", "2"]) == 0
    a, s = tmp_path / "all" / "0-1", tmp_path / "summ" / "0-1"
    assert json.loads((s / "summary.json").read_text()) == {"count": 6, "burn_in": 2, "thin": 1, "batch": 2, "nbatch": 3}
    assert json.loads((tmp_path / "summ" / "args.json").read_text())["batch"] == 2
    for key, stem in (("signal_cr", "gcr-eor"), ("fg_amps", "fg-amps")):
        samples = np.load(a / f"{stem}.npy")[2:]
        got = {f"{key}_{q}": np.load(s / f"{stem}-{q}.npy") for q in ("mcse", "ess")}
        got.update(batch=2, nbatch=3)
        check_against(got, key, samples, 2)
        assert rel(np.load(s / f"{stem}-mean.npy"), samples.mean(axis=0)) <= tgs.MEAN_TOL, stem
