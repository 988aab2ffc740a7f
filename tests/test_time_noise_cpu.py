"""Per-time diagonal noise, host side: the oracle's semantics, the split of a 3-D Ninv (pspec._time_noise_model), the
driver's --noise_weights and the device-budget estimate.  CPU only -- no compute entry point is called."""
import argparse

import numpy as np
import pytest

from oracle import hydra_oracle as ho
import time_noise_oracle as tno


def crandn(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def make_case(nt, nf, nm, seed):
    rng = np.random.default_rng(seed)
    F = np.linalg.qr(crandn(rng, nf, nm))[0]
    fop = ho.fourier_operator(nf)
    S0 = fop.conj().T @ np.diag((0.5 + rng.random(nf)) / nf ** 2) @ fop
    vis = crandn(rng, nt, nf) + (4 * crandn(rng, nt, nm)) @ F.T
    prior = np.zeros((2, nf))
    prior[0, nf // 2] = 40.0
    prior[1, nf // 2] = 0.2
    draws = (crandn(rng, nt, nf), crandn(rng, nt, nf), rng.random((3, nf)))
    return rng, vis, S0, F, prior, draws


@pytest.mark.parametrize("solver", ["direct", "cg"])
@pytest.mark.parametrize("per_time_flags", [False, True])
def test_identical_slices_equal_2d_oracle(solver, per_time_flags):
    rng, vis, S0, F, prior, draws = make_case(5, 24, 3, 1)
    ninv = 1.0 + rng.random(24)
    flags = rng.random((5, 24)) > 0.15 if per_time_flags else rng.random(24) > 0.15
    a = ho.gibbs_sample_with_fg(vis, flags, S0, F, np.diag(ninv), prior, Niter=3, solver=solver, draws=draws)
    b = tno.gibbs_sample_with_fg(vis, flags, S0, F, tno.diag_stack(np.tile(ninv, (5, 1))), prior, Niter=3, solver=solver,
                                 draws=draws)
    for x, y in zip(a, b):
        if solver == "cg" or per_time_flags:   # the same per-time solves: bit for bit
            np.testing.assert_array_equal(x, y)
        else:                                  # one LU for all times (2-D) vs one solve per time
            np.testing.assert_allclose(y, x, rtol=1e-12, atol=1e-12 * np.max(np.abs(x)))


def test_per_time_solve_is_reference_system():
    """Each time's GCR solution is np.linalg.solve of the reference's A_t with that time's Ninv[t] and flags."""
    rng, vis, S0, F, prior, draws = make_case(6, 20, 2, 2)
    flags = rng.random((6, 20)) > 0.2
    ninv_t = (0.5 + rng.random((6, 20))) * (rng.random((6, 20)) > 0.1)
    Ninv = tno.diag_stack(ninv_t)
    oma, omb, u = draws
    out = tno.gibbs_step_fgmodes(vis * flags, flags, S0, F, Ninv, prior, oma, omb, u[0])
    for t in range(6):
        m = ho.build_matrices(flags[t], S0, Ninv[t], F, need_pinv=False)
        b = ho.gcr_rhs(vis[t] * flags[t], flags[t], m, F, oma[t], omb[t])
        x = np.linalg.solve(m["A"], b)
        np.testing.assert_allclose(out[0][t], x[:20], rtol=0, atol=1e-12 * np.max(np.abs(x)))
        np.testing.assert_allclose(out[3][t], x[20:], rtol=0, atol=1e-12 * np.max(np.abs(x)))
    # chi^2 weights per time
    resid = vis * flags - out[0] - out[3] @ F.T
    np.testing.assert_allclose(out[4], np.abs(resid) ** 2 * ninv_t, rtol=1e-14)


def test_time_noise_model_split():
    from hydra_pspec_b200 import pspec
    T, n = 4, 6
    rng = np.random.default_rng(3)
    flags1 = rng.random(n) > 0.3
    ninv = np.diag(1.0 + rng.random(n))
    # 2-D: untouched
    N2, f2, nt = pspec._time_noise_model(ninv, flags1, T, n)
    assert nt is None and np.array_equal(N2, ninv) and f2 is flags1
    # identical slices: the 2-D matrix, flags as given
    N2, f2, nt = pspec._time_noise_model(np.stack([ninv] * T), flags1, T, n)
    assert nt is None and np.array_equal(N2, ninv) and f2 is flags1
    # diagonal slices: per-time weights, 1-D flags broadcast
    w = rng.random((T, n))
    w[1, 2] = 0.0
    N2, f2, nt = pspec._time_noise_model(tno.diag_stack(w), flags1, T, n)
    assert N2 is None and nt.dtype == np.float64 and np.array_equal(nt, w)
    assert f2.shape == (T, n) and np.array_equal(f2, np.broadcast_to(flags1, (T, n)))
    # per-time flags pass through
    flags2 = rng.random((T, n)) > 0.3
    _, f2, _ = pspec._time_noise_model(tno.diag_stack(w), flags2, T, n)
    assert np.array_equal(f2, flags2)
    # non-diagonal slice
    bad = tno.diag_stack(w)
    bad[2, 0, 1] = bad[2, 1, 0] = 0.1
    with pytest.raises(NotImplementedError):
        pspec._time_noise_model(bad, flags1, T, n)
    # negative, non-finite, complex diagonals
    for v in (-1.0, np.nan, np.inf):
        bad = tno.diag_stack(w)
        bad[3, 4, 4] = v
        with pytest.raises(ValueError):
            pspec._time_noise_model(bad, flags1, T, n)
    bad = tno.diag_stack(w).astype(complex)
    bad[0, 0, 0] += 1e-3j
    with pytest.raises(ValueError):
        pspec._time_noise_model(bad, flags1, T, n)
    # wrong leading dimension
    with pytest.raises(ValueError):
        pspec._time_noise_model(tno.diag_stack(w[:3]), flags1, T, n)


def test_time_noise_refused_with_reference_cg():
    """solver='reference-cg' has no per-time counterpart in the reference; refused before any device call."""
    from hydra_pspec_b200 import pspec
    with pytest.raises(NotImplementedError):
        pspec._check_per_time_supported("reference-cg", None, None)


def test_device_budget_time_noise():
    from hydra_pspec_b200 import pspec
    args = (512, 256, 16, 100, "philox", 3 * 2 ** 20, False, False, True, False)
    base = pspec._device_bytes_per_chain(*args)
    assert pspec._device_bytes_per_chain(*args, time_noise=False) == base
    assert pspec._device_bytes_per_chain(*args, time_noise=True) == base + 8 * 512 * 256
    args = (37, 96, 8, 10, "numpy", 2 ** 20, False, False, False, True)
    assert pspec._device_bytes_per_chain(*args, batch=True, time_noise=True) == \
        pspec._device_bytes_per_chain(*args, batch=True) + 8 * 48 * 96


def _driver_args(**kw):
    base = dict(flags=None, flags_file=None, nsamples="ns.npy", nsamples_file=None, noise=None, noise_file=None,
                sigcov0=None, sigcov0_file=None, noise_cov=None, noise_cov_file=None, fgmodes=None, fgmodes_file=None,
                dpss_alpha=None, Nfgmodes=2, noise_weights="nsamples")
    base.update(kw)
    return argparse.Namespace(**base)


def test_driver_builds_ninv_t_from_nsamples(tmp_path, monkeypatch):
    import run_hydra_pspec_b200 as drv
    T, n = 5, 16
    rng = np.random.default_rng(4)
    nsamples = rng.integers(0, 4, size=(T, n)).astype(float)
    np.save(tmp_path / "ns.npy", nsamples)
    monkeypatch.chdir(tmp_path)
    freqs = np.linspace(100e6, 110e6, n)
    d = crandn(rng, T, n)
    get = lambda ap: (d, np.zeros((T, n), dtype=bool))  # noqa: E731
    out = drv.assemble_baselines(_driver_args(), [(0, 1)], freqs, get, tmp_path)
    ninv = np.real(np.diagonal(out[0]["Ninv"]))
    np.testing.assert_array_equal(out[0]["ninv_t"], nsamples * ninv[None, :])
    full = drv.time_noise_ninv(out[0]["ninv_t"])
    assert full.shape == (T, n, n)
    for t in range(T):
        np.testing.assert_array_equal(full[t], np.diag(nsamples[t] * ninv))
    # without --noise_weights: no per-time weights, today's behaviour
    out = drv.assemble_baselines(_driver_args(noise_weights="none"), [(0, 1)], freqs, get, tmp_path)
    assert out[0]["ninv_t"] is None


def test_driver_noise_weights_option():
    import run_hydra_pspec_b200 as drv
    _, args = drv.parse_args(["x.uvh5"])
    assert not hasattr(args, "noise_weights")   # default: none (one Ninv for all times)
    _, args = drv.parse_args(["--noise_weights", "nsamples", "--nsamples", "ns.npy", "x.uvh5"])
    assert args.noise_weights == "nsamples"
    with pytest.raises(SystemExit):
        drv.parse_args(["--noise_weights", "rms", "x.uvh5"])
    with pytest.raises(SystemExit):   # needs --nsamples
        drv.main(["--noise_weights", "nsamples", "x.uvh5"])
    with pytest.raises(SystemExit):   # needs a diagonal Ninv
        drv.main(["--noise_weights", "nsamples", "--nsamples", "ns.npy", "--noise_cov", "nc.npy", "x.uvh5"])
