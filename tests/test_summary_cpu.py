"""Host side of the on-device posterior summary: driver arguments, validation of ``summary=``, device-budget arithmetic.
CPU only -- no compute entry point is called."""
import numpy as np
import pytest

import run_hydra_pspec_b200 as drv

# the driver's argument namespace before --samples / --burn_in / --thin existed
ARGS_BEFORE = {"Nfgmodes", "Niter", "Nproc", "ant_str", "clobber", "config", "dirname", "dpss_alpha", "fgmodes", "fgmodes_file",
               "file_paths", "flags", "flags_file", "freq_range", "map_estimate", "n_ps_prior_bins", "noise", "noise_cov",
               "noise_cov_file", "noise_file", "nsamples", "nsamples_file", "out_dir", "ps_prior_hi", "ps_prior_lo", "rng", "seed",
               "sigcov0", "sigcov0_file", "solver", "time_flags", "verbose", "write_Niter"}


def test_driver_samples_defaults():
    _, args = drv.parse_args(["x.uvh5"])
    d = vars(args)
    assert set(d) == ARGS_BEFORE | {"samples", "burn_in", "thin"}
    assert (d["samples"], d["burn_in"], d["thin"]) == ("all", 0, 1)
    _, args = drv.parse_args(["--samples", "summary", "--burn_in", "200", "--thin", "5", "x.uvh5"])
    assert (args.samples, args.burn_in, args.thin) == ("summary", 200, 5)
    with pytest.raises(SystemExit):
        drv.parse_args(["--samples", "mean", "x.uvh5"])


@pytest.mark.parametrize("bad", [["--burn_in", "-1"], ["--thin", "0"]])
def test_driver_refuses_bad_thinning(bad):
    with pytest.raises(SystemExit):
        drv.main(["--samples", "summary"] + bad + ["x.uvh5"])


def test_check_summary():
    from hydra_pspec_b200 import pspec
    assert pspec._check_summary(None) is None
    assert pspec._check_summary({}) == {"burn_in": 0, "thin": 1}
    assert pspec._check_summary(dict(burn_in=np.int64(3), thin=2)) == {"burn_in": 3, "thin": 2}
    for bad, exc in ((dict(thin=0), ValueError), (dict(burn_in=-1), ValueError), (dict(burn=1), ValueError),
                     (dict(thin=1.5), TypeError), (dict(burn_in=True), TypeError), ((1, 2), TypeError)):
        with pytest.raises(exc):
            pspec._check_summary(bad)


def test_sampling_functions_validate_summary_before_the_device():
    from hydra_pspec_b200 import pspec
    with pytest.raises(ValueError, match="thin"):
        pspec.gibbs_sample_with_fg(np.ones((4, 8), complex), np.ones(8, bool), np.eye(8), np.ones((8, 2)), np.eye(8),
                                   np.zeros((2, 8)), Niter=1, verbose=False, summary=dict(thin=0))
    bl = dict(vis=np.ones((4, 8), complex), flags=np.ones(8, bool), S_initial=np.eye(8), fgmodes=np.ones((8, 2)), Ninv=np.eye(8))
    with pytest.raises(ValueError, match="burn_in"):
        pspec.gibbs_sample_batch([bl], Niter=1, summary=dict(burn_in=-2))


@pytest.mark.parametrize("rng,general,dense,per_time", [("philox", False, False, False), ("numpy", True, False, False),
                                                        ("philox", False, True, False), ("philox", False, False, True)])
def test_device_budget_with_summary(rng, general, dense, per_time):
    """The posterior moments add a complex mean and a real M2 per (time, channel | mode) of a chain: 24 T (n + m) bytes."""
    from hydra_pspec_b200 import pspec
    T, n, m, niter = 1024, 384, 32, 100
    big = pspec._big_bytes_per_iter(1, T, n, m, ("cr", "fg", "chisq"))
    off = pspec._device_bytes_per_chain(T, n, m, niter, rng, big, general, dense, per_time, False)
    on = pspec._device_bytes_per_chain(T, n, m, niter, rng, big, general, dense, per_time, True)
    assert on - off == 24 * T * (n + m)
