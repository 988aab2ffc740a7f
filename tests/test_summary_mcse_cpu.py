"""Host side of the batch-means Monte-Carlo standard errors of the on-device posterior means: the driver's --batch,
validation of ``summary=dict(batch=...)``, device-budget arithmetic and the summary files.  CPU only -- no compute entry
point is called."""
import json

import numpy as np
import pytest
import yaml

import run_hydra_pspec_b200 as drv


def test_driver_batch_absent_unless_given():
    _, args = drv.parse_args(["--samples", "summary", "x.uvh5"])
    assert "batch" not in vars(args)
    _, args = drv.parse_args(["--samples", "both", "--batch", "7", "x.uvh5"])
    assert args.batch == 7


@pytest.mark.parametrize("argv", [["--batch", "4"],                                   # --samples all (the default)
                                  ["--samples", "all", "--batch", "4"],
                                  ["--samples", "summary", "--batch", "0"],
                                  ["--samples", "both", "--batch", "-3"]])
def test_driver_refuses_batch(argv):
    with pytest.raises(SystemExit):
        drv.main(argv + ["x.uvh5"])


def test_driver_batch_from_config_file(tmp_path):
    cfg = tmp_path / "config.yaml"
    cfg.write_text(yaml.safe_dump({"samples": "summary", "batch": 5}))
    _, args = drv.parse_args(["--config", str(cfg), "x.uvh5"])
    assert (args.samples, args.batch) == ("summary", 5)
    _, args = drv.parse_args(["--config", str(cfg), "--batch", "9", "x.uvh5"])   # the command line wins
    assert args.batch == 9
    cfg.write_text(yaml.safe_dump({"batch": 5}))
    with pytest.raises(SystemExit):
        drv.main(["--config", str(cfg), "x.uvh5"])                                # still needs --samples summary / both


def test_check_summary_batch():
    from hydra_pspec_b200 import pspec
    assert pspec._check_summary({}) == {"burn_in": 0, "thin": 1}
    assert pspec._check_summary(dict(batch=0)) == {"burn_in": 0, "thin": 1, "batch": 0}
    assert pspec._check_summary(dict(burn_in=2, batch=np.int32(4))) == {"burn_in": 2, "thin": 1, "batch": 4}
    assert type(pspec._check_summary(dict(batch=np.int64(3)))["batch"]) is int
    for bad, exc in ((dict(batch=-1), ValueError), (dict(batch=True), TypeError), (dict(batch=2.0), TypeError),
                     (dict(batch="2"), TypeError), (dict(batches=2), ValueError)):
        with pytest.raises(exc):
            pspec._check_summary(bad)


@pytest.mark.parametrize("rng,general,dense,per_time", [("philox", False, False, False), ("numpy", True, False, False),
                                                        ("philox", False, True, False), ("philox", False, False, True)])
def test_device_budget_with_batch_means(rng, general, dense, per_time):
    """Batch means add a complex snapshot and a real M2_bm per (time, channel | mode) of a chain: 24 T (n + m) bytes."""
    from hydra_pspec_b200 import pspec
    T, n, m, niter = 1024, 384, 32, 100
    big = pspec._big_bytes_per_iter(1, T, n, m, ())
    args = (T, n, m, niter, rng, big, general, dense, per_time)
    on = pspec._device_bytes_per_chain(*args, True)
    assert pspec._device_bytes_per_chain(*args, True, batch=False) == on
    assert pspec._device_bytes_per_chain(*args, True, batch=True) - on == 24 * T * (n + m)


def _moments(T=3, n=5, m=2, batch=False):
    rng = np.random.default_rng(0)
    mom = {"count": 9}
    for key, w in (("signal_cr", n), ("fg_amps", m)):
        mom[f"{key}_mean"] = rng.standard_normal((T, w)) + 1j * rng.standard_normal((T, w))
        mom[f"{key}_var"] = rng.random((T, w))
    if batch:
        for key, w in (("signal_cr", n), ("fg_amps", m)):
            mom[f"{key}_mcse"] = rng.random((T, w))
            mom[f"{key}_ess"] = rng.random((T, w)) * 9
        mom.update(batch=4, nbatch=2)
    return mom


def test_write_summary_files_without_batch_unchanged(tmp_path):
    from hydra_pspec_b200 import utils
    mom = _moments()
    utils.write_summary_files(tmp_path, mom, burn_in=2, thin=3)
    assert sorted(p.name for p in tmp_path.iterdir()) == ["fg-amps-mean.npy", "fg-amps-var.npy", "gcr-eor-mean.npy",
                                                          "gcr-eor-var.npy", "summary.json"]
    assert (tmp_path / "summary.json").read_text() == json.dumps({"count": 9, "burn_in": 2, "thin": 3}, indent=2)
    # batch=0 is "off": byte for byte the same output
    off = tmp_path / "off"
    off.mkdir()
    utils.write_summary_files(off, _moments(batch=True), burn_in=2, thin=3, batch=0)
    for p in tmp_path.iterdir():
        if p.is_file():
            assert (off / p.name).read_bytes() == p.read_bytes(), p.name
    assert sorted(p.name for p in off.iterdir()) == sorted(p.name for p in tmp_path.iterdir() if p.is_file())


def test_write_summary_files_with_batch(tmp_path):
    from hydra_pspec_b200 import utils
    mom = _moments(batch=True)
    utils.write_summary_files(tmp_path, mom, burn_in=2, thin=3, batch=4)
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(
        [f"{s}-{q}.npy" for s in ("gcr-eor", "fg-amps") for q in ("mean", "var", "mcse", "ess")] + ["summary.json"])
    assert json.loads((tmp_path / "summary.json").read_text()) == {"count": 9, "burn_in": 2, "thin": 3, "batch": 4,
                                                                   "nbatch": 2}
    for key, stem in (("signal_cr", "gcr-eor"), ("fg_amps", "fg-amps")):
        for q in ("mean", "var", "mcse", "ess"):
            assert np.array_equal(np.load(tmp_path / f"{stem}-{q}.npy"), mom[f"{key}_{q}"]), (stem, q)
