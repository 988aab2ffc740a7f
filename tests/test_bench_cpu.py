"""Host side of bench.py that needs no GPU: synthetic inputs, and the reference arm on the smallest configuration."""
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bench  # noqa: E402


def test_synthetic_inputs_are_deterministic_and_shaped():
    a = bench.make_baseline(5, 16, 32, 4)
    b = bench.make_baseline(5, 16, 32, 4)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    vis, flags, F, nd, l0 = a
    assert vis.shape == (16, 32) and flags.shape == (32,) and F.shape == (32, 4) and not flags.all()
    assert np.allclose(F.conj().T @ F, np.eye(4), atol=1e-12)
    assert bench.make_baseline(5, 16, 32, 4, flagged=False)[1].all()
    pt = bench.per_time_flags(5, flags, 16)
    assert pt.shape == (16, 32) and not np.any(pt[:, ~flags]) and len({r.tobytes() for r in pt}) > 1
    Ni = bench.dense_ninv(24)
    assert np.allclose(Ni, Ni.conj().T) and np.all(np.linalg.eigvalsh(Ni) > 0)


def test_every_config_names_its_metric_and_workload():
    for k in (0, 1, 2, 3, 4):
        assert "baseline-Gibbs-iterations/sec" in bench.metric_name(k)
        assert f"configs[{k}]" in bench.workload_name(k, 3)
    assert bench.metric_name(3) == bench.METRIC


def test_cpu_arm_runs_on_the_smallest_config():
    """One Gibbs iteration of configs[1] through the CPU arm's worker: the unmodified reference when baseline/_ref is
    installed (pip install --target, DESIGN.md), else the oracle port."""
    dt, kind = bench._cpu_worker((1, 3, 16, 1))
    assert dt > 0 and kind.split(" ")[0] in ("reference", "port")
    if (bench.ROOT / "baseline" / "_ref" / "hydra_pspec" / "pspec.py").is_file():
        assert kind.startswith("reference")


class _FakeEngine:
    """The read side of GibbsEngine at the configs[3] shape; every value encodes (chain, iteration)."""

    def __init__(self, B=128, T=1024, n=384, m=32):
        self.nchains, self.ntimes, self.nfreqs, self.nmodes = B, T, n, m

    def _fill(self, c, it, shape, dtype=np.float64):
        a = np.full(shape, 1000.0 * c + it, dtype=dtype)
        if np.iscomplexobj(a):
            a += 0.5j
        return a

    def signal_ps(self, c, it, k):
        return self._fill(c, it, (k, self.nfreqs))

    def ln_post(self, c, it, k):
        return self._fill(c, it, (k,))

    def signal_cr(self, c, it, k):
        return self._fill(c, it, (k, self.ntimes, self.nfreqs), np.complex128)

    def fg_amps(self, c, it, k):
        return self._fill(c, it, (k, self.ntimes, self.nmodes), np.complex128)

    def chisq(self, c, it, k):
        return self._fill(c, it, (k, self.ntimes, self.nfreqs))


def test_dump_outputs_writes_a_seeded_float64_sample_within_64_MB(tmp_path):
    eng = _FakeEngine()
    chains = bench.dump_outputs(eng, tmp_path / "a", 22)
    assert np.array_equal(chains, bench.dump_outputs(eng, tmp_path / "b", 22))
    assert 1 <= len(chains) < eng.nchains and np.all(np.diff(chains) > 0)
    files = {p.name: p for p in (tmp_path / "a").iterdir()}
    assert sorted(files) == sorted(f"{k}.npy" for k in ("signal_ps", "ln_post", "signal_cr", "fg_amps", "chisq"))
    assert sum(p.stat().st_size for p in files.values()) <= 64 * 2 ** 20
    out = {k[:-4]: np.load(p) for k, p in files.items()}
    assert all(a.dtype == np.float64 for a in out.values())
    assert np.array_equal(out["signal_ps"][:, 0], 1000.0 * np.arange(eng.nchains) + 22)
    assert np.array_equal(out["ln_post"], 1000.0 * np.arange(eng.nchains) + 22)
    assert out["signal_cr"].shape == (len(chains), 1024, 384, 2) and out["fg_amps"].shape == (len(chains), 1024, 32, 2)
    assert out["chisq"].shape == (len(chains), 1024, 384)
    assert np.array_equal(out["signal_cr"][:, 0, 0], np.stack([1000.0 * chains + 22, np.full(len(chains), 0.5)], axis=1))
    assert np.array_equal(out["chisq"][:, 5, 7], 1000.0 * chains + 22)


def test_steps_and_dump_arguments():
    assert bench.parse_args(["--steps", "7"]).steps == 7
    for bad in (["--steps", "0"], ["--config", "0", "--dump-outputs", "x"], ["--impl", "reference", "--dump-outputs", "x"]):
        with pytest.raises(SystemExit):
            bench.parse_args(bad)
