"""bench.py --dump-outputs on the device: the last timed step of two runs with the same arguments is identical."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent


def test_dump_outputs_are_reproducible(tmp_path):
    outs = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--config", "1", "--steps", "4", "--warmup", "3",
                            "--no-cpu-baseline", "--no-e2e", "--no-parity", "--dump-outputs", str(tmp_path / run)],
                           capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 4 and line["dump_outputs"]["iteration"] == 3 + 4 - 1
        assert line["dump_outputs"]["sampled_chains"] == [0]
        outs.append({p.stem: np.load(p) for p in (tmp_path / run).glob("*.npy")})
    assert sorted(outs[0]) == ["chisq", "fg_amps", "ln_post", "signal_cr", "signal_ps"]
    for k, a in outs[0].items():
        assert a.dtype == np.float64 and np.all(np.isfinite(a)), k
        assert np.array_equal(a, outs[1][k]), k
    assert outs[0]["signal_cr"].shape == (1, 64, 128, 2) and outs[0]["signal_ps"].shape == (1, 128)
