"""Step time of per-time diagonal noise at the configs[2] shape (128 baselines x 512 times, Nfreqs 256, Nmodes 16), one GPU.

  (a) per-time flags, one factorisation per time (force_dense_solve);
  (b) the same flags plus nsamples weights that change only where the flags change (the same factorisations as (a));
  (c) weights that change at every time (one factorisation per time, no re-use).

The three engines are resident together; after a warm-up the cases are timed in turn, three rounds, each a host clock
around `steps` Gibbs iterations that ends in a device synchronisation.  Prints one JSON line (also written to --out) with
the card name and power limit read in the same run.

    python profiles/scripts/time_noise_probe.py --out time_noise_probe.json
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[2]))
from hydra_pspec_b200 import pspec  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out
    except Exception as exc:  # noqa: BLE001
        return f"unknown ({exc})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nbl", type=int, default=128)
    ap.add_argument("--ntimes", type=int, default=512)
    ap.add_argument("--nfreqs", type=int, default=256)
    ap.add_argument("--nmodes", type=int, default=16)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    C, T, n, m = a.nbl, a.ntimes, a.nfreqs, a.nmodes
    rng = np.random.default_rng(0)
    F = np.linalg.qr(rng.standard_normal((n, m)) + 1j * rng.standard_normal((n, m)))[0]
    lam0sq = np.full(n, 1.0 / n)
    ninv = np.full(n, 1.0 / 100.0)
    seg = 16                                   # flags (and the weights of case b) change every 16 times
    nseg = (T + seg - 1) // seg
    engines = {}
    for case in ("a", "b", "c"):
        engines[case] = pspec.GibbsEngine(C, T, n, m, max_iters=a.steps, rng="philox", keep=(), seed=1, time_flags=True,
                                          force_dense_solve=True, substreams=4)
    for c in range(C):
        vis = (rng.standard_normal((T, n)) + 1j * rng.standard_normal((T, n))) * 0.1
        flags = np.ones((T, n), dtype=bool)
        flags[:, rng.choice(n, 8, replace=False)] = False                    # persistent RFI
        segflag = rng.random((nseg, n)) > 0.03                                # intermittent RFI, per segment
        flags &= np.repeat(segflag, seg, axis=0)[:T]
        nseg_w = np.repeat(1.0 + rng.integers(0, 4, size=(nseg, n)), seg, axis=0)[:T]
        engines["a"].load_chain(c, vis, flags, F, ninv, lam0sq)
        engines["b"].load_chain(c, vis, flags, F, None, lam0sq, ninv_t=nseg_w * ninv[None, :])
        engines["c"].load_chain(c, vis, flags, F, None, lam0sq, ninv_t=(0.5 + 3.0 * rng.random((T, n))) * ninv[None, :])
    for eng in engines.values():   # warm-up: every shape once
        eng.run(a.steps)
        eng.sync()
    times = {k: [] for k in engines}
    for _ in range(a.rounds):
        for k, eng in engines.items():
            eng.rewind()
            t0 = time.perf_counter()
            eng.run(a.steps)
            eng.sync()
            times[k].append((time.perf_counter() - t0) / a.steps * 1e3)
    for k, eng in engines.items():
        assert np.all(eng.info() == 0), k
        assert eng.pt_form()[0] == "direct", k
        eng.close()
    res = {"card": card(), "shape": dict(nbl=C, ntimes=T, nfreqs=n, nmodes=m), "steps_per_sample": a.steps,
           "step_ms": {k: [round(v, 2) for v in vs] for k, vs in times.items()},
           "step_ms_median": {k: round(float(np.median(vs)), 2) for k, vs in times.items()}}
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
