#!/usr/bin/env python
"""GCR solve between k_solve3's range and the dense-product solve: a config-3-like engine (128 baselines x 1024 times,
Philox, time-invariant flags, 4 sub-batches, 2-slot device ring) at (Nfreqs, Nmodes) = (448, 32) and (512, 32), i.e.
Np = 480 and 544, where the engine takes the resident round-1 k_solve (hp_solve.cu).

Prints one JSON line with, per shape,
  1. the device-resident Gibbs step time: host clock around eng.run(K) ending in a device synchronise, after warm-up,
     three windows;
  2. the "solve" class time per step from the engine's own CUDA-event timings (kernel_ms), in a separate profiled run
     with sub-batches off so that kernels do not overlap;
and the card's name and power limit, read with nvidia-smi in the same run.

    python profiles/scripts/solve_fallback_probe.py [--label TEXT]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

B, NT, NM = 128, 1024, 32
SHAPES = [(448, NM), (512, NM)]
SUBSTREAMS = 4
K, W, KP, WINDOWS = 10, 3, 3, 3


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    name, plim = (f.strip() for f in out[0].split(",")) if out else ("unknown", "unknown")
    return name, plim


def probe_shape(nf, nm, tstream):
    import torch
    import bench
    from hydra_pspec_b200 import pspec

    eng = pspec.GibbsEngine(B, NT, nf, nm, max_iters=K + W, rng="philox", cg_compat=False, refresh_omega=True,
                            keep=("cr", "fg", "chisq"), ring_iters=2, seed=1234, stream=tstream.cuda_stream,
                            substreams=SUBSTREAMS)
    eng.set_chain_ids(np.arange(B, dtype=np.int32))
    for ch in range(B):
        eng.load_chain(ch, *bench.make_baseline(ch, NT, nf, nm, flagged=True))

    def window(k):
        eng.rewind()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.run(k)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / k

    window(W)
    step_ms = [window(K) for _ in range(WINDOWS)]

    eng.set_substreams(1)
    window(W)
    eng.rewind()
    eng.set_profile(True)
    eng.kernel_ms(reset=True)
    eng.run(KP)
    kms = eng.kernel_ms(reset=True)
    eng.set_profile(False)
    bad = int(np.count_nonzero(eng.info()))
    eng.close()
    return {"nfreqs": nf, "nmodes": nm, "Np": 32 * ((nf + nm + 31) // 32),
            "step_ms": step_ms, "step_ms_median": float(np.median(step_ms)),
            "solve_ms_per_step": kms["solve"][0] / KP, "solve_launches_per_step": kms["solve"][1] / KP,
            "chains_with_bad_pivot": bad}


def main():
    import torch

    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--label", default="", help="free text copied into the JSON line (which build or setting ran)")
    opts = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("solve_fallback_probe.py: no CUDA device")
    name, plim = card()
    torch.cuda.set_device(0)
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    shapes = [probe_shape(nf, nm, tstream) for nf, nm in SHAPES]
    print(json.dumps({"probe": "solve_fallback", "label": opts.label, "device": name, "power_limit": plim,
                      "baselines": B, "ntimes": NT, "substreams": SUBSTREAMS, "steps_per_window": K, "shapes": shapes}))


if __name__ == "__main__":
    main()
