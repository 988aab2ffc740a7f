#!/usr/bin/env python
"""Cost of the on-device posterior summary (k_moments, hp_engine_set_summary) at the headline shape: 128 baselines x 1024
times x 384 channels x 32 foreground modes, Philox, time-invariant flags, 4 sub-batches (bench.py --config 3).

Prints one JSON line with
  1. the device-resident Gibbs step time without and with the summary (thin = 1), same engine (2-slot ring, the bench's
     set-up), the two settings alternated three times;
  2. k_moments' time per launch from a separate torch.profiler run (CUDA activities; its table is written under OUT_DIR),
     and the achieved bytes/s of the 64 B / complex element model (16 B sample read, 32 B mean read + write, 16 B M2
     read + write) as a fraction of the 7.7 TB/s data-sheet HBM bandwidth;
  3. end-to-end baseline-iterations/s for 64 iterations from pinned inputs: the full return set streamed to pinned host
     arrays (the bench's e2e call) against keep=() + summary through the engine, and through gibbs_sample_batch.
The card's name and power limit are read with nvidia-smi in the same run.

With --batch B (batch means, k_moments_batch) the JSON line also has
  4. the step time with batch means over B accumulated samples, alternated with the two settings of 1 (thin = 1, so one
     iteration in B closes a batch and runs k_moments_batch instead of k_moments);
  5. k_moments_batch's time per launch from a profiler run of its own (batch = 1: every launch closes a batch), against
     its 112 B / complex element model (the 64 B above, 32 B snapshot read + write, 16 B M2_bm read + write).

    python profiles/scripts/summary_probe.py [--batch B] [OUT_DIR]      (default: a new temporary directory)
"""
import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

B, NT, NF, NM = 128, 1024, 384, 32
SUBSTREAMS = 4
HBM_BYTES_PER_S = 7.7e12
BYTES_PER_ELEMENT = 64
BYTES_PER_ELEMENT_BATCH = 112


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    name, plim = (f.strip() for f in out[0].split(",")) if out else ("unknown", "unknown")
    return name, plim


def main():
    import torch
    import bench
    from hydra_pspec_b200 import _lib, pspec

    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("out_dir", nargs="?", default=None)
    ap.add_argument("--batch", type=int, default=0, help="also measure batch means over BATCH accumulated samples")
    opts = ap.parse_args()
    if opts.batch < 0:
        ap.error("--batch must be >= 0")
    if not torch.cuda.is_available():
        raise SystemExit("summary_probe.py: no CUDA device")
    out_dir = Path(opts.out_dir if opts.out_dir is not None else tempfile.mkdtemp(prefix="summary_probe_"))
    out_dir.mkdir(parents=True, exist_ok=True)
    name, plim = card()
    torch.cuda.set_device(0)
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    inputs = [bench.make_baseline(ch, NT, NF, NM, flagged=True) for ch in range(B)]

    # ---- 1. device-resident step time, summary off / on, alternated
    K, W = 10, 3
    eng = pspec.GibbsEngine(B, NT, NF, NM, max_iters=K, rng="philox", keep=("cr", "fg", "chisq"), ring_iters=2, seed=1234,
                            stream=tstream.cuda_stream, substreams=SUBSTREAMS)
    eng.set_chain_ids(np.arange(B, dtype=np.int32))
    for ch, (v, fl, F, nd, l0) in enumerate(inputs):
        eng.load_chain(ch, v, fl, F, nd, l0)

    def steps(on, k, batch=0):
        eng.rewind()
        eng.set_summary(("cr", "fg") if on else (), burn_in=0, thin=1, batch=batch)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.run(k)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k

    steps(False, W)
    steps(True, W)
    if opts.batch:
        steps(True, W, batch=1)   # every iteration launches k_moments_batch (first-launch module load)
    off_ms, on_ms, batch_ms = [], [], []
    for _ in range(3):
        off_ms.append(steps(False, K))
        on_ms.append(steps(True, K))
        if opts.batch:
            batch_ms.append(steps(True, K, batch=opts.batch))
    assert eng.summary(0)["count"] == K

    # ---- 2. k_moments per launch (profiler run of its own; sub-batches off so that kernels do not overlap)
    eng.set_substreams(1)
    steps(True, 2)
    from torch.profiler import ProfilerActivity, profile
    KP = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        steps(True, KP)
    durs = [ev.time_range.elapsed_us() for ev in prof.events() if "k_moments" in ev.name and str(ev.device_type).endswith("CUDA")]
    (out_dir / "summary_probe_profile.txt").write_text(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30))
    if opts.batch:
        # ---- 5. k_moments_batch per launch: batch = 1, so that every accumulated iteration closes a batch
        steps(True, 2, batch=1)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            steps(True, KP, batch=1)
        bdurs = [ev.time_range.elapsed_us() for ev in prof.events()
                 if "k_moments_batch" in ev.name and str(ev.device_type).endswith("CUDA")]
        (out_dir / "summary_probe_batch_profile.txt").write_text(
            prof.key_averages().table(sort_by="cuda_time_total", row_limit=30))
    eng.close()
    kmom_ms = float(np.mean(durs)) / 1e3 if durs else None
    bytes_per_launch = BYTES_PER_ELEMENT * B * NT * (NF + NM)   # one launch covers the whole batch here
    kmom = {"launches": len(durs), "ms_per_launch": kmom_ms, "bytes_per_launch": bytes_per_launch,
            "bytes_per_s": bytes_per_launch / (kmom_ms * 1e-3) if kmom_ms else None}
    kmom["fraction_of_7.7TBps"] = kmom["bytes_per_s"] / HBM_BYTES_PER_S if kmom_ms else None
    if opts.batch:
        kb_ms = float(np.mean(bdurs)) / 1e3 if bdurs else None
        kb_bytes = BYTES_PER_ELEMENT_BATCH * B * NT * (NF + NM)
        kbatch = {"launches": len(bdurs), "ms_per_launch": kb_ms, "bytes_per_launch": kb_bytes,
                  "bytes_per_s": kb_bytes / (kb_ms * 1e-3) if kb_ms else None}
        kbatch["fraction_of_7.7TBps"] = kbatch["bytes_per_s"] / HBM_BYTES_PER_S if kb_ms else None

    # ---- 3. end to end, 64 iterations from pinned inputs
    Ke, chunk = 64, 2
    pin = []
    for v, *_ in inputs:
        pv = _lib.pinned_empty(v.shape, np.complex128)
        pv[...] = v
        pin.append(pv)
    stage = {}

    def engine_call(keep, summary):
        e = pspec.GibbsEngine(B, NT, NF, NM, max_iters=Ke, rng="philox", keep=keep, ring_iters=3, seed=99,
                              stream=tstream.cuda_stream, substreams=SUBSTREAMS)
        e.set_chain_ids(np.arange(B, dtype=np.int32))
        if keep not in stage:
            stage[keep] = e.host_buffers(chunk, iter_major=True)
        for ch, (v, fl, F, nd, l0) in enumerate(inputs):
            e.load_chain(ch, pin[ch], fl, F, nd, l0)
        if summary:
            e.set_summary(("cr", "fg"), burn_in=0, thin=1)
        done = 0
        while done < Ke:
            n_ = min(chunk, Ke - done)
            e.run_to_host(n_, stage[keep], first_iter=done, iter_major=True, read_ahead=(2 if done + n_ < Ke else 0))
            done += n_
        if summary:
            for ch in range(B):
                e.summary(ch)
        e.close()

    bls = [dict(vis=pin[ch], flags=fl, S_initial=np.eye(NF), fgmodes=F, Ninv=np.diag(nd), ps_prior=None)
           for ch, (v, fl, F, nd, l0) in enumerate(inputs)]

    def batch_call():
        pspec.gibbs_sample_batch(bls, Niter=Ke, seed=99, rng="philox", keep=(), substreams=SUBSTREAMS,
                                 summary=dict(burn_in=0, thin=1))

    def rate(fn, reps=2):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return B * Ke * reps / (time.perf_counter() - t0)

    e2e = {"iterations": Ke,
           "full_return_set": rate(lambda: engine_call(("cr", "fg", "chisq"), False)),
           "summary_engine": rate(lambda: engine_call((), True)),
           "summary_gibbs_sample_batch": rate(batch_call),
           "unit": "baseline-iterations/s"}

    res = {"probe": "summary", "device": name, "power_limit": plim,
           "shape": {"baselines": B, "ntimes": NT, "nfreqs": NF, "nmodes": NM, "substreams": SUBSTREAMS},
           "step_ms_off": off_ms, "step_ms_on": on_ms,
           "step_ms_off_median": float(np.median(off_ms)), "step_ms_on_median": float(np.median(on_ms)),
           "step_overhead_ms": float(np.median(on_ms) - np.median(off_ms)),
           "step_overhead_fraction": float(np.median(on_ms) / np.median(off_ms) - 1.0),
           "k_moments": kmom, "e2e": e2e}
    if opts.batch:
        res.update({"batch": opts.batch, "step_ms_batch": batch_ms, "step_ms_batch_median": float(np.median(batch_ms)),
                    "batch_overhead_ms": float(np.median(batch_ms) - np.median(on_ms)),
                    "batch_overhead_fraction": float(np.median(batch_ms) / np.median(on_ms) - 1.0),
                    "k_moments_batch": kbatch})
    print(json.dumps(res))


if __name__ == "__main__":
    main()
