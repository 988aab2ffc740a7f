#!/usr/bin/env python
"""bench.py -- baseline-Gibbs-iterations/sec of the BASELINE.json configurations (default: configs[3], the headline).

    python bench.py [--config K] --gpus N --steps K --warmup W        (N>1: launched under torch.distributed.run)
    python bench.py --impl reference [--config K] --gpus N --steps K --warmup W

A "step" is one Gibbs iteration (GCR solve for all times + power-spectrum draw) of every baseline resident on the GPU.
One JSON line is printed by rank 0.

  --config 3 (default)  HERA-like: Nfreq=384, Ntimes=1024, Nfg=32, 1024 baselines / 8 GPUs = 128 per GPU (weak scaling)
  --config 1            one baseline, Nfreq=128, Ntimes=64, Nfg=8, no flags (every GPU runs a replica)
  --config 2            128 baselines in total, Nfreq=256, Ntimes=512, Nfg=16, per-time RFI flags (strong scaling)
  --config 4            Nfreq=1024, Nfg=64, Ntimes=1024, dense noise covariance, 32 baselines per GPU (weak scaling)
  --config 0            the reference's test_data run through the driver (run_hydra_pspec_b200.py), one baseline

`--impl reference` runs the UNMODIFIED reference (baseline/_ref: `pip install --target` of /root/reference, see DESIGN.md)
on the host cores, one single-threaded process per core (the layout of `mpirun -n <cores> run-hydra-pspec.py`).

`--dump-outputs DIR` (configs 1-4) writes what the last timed step computed as float64 DIR/<name>.npy, so that two builds
can be compared output for output (the inputs and the Philox draws are seeded): signal_ps and ln_post of every chain on
rank 0, and signal_cr, fg_amps and chisq (complex arrays with a trailing (real, imag) axis) of a fixed, seeded sample of
its chains, as many as fit in 64 MB in all.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "baseline-Gibbs-iterations/sec at Nfreq=384, Ntimes=1024, Nfg=32 on 1/8 B200"
UNIT = "baseline-iterations/s"
FP64_PEAK_NOMINAL_TFLOPS = 37.2  # 148 SMs x 64 FP64 FMA/clk x 2 x 1.965 GHz

# BASELINE.json configs[k]: shape, baselines, engine mode, default steps
CONFIGS = {
    1: dict(nt=64, nf=128, nm=8, per_gpu=1, total=None, mode="std", flags=False, scaling="replicas", steps=200,
            what="single synthetic baseline, diagonal noise, no flags (one replica per GPU)"),
    2: dict(nt=512, nf=256, nm=16, per_gpu=None, total=128, mode="pertime", flags=True, scaling="strong", steps=40,
            what="128 baselines in total, a different random RFI mask at every time (in-painting: every time has its own GCR system)"),
    3: dict(nt=1024, nf=384, nm=32, per_gpu=128, total=None, mode="std", flags=True, scaling="weak", steps=20,
            what="HERA-like, 128 baselines per GPU (1024 / 8), time-invariant flags (5 %), diagonal noise"),
    4: dict(nt=1024, nf=1024, nm=64, per_gpu=32, total=None, mode="dense", flags=True, scaling="weak", steps=10,
            what="stress case, full non-diagonal noise covariance, 32 baselines per GPU (256 / 8)"),
}


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[0, 1, 2, 3, 4])
    ap.add_argument("--baselines-per-gpu", type=int, default=None)
    ap.add_argument("--e2e-iters", type=int, default=64)   # the set-up of the call (create + load_chain, ~0.1 s) is inside the timed region
    ap.add_argument("--substreams", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None)
    a = ap.parse_args(argv)
    if a.steps is not None and a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.config == 0):
        ap.error("--dump-outputs needs --impl b200 and --config 1..4")
    return a


# ------------------------------------------------------------------------------------------------
def make_baseline(seed, nt, nf, nm, flagged=True):
    """Synthetic HERA-like baseline: flat-ish EoR delay spectrum, smooth foreground modes with a
    steep amplitude spectrum, white noise, ~5 % of the channels flagged at all times."""
    rng = np.random.default_rng(seed)
    x = np.linspace(-1.0, 1.0, nf)
    F = np.linalg.qr(np.polynomial.legendre.legvander(x, nm - 1))[0].astype(np.complex128)
    crandn = lambda *s: (rng.standard_normal(s) + 1j * rng.standard_normal(s)) / np.sqrt(2)  # noqa: E731
    eor = crandn(nt, nf)
    amps = crandn(nt, nm) * np.logspace(3, 0, nm)
    sigma = 0.5
    vis = eor + amps @ F.T + sigma * crandn(nt, nf)
    flags = np.ones(nf, dtype=bool)
    if flagged:
        flags[rng.choice(nf, max(1, nf // 20), replace=False)] = False
    ninv_diag = np.full(nf, 1.0 / sigma ** 2)
    lam0sq = np.ones(nf)  # S_initial = identity (run-hydra-pspec.py:425)
    return vis, flags, F, ninv_diag, lam0sq


def per_time_flags(seed, flags, nt):
    """configs[2]: the time-invariant mask AND a different random 5 % mask at every time."""
    nf = flags.size
    return np.broadcast_to(flags, (nt, nf)) & (np.random.default_rng(1000 + seed).random((nt, nf)) > 0.05)


def dense_ninv(nf):
    """configs[4]: inverse of a full noise covariance of the calc-vis-cov-matrices.py form (sample covariance + ridge)."""
    rng = np.random.default_rng(99)
    Xn = (rng.standard_normal((nf, 2 * nf)) + 1j * rng.standard_normal((nf, 2 * nf))) / np.sqrt(2)
    return np.linalg.inv(0.25 * (Xn @ Xn.conj().T / (2 * nf) + 0.2 * np.eye(nf)))


DUMP_BYTES = 64 * 2 ** 20


def dump_outputs(eng, out_dir, it):
    """--dump-outputs: iteration `it` of every output the engine keeps, as float64 .npy files under `out_dir` (module
    docstring).  Returns the indices of the chains whose signal_cr / fg_amps / chisq were written."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    B, T, n, m = eng.nchains, eng.ntimes, eng.nfreqs, eng.nmodes
    out = {"signal_ps": np.stack([eng.signal_ps(c, it, 1)[0] for c in range(B)]),
           "ln_post": np.concatenate([eng.ln_post(c, it, 1) for c in range(B)])}
    per_chain = 8 * T * (2 * n + 2 * m + n)   # signal_cr + fg_amps + chisq of one chain
    room = DUMP_BYTES - sum(a.nbytes for a in out.values())
    chains = np.sort(np.random.default_rng(0).choice(B, min(B, room // per_chain), replace=False))
    for name in ("signal_cr", "fg_amps", "chisq"):
        out[name] = np.stack([getattr(eng, name)(int(c), it, 1)[0] for c in chains])
    for name, a in out.items():
        if np.iscomplexobj(a):
            a = np.ascontiguousarray(a).view(np.float64).reshape(a.shape + (2,))
        np.save(out_dir / f"{name}.npy", a)
    return chains


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.stop = index, [], threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([f.strip() for f in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=3)

    def summary(self):
        sm = sorted(float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 3 + i and s[3 + i].lower() == "active" for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "power_w_max": max(float(s[2]) for s in self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU side: the unmodified reference (baseline/_ref), or -- where it has no such code path -- the oracle port
def load_reference():
    """hydra_pspec from baseline/_ref (unmodified; pyuvdata / astropy are not installed in this image and are only used
    by the reference's uvh5 helpers, so they are stubbed).  None when baseline/_ref is absent."""
    ref = ROOT / "baseline" / "_ref"
    if not (ref / "hydra_pspec" / "pspec.py").is_file():
        return None
    for name in ["pyuvdata", "pyuvdata.utils", "astropy", "astropy.units"]:
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["pyuvdata"].UVData = type("UVData", (), {})
    sys.modules["pyuvdata"].utils = sys.modules["pyuvdata.utils"]
    sys.modules["astropy"].units = sys.modules["astropy.units"]
    sys.modules["astropy.units"].Quantity = type("Quantity", (), {})
    if str(ref) not in sys.path:
        sys.path.insert(0, str(ref))
    try:
        import hydra_pspec
    except Exception:  # noqa: BLE001
        return None
    # gcr_fgmodes (pspec.py:285) maps its per-time solves over `multiprocess.Pool(nproc)`; with nproc = 1 that is a serial map
    # in one child process.  On this image Pool.__exit__ sporadically blocks for minutes (profiles/r2_reference_pool_stall.txt:
    # 635 s for 16 times, 2 s for 64), so the benchmark arm maps in-process instead; every solve is still the reference's
    # gcr_fgmodes_1d.  This replaces a runtime object of the imported module, not its source.
    hydra_pspec.pspec.Pool = _SerialPool
    return hydra_pspec


class _SerialPool:
    """Stand-in for multiprocess.Pool(1): `with Pool(1) as pool: pool.map(f, xs)` evaluated in-process."""

    def __init__(self, *a, **kw):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def map(self, f, xs):
        return [f(x) for x in xs]


def _cpu_worker(job):
    """One baseline on one core: `niter` Gibbs iterations, each restarting from S_initial = I (the per-iteration cost of the
    reference's algorithm -- 2 x sqrtm, pinv, Ntimes preconditioned CG solves -- without the risk of its CG stagnating
    for 1e5 iterations per time on a later, coloured S sample; DESIGN.md section 1).  Returns (seconds, kind)."""
    import warnings
    cfg_id, seed, nt_sample, niter = job
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    c = CONFIGS[cfg_id]
    nf, nm = c["nf"], c["nm"]
    vis, flags, F, ninv_diag, _ = make_baseline(seed, nt_sample, nf, nm, flagged=c["flags"])
    Ninv = dense_ninv(nf) if c["mode"] == "dense" else np.diag(ninv_diag)
    prior = np.zeros((2, nf))
    hp = load_reference() if c["mode"] != "pertime" else None   # the reference asserts 1-D flags (pspec.py:428)
    kind = "reference" if hp is not None else "port"
    if hp is not None and not np.all(flags):
        # build_matrices (pspec.py:362) takes scipy's sqrtm of the flagged N^-1; with this image's scipy that is NaN for most
        # masks with several flagged channels -- the reference's whole chain is then NaN and every CG runs its 1e5 iterations
        # (~30 s per time).  The unmodified reference is therefore timed on the same baseline without flags: same shapes, same
        # dense operations per iteration.
        import scipy.linalg
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            fl = flags.astype(float)
            if not np.all(np.isfinite(scipy.linalg.sqrtm((fl * Ninv * fl).astype(complex)))):
                flags = np.ones(nf, dtype=bool)
                kind = "reference (unflagged: scipy sqrtm of its flagged N^-1 is NaN)"
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if hp is not None:
            for it in range(niter):
                hp.pspec.gibbs_sample_with_fg(vis.copy(), flags.copy(), np.eye(nf, dtype=complex), F, Ninv, prior, Niter=1,
                                              seed=seed + it, verbose=False, nproc=1)
        else:
            from oracle import hydra_oracle as ho
            fl = per_time_flags(seed, flags, nt_sample) if c["mode"] == "pertime" else flags
            for it in range(niter):
                ho.gibbs_sample_with_fg(vis, fl, np.eye(nf), F, Ninv, prior, Niter=1, seed=seed + it, solver="cg")
    return time.perf_counter() - t0, kind


def cpu_throughput(cfg_id, steps, warmup):
    """baseline-iterations/s of the CPU implementation on all host cores: `cores` baselines x `steps` iterations.  configs[2]
    and configs[4] use a bounded sample of the times (the cost per baseline-iteration is linear in Ntimes once the operators
    are built; the operator build is charged in full)."""
    import multiprocessing as mp
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):   # before the workers import numpy
        os.environ[k] = "1"
    c = CONFIGS[cfg_id]
    cores = os.cpu_count() or 1
    # bounded sample: about two minutes of wall clock for the whole call (one headline iteration of the unmodified reference
    # takes ~23 s per core: 1024 scipy CG solves plus the right-hand-side assembly of gcr_fgmodes_1d)
    if cfg_id == 1:
        nt_sample = c["nt"]
    elif cfg_id == 3:
        nt_sample = int(min(c["nt"], max(32, (c["nt"] * 120 // (23 * max(steps, 1))) // 16 * 16)))
    else:
        nt_sample = min(c["nt"], 32 if cfg_id == 2 else 128)
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        if warmup:
            pool.map(_cpu_worker, [(1, 1000 + i, CONFIGS[1]["nt"], 1) for i in range(cores)])   # imports, first touch
        t0 = time.perf_counter()
        res = pool.map(_cpu_worker, [(cfg_id, i, nt_sample, steps) for i in range(cores)])
        dt = time.perf_counter() - t0
    kind_full = res[0][1]
    kind = kind_full.split(" ")[0]
    frac = nt_sample / c["nt"]   # fraction of a baseline-iteration that one sampled iteration is
    sample = (f"{cores} baselines x {steps} Gibbs iteration(s), one single-threaded process per core, "
              f"{'the unmodified reference (baseline/_ref)' if kind == 'reference' else 'the oracle port'}"
              + (f", {nt_sample} of {c['nt']} times per baseline (scaled by {frac:.4f})" if frac < 1 else "")
              + f"; every iteration restarts from S_initial = I; {dt:.1f} s")
    if kind == "reference":
        sample += "; multiprocess.Pool(1) of gcr_fgmodes mapped in-process (its teardown stalls sporadically on this image)"
        if kind_full != kind:
            sample += "; " + kind_full[len(kind) + 1:].strip("()")
    return cores * steps * frac / dt, cores, dt, kind, sample


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg_id = args.config
    steps = max(1, args.steps or 1)
    if cfg_id == 0:
        line = run_config0_reference(steps)
    else:
        c = CONFIGS[cfg_id]
        val, cores, dt, kind, sample = cpu_throughput(cfg_id, steps, args.warmup)
        line = {
            "impl": "reference", "metric": metric_name(cfg_id), "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": c["scaling"],
            "vs_baseline": None, "dtype": "f64 (complex128)", "data": "synthetic",
            "config": {"workload": workload_name(cfg_id, None), "sample": sample},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
    print(json.dumps(line))


def metric_name(cfg_id):
    if cfg_id == 3:
        return METRIC
    if cfg_id == 0:
        return "baseline-Gibbs-iterations/sec on the reference's test_data run (BASELINE.json configs[0])"
    c = CONFIGS[cfg_id]
    return f"baseline-Gibbs-iterations/sec at Nfreq={c['nf']}, Ntimes={c['nt']}, Nfg={c['nm']} (BASELINE.json configs[{cfg_id}])"


def workload_name(cfg_id, B):
    if cfg_id == 0:
        return "BASELINE.json configs[0]: test_data/vis-eor-fgs.uvh5, baseline (0, 1), 203 x 120, 12 foreground modes"
    c = CONFIGS[cfg_id]
    return (f"BASELINE.json configs[{cfg_id}]: {c['what']}; Nfreq={c['nf']} Ntimes={c['nt']} Nfg={c['nm']}"
            + (f", {B} baselines on this GPU" if B else ""))


# ------------------------------------------------------------------------------------------------
# configs[0]: the reference's own test_data run
def _config0_inputs(tmp):
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    from testdata_fixture import materialize
    from make_golden_testdata import driver_argv
    td = materialize(Path(tmp) / "td")
    return td, driver_argv


def run_config0_reference(steps):
    """The unmodified reference sampler on its test_data inputs (assembled by this repo's driver functions: pyuvdata is
    not installed), one core, `steps` iterations -- the CPU run BASELINE.json configs[0] names."""
    import tempfile
    import warnings
    import run_hydra_pspec_b200 as drv
    with tempfile.TemporaryDirectory() as tmp:
        td, driver_argv = _config0_inputs(tmp)
        _, a = drv.parse_args(driver_argv(td, tmp))
        antpairs, freqs, get = drv.read_visibilities([Path(p) for p in a.file_paths], a.ant_str, a.freq_range)
        b = drv.assemble_baselines(a, antpairs, freqs, get, Path(tmp))[0]
        w = drv.time_invariant_flags(~np.asarray(b["w"], dtype=bool))
        pr = drv.ps_prior_for(a, b["d"].shape[1])
        hp = load_reference()   # (after the inputs are read: it stubs pyuvdata, which the reference's utils.py imports)
        t0 = time.perf_counter()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            if hp is not None:
                hp.pspec.gibbs_sample_with_fg(b["d"], w, b["S_initial"], b["fgmodes"], b["Ninv"], pr, Niter=steps,
                                              seed=a.seed, verbose=False, nproc=1)
                kind = "reference"
            else:
                from oracle import hydra_oracle as ho
                ho.gibbs_sample_with_fg(b["d"], w, b["S_initial"], b["fgmodes"], b["Ninv"], pr, Niter=steps, seed=a.seed)
                kind = "port"
        dt = time.perf_counter() - t0
    val = steps / dt
    sample = f"1 baseline x {steps} iterations on one core ({kind}); {dt:.1f} s"
    return {"impl": "reference", "metric": metric_name(0), "value": val, "unit": UNIT, "n_gpus": 1, "steps": steps, "warmup": 0,
            "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "replicas", "vs_baseline": None,
            "dtype": "f64 (complex128)", "data": "the reference's test_data", "config": {"workload": workload_name(0, 1), "sample": sample},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def run_config0_b200(args):
    """configs[0] end to end through the driver (uvh5 read, input assembly, chain, .npy output), numpy draws + the scalar
    model of the reference's CG: the run reproduces the reference's files (tests/test_driver_cli.py)."""
    import tempfile
    import torch
    import run_hydra_pspec_b200 as drv
    from hydra_pspec_b200 import _lib
    niter = args.steps or 1000   # test_data/config.yaml: Niter 1000
    with tempfile.TemporaryDirectory() as tmp:
        td, driver_argv = _config0_inputs(tmp)
        argv = driver_argv(td, tmp)
        argv[argv.index("--Niter") + 1] = str(niter)
        drv.main(argv[:argv.index("--Niter") + 1] + ["3"] + argv[argv.index("--Niter") + 2:])   # warm-up (arena, first touch)
        torch.cuda.synchronize()
        with ClockSampler(0) as clk:
            t0 = time.perf_counter()
            rc = drv.main(argv)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
    assert rc == 0
    val = niter / dt
    cpu = None
    if not args.no_cpu_baseline:
        r = run_config0_reference(3)
        cpu = r["cpu_baseline"]
    out_bytes = niter * (203 * 120 * 24 + 203 * 12 * 16 + 120 * 8 + 8)
    return {"metric": metric_name(0), "value": val, "unit": UNIT, "n_gpus": 1, "steps": niter, "warmup": 3,
            "ms_per_step": 1e3 * dt / niter, "higher_is_better": True, "scaling": "replicas", "vs_baseline": None,
            "dtype": "f64 (complex128)", "data": "the reference's test_data",
            "config": {"workload": workload_name(0, 1), "call": "run_hydra_pspec_b200.main(argv): uvh5 read + assembly + chain + .npy files",
                       "l2": "single small baseline: working set fits L2; every iteration rewrites it"},
            "roofline": {"bound": "latency", "note": "one 132 x 132 system, 203 times: launch / latency bound, no roofline claimed",
                         "achieved": None, "peak": _lib.lib().hp_fp64_peak_tflops(0, 0.2), "unit": "TFLOP/s", "frac": None, "traffic": None},
            "cpu_baseline": cpu,
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": int(203 * 120 * 16 / niter), "d2h_bytes_per_step": int(out_bytes / niter),
                    "call": "the driver run above is the end-to-end call (host file in, host files out)"},
            "gpu_launches": None, "clocks": clk.summary()}


# ------------------------------------------------------------------------------------------------
def ncu_traffic(kernel):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this workload
    (profiles/r2_ncu_traffic.json, written from the .ncu-rep by profiles/ncu_summary.py); None when there is no capture."""
    try:
        d = json.load(open(ROOT / "profiles" / "r2_ncu_traffic.json"))
        e = d[kernel]
        return e["dram_bytes_read"] + e["dram_bytes_write"], e["source"]
    except Exception:  # noqa: BLE001
        return None, None


def run_b200(args):
    import torch
    import torch.distributed as dist
    from hydra_pspec_b200 import _lib, pspec, driver

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (hydra_pspec_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    numa_node = _lib.bind_to_device_numa(local_rank, verbose=True) if world > 1 else None
    # stdout carries exactly one JSON line: anything libraries print at the fd level while the job runs
    # (NCCL's "NCCL version ..." banner on a box with NCCL_DEBUG set) goes to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if args.config == 0:
        if rank == 0:
            os.write(json_fd, (json.dumps(run_config0_b200(args)) + "\n").encode())
        return
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cfg_id = args.config
    c = CONFIGS[cfg_id]
    nt, nf, nm = c["nt"], c["nf"], c["nm"]
    if args.baselines_per_gpu:
        B = args.baselines_per_gpu
    elif c["total"]:
        B = driver.shard_counts(c["total"], world)[rank]   # strong scaling: the fixed set of baselines is sharded
    else:
        B = c["per_gpu"]
    first = rank * B if not c["total"] else sum(driver.shard_counts(c["total"], world)[:rank])
    K, W = args.steps or c["steps"], max(args.warmup, 3)
    KP = 3  # extra, untimed steps on a single stream for the per-kernel CUDA-event timings
    N = nf + nm
    tstream = torch.cuda.Stream()   # a non-default torch stream: the engine launches on it, and torch.cuda.Event times it
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    substreams = args.substreams if cfg_id == 3 else (2 if cfg_id == 4 else 1)

    def barrier():
        if world > 1:
            dist.barrier()

    Ninv_dense = dense_ninv(nf) if c["mode"] == "dense" else None

    def host_inputs(seed):
        """(vis, flags, fgmodes, ninv_diag, lam0sq) of one synthetic baseline in the form load_chain takes for this config"""
        v, flags, F, nd, l0 = make_baseline(seed, nt, nf, nm, flagged=c["flags"])
        if c["mode"] == "pertime":
            flags = per_time_flags(seed, flags, nt)
        elif c["mode"] == "dense":
            nd = np.real(np.diagonal(Ninv_dense)).copy()
        return v, flags, F, nd, l0

    def load(eng, chain, inp, vis=None):
        v, flags, F, nd, l0 = inp
        eng.load_chain(chain, v if vis is None else vis, flags, F, nd, l0, ninv_dense=Ninv_dense)

    # ---- resident chains (baselines are independent: rank r holds global baselines first .. first + B - 1).  The big
    # per-iteration outputs (signal_cr, fg_amps, chisq) are written to a 2-slot device ring in every step.
    mode_kw = dict(time_flags=(c["mode"] == "pertime"), dense_noise=(c["mode"] == "dense"))
    eng = pspec.GibbsEngine(B, nt, nf, nm, max_iters=K + W + KP, rng="philox", cg_compat=False, refresh_omega=True,
                            keep=("cr", "fg", "chisq"), ring_iters=2, seed=1234, device=local_rank, stream=stream,
                            substreams=substreams, **mode_kw)
    eng.set_chain_ids(np.arange(first, first + B, dtype=np.int32))   # one key for the job, chain id = global baseline index
    t_load = time.perf_counter()
    for ch in range(B):
        load(eng, ch, host_inputs(first + ch))
    t_load = time.perf_counter() - t_load

    eng.run(W)
    eng.sync()
    torch.cuda.synchronize()
    barrier()
    l0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        ev0.record()
        eng.run(K)
        ev1.record()
        torch.cuda.synchronize()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count - l0
    dumped = dump_outputs(eng, args.dump_outputs, W + K - 1) if (args.dump_outputs and rank == 0) else None
    # per-kernel durations: same engine, sub-batches off so that the kernels do not overlap
    eng.set_substreams(1)
    eng.set_profile(True)
    eng.kernel_ms(reset=True)
    eng.run(KP)
    kms = eng.kernel_ms(reset=True)
    eng.set_profile(False)
    bad = int(np.count_nonzero(eng.info()))
    ps_last = eng.signal_ps(0, W + K + KP - 1, 1)
    finite = bool(np.all(np.isfinite(ps_last)))
    t = torch.tensor([ms, float(B)], dtype=torch.float64, device="cuda")
    if world > 1:
        tm = t.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ms_max, Btot = float(tm[0].item()), float(t[1].item())
    else:
        ms_max, Btot = ms, float(B)
    value = Btot * K / (ms_max * 1e-3)

    # ---- roofline of the dominant kernel
    peak = _lib.lib().hp_fp64_peak_tflops(local_rank, 0.3)
    solve_ms, solve_launches = kms["solve"]
    pt_form, pt_kmax = eng.pt_form() if c["mode"] == "pertime" else (None, 0)
    direct_flops = (4.0 * N ** 3 / 3 + 8.0 * N * N) * nt * B   # one factorisation + two substitutions per (baseline, time)
    if c["mode"] == "pertime" and pt_form == "direct":
        kernel = "k_pt_cholsolve"
        flops_per_launch = direct_flops
        note = "4 N^3/3 + 8 N^2 flops per (baseline, time) system"
    elif c["mode"] == "pertime":
        # low-rank form (csrc/hp_ptlow.cu): one shared factorisation per baseline; k_solve3 solves the Ntimes right-hand sides
        # and the Nfreq columns of A = D [Q|F]^H sqrt(wbar N^-1); per time a rank-k_t correction (k_pt_lowrank)
        kernel = "k_solve3"
        flops_per_launch = 8.0 * N * N * (nt + nf) * B
        note = ("8 N^2 (Ntimes + Nfreq) flops per baseline-iteration: two triangular products with W = L^-1 for the Ntimes right-hand "
                "sides and the Nfreq columns of A (low-rank form of the per-time systems)")
    else:
        kernel = "k_solve3" if N <= 448 else ("k_solve2 / k_solve" if N <= 576 else "k_zgemm2 (dense-product solve)")
        flops_per_launch = 8.0 * N * N * nt * B
        note = "8 N^2 Ntimes flops per baseline-iteration (two triangular products with W = L^-1)"
    achieved = flops_per_launch / (solve_ms / KP * 1e-3) * 1e-12 if solve_ms > 0 else None
    traffic, traffic_src = ncu_traffic(kernel) if (cfg_id == 3 and B == 128) else (None, None)
    roofline = {
        "bound": "tensor", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
        "frac": achieved / peak if (achieved and peak > 0) else None,
        "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)", "traffic_source": traffic_src,
        "algorithmic_bytes_per_launch": 16.0 * (2 * nt * N + N * N) * B if c["mode"] != "pertime" else None,
        "peak_source": "FP64 DMMA.8x8x4 issue loop measured in this run (hp_fp64_peak_tflops); MEASURED_PEAKS.json has no FP64 entry; nominal 37.2",
        "flops_per_launch": flops_per_launch, "flops_note": note,
        "step_share": {k: v[0] / max(sum(x[0] for x in kms.values()), 1e-9) for k, v in kms.items()},
        "kernel_ms_per_step": {k: v[0] / KP for k, v in kms.items()},
        "kernel_launches_per_step": {k: v[1] / KP for k, v in kms.items()},
        "kernel_timing": f"CUDA events around each kernel class, {KP} extra steps on one stream after the timed region",
    }
    # algorithmic flops of a step: complex Cholesky N^3/6 complex MACs (= 4 N^3 / 3 real flops) + two triangular
    # solves for T right-hand sides (N^2 T complex MACs = 8 N^2 T); the explicit W = L^-1 is an implementation choice
    if c["mode"] == "pertime" and pt_form == "low-rank":
        # + P = A^H R (Hermitian: 4 n^2 N) + per time a k x k Cholesky and 2 k N complex MACs (mean k = rank of the correction)
        kbar = float(np.mean([np.mean(np.sum(f.any(axis=0)[None, :] & ~f, axis=1)) for f in
                              (host_inputs(first + ch)[1] for ch in range(min(B, 4)))]))
        step_flops = (4.0 * N ** 3 / 3 + 8.0 * N * N * (nt + nf) + 4.0 * nf * nf * N + nt * (4.0 * kbar ** 3 / 3 + 16.0 * kbar * N)) * B
        roofline["per_time_form"] = {"form": pt_form, "max_rank": pt_kmax, "mean_rank": kbar,
                                     "lowrank_ms_per_step": kms["lowrank"][0] / KP,
                                     "direct_form_equivalent_tflops": direct_flops * K / (ms * 1e-3) * 1e-12,
                                     "note": "step_tflops counts the flops of the low-rank form; direct_form_equivalent_tflops is what "
                                             "one factorisation per (baseline, time) would need at this rate (may exceed the peak)"}
    else:
        step_flops = flops_per_launch if c["mode"] == "pertime" else (4.0 * N ** 3 / 3 + 8.0 * N * N * nt) * B
    roofline["step_tflops"] = step_flops * K / (ms * 1e-3) * 1e-12
    roofline["step_frac_of_peak"] = roofline["step_tflops"] / peak if peak > 0 else None
    if c["mode"] != "pertime":
        post_ms, chol_ms = kms["post"][0] / KP, kms["chol"][0] / KP
        post_bytes = (16.0 * nt * (N + 2 * nf) + 8.0 * nt * nf + 16.0 * nt * nm) * B   # X, flags*vis in; signal_cr, chisq, fg_amps out
        ok = {"k_post_fft": {"bound": "hbm", "achieved": post_bytes / (post_ms * 1e-3) * 1e-9 if post_ms > 0 else None, "unit": "GB/s",
                             "algorithmic_bytes_per_launch": post_bytes},
              "k_chol_col + k_trinv": {"bound": "tensor", "unit": "TFLOP/s", "peak": peak,
                                       "achieved": (8.0 * N ** 3 / 3) * B / (chol_ms * 1e-3) * 1e-12 if chol_ms > 0 else None,
                                       "flops_per_step": (8.0 * N ** 3 / 3) * B,
                                       "note": "4 N^3/3 (Cholesky) + 4 N^3/3 (explicit inverse of the factor)"}}
        ck = ok["k_chol_col + k_trinv"]
        ck["frac"] = ck["achieved"] / peak if (ck["achieved"] and peak > 0) else None
        try:
            peaks = json.load(open(ROOT / "MEASURED_PEAKS.json"))
            if ok["k_post_fft"]["achieved"]:
                ok["k_post_fft"]["peak"] = peaks["hbm_gbs"]
                ok["k_post_fft"]["frac"] = ok["k_post_fft"]["achieved"] / peaks["hbm_gbs"]
        except Exception:  # noqa: BLE001
            pass
        roofline["other_kernels"] = ok

    # ---- parity: one injected-draw iteration of this rank's first baseline at the benchmark shape against the oracle
    parity = None
    if rank == 0 and not args.no_parity and cfg_id in (1, 3):
        from oracle import hydra_oracle as ho   # checker only
        v, flags, F, nd, _ = make_baseline(first, nt, nf, nm, flagged=c["flags"])
        want = ho.gibbs_sample_with_fg(v, flags, np.eye(nf), F, np.diag(nd), np.zeros((2, nf)), Niter=1, seed=11, solver="direct")
        got = pspec.gibbs_sample_with_fg(v, flags, np.eye(nf), F, np.diag(nd), np.zeros((2, nf)), Niter=1, seed=11, verbose=False,
                                         solver="exact", device=local_rank)
        parity = {k: float(np.max(np.abs(np.asarray(g) - np.asarray(w_))) / np.max(np.abs(w_)))
                  for g, w_, k in zip(got[:6], want, ["signal_cr", "signal_S", "signal_ps", "fg_amps", "chisq", "ln_post"])}
        parity["max"] = max(parity.values())
        parity["what"] = ("one Gibbs iteration of global baseline %d at this shape, the reference's numpy draws injected, exact "
                          "solves: max relative error of every output against oracle.gibbs_sample_with_fg(solver='direct')" % first)

    # ---- gather of the sample arrays over NCCL (the only collective of the job)
    gather = None
    if world > 1:
        ps_loc = np.stack([eng.signal_ps(ch, W, K) for ch in range(B)])
        lp_loc = np.stack([eng.ln_post(ch, W, K) for ch in range(B)])
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        if c["total"]:
            ps_all = driver.gather_samples(ps_loc, int(Btot))
            lp_all = driver.gather_samples(lp_loc, int(Btot))
        else:   # equal shards
            ps_all = driver.gather_samples(ps_loc, int(Btot))
            lp_all = driver.gather_samples(lp_loc, int(Btot))
        torch.cuda.synchronize()
        dtg = time.perf_counter() - t0
        tg = torch.tensor([dtg], dtype=torch.float64, device="cuda")
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        gather = {"seconds": float(tg.item()), "bytes_per_rank": int(ps_loc.nbytes + lp_loc.nbytes), "shape": list(ps_all.shape),
                  "what": f"driver.gather_samples (NCCL all_gather) of signal_ps + ln_post of the {K} timed iterations, all ranks",
                  "finite": bool(np.all(np.isfinite(ps_all)) and np.all(np.isfinite(lp_all)))}
    eng.close()

    # ---- end to end through the public API with host buffers (the reference's full return set)
    e2e = None
    if not args.no_e2e:
        Ke = args.e2e_iters
        pin, hin = [], []
        for ch in range(B):   # host inputs of the call, prepared once: the visibilities in page-locked memory
            inp = host_inputs(10_000 + first + ch)
            pv = _lib.pinned_empty(inp[0].shape, np.complex128)
            pv[...] = inp[0]
            pin.append(pv)
            hin.append(inp)
        stage = {}
        chunk = 2   # iterations of page-locked staging (bounded: the host side of a long chain re-uses it)

        def one_call(keep):
            e = pspec.GibbsEngine(B, nt, nf, nm, max_iters=Ke, rng="philox", keep=keep, ring_iters=3, seed=99, device=local_rank,
                                  stream=stream, substreams=substreams, **mode_kw)
            e.set_chain_ids(np.arange(first, first + B, dtype=np.int32))
            if keep not in stage:
                stage[keep] = e.host_buffers(chunk, iter_major=True)   # page-locked destination arrays, allocated once by the caller
            for ch in range(B):
                load(e, ch, hin[ch], vis=pin[ch])
            done = 0
            while done < Ke:
                n_ = min(chunk, Ke - done)
                # compute overlapped with the device-to-host copies; read-ahead: the next chunk's first iterations are computed
                # under this chunk's last copies (hp_host_sink.read_ahead)
                e.run_to_host(n_, stage[keep], first_iter=done, iter_major=True, read_ahead=(2 if done + n_ < Ke else 0))
                done += n_
            e.close()

        def timed(keep):
            one_call(keep)  # warm-up (allocation paths, first touch)
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            reps = 2
            for _ in range(reps):
                one_call(keep)
            torch.cuda.synchronize()
            dt_ = (time.perf_counter() - t0) / reps
            tt = torch.tensor([dt_], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())

        full = ("cr", "fg", "chisq")
        dt = timed(full)
        dt_ps = timed(())
        h2d = sum(p.nbytes for p in pin) / Ke
        d2h = sum(v.nbytes for v in stage[full].values()) / chunk
        e2e = {"value": Btot * Ke / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "call": f"GibbsEngine(create) + load_chain x{B} from pinned host arrays + run_to_host({Ke} iterations, staging area of "
                       f"{chunk}): signal_cr/fg_amps/chisq/signal_ps/ln_post of every iteration (the reference's full return set) land "
                       "in pinned host arrays through a 3-slot device ring; PCIe-bound",
               "baselines": B, "iterations": Ke, "substreams": substreams, "pcie_gbs": d2h * Ke / dt * 1e-9, "numa_node": numa_node,
               "power_spectrum_only": {"value": Btot * Ke / dt_ps, "unit": UNIT,
                                       "d2h_bytes_per_step": int(sum(v.nbytes for v in stage[()].values()) / chunk),
                                       "call": "same call with keep=(): only signal_ps + ln_post are read back"}}

    # ---- CPU baseline on this box (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v_, cores, dtc, kind, sample = cpu_throughput(cfg_id, 1, 1)
        cpu = {"value": v_, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}

    if rank == 0:
        line = {
            "metric": metric_name(cfg_id), "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": c["scaling"], "vs_baseline": None,
            "dtype": "f64 (complex128)", "data": "synthetic",
            "config": {"workload": workload_name(cfg_id, B) + "; device Philox draws, exact solves",
                       "baselines_per_gpu": B, "baselines_total": int(Btot), "substreams": substreams,
                       "parallelism": f"baseline-sharded x{world}, no hot-path collective",
                       "l2": f"per-step working set ~{B * 16 * (4 * nt * N + 4 * nt * nf) / 2**30:.1f} GiB per GPU vs 126 MB L2"
                             + ("" if B * 16 * 4 * nt * N > 2 ** 28 else " (fits: a single small baseline, every iteration rewrites it)"),
                       "outputs_kept": "signal_cr + fg_amps + chisq written to a 2-slot device ring and signal_ps + ln_post per iteration "
                                       "(value); the same streamed to pinned host arrays (e2e)",
                       "load_s": round(t_load, 2)},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "parity_check": parity,
            "gather": gather, "clocks": clk.summary(), "chol_failures": bad, "finite": finite,
        }
        if dumped is not None:
            line["dump_outputs"] = {"dir": args.dump_outputs, "iteration": W + K - 1, "sampled_chains": dumped.tolist()}
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
