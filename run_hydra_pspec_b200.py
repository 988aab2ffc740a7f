#!/usr/bin/env python
"""Driver: the reference's ``run-hydra-pspec.py`` with the Gibbs hot path on B200s.

Same command line, config file keys, input files and output files as the reference driver
(run-hydra-pspec.py:38-260 arguments, :290-480 per-baseline input assembly, :482-557 sampling,
:559-589 timing files), with these differences:

* MPI ranks become one process per GPU.  Launch with ``python run_hydra_pspec_b200.py ...`` (one GPU)
  or ``python -m torch.distributed.run --nproc-per-node N run_hydra_pspec_b200.py ...``; baselines are
  split over ranks exactly like ``split_data_for_scatter`` and never exchanged during sampling.
* ``--rng numpy`` (default) reproduces the reference's random streams and CG truncation, one chain
  after the other (bit-for-bit comparable outputs, tolerance 1e-10); ``--rng philox`` is the
  production mode: all baselines of a rank advance together in one batched engine with device draws
  and exact solves.
* ``--config`` is read with PyYAML (jsonargparse is not a dependency); keys are the long option
  names, relative ``file_paths`` are resolved against the config file's directory like jsonargparse's
  ``Path_fr`` does, everything else against the working directory.
* uvh5 input goes through pyuvdata when it is importable, else through the built-in reader
  (``hydra_pspec_b200.uvh5``).
* ``--Nproc`` is accepted and ignored (all times of all resident baselines are solved in one launch).
* ``--samples summary`` (or ``both``) writes the posterior mean and variance of the in-painted signal and of the foreground
  amplitudes after ``--burn_in`` iterations, thinned by ``--thin``, accumulated on the GPU: ``gcr-eor-mean.npy``,
  ``gcr-eor-var.npy``, ``fg-amps-mean.npy``, ``fg-amps-var.npy`` and ``summary.json``.  With ``summary`` the per-sample files
  ``gcr-eor.npy`` / ``fg-amps.npy`` / ``chisq.npy`` are not written, and those samples never leave the GPU.  ``--batch B`` adds
  the batch-means Monte-Carlo standard error and effective sample size of each mean (``*-mcse.npy``, ``*-ess.npy``).
"""
import argparse
import json
import os
import sys
import time
from pathlib import Path
from pprint import pprint
from resource import getrusage, RUSAGE_SELF

import numpy as np
import scipy.special


def build_parser():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--ant_str", type=str, default="cross")
    p.add_argument("--sigcov0", type=str)
    p.add_argument("--sigcov0_file", type=str)
    p.add_argument("--Nfgmodes", type=int, default=8)
    p.add_argument("--fgmodes", type=str)
    p.add_argument("--fgmodes_file", type=str)
    p.add_argument("--freq_range", type=str)
    p.add_argument("--flags", type=str)
    p.add_argument("--flags_file", type=str)
    p.add_argument("--noise", type=str)
    p.add_argument("--noise_file", type=str)
    p.add_argument("--noise_cov", type=str)
    p.add_argument("--noise_cov_file", type=str)
    p.add_argument("--nsamples", type=str)
    p.add_argument("--nsamples_file", type=str)
    p.add_argument("--n_ps_prior_bins", type=int, default=3)
    p.add_argument("--ps_prior_lo", type=float, default=0.0)
    p.add_argument("--ps_prior_hi", type=float, default=0.0)
    p.add_argument("--map_estimate", action="store_true")
    p.add_argument("--Niter", type=int, default=100)
    p.add_argument("--seed", type=int, default=None)
    p.add_argument("-v", "--verbose", dest="verbose", action="store_true", default=False)
    p.add_argument("--Nproc", type=int, default=1)
    p.add_argument("--out_dir", type=str, default="./")
    p.add_argument("--dirname", type=str)
    p.add_argument("--clobber", action="store_true", default=False)
    p.add_argument("--write_Niter", type=int, default=100)
    p.add_argument("file_paths", type=str, nargs="*")
    p.add_argument("--config", type=str, action="append")
    # additions
    p.add_argument("--rng", choices=("numpy", "philox"), default="numpy",
                   help="numpy: the reference's random streams, chain by chain; philox: batched device draws")
    p.add_argument("--solver", choices=("reference-cg", "exact"), default=None)
    p.add_argument("--dpss_alpha", type=float, default=None,
                   help="without --fgmodes: use Nfgmodes DPSS modes of this bandwidth factor (hydra_pspec/dpss.py:70-73) "
                        "instead of the reference driver's Legendre polynomials")
    p.add_argument("--time_flags", choices=("any", "per-time"), default="any",
                   help="any: a channel flagged at any time is flagged at all times (the reference, "
                        "run-hydra-pspec.py:520-526); per-time: keep the (Ntimes, Nfreqs) flags (in-painting)")
    p.add_argument("--noise_weights", choices=("none", "nsamples"), default=argparse.SUPPRESS,
                   help="none (default): one inverse noise covariance for all times; nsamples: diagonal noise per time and channel, "
                        "N_t^-1 = nsamples[t] * diag(N^-1) (needs --nsamples and a diagonal N^-1, i.e. no --noise_cov)")
    p.add_argument("--samples", choices=("all", "summary", "both"), default="all",
                   help="all: every sample of signal_cr / fg_amps / chisq (gcr-eor.npy, fg-amps.npy, chisq.npy); summary: only "
                        "their posterior mean and variance, accumulated on the GPU (gcr-eor-mean.npy, gcr-eor-var.npy, "
                        "fg-amps-mean.npy, fg-amps-var.npy, summary.json); both: the two")
    p.add_argument("--burn_in", type=int, default=0, help="--samples summary / both: iterations skipped before accumulating")
    p.add_argument("--thin", type=int, default=1, help="--samples summary / both: accumulate every thin-th iteration")
    p.add_argument("--batch", type=int, default=argparse.SUPPRESS,
                   help="--samples summary / both: also write the batch-means Monte-Carlo standard error and effective "
                        "sample size of each mean (gcr-eor-mcse.npy, gcr-eor-ess.npy, fg-amps-mcse.npy, fg-amps-ess.npy), "
                        "from batches of BATCH accumulated (i.e. thinned) samples.  Choose BATCH well above the "
                        "autocorrelation time, about sqrt of the accumulated samples; fewer than 2 complete batches give NaN")
    return p


def parse_args(argv=None):
    """Command line over config file(s) over defaults, the precedence jsonargparse gives
    ``ActionConfigFile`` when the config is named first."""
    import yaml
    parser = build_parser()
    args = parser.parse_args(argv)
    if args.config:
        merged = {}
        for cfg in args.config:
            cfg_path = Path(cfg)
            with open(cfg_path) as f:
                d = yaml.safe_load(f) or {}
            if "file_paths" in d:
                d["file_paths"] = [str(p if Path(p).is_absolute() else (cfg_path.parent / p)) for p in d["file_paths"]]
            merged.update(d)
        known = {a.dest for a in parser._actions}
        unknown = set(merged) - known
        if unknown:
            parser.error(f"unknown key(s) in config file: {sorted(unknown)}")
        cli_paths = args.file_paths
        parser.set_defaults(**merged)
        args = parser.parse_args(argv)
        if cli_paths:
            args.file_paths = cli_paths
        elif "file_paths" in merged:
            args.file_paths = merged["file_paths"]
    return parser, args


def check_shape(shape, d_shape, desc=""):
    assert shape == d_shape, (f"The {desc} array has shape {shape} which does not match the shape of the "
                              f"per-baseline data, {d_shape}.")


def check_load_path(fp):
    fp = Path(fp)
    if fp.is_dir():
        return True, None
    return False, np.load(fp)


def _per_baseline(path, file_name, bl_str):
    is_dir, data = check_load_path(path)
    if is_dir:
        data = np.load(Path(path) / bl_str / file_name)
    return data


def read_visibilities(file_paths, ant_str, freq_range):
    """run-hydra-pspec.py:305-322: read, select antenna pairs / frequencies, conjugate to ant1 < ant2,
    form pseudo-Stokes I in the XX slot."""
    from hydra_pspec_b200 import utils
    try:
        from pyuvdata import UVData  # pragma: no cover - not in this image
        have_pyuvdata = hasattr(UVData, "read")   # (a stub module stands in for it when the reference is imported)
    except ImportError:
        have_pyuvdata = False
    if have_pyuvdata:  # pragma: no cover
        uvd = UVData()
        keep = None
        if freq_range:
            uvd.read(file_paths[0], read_data=False)
            keep = utils.filter_freqs(freq_range, np.asarray(uvd.freq_array).reshape(-1) / 1e6) * 1e6
        uvd.read(file_paths, ant_str=ant_str, frequencies=keep)
        uvd.conjugate_bls()
        uvd = utils.form_pseudo_stokes_vis(uvd)
        freqs = np.asarray(uvd.freq_array).reshape(-1)
        get = lambda ap: (uvd.get_data(ap + ("xx",), force_copy=True), uvd.get_flags(ap + ("xx",)))  # noqa: E731
        return uvd.get_antpairs(), freqs, get
    from hydra_pspec_b200.uvh5 import read_uvh5
    uvd = read_uvh5(file_paths[0] if len(file_paths) == 1 else list(file_paths))
    keep = None
    if freq_range:
        keep = utils.filter_freqs(freq_range, uvd.freq_array / 1e6) * 1e6
    uvd.select(ant_str=ant_str, frequencies=keep)
    uvd.conjugate_bls()
    uvd = utils.form_pseudo_stokes_vis(uvd)
    get = lambda ap: (uvd.get_data(ap + ("xx",)), uvd.get_flags(ap + ("xx",)))  # noqa: E731
    return uvd.get_antpairs(), uvd.freq_array, get


def assemble_baselines(args, antpairs, freqs, get, out_dir):
    """Per-baseline inputs (run-hydra-pspec.py:357-470)."""
    Nfreqs = freqs.size
    fmhz = freqs / 1e6
    freq_str = f"{fmhz.min():.3f}-{fmhz.max():.3f}MHz"
    all_data_weights = []
    for antpair in antpairs:
        bl_str = f"{antpair[0]}-{antpair[1]}"
        d, uv_flags = get(tuple(antpair))
        bl_data_shape = d.shape
        cov_ff_shape = (Nfreqs, Nfreqs)
        if args.flags:
            flags = _per_baseline(args.flags, args.flags_file, bl_str)
            check_shape(flags.shape, bl_data_shape, desc="flags")
        else:
            flags = uv_flags
        nsamples = None
        if args.nsamples:
            nsamples = _per_baseline(args.nsamples, args.nsamples_file, bl_str)
            check_shape(nsamples.shape, bl_data_shape, desc="nsamples")
        if args.noise:
            noise = _per_baseline(args.noise, args.noise_file, bl_str)
            check_shape(noise.shape, bl_data_shape, desc="noise")
            if nsamples is not None:
                noise = noise / np.sqrt(nsamples)
            d = d + noise
        if args.sigcov0:
            sigcov0 = _per_baseline(args.sigcov0, args.sigcov0_file, bl_str)
            check_shape(sigcov0.shape, cov_ff_shape, desc="signal covariance")
        else:
            sigcov0 = np.eye(Nfreqs)
        if args.noise_cov:
            noise_cov = _per_baseline(args.noise_cov, args.noise_cov_file, bl_str)
            check_shape(noise_cov.shape, cov_ff_shape, desc="noise covariance")
            Ninv = np.linalg.inv(noise_cov)
        else:
            Ninv = np.eye(Nfreqs) / (10.0) ** 2.0
        if args.fgmodes:
            is_dir, fgmodes = check_load_path(args.fgmodes)
            if is_dir:
                name = args.fgmodes_file if args.fgmodes_file else f"evecs-{freq_str}.npy"
                fgmodes = np.load(Path(args.fgmodes) / bl_str / name)
            fgmodes = fgmodes[:, :args.Nfgmodes]
            check_shape(fgmodes.shape, (Nfreqs, args.Nfgmodes), desc="fgmodes")
        elif args.dpss_alpha is not None:
            from hydra_pspec_b200.dpss import dpss_modes
            fgmodes = dpss_modes(freqs.size, args.Nfgmodes, args.dpss_alpha).T
        else:
            fgmodes = np.array([scipy.special.legendre(i)(np.linspace(-1.0, 1.0, freqs.size))
                                for i in range(args.Nfgmodes)]).T
        ninv_t = None
        if getattr(args, "noise_weights", "none") == "nsamples":
            # the noise of a cell averaged over nsamples samples has variance sigma^2 / nsamples (the simulated noise above)
            ninv_t = np.asarray(nsamples, dtype=np.float64) * np.real(np.diagonal(Ninv))[None, :]
        all_data_weights.append({"antpair": tuple(int(a) for a in antpair), "d": d, "w": flags, "fgmodes": fgmodes,
                                 "S_initial": sigcov0, "Ninv": Ninv, "ninv_t": ninv_t, "out_dir": out_dir})
    return all_data_weights


def ps_prior_for(args, Nfreqs):
    """run-hydra-pspec.py:497-510."""
    ps_prior = np.zeros((2, Nfreqs))
    if args.ps_prior_lo != 0 or args.ps_prior_hi != 0:
        inds = slice(Nfreqs // 2 - args.n_ps_prior_bins, Nfreqs // 2 + args.n_ps_prior_bins + 1)
        ps_prior[0, inds] = args.ps_prior_hi
        ps_prior[1, inds] = args.ps_prior_lo
    return ps_prior


def time_noise_ninv(ninv_t):
    """(Ntimes, Nfreqs, Nfreqs) inverse noise covariance with diagonal slices diag(ninv_t[t])."""
    T, n = ninv_t.shape
    out = np.zeros((T, n, n), dtype=np.float64)
    out[:, np.arange(n), np.arange(n)] = ninv_t
    return out


def time_invariant_flags(w):
    """A channel flagged at any time is dropped at all times (run-hydra-pspec.py:520-526).
    ``w``: (Ntimes, Nfreqs) bool, True = unflagged."""
    return np.all(w, axis=0)


def main(argv=None):
    parser, args = parse_args(argv)
    if args.burn_in < 0 or args.thin < 1:
        parser.error("--burn_in must be >= 0 and --thin >= 1")
    batch = getattr(args, "batch", 0)   # absent from the namespace unless given
    if hasattr(args, "batch"):
        if args.samples == "all":
            parser.error("--batch needs --samples summary or both")
        if batch < 1:
            parser.error("--batch must be >= 1")
    if getattr(args, "noise_weights", "none") == "nsamples":   # absent from the namespace unless given
        if not args.nsamples:
            parser.error("--noise_weights nsamples needs --nsamples")
        if args.noise_cov:
            parser.error("--noise_weights nsamples needs a diagonal inverse noise covariance: it cannot be combined with "
                         "--noise_cov")
    summary = None if args.samples == "all" else dict(burn_in=args.burn_in, thin=args.thin)
    if batch:
        summary["batch"] = batch
    rank = int(os.environ.get("RANK", "0"))
    size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if size > 1:
        import torch
        import torch.distributed as dist
        backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
        dist.init_process_group(backend)

    from hydra_pspec_b200 import pspec, driver, utils, _lib
    _lib.bind_to_device_numa(local_rank)  # page-locked output staging next to this rank's GPU

    time_load_start = time.perf_counter()
    # Every rank reads the (small) inputs itself: the reference's rank-0 load + MPI scatter of pickled
    # arrays is replaced by an identical deterministic split on every rank.
    if not args.file_paths:
        print("Must pass file(s) to analyze via --file_paths.  Exiting.")
        return 1
    file_paths = sorted(Path(fp) for fp in args.file_paths)
    if rank == 0:
        if args.config:
            print(f"Loading config file {args.config[0]}", end="\n\n")
        pprint(vars(args))
        print(f"\nReading {len(file_paths)} file(s)")
    antpairs, freqs, get = read_visibilities(file_paths, args.ant_str, args.freq_range)
    fmhz = freqs / 1e6
    freq_str = f"{fmhz.min():.3f}-{fmhz.max():.3f}MHz"
    out_dir = Path(args.out_dir)
    if not args.dirname:
        out_dir /= f"results-{freq_str}-Niter-{args.Niter}"
    elif args.map_estimate:
        out_dir /= args.dirname + "-map-estimate"
    else:
        out_dir /= args.dirname
    if rank == 0:
        if out_dir.exists() and not args.clobber:
            utils.add_mtime_to_filepath(out_dir)
        out_dir.mkdir(exist_ok=True, parents=True)
        print(f"\nWriting output(s) to {out_dir.absolute()}", end="\n\n")
        with open(out_dir / "git.json", "w") as f:
            json.dump("", f, indent=2)
        with open(out_dir / "args.json", "w") as f:
            json.dump(vars(args), f, indent=2, default=str)
        if "SLURM_JOB_ID" in os.environ:
            (out_dir / os.environ["SLURM_JOB_ID"]).touch()
    if dist is not None:
        dist.barrier()
    all_data_weights = assemble_baselines(args, antpairs, freqs, get, out_dir)
    list_of_baselines = driver.split_data_for_scatter(all_data_weights, size)[rank]
    global_ids = driver.split_data_for_scatter(list(range(len(all_data_weights))), size)[rank]
    time_load_end = time.perf_counter()

    verbose = args.verbose and rank == 0
    jobs = []
    for data in list_of_baselines:
        antpair = data["antpair"]
        bl_dir = data["out_dir"] / f"{antpair[0]}-{antpair[1]}"
        bl_dir.mkdir(exist_ok=True, parents=True)
        w = ~np.asarray(data["w"], dtype=bool)
        flags = w if args.time_flags == "per-time" else time_invariant_flags(w)
        jobs.append(dict(vis=data["d"], flags=flags, S_initial=data["S_initial"], fgmodes=data["fgmodes"],
                         Ninv=data["Ninv"], ninv_t=data["ninv_t"], ps_prior=ps_prior_for(args, data["d"].shape[1]),
                         out_dir=bl_dir, antpair=antpair))

    ant_pairs, write_times = [], []
    if args.rng == "numpy":
        for job in jobs:  # one chain after the other, the reference's streams
            if verbose:
                print(f"Printing status messages for:\nRank:     {rank}\nBaseline: {job['antpair']}", end="\n\n")
            if job["ninv_t"] is not None and args.samples != "summary":
                # the drop-in takes per-time noise as a 3-D Ninv; built for one baseline at a time
                job = dict(job, Ninv=time_noise_ninv(job["ninv_t"]), ninv_t=None)
            if args.samples == "summary":
                # the same chain through the batched form, which can leave the samples on the device (keep=())
                res = pspec.gibbs_sample_batch([job], Niter=args.Niter, seed=args.seed, rng="numpy", solver=args.solver,
                                               keep=(), write_Niter=args.write_Niter, map_estimate=args.map_estimate,
                                               device=local_rank, verbose=verbose, summary=summary)[0]
            else:
                res = pspec.gibbs_sample_with_fg(job["vis"], job["flags"], job["S_initial"], job["fgmodes"], job["Ninv"],
                                                 job["ps_prior"], Niter=args.Niter, seed=args.seed,
                                                 map_estimate=args.map_estimate, verbose=verbose, nproc=args.Nproc,
                                                 write_Niter=args.write_Niter, out_dir=job["out_dir"], rng="numpy",
                                                 solver=args.solver, device=local_rank, summary=summary)
            ant_pairs.append(f"{job['antpair'][0]}_{job['antpair'][1]}")
            write_times.append(res[6])
    else:
        # one Philox key for the whole job, chain id = global baseline index: the samples of a baseline do not
        # depend on the number of ranks / GPUs
        seed = 0 if args.seed is None else args.seed
        keep = () if args.samples == "summary" else ("cr", "fg", "chisq")
        res = pspec.gibbs_sample_batch(jobs, Niter=args.Niter, seed=int(seed) & 0xFFFFFFFFFFFFFFFF, rng="philox",
                                       solver=args.solver, keep=keep, write_Niter=args.write_Niter,
                                       map_estimate=args.map_estimate, device=local_rank, verbose=verbose,
                                       chain_ids=global_ids, summary=summary)
        for job, r in zip(jobs, res):
            ant_pairs.append(f"{job['antpair'][0]}_{job['antpair'][1]}")
            write_times.append(r[6])
    write_timings = {"rank": rank, "ant_pairs": ant_pairs, "write_times": write_times}
    if dist is not None:
        gathered = [None] * size
        dist.all_gather_object(gathered, write_timings)
        pre = time.perf_counter()
        dist.barrier()
        time_barrier = time.perf_counter() - pre
    else:
        gathered, time_barrier = [write_timings], 0.0

    if rank == 0:
        time_stop = time.perf_counter()
        timings = {"num_ranks": size, "num_baselines": len(antpairs),
                   "rank_0_timers": {"load_data": time_load_end - time_load_start, "scatter": 0.0,
                                     "process": time_stop - time_load_end, "barrier": time_barrier,
                                     "total": time_stop - time_load_start},
                   "write_data": gathered}
        with open(out_dir / "timings.json", "w") as f:
            json.dump(timings, f, indent=2)
        r = getrusage(RUSAGE_SELF)
        with open(out_dir / "resources.json", "w") as f:
            json.dump({"ru_maxrss": r.ru_maxrss, "ru_utime": r.ru_utime, "ru_stime": r.ru_stime}, f, indent=2)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
