"""Drop-in for ``hydra_pspec.pspec`` (reference: hydra_pspec/pspec.py) on B200.

Same function names, argument meaning, return values and error behaviour as the reference for
the Gibbs hot path; the work is done by hand-written sm_100a kernels behind the C ABI in
``include/hydra_pspec_b200.h``.  The host code in this module only validates and stages the
inputs, reproduces the reference's numpy random streams when asked to (``rng="numpy"``), and
copies the sample arrays back.

Two fidelity modes
------------------
``rng="numpy"`` (default of the drop-in functions)
    The draws are the reference's: ``np.random.seed(912983 + t)`` normals per time for the GCR
    fluctuation terms (pspec.py:195-217, identical in every iteration) and one uniform per delay
    bin per iteration from ``np.random.seed(seed)`` for ``sample_S`` (pspec.py:58, 125).  With
    ``solver="reference-cg"`` (default in this mode) each solve is additionally scaled by the
    scalar model of the reference's truncated CG, so a chain reproduces the reference's numbers
    to ~1e-10.  ``solver="exact"`` returns the exact solution of the same linear system.
``rng="philox"``
    Device Philox4x32-10 draws, exact solves, new fluctuation terms every iteration
    (``refresh_omega=True``) -- the production mode used by :class:`GibbsEngine` and ``bench.py``.
"""
import os
import time

import numpy as np
import scipy.special
from scipy.interpolate import interp1d
from scipy.stats import invgamma

from . import _lib, utils

GCR_SEED_BASE = 912983  # pspec.py:153

# Test switch: apply the Fourier operator as dense products instead of the fused FFT kernels (the
# path Nfreqs with a prime factor > 31 takes anyway).
_FORCE_DENSE_TRANSFORMS = False
_FORCE_DENSE_SOLVE = False  # tests: take the large-N dense-product solve at any size


# --------------------------------------------------------------------------------------------
# host-side helpers of the reference API (not on the hot path)
def inversion_sample_invgamma(alpha, beta, prior_min, prior_max, ngrid=1000):
    """pspec.py:11-64.  Host version (the chain uses the device implementation in k_sample)."""
    if prior_min <= 0:
        raise ValueError("prior_min must be greater than zero")
    if prior_max <= 0:
        raise ValueError("prior_max must be greater than zero")
    if not np.isfinite(prior_max):
        raise ValueError("prior_max must be finite")
    if prior_max <= prior_min:
        raise ValueError("prior_max must be greater than prior_min")
    x = np.logspace(np.log10(prior_min), np.log10(prior_max), ngrid)
    cdf = invgamma.cdf(x, a=alpha, loc=0, scale=beta)
    cdf -= cdf.min()
    cdf /= cdf.max()
    cdf_unique, idxs_unique = np.unique(cdf, return_index=True)
    u = np.random.uniform()
    return interp1d(cdf_unique, x[idxs_unique], kind="linear")(u)


def covariance_from_pspec(ps, fourier_op):
    """pspec.py:313-322."""
    ps = np.asarray(ps)
    return fourier_op.T.conj() @ (ps.astype(complex)[:, None] * fourier_op)


def sprior(signals, bins, factor):
    """pspec.py:130-148."""
    nobs, nfreq = signals.shape
    sk_ = np.fft.fft(signals, axis=-1)
    ds = np.sum(sk_ * sk_.conj(), axis=0).real
    prior = np.zeros((2, nfreq))
    prior[0] = ds * factor
    prior[1] = ds / factor
    prior[0, bins + 1:-bins] = 0
    prior[1, bins + 1:-bins] = 0
    return prior / (nobs / 2 - 1)


# --------------------------------------------------------------------------------------------
# the reference's numpy draw streams
def _reference_gcr_draws(ntimes, nfreqs):
    """(omega_a, omega_b): pspec.py:195-217 -- reseeded per time index, four randn vectors."""
    oma = np.empty((ntimes, nfreqs), dtype=np.complex128)
    omb = np.empty((ntimes, nfreqs), dtype=np.complex128)
    for idx in range(ntimes):
        rs = np.random.RandomState(GCR_SEED_BASE + idx)
        omi, omj = rs.randn(nfreqs), rs.randn(nfreqs)
        omk, oml = rs.randn(nfreqs), rs.randn(nfreqs)
        oma[idx] = (omi + 1.0j * omj) / 2 ** 0.5
        omb[idx] = (omk + 1.0j * oml) / 2 ** 0.5
    return oma, omb


def _s_draws_from_uniforms(u, ps_prior, ntimes):
    """Turn the per-bin uniforms of sample_S into what the device consumes: u itself for
    prior-bounded bins (pspec.py:58), the invgamma(a = Ntimes - 1) variate for the others
    (pspec.py:125; scipy evaluates rvs as ppf(u) = 1 / gammainccinv(a, u))."""
    u = np.atleast_2d(np.asarray(u, dtype=np.float64))
    has_prior = np.any(np.asarray(ps_prior) > 0, axis=0)
    y = 1.0 / scipy.special.gammainccinv(ntimes - 1.0, u)
    return np.where(has_prior[None, :], u, y)


def _check_prior(ps_prior, nfreqs):
    """Raise the reference's errors (pspec.py:40-47) up front instead of mid-chain."""
    if ps_prior is None:
        return np.zeros((2, nfreqs))
    ps_prior = np.asarray(ps_prior, dtype=np.float64)
    if ps_prior.shape != (2, nfreqs):
        raise ValueError(f"ps_prior must have shape (2, {nfreqs})")
    for i in np.nonzero(np.any(ps_prior > 0, axis=0))[0]:
        pmax, pmin = ps_prior[0, i], ps_prior[1, i]
        if pmin <= 0:
            raise ValueError("prior_min must be greater than zero")
        if pmax <= 0:
            raise ValueError("prior_max must be greater than zero")
        if not np.isfinite(pmax):
            raise ValueError("prior_max must be finite")
        if pmax <= pmin:
            raise ValueError("prior_max must be greater than prior_min")
    return ps_prior


_UNITARY_CACHE = {}


def _unitary_dft(n):
    if n not in _UNITARY_CACHE:
        idx = np.arange(n) - n // 2
        _UNITARY_CACHE[n] = np.exp(-2j * np.pi * (np.outer(idx, idx) % n) / n) / np.sqrt(n)
    return _UNITARY_CACHE[n]


def _delay_diagonal(S):
    """Eigenvalues of a delay-diagonal S = U^H diag(d) U (U = fourier_operator / sqrt(n)), or None.  Such an S is circulant,
    S[x, x'] = c[(x - x') mod n]; checked in O(n^2), d from one FFT of its first column (no matrix product)."""
    S = np.asarray(S)
    n = S.shape[0]
    c = S[:, 0]
    idx = (np.arange(n)[:, None] - np.arange(n)[None, :]) % n
    scale = max(np.max(np.abs(np.diagonal(S))), 1e-300)
    if np.max(np.abs(S - c[idx])) > 1e-13 * scale:
        return None
    d = np.roll(np.fft.fft(c), n // 2)          # d[k] = sum_j c[j] exp(-2 pi i (k - n/2) j / n)
    if np.max(np.abs(d.imag)) > 1e-13 * max(np.max(np.abs(d.real)), 1e-300) * n:
        return None
    return np.ascontiguousarray(d.real, dtype=np.float64)


def device_eigh(mats, device=0):
    """Batched Hermitian eigendecomposition on the GPU (csrc/hp_eigh.cu: one-sided Jacobi, one CTA per matrix).
    ``mats``: (batch, n, n); returns ``(w, V)`` like ``numpy.linalg.eigh`` (eigenvalues unordered)."""
    mats = np.ascontiguousarray(mats, dtype=np.complex128)
    batch, n, _ = mats.shape
    V = np.empty_like(mats)
    w = np.empty((batch, n), dtype=np.float64)
    _lib.check(_lib.lib().hp_eigh_batch(int(device), n, batch, _lib.ptr(mats), _lib.ptr(V), _lib.ptr(w), None))
    return w, V


def _analyse_signal_covs(covs, device=0, eigh=None):
    """Eigen-structure of the signal covariances handed to the device, for a list of baselines.

    Returns a list of (basis0 or None, lam0sq).  A delay-diagonal S (every covariance the chain itself produces, the
    reference's test data, and the identity default) needs no decomposition: its eigenvectors are the columns of U^H.
    Everything else is decomposed once, all such matrices of the list in one batched device call (``device_eigh``; the first
    iteration then runs in that basis).  ``eigh``: replacement for the decomposition (host-logic tests without a GPU).
    """
    out = [None] * len(covs)
    todo = []
    for i, S in enumerate(covs):
        S = np.asarray(S)
        d = _delay_diagonal(S)
        if d is not None:
            # eigenvalues are clipped at zero: a rank-deficient or barely positive semi-definite S (e.g. a sample covariance
            # passed as --sigcov0) has eigenvalues ~ -1e-17, whose square root would turn the whole chain into NaN
            # (the reference's sqrtm tolerates them, pspec.py:355)
            out[i] = (None, np.clip(d, 0.0, None))
        else:
            todo.append(i)
    if todo:
        Sh = np.stack([0.5 * (np.asarray(covs[i]) + np.asarray(covs[i]).conj().T) for i in todo])
        w, V = (eigh or (lambda m: device_eigh(m, device)))(Sh)
        for j, i in enumerate(todo):
            out[i] = (np.ascontiguousarray(V[j], dtype=np.complex128), np.ascontiguousarray(np.clip(w[j], 0.0, None), dtype=np.float64))
    return out


def _analyse_signal_cov(S, device=0, eigh=None):
    """One covariance: (basis0 or None, lam0sq); see :func:`_analyse_signal_covs`."""
    return _analyse_signal_covs([S], device=device, eigh=eigh)[0]


def _noise_model(Ninv, flags, nfreqs, need_sqrt):
    """Split the inverse noise covariance into what the device needs.

    Returns ``(ninv_diag, ninv_dense, nih_dense)``: the real diagonal (chi^2 weights, pspec.py:452) and,
    for a non-diagonal ``Ninv``, the full matrix plus -- only when the reference's draws are injected
    (``need_sqrt``) -- the principal square root of the flagged matrix (pspec.py:362).  With flagged
    channels and a non-diagonal ``Ninv`` the flags are applied to rows *and* columns (the reference's
    ``flags.T * Ninv * flags`` masks columns only, its own FIXME at pspec.py:361; the two agree without
    flags or for a diagonal ``Ninv``).
    """
    Ninv = np.asarray(Ninv)
    if Ninv.ndim == 3:
        raise NotImplementedError("per-time Ninv (Ntimes, Nfreqs, Nfreqs) is not supported by the reference's "
                                  "build_matrices either (pspec.py:361)")
    if Ninv.shape != (nfreqs, nfreqs):
        raise ValueError("Ninv shape must be (Nfreqs, Nfreqs)")
    d = np.ascontiguousarray(np.real(np.diagonal(Ninv)), dtype=np.float64)
    if not np.any(Ninv - np.diag(np.diagonal(Ninv)) != 0):
        return d, None, None
    dense = np.ascontiguousarray(Ninv, dtype=np.complex128)
    nih = None
    if np.asarray(flags).ndim == 2:
        raise NotImplementedError("per-time flags need a diagonal Ninv")
    if need_sqrt:
        w = np.asarray(flags).astype(float)
        Ni = w[:, None] * dense * w[None, :]
        ev, V = np.linalg.eigh(0.5 * (Ni + Ni.conj().T))
        nih = np.ascontiguousarray((V * np.sqrt(np.clip(ev, 0.0, None))) @ V.conj().T)
    return d, dense, nih


def _time_noise_model(Ninv, flags, ntimes, nfreqs):
    """Per-time inverse noise covariance ``Ninv`` of shape ``(Ntimes, Nfreqs, Nfreqs)`` (an extension: the reference's
    build_matrices takes one matrix, pspec.py:361).  Returns ``(Ninv, flags, ninv_t)``:

    - ``Ninv`` 2-D: unchanged, ``ninv_t = None``;
    - all slices identical: ``Ninv[0]`` and ``ninv_t = None`` -- the chain is exactly the one of the 2-D matrix;
    - all slices diagonal: ``Ninv = None``, the flags as ``(Ntimes, Nfreqs)`` (1-D flags are broadcast) and ``ninv_t``, the
      ``(Ntimes, Nfreqs)`` diagonals: time t uses ``Ninv[t]`` in its GCR system and as its chi^2 / ln-posterior weight,
      one factorisation per time on the device (csrc/hp_pertime.cu).

    A non-diagonal slice raises ``NotImplementedError`` (a dense rank change per time); a diagonal that is not real, finite
    and non-negative raises ``ValueError``.
    """
    Ninv = np.asarray(Ninv)
    if Ninv.ndim != 3:
        return Ninv, flags, None
    if Ninv.shape != (ntimes, nfreqs, nfreqs):
        raise ValueError("Ninv shape must be (Ntimes, Nfreqs, Nfreqs) or (Nfreqs, Nfreqs)")
    if np.all(Ninv == Ninv[0]):
        return Ninv[0], flags, None
    d = np.diagonal(Ninv, axis1=1, axis2=2)
    if np.count_nonzero(Ninv) != np.count_nonzero(d):
        raise NotImplementedError("per-time Ninv: only diagonal slices are supported (a non-diagonal N_t^-1 is a dense rank "
                                  "change per time)")
    flags, ninv_t = _time_noise_diag(d, flags, ntimes, nfreqs)
    return None, flags, ninv_t


def _time_noise_diag(d, flags, ntimes, nfreqs):
    """``(flags, ninv_t)`` of per-time noise given by its ``(Ntimes, Nfreqs)`` diagonals ``d``: checked to be real, finite and
    non-negative (``ValueError`` otherwise), the flags broadcast to ``(Ntimes, Nfreqs)``."""
    d = np.asarray(d)
    if d.shape != (ntimes, nfreqs):
        raise ValueError("per-time noise diagonals must have shape (Ntimes, Nfreqs)")
    if np.any(np.imag(d) != 0) or not np.all(np.isfinite(d)) or np.any(np.real(d) < 0):
        raise ValueError("per-time Ninv: the diagonals must be real, finite and non-negative")
    flags = np.asarray(flags)
    if flags.ndim == 1:
        flags = np.broadcast_to(flags, (ntimes, nfreqs))
    return np.ascontiguousarray(flags), np.ascontiguousarray(np.real(d), dtype=np.float64)


# --------------------------------------------------------------------------------------------
class GibbsEngine:
    """Batched Gibbs sampler: ``nchains`` baselines of identical shape resident on one GPU.

    This is the production interface (one process per GPU, baselines sharded across ranks with
    no collective on the hot path); the drop-in functions below are thin single-chain wrappers.
    """

    def __init__(self, nchains, ntimes, nfreqs, nmodes, max_iters, rng="philox", cg_compat=False,
                 refresh_omega=True, keep=("cr", "fg", "chisq"), general_basis0=False, seed=0, device=0,
                 stream=None, profile=False, force_dense_transforms=False, dense_noise=False, substreams=1,
                 time_flags=False, force_dense_solve=False, ring_iters=0):
        self._h = None
        L = _lib.lib()
        cfg = _lib.HPConfig()
        cfg.device = int(device)
        cfg.nchains, cfg.ntimes, cfg.nfreqs, cfg.nmodes = int(nchains), int(ntimes), int(nfreqs), int(nmodes)
        cfg.rng_mode = _lib.HP_RNG_PHILOX if rng == "philox" else _lib.HP_RNG_INJECTED
        cfg.cg_compat = int(bool(cg_compat))
        cfg.refresh_omega = int(bool(refresh_omega))
        k = 0
        for name, bit in (("cr", _lib.HP_KEEP_CR), ("fg", _lib.HP_KEEP_FG), ("chisq", _lib.HP_KEEP_CHISQ)):
            if name in keep:
                k |= bit
        cfg.keep = k
        cfg.max_iters = int(max_iters)
        cfg.general_basis0 = int(bool(general_basis0))
        cfg.profile = int(bool(profile))
        cfg.force_dense_transforms = int(bool(force_dense_transforms))
        cfg.dense_noise = int(bool(dense_noise))
        cfg.substreams = int(substreams)
        cfg.time_flags = int(bool(time_flags))
        cfg.force_dense_solve = int(bool(force_dense_solve or _FORCE_DENSE_SOLVE))
        cfg.ring_iters = int(ring_iters)
        cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        cfg.stream = stream
        h = _lib.C.c_void_p()
        _lib.check(L.hp_engine_create(_lib.C.byref(cfg), _lib.C.byref(h)))
        self._h = h
        self.nchains, self.ntimes, self.nfreqs, self.nmodes = int(nchains), int(ntimes), int(nfreqs), int(nmodes)
        self.max_iters = int(max_iters)
        self.rng = rng
        self.keep = tuple(keep)
        self.general_basis0 = bool(general_basis0)
        self.time_flags = bool(time_flags)
        self.summary_what = ()
        self.summary_batch = 0

    def close(self):
        if self._h is not None:
            _lib.lib().hp_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- loading
    def load_chain(self, chain, vis, flags, fgmodes, ninv_diag, lam0sq, ps_prior=None, basis0=None, ninv_dense=None,
                   nih_dense=None, ninv_t=None):
        """Load one baseline.  ``ninv_t``: ``(Ntimes, Nfreqs)`` diagonal of the inverse noise covariance of every time (engines
        with ``time_flags``; ``ninv_diag`` is then ignored): the chain runs one factorisation per time
        (``hp_engine_load_chain_time_noise``)."""
        T, n, m = self.ntimes, self.nfreqs, self.nmodes
        vis = _lib.c128(vis)
        assert vis.shape == (T, n)
        fl = np.ascontiguousarray(np.asarray(flags).astype(np.uint8))
        if self.time_flags:
            assert fl.shape == (T, n), "`flags` array must have shape (Ntimes, Nfreqs) in per-time mode"
        else:
            assert fl.shape == (n,), "`flags` array must have shape (Nfreqs,)"
        F = _lib.c128(fgmodes)
        assert F.shape == (n, m), "fgmodes must have shape (Nfreqs, Nmodes)"
        l0 = _lib.f64(lam0sq)
        pr = None if ps_prior is None else _lib.f64(ps_prior)
        b0 = None if basis0 is None else _lib.c128(basis0)
        if ninv_t is not None:
            if not self.time_flags:
                raise ValueError("ninv_t (per-time noise) needs an engine created with time_flags=True")
            nt = _lib.f64(ninv_t)
            assert nt.shape == (T, n), "ninv_t must have shape (Ntimes, Nfreqs)"
            _lib.check(_lib.lib().hp_engine_load_chain_time_noise(self._h, int(chain), _lib.ptr(vis), _lib.ptr(fl), _lib.ptr(F),
                                                                  _lib.ptr(nt), _lib.ptr(b0), _lib.ptr(l0), _lib.ptr(pr)))
            return
        nd = _lib.f64(ninv_diag)
        if ninv_dense is not None:
            nD = _lib.c128(ninv_dense)
            nH = None if nih_dense is None else _lib.c128(nih_dense)
            _lib.check(_lib.lib().hp_engine_load_chain_dense(self._h, int(chain), _lib.ptr(vis), _lib.ptr(fl), _lib.ptr(F),
                                                             _lib.ptr(nd), _lib.ptr(nD), _lib.ptr(nH), _lib.ptr(b0),
                                                             _lib.ptr(l0), _lib.ptr(pr)))
            return
        _lib.check(_lib.lib().hp_engine_load_chain(self._h, int(chain), _lib.ptr(vis), _lib.ptr(fl), _lib.ptr(F),
                                                   _lib.ptr(nd), _lib.ptr(b0), _lib.ptr(l0), _lib.ptr(pr)))

    def set_draws(self, chain, omega_a, omega_b, s_draws):
        oa = None if omega_a is None else _lib.c128(omega_a)
        ob = None if omega_b is None else _lib.c128(omega_b)
        sd = None if s_draws is None else _lib.f64(s_draws)
        nd = 0 if sd is None else sd.shape[0]
        _lib.check(_lib.lib().hp_engine_set_draws(self._h, int(chain), _lib.ptr(oa), _lib.ptr(ob), _lib.ptr(sd), int(nd)))

    # -- running
    def run(self, niter):
        _lib.check(_lib.lib().hp_engine_run(self._h, int(niter)))

    def host_buffers(self, iters=None, pinned=True, iter_major=False):
        """Host arrays for :meth:`run_to_host` (page-locked by default): ``[nchains][iters][...]``, or -- ``iter_major`` --
        ``[iters][nchains][...]`` for the big arrays (signal_cr, fg_amps, chisq): an iteration's array of all chains is then
        one contiguous block on both sides of the copy (``signal_ps`` / ``ln_post`` stay ``[nchains][iters]``)."""
        iters = self.max_iters if iters is None else iters
        mk = _lib.pinned_empty if pinned else (lambda shape, dt: np.empty(shape, dtype=dt))
        C, T, n, m = self.nchains, self.ntimes, self.nfreqs, self.nmodes
        lead = (iters, C) if iter_major else (C, iters)
        out = {"signal_ps": mk((C, iters, n), np.float64), "ln_post": mk((C, iters), np.float64)}
        if "cr" in self.keep:
            out["signal_cr"] = mk(lead + (T, n), np.complex128)
        if "fg" in self.keep:
            out["fg_amps"] = mk(lead + (T, m), np.complex128)
        if "chisq" in self.keep:
            out["chisq"] = mk(lead + (T, n), np.float64)
        return out

    def run_to_host(self, niter, bufs, first_iter=0, iter_major=False, read_ahead=0):
        """Run ``niter`` iterations and stream every iteration's arrays into ``bufs`` (from
        :meth:`host_buffers`) while the next iteration computes; returns when all data has landed.
        Iteration ``i`` of the chain lands in slot ``i - first_iter`` of the host arrays: a bounded staging area is
        re-used chunk after chunk by passing the index of the chunk's first iteration.  ``read_ahead`` > 0: the next
        iterations of the chain (at most ring_iters - 1) are computed into free device ring slots before the call
        returns, so that the next chunk starts copying at once (``hp_host_sink.read_ahead``; pass 0 in the last call)."""
        sink = _lib.HPHostSink()
        for k in ("signal_ps", "ln_post", "signal_cr", "fg_amps", "chisq"):
            a = bufs.get(k)
            if a is not None:
                big = iter_major and k in ("signal_cr", "fg_amps", "chisq")
                assert a.flags["C_CONTIGUOUS"] and a.shape[1 if big else 0] == self.nchains
                setattr(sink, k, a.ctypes.data)
        sink.iters = int(bufs["signal_ps"].shape[1])
        sink.first_iter = int(first_iter)
        sink.iter_major = int(bool(iter_major))
        sink.read_ahead = int(read_ahead)
        _lib.check(_lib.lib().hp_engine_run_to_host(self._h, int(niter), _lib.C.byref(sink)))

    def gcr(self):
        _lib.check(_lib.lib().hp_engine_gcr(self._h))

    def sync(self):
        _lib.check(_lib.lib().hp_engine_sync(self._h))

    def rewind(self):
        _lib.check(_lib.lib().hp_engine_rewind(self._h))

    @property
    def iterations_done(self):
        return _lib.lib().hp_engine_iterations_done(self._h)

    @property
    def launch_count(self):
        return _lib.lib().hp_engine_launch_count(self._h)

    def pt_form(self):
        """Per-time flags: ("low-rank" | "direct", largest number of channels flagged at one time beyond the all-times
        mask) for the chains loaded so far (csrc/hp_ptlow.cu / csrc/hp_pertime.cu)."""
        import ctypes as C
        low, kmax = C.c_int(0), C.c_int(0)
        _lib.check(_lib.lib().hp_engine_pt_form(self._h, C.byref(low), C.byref(kmax)))
        return ("low-rank" if low.value else "direct"), kmax.value

    def set_chain_ids(self, ids):
        """Philox chain id of every chain (default: its index).  Passing the global baseline indices (and the same
        seed on every rank) makes the device draws independent of how baselines are sharded over GPUs."""
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        assert ids.shape == (self.nchains,)
        _lib.check(_lib.lib().hp_engine_set_chain_ids(self._h, _lib.ptr(ids)))

    def set_substreams(self, n):
        _lib.check(_lib.lib().hp_engine_set_substreams(self._h, int(n)))

    def set_profile(self, on):
        _lib.check(_lib.lib().hp_engine_set_profile(self._h, int(bool(on))))

    def kernel_ms(self, reset=False):
        ms = np.zeros(_lib.HP_NUM_KERNEL_CLASSES)
        nl = np.zeros(_lib.HP_NUM_KERNEL_CLASSES, dtype=np.int32)
        _lib.check(_lib.lib().hp_engine_kernel_ms(self._h, _lib.ptr(ms), _lib.ptr(nl), int(reset)))
        names = [_lib.lib().hp_kernel_class_name(i).decode() for i in range(_lib.HP_NUM_KERNEL_CLASSES)]
        return {k: (float(a), int(b)) for k, a, b in zip(names, ms, nl)}

    def info(self):
        out = np.zeros(self.nchains, dtype=np.int32)
        _lib.check(_lib.lib().hp_engine_info(self._h, _lib.ptr(out)))
        return out

    # -- reading
    def _read(self, chain, buf, shape, dtype, iter0=0, niter=0):
        out = np.empty(shape, dtype=dtype)
        _lib.check(_lib.lib().hp_engine_read(self._h, int(chain), int(buf), int(iter0), int(niter), _lib.ptr(out),
                                             out.nbytes))
        return out

    def signal_ps(self, chain, iter0=0, niter=None):
        niter = self.iterations_done - iter0 if niter is None else niter
        return self._read(chain, _lib.HP_BUF_PS, (niter, self.nfreqs), np.float64, iter0, niter)

    def ln_post(self, chain, iter0=0, niter=None):
        niter = self.iterations_done - iter0 if niter is None else niter
        return self._read(chain, _lib.HP_BUF_LNPOST, (niter,), np.float64, iter0, niter)

    def signal_cr(self, chain, iter0=0, niter=None):
        niter = self.iterations_done - iter0 if niter is None else niter
        return self._read(chain, _lib.HP_BUF_CR, (niter, self.ntimes, self.nfreqs), np.complex128, iter0, niter)

    def fg_amps(self, chain, iter0=0, niter=None):
        niter = self.iterations_done - iter0 if niter is None else niter
        return self._read(chain, _lib.HP_BUF_FG, (niter, self.ntimes, self.nmodes), np.complex128, iter0, niter)

    def chisq(self, chain, iter0=0, niter=None):
        niter = self.iterations_done - iter0 if niter is None else niter
        return self._read(chain, _lib.HP_BUF_CHISQ, (niter, self.ntimes, self.nfreqs), np.float64, iter0, niter)

    def last_gcr(self, chain):
        """(Ntimes, Nfreqs + Nmodes) solution of the most recent GCR step (pspec.py:301)."""
        s = self._read(chain, _lib.HP_BUF_LAST_CR, (self.ntimes, self.nfreqs), np.complex128)
        f = self._read(chain, _lib.HP_BUF_LAST_FG, (self.ntimes, self.nmodes), np.complex128)
        return np.concatenate([s, f], axis=1)

    def current_ps(self, chain):
        return self._read(chain, _lib.HP_BUF_PS_CUR, (self.nfreqs,), np.float64)

    def signal_S(self, chain):
        out = np.empty((self.nfreqs, self.nfreqs), dtype=np.complex128)
        _lib.check(_lib.lib().hp_engine_read_signal_S(self._h, int(chain), _lib.ptr(out)))
        return out

    # -- posterior summary (hp_engine_set_summary)
    _SUMMARY = {"cr": (_lib.HP_SUMMARY_CR, "signal_cr"), "fg": (_lib.HP_SUMMARY_FG, "fg_amps")}

    def set_summary(self, what=("cr", "fg"), burn_in=0, thin=1, batch=0):
        """(Re)start the on-device posterior moments of ``signal_cr`` ("cr") and / or ``fg_amps`` ("fg"): of the iterations
        computed from now on the first ``burn_in`` are skipped, then every ``thin``-th is accumulated.  ``what=()`` stops.
        ``batch > 0`` also keeps batch means over ``batch`` accumulated samples, for the Monte-Carlo standard error and
        effective sample size of each mean (:meth:`summary`)."""
        what = tuple(what)
        bad = [w for w in what if w not in self._SUMMARY]
        if bad:
            raise ValueError(f"set_summary: unknown quantities {bad} (expected 'cr' and / or 'fg')")
        mask = 0
        for w in what:
            mask |= self._SUMMARY[w][0]
        _lib.check(_lib.lib().hp_engine_set_summary_batched(self._h, mask, int(burn_in), int(thin), int(batch)))
        self.summary_what = what
        self.summary_batch = int(batch)

    def summary(self, chain):
        """``{"count", "signal_cr_mean", "signal_cr_var", "fg_amps_mean", "fg_amps_var"}`` of one chain, with only the
        quantities being accumulated: means (Ntimes, Nfreqs | Nmodes) complex128, variances E|x - mean|^2 (ddof = 0, as
        ``numpy.var`` of the complex samples), count = accumulated iterations.

        With batch means on (``set_summary(batch=b)``) the dict also has ``"<name>_mcse"`` and ``"<name>_ess"`` (float64,
        same shape), ``"batch"`` and ``"nbatch"``: with k = count, nb = k // b complete batches of means Ybar_j and their
        mean Ybar, ``s2_bm = sum_j |Ybar_j - Ybar|^2 / (nb - 1)``, ``mcse = sqrt(b s2_bm / k)`` (the standard error of the
        mean) and ``ess = var / mcse**2``; NaN while nb < 2."""
        if not self.summary_what:
            raise ValueError("summary: no posterior summary is being accumulated (set_summary)")
        out = {}
        count, nbatch = _lib.C.c_int(0), _lib.C.c_int(0)
        for w in self.summary_what:
            bit, name = self._SUMMARY[w]
            width = self.nfreqs if w == "cr" else self.nmodes
            mean = np.empty((self.ntimes, width), dtype=np.complex128)
            var = np.empty((self.ntimes, width), dtype=np.float64)
            _lib.check(_lib.lib().hp_engine_read_summary(self._h, int(chain), bit, _lib.ptr(mean), _lib.ptr(var), mean.nbytes,
                                                         _lib.C.byref(count)))
            out[f"{name}_mean"], out[f"{name}_var"] = mean, var
            if self.summary_batch > 0:
                mcse = np.empty((self.ntimes, width), dtype=np.float64)
                ess = np.empty((self.ntimes, width), dtype=np.float64)
                _lib.check(_lib.lib().hp_engine_read_summary_mcse(self._h, int(chain), bit, _lib.ptr(mcse), _lib.ptr(ess),
                                                                  mcse.nbytes, _lib.C.byref(nbatch)))
                out[f"{name}_mcse"], out[f"{name}_ess"] = mcse, ess
        out["count"] = int(count.value)
        if self.summary_batch > 0:
            out["batch"], out["nbatch"] = self.summary_batch, int(nbatch.value)
        return out



# Device slots of the big per-iteration outputs when they are streamed to the host (cfg.ring_iters): the device footprint
# of a chain does not grow with Niter (the reference keeps one baseline's samples in host RAM, pspec.py:590-596).
_RING_ITERS = 3
_STAGING_BYTES = int(float(os.environ.get("HP_STAGING_GB", "2")) * 2 ** 30)   # page-locked staging area


def _device_bytes_per_chain(ntimes, nfreqs, nmodes, Niter, rng, big_per_iter, general, dense, per_time, summary,
                            batch=False, time_noise=False):
    """Estimated device memory of one chain of an engine (how many chains share an engine in gibbs_sample_batch).
    ``big_per_iter``: host bytes of one chain's kept outputs per iteration (``_big_bytes_per_iter`` / nchains).
    ``summary`` / ``batch``: the posterior moments / their batch means are accumulated.  ``time_noise``: some chain of the
    engine has per-time noise (the weights of every time)."""
    Np = 32 * ((nfreqs + nmodes + 31) // 32)
    Tp = 16 * ((ntimes + 15) // 16)
    per_chain = 16 * Tp * Np * (4 if rng == "numpy" else 3) + 16 * Tp * nfreqs * 3 + 16 * nfreqs * Np * (2 if general else 1) \
        + 8 * 3 * (Np * Np // 2 + 18 * Np) * 2 + _RING_ITERS * big_per_iter + 8 * Niter * nfreqs * (2 if rng == "numpy" else 1)
    if dense:
        per_chain += 16 * nfreqs * nfreqs * 3 + 16 * Tp * nfreqs * 2
    if per_time:
        # low-rank form (csrc/hp_ptlow.cu): Nfreqs more right-hand sides ride through the solve, plus P and the flag lists
        Tx = Tp + 16 * ((nfreqs + 15) // 16)
        per_chain = per_chain * Tx // Tp + 16 * Tx * (1 + nmodes) * Np + 8 * Tx * nfreqs + 16 * nfreqs * nfreqs + 132 * ntimes
    if summary:
        per_chain += 24 * ntimes * (nfreqs + nmodes)   # posterior moments: complex mean + real M2 per element
    if batch:
        per_chain += 24 * ntimes * (nfreqs + nmodes)   # batch means: complex snapshot + real M2_bm per element
    if time_noise:
        per_chain += 8 * Tp * nfreqs   # diag(N_t^-1) of every (padded) time
    return per_chain


def _check_summary(summary):
    """Validate the ``summary=`` argument of the sampling functions: None, or a dict with the optional keys ``burn_in``
    (integer >= 0, default 0), ``thin`` (integer >= 1, default 1) and ``batch`` (integer >= 0, batch means over that many
    accumulated samples, 0: off).  Returns None or ``{"burn_in", "thin"}``, plus ``"batch"`` when it was given."""
    if summary is None:
        return None
    if not isinstance(summary, dict):
        raise TypeError("summary must be None or a dict(burn_in=..., thin=..., batch=...)")
    unknown = set(summary) - {"burn_in", "thin", "batch"}
    if unknown:
        raise ValueError(f"summary: unknown keys {sorted(unknown)} (expected burn_in, thin, batch)")
    out = {"burn_in": summary.get("burn_in", 0), "thin": summary.get("thin", 1)}
    if "batch" in summary:
        out["batch"] = summary["batch"]
    for k, v in out.items():
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
            raise TypeError(f"summary: {k} must be an integer")
        out[k] = int(v)
    if out["burn_in"] < 0:
        raise ValueError("summary: burn_in must be >= 0")
    if out["thin"] < 1:
        raise ValueError("summary: thin must be >= 1")
    if out.get("batch", 0) < 0:
        raise ValueError("summary: batch must be >= 0")
    return out


def _big_bytes_per_iter(nchains, ntimes, nfreqs, nmodes, keep):
    per = 0
    if "cr" in keep:
        per += ntimes * nfreqs * 16
    if "fg" in keep:
        per += ntimes * nmodes * 16
    if "chisq" in keep:
        per += ntimes * nfreqs * 8
    return nchains * (per + nfreqs * 8 + 8)


# threads of the staging -> destination copy: HP_COPY_THREADS, else the host cores shared by the ranks of this node (at most 16)
_COPY_THREADS = max(1, int(os.environ.get("HP_COPY_THREADS", "0")) or
                    min(16, (os.cpu_count() or 1) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))
_copy_pool = None


def _scatter_chunk(dest, stage, done, c):
    """Move iterations [done, done + c) of a chunk from the iteration-major staging arrays ``stage[k][iter][chain]...`` into
    the chain-major destination arrays ``dest[k][chain][iter]...``.  One numpy copy of a headline-size chunk (1.3 GB per
    iteration) runs at a few GB/s on one core -- ten times longer than the GPU needs for the iteration -- so the chains are
    split over a small thread pool (numpy releases the GIL while it copies)."""
    global _copy_pool
    jobs = []
    for k, a in dest.items():
        if a is None:
            continue
        big = k in ("signal_cr", "fg_amps", "chisq")
        nch = a.shape[0]
        if not big or _COPY_THREADS == 1 or stage[k][:c].nbytes < (32 << 20):
            a[:, done:done + c] = np.swapaxes(stage[k][:c], 0, 1) if big else stage[k][:, :c]
            continue
        step = -(-nch // _COPY_THREADS)
        for c0 in range(0, nch, step):
            jobs.append((a, stage[k], c0, min(nch, c0 + step)))
    if jobs:
        if _copy_pool is None:
            from concurrent.futures import ThreadPoolExecutor
            _copy_pool = ThreadPoolExecutor(max_workers=_COPY_THREADS, thread_name_prefix="hp-copy")

        def work(job):
            a, st, c0, c1 = job
            a[c0:c1, done:done + c] = np.swapaxes(st[:c, c0:c1], 0, 1)

        list(_copy_pool.map(work, jobs))


def _staged_run(eng, Niter, dest, write_Niter=None, after_chunk=None):
    """Run ``Niter`` iterations of ``eng`` through a bounded page-locked staging area.

    ``dest``: dict of host arrays ``[nchains][Niter][...]`` (numpy arrays or ``np.memmap``) that receive the samples;
    ``after_chunk(done)`` is called whenever ``done`` is a multiple of ``write_Niter`` (and at the end).
    """
    per_iter = _big_bytes_per_iter(eng.nchains, eng.ntimes, eng.nfreqs, eng.nmodes, eng.keep)
    chunk = max(1, min(Niter, _STAGING_BYTES // max(per_iter, 1)))
    if write_Niter:
        chunk = min(chunk, write_Niter)
    stage = eng.host_buffers(chunk, iter_major=True)   # iteration-major staging: one plain copy per array and iteration
    done = 0
    while done < Niter:
        c = min(chunk, Niter - done)
        if write_Niter:   # never run past a write boundary (pspec.py:625: files every write_Niter iterations)
            c = min(c, write_Niter - done % write_Niter)
        # read-ahead: the device computes the next iterations while this chunk's last copies land and while the host moves the
        # chunk out of the staging area; not across a write boundary (the callback reads the chain's current signal_S)
        at_boundary = after_chunk is not None and (done + c == Niter or (write_Niter and (done + c) % write_Niter == 0))
        ra = 0 if (done + c >= Niter or at_boundary) else _RING_ITERS - 1
        eng.run_to_host(c, stage, first_iter=done, iter_major=True, read_ahead=ra)
        _scatter_chunk(dest, stage, done, c)
        done += c
        if after_chunk is not None and (done == Niter or (write_Niter and done % write_Niter == 0)):
            after_chunk(done)

# --------------------------------------------------------------------------------------------
class GCRMatrices:
    """What :func:`build_matrices` returns on the device path.

    The reference materialises sqrtm(S), sqrtm(N^-1), A and pinv(A) (pspec.py:355-372); the GPU
    path never forms them (it factors the whitened Hermitian system instead), so this object just
    carries the operands.  ``m[0][1]`` (S) and ``m[0][2]`` (N^-1 with the flags applied) index like
    the reference's list so code that peeks at them keeps working.
    """

    def __init__(self, flags, signal_S, Ninv, fgmodes):
        self.flags = np.asarray(flags, dtype=bool)
        self.S = np.array(signal_S, dtype=complex)
        fl = self.flags.astype(float)
        self.Ni = (fl * np.asarray(Ninv) * fl).astype(complex)  # pspec.py:361
        self.fgmodes = np.asarray(fgmodes)

    def __getitem__(self, i):
        if i == 0:
            return {1: self.S, 2: self.Ni}
        raise IndexError("the device path does not materialise A / pinv(A) (pspec.py:365-372)")


def build_matrices(Nparams, flags, signal_S, Ninv, fgmodes):
    """pspec.py:325-374."""
    nfreqs = np.asarray(signal_S).shape[0]
    assert Nparams == nfreqs + np.asarray(fgmodes).shape[1]
    return GCRMatrices(flags, signal_S, Ninv, fgmodes)


def _check_per_time_supported(solver, basis0, ninv_dense):
    """Per-time flags ``(Ntimes, Nfreqs)`` are an extension of the reference (it asserts 1-D flags,
    pspec.py:428, and its driver collapses them, run-hydra-pspec.py:520-526): every time gets its own
    factorisation (csrc/hp_pertime.cu), or -- when no time has more than 64 channels flagged beyond the all-times
    mask -- as a low-rank correction of one shared factorisation (csrc/hp_ptlow.cu)."""
    if solver != "exact":
        raise NotImplementedError("per-time flags: only solver='exact' (the reference has no per-time CG to reproduce)")
    # (a non-delay-diagonal S_initial is taken by the low-rank form only: the engine refuses it when Nfreqs + Nmodes > 448 or
    #  when a time has more than 64 channels flagged beyond the all-times mask)
    if ninv_dense is not None:
        raise NotImplementedError("per-time flags need a diagonal Ninv")


def _single_chain_engine(vis, flags, S, fgmodes, Ninv, ps_prior, max_iters, rng, solver, map_estimate, keep,
                         seed, device, s_uniforms=None, ring_iters=0, ninv_t=None):
    """Engine with one chain loaded and (numpy mode) its draws injected.  ``ninv_t``: per-time noise diagonals
    (:func:`_time_noise_model`; ``Ninv`` is then not read)."""
    vis = np.asarray(vis)
    ntimes, nfreqs = vis.shape
    nmodes = np.asarray(fgmodes).shape[1]
    per_time = np.asarray(flags).ndim == 2
    if ninv_t is not None:
        ninv_diag, ninv_dense, nih_dense = None, None, None
    else:
        ninv_diag, ninv_dense, nih_dense = _noise_model(Ninv, flags, nfreqs, need_sqrt=(rng == "numpy" and not map_estimate))
    basis0, lam0sq = _analyse_signal_cov(S, device=device)
    if solver is None:
        solver = "reference-cg" if (rng == "numpy" and not per_time) else "exact"
    if solver not in ("reference-cg", "exact"):
        raise ValueError("solver must be 'reference-cg' or 'exact'")
    if per_time:
        _check_per_time_supported(solver, basis0, ninv_dense)
    eng = GibbsEngine(1, ntimes, nfreqs, nmodes, max_iters, rng=rng, cg_compat=(solver == "reference-cg"),
                      refresh_omega=(rng == "philox"), keep=keep, general_basis0=basis0 is not None,
                      seed=0 if seed is None else seed, device=device,
                      force_dense_transforms=_FORCE_DENSE_TRANSFORMS and not per_time, dense_noise=ninv_dense is not None,
                      time_flags=per_time, ring_iters=ring_iters)
    eng.load_chain(0, vis, flags, fgmodes, ninv_diag, lam0sq, ps_prior=ps_prior, basis0=basis0, ninv_dense=ninv_dense,
                   nih_dense=nih_dense, ninv_t=ninv_t)
    if rng == "numpy":
        if map_estimate:
            oma = omb = None  # pspec.py:210-212
        else:
            oma, omb = _reference_gcr_draws(ntimes, nfreqs)
        sd = None
        if s_uniforms is not None:
            sd = _s_draws_from_uniforms(s_uniforms, ps_prior if ps_prior is not None else np.zeros((2, nfreqs)), ntimes)
        eng.set_draws(0, oma, omb, sd)
    return eng


def gcr_fgmodes(vis, w, matrices, fgmodes, f0=None, nproc=1, map_estimate=False, verbose=False,
                rng="numpy", solver=None, device=0):
    """GCR step for all times (pspec.py:238-310).  Returns ``(Ntimes, Nfreqs + Nmodes)`` samples.

    ``f0`` / ``nproc`` are accepted for signature compatibility (the reference's CG ignores the
    initial guess up to its tolerance; the device solve is direct and batched over times).
    """
    S = matrices[0][1]
    Ni = matrices[0][2]
    vis = np.asarray(vis)
    # the reference multiplies the data by w again (pspec.py:221); Ni already carries the flags
    eng = _single_chain_engine(vis, np.asarray(w), S, fgmodes, Ni, None, 1, rng, solver, map_estimate, (), None, device)
    try:
        eng.gcr()
        out = eng.last_gcr(0)
    finally:
        eng.close()
    return out


def sample_S(s=None, sk=None, prior=None, device=0):
    """pspec.py:67-127.  Draws one uniform per delay bin from numpy's global stream, like the
    reference (explicitly for prior-bounded bins, inside ``invgamma.rvs`` for the others)."""
    if s is None and sk is None:
        raise ValueError("Must pass in s (real space) or sk (Fourier space) vector.")
    if s is None:
        sk = np.asarray(sk)
        n = sk.shape[1]
        U = _unitary_dft(n)
        s = (sk / np.sqrt(n)) @ U.conj()  # sk = sqrt(n) U s  =>  s = U^H sk / sqrt(n)
    s = _lib.c128(s)
    nobs, nfreqs = s.shape
    pr = _check_prior(prior, nfreqs)
    u = np.array([np.random.uniform() for _ in range(nfreqs)])
    draws = _lib.f64(_s_draws_from_uniforms(u, pr, nobs)[0])
    out = np.empty(nfreqs)
    pr = _lib.f64(pr)
    _lib.check(_lib.lib().hp_sample_S(int(device), int(nobs), int(nfreqs), _lib.ptr(s), _lib.ptr(pr), _lib.ptr(draws),
                                      _lib.ptr(out)))
    return out


def gibbs_step_fgmodes(vis, flags, signal_S, fgmodes, Ninv, ps_prior=None, f0=None, nproc=1, map_estimate=False,
                       verbose=False, rng="numpy", solver=None, device=0):
    """One Gibbs iteration (pspec.py:377-490).  ``vis`` is expected pre-multiplied by the flags,
    as gibbs_sample_with_fg passes it (pspec.py:613)."""
    vis = np.asarray(vis)
    nfreqs = vis.shape[1]
    flags = np.asarray(flags)
    assert flags.shape == (nfreqs,), "`flags` array must have shape (Nfreqs,)"
    Ninv, flags, ninv_t = _time_noise_model(Ninv, flags, vis.shape[0], nfreqs)
    pr = _check_prior(ps_prior, nfreqs)
    u = np.array([np.random.uniform() for _ in range(nfreqs)])[None, :] if rng == "numpy" else None
    eng = _single_chain_engine(vis, flags, signal_S, fgmodes, Ninv, pr, 1, rng, solver, map_estimate,
                               ("cr", "fg", "chisq"), None, device, s_uniforms=u, ninv_t=ninv_t)
    try:
        eng.run(1)
        out = (eng.signal_cr(0)[0], eng.signal_S(0), eng.signal_ps(0)[0], eng.fg_amps(0)[0], eng.chisq(0)[0],
               float(eng.ln_post(0)[0]))
    finally:
        eng.close()
    if verbose:
        print(f"{out[5]:<12.1f}")
    return out


def gibbs_sample_with_fg(vis, flags, S_initial, fgmodes, Ninv, ps_prior, Niter=100, seed=None, verbose=True,
                         nproc=1, write_Niter=100, out_dir=None, map_estimate=False, rng="numpy", solver=None,
                         device=0, summary=None):
    """Gibbs chain for one baseline (pspec.py:493-658); same arguments and return tuple:
    ``signal_cr, signal_S, signal_ps, fg_amps, chisq, ln_post, write_time``.

    ``Ninv`` may be ``(Ntimes, Nfreqs, Nfreqs)``: identical slices run the 2-D path, diagonal slices a per-time noise model
    (time t uses ``Ninv[t]``, :func:`_time_noise_model`; one factorisation per time, ``solver="exact"``).
    Extra keyword arguments: ``rng`` / ``solver`` (see the module docstring) and ``device``.
    ``nproc`` is accepted and ignored (all times are solved in one batched launch).
    ``summary=dict(burn_in=..., thin=...)``: the posterior moments of signal_cr and fg_amps are accumulated on the device
    (:meth:`GibbsEngine.set_summary`) and returned as an 8th element, the dict of :meth:`GibbsEngine.summary`; with
    ``out_dir`` they are also written (``utils.write_summary_files``) at every ``write_Niter`` boundary and at the end.
    ``summary=dict(..., batch=b)`` adds the batch-means Monte-Carlo standard error and effective sample size of each mean.
    """
    t_start = time.perf_counter()
    summary = _check_summary(summary)
    if map_estimate:
        Niter = 1
        write_Niter = 1
    vis = np.asarray(vis)
    ntimes, nfreqs = vis.shape
    flags = np.asarray(flags)
    fgmodes = np.asarray(fgmodes)
    assert flags.shape in ((nfreqs,), (ntimes, nfreqs)), "`flags` array must have shape (Nfreqs,) [or (Ntimes, Nfreqs)]"
    assert fgmodes.shape[0] == nfreqs, "fgmodes must have shape (Nfreqs, Nmodes)"
    Ninv = np.asarray(Ninv)
    if len(Ninv.shape) == 3:
        assert Ninv.shape[0] == ntimes, "Ninv shape must be (Ntimes, Nfreqs, Nfreqs) or (Nfreqs, Nfreqs)"
    Ninv, flags, ninv_t = _time_noise_model(Ninv, flags, ntimes, nfreqs)
    pr = _check_prior(ps_prior, nfreqs)
    u = None
    if rng == "numpy":
        if map_estimate:
            u = np.array([np.random.uniform() for _ in range(nfreqs)])[None, :]  # global stream, not reseeded
        else:
            u = np.random.RandomState(seed).uniform(size=(Niter, nfreqs))  # pspec.py:577
    nmodes = fgmodes.shape[1]
    eng = _single_chain_engine(vis, flags, S_initial, fgmodes, Ninv, pr, Niter, rng, solver, map_estimate,
                               ("cr", "fg", "chisq"), seed, device, s_uniforms=u, ring_iters=_RING_ITERS, ninv_t=ninv_t)
    write_time = [0.0]
    moments = None
    try:
        if summary is not None:
            eng.set_summary(("cr", "fg"), **summary)
        # the reference's return arrays (pspec.py:590-596), filled chunk by chunk from a bounded page-locked staging area
        signal_cr = np.empty((1, Niter, ntimes, nfreqs), dtype=np.complex128)
        signal_ps = np.empty((1, Niter, nfreqs))
        fg_amps = np.empty((1, Niter, ntimes, nmodes), dtype=np.complex128)
        chisq = np.empty((1, Niter, ntimes, nfreqs))
        ln_post = np.empty((1, Niter))
        dest = dict(signal_cr=signal_cr, signal_ps=signal_ps, fg_amps=fg_amps, chisq=chisq, ln_post=ln_post)

        def write(done):
            t0 = time.perf_counter()
            utils.write_numpy_files(out_dir, signal_cr[0, :done], eng.signal_S(0), signal_ps[0, :done], fg_amps[0, :done],
                                    chisq[0, :done], ln_post[0, :done])
            if summary is not None:
                utils.write_summary_files(out_dir, eng.summary(0), **summary)
            write_time[0] += time.perf_counter() - t0

        _staged_run(eng, Niter, dest, write_Niter=write_Niter if out_dir is not None else None,
                    after_chunk=write if out_dir is not None else None)
        bad = eng.info()
        if np.any(bad != 0):
            raise np.linalg.LinAlgError("GCR system not positive definite (Cholesky failed in block column "
                                        f"{int(bad[0]) - 1})")
        signal_S = eng.signal_S(0)
        if summary is not None:
            moments = eng.summary(0)
        signal_cr, signal_ps, fg_amps, chisq, ln_post = signal_cr[0], signal_ps[0], fg_amps[0], chisq[0], ln_post[0]
    finally:
        eng.close()
    write_time = write_time[0]
    if verbose:
        # the reference's per-iteration table (pspec.py:602-604, 306-309, 453-458), printed after the run: the chain never
        # leaves the device between iterations.  Time = wall time of the call / Niter; Info = 0 and |Ax - b| = "exact" for the
        # direct solves (the reference prints its CG status and residual there)
        per_it = (time.perf_counter() - t_start) / max(Niter, 1)
        fl = flags if flags.ndim == 1 else None
        print("Iter     Time [s]    Info    |Ax - b|    Chisq    ln Post")
        print("-----    --------    ----    --------    -----    -------")
        for i, lp in enumerate(ln_post):
            cm = float(chisq[i][:, fl].mean()) if fl is not None else float(chisq[i][flags].mean())
            cs = f"{cm:<9.1e}" if cm > 10 else f"{cm:<9.3f}"
            eff = solver or ("reference-cg" if (rng == "numpy" and flags.ndim == 1) else "exact")
            res = "exact" if eff != "reference-cg" else "(cg)"
            print(f"{i + 1:<9d}{per_it:<12.4f}{0.0:<8.1f}{res:<12s}{cs}{lp:<12.1f}")
        print()
    if summary is not None:
        return signal_cr, signal_S, signal_ps, fg_amps, chisq, ln_post, write_time, moments
    return signal_cr, signal_S, signal_ps, fg_amps, chisq, ln_post, write_time


def gibbs_sample_batch(baselines, Niter=100, seed=None, rng="philox", solver=None, keep=("cr", "fg", "chisq"),
                       write_Niter=100, map_estimate=False, device=0, verbose=False, substreams=1, chain_ids=None, summary=None):
    """Advance the Gibbs chains of several baselines of identical shape together on one GPU.

    This is the batched form of the reference's per-rank loop over baselines
    (run-hydra-pspec.py:487-557): ``baselines`` is a list of dicts with the arguments of
    :func:`gibbs_sample_with_fg` (``vis, flags, S_initial, fgmodes, Ninv, ps_prior`` and optionally
    ``out_dir``); all chains live in one :class:`GibbsEngine` and every kernel launch covers all of
    them.  ``Ninv`` may be ``(Ntimes, Nfreqs, Nfreqs)`` with diagonal slices (per-time noise, :func:`_time_noise_model`); an
    optional ``ninv_t`` of shape ``(Ntimes, Nfreqs)`` gives the same diagonals directly, in place of ``Ninv``, without the
    Ntimes Nfreqs^2 host array.  Such baselines run one factorisation per time.  Returns one ``gibbs_sample_with_fg``-style tuple per baseline (arrays that were not kept
    are ``None``).  With ``rng="numpy"`` each chain gets the reference's draws for ``seed`` (every
    baseline the same streams, as in the reference, where each chain reseeds numpy).

    ``summary=dict(burn_in=..., thin=...)``: the posterior moments of signal_cr and fg_amps are accumulated on the device
    and each tuple gains an 8th element, the dict of :meth:`GibbsEngine.summary`.  Baselines with an ``out_dir`` also get
    them written (``utils.write_summary_files``) at every ``write_Niter`` boundary and at the end.  With ``keep=()`` only
    signal_ps / ln_post leave the device per iteration, and no ``out_dir`` is needed however long the chain.
    ``summary=dict(..., batch=b)`` adds the batch-means Monte-Carlo standard error and effective sample size of each mean.
    """
    summary = _check_summary(summary)
    if not baselines:
        return []
    if map_estimate:
        Niter = 1
        write_Niter = 1
    nb = len(baselines)
    ntimes, nfreqs = np.asarray(baselines[0]["vis"]).shape
    nmodes = np.asarray(baselines[0]["fgmodes"]).shape[1]
    solver_default = solver is None
    if solver is None:
        solver = "reference-cg" if rng == "numpy" else "exact"
    if solver not in ("reference-cg", "exact"):
        raise ValueError("solver must be 'reference-cg' or 'exact'")
    prep = []
    for b in baselines:
        vis = np.asarray(b["vis"])
        assert vis.shape == (ntimes, nfreqs), "all baselines of a batch must have the same (Ntimes, Nfreqs)"
        flags = np.asarray(b["flags"])
        assert flags.shape in ((nfreqs,), (ntimes, nfreqs)), "`flags` array must have shape (Nfreqs,) [or (Ntimes, Nfreqs)]"
        F = np.asarray(b["fgmodes"])
        assert F.shape == (nfreqs, nmodes), "fgmodes must have shape (Nfreqs, Nmodes)"
        if b.get("ninv_t") is not None:
            Ninv = None
            flags, nt = _time_noise_diag(b["ninv_t"], flags, ntimes, nfreqs)
        else:
            Ninv, flags, nt = _time_noise_model(b["Ninv"], flags, ntimes, nfreqs)
        if nt is None:
            nd, nD, nH = _noise_model(Ninv, flags, nfreqs, need_sqrt=(rng == "numpy" and not map_estimate))
        else:
            nd, nD, nH = None, None, None
        prep.append(dict(vis=vis * flags, flags=flags, F=F, nd=nd, nD=nD, nH=nH, nt=nt,
                         prior=_check_prior(b.get("ps_prior"), nfreqs)))
    # one batched device eigendecomposition for all baselines with a non-delay-diagonal S_initial
    covs = [np.eye(nfreqs) if b.get("S_initial") is None else b["S_initial"] for b in baselines]
    for pr_, (basis0, lam0sq) in zip(prep, _analyse_signal_covs(covs, device=device)):
        pr_["basis0"], pr_["lam0sq"] = basis0, lam0sq
    general = any(p["basis0"] is not None for p in prep)
    dense = any(p["nD"] is not None for p in prep)
    time_noise = any(p["nt"] is not None for p in prep)   # per-time noise: those baselines have (Ntimes, Nfreqs) flags
    per_time = any(p["flags"].ndim == 2 for p in prep)
    if per_time:
        if solver_default and rng == "numpy":
            solver = "exact"
        _check_per_time_supported(solver, True if general else None, True if dense else None)
        for p in prep:  # a batch is per-time as a whole
            if p["flags"].ndim == 1:
                p["flags"] = np.broadcast_to(p["flags"], (ntimes, nfreqs)).copy()
    ids = np.arange(nb, dtype=np.int32) if chain_ids is None else np.ascontiguousarray(chain_ids, dtype=np.int32)
    assert ids.shape == (nb,)
    keep = tuple(keep)
    if rng == "numpy":
        oma, omb = (None, None) if map_estimate else _reference_gcr_draws(ntimes, nfreqs)
        if map_estimate:
            u = np.array([np.random.uniform() for _ in range(nfreqs)])[None, :]
        else:
            u = np.random.RandomState(seed).uniform(size=(Niter, nfreqs))

    # ---- where the samples go.  In host RAM when they fit (HP_HOST_BUDGET_GB, default: half of the available memory);
    # otherwise every baseline must have an out_dir and its big arrays are written through np.memmap'ed .npy files
    # (the reference's file names), chunk by chunk -- neither host nor device memory grows with Niter x Nbaselines.
    per_iter = _big_bytes_per_iter(nb, ntimes, nfreqs, nmodes, keep)
    budget = os.environ.get("HP_HOST_BUDGET_GB")
    if budget is not None:
        budget = float(budget) * 2 ** 30
    else:
        try:
            import psutil
            budget = 0.5 * psutil.virtual_memory().available
        except Exception:  # noqa: BLE001
            budget = 64 * 2 ** 30
    in_ram = per_iter * Niter <= budget
    if not in_ram and any(b.get("out_dir") is None for b in baselines) and any(k in keep for k in ("cr", "fg", "chisq")):
        raise MemoryError(f"the sample arrays of this batch need {per_iter * Niter / 2 ** 30:.1f} GiB of host memory: pass an "
                          "out_dir per baseline (they are then written through memory-mapped .npy files), or keep=()")
    shapes = dict(signal_cr=((Niter, ntimes, nfreqs), np.complex128, "cr", "gcr-eor.npy"),
                  fg_amps=((Niter, ntimes, nmodes), np.complex128, "fg", "fg-amps.npy"),
                  chisq=((Niter, ntimes, nfreqs), np.float64, "chisq", "chisq.npy"))
    results = [dict(signal_ps=np.empty((Niter, nfreqs)), ln_post=np.empty(Niter)) for _ in range(nb)]
    for c, b in enumerate(baselines):
        for k, (shape, dt, kk, fname) in shapes.items():
            if kk not in keep:
                results[c][k] = None
            elif in_ram:
                results[c][k] = np.empty(shape, dtype=dt)
            else:
                results[c][k] = np.lib.format.open_memmap(os.path.join(str(b["out_dir"]), fname), mode="w+", dtype=dt, shape=shape)

    # ---- how many chains share an engine: all of them unless the device arena would not fit (then groups run one after
    # the other; the Philox chain ids keep the samples independent of the grouping)
    per_chain = _device_bytes_per_chain(ntimes, nfreqs, nmodes, Niter, rng, per_iter // nb, general, dense, per_time,
                                        summary is not None, batch=summary is not None and summary.get("batch", 0) > 0,
                                        time_noise=time_noise)
    dev_budget = float(os.environ.get("HP_DEVICE_BUDGET_GB", "150")) * 2 ** 30
    group = max(1, min(nb, int(dev_budget // per_chain)))
    write_times = [0.0] * nb
    signal_S = [None] * nb
    moments = [None] * nb
    any_out = any(b.get("out_dir") is not None for b in baselines)

    for g0 in range(0, nb, group):
        cs = list(range(g0, min(nb, g0 + group)))
        eng = GibbsEngine(len(cs), ntimes, nfreqs, nmodes, Niter, rng=rng, cg_compat=(solver == "reference-cg"),
                          refresh_omega=(rng == "philox"), keep=keep, general_basis0=general,
                          seed=0 if seed is None else seed, device=device,
                          force_dense_transforms=_FORCE_DENSE_TRANSFORMS and not per_time, dense_noise=dense,
                          time_flags=per_time, substreams=substreams, ring_iters=_RING_ITERS)
        try:
            eng.set_chain_ids(ids[cs])
            for lc, c in enumerate(cs):
                p = prep[c]
                b0, nD, nH = p["basis0"], p["nD"], p["nH"]
                if general and b0 is None:
                    b0 = np.ascontiguousarray(_unitary_dft(nfreqs).conj().T)
                if dense and nD is None:
                    nD = np.diag(p["nd"]).astype(np.complex128)
                    if rng == "numpy" and not map_estimate:
                        nH = np.diag(np.sqrt(p["nd"] * p["flags"].astype(float))).astype(np.complex128)
                eng.load_chain(lc, p["vis"], p["flags"], p["F"], p["nd"], p["lam0sq"], ps_prior=p["prior"], basis0=b0,
                               ninv_dense=nD, nih_dense=nH, ninv_t=p["nt"])
                if rng == "numpy":
                    eng.set_draws(lc, oma, omb, _s_draws_from_uniforms(u, p["prior"], ntimes))
            if summary is not None:
                eng.set_summary(("cr", "fg"), **summary)

            class _Dest:
                """[chain][iteration] view over the per-baseline destination arrays of this group."""
                def __init__(self, key):
                    self.key = key

                    self.shape = (len(cs),)      # chains of this group (what _scatter_chunk splits over its threads)

                def __setitem__(self, idx, val):
                    chs, its = idx               # (slice of the group's chains, slice of iterations)
                    for j, lc in enumerate(range(*chs.indices(len(cs)))):
                        results[cs[lc]][self.key][its] = val[j]

            dest = {k: (_Dest(k) if (k in ("signal_ps", "ln_post") or results[cs[0]][k] is not None) else None)
                    for k in ("signal_ps", "ln_post", "signal_cr", "fg_amps", "chisq")}

            def write(done):
                for lc, c in enumerate(cs):
                    b = baselines[c]
                    if b.get("out_dir") is None:
                        continue
                    t0 = time.perf_counter()
                    r = results[c]
                    if summary is not None:
                        # the sample files of the kept arrays only, and the moments
                        for k, (_, _, _, fname) in shapes.items():
                            if r[k] is not None:
                                if in_ram:
                                    np.save(os.path.join(str(b["out_dir"]), fname), r[k][:done])
                                else:
                                    r[k].flush()
                        np.save(os.path.join(str(b["out_dir"]), "cov-eor.npy"), eng.signal_S(lc))
                        np.save(os.path.join(str(b["out_dir"]), "dps-eor.npy"), r["signal_ps"][:done])
                        np.save(os.path.join(str(b["out_dir"]), "ln-post.npy"), r["ln_post"][:done])
                        utils.write_summary_files(b["out_dir"], eng.summary(lc), **summary)
                    elif in_ram:
                        z = lambda k: r[k][:done] if r[k] is not None else np.zeros(0)  # noqa: E731
                        utils.write_numpy_files(b["out_dir"], z("signal_cr"), eng.signal_S(lc), r["signal_ps"][:done],
                                                z("fg_amps"), z("chisq"), r["ln_post"][:done])
                    else:
                        for k in ("signal_cr", "fg_amps", "chisq"):
                            if r[k] is not None:
                                r[k].flush()
                        np.save(os.path.join(str(b["out_dir"]), "cov-eor.npy"), eng.signal_S(lc))
                        np.save(os.path.join(str(b["out_dir"]), "dps-eor.npy"), r["signal_ps"][:done])
                        np.save(os.path.join(str(b["out_dir"]), "ln-post.npy"), r["ln_post"][:done])
                    write_times[c] += time.perf_counter() - t0

            _staged_run(eng, Niter, dest, write_Niter=write_Niter if any_out else None, after_chunk=write if any_out else None)
            bad = eng.info()
            if np.any(bad != 0):
                lc = int(np.flatnonzero(bad)[0])
                raise np.linalg.LinAlgError(f"GCR system of baseline {cs[lc]} of the batch is not positive definite "
                                            f"(Cholesky failed in block column {int(bad[lc]) - 1})")
            for lc, c in enumerate(cs):
                signal_S[c] = eng.signal_S(lc)
                if summary is not None:
                    moments[c] = eng.summary(lc)
        finally:
            eng.close()
    out = [(results[c]["signal_cr"], signal_S[c], results[c]["signal_ps"], results[c]["fg_amps"], results[c]["chisq"],
            results[c]["ln_post"], write_times[c]) + ((moments[c],) if summary is not None else ()) for c in range(nb)]
    if verbose:
        for c in range(nb):
            print(f"baseline {c}: ln_post[-1] = {out[c][5][-1]:.1f}")
    return out
