"""CPU oracle of the Gibbs step with a per-time inverse noise covariance ``Ninv`` of shape ``(Ntimes, Nfreqs, Nfreqs)``.

TEST INFRASTRUCTURE ONLY (checker of tests/test_time_noise_cpu.py and tests/test_gpu_time_noise.py).  The reference's
build_matrices takes one ``Ninv`` (pspec.py:361); this extends ``oracle/hydra_oracle.py`` the way its 2-D flags do, with
the same building blocks:

- time ``t`` uses ``build_matrices(flags_t, S, Ninv[t], ...)``, ``flags_t`` being the 1-D flags or ``flags[t]``;
- ``chisq[t] = |resid_t|^2 * real(diag(Ninv[t]))``;
- the ln-posterior term of time ``t`` uses ``Ninv[t][f][:, f]``.

A 2-D ``Ninv`` goes to ``hydra_oracle`` unchanged.
"""
import numpy as np

from oracle import hydra_oracle as ho


def gibbs_step_fgmodes(vis, flags, signal_S, fgmodes, Ninv, ps_prior, oma, omb, u, map_estimate=False, solver="direct"):
    """One Gibbs iteration (``vis`` already multiplied by the flags).  Returns signal_cr, S_sample, ps_sample, fg_amps,
    chisq, ln_post as ``hydra_oracle.gibbs_step_fgmodes``."""
    Ninv = np.asarray(Ninv)
    if Ninv.ndim == 2:
        return ho.gibbs_step_fgmodes(vis, flags, signal_S, fgmodes, Ninv, ps_prior, oma, omb, u,
                                     map_estimate=map_estimate, solver=solver)
    ntimes, nfreqs = vis.shape
    flags = np.asarray(flags, dtype=bool)
    fl = [flags[t] if flags.ndim == 2 else flags for t in range(ntimes)]
    need_pinv = solver == "cg"
    cache, mats = {}, []
    for t in range(ntimes):
        key = (fl[t].tobytes(), Ninv[t].tobytes())
        if key not in cache:
            cache[key] = ho.build_matrices(fl[t], signal_S, Ninv[t], fgmodes, need_pinv)
        mats.append(cache[key])
    cr = ho.gcr_fgmodes(vis, fl, mats, fgmodes, oma, omb, map_estimate=map_estimate, solver=solver)
    signal_cr = cr[:, :nfreqs]
    fg_amps = cr[:, nfreqs:]
    resid = vis - (signal_cr + fg_amps @ fgmodes.T)
    chisq = np.abs(resid) ** 2 * np.real(np.diagonal(Ninv, axis1=1, axis2=2))
    ps_sample, _ = ho.sample_S(s=signal_cr, prior=ps_prior, u=u)
    S_sample = ho.covariance_from_pspec(ps_sample / nfreqs ** 2, ho.fourier_operator(nfreqs))
    Sinv = np.linalg.inv(S_sample)
    ln_post = 0.0
    for t in range(ntimes):
        f = fl[t]
        r = resid[t, f]
        s = signal_cr[t, f]
        ln_post += -(r.conj() @ Ninv[t][f][:, f] @ r) - (s.conj() @ Sinv[f][:, f] @ s)
    return signal_cr, S_sample, ps_sample, fg_amps, chisq, float(np.real(ln_post))


def gibbs_sample_with_fg(vis, flags, S_initial, fgmodes, Ninv, ps_prior, Niter=100, seed=None, map_estimate=False,
                         solver="direct", draws=None):
    """Chain for one baseline with the reference's draw sequence (or ``draws=(oma, omb, u[Niter, Nfreqs])``), as
    ``hydra_oracle.gibbs_sample_with_fg``."""
    if np.asarray(Ninv).ndim == 2:
        return ho.gibbs_sample_with_fg(vis, flags, S_initial, fgmodes, Ninv, ps_prior, Niter=Niter, seed=seed,
                                       map_estimate=map_estimate, solver=solver, draws=draws)
    if map_estimate:
        Niter = 1
    ntimes, nfreqs = vis.shape
    nmodes = fgmodes.shape[1]
    flags = np.asarray(flags, dtype=bool)
    if draws is None:
        oma, omb = ho.reference_gcr_draws(ntimes, nfreqs)
        sd = ho.ReferenceSDraws(seed)
        u_all = None
    else:
        oma, omb, u_all = draws
    signal_cr = np.zeros((Niter, ntimes, nfreqs), dtype=complex)
    signal_ps = np.zeros((Niter, nfreqs))
    fg_amps = np.zeros((Niter, ntimes, nmodes), dtype=complex)
    chisq = np.zeros((Niter, ntimes, nfreqs))
    ln_post = np.zeros(Niter)
    signal_S = np.array(S_initial, dtype=complex)
    visf = vis * flags
    for i in range(Niter):
        u = sd.next(nfreqs) if u_all is None else u_all[i]
        signal_cr[i], signal_S, signal_ps[i], fg_amps[i], chisq[i], ln_post[i] = gibbs_step_fgmodes(
            visf, flags, signal_S, fgmodes, Ninv, ps_prior, oma, omb, u, map_estimate=map_estimate, solver=solver)
    return signal_cr, signal_S, signal_ps, fg_amps, chisq, ln_post


def diag_stack(ninv_t):
    """``(Ntimes, Nfreqs, Nfreqs)`` with diagonal slices ``diag(ninv_t[t])``."""
    ninv_t = np.asarray(ninv_t, dtype=float)
    T, n = ninv_t.shape
    out = np.zeros((T, n, n))
    out[:, np.arange(n), np.arange(n)] = ninv_t
    return out
