"""The ``hydra_pspec.utils`` helpers used by the Gibbs hot path (reference: hydra_pspec/utils.py).

The uvh5 / pyuvdata helpers of the reference's utils module are outside the hot path and are
not duplicated here.
"""
from pathlib import Path

import numpy as np


def fourier_operator(n):
    """Shifted DFT matrix ``F[k, x] = exp(-2 pi i (k - n//2)(x - n//2) / n)``.

    Same operator as hydra_pspec/utils.py:14-40 (equivalent to ifftshift -> fft -> fftshift);
    computed on the device by ``hp_fourier_operator``.
    """
    from . import _lib
    out = np.empty((n, n), dtype=np.complex128)
    _lib.check(_lib.lib().hp_fourier_operator(0, int(n), _lib.ptr(out)))
    return out


def write_numpy_files(fp, signal_cr, signal_S, signal_ps, fg_amps, chisq, ln_post):
    """Write the sample arrays with the reference's file names (hydra_pspec/utils.py:269-312)."""
    fp = Path(fp)
    np.save(fp / "gcr-eor.npy", signal_cr)
    np.save(fp / "cov-eor.npy", signal_S)
    np.save(fp / "dps-eor.npy", signal_ps)
    np.save(fp / "fg-amps.npy", fg_amps)
    np.save(fp / "chisq.npy", chisq)
    np.save(fp / "ln-post.npy", ln_post)


def write_summary_files(fp, moments, burn_in, thin, batch=0):
    """Posterior moments of a chain (``GibbsEngine.summary``): ``gcr-eor-mean.npy`` / ``gcr-eor-var.npy`` (signal_cr),
    ``fg-amps-mean.npy`` / ``fg-amps-var.npy`` (fg_amps) and ``summary.json`` (count, burn_in, thin).  With ``batch > 0``
    also the batch-means standard errors and effective sample sizes, ``gcr-eor-mcse.npy`` / ``gcr-eor-ess.npy`` /
    ``fg-amps-mcse.npy`` / ``fg-amps-ess.npy``, and ``batch`` / ``nbatch`` in ``summary.json``."""
    import json
    fp = Path(fp)
    for key, stem in (("signal_cr", "gcr-eor"), ("fg_amps", "fg-amps")):
        if f"{key}_mean" in moments:
            np.save(fp / f"{stem}-mean.npy", moments[f"{key}_mean"])
            np.save(fp / f"{stem}-var.npy", moments[f"{key}_var"])
            if batch > 0:
                np.save(fp / f"{stem}-mcse.npy", moments[f"{key}_mcse"])
                np.save(fp / f"{stem}-ess.npy", moments[f"{key}_ess"])
    meta = {"count": int(moments["count"]), "burn_in": int(burn_in), "thin": int(thin)}
    if batch > 0:
        meta.update(batch=int(batch), nbatch=int(moments["nbatch"]))
    with open(fp / "summary.json", "w") as f:
        json.dump(meta, f, indent=2)


def filter_freqs(freq_str, freqs_in):
    """Subset of ``freqs_in`` (MHz) selected by ``freq_str`` (hydra_pspec/utils.py:137-196): a single
    frequency, a comma list (closest channels are kept) or ``'lo-hi'``.  Plain floats in MHz stand in
    for the reference's astropy ``Quantity`` (astropy is not a dependency here)."""
    import ast
    freqs_in = np.asarray(freqs_in, dtype=float)
    rng = f"{freqs_in.min():.2f} - {freqs_in.max():.2f} MHz"
    if "-" in freq_str:
        lo, hi = (float(ast.literal_eval(x)) for x in freq_str.split("-"))
        mask = np.logical_and(freqs_in >= lo, freqs_in <= hi)
        if mask.sum() == 0:
            print(f"Frequency range {freq_str} MHz outside of the frequencies in `freqs_in`, {rng}.")
    else:
        want = np.array([float(ast.literal_eval(f)) for f in freq_str.split(",")])
        outside = (want < freqs_in.min()) | (want > freqs_in.max())
        if outside.any():
            print(f"Frequency(ies) {want[outside]} are not within the range of frequencies in `freqs_in`, {rng}.")
        mask = np.zeros(freqs_in.size, dtype=bool)
        mask[[int(np.argmin(np.abs(freqs_in - f))) for f in want]] = True
    return freqs_in[mask]


def add_mtime_to_filepath(fp, join_char="-"):
    """Rename an existing file / directory by appending its mtime (hydra_pspec/utils.py:235-265)."""
    import os
    import shutil
    from datetime import datetime
    fp = Path(fp)
    mtime = datetime.fromtimestamp(os.path.getmtime(fp)).isoformat()
    if fp.is_file():
        fp.rename(fp.with_stem(f"{fp.stem}{join_char}{mtime}"))
    elif fp.is_dir():
        shutil.move(fp, fp.with_name(f"{fp.name}{join_char}{mtime}"))


def form_pseudo_stokes_vis(uvd, convention=1.0):
    """pI = convention * (XX + YY), stored in the XX slot (hydra_pspec/utils.py:104-135).  ``uvd`` is a
    :class:`hydra_pspec_b200.uvh5.UVH5Data` or a ``pyuvdata.UVData``."""
    if hasattr(uvd, "form_pseudo_stokes_vis"):
        uvd.form_pseudo_stokes_vis(convention)
        return uvd
    from pyuvdata import utils as uvutils  # pragma: no cover - pyuvdata is optional
    if uvutils.polstr2num("pI") not in uvd.polarization_array:
        ix = np.where(uvd.polarization_array == uvutils.polstr2num("xx"))[0]
        iy = np.where(uvd.polarization_array == uvutils.polstr2num("yy"))[0]
        uvd.data_array[..., ix] += uvd.data_array[..., iy]
        uvd.data_array *= convention
        uvd.select(polarizations=["xx"])
    return uvd
