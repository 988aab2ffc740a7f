"""ctypes binding of libhydra_pspec_b200.so (C ABI: include/hydra_pspec_b200.h)."""
import ctypes as C
import os
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("HP_LIB_PATH", _HERE / "csrc" / "libhydra_pspec_b200.so"))   # (HP_LIB_PATH: experiments)

HP_RNG_INJECTED, HP_RNG_PHILOX = 0, 1
HP_KEEP_CR, HP_KEEP_FG, HP_KEEP_CHISQ = 1, 2, 4
(HP_BUF_PS, HP_BUF_LNPOST, HP_BUF_CR, HP_BUF_FG, HP_BUF_CHISQ, HP_BUF_LAST_CR, HP_BUF_LAST_FG,
 HP_BUF_PS_CUR) = range(8)
HP_NUM_KERNEL_CLASSES = 6
HP_SUMMARY_CR, HP_SUMMARY_FG = 1, 2


class HPConfig(C.Structure):
    _fields_ = [
        ("device", C.c_int), ("nchains", C.c_int), ("ntimes", C.c_int), ("nfreqs", C.c_int),
        ("nmodes", C.c_int), ("rng_mode", C.c_int), ("cg_compat", C.c_int), ("refresh_omega", C.c_int),
        ("keep", C.c_int), ("max_iters", C.c_int), ("general_basis0", C.c_int), ("profile", C.c_int), ("substreams", C.c_int), ("dense_noise", C.c_int),
        ("force_dense_transforms", C.c_int), ("force_dense_solve", C.c_int), ("time_flags", C.c_int),
        ("ring_iters", C.c_int), ("seed", C.c_uint64), ("stream", C.c_void_p),
    ]


class HPHostSink(C.Structure):
    _fields_ = [("signal_ps", C.c_void_p), ("ln_post", C.c_void_p), ("signal_cr", C.c_void_p),
                ("fg_amps", C.c_void_p), ("chisq", C.c_void_p), ("iters", C.c_int), ("first_iter", C.c_int),
                ("iter_major", C.c_int), ("read_ahead", C.c_int)]


class HydraLibError(RuntimeError):
    pass


_lib = None

_dp = C.POINTER(C.c_double)
_SIGNATURES = {
    "hp_engine_create": (C.c_int, [C.POINTER(HPConfig), C.POINTER(C.c_void_p)]),
    "hp_engine_destroy": (C.c_int, [C.c_void_p]),
    "hp_engine_load_chain": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "hp_engine_load_chain_dense": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 9),
    "hp_engine_set_draws": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "hp_engine_run": (C.c_int, [C.c_void_p, C.c_int]),
    "hp_engine_run_to_host": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(HPHostSink)]),
    "hp_engine_gcr": (C.c_int, [C.c_void_p]),
    "hp_engine_sync": (C.c_int, [C.c_void_p]),
    "hp_engine_iterations_done": (C.c_int, [C.c_void_p]),
    "hp_engine_rewind": (C.c_int, [C.c_void_p]),
    "hp_engine_read": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "hp_engine_read_signal_S": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "hp_engine_info": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hp_engine_kernel_ms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "hp_engine_set_substreams": (C.c_int, [C.c_void_p, C.c_int]),
    "hp_engine_set_chain_ids": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hp_engine_set_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "hp_engine_launch_count": (C.c_longlong, [C.c_void_p]),
    "hp_engine_set_summary": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "hp_engine_read_summary": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                         C.POINTER(C.c_int)]),
    "hp_engine_set_summary_batched": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "hp_engine_read_summary_mcse": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                              C.POINTER(C.c_int)]),
    "hp_engine_pt_form": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "hp_kernel_class_name": (C.c_char_p, [C.c_int]),
    "hp_sample_S": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hp_fourier_operator": (C.c_int, [C.c_int, C.c_int, C.c_void_p]),
    "hp_eigh_batch": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hp_test_zgemm": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                C.c_int, C.c_void_p, C.c_void_p]),
    "hp_test_chol_solve": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hp_test_solve3": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "hp_test_solve3_schedule": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "hp_fp64_peak_tflops": (C.c_double, [C.c_int, C.c_double]),
    "hp_release_cached_memory": (None, []),
    "hp_pinned_alloc": (C.c_void_p, [C.c_size_t]),
    "hp_pinned_free": (None, [C.c_void_p]),
    "hp_last_error": (C.c_char_p, []),
    "hp_version": (C.c_char_p, []),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib():
    """The loaded library.  Fails loudly when it has not been built (no CPU fallback)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise HydraLibError(
                f"{LIB_PATH} not found: build it with hydra_pspec_b200/csrc/build.sh "
                "(hydra_pspec_b200 has no CPU fallback)")
        L = C.CDLL(os.fspath(LIB_PATH))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise HydraLibError(f"hydra_pspec_b200 error {rc}: {lib().hp_last_error().decode()}")


def ptr(a):
    """Host pointer of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def c128(a):
    return np.ascontiguousarray(a, dtype=np.complex128)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def pinned_empty(shape, dtype):
    """numpy array over page-locked host memory (freed when the array is garbage collected)."""
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    p = lib().hp_pinned_alloc(max(nbytes, 1))
    if not p:
        raise HydraLibError("cudaHostAlloc failed")
    buf = (C.c_char * max(nbytes, 1)).from_address(p)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    import weakref
    weakref.finalize(buf, lib().hp_pinned_free, p)
    return arr


def bind_to_device_numa(device, verbose=False):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, so that page-locked staging
    buffers (first touch / cudaHostAlloc) land in that node's memory and device-to-host copies do not
    cross the socket interconnect.  With one process per GPU on a dual-socket box this is what keeps the
    end-to-end (PCIe-bound) rate from collapsing when all GPUs stream at once.  Best effort: returns the
    node, or None when the topology cannot be read or the node's CPUs are not available to the process.
    Disabled by HP_NO_NUMA_BIND=1."""
    import os
    import subprocess
    if os.environ.get("HP_NO_NUMA_BIND") == "1":
        return None
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(int(device))],
                             capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0].strip().lower()
        dom, rest = out.split(":", 1)
        bus = f"{dom[-4:]}:{rest}"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if verbose:
            import sys
            print(f"[numa] device {device} bus {bus} node {node}: {len(use)} of {len(allowed)} allowed CPUs on that node",
                  file=sys.stderr)
        if not use:
            return None
        os.sched_setaffinity(0, use)
        return node
    except Exception:  # noqa: BLE001 - topology files missing, nvidia-smi absent, ...
        return None
