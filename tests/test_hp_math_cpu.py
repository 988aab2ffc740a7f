"""Device math (csrc/hp_math.h) compiled for the host and checked against scipy / the reference
goldens.  CPU only: this is how the k_sample / cg_compat arithmetic is tested without a GPU."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest
import scipy.special as sc
from scipy import stats

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "hydra_pspec_b200" / "csrc"


@pytest.fixture(scope="module")
def hm():
    so = CSRC / "libhp_math_host.so"
    src = CSRC / "hp_math_host.cpp"
    if not so.exists() or so.stat().st_mtime < max(src.stat().st_mtime, (CSRC / "hp_math.h").stat().st_mtime):
        subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-o", str(so), str(src)], check=True)
    L = C.CDLL(str(so))
    L.hp_host_igamc.restype = C.c_double
    L.hp_host_igamc.argtypes = [C.c_double, C.c_double]
    L.hp_host_invsamp.restype = C.c_double
    L.hp_host_invsamp.argtypes = [C.c_double] * 5 + [C.c_int]
    L.hp_host_cg_theta.argtypes = [C.c_double, C.c_double, C.c_double, C.c_void_p]
    L.hp_host_philox.argtypes = [C.c_uint32] * 6 + [C.c_void_p]
    L.hp_host_normals.argtypes = [C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
    L.hp_host_normals_fast.argtypes = [C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
    L.hp_host_gammas.argtypes = [C.c_double, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
    L.hp_host_normal_pair.argtypes = [C.c_uint32] * 6 + [C.c_int, C.c_void_p]
    return L


def test_philox_known_answer(hm):
    # Random123 known-answer vectors for philox4x32-10
    out = (C.c_uint32 * 4)()
    hm.hp_host_philox(0, 0, 0, 0, 0, 0, out)
    assert list(out) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    hm.hp_host_philox(0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, out)
    assert list(out) == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    hm.hp_host_philox(0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, 0xA4093822, 0x299F31D0, out)
    assert list(out) == [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_normals_are_standard(hm):
    n = 400_000
    x = np.empty(n)
    hm.hp_host_normals(12345, 678, n, x.ctypes.data_as(C.c_void_p))
    assert abs(x.mean()) < 4 / np.sqrt(n)
    assert abs(x.var() - 1) < 4 * np.sqrt(2 / n)
    assert stats.kstest(x, "norm").pvalue > 1e-3
    assert abs(np.corrcoef(x[0::2], x[1::2])[0, 1]) < 4 / np.sqrt(n / 2)


def test_fast_normals_are_standard(hm):
    """Single-precision Box-Muller used for the GCR fluctuation draws (hp_math.h: normal_pair_fast)."""
    n = 2_000_000
    x = np.empty(n)
    hm.hp_host_normals_fast(4321, 99, n, x.ctypes.data_as(C.c_void_p))
    assert abs(x.mean()) < 4 / np.sqrt(n)
    assert abs(x.var() - 1) < 4 * np.sqrt(2 / n)
    assert abs(np.mean(x ** 4) - 3) < 4 * np.sqrt(96 / n)
    assert stats.kstest(x, "norm").pvalue > 1e-3
    assert abs(np.corrcoef(x[0::2], x[1::2])[0, 1]) < 4 / np.sqrt(n / 2)
    # tails are populated as expected: P(|x| > 4) = 6.33e-5
    frac = np.mean(np.abs(x) > 4)
    assert abs(frac - 6.334e-5) < 5 * np.sqrt(6.334e-5 / n)


def test_normal_pair_of_any_counter(hm):
    """hp_host_normal_pair (the draws of one general Philox counter, used by the GPU kernel tests) with counters (i, 0, 0, 0)
    is the stream of hp_host_normals / hp_host_normals_fast, and every counter word and key word changes the draw."""
    n = 2000
    out = np.empty(2)
    for fast, stream in ((0, hm.hp_host_normals), (1, hm.hp_host_normals_fast)):
        x = np.empty(n)
        stream(0xA5A5A5A5, 77, n, x.ctypes.data_as(C.c_void_p))
        got = np.empty(n)
        for i in range(n // 2):
            hm.hp_host_normal_pair(i, 0, 0, 0, 0xA5A5A5A5, 77, fast, got[2 * i:].ctypes.data_as(C.c_void_p))
        assert np.array_equal(got, x)
        hm.hp_host_normal_pair(3, 0, 0, 0, 0xA5A5A5A5, 77, fast, out.ctypes.data_as(C.c_void_p))
        base = out.copy()
        for args in ((3, 1, 0, 0, 0xA5A5A5A5, 77), (3, 0, 1, 0, 0xA5A5A5A5, 77), (3, 0, 0, 1, 0xA5A5A5A5, 77),
                     (0x80000003, 0, 0, 0, 0xA5A5A5A5, 77), (3, 0, 0, 0, 0xA5A5A5A4, 77), (3, 0, 0, 0, 0xA5A5A5A5, 76)):
            hm.hp_host_normal_pair(*args, fast, out.ctypes.data_as(C.c_void_p))
            assert not np.any(out == base), args


@pytest.mark.parametrize("alpha", [1.0, 15.0, 202.0, 1023.0])
def test_gamma_draws(hm, alpha):
    n = 100_000
    x = np.empty(n)
    hm.hp_host_gammas(alpha, 7, 9, n, x.ctypes.data_as(C.c_void_p))
    assert stats.kstest(x, "gamma", args=(alpha,)).pvalue > 1e-3


@pytest.mark.parametrize("a", [1.5, 8.0, 12.0, 24.0, 203.0, 204.0, 1024.0, 4096.0])
def test_igamc_matches_scipy(hm, a):
    xs = a * np.concatenate([np.logspace(-2, 1.5, 300), 1 + np.linspace(-0.3, 0.3, 201)])
    mine = np.array([hm.hp_host_igamc(a, x) for x in xs])
    ref = sc.gammaincc(a, xs)
    m = ref > 1e-280
    assert np.max(np.abs(mine[m] - ref[m]) / ref[m]) < 2e-11
    assert np.all(mine[~m] < 1e-270)


def test_inversion_sampler_matches_reference(hm, golden_dir):
    g = np.load(golden_dir / "functions.npz")
    for (alpha, beta, lo, hi), u, want in zip(g["invsamp_cases"], g["invsamp_u"], g["invsamp_out"]):
        got = hm.hp_host_invsamp(alpha, beta, lo, hi, u, 1000)
        assert abs(got - want) < 1e-12 * abs(want)


def test_cg_theta_matches_oracle(hm):
    from oracle import hydra_oracle as ho
    out = (C.c_double * 2)()
    rng = np.random.default_rng(0)
    for phase in [0.0, 1e-6, 3e-4, 2e-3, 0.01, 0.03, -0.0734]:
        for bnorm in [1e-7, 0.5, 8.0, 2.6e6]:
            c = (10 ** rng.uniform(-2, 6)) * np.exp(1j * phase)
            want = ho.cg_theta(c, bnorm)
            hm.hp_host_cg_theta(c.real, c.imag, bnorm, out)
            got = out[0] + 1j * out[1]
            assert abs(got - want) < 1e-12 * max(abs(want), 1e-300) or abs(want) == 0 == abs(got)
