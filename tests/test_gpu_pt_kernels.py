"""Kernel-level tests of the two per-time solves, each against plain float64 numpy solves of every time's own system.  GPU only.

* ``k_pt_lowrank`` (csrc/hp_ptlow.cu): the Woodbury correction of one shared factorisation, x_t = x0_t + R_f K_t^-1 (R^H b_t)_f.
  The inputs are built from a random ``A`` (N x n): ``M_0 = J + A A^H``, ``R = M_0^-1 A``, ``P = A^H R``, ``x0_t = M_0^-1 b_t``;
  the expectation is ``solve(M_0 - A_f A_f^H, b_t)``, not the Woodbury algebra again.
* ``k_pt_cholsolve`` (csrc/hp_pertime.cu): one factorisation per time of ``M_t = J + D G_t D``, ``G_t = B^H diag(v_t) B``,
  ``B = [U^H | F]`` (circulant signal block); the expectation is ``solve(M_t, lam * Rfix + [wa; 0])``.

Both kernels add Philox draws whose counters are fully determined, so the tests reproduce them on the host
(``hp_host_normal_pair``) and compare draw by draw: ``zeta`` of ``k_pt_lowrank`` with ``normal_pair`` (round-off), ``xi`` of
``k_pt_cholsolve`` with ``normal_pair_fast`` (single-precision transcendentals on both sides: 1e-5).  A wrong counter is an O(1)
difference.  The hooks (csrc/hp_testhooks.cu) fill every device element the kernels must not read with NaN.
"""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest
import scipy.linalg as sla

pytestmark = pytest.mark.gpu

from hydra_pspec_b200 import _lib as L  # noqa: E402

CSRC = Path(__file__).resolve().parent.parent / "hydra_pspec_b200" / "csrc"
KEY0, KEY1, ITER = 0x1234ABCD, 0x0BADF00D, 12345
MAXRANK = 64   # kPtLowMaxRank


def crandn(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


@pytest.fixture(scope="module")
def host_math():
    so = CSRC / "libhp_math_host.so"
    if not so.exists() or so.stat().st_mtime < max((CSRC / "hp_math_host.cpp").stat().st_mtime, (CSRC / "hp_math.h").stat().st_mtime):
        subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-o", str(so), str(CSRC / "hp_math_host.cpp")], check=True)
    hm = C.CDLL(str(so))
    hm.hp_host_normal_pair.argtypes = [C.c_uint32] * 6 + [C.c_int, C.c_void_p]
    return hm


def cnormal(hm, c0, c1, c2, c3, key1, fast):
    """(n0 + i n1) / sqrt(2) of the Philox block of counter (c0, c1, c2, c3), key (KEY0, key1)."""
    out = np.empty(2)
    hm.hp_host_normal_pair(c0 & 0xFFFFFFFF, c1, c2, c3 & 0xFFFFFFFF, KEY0, key1, int(fast), out.ctypes.data_as(C.c_void_p))
    return (out[0] + 1j * out[1]) / np.sqrt(2)


def rel_err(x, ref):
    """Per-time relative error max |x - ref| / max |ref| over the last axis."""
    return np.max(np.abs(x - ref), axis=-1) / np.max(np.abs(ref), axis=-1)


def tol_for(cond):
    """1e-11 for the condition numbers of these inputs (<= 1e3), growing with it beyond."""
    return 1e-11 * np.maximum(1.0, cond / 1e3)


def hermitian_cond(M):
    ev = np.linalg.eigvalsh(M)
    return ev[..., -1] / ev[..., 0]


# ---- k_pt_lowrank -------------------------------------------------------------------------------------------------------

def channel_lists(rng, n, ranks):
    """fidx [nsys][T][64], fcnt [nsys][T] for the given ranks: unsorted channel lists; every other list of two or more
    channels starts with channel n - 1 and ends with channel 0."""
    nsys, T = ranks.shape
    fidx = np.zeros((nsys, T, MAXRANK), dtype=np.uint16)
    lists = []
    for s in range(nsys):
        row = []
        for t in range(T):
            k = int(ranks[s, t])
            if k >= 2 and (s + t) % 2 == 0:
                f = np.r_[n - 1, rng.choice(np.arange(1, n - 1), k - 2, replace=False), 0]
            else:
                f = rng.choice(n, k, replace=False)
            fidx[s, t, :k] = f
            row.append(f.astype(int))
        lists.append(row)
    return fidx, ranks.astype(np.int32), lists


def lowrank_case(rng, n, m, ranks, wa=True):
    """Inputs of k_pt_lowrank for nsys = ranks.shape[0] systems and T = ranks.shape[1] times, and for every (system, time) the
    system M_t = M_0 - A_f A_f^H and its right-hand side b_t."""
    nsys, T = ranks.shape
    N = n + m
    J = np.diag(np.r_[np.ones(n), np.zeros(m)])
    lam = np.concatenate([0.5 + 1.5 * rng.random((nsys, n)), np.ones((nsys, m))], axis=1)
    Rfix = crandn(rng, nsys, T, N)
    Wa = crandn(rng, nsys, T, n) if wa else None
    fidx, fcnt, lists = channel_lists(rng, n, ranks)
    X0 = np.empty((nsys, T, N), complex)
    X0n = np.empty((nsys, T, N), complex)
    Rcols = np.empty((nsys, n, N), complex)
    P = np.empty((nsys, n, n), complex)
    Mt = np.empty((nsys, T, N, N), complex)
    b = np.empty((nsys, T, N), complex)
    Rf = []
    for s in range(nsys):
        A = crandn(rng, N, n) * np.sqrt(2.0 / n)
        M0 = J + A @ A.conj().T
        b[s] = lam[s] * Rfix[s]
        X0n[s] = np.linalg.solve(M0, b[s].T).T
        if wa:
            b[s, :, :n] += Wa[s]
        X0[s] = np.linalg.solve(M0, b[s].T).T
        R = np.linalg.solve(M0, A)
        Rcols[s] = R.T
        P[s] = A.conj().T @ R
        Rf.append([R[:, f] for f in lists[s]])
        for t in range(T):
            f = lists[s][t]
            Mt[s, t] = M0 - A[:, f] @ A[:, f].conj().T
    Pin = P.copy()
    iu = np.triu_indices(n, 1)
    Pin[:, iu[0], iu[1]] = np.nan          # the kernel reads the lower triangle of P only
    return dict(n=n, N=N, T=T, nsys=nsys, lam=lam, Rfix=Rfix, wa=Wa, X0=X0, X0n=X0n, Rcols=Rcols, P=P, Pin=Pin, fidx=fidx,
                fcnt=fcnt, lists=lists, Mt=Mt, b=b, Rf=Rf)


def run_lowrank(c, philox=False, chain_ids=None, wa=True, P=None):
    X = np.full((c["nsys"], c["T"], c["N"]), np.nan, complex)
    info = np.full(c["nsys"], -7, np.int32)
    ch = np.ascontiguousarray(chain_ids if chain_ids is not None else np.arange(c["nsys"]), np.int32)
    wa_arr = L.c128(c["wa"]) if (wa and c["wa"] is not None) else None
    X0 = c["X0"] if wa_arr is not None else c["X0n"]     # x0_t = M_0^-1 b_t of the right-hand side the kernel is given
    L.check(L.lib().hp_test_pt_lowrank(c["n"], c["N"], c["T"], c["nsys"], L.ptr(L.f64(c["lam"])), L.ptr(L.c128(c["Rfix"])),
                                       L.ptr(wa_arr), L.ptr(L.c128(X0)), L.ptr(L.c128(c["Rcols"])),
                                       L.ptr(L.c128(c["Pin"] if P is None else P)), L.ptr(np.ascontiguousarray(c["fidx"])),
                                       L.ptr(np.ascontiguousarray(c["fcnt"])), int(philox), KEY0, KEY1, ITER, L.ptr(ch),
                                       L.ptr(X), L.ptr(info)))
    return X, info


def lowrank_expected(c, wa=True):
    b = c["b"]
    if not wa and c["wa"] is not None:
        b = b.copy()
        b[:, :, :c["n"]] -= c["wa"]
    x = np.linalg.solve(c["Mt"], b[..., None])[..., 0]
    return x, hermitian_cond(c["Mt"])


def lowrank_zeta_part(c, hm, chain_ids, keep):
    """R_f L_K^-H zeta with L_K = chol(I - P_ff) in the order of the channel list and zeta_e from counter
    (0x80000000 + e, t, iter, chain), key (key0, key1 ^ 0xA5A5A5A5), double-precision Box-Muller."""
    out = np.zeros((c["nsys"], c["T"], c["N"]), complex)
    for s in range(c["nsys"]):
        for t, f in enumerate(c["lists"][s]):
            k = len(f)
            if k == 0 or not keep[s, t]:
                continue
            LK = np.linalg.cholesky(np.eye(k) - c["P"][s][np.ix_(f, f)])
            zeta = np.array([cnormal(hm, 0x80000000 + e, t, ITER, int(chain_ids[s]), KEY1 ^ 0xA5A5A5A5, False)
                             for e in range(k)])
            out[s, t] = c["Rf"][s][t] @ sla.solve_triangular(LK.conj().T, zeta, lower=False)
    return out


def check_lowrank(c, hm, chain_ids=None, skip=()):
    """Deterministic launch (with wa) and Philox launch (without) against the direct solves; (system, time) pairs in `skip`
    are not compared."""
    ids = np.arange(c["nsys"]) if chain_ids is None else np.asarray(chain_ids)
    keep = np.ones((c["nsys"], c["T"]), bool)
    for s, t in skip:
        keep[s, t] = False
    X, info = run_lowrank(c, chain_ids=ids)
    want, cond = lowrank_expected(c)
    err = rel_err(X, want)
    tol = tol_for(cond)
    assert np.all(err[keep] < tol[keep]), (np.max(err[keep] / tol[keep]), np.argwhere((err >= tol) & keep)[:5])
    Xp, infop = run_lowrank(c, philox=True, chain_ids=ids, wa=False)
    want0, _ = lowrank_expected(c, wa=False)
    zpart = lowrank_zeta_part(c, hm, ids, keep)
    has = keep & (c["fcnt"] > 0)
    zerr = np.max(np.abs(Xp - want0 - zpart), axis=-1) / np.maximum(np.max(np.abs(zpart), axis=-1), np.max(np.abs(want0), axis=-1))
    assert np.all(zerr[has] < tol[has]), (np.max(zerr[has] / tol[has]), np.argwhere((zerr >= tol) & has)[:5])
    # a time without extra flagged channels is x0_t exactly (the kernel skips it)
    none = keep & (c["fcnt"] == 0)
    assert np.array_equal(Xp[none], c["X0n"][none]) and np.array_equal(X[none], c["X0"][none])
    return info, infop


RANKS = [0, 1, 2, 3, 31, 32, 33, 63, 64]


# every instantiation (<5>: N <= 160, <9>: N <= 288, <14>: N <= 448) and both sides of each boundary; ranks 0..64 mixed in one
# launch (kcap 64: two warps per CTA)
@pytest.mark.parametrize("n,m", [(40, 4), (144, 16), (145, 16), (256, 16), (256, 32), (257, 32), (384, 32), (416, 32)])
def test_pt_lowrank_matches_direct_solves(n, m, host_math):
    rng = np.random.default_rng(n + 1000 * m)
    ranks = [r for r in RANKS if r <= n - m - 4]
    ranks = np.stack([ranks, ranks[::-1]])
    c = lowrank_case(rng, n, m, ranks)
    info, infop = check_lowrank(c, host_math, chain_ids=[3, 0])
    assert np.all(info == 0) and np.all(infop == 0)


@pytest.mark.parametrize("kmax", [4, 36, 37, 64])
def test_pt_lowrank_warp_configurations(kmax, host_math):
    """kcap (the largest rank rounded up to a multiple of 4) 4 and 36: 8 warps per CTA (36: the largest shared-memory
    footprint that keeps 8), 37 -> 40: 4 warps, 64: 2 warps."""
    rng = np.random.default_rng(kmax)
    T = 24
    ranks = rng.integers(0, kmax + 1, size=(3, T))
    ranks[1, 5] = kmax
    ranks[2, ::7] = 1                      # odd ranks: the paired dot product re-reads the last row
    c = lowrank_case(rng, 256, 16, ranks)
    info, infop = check_lowrank(c, host_math, chain_ids=[11, 2, 9])
    assert np.all(info == 0) and np.all(infop == 0)


def test_pt_lowrank_warps_stride_over_many_items(host_math):
    """4 x 1000 (system, time) pairs at N = 44 and kcap 4: more items than the persistent grid has warps (148 SMs x 2 CTAs x 8
    warps), so every warp takes several; non-contiguous chain ids in the draws."""
    rng = np.random.default_rng(5)
    ranks = rng.integers(0, 5, size=(4, 1000))
    c = lowrank_case(rng, 40, 4, ranks)
    info, infop = check_lowrank(c, host_math, chain_ids=[7, 1000, 2, 0x7FFFFFF0])
    assert np.all(info == 0) and np.all(infop == 0)


def test_pt_lowrank_singular_time_reports_its_system_only(host_math):
    """One time of system 1 lists all n channels (n <= 64, m > 0 flat-prior modes): M_t = J is singular, info = nblk + 1 for
    that system alone, and every other (system, time) -- of system 1 too -- is still solved."""
    rng = np.random.default_rng(17)
    n, m = 40, 4
    ranks = rng.integers(0, 12, size=(3, 6))
    ranks[1, 2] = n
    c = lowrank_case(rng, n, m, ranks)
    info, infop = check_lowrank(c, host_math, chain_ids=[4, 5, 6], skip=[(1, 2)])
    nblk = (n + m + 31) // 32
    assert list(info) == [0, nblk + 1, 0] and list(infop) == [0, nblk + 1, 0]


def test_pt_lowrank_pivot_threshold():
    """K_t = I - P_ff has its diagonal in (0, 1]; a pivot at or below 1.5e-14 means a singular system.  With P diagonal the
    pivot of a one-channel list is 1 - P_jj: 1e-15 and 0 are reported, 2e-14 and 1e-3 are not."""
    rng = np.random.default_rng(3)
    n, m = 40, 4
    ranks = np.ones((4, 2), int)
    c = lowrank_case(rng, n, m, ranks)
    d = np.array([1e-15, 2e-14, 0.0, 1e-3])
    P = np.zeros((4, n, n), complex)
    for s in range(4):
        P[s] = np.diag(1.0 - np.full(n, 0.5))
        for t in range(2):
            P[s, c["lists"][s][t][0], c["lists"][s][t][0]] = 1.0 - d[s]
    _, info = run_lowrank(c, P=P)
    nblk = (n + m + 31) // 32
    assert list(info) == [nblk + 1, 0, nblk + 1, 0]


def test_pt_lowrank_refuses_sizes_it_does_not_take():
    """A rank above 64 and N > 448 (more rows per lane than k_pt_lowrank<14> holds) are refused with HP_ERR_SIZE before
    anything is launched."""
    n, T = 40, 2
    fidx = np.zeros((1, T, MAXRANK), np.uint16)
    for N, k in ((44, 65), (449, 1)):
        fcnt = np.full((1, T), k, np.int32)
        vec = np.zeros((1, T, N), complex)
        X = np.empty((1, T, N), complex)
        info = np.empty(1, np.int32)
        rc = L.lib().hp_test_pt_lowrank(n, N, T, 1, L.ptr(np.ones((1, N))), L.ptr(vec), None, L.ptr(vec),
                                        L.ptr(np.zeros((1, n, N), complex)), L.ptr(np.zeros((1, n, n), complex)), L.ptr(fidx),
                                        L.ptr(fcnt), 0, 0, 0, 0, None, L.ptr(X), L.ptr(info))
        assert rc == -3, (N, k, rc)        # HP_ERR_SIZE


# ---- k_pt_cholsolve -----------------------------------------------------------------------------------------------------

def cholsolve_case(rng, n, m, vidx, wa=True, zero=None):
    """Inputs of k_pt_cholsolve.  vidx [nsys][T]: which weight row v a time uses (equal index: equal system); zero: (s, t) whose
    weights are all zero."""
    nsys, T = vidx.shape
    N = n + m
    k = np.arange(n)
    U = np.exp(-2j * np.pi * np.outer(k, k) / n) / np.sqrt(n)
    F = np.linalg.qr(crandn(rng, n, m))[0] if m else np.zeros((n, 0), complex)
    B = np.concatenate([U.conj().T, F], axis=1)                   # n x N
    J = np.diag(np.r_[np.ones(n), np.zeros(m)])
    lam = np.concatenate([0.2 + 1.8 * rng.random((nsys, n)), np.ones((nsys, m))], axis=1)
    V = (0.5 + 2.5 * rng.random((nsys, int(vidx.max()) + 1, n))) * (rng.random((nsys, int(vidx.max()) + 1, n)) > 0.1)
    H = np.zeros((nsys, T, 1 + m, N), complex)
    Mt = np.empty((nsys, T, N, N), complex)
    for s in range(nsys):
        for t in range(T):
            v = V[s, vidx[s, t]] * (0.0 if zero == (s, t) else 1.0)
            G = B.conj().T @ (v[:, None] * B)
            chat = G[:n, 0]
            assert np.allclose(G[:n, :n], chat[(k[:, None] - k[None, :]) % n], rtol=0, atol=1e-13 * np.max(np.abs(chat)) + 1e-300)
            H[s, t, 0, :n] = chat
            H[s, t, 1:] = G[:, n:].T
            Mt[s, t] = J + lam[s][:, None] * G * lam[s][None, :]
    Rfix = crandn(rng, nsys, T, N)
    Wa = crandn(rng, nsys, T, n) if wa else None
    b = lam[:, None, :] * Rfix
    if wa:
        b[:, :, :n] += Wa
    return dict(n=n, m=m, N=N, T=T, nsys=nsys, H=H, lam=lam, Rfix=Rfix, wa=Wa, Mt=Mt, b=b)


def run_cholsolve(c, philox=False, chain_ids=None, wa=True, same_prev=None, grid=0):
    X = np.full((c["nsys"], c["T"], c["N"]), np.nan, complex)
    info = np.full(c["nsys"], -7, np.int32)
    ch = np.ascontiguousarray(chain_ids if chain_ids is not None else np.arange(c["nsys"]), np.int32)
    wa_arr = L.c128(c["wa"]) if (wa and c["wa"] is not None) else None
    sp = None if same_prev is None else np.ascontiguousarray(same_prev, np.int32)
    L.check(L.lib().hp_test_pt_cholsolve(c["n"], c["m"], c["T"], c["nsys"], L.ptr(L.c128(c["H"])), L.ptr(L.f64(c["lam"])),
                                         L.ptr(L.c128(c["Rfix"])), L.ptr(wa_arr), L.ptr(sp), int(grid), int(philox), KEY0, KEY1,
                                         ITER, L.ptr(ch), L.ptr(X), L.ptr(info)))
    return X, info


def cholsolve_xi_part(c, hm, chain_ids, keep):
    """L_t^-H xi with M_t = L_t L_t^H and xi_row from counter (row, t, iter, chain), key (key0, key1 ^ 0xA5A5A5A5),
    normal_pair_fast."""
    out = np.zeros((c["nsys"], c["T"], c["N"]), complex)
    for s in range(c["nsys"]):
        for t in range(c["T"]):
            if not keep[s, t]:
                continue
            xi = np.array([cnormal(hm, r, t, ITER, int(chain_ids[s]), KEY1 ^ 0xA5A5A5A5, True) for r in range(c["N"])])
            Lt = np.linalg.cholesky(c["Mt"][s, t])
            out[s, t] = sla.solve_triangular(Lt.conj().T, xi, lower=False)
    return out


def check_cholsolve(c, hm, chain_ids=None, same_prev=None, grid=0, skip=(), philox=True):
    ids = np.arange(c["nsys"]) if chain_ids is None else np.asarray(chain_ids)
    keep = np.ones((c["nsys"], c["T"]), bool)
    for s, t in skip:
        keep[s, t] = False
    X, info = run_cholsolve(c, chain_ids=ids, same_prev=same_prev, grid=grid)
    Mk = c["Mt"][keep]
    want = np.linalg.solve(Mk, c["b"][keep][..., None])[..., 0]
    cond = hermitian_cond(Mk)
    err = rel_err(X[keep], want)
    tol = tol_for(cond)
    assert np.all(err < tol), (np.max(err / tol), np.max(cond))
    if not philox:
        return info, None
    Xp, infop = run_cholsolve(c, philox=True, chain_ids=ids, wa=False, same_prev=same_prev, grid=grid)
    b0 = c["b"].copy()
    b0[:, :, :c["n"]] -= c["wa"]
    want0 = np.linalg.solve(Mk, b0[keep][..., None])[..., 0]
    xpart = cholsolve_xi_part(c, hm, ids, keep)[keep]
    xerr = np.max(np.abs(Xp[keep] - want0 - xpart), axis=-1) / np.max(np.abs(xpart), axis=-1)
    # device sincospif / logf against host sinf / logf: single-precision round-off of the draws; a wrong counter is O(1)
    assert np.all(xerr < 1e-5), np.max(xerr)
    return info, infop


# nblk = 1, 2, 9, 13 (the headline 384 + 32), 14, 15, 17, 18 and 34 (1024 + 64)
@pytest.mark.parametrize("n,m", [(24, 4), (48, 8), (272, 8), (384, 32), (432, 10), (448, 12), (512, 16), (544, 24), (1024, 64)])
def test_pt_cholsolve_matches_direct_solves(n, m, host_math):
    rng = np.random.default_rng(n + m)
    T = 3 if n >= 512 else 4
    vidx = np.arange(2 * T).reshape(2, T)
    c = cholsolve_case(rng, n, m, vidx)
    info, infop = check_cholsolve(c, host_math, chain_ids=[9, 4])
    assert np.all(info == 0) and np.all(infop == 0)


def test_pt_cholsolve_factor_reuse_across_cta_chunks(host_math):
    """2 systems x 7 times on 3 CTAs (chunks of 5 items start at items 0, 5, 10).  Equal weight rows in runs that cross the
    chunk boundaries re-use the factor of t - 1 within a chunk only; same_prev = 1 on t = 0 of a system and on a chunk's first
    item whose system differs from the time before must not re-use (the scratch starts as NaN)."""
    rng = np.random.default_rng(21)
    vidx = np.array([[0, 0, 1, 1, 1, 1, 2],
                     [3, 3, 4, 5, 5, 5, 5]])
    same = np.zeros_like(vidx)
    same[:, 1:] = vidx[:, 1:] == vidx[:, :-1]
    same[:, 0] = 1          # t = 0: no previous time of this system (item 7 follows system 0's last time on CTA 1)
    same[1, 3] = 1          # item 10, first of CTA 2: M_t differs from t - 1
    assert same[0, 5] == 1  # item 5, first of CTA 1: equal to t - 1, but the factor is on CTA 0
    c = cholsolve_case(rng, 64, 8, vidx)
    info, infop = check_cholsolve(c, host_math, chain_ids=[1, 0], same_prev=same, grid=3)
    assert np.all(info == 0) and np.all(infop == 0)
    # the same inputs on one CTA per item (no re-use at all) and on one CTA (re-use wherever same_prev is true at t > 0)
    same[1, 3] = 0
    for grid in (14, 1):
        check_cholsolve(c, host_math, same_prev=same, grid=grid, philox=False)


def test_pt_cholsolve_zero_weight_time_reports_its_system_only(host_math):
    """A time of system 1 with all weights zero and m > 0 flat-prior modes: M_t = J is singular (zero foreground block, block
    column 1), info = 2 for that system alone; every other (system, time) is still solved."""
    rng = np.random.default_rng(8)
    vidx = np.arange(12).reshape(3, 4)
    c = cholsolve_case(rng, 48, 8, vidx, zero=(1, 2))
    info, infop = check_cholsolve(c, host_math, chain_ids=[2, 7, 5], skip=[(1, 2)], grid=5)
    assert list(info) == [0, 2, 0] and list(infop) == [0, 2, 0]
