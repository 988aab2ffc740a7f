// hp_ptlow.cu -- per-time flags as a low-rank change of one shared system (BASELINE.json configs[2]).
//
// With a separate flag vector w_t per time every time has its own GCR system (gcr_fgmodes_1d, pspec.py:151-235, called
// with that time's operators), M_t = J + D [Q|F]^H (w_t N^-1) [Q|F] D.  hp_pertime.cu factors each of them: 4 N^3 / 3
// FLOP per (baseline, time).  But the systems of one baseline differ only in the channels that are flagged at time t
// and not at all times.  With wbar = OR_t w_t, s = sqrt(wbar N^-1), A = D [Q|F]^H diag(s) (N x n):
//
//      M_0 = J + A A^H                         one factorisation per baseline and iteration, as without per-time flags
//      M_t = M_0 - A_f A_f^H                   f = f_t: the k_t channels with wbar = 1, w_t = 0 (columns of A)
//      M_t^-1 = M_0^-1 + R_f K_t^-1 R_f^H      R = M_0^-1 A,  K_t = I_k - P_ff,  P = A^H R          (Woodbury)
//
// so that  x_t = M_t^-1 b_t = x0_t + R_f K_t^-1 (R^H b_t)_f  with x0_t = M_0^-1 b_t from the shared two-pass solve.  The
// columns of A ride through k_solve3 as n more right-hand sides (rows Tp0 + x of the right-hand-side and solution
// arrays), P is one batched product, and what is left per time is a k_t x k_t Cholesky and 2 k_t N complex MACs:
// k_pt_lowrank, one warp per (baseline, time).
//
// Device draws: k_solve3 adds xi ~ CN(0, I) between its passes, i.e. x0_t carries fluctuations of covariance M_0^-1.
// The missing part M_t^-1 - M_0^-1 = R_f K_t^-1 R_f^H is added as R_f L_K^-H zeta with zeta ~ CN(0, I_k) independent of
// xi (K_t = L_K L_K^H), and the mean uses the noise-free right-hand side:
//      x_t = x0_t + R_f L_K^-H (L_K^-1 (R^H r_t)_f + zeta).
// With injected draws b_t is explicit (k_rhs_tile) and zeta is absent.
//
// K_t is positive definite exactly when M_t is; cond(K_t) <= cond(M_t), so the result is as accurate as the direct
// factorisation (tests/test_gpu_pertime.py: 1e-10 against the oracle's time-by-time solves).
#include "hp_kernels.cuh"
#include "hp_math.h"

namespace hp {
namespace {

constexpr int kPLMaxJ = 14;   // Np / 32 <= 14 (k_solve3 sizes); the kernel is instantiated for 5, 9 and 14 rows per lane

__device__ __forceinline__ double2 cmul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ double2 cmulc(double2 a, double2 b) {   // a conj(b)
    return make_double2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}
__device__ __forceinline__ int tri(int i) { return i * (i + 1) / 2; }

__global__ void __launch_bounds__(256) k_pt_arows(double* __restrict__ Rfix, const double* __restrict__ Bmat,
                                                  const double* __restrict__ ni, int n, int Np, int Tp0) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)n * Np) return;
    const int x = (int)(e / Np);
    const double s = sqrt(ni[x]);
    const double2 b = reinterpret_cast<const double2*>(Bmat)[e];
    reinterpret_cast<double2*>(Rfix)[(size_t)Tp0 * Np + e] = make_double2(s * b.x, -s * b.y);
}

// Shared memory: a CTA-wide table that maps a packed lower-triangle index e to (row, column) (the inverse of
// tri(r) + c: lets a warp spread a triangle of entries over its lanes), then per warp the packed K_t, three k-vectors
// (c / z, w, 1 / L_jj) and the channel list.
#ifndef HP_PTLOW_MINB
#define HP_PTLOW_MINB 2   // resident CTAs per SM the register budget is sized for
#endif
template <int kNJ>
__global__ void __launch_bounds__(256, HP_PTLOW_MINB) k_pt_lowrank(PtLowArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int kcap = a.kcap, ntri = tri(kcap);
    uint16_t* tab = reinterpret_cast<uint16_t*>(smem_raw);    // tab[tri(r) + c] = r << 8 | c
    const size_t tab_bytes = ((size_t)ntri * 2 + 15) & ~size_t(15);
    const size_t per_warp = ((size_t)ntri * 16 + (size_t)kcap * (16 + 16 + 8 + 4) + 15) & ~size_t(15);
    unsigned char* base = smem_raw + tab_bytes + (size_t)warp * per_warp;
    double2* Kp = reinterpret_cast<double2*>(base);           // packed lower triangle, row i at tri(i)
    double2* cv = Kp + ntri;                                  // (R^H b)_f, later z
    double2* wv = cv + kcap;                                  // forward-substitution result w = L^-1 c (+ zeta)
    double* dv = reinterpret_cast<double*>(wv + kcap);        // 1 / L_jj
    int* fl = reinterpret_cast<int*>(dv + kcap);
    for (int e = threadIdx.x; e < ntri; e += blockDim.x) {
        int r = (int)((sqrtf(8.0f * (float)e + 1.0f) - 1.0f) * 0.5f);
        while (tri(r + 1) <= e) ++r;
        while (tri(r) > e) --r;
        tab[e] = (uint16_t)((r << 8) | (e - tri(r)));
    }
    __syncthreads();
    const int Np = a.Np, N = a.N, n = a.n;
    const long long nitems = (long long)a.nsys * a.T;
    const long long gw = (long long)blockIdx.x * nwarp + warp, gstride = (long long)gridDim.x * nwarp;
    const int nj = (N + 31) >> 5;

    for (long long item = gw; item < nitems; item += gstride) {
        const int sys = (int)(item / a.T), t = (int)(item - (long long)sys * a.T);
        const int k = a.fcnt[(size_t)sys * a.T + t];
        if (k <= 0) continue;                                  // no channel beyond the all-times mask: x_t = x0_t
        __syncwarp();
        for (int e = lane; e < k; e += 32) fl[e] = a.fidx[((size_t)sys * a.T + t) * kPtLowMaxRank + e];
        const double2* Rf = reinterpret_cast<const double2*>(a.Rfix) + ((size_t)sys * a.Tp + t) * Np;
        const double2* Wa = a.wa ? reinterpret_cast<const double2*>(a.wa) + ((size_t)sys * a.Tp + t) * Np : nullptr;
        const double* lam = a.lam + (size_t)sys * Np;
        double2* Xs = reinterpret_cast<double2*>(a.X) + (size_t)sys * a.Tp * Np;
        const double2* Rr = Xs + (size_t)a.Tp0 * Np;           // row x: R[:, x]
        const double2* Pm = reinterpret_cast<const double2*>(a.Pm) + (size_t)sys * n * n;
        // right-hand side of this time, lane owns rows lane + 32 i
        double2 b[kNJ];
#pragma unroll
        for (int i = 0; i < kNJ; ++i) {
            const int j = lane + 32 * i;
            b[i] = make_double2(0.0, 0.0);
            if (i < nj && j < N) {
                const double l = lam[j];
                const double2 r = Rf[j];
                b[i] = make_double2(l * r.x, l * r.y);
                if (Wa && j < n) { const double2 w = Wa[j]; b[i].x += w.x; b[i].y += w.y; }
            }
        }
        __syncwarp();
        // K = I - P_ff (lower triangle): the k (k + 1) / 2 entries spread over the lanes, all loads independent
        const int ktri = tri(k);
        for (int e = lane; e < ktri; e += 32) {
            const int rc = tab[e], r = rc >> 8, c = rc & 255;
            const double2 p = Pm[(size_t)fl[r] * n + fl[c]];
            Kp[e] = make_double2((c == r ? 1.0 : 0.0) - p.x, c == r ? 0.0 : -p.y);
        }
        // c = (R^H b)_f, two channels at a time
        for (int r = 0; r < k; r += 2) {
            const double2* row0 = Rr + (size_t)fl[r] * Np;
            const double2* row1 = Rr + (size_t)fl[r + 1 < k ? r + 1 : r] * Np;
            double2 s0 = make_double2(0.0, 0.0), s1 = make_double2(0.0, 0.0);
#pragma unroll
            for (int i = 0; i < kNJ; ++i) {
                const int j = lane + 32 * i;
                if (i < nj && j < N) {
                    const double2 v0 = row0[j], v1 = row1[j];
                    // conj(v) b
                    s0.x += v0.x * b[i].x + v0.y * b[i].y; s0.y += v0.x * b[i].y - v0.y * b[i].x;
                    s1.x += v1.x * b[i].x + v1.y * b[i].y; s1.y += v1.x * b[i].y - v1.y * b[i].x;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s0.x += __shfl_xor_sync(0xffffffffu, s0.x, o); s0.y += __shfl_xor_sync(0xffffffffu, s0.y, o);
                s1.x += __shfl_xor_sync(0xffffffffu, s1.x, o); s1.y += __shfl_xor_sync(0xffffffffu, s1.y, o);
            }
            if (lane == 0) { cv[r] = s0; if (r + 1 < k) cv[r + 1] = s1; }
        }
        __syncwarp();
        // Cholesky K = L L^H, right-looking, with the forward substitution w = L^-1 c folded in.  Column j is kept unscaled
        // (L_ij = K_ij / sqrt(d_j), 1 / sqrt(d_j) in dv): nothing is written where the step reads, one warp barrier per column.
        bool bad = false;
        for (int j = 0; j < k; ++j) {
            const int tj = tri(j);
            const double djj = Kp[tj + j].x;
            // the diagonal of K_t lies in (0, 1]: a pivot at round-off level means M_t is singular (e.g. a fully flagged time
            // with flat-prior foreground modes), which the direct factorisation reports through an exactly zero pivot
            if (!(djj > 1.5e-14)) bad = true;
            double inv = bad ? 1.0 : rsqrt(djj);
            inv = bad ? 1.0 : inv * (1.5 - 0.5 * djj * inv * inv);        // one Newton step: full double precision
            const double rd = inv * inv;                                      // 1 / d_j
            const double2 cj = cv[j];
            const double2 wj = make_double2(cj.x * inv, cj.y * inv);         // w_j = c_j / L_jj
            if (lane == 0) { wv[j] = wj; dv[j] = inv; }
            // c_i -= L_ij w_j = K_ij w_j / sqrt(d_j)
            for (int i = j + 1 + lane; i < k; i += 32) {
                const double2 u = cmul(Kp[tri(i) + j], make_double2(wj.x * inv, wj.y * inv));
                cv[i].x -= u.x; cv[i].y -= u.y;
            }
            // trailing update K_il -= K_ij conj(K_lj) / d_j over the pairs j < l <= i < k
            const int mrem = k - j - 1, npair = tri(mrem);
            for (int e = lane; e < npair; e += 32) {
                const int rc = tab[e], i = j + 1 + (rc >> 8), l = j + 1 + (rc & 255);
                const double2 aij = Kp[tri(i) + j], alj = Kp[tri(l) + j];
                const double2 u = cmulc(aij, alj);
                double2* dst = Kp + tri(i) + l;
                dst->x -= u.x * rd; dst->y -= u.y * rd;
            }
            __syncwarp();
        }
        if (bad && lane == 0) atomicMax(a.info + sys, a.nblk + 1);
        if (a.philox) {
            const uint32_t chain = (uint32_t)a.dk.chain_ids[sys];
            for (int e = lane; e < k; e += 32) {
                u32x4 ctr; ctr.x = 0x80000000u + (uint32_t)e; ctr.y = (uint32_t)t; ctr.z = a.dk.iter; ctr.w = chain;
                double x0, x1;
                normal_pair(philox4x32_10(ctr, a.dk.key0, a.dk.key1 ^ 0xA5A5A5A5u), x0, x1);
                wv[e].x += x0 * 0.70710678118654752440; wv[e].y += x1 * 0.70710678118654752440;
            }
            __syncwarp();
        }
        // backward substitution L^H z = w:  z_j = w_j / L_jj, then w_i -= conj(L_ji) z_j for i < j (row j of K, unscaled)
        for (int j = k - 1; j >= 0; --j) {
            const double2 wj = wv[j];
            const double dj = dv[j];
            const double2 zj = make_double2(wj.x * dj, wj.y * dj);
            if (lane == 0) cv[j] = zj;
            const double2* row = Kp + tri(j);
            for (int i = lane; i < j; i += 32) {
                const double di = dv[i];
                const double2 u = cmul(make_double2(row[i].x * di, -row[i].y * di), zj);
                wv[i].x -= u.x; wv[i].y -= u.y;
            }
            __syncwarp();
        }
        // x_t += R_f z
        double2 acc[kNJ];
#pragma unroll
        for (int i = 0; i < kNJ; ++i) acc[i] = make_double2(0.0, 0.0);
        for (int r = 0; r < k; ++r) {
            const double2* row = Rr + (size_t)fl[r] * Np;
            const double2 z = cv[r];
#pragma unroll
            for (int i = 0; i < kNJ; ++i) {
                const int j = lane + 32 * i;
                if (i < nj && j < N) {
                    const double2 v = row[j];
                    acc[i].x += v.x * z.x - v.y * z.y; acc[i].y += v.x * z.y + v.y * z.x;
                }
            }
        }
        double2* xt = Xs + (size_t)t * Np;
#pragma unroll
        for (int i = 0; i < kNJ; ++i) {
            const int j = lane + 32 * i;
            if (i < nj && j < N) { double2 v = xt[j]; v.x += acc[i].x; v.y += acc[i].y; xt[j] = v; }
        }
    }
}

}  // namespace

size_t pt_lowrank_smem_bytes(int kcap, int warps) {
    const size_t ntri = (size_t)kcap * (kcap + 1) / 2;
    const size_t tab = (ntri * 2 + 15) & ~size_t(15);
    const size_t per_warp = (ntri * 16 + (size_t)kcap * (16 + 16 + 8 + 4) + 15) & ~size_t(15);
    return tab + per_warp * warps;
}

void launch_pt_lowrank(const PtLowArgs& a_in, cudaStream_t st) {
    PtLowArgs a = a_in;
    if (a.kcap < 1) return;               // no time has a channel beyond the all-times mask
    static int num_sm = 0;
    if (!num_sm) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sm, cudaDevAttrMultiProcessorCount, dev);
    }
    a.kcap = (a.kcap + 3) & ~3;
    const long long nitems = (long long)a.nsys * a.T;
    // (a 128-thread CTA per system with the rows R[:, x] parked in shared memory between the two products -- half the L2
    //  traffic -- was 2.6x slower: the kernel is bound by the per-system dependency chain, not by L2 bandwidth;
    //  profiles/r2_summary.md)
    // warps per CTA: as many as keep >= 2 CTAs (<= 100 KB each) on an SM, at most 8
    int warps = 8;
    while (warps > 1 && pt_lowrank_smem_bytes(a.kcap, warps) > 100 * 1024) warps >>= 1;
    const size_t smem = pt_lowrank_smem_bytes(a.kcap, warps);
    static size_t attr_dev[kMaxDev] = {0};
    size_t& attr_smem = attr_dev[current_device_slot()];
    if (smem > attr_smem) {
        cudaFuncSetAttribute(k_pt_lowrank<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_pt_lowrank<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_pt_lowrank<kPLMaxJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_smem = smem;
    }
    const int nj = (a.N + 31) / 32;   // rows of the system per lane
    // resident CTAs per SM for this (instantiation, CTA size, shared memory): queried once per device and configuration
    struct OccKey { size_t smem; int warps, cls, per_sm; };
    static OccKey occ_dev[kMaxDev] = {};
    OccKey& occ = occ_dev[current_device_slot()];
    const int cls = nj <= 5 ? 5 : (nj <= 9 ? 9 : kPLMaxJ);
    if (occ.per_sm < 1 || occ.smem != smem || occ.warps != warps || occ.cls != cls) {
        int per = 0;
        if (cls == 5) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_pt_lowrank<5>, 32 * warps, smem);
        else if (cls == 9) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_pt_lowrank<9>, 32 * warps, smem);
        else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_pt_lowrank<kPLMaxJ>, 32 * warps, smem);
        occ = OccKey{smem, warps, cls, per < 1 ? 1 : per};
    }
    const int per_sm = occ.per_sm;
    long long grid = (nitems + warps - 1) / warps;
    const long long cap = (long long)num_sm * per_sm;   // persistent: every resident warp strides over the systems
    if (grid > cap) grid = cap;
    if (nj <= 5) k_pt_lowrank<5><<<(int)grid, 32 * warps, smem, st>>>(a);
    else if (nj <= 9) k_pt_lowrank<9><<<(int)grid, 32 * warps, smem, st>>>(a);
    else k_pt_lowrank<kPLMaxJ><<<(int)grid, 32 * warps, smem, st>>>(a);
}

void launch_pt_arows(double* Rfix_sys, const double* Bmat_sys, const double* ni_sys, int n, int Np, int Tp0, cudaStream_t st) {
    const long long tot = (long long)n * Np;
    k_pt_arows<<<(int)((tot + 255) / 256), 256, 0, st>>>(Rfix_sys, Bmat_sys, ni_sys, n, Np, Tp0);
}

}  // namespace hp
