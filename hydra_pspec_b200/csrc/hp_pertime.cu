// hp_pertime.cu -- GCR step with a separate flag vector per time (BASELINE.json configs[2]).
//
// The reference collapses per-time flags to "flagged at any time" (run-hydra-pspec.py:520-526, its
// FIXME) because its gcr_fgmodes shares one set of operators between all times (pspec.py:238-310).
// With per-time flags w_t every time has its own system
//
//      M_t = J + D G_t D,      G_t = [Q|F]^H (w_t N^-1) [Q|F]
//
// so nothing is shared and each (baseline, time) pair is factored and solved on its own: one
// 512-thread CTA per pair, persistent over the pairs, two CTAs per SM so that one CTA's latency-bound
// diagonal-block factorisation runs under the other's DMMA block products.
//
// M_t is never stored.  In the delay eigenbasis Q = U^H the signal block of G_t is circulant,
// G_t[k][k'] = chat_t[(k - k') mod n] with chat_t the (shifted) DFT of w_t N^-1 / n, so a system is
// described by n + (n + m) m numbers: chat_t and the foreground columns [Q|F]^H (w_t N^-1) F
// (`H`, built once per baseline by k_zgemm2 when the chain is loaded).
//
// The factor L lives in a per-CTA global scratch slot (L2 / HBM), streamed through shared memory by
// cp.async, double buffered as in k_chol_w.  The forward substitution y = L^-1 r is folded into the
// factorisation (the blocks L_kj pass through shared memory anyway when the diagonal block k is
// updated), the Philox fluctuation xi ~ CN(0, I) is added to y, and the backward substitution
// x = L^-H (y + xi) re-reads L once from the scratch slot.
#include "hp_kernels.cuh"
#include "hp_math.h"
#include "hp_mma.cuh"
#include "hp_diag.cuh"

namespace hp {
// Phase timers of k_pt_cholsolve (build with -DHP_PT_TIMERS; profiles/scripts/pt_timers.py): clock64 deltas of thread 0
// of every CTA, accumulated per phase.
#ifdef HP_PT_TIMERS
__device__ unsigned long long g_pt_cycles[8];
#define PT_T(idx) do { if (tid == 0) { long long _n = clock64(); tacc[idx] += _n - tlast; tlast = _n; } } while (0)
#else
#define PT_T(idx) do { } while (0)
#endif
namespace {

constexpr int kPT = 512;  // 16 warps: one 8x8 tile of a 32x32 block each

__device__ __forceinline__ void pt_cp_async16(void* smem_dst, const void* gmem_src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void pt_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void pt_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void pt_load_block(double* s, const double* g) {
    for (int c = threadIdx.x; c < kLBlkDoubles / 2; c += kPT) pt_cp_async16(s + 2 * c, g + 2 * c);
}

struct PtSmem {
    double A[2][kLBlkDoubles];   // L_ij (double buffered); A[0] also holds the block being finished
    double B[2][kLBlkDoubles];   // L_kj (double buffered); B[0] doubles as reduction scratch
    double V[kLBlkDoubles];      // inverse of the current diagonal block
    double tv[64];               // 32-vector (re | im) between the two halves of a substitution step
    // followed by:  y[2 Np] (re | im planes), lam[Np], chat[2 n] (re | im planes)
};

__global__ void __launch_bounds__(kPT, 2) k_pt_cholsolve(PtArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PtSmem& s = *reinterpret_cast<PtSmem*>(smem_raw);
    const int nblk = a.nblk, Np = nblk * 32, n = a.n, N = a.N, m = a.m;
    double* yr = reinterpret_cast<double*>(smem_raw + sizeof(PtSmem));
    double* yi = yr + Np;
    double* lamS = yi + Np;
    double* chr = lamS + Np;
    double* chi = chr + n;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, q = lane & 3;
    const int ti = warp >> 2, tj = warp & 3;   // warp tile: rows 8 ti .. +8, cols 8 tj .. +8
    const int mr = tid >> 4, ms = tid & 15;    // block mat-vec mapping: row mr, columns 2 ms, 2 ms + 1
    double* Ar = s.A[0];
    double* Ai = s.A[0] + kLPlane;
    double* Vr = s.V;
    double* Vi = s.V + kLPlane;
    double* redr = s.B[0];
    double* redi = s.B[0] + 16 * 32;
    const size_t tri = tri_blocks(nblk);
    double* Lp = a.scratch + (size_t)blockIdx.x * (tri + nblk) * kLBlkDoubles;
    double* Vp = Lp + tri * kLBlkDoubles;
    const long long nitems = (long long)a.nsys * a.T;
#ifdef HP_PT_TIMERS
    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock64();
#endif

    // Every CTA walks a contiguous range of (system, time) pairs.  Consecutive times of a baseline often carry the
    // same flag vector (persistent RFI channels): `same_prev[sys][t]` marks a time whose mask equals that of t - 1,
    // and such a pair re-uses the factor that is already in the CTA's scratch slot: only the two substitutions
    // are done (the time-invariant case of the reference, one factorisation for all times, is the limit of this).
    const long long chunk = (nitems + gridDim.x - 1) / gridDim.x;
    const long long item_begin = (long long)blockIdx.x * chunk;
    const long long item_end = item_begin + chunk < nitems ? item_begin + chunk : nitems;
    for (long long item = item_begin; item < item_end; ++item) {
        const int sys = (int)(item / a.T), t = (int)(item % a.T);
        const bool reuse = item > item_begin && t > 0 && a.same_prev && a.same_prev[(size_t)sys * a.Tp + t] != 0;
        const double2* H = reinterpret_cast<const double2*>(a.H) + ((size_t)sys * a.Tp + t) * (size_t)(1 + m) * Np;
        const double* lam = a.lam + (size_t)sys * Np;
        const double2* R = reinterpret_cast<const double2*>(a.Rfix) + ((size_t)sys * a.Tp + t) * Np;
        const double2* WA = a.wa ? reinterpret_cast<const double2*>(a.wa) + ((size_t)sys * a.Tp + t) * Np : nullptr;
        __syncthreads();  // the previous item is done with shared memory
        for (int e = tid; e < Np; e += kPT) {
            const double l = lam[e];
            double2 r = R[e];
            r.x *= l; r.y *= l;
            if (WA) { double2 w = WA[e]; r.x += w.x; r.y += w.y; }
            lamS[e] = l; yr[e] = r.x; yi[e] = r.y;
        }
        for (int e = tid; e < n; e += kPT) { double2 c = H[e]; chr[e] = c.x; chi[e] = c.y; }
        __syncthreads();
        int bad = 0;
        PT_T(0);  // item prologue

        if (reuse) {
            // ---- forward substitution only, y_k = V_kk (r_k - sum_{j<k} L_kj y_j), with the factor of the previous time
            {   // start the whole factor on its way from DRAM to L2 (1 MB: 16 lines per thread)
                const char* base = reinterpret_cast<const char*>(Lp);
                const size_t bytes = (tri + nblk) * (size_t)kLBlkDoubles * 8;
                for (size_t off = (size_t)tid * 128; off < bytes; off += (size_t)kPT * 128)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
            }
            for (int k = 0; k < nblk; ++k) {
                double f0r = 0.0, f0i = 0.0, f1r = 0.0, f1i = 0.0;
                for (int j = 0; j < k; ++j) {
                    const double* Lb = Lp + blk_index(k, j) * kLBlkDoubles + mr * kLdBlk + 2 * ms;
                    const double lr0 = __ldcg(Lb), lr1 = __ldcg(Lb + 1), li0 = __ldcg(Lb + kLPlane), li1 = __ldcg(Lb + kLPlane + 1);
                    const double2 vr = *reinterpret_cast<const double2*>(yr + 32 * j + 2 * ms);
                    const double2 vi = *reinterpret_cast<const double2*>(yi + 32 * j + 2 * ms);
                    f0r += lr0 * vr.x - li0 * vi.x; f0i += lr0 * vi.x + li0 * vr.x;
                    f1r += lr1 * vr.y - li1 * vi.y; f1i += lr1 * vi.y + li1 * vr.y;
                }
                double fr = f0r + f1r, fi = f0i + f1i;
                for (int o = 8; o > 0; o >>= 1) {
                    fr += __shfl_xor_sync(0xffffffffu, fr, o);
                    fi += __shfl_xor_sync(0xffffffffu, fi, o);
                }
                if (ms == 0) { s.tv[mr] = yr[32 * k + mr] - fr; s.tv[32 + mr] = yi[32 * k + mr] - fi; }
                __syncthreads();
                {
                    const double* Vb = Vp + (size_t)k * kLBlkDoubles + mr * kLdBlk + 2 * ms;
                    const double vr0 = __ldcg(Vb), vr1 = __ldcg(Vb + 1), vi0 = __ldcg(Vb + kLPlane), vi1 = __ldcg(Vb + kLPlane + 1);
                    const double2 xr = *reinterpret_cast<const double2*>(s.tv + 2 * ms);
                    const double2 xi = *reinterpret_cast<const double2*>(s.tv + 32 + 2 * ms);
                    double pr = vr0 * xr.x - vi0 * xi.x + vr1 * xr.y - vi1 * xi.y;
                    double pi = vr0 * xi.x + vi0 * xr.x + vr1 * xi.y + vi1 * xr.y;
                    for (int o = 8; o > 0; o >>= 1) {
                        pr += __shfl_xor_sync(0xffffffffu, pr, o);
                        pi += __shfl_xor_sync(0xffffffffu, pi, o);
                    }
                    if (ms == 0) { yr[32 * k + mr] = pr; yi[32 * k + mr] = pi; }
                }
                __syncthreads();
            }
        } else
        for (int k = 0; k < nblk; ++k) {
            double fr = 0.0, fi = 0.0;  // partial of sum_{j<k} L_kj y_j for row mr (columns 2 ms, 2 ms + 1)
            for (int i = k; i < nblk; ++i) {
                double cr[1][1][2], ci[1][1][2];
                warp_zero<1, 1>(cr, ci);
                double P3m[3][1][1][2];
                warp_zero3m<1, 1>(P3m);
                __syncthreads();  // buffers free (previous block finished: its TRSM / write-out still read A[0] and V)
                if (k > 0) {
                    pt_load_block(s.A[0], Lp + blk_index(i, 0) * kLBlkDoubles);
                    if (i != k) pt_load_block(s.B[0], Lp + blk_index(k, 0) * kLBlkDoubles);
                    pt_commit();
                }
                for (int j = 0; j < k; ++j) {
                    const int st = j & 1;
                    if (j + 1 < k) {
                        pt_load_block(s.A[st ^ 1], Lp + blk_index(i, j + 1) * kLBlkDoubles);
                        if (i != k) pt_load_block(s.B[st ^ 1], Lp + blk_index(k, j + 1) * kLBlkDoubles);
                        pt_commit();
                        pt_wait<1>();
                    } else {
                        pt_wait<0>();
                    }
                    __syncthreads();
                    const double* ar = s.A[st];
                    const double* br = (i != k) ? s.B[st] : s.A[st];
                    warp_zgemm3m<1, 1, false, false, true, true>(P3m, ar + 8 * ti * kLdBlk, ar + kLPlane + 8 * ti * kLdBlk,
                                                               kLdBlk, br + 8 * tj * kLdBlk, br + kLPlane + 8 * tj * kLdBlk,
                                                               kLdBlk, 32);
                    if (i == k) {
                        // forward substitution rides along: the blocks L_kj are in shared memory right now
                        const double2 lr = *reinterpret_cast<const double2*>(ar + mr * kLdBlk + 2 * ms);
                        const double2 li = *reinterpret_cast<const double2*>(ar + kLPlane + mr * kLdBlk + 2 * ms);
                        const double2 vr = *reinterpret_cast<const double2*>(yr + 32 * j + 2 * ms);
                        const double2 vi = *reinterpret_cast<const double2*>(yi + 32 * j + 2 * ms);
                        fr += lr.x * vr.x - li.x * vi.x + lr.y * vr.y - li.y * vi.y;
                        fi += lr.x * vi.x + li.x * vr.x + lr.y * vi.y + li.y * vr.y;
                    }
                    __syncthreads();  // stage st may be overwritten by the load issued in the next iteration
                }
                PT_T(1);  // j loop
                warp_zgemm3m_finish<1, 1, false, true>(P3m, cr, ci);
                // C = M_ik - acc with M generated on the fly
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int r = 8 * ti + g, c = 8 * tj + 2 * q + e;
                    const int gi = 32 * i + r, gj = 32 * k + c;
                    double vr, vi;
                    if (gi >= N || gj >= N) {
                        vr = gi == gj ? 1.0 : 0.0; vi = 0.0;
                    } else if (gi < n && gj < n) {
                        int d = gi - gj;
                        if (d < 0) d += n;
                        const double sc = lamS[gi] * lamS[gj];
                        vr = sc * chr[d]; vi = sc * chi[d];
                        if (gi == gj) vr += 1.0;
                    } else if (gj >= n) {
                        const double2 h = H[(size_t)(1 + gj - n) * Np + gi];
                        const double sc = lamS[gi];
                        vr = sc * h.x; vi = sc * h.y;
                    } else {
                        const double2 h = H[(size_t)(1 + gi - n) * Np + gj];
                        const double sc = lamS[gj];
                        vr = sc * h.x; vi = -sc * h.y;
                    }
                    Ar[r * kLdBlk + c] = vr - cr[0][0][e];
                    Ai[r * kLdBlk + c] = vi - ci[0][0][e];
                }
                __syncthreads();
                PT_T(2);  // generation
                if (i == k) {
                    // ---- Cholesky of the 32x32 diagonal block and its inverse, blocked 8x8 (hp_diag.cuh)
                    if (diag_chol_inverse_block(Ar, Ai, Vr, Vi, tid, kPT)) bad = k + 1;
                    __syncthreads();
                    PT_T(3);  // diagonal block
                    // ---- y_k = V (r_k - sum_{j<k} L_kj y_j)
                    for (int o = 8; o > 0; o >>= 1) {
                        fr += __shfl_xor_sync(0xffffffffu, fr, o);
                        fi += __shfl_xor_sync(0xffffffffu, fi, o);
                    }
                    if (ms == 0) { s.tv[mr] = yr[32 * k + mr] - fr; s.tv[32 + mr] = yi[32 * k + mr] - fi; }
                    __syncthreads();
                    {
                        const double2 vr = *reinterpret_cast<const double2*>(Vr + mr * kLdBlk + 2 * ms);
                        const double2 vi = *reinterpret_cast<const double2*>(Vi + mr * kLdBlk + 2 * ms);
                        const double2 xr = *reinterpret_cast<const double2*>(s.tv + 2 * ms);
                        const double2 xi = *reinterpret_cast<const double2*>(s.tv + 32 + 2 * ms);
                        double pr = vr.x * xr.x - vi.x * xi.x + vr.y * xr.y - vi.y * xi.y;
                        double pi = vr.x * xi.x + vi.x * xr.x + vr.y * xi.y + vi.y * xr.y;
                        for (int o = 8; o > 0; o >>= 1) {
                            pr += __shfl_xor_sync(0xffffffffu, pr, o);
                            pi += __shfl_xor_sync(0xffffffffu, pi, o);
                        }
                        if (ms == 0) { yr[32 * k + mr] = pr; yi[32 * k + mr] = pi; }
                    }
                    // L_kk and V to the scratch slot
                    double* Lb = Lp + blk_index(k, k) * kLBlkDoubles;
                    double* Vb = Vp + (size_t)k * kLBlkDoubles;
                    for (int e = tid; e < kLBlkDoubles; e += kPT) {
                        Lb[e] = s.A[0][e];
                        Vb[e] = s.V[e];
                    }
                    PT_T(4);  // y_k + store
                } else {
                    // L_ik = C . V^H
                    double dr[1][1][2], di[1][1][2];
                    warp_zero<1, 1>(dr, di);
                    double Q3m[3][1][1][2];
                    warp_zero3m<1, 1>(Q3m);
                    warp_zgemm3m<1, 1, false, false, true, true>(Q3m, Ar + 8 * ti * kLdBlk, Ai + 8 * ti * kLdBlk, kLdBlk,
                                                               Vr + 8 * tj * kLdBlk, Vi + 8 * tj * kLdBlk, kLdBlk, 32);
                    warp_zgemm3m_finish<1, 1, false, true>(Q3m, dr, di);
                    double* Lb = Lp + blk_index(i, k) * kLBlkDoubles;
                    const int r = 8 * ti + g, c = 8 * tj + 2 * q;
                    *reinterpret_cast<double2*>(Lb + r * kLdBlk + c) = make_double2(dr[0][0][0], dr[0][0][1]);
                    *reinterpret_cast<double2*>(Lb + kLPlane + r * kLdBlk + c) = make_double2(di[0][0][0], di[0][0][1]);
                    PT_T(5);  // trsm
                }
            }
        }
        __syncthreads();  // y complete; every L block is in the scratch slot
        if (bad && tid == 0 && a.info) atomicMax(a.info + sys, bad);

        // ---- fluctuation term: y += xi, xi ~ CN(0, I)   (same counter layout as k_solve)
        if (a.philox_wa) {
            const uint32_t chain = (uint32_t)a.dk.chain_ids[sys];
            for (int row = tid; row < N; row += kPT) {
                u32x4 ctr; ctr.x = (uint32_t)row; ctr.y = (uint32_t)t; ctr.z = a.dk.iter; ctr.w = chain;
                double n0, n1;
                normal_pair_fast(philox4x32_10(ctr, a.dk.key0, a.dk.key1 ^ 0xA5A5A5A5u), n0, n1);
                yr[row] += n0 * 0.70710678118654752440;
                yi[row] += n1 * 0.70710678118654752440;
            }
        }
        __syncthreads();

        // ---- backward substitution  x_i = V_ii^H (y_i - sum_{j>i} L_ji^H x_j), in place in y
        // The scratch slots of all CTAs (245 MB at configs[2]) do not stay in L2, so the blocks of a row would be
        // fetched from DRAM by a chain of dependent loads.  Each row therefore starts by asking L2 for the blocks of
        // the NEXT row (prefetch.global.L2, one 128-byte line per thread and step): by the time they are needed the
        // loads hit L2.
        auto prefetch_row = [&](int i) {   // V_ii and L_ji, j > i
            const char* vb = reinterpret_cast<const char*>(Vp + (size_t)i * kLBlkDoubles);
            for (int off = tid * 128; off < (int)(kLBlkDoubles * 8); off += kPT * 128)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(vb + off));
            for (int j = i + 1; j < nblk; ++j) {
                const char* lb = reinterpret_cast<const char*>(Lp + blk_index(j, i) * kLBlkDoubles);
                for (int off = tid * 128; off < (int)(kLBlkDoubles * 8); off += kPT * 128)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(lb + off));
            }
        };
        prefetch_row(nblk - 1);
        for (int i = nblk - 1; i >= 0; --i) {
            if (i > 0) prefetch_row(i - 1);
            double pr = 0.0, pi = 0.0;
            for (int j = i + 1 + warp; j < nblk; j += 16) {
                const double* Lr = Lp + blk_index(j, i) * kLBlkDoubles + lane;
                const double* Li = Lr + kLPlane;
                const double* xr = yr + 32 * j;
                const double* xi = yi + 32 * j;
#pragma unroll 8
                for (int r = 0; r < 32; ++r) {
                    const double lr = __ldcg(Lr + r * kLdBlk), li = __ldcg(Li + r * kLdBlk);
                    pr += lr * xr[r] + li * xi[r];
                    pi += lr * xi[r] - li * xr[r];
                }
            }
            redr[warp * 32 + lane] = pr; redi[warp * 32 + lane] = pi;
            __syncthreads();
            if (tid < 32) {
                double tr = 0.0, tim = 0.0;
#pragma unroll
                for (int pp = 0; pp < 16; ++pp) { tr += redr[pp * 32 + lane]; tim += redi[pp * 32 + lane]; }
                s.tv[lane] = yr[32 * i + lane] - tr;
                s.tv[32 + lane] = yi[32 * i + lane] - tim;
            }
            __syncthreads();
            {
                const double* Vg = Vp + (size_t)i * kLBlkDoubles + lane;
                pr = 0.0; pi = 0.0;
#pragma unroll
                for (int rr = 0; rr < 2; ++rr) {
                    const int r = 2 * warp + rr;
                    const double vr = __ldcg(Vg + r * kLdBlk), vi = __ldcg(Vg + kLPlane + r * kLdBlk);
                    pr += vr * s.tv[r] + vi * s.tv[32 + r];
                    pi += vr * s.tv[32 + r] - vi * s.tv[r];
                }
                redr[warp * 32 + lane] = pr; redi[warp * 32 + lane] = pi;
            }
            __syncthreads();
            if (tid < 32) {
                double tr = 0.0, tim = 0.0;
#pragma unroll
                for (int pp = 0; pp < 16; ++pp) { tr += redr[pp * 32 + lane]; tim += redi[pp * 32 + lane]; }
                yr[32 * i + lane] = tr;
                yi[32 * i + lane] = tim;
            }
            __syncthreads();
        }
        PT_T(6);  // noise + backward substitution
        double2* X = reinterpret_cast<double2*>(a.X) + ((size_t)sys * a.Tp + t) * Np;
        for (int e = tid; e < Np; e += kPT) X[e] = make_double2(yr[e], yi[e]);
        PT_T(7);
    }
#ifdef HP_PT_TIMERS
    if (tid == 0) for (int i = 0; i < 8; ++i) atomicAdd(&g_pt_cycles[i], (unsigned long long)tacc[i]);
#endif
}

}  // namespace

size_t pt_smem_bytes(int nblk, int n) { return sizeof(PtSmem) + sizeof(double) * ((size_t)3 * nblk * 32 + 2 * n); }
size_t pt_scratch_doubles_per_cta(int nblk) { return (tri_blocks(nblk) + nblk) * (size_t)kLBlkDoubles; }

int pt_grid(int nsys, int T) {
    static int ctas = 0;
    if (!ctas) {
        int dev = 0, sms = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        ctas = 2 * (sms > 0 ? sms : 148);
    }
    long long items = (long long)nsys * T;
    return (int)(items < ctas ? items : ctas);
}

#ifdef HP_PT_TIMERS
extern "C" void hp_pt_timers(unsigned long long* out, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_pt_cycles, sizeof(unsigned long long) * 8);
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_pt_cycles, z, sizeof(z)); }
}
#endif
void launch_pt_cholsolve(const PtArgs& a, int grid, cudaStream_t st) {
    const size_t smem = pt_smem_bytes(a.nblk, a.n);
    static size_t attr_dev[kMaxDev] = {0};
    size_t& attr_set = attr_dev[current_device_slot()];
    if (attr_set < smem) {
        cudaFuncSetAttribute(k_pt_cholsolve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_set = smem;
    }
    k_pt_cholsolve<<<grid, kPT, smem, st>>>(a);
}

}  // namespace hp
