// hp_kernels.cu -- sm_100a kernels of the per-baseline Gibbs hot path.
//
// Reference behaviour being reproduced: hydra_pspec/pspec.py (build_matrices :325-374,
// gcr_fgmodes_1d :151-235, sample_S :67-127, gibbs_step_fgmodes :377-490).  The algebra is
// re-derived for the GPU (see DESIGN.md): the GCR system is whitened and written in the
// eigenbasis Q of the current signal covariance S = Q diag(lam^2) Q^H,
//
//      M = J + D G D,   G = [Q|F]^H N^-1 [Q|F],   D = diag(lam, 1),   J = diag(1_n, 0_m)
//
// so that one iteration needs a Hermitian positive definite factorisation M = L L^H with the explicit
// inverse W = L^-1 (k_chol_w, here) and two triangular products x = W^H (W r + xi) for all Ntimes
// right-hand sides (k_solve3, hp_solve3.cu); every O(N^3) / O(N^2 T) contraction runs on the FP64
// tensor pipe (hp_mma.cuh).  Also here: the set-up kernels k_fourier_operator and k_pack_lower, the
// residual / chi^2 / ln-posterior terms (k_post, k_colsumsq) and the power-spectrum draw (k_sample).
#include "hp_kernels.cuh"
#include "hp_math.h"
#include "hp_mma.cuh"
#include "hp_diag.cuh"

namespace hp {

// ==========================================================================================
// small helpers
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ==========================================================================================
__global__ void k_fourier_operator(double* out, int n, double scale) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)n * n) return;
    int k = (int)(e / n), x = (int)(e % n);
    long long a = (long long)(k - n / 2) * (long long)(x - n / 2);
    long long r = a % n;  // exact argument reduction: exp(-2 pi i a / n) depends on a mod n only
    if (r < 0) r += n;
    double s, c;
    sincospi(-2.0 * (double)r / (double)n, &s, &c);
    out[2 * e] = c * scale;
    out[2 * e + 1] = s * scale;
}
void launch_fourier_operator(double* out, int n, double scale, cudaStream_t st) {
    long long tot = (long long)n * n;
    k_fourier_operator<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(out, n, scale);
}

__global__ void k_pack_lower(const double* dense, long long ld, long long bs, double* packed, int N, int nblk) {
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj > bi) return;
    const double* D = dense + 2 * bs * blockIdx.z;
    double* P = packed + ((size_t)blockIdx.z * tri_blocks(nblk) + blk_index(bi, bj)) * kBlkDoubles;
    for (int e = threadIdx.x; e < 1024; e += blockDim.x) {
        int r = e >> 5, c = e & 31;
        int gi = bi * 32 + r, gj = bj * 32 + c;
        double xr = 0.0, xi = 0.0;
        if (gi < N && gj < N) { xr = D[2 * (gi * ld + gj)]; xi = D[2 * (gi * ld + gj) + 1]; }
        P[e] = xr; P[1024 + e] = xi;
    }
}
void launch_pack_lower(const double* dense, long long ld, long long bs, double* packed, int N, int nblk, int batch,
                       cudaStream_t st) {
    k_pack_lower<<<dim3(nblk, nblk, batch), 256, 0, st>>>(dense, ld, bs, packed, N, nblk);
}

// ==========================================================================================
constexpr int kCT = 512;  // threads of k_chol_w: 16 warps, one 8x8 tile of a 32x32 block each

// global L block -> shared memory, async, by all kCT threads
__device__ __forceinline__ void load_block_async_ct(double* s, const double* g) {
    for (int c = threadIdx.x; c < kLBlkDoubles / 2; c += kCT) cp_async16(s + 2 * c, g + 2 * c);
}

struct CholWSmem {
    double A[2][kLBlkDoubles];   // L_ij (double buffered); A[0] also holds the block being finished
    double B[2][kLBlkDoubles];   // L_kj (double buffered)
    double V[kLBlkDoubles];      // V_kk
};
// Fragment-major copies of W for k_solve3 (hp_solve3.cu).  One k-step (4 values of k) of one 16-row strip is 2 row groups x
// 32 lanes x [re, im] = 128 doubles: lane 4 g + q holds A[8 wi + g][4 t + q] at [wi][lane][re, im], so that each of the two
// 16-byte loads of a warp covers 512 contiguous, fully used bytes.
//   pass 1: A = W1 (rows R, k = column C);  strip R / 16 stores k-steps t < 4 (strip + 1) from offset 2 s (s + 1)
//   pass 2: A = W^H (rows = columns C of W, k = row R);  strip C / 16 stores k-steps t >= 4 strip from offset 8 nblk s - 2 s (s - 1)
__device__ __forceinline__ void store_frag1(double* Wf1, int R, int C, double re, double im) {
    const int s = R >> 4, t = C >> 2;
    double* d = Wf1 + ((size_t)(2 * s * (s + 1) + t) * 128 + 64 * ((R >> 3) & 1) + (4 * (R & 7) + (C & 3)) * 2);
    *reinterpret_cast<double2*>(d) = make_double2(re, im);
}
__device__ __forceinline__ void store_frag2(double* Wf2, int nblk, int R, int C, double re, double im) {
    const int s = C >> 4, t = R >> 2;
    double* d = Wf2 + ((size_t)(8 * nblk * s - 2 * s * (s - 1) + t - 4 * s) * 128 + 64 * ((C >> 3) & 1) + (4 * (C & 7) + (R & 3)) * 2);
    *reinterpret_cast<double2*>(d) = make_double2(re, im);
}

// ------------------------------------------------------------------------------------------
// k_chol_w: left-looking blocked Cholesky of M = J + D G D with 32x32 blocks (M is never materialised: G blocks are
// scaled by lam on the fly), with the inverse W = L^-1 built on the way, row by row:
//      W_kk = V_kk,     W_kj' = -V_kk sum_{j = j'}^{k-1} L_kj W_jj'      (j' < k)
// where V_kk = L_kk^-1 comes with the factorisation of the diagonal block (hp_diag.cuh).  Off-diagonal work is DMMA.
// One launch per block column and one CTA per block: the blocks of a column are independent, so a column's work spreads
// over (nblk - k) x nsys CTAs, where one CTA per system would leave 116 of 148 SMs idle with 32 systems resident
// (BASELINE.json configs[4]).
// Row k of W needs row k of L (finished by the panel launches of the columns < k), the rows < k of W and V_kk, i.e.
// exactly what the panel launch of column k waits for: its grid takes the nblk - k - 1 panel blocks (i, k) AND the k
// blocks (k, j') of W.  The number of CTAs per launch is nblk - 1 for every column, so the late columns, whose panels
// leave most SMs idle (one or two blocks per system), carry most of the inverse: a separate launch for W (0.65 ms at the
// headline shape) disappears into launches that were under-filled.
// The diagonal block of the NEXT column rides along as well (look-ahead): block (k + 1, k + 1) needs row k + 1 of L up to
// column k, and its last piece L_{k+1,k} is the first panel block of this launch -- the CTA that computes it goes on to
// update, factor and invert block (k + 1, k + 1) while the other CTAs of the launch work through the rest of the column.
// So the diagonal blocks need no launches of their own, which would be latency bound (128 CTAs with one 32 x 32
// factorisation each, 17 - 30 us) and sit between the panel launches.
//   first = 1: grid (nsys, 1):        block (0, 0) (for nblk = 1 the whole factorisation)
//   first = 0: grid (nsys, nblk - 1): blockIdx.y = 0: panel block (k + 1, k), then diagonal block (k + 1, k + 1);
//              0 < blockIdx.y < nblk - k - 1: panel block (k + 1 + blockIdx.y, k);  else W block (k, j')
//              (systems along x: the look-ahead CTAs of all systems start in the first wave)
__global__ void __launch_bounds__(kCT, 2) k_chol_w(CholArgs a, TrinvExtra ex, double* Wp_all, int k, int first) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CholWSmem& s = *reinterpret_cast<CholWSmem*>(smem_raw);
    const int sys = blockIdx.x;
    const int nblk = a.nblk, Np = nblk * 32;
    const int npanel = nblk - k - 1;
    const bool wrow = !first && (int)blockIdx.y >= npanel;
    const int jp = wrow ? (int)blockIdx.y - npanel : 0;    // W block column
    const double* Gp = a.Gp + (size_t)sys * tri_blocks(nblk) * kBlkDoubles;
    double* Lp = a.Lp + (size_t)sys * tri_blocks(nblk) * kLBlkDoubles;
    double* Linvp = a.Linvp + (size_t)sys * nblk * kLBlkDoubles;
    double* Wp = Wp_all + (size_t)sys * tri_blocks(nblk) * kLBlkDoubles;
    const double* lam = a.lam + (size_t)sys * Np;
    const size_t wf = (size_t)4 * nblk * (2 * nblk + 1) * 128;
    double* Wf1 = ex.Wf1 ? ex.Wf1 + (size_t)sys * wf : nullptr;
    double* Wf2 = ex.Wf2 ? ex.Wf2 + (size_t)sys * wf : nullptr;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, q = lane & 3;
    const int ti = warp >> 2, tj = warp & 3;
    double* Ar = s.A[0];
    double* Ai = s.A[0] + kLPlane;
    double* Vr = s.V;
    double* Vi = s.V + kLPlane;

    if (wrow) {
        // ---- W block (k, jp):  -V_kk sum_{j = jp}^{k-1} L_kj W_j,jp
        const double* lamj = ex.lam ? ex.lam + (size_t)sys * Np + 32 * jp : nullptr;
        double P3m[3][1][1][2], cr[1][1][2], ci[1][1][2];
        warp_zero3m<1, 1>(P3m);
        load_block_async_ct(s.V, Linvp + (size_t)k * kLBlkDoubles);
        load_block_async_ct(s.A[0], Lp + blk_index(k, jp) * kLBlkDoubles);
        load_block_async_ct(s.B[0], Wp + blk_index(jp, jp) * kLBlkDoubles);
        cp_async_commit();
        for (int j = jp; j < k; ++j) {
            // one barrier per block step: it publishes stage st AND says that every warp is done with stage st ^ 1 (read by
            // the previous step), which the loads issued right after it refill while this step multiplies
            const int st = (j - jp) & 1;
            cp_async_wait<0>();
            __syncthreads();
            if (j + 1 < k) {
                load_block_async_ct(s.A[st ^ 1], Lp + blk_index(k, j + 1) * kLBlkDoubles);
                load_block_async_ct(s.B[st ^ 1], Wp + blk_index(j + 1, jp) * kLBlkDoubles);
                cp_async_commit();
            }
            warp_zgemm3m<1, 1, false, false, false, false>(P3m, s.A[st] + 8 * ti * kLdBlk, s.A[st] + kLPlane + 8 * ti * kLdBlk, kLdBlk,
                                                           s.B[st] + 8 * tj, s.B[st] + kLPlane + 8 * tj, kLdBlk, 32);
        }
        __syncthreads();   // every warp is done with the operand stages: s.A[0] takes the accumulated sum
        warp_zgemm3m_finish<1, 1, false, false>(P3m, cr, ci);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int r = 8 * ti + g, c = 8 * tj + 2 * q + e;
            s.A[0][r * kLdBlk + c] = -cr[0][0][e];
            s.A[0][kLPlane + r * kLdBlk + c] = -ci[0][0][e];
        }
        __syncthreads();
        double dr[1][1][2], di[1][1][2], Q3m[3][1][1][2];
        warp_zero3m<1, 1>(Q3m);
        // V_kk is lower triangular: rows 8 ti.. only need k < 8 (ti + 1)
        warp_zgemm3m<1, 1, false, false, false, false>(Q3m, s.V + 8 * ti * kLdBlk, s.V + kLPlane + 8 * ti * kLdBlk, kLdBlk,
                                                       s.A[0] + 8 * tj, s.A[0] + kLPlane + 8 * tj, kLdBlk, 8 * (ti + 1));
        warp_zgemm3m_finish<1, 1, false, false>(Q3m, dr, di);
        double* Wb = Wp + blk_index(k, jp) * kLBlkDoubles;
        const int r = 8 * ti + g, c = 8 * tj + 2 * q;
        *reinterpret_cast<double2*>(Wb + r * kLdBlk + c) = make_double2(dr[0][0][0], dr[0][0][1]);
        *reinterpret_cast<double2*>(Wb + kLPlane + r * kLdBlk + c) = make_double2(di[0][0][0], di[0][0][1]);
        if (Wf1 || Wf2) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int R = 32 * k + r, C = 32 * jp + c + e;
                if (Wf1) {
                    const double l = lamj ? lamj[c + e] : 1.0;
                    store_frag1(Wf1, R, C, l * dr[0][0][e], l * di[0][0][e]);
                }
                if (Wf2) store_frag2(Wf2, nblk, R, C, dr[0][0][e], di[0][0][e]);
            }
        }
        return;
    }

    // ---- Cholesky block (i, kc): the update, then the factorisation + inverse (diag) or L_i,kc = C V_kc^H
    auto chol_block = [&](int i, int kc, bool diag) {
        double cr[1][1][2], ci[1][1][2], P3m[3][1][1][2];
        warp_zero<1, 1>(cr, ci);
        warp_zero3m<1, 1>(P3m);
        double mr_[2], mi_[2];
        {
            const double* Gb = Gp + blk_index(i, kc) * kBlkDoubles;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int r = 8 * ti + g, c = 8 * tj + 2 * q + e;
                const int gi = 32 * i + r, gj = 32 * kc + c;
                const double sc = lam[gi] * lam[gj];
                mr_[e] = sc * Gb[r * 32 + c];
                mi_[e] = sc * Gb[1024 + r * 32 + c];
                if (gi == gj && (gi < a.n || gi >= a.N)) mr_[e] += 1.0;
            }
        }
        if (!diag) load_block_async_ct(s.V, Linvp + (size_t)kc * kLBlkDoubles);
        if (kc > 0) {
            load_block_async_ct(s.A[0], Lp + blk_index(i, 0) * kLBlkDoubles);
            if (!diag) load_block_async_ct(s.B[0], Lp + blk_index(kc, 0) * kLBlkDoubles);
        }
        cp_async_commit();
        for (int j = 0; j < kc; ++j) {
            const int st = j & 1;
            cp_async_wait<0>();
            __syncthreads();   // stage st has landed; every warp is done with stage st ^ 1 (one barrier per block step)
            if (j + 1 < kc) {
                load_block_async_ct(s.A[st ^ 1], Lp + blk_index(i, j + 1) * kLBlkDoubles);
                if (!diag) load_block_async_ct(s.B[st ^ 1], Lp + blk_index(kc, j + 1) * kLBlkDoubles);
                cp_async_commit();
            }
            const double* ar = s.A[st];
            const double* br = diag ? s.A[st] : s.B[st];
            warp_zgemm3m<1, 1, false, false, true, true>(P3m, ar + 8 * ti * kLdBlk, ar + kLPlane + 8 * ti * kLdBlk, kLdBlk,
                                                         br + 8 * tj * kLdBlk, br + kLPlane + 8 * tj * kLdBlk, kLdBlk, 32);
        }
        cp_async_wait<0>();
        __syncthreads();   // V_kk landed (kc = 0: nothing else waited for it); every warp is done with the operand stages
        warp_zgemm3m_finish<1, 1, false, true>(P3m, cr, ci);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            int r = 8 * ti + g, c = 8 * tj + 2 * q + e;
            Ar[r * kLdBlk + c] = mr_[e] - cr[0][0][e];
            Ai[r * kLdBlk + c] = mi_[e] - ci[0][0][e];
        }
        __syncthreads();
        if (diag) {
            const bool bad = diag_chol_inverse_block(Ar, Ai, Vr, Vi, tid, kCT);
            __syncthreads();
            double* Lb = Lp + blk_index(kc, kc) * kLBlkDoubles;
            double* Vb = Linvp + (size_t)kc * kLBlkDoubles;
            double* Wb = Wp + blk_index(kc, kc) * kLBlkDoubles;
            const double* lamk = ex.lam ? ex.lam + (size_t)sys * Np + 32 * kc : nullptr;
            for (int e = tid; e < kLBlkDoubles; e += kCT) {
                const double v = s.V[e];
                Lb[e] = s.A[0][e];
                Vb[e] = v;
                Wb[e] = v;                                   // W_kk = V_kk
            }
            if (Wf1 || Wf2) {
                // diagonal block (lower triangular; the zeros above the diagonal are part of the 16-row strips' k range)
                for (int e = tid; e < 1024; e += kCT) {
                    const int r = e >> 5, c = e & 31;
                    const double re = Vr[r * kLdBlk + c], im = Vi[r * kLdBlk + c];
                    if (Wf1 && c < 16 * ((r >> 4) + 1)) {
                        const double l = lamk ? lamk[c] : 1.0;
                        store_frag1(Wf1, 32 * kc + r, 32 * kc + c, l * re, l * im);
                    }
                    if (Wf2 && r >= 16 * (c >> 4)) store_frag2(Wf2, nblk, 32 * kc + r, 32 * kc + c, re, im);
                }
            }
            if (bad && tid == 0 && a.info) atomicMax(a.info + sys, kc + 1);
        } else {
            double dr[1][1][2], di[1][1][2], Q3m[3][1][1][2];
            warp_zero3m<1, 1>(Q3m);
            warp_zgemm3m<1, 1, false, false, true, true>(Q3m, Ar + 8 * ti * kLdBlk, Ai + 8 * ti * kLdBlk, kLdBlk, Vr + 8 * tj * kLdBlk,
                                                         Vi + 8 * tj * kLdBlk, kLdBlk, 32);
            warp_zgemm3m_finish<1, 1, false, true>(Q3m, dr, di);
            double* Lb = Lp + blk_index(i, kc) * kLBlkDoubles;
            int r = 8 * ti + g, c = 8 * tj + 2 * q;
            *reinterpret_cast<double2*>(Lb + r * kLdBlk + c) = make_double2(dr[0][0][0], dr[0][0][1]);
            *reinterpret_cast<double2*>(Lb + kLPlane + r * kLdBlk + c) = make_double2(di[0][0][0], di[0][0][1]);
        }
    };
    if (first) { chol_block(0, 0, true); return; }
    chol_block(k + 1 + (int)blockIdx.y, k, false);
    if (blockIdx.y == 0) {
        // look-ahead: this CTA has just written L_{k+1,k}, the last block row k + 1 of L was waiting for
        __syncthreads();   // its global stores are visible to the whole CTA (the cp.async reads below are the CTA's own)
        chol_block(k + 1, k + 1, true);
    }
}

// Cholesky + explicit inverse of the factor in one sequence of block-column launches
int launch_chol_trinv(const CholArgs& a, double* Wp, const TrinvExtra& ex, cudaStream_t st) {
    static bool attr_dev[kMaxDev] = {false};
    bool& attr_set = attr_dev[current_device_slot()];
    if (!attr_set) {
        cudaFuncSetAttribute(k_chol_w, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CholWSmem));
        attr_set = true;
    }
    if (a.info) cudaMemsetAsync(a.info, 0, sizeof(int) * a.nsys, st);
    k_chol_w<<<dim3(a.nsys, 1), kCT, sizeof(CholWSmem), st>>>(a, ex, Wp, 0, 1);
    if (a.nblk == 1) return 1;   // block (0, 0) is the whole matrix; the column launches would have no CTAs
    for (int k = 0; k < a.nblk; ++k) k_chol_w<<<dim3(a.nsys, a.nblk - 1), kCT, sizeof(CholWSmem), st>>>(a, ex, Wp, k, 0);
    return a.nblk + 1;
}

// ==========================================================================================
// k_post: one CTA per (time, system): model = s + F f, residual, chi^2, flagged copies.
__global__ void __launch_bounds__(128) k_post(PostArgs a) {
    extern __shared__ double fsh[];  // f_t: 2*m doubles
    const int sys = blockIdx.y, t = blockIdx.x;
    const double* X = a.X + 2 * ((size_t)sys * a.Tp + t) * a.Np;
    for (int j = threadIdx.x; j < 2 * a.m; j += blockDim.x) fsh[j] = X[2 * a.n + j];
    __syncthreads();
    if (a.fg_out && t < a.T)
        for (int j = threadIdx.x; j < 2 * a.m; j += blockDim.x) a.fg_out[(size_t)sys * a.fg_bs + (size_t)t * 2 * a.m + j] = fsh[j];
    const double* Sf = a.Sf + 2 * ((size_t)sys * a.sf_bs + (size_t)t * a.n);
    const double* wd = a.wd + 2 * ((size_t)sys * a.Tp + t) * a.n;
    const double* Ft = a.Ft + 2 * (size_t)sys * a.m * a.n;
    const double* w = a.w + (size_t)sys * a.n;
    const double* nd = a.ninvd + (size_t)sys * a.n;
    double part = 0.0;
    for (int x = threadIdx.x; x < a.n; x += blockDim.x) {
        double sr = 0.0, si = 0.0;
        if (t < a.T) { sr = Sf[2 * x]; si = Sf[2 * x + 1]; }
        double mr = sr, mi = si;
        for (int j = 0; j < a.m; ++j) {
            double fr = Ft[2 * ((size_t)j * a.n + x)], fi = Ft[2 * ((size_t)j * a.n + x) + 1];
            double ar = fsh[2 * j], ai = fsh[2 * j + 1];
            mr += ar * fr - ai * fi;
            mi += ar * fi + ai * fr;
        }
        double rr = wd[2 * x] - mr, ri = wd[2 * x + 1] - mi;
        double r2 = rr * rr + ri * ri;
        if (t < a.T) {
            if (a.chisq_out) a.chisq_out[(size_t)sys * a.chisq_bs + (size_t)t * a.n + x] = r2 * nd[x];
            part += w[x] * nd[x] * r2;
            if (a.Rm) {
                double* p = a.Rm + 2 * (((size_t)sys * a.Tp + t) * a.n + x);
                p[0] = w[x] * rr; p[1] = w[x] * ri;
            }
        }
        if (a.Wm) {
            double* p = a.Wm + 2 * (((size_t)sys * a.Tp + t) * a.n + x);
            p[0] = w[x] * sr; p[1] = w[x] * si;
        }
    }
    // block reduce
    __shared__ double redp[4];
    for (int o = 16; o > 0; o >>= 1) part += __shfl_down_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) redp[threadIdx.x >> 5] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += redp[i];
        a.lnp1[(size_t)sys * a.Tp + t] = t < a.T ? s : 0.0;
    }
}
void launch_post(const PostArgs& a, cudaStream_t st) {
    k_post<<<dim3(a.Tp, a.nsys), 128, 2 * a.m * sizeof(double), st>>>(a);
}

// ==========================================================================================
__global__ void __launch_bounds__(256) k_colsumsq(const double* A, double* out, int T, int Tp, int n, int ld) {
    __shared__ double red[8][33];
    const int sys = blockIdx.y;
    const int k = blockIdx.x * 32 + (threadIdx.x & 31), tg = threadIdx.x >> 5;
    double acc = 0.0;
    if (k < n)
        for (int t = tg; t < T; t += 8) {
            const double* p = A + 2 * (((size_t)sys * Tp + t) * ld + k);
            acc += p[0] * p[0] + p[1] * p[1];
        }
    red[tg][threadIdx.x & 31] = acc;
    __syncthreads();
    if (tg == 0 && k < n) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += red[i][threadIdx.x & 31];
        out[(size_t)sys * n + k] = s;
    }
}
void launch_colsumsq(const double* A, double* out, int T, int Tp, int n, int nsys, cudaStream_t st, int ld) {
    k_colsumsq<<<dim3((n + 31) / 32, nsys), 256, 0, st>>>(A, out, T, Tp, n, ld > 0 ? ld : n);
}

// ==========================================================================================
// k_sample: one CTA (1024 threads) per system.  beta -> new power spectrum sample
// (pspec.py:67-127), lam for the next iteration, and ln_post (pspec.py:466-485).
__device__ __forceinline__ double block_reduce(double v, double* sh, int op) {
    // op 0 sum, 1 min, 2 max ; 1024 threads
    for (int o = 16; o > 0; o >>= 1) {
        double w = __shfl_xor_sync(0xffffffffu, v, o);
        v = op == 0 ? v + w : (op == 1 ? fmin(v, w) : fmax(v, w));
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        double x = sh[threadIdx.x];
        for (int o = 16; o > 0; o >>= 1) {
            double w = __shfl_xor_sync(0xffffffffu, x, o);
            x = op == 0 ? x + w : (op == 1 ? fmin(x, w) : fmax(x, w));
        }
        if (threadIdx.x == 0) sh[32] = x;
    }
    __syncthreads();
    return sh[32];
}

__global__ void __launch_bounds__(1024) k_sample(SampleArgs a) {
    __shared__ double sh[40];
    __shared__ double cdf[kInvGrid + 24];
    __shared__ double pmx[kInvGrid + 24];
    __shared__ double wmax[33];
    __shared__ double beta_s;
    const int sys = blockIdx.x, tid = threadIdx.x;
    const int n = a.n;
    double* ps = a.ps + (size_t)sys * n;
    double* lam = a.lam + (size_t)sys * a.Np;
    const double* prior = a.prior + (size_t)sys * 2 * n;
    const double* draws = a.draws ? a.draws + (size_t)sys * a.draws_bs : nullptr;
    const double alpha = (double)a.T - 1.0;  // pspec.py:108
    const uint32_t chain = a.philox ? (uint32_t)a.dk.chain_ids[sys] : 0u;

    double lp2 = 0.0;  // sum_k E_k / Lambda'_k
    for (int k0 = 0; k0 < n; k0 += 1024) {
        int k = k0 + tid;
        double beta = 0.0, newps = 0.0;
        bool has_prior = false;
        if (k < n) {
            if (a.beta_mode == 0) {
                double s = 0.0;
                for (int tl = 0; tl < a.ntiles; ++tl) s += a.Ppart[((size_t)sys * a.ntiles + tl) * n + k];
                beta = ps[k] * s;  // |sk|^2 = n lam^2 |ytilde|^2 = ps |ytilde|^2
            } else if (a.ntilesE > 0) {
                double s = 0.0;
                for (int tl = 0; tl < a.ntilesE; ++tl) s += a.Eu[((size_t)sys * a.ntilesE + tl) * n + k];
                beta = (double)n * s;
            } else {
                beta = (double)n * a.Eu[(size_t)sys * n + k];
            }
            has_prior = prior[k] > 0.0 || prior[n + k] > 0.0;  // pspec.py:114
            if (!has_prior) {
                if (!a.philox) newps = draws[k] * beta;  // invgamma.rvs(a=alpha) * beta, pspec.py:125
                else newps = beta / gamma_mt(alpha, (uint32_t)k, a.dk.iter, chain, a.dk.key0, a.dk.key1 ^ 0x5A5A5A5Au);
            }
        }
        // prior-bounded bins: inversion sampling, one bin at a time, grid evaluated by the CTA
        for (int kk = k0; kk < min(k0 + 1024, n); ++kk) {
            bool hp_ = prior[kk] > 0.0 || prior[n + kk] > 0.0;
            if (!hp_) continue;
            if (tid == kk - k0) beta_s = beta;
            __syncthreads();
            const double b = beta_s;
            const double l0 = log10(prior[n + kk]), l1 = log10(prior[kk]);
            double xj = 0.0, cj = 0.0;
            if (tid < kInvGrid) {
                xj = invsamp_grid_x(l0, l1, tid, kInvGrid);
                cj = igamc(alpha + 1.0, b / xj);  // invgamma.cdf(x, a=alpha+1, scale=beta), pspec.py:51,121
            }
            double mn = block_reduce(tid < kInvGrid ? cj : INFINITY, sh, 1);
            cj -= mn;
            double mx = block_reduce(tid < kInvGrid ? cj : -INFINITY, sh, 2);
            cj /= mx;
            if (tid < kInvGrid) cdf[tid] = cj;
            __syncthreads();
            // exclusive prefix max -> first occurrences of a non-decreasing sequence (np.unique)
            double run = tid < kInvGrid ? cj : -INFINITY;
            for (int o = 1; o < 32; o <<= 1) {
                double w = __shfl_up_sync(0xffffffffu, run, o);
                if ((tid & 31) >= o) run = fmax(run, w);
            }
            if ((tid & 31) == 31) wmax[tid >> 5] = run;
            __syncthreads();
            if (tid < 32) {
                double w = wmax[tid];
                for (int o = 1; o < 32; o <<= 1) {
                    double v = __shfl_up_sync(0xffffffffu, w, o);
                    if (tid >= o) w = fmax(w, v);
                }
                wmax[tid] = w;
            }
            __syncthreads();
            double incl = run;
            if ((tid >> 5) > 0) incl = fmax(incl, wmax[(tid >> 5) - 1]);
            if (tid < kInvGrid) pmx[tid] = incl;
            __syncthreads();
            bool keep = tid < kInvGrid && (tid == 0 || cj > pmx[tid - 1]);
            double u;
            if (!a.philox) u = draws[kk];
            else {
                u32x4 ctr; ctr.x = (uint32_t)kk; ctr.y = a.dk.iter; ctr.z = 0xFFFFu; ctr.w = chain;
                u32x4 r = philox4x32_10(ctr, a.dk.key0, a.dk.key1 ^ 0x5A5A5A5Au);
                u = u53(r.x, r.y);
            }
            // bracket: lo = last kept with cdf <= u ; hi = first kept with cdf > u
            double lo = block_reduce((keep && cj <= u) ? (double)tid : -1.0, sh, 2);
            double hi = block_reduce((keep && cj > u) ? (double)tid : 1e9, sh, 1);
            if (tid == kk - k0) {
                if (lo < 0.0 || hi > 1e8) newps = NAN;
                else {
                    int il = (int)lo, ih = (int)hi;
                    double xl = invsamp_grid_x(l0, l1, il, kInvGrid), xh = invsamp_grid_x(l0, l1, ih, kInvGrid);
                    double slope = (xh - xl) / (cdf[ih] - cdf[il]);
                    newps = slope * (u - cdf[il]) + xl;
                }
            }
            __syncthreads();
        }
        if (k < n) {
            ps[k] = newps;
            lam[k] = sqrt(newps / (double)n);
            a.ps_out[(size_t)sys * a.ps_bs + k] = newps;
            double E = beta / (double)n;
            if (a.Em) {
                if (a.ntilesE > 0) {
                    E = 0.0;
                    for (int tl = 0; tl < a.ntilesE; ++tl) E += a.Em[((size_t)sys * a.ntilesE + tl) * n + k];
                } else {
                    E = a.Em[(size_t)sys * n + k];
                }
            }
            lp2 += E / (newps / (double)n);
        }
    }
    double s2 = block_reduce(lp2, sh, 0);
    double l1 = 0.0;
    const double* lnp1 = a.lnp1 + (size_t)sys * a.Tp;
    for (int t = tid; t < a.T; t += 1024) l1 += lnp1[t];
    double s1 = block_reduce(l1, sh, 0);
    if (tid == 0) a.lnpost_out[(size_t)sys * a.lnpost_bs] = -s1 - s2;
}
void launch_sample(const SampleArgs& a, cudaStream_t st) { k_sample<<<a.nsys, 1024, 0, st>>>(a); }

}  // namespace hp
