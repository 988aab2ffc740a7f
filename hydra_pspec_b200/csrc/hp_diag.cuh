// hp_diag.cuh -- 32x32 complex diagonal block: Cholesky factor and its triangular inverse, blocked 8x8.
//
// The block lives in shared memory (planar re / im, row stride kLdBlk).  History: (1) all 512 threads,
// two __syncthreads per column (128 block-wide barriers per block); (2) a two-warp pipeline, one named
// barrier per column, ~20 us per block (measured by removing it: 30 % of k_pt_cholsolve, 17 % of the round-1 Cholesky kernel).
// This version is a right-looking factorisation over the 4 x 4 grid of 8x8 sub-blocks:
//
//   for kk = 0..3:  one warp factors the 8x8 diagonal sub-block in registers (lane = row, shuffles for
//                   the column broadcasts, fully unrolled) and inverts it;  barrier;
//                   panel    L[R][kk]  = A[R][kk] . inv8^H          one warp per sub-block, DMMA, K = 8
//                   trailing A[R][C]  -= L[R][kk] . L[C][kk]^H      one warp per sub-block, DMMA, K = 8
//   inverse: V[R][R] = inv8_R;  V[R][C] = -inv8_R . sum_{C <= p < R} L[R][p] V[p][C]  by distance R - C
//
// 13 block-wide barriers and ~40 DMMA k-steps instead of ~1000 dependent scalar steps.
#pragma once
#include "hp_kernels.cuh"
#include "hp_mma.cuh"

namespace hp {

// One warp.  (Ar, Ai): 8x8 Hermitian sub-block (lower part used), overwritten with its Cholesky factor (upper
// part zeroed); (Vr, Vi): receives the inverse of the factor (upper part zeroed).  Returns true on a
// non-positive pivot.  All 32 lanes must call; lanes >= 8 only take part in the shuffles.
__device__ __forceinline__ bool diag_chol_inverse8(double* Ar, double* Ai, double* Vr, double* Vi) {
    const int lane = threadIdx.x & 31;
    const int r = lane & 7;
    const bool act = lane < 8;
    bool bad = false;
    {
        // factor: lane = row, the row lives in 16 registers; 1 / L[c][c] is parked on the diagonal of V
        double ar[8], ai[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) { ar[c] = Ar[r * kLdBlk + c]; ai[c] = Ai[r * kLdBlk + c]; }
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const double piv = __shfl_sync(0xffffffffu, ar[c], c);
            if (!(piv > 0.0)) bad = true;
            const double inv = rsqrt(piv);
            double lr = ar[c] * inv, li = ai[c] * inv;
            if (r == c) { lr = piv * inv; li = 0.0; }
            if (r < c) { lr = 0.0; li = 0.0; }
            if (act) {
                Ar[r * kLdBlk + c] = lr; Ai[r * kLdBlk + c] = li;
                if (r == c) Vr[c * kLdBlk + c] = inv;
            }
#pragma unroll
            for (int c2 = c + 1; c2 < 8; ++c2) {
                const double yr = __shfl_sync(0xffffffffu, lr, c2), yi = __shfl_sync(0xffffffffu, li, c2);
                ar[c2] -= lr * yr + li * yi;     // a[r][c2] -= l[r][c] conj(l[c2][c])
                ai[c2] -= li * yr - lr * yi;
            }
        }
    }
    __syncwarp();
    {
        // inverse, lane = column c:  V[q][c] = (delta_qc - sum_{p<q} L[q][p] V[p][c]) / L[q][q]   (L, 1/L[q][q]: broadcast reads)
        double vr[8], vi[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            double sr = 0.0, si = 0.0;
#pragma unroll
            for (int p = 0; p < q; ++p) {
                const double lr = Ar[q * kLdBlk + p], li = Ai[q * kLdBlk + p];
                sr += lr * vr[p] - li * vi[p];
                si += lr * vi[p] + li * vr[p];
            }
            const double dinv = Vr[q * kLdBlk + q];
            vr[q] = r < q ? -sr * dinv : (r == q ? dinv : 0.0);
            vi[q] = r < q ? -si * dinv : 0.0;
        }
        __syncwarp();  // every lane has read the parked reciprocals
        if (act) {
#pragma unroll
            for (int q = 0; q < 8; ++q) { Vr[q * kLdBlk + r] = vr[q]; Vi[q * kLdBlk + r] = vi[q]; }
        }
    }
    __syncwarp();
    return bad;
}

// All threads of the CTA must call (it contains __syncthreads); `tid` / `nthreads` identify the thread within the
// team of >= 6 warps that owns this block (the whole CTA, or one of the lockstep teams of k_pt_cholsolve).  In place: lower triangle of (Ar, Ai) := L
// (upper part zeroed), (Vr, Vi) := L^-1 (upper part zeroed).  Returns (on warp 0) true if a pivot was not positive.
__device__ __forceinline__ bool diag_chol_inverse_block(double* Ar, double* Ai, double* Vr, double* Vi, int tid, int nthreads) {
    const int warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, q = lane & 3;
    bool bad = false;
    auto sub = [](double* base, int R, int C) { return base + (8 * R) * kLdBlk + 8 * C; };
    // zero V and the strictly upper sub-blocks of A
    for (int e = tid; e < kLBlkDoubles; e += nthreads) Vr[e] = 0.0;   // both planes are contiguous: Vi = Vr + kLPlane
    if (warp < 6) {
        const int R = warp < 3 ? 0 : (warp < 5 ? 1 : 2), C = warp < 3 ? warp + 1 : (warp < 5 ? warp - 1 : 3);
        for (int e = lane; e < 64; e += 32) { sub(Ar, R, C)[(e >> 3) * kLdBlk + (e & 7)] = 0.0; sub(Ai, R, C)[(e >> 3) * kLdBlk + (e & 7)] = 0.0; }
    }
    __syncthreads();
    for (int kk = 0; kk < 4; ++kk) {
        if (warp == 0) bad |= diag_chol_inverse8(sub(Ar, kk, kk), sub(Ai, kk, kk), sub(Vr, kk, kk), sub(Vi, kk, kk));
        if (kk == 3) break;
        __syncthreads();
        if (warp < 3 - kk) {
            // panel: L[R][kk] = A[R][kk] . inv8^H
            const int R = kk + 1 + warp;
            double P[3][1][1][2], cr[1][1][2], ci[1][1][2];
            warp_zero3m<1, 1>(P);
            warp_zgemm3m<1, 1, false, false, true, true>(P, sub(Ar, R, kk), sub(Ai, R, kk), kLdBlk, sub(Vr, kk, kk), sub(Vi, kk, kk),
                                                         kLdBlk, 8);
            warp_zgemm3m_finish<1, 1, false, true>(P, cr, ci);
            __syncwarp();  // every lane has read its fragments of A[R][kk] before it is overwritten
            *reinterpret_cast<double2*>(sub(Ar, R, kk) + g * kLdBlk + 2 * q) = make_double2(cr[0][0][0], cr[0][0][1]);
            *reinterpret_cast<double2*>(sub(Ai, R, kk) + g * kLdBlk + 2 * q) = make_double2(ci[0][0][0], ci[0][0][1]);
        }
        __syncthreads();
        const int ntr = (3 - kk) * (4 - kk) / 2;
        if (warp < ntr) {
            // trailing update: A[R][C] -= L[R][kk] . L[C][kk]^H   for kk < C <= R <= 3
            int R = kk + 1, C = kk + 1, w = warp;
            while (w > R - (kk + 1)) { w -= R - kk; ++R; }
            C = kk + 1 + w;
            double P[3][1][1][2], cr[1][1][2], ci[1][1][2];
            warp_zero3m<1, 1>(P);
            warp_zgemm3m<1, 1, false, false, true, true>(P, sub(Ar, R, kk), sub(Ai, R, kk), kLdBlk, sub(Ar, C, kk), sub(Ai, C, kk),
                                                         kLdBlk, 8);
            warp_zgemm3m_finish<1, 1, false, true>(P, cr, ci);
            double2* dr = reinterpret_cast<double2*>(sub(Ar, R, C) + g * kLdBlk + 2 * q);
            double2* di = reinterpret_cast<double2*>(sub(Ai, R, C) + g * kLdBlk + 2 * q);
            double2 xr = *dr, xi = *di;
            xr.x -= cr[0][0][0]; xr.y -= cr[0][0][1]; xi.x -= ci[0][0][0]; xi.y -= ci[0][0][1];
            *dr = xr; *di = xi;
        }
        __syncthreads();
    }
    __syncthreads();
    // inverse: V[R][C] = -inv8_R . sum_{C <= p < R} L[R][p] V[p][C], by distance d = R - C
    for (int d = 1; d < 4; ++d) {
        if (warp < 4 - d) {
            const int C = warp, R = C + d;
            double P[3][1][1][2], cr[1][1][2], ci[1][1][2];
            warp_zero3m<1, 1>(P);
            warp_zgemm3m<1, 1, false, false, false, false>(P, sub(Ar, R, C), sub(Ai, R, C), kLdBlk, sub(Vr, C, C), sub(Vi, C, C),
                                                           kLdBlk, 8 * d);
            warp_zgemm3m_finish<1, 1, false, false>(P, cr, ci);
            // park T in V[R][C] (zero so far), then V[R][C] = -inv8_R . T
            *reinterpret_cast<double2*>(sub(Vr, R, C) + g * kLdBlk + 2 * q) = make_double2(cr[0][0][0], cr[0][0][1]);
            *reinterpret_cast<double2*>(sub(Vi, R, C) + g * kLdBlk + 2 * q) = make_double2(ci[0][0][0], ci[0][0][1]);
            __syncwarp();
            warp_zero3m<1, 1>(P);
            warp_zgemm3m<1, 1, false, false, false, false>(P, sub(Vr, R, R), sub(Vi, R, R), kLdBlk, sub(Vr, R, C), sub(Vi, R, C),
                                                           kLdBlk, 8);
            warp_zgemm3m_finish<1, 1, false, false>(P, cr, ci);
            __syncwarp();
            *reinterpret_cast<double2*>(sub(Vr, R, C) + g * kLdBlk + 2 * q) = make_double2(-cr[0][0][0], -cr[0][0][1]);
            *reinterpret_cast<double2*>(sub(Vi, R, C) + g * kLdBlk + 2 * q) = make_double2(-ci[0][0][0], -ci[0][0][1]);
        }
        __syncthreads();
    }
    return bad;
}

}  // namespace hp
