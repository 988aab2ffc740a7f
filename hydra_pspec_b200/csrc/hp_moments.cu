// hp_moments.cu -- k_moments / k_moments_batch: on-device posterior moments of signal_cr and fg_amps (Welford, FP64).
//
// One launch per sub-batch and accumulated iteration updates the per-chain accumulators of both arrays:
//   d = x - mean;  mean += d / k;  M2 += Re(d conj(x - mean))   (= |d|^2 (k - 1) / k)
// The update order is the iteration order, so the moments of a chain do not depend on how its iterations were split over
// calls, sub-streams or read-ahead.  Bandwidth-bound: 16 B sample read + 32 B mean read/write + 16 B M2 read/write per
// complex element.  A thread takes two neighbouring elements of a chain (per-chain accumulator rows are padded to an even
// length), so every access is a 16-byte vector; no shared memory, no atomics.
//
// k_moments_batch replaces k_moments on the accumulated iterations that close a batch of b (batch means, for the
// Monte-Carlo standard error of the mean).  The running mean of the first j b samples is the mean of the first j batch
// means, so Welford over the batch means needs no batch sum: after the normal update has produced mean_k (k = j b),
//   d = mean_k - snap;  M2_bm += j (j - 1) |d|^2;  snap = mean_k
// with snap the mean at the previous batch boundary (Ybar_j - mu_{j-1} = j d, Ybar_j - mu_j = (j - 1) d).  A closing
// launch moves 112 B per complex element: the 64 B above plus 32 B snap read/write and 16 B M2_bm read/write.
#include "hp_kernels.cuh"

namespace hp {
namespace {

constexpr int kMomThreads = 256;

__device__ __forceinline__ void welford(double2 x, double2& mu, double& m2, double invk) {
    const double dr = x.x - mu.x, di = x.y - mu.y;
    mu.x += dr * invk;
    mu.y += di * invk;
    m2 += dr * (x.x - mu.x) + di * (x.y - mu.y);
}

// element i of chain row: sample offset (complex elements) inside the chain's block of the source
__device__ __forceinline__ long long src_off(const MomentsArr& a, int i) {
    return a.w == a.rs ? (long long)i : (long long)(i / a.w) * a.rs + (i % a.w);
}

// the batch-means step of one element: mu = mean_k at the close of batch j, jj1 = j (j - 1)
__device__ __forceinline__ void close_batch(double2 mu, double2& snap, double& m2bm, double jj1) {
    const double dr = mu.x - snap.x, di = mu.y - snap.y;
    m2bm += jj1 * (dr * dr + di * di);
    snap = mu;
}

template <bool kBatch>
__device__ __forceinline__ void moments_pair(const MomentsArr& a, const MomentsBatch& bm, long long p, double invk,
                                             double jj1) {
    const long long P = a.ld >> 1;   // element pairs per chain
    if (p >= (long long)a.nsys * P) return;
    const int c = (int)(p / P);
    const int i0 = (int)(p - (long long)c * P) * 2;
    const bool two = i0 + 1 < a.L;
    const double2* src = reinterpret_cast<const double2*>(a.src) + (long long)c * a.src_cs;
    double2* mean = reinterpret_cast<double2*>(a.mean) + (long long)c * a.ld + i0;
    double2* m2p = reinterpret_cast<double2*>(a.m2 + (long long)c * a.ld + i0);
    const double2 x0 = __ldg(src + src_off(a, i0));
    const double2 x1 = __ldg(src + src_off(a, two ? i0 + 1 : i0));   // (an odd L: the pad element re-reads x0, unused)
    double2 mu0 = mean[0];
    double2 mu1 = two ? mean[1] : make_double2(0.0, 0.0);
    double2 m2 = *m2p;
    welford(x0, mu0, m2.x, invk);
    mean[0] = mu0;
    if (two) {
        welford(x1, mu1, m2.y, invk);
        mean[1] = mu1;
    }
    *m2p = m2;
    if constexpr (kBatch) {
        double2* snap = reinterpret_cast<double2*>(bm.snap) + (long long)c * a.ld + i0;
        double2* m2bp = reinterpret_cast<double2*>(bm.m2 + (long long)c * a.ld + i0);
        double2 s0 = snap[0];
        double2 s1 = two ? snap[1] : make_double2(0.0, 0.0);
        double2 mb = *m2bp;
        close_batch(mu0, s0, mb.x, jj1);
        snap[0] = s0;
        if (two) {
            close_batch(mu1, s1, mb.y, jj1);
            snap[1] = s1;
        }
        *m2bp = mb;
    }
}

__global__ void __launch_bounds__(kMomThreads) k_moments(MomentsArr a0, MomentsArr a1, long long nblk0, double invk) {
    const long long b = blockIdx.x;
    if (b < nblk0) moments_pair<false>(a0, MomentsBatch{}, b * kMomThreads + threadIdx.x, invk, 0.0);
    else moments_pair<false>(a1, MomentsBatch{}, (b - nblk0) * kMomThreads + threadIdx.x, invk, 0.0);
}

__global__ void __launch_bounds__(kMomThreads) k_moments_batch(MomentsArr a0, MomentsArr a1, MomentsBatch b0, MomentsBatch b1,
                                                               long long nblk0, double invk, double jj1) {
    const long long b = blockIdx.x;
    if (b < nblk0) moments_pair<true>(a0, b0, b * kMomThreads + threadIdx.x, invk, jj1);
    else moments_pair<true>(a1, b1, (b - nblk0) * kMomThreads + threadIdx.x, invk, jj1);
}

long long moments_blocks(const MomentsArr& a) {
    if (!a.src || a.L <= 0 || a.nsys <= 0) return 0;
    return ((long long)a.nsys * (a.ld >> 1) + kMomThreads - 1) / kMomThreads;
}

}  // namespace

int launch_moments(const MomentsArr& cr, const MomentsArr& fg, double invk, cudaStream_t st) {
    const long long n0 = moments_blocks(cr), n1 = moments_blocks(fg);
    if (n0 + n1 == 0) return 0;
    k_moments<<<(unsigned)(n0 + n1), kMomThreads, 0, st>>>(cr, fg, n0, invk);
    return 1;
}

int launch_moments_batch(const MomentsArr& cr, const MomentsArr& fg, const MomentsBatch& crb, const MomentsBatch& fgb,
                         double invk, double jj1, cudaStream_t st) {
    const long long n0 = moments_blocks(cr), n1 = moments_blocks(fg);
    if (n0 + n1 == 0) return 0;
    k_moments_batch<<<(unsigned)(n0 + n1), kMomThreads, 0, st>>>(cr, fg, crb, fgb, n0, invk, jj1);
    return 1;
}

}  // namespace hp
