// hp_moments.cu -- k_moments: on-device posterior moments of signal_cr and fg_amps (Welford, FP64).
//
// One launch per sub-batch and accumulated iteration updates the per-chain accumulators of both arrays:
//   d = x - mean;  mean += d / k;  M2 += Re(d conj(x - mean))   (= |d|^2 (k - 1) / k)
// The update order is the iteration order, so the moments of a chain do not depend on how its iterations were split over
// calls, sub-streams or read-ahead.  Bandwidth-bound: 16 B sample read + 32 B mean read/write + 16 B M2 read/write per
// complex element.  A thread takes two neighbouring elements of a chain (per-chain accumulator rows are padded to an even
// length), so every access is a 16-byte vector; no shared memory, no atomics.
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

__device__ __forceinline__ void moments_pair(const MomentsArr& a, long long p, double invk) {
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
}

__global__ void __launch_bounds__(kMomThreads) k_moments(MomentsArr a0, MomentsArr a1, long long nblk0, double invk) {
    const long long b = blockIdx.x;
    if (b < nblk0) moments_pair(a0, b * kMomThreads + threadIdx.x, invk);
    else moments_pair(a1, (b - nblk0) * kMomThreads + threadIdx.x, invk);
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

}  // namespace hp
