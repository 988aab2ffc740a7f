// hp_fft2.cu -- k_post_fft2: the fused delay-transform kernel with register-resident FFTs.
//
// Same work as k_post_fft (hp_fft.cu; reference: gibbs_step_fgmodes, pspec.py:442-485, and the dense Fourier operator of
// utils.py:14-40 / pspec.py:91-95): per (baseline, time)  s = U^H (lam * ytilde),  model = s + F f,  residual, chi^2,
// ln-posterior partial sums, and |U (w s)|^2 partial sums.  ncu on the round-1 kernel: 81 % L1/TEX throughput, 32 % of the
// shared-memory wavefronts were bank-conflict replays of the five Stockham passes, 13 % DMMA pipe; this version
//
//   * keeps a whole FFT in the registers of one warp (E = Nfreqs / 32 points per lane; radices that divide E, so a lane owns
//     whole butterflies): between two passes the points cross shared memory once (E 16-byte stores + E 16-byte loads per
//     lane, index i stored at i + i / 8: conflict-free for the stride-Ns Stockham stores), with warp-level synchronisation
//     only; 384 points = 6 x 4 x 4 x 4 -> three crossings instead of five passes of load-compute-store with CTA barriers;
//   * reads ytilde straight from global into the first pass and leaves the last pass in registers (signal_cr goes from there
//     to global); the second transform runs its passes in the reverse radix order;
//   * computes F f on the tensor pipe (3M) and finishes the residual in the accumulator layout: the foreground model never
//     goes to shared memory (one buffer instead of two: three CTAs per SM instead of two).
//
// Taken for Nfreqs = 128, 256, 384, 512, 1024 (plans 4.4.4.2, 8.8.4, 6.4.4.4, 8.8.4.2, 8.8.4.4 as template parameters; from 512 on one
// CTA per SM: 16 / 32 points per lane need the whole register file: all index arithmetic but the lane is
// compile-time -- the run-time version spent half of its 6.6 k instructions per transform pair on it); everything else (and
// the general-basis first iteration) stays on k_post_fft.
#include "hp_kernels.cuh"
#include "hp_math.h"
#include "hp_mma.cuh"

namespace hp {

namespace {

constexpr int kTP2 = 8;   // times per CTA = warps per CTA
constexpr int kFft2Ctas = 2;   // resident CTAs per SM the register budget is sized for

__device__ __forceinline__ double2 cmul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 mul_mi(double2 a) { return make_double2(a.y, -a.x); }   // a * (-i)

// in-place forward DFT of R points:  a[q] <- sum_r a[r] exp(-2 pi i q r / R)
template <int R>
__device__ __forceinline__ void butterfly(double2* a);
template <>
__device__ __forceinline__ void butterfly<2>(double2* a) {
    const double2 t = a[1];
    a[1] = csub(a[0], t);
    a[0] = cadd(a[0], t);
}
template <>
__device__ __forceinline__ void butterfly<3>(double2* a) {
    const double S3 = 0.86602540378443864676;
    const double2 t1 = cadd(a[1], a[2]);
    const double2 t2 = make_double2(a[0].x - 0.5 * t1.x, a[0].y - 0.5 * t1.y);
    const double2 t3 = make_double2(S3 * (a[1].y - a[2].y), -S3 * (a[1].x - a[2].x));   // -i sqrt(3)/2 (a1 - a2)
    a[0] = cadd(a[0], t1);
    a[1] = cadd(t2, t3);
    a[2] = csub(t2, t3);
}
template <>
__device__ __forceinline__ void butterfly<4>(double2* a) {
    const double2 b0 = cadd(a[0], a[2]), b1 = csub(a[0], a[2]), b2 = cadd(a[1], a[3]), b3 = mul_mi(csub(a[1], a[3]));
    a[0] = cadd(b0, b2); a[1] = cadd(b1, b3); a[2] = csub(b0, b2); a[3] = csub(b1, b3);
}
template <>
__device__ __forceinline__ void butterfly<6>(double2* a) {
    // 6 = 2 x 3 (Good-Thomas: no twiddles): three-point DFTs of (a0, a2, a4) and (a3, a5, a1), then two-point combinations
    double2 e[3] = {a[0], a[2], a[4]}, o[3] = {a[3], a[5], a[1]};
    butterfly<3>(e);
    butterfly<3>(o);
    // X[q] = E[q mod 3] + (-1)^q O[q mod 3]
    a[0] = cadd(e[0], o[0]); a[3] = csub(e[0], o[0]);
    a[4] = cadd(e[1], o[1]); a[1] = csub(e[1], o[1]);
    a[2] = cadd(e[2], o[2]); a[5] = csub(e[2], o[2]);
}
template <>
__device__ __forceinline__ void butterfly<8>(double2* a) {
    const double H = 0.70710678118654752440;
    double2 e[4] = {a[0], a[2], a[4], a[6]}, o[4] = {a[1], a[3], a[5], a[7]};
    butterfly<4>(e);
    butterfly<4>(o);
    // twiddles exp(-2 pi i q / 8), q = 0..3:  1,  (1 - i)/sqrt2,  -i,  (-1 - i)/sqrt2
    const double2 o1 = make_double2(H * (o[1].x + o[1].y), H * (o[1].y - o[1].x));
    const double2 o2 = mul_mi(o[2]);
    const double2 o3 = make_double2(H * (o[3].y - o[3].x), -H * (o[3].x + o[3].y));
    a[0] = cadd(e[0], o[0]); a[4] = csub(e[0], o[0]);
    a[1] = cadd(e[1], o1);   a[5] = csub(e[1], o1);
    a[2] = cadd(e[2], o2);   a[6] = csub(e[2], o2);
    a[3] = cadd(e[3], o3);   a[7] = csub(e[3], o3);
}

__device__ __forceinline__ int phys(int i) { return i + (i >> 3); }

// One Stockham pass of one warp's FFT with everything but the lane known at compile time.
//   v[u * R + r] = input r of butterfly j = lane + 32 u (index j + r * nb, nb = n / R)
//   NS    : product of the radices of the earlier passes;  k = j mod NS, jq = j / NS
//   kLoad : fetch the inputs from `row` (shared memory, index i at phys(i)); else they are in v already
//   kStore: write the outputs to `row` (index jq NS R + k + r NS) between two __syncwarp; else they stay in v as output r of
//           butterfly j = index j + r * NS (only the last pass: NS R = n)
//   twt   : this pass's twiddle table, twt[k * (R - 1) + r - 1] = exp(-2 pi i r k / (NS R)): consecutive lanes read consecutive
//           entries (a look-up in the plain table exp(-2 pi i j / n) has a power-of-two stride and conflicts 8 - 16 ways)
template <int E, int R, int NS, bool kLoad, bool kStore>
__device__ __forceinline__ void fft_pass(double2 (&v)[E], double2* row, const double2* __restrict__ twt, int lane) {
    constexpr int n = 32 * E, NB = E / R, nb = n / R;
    static_assert(E % R == 0 && nb % 8 == 0, "a lane owns whole butterflies; rows of a butterfly are 8-aligned");
    if (kLoad) {
        // phys(lane + 32 u + r nb) = phys(lane) + 36 u + r (9 nb / 8): one base, compile-time offsets
        const double2* src = row + phys(lane);
#pragma unroll
        for (int u = 0; u < NB; ++u)
#pragma unroll
            for (int r = 0; r < R; ++r) v[u * R + r] = src[36 * u + r * (nb / 8 * 9)];
    }
#pragma unroll
    for (int u = 0; u < NB; ++u) {
        if (NS > 1) {
            const int k = (lane + 32 * u) % NS;
#pragma unroll
            for (int r = 1; r < R; ++r) v[u * R + r] = cmul(v[u * R + r], twt[k * (R - 1) + r - 1]);
        }
        butterfly<R>(&v[u * R]);
    }
    if (kStore) {
        __syncwarp();   // every lane has its inputs in registers: the row may be overwritten
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            const int j = lane + 32 * u, jq = j / NS, k = j - jq * NS;
            const int base = jq * (NS * R) + k;
#pragma unroll
            for (int r = 0; r < R; ++r) row[phys(base + r * NS)] = v[u * R + r];
        }
        __syncwarp();
    }
}

// A whole transform: radices P0 P1 P2 (P3) (P3 = 1: three passes); the first pass takes its inputs from v (kFromRegs) or from
// the row; the last pass leaves element u * R + r = index (lane + 32 u) + r * (n / R) in v.  Twiddle tables of pass p >= 1 at
// tw + (NS_p - P0).
template <int E, int P0, int P1, int P2, int P3, bool kFromRegs>
__device__ __forceinline__ void fft_run(double2 (&v)[E], double2* row, const double2* __restrict__ tw, int lane) {
    fft_pass<E, P0, 1, !kFromRegs, true>(v, row, tw, lane);
    fft_pass<E, P1, P0, true, true>(v, row, tw, lane);
    if constexpr (P3 > 1) {
        fft_pass<E, P2, P0 * P1, true, true>(v, row, tw + (P0 * P1 - P0), lane);
        fft_pass<E, P3, P0 * P1 * P2, true, false>(v, row, tw + (P0 * P1 * P2 - P0), lane);
    } else {
        fft_pass<E, P2, P0 * P1, true, false>(v, row, tw + (P0 * P1 - P0), lane);
    }
}

// per-pass twiddle tables of a plan, packed one after the other (pass p starts at NS_p - P0; n - P0 entries in all)
template <int E, int P0, int P1, int P2, int P3>
__device__ __forceinline__ void build_twiddle_tables(double2* dst, const double2* __restrict__ twg, int tid, int nthreads) {
    constexpr int n = 32 * E;
    constexpr int rad[4] = {P0, P1, P2, P3};
    int Ns = P0;
#pragma unroll
    for (int ps = 1; ps < 4; ++ps) {
        const int R = rad[ps];
        if (R <= 1) break;
        const int tstep = n / (Ns * R), cnt = Ns * (R - 1);
        double2* t = dst + (Ns - P0);
        for (int e = tid; e < cnt; e += nthreads) {
            const int k = e / (R - 1), r = e - k * (R - 1) + 1;
            t[e] = twg[r * k * tstep];
        }
        Ns *= R;
    }
}

}  // namespace

// Nfreqs covered by k_post_fft2: its radices are template parameters, 128 = 4.4.4.2, 256 = 8.8.4, 384 = 6.4.4.4,
// 512 = 8.8.4.2, 1024 = 8.8.4.4
bool postfft2_ok(int n) { return n == 128 || n == 256 || n == 384 || n == 512 || n == 1024; }

size_t postfft2_smem_bytes(int n, int m) {
    const int mk = ((m + 3) / 4) * 4;
    const int ld = n + n / 8 + 1;   // padded row: index i at i + i / 8, row stride == 1 (mod 8) sixteen-byte units
    return sizeof(double2) * ((size_t)kTP2 * ld + 2 * (size_t)n + (size_t)kTP2 * (((mk + 7) / 8) * 8 + 4)) + 80 * sizeof(double);
}

// E = Nfreqs / 32; forward radices P0 P1 P2 (P3); the second transform runs them in reverse order
template <int E, int P0, int P1, int P2, int P3>
__global__ void __launch_bounds__(32 * kTP2, (E >= 16 ? 1 : kFft2Ctas)) k_post_fft2(PostFftArgs a) {
    constexpr int kThreads = 32 * kTP2;
    constexpr int n = 32 * E, ld = n + n / 8 + 1;
    constexpr int RL = P3 > 1 ? P3 : P2;      // last forward radix = first reverse radix
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int m = a.m, mk = ((m + 3) / 4) * 4, ldf = ((mk + 7) / 8) * 8 + 4;   // ldf == 4 (mod 8): conflict-free fragment loads
    double2* A = reinterpret_cast<double2*>(smem_raw);          // [8][ld]: one FFT row per warp; later s in frequency space
    double2* tw = A + (size_t)kTP2 * ld;                         // [2][n] per-pass twiddle tables: forward plan, reverse plan
    double2* fs = tw + 2 * (size_t)n;                            // [8][ldf] foreground amplitudes of the tile's times
    double* red = reinterpret_cast<double*>(fs + (size_t)kTP2 * ldf);   // [8 warps][8 times]
    const int sys = blockIdx.y, tile = blockIdx.x, t0 = tile * kTP2;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const double* X = a.X + 2 * ((size_t)sys * a.Tp + t0) * a.Np;
    const double* lam = a.lam + (size_t)sys * a.Np;
    const double* w = a.w + (size_t)sys * a.w_bs + (size_t)t0 * a.w_ts;
    const double* wd = a.wd + 2 * ((size_t)sys * a.Tp + t0) * n;
    double* Sf = a.Sf + 2 * ((size_t)sys * a.sf_bs + (size_t)t0 * n);
    const double2* twg = reinterpret_cast<const double2*>(a.tw);
    const double rsn = rsqrt((double)n);

    {   // the data rows are consumed in the residual phase: start them on their way from DRAM to L2 now
        const char* wdp = reinterpret_cast<const char*>(wd);
        const size_t bytes = (size_t)min(kTP2, a.T - t0) * n * 16;
        for (size_t off = (size_t)tid * 128; off < bytes; off += kThreads * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(wdp + off));
    }
    // ---- first pass inputs straight from global:  conj(lam * ytilde) * (-1)^k  (U^H a = conj(U conj(a)); n is even)
    const int t = warp;                    // this warp's time
    const bool live = t0 + t < a.T;
    double2 v[E];
    {
        constexpr int nb0 = n / P0;
        const double* xr = X + 2 * (size_t)t * a.Np;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            // element e = u * P0 + r  <->  index (lane + 32 u) + r * nb0
            const int u = e / P0, r = e - u * P0;
            const int k = lane + 32 * u + r * nb0;
            double2 y = make_double2(0.0, 0.0);
            double l = 0.0;
            if (live) { y = *reinterpret_cast<const double2*>(xr + 2 * k); l = lam[k]; }
            const double sg = (k & 1) ? -l : l;
            v[e] = make_double2(sg * y.x, -sg * y.y);
        }
    }
    // the tables were built once per engine: a straight, coalesced copy (the per-CTA build is ~760 scattered 16-byte gathers
    // with index arithmetic in front of every CTA's first pass)
    const double2* t2 = reinterpret_cast<const double2*>(a.tw2);
    const int cnt = a.Empart ? 2 * n : n;
#pragma unroll 8   // the compiler's default unrolling hoists these loads over the first pass: 6 more registers at 1024 channels
    for (int e = tid; e < cnt; e += kThreads) tw[e] = t2[e];
    for (int e = tid; e < kTP2 * ldf; e += kThreads) {
        const int tt = e / ldf, j = e - tt * ldf;
        double2 f = make_double2(0.0, 0.0);
        if (j < m && t0 + tt < a.T) f = *reinterpret_cast<const double2*>(X + 2 * ((size_t)tt * a.Np + n + j));
        fs[e] = f;
        if (j < m && t0 + tt < a.T && a.fg_out)
            *reinterpret_cast<double2*>(a.fg_out + (size_t)sys * a.fg_bs + 2 * ((size_t)(t0 + tt) * m + j)) = f;
    }
    __syncthreads();   // twiddles and f in shared memory
    double2* row = A + (size_t)t * ld;
    // ---- FFT 1 (forward plan): first pass from registers, middle passes through the row, last pass stays in registers
    {
        fft_run<E, P0, P1, P2, P3, true>(v, row, tw, lane);
        // outputs: element u * R + r = index x = lane + 32 u + r * Ns (Ns = n / R).  s = conj(out * (-1)^x * c0) / sqrt(n)
        constexpr int R = RL, Ns = n / RL;
        const double2 c0 = twg[(int)(((long long)(n / 2) * (n / 2)) % n)];   // exp(-2 pi i h^2 / n), h = n / 2
        __syncwarp();   // the last pass has read the row
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int u = e / R, r = e - u * R;
            const int x = lane + 32 * u + r * Ns;
            double2 o = cmul(v[e], c0);
            const double sg = (x & 1) ? -rsn : rsn;
            o = make_double2(sg * o.x, -sg * o.y);
            row[phys(x)] = o;
            if (live) *reinterpret_cast<double2*>(Sf + 2 * ((size_t)t * n + x)) = o;
        }
    }
    __syncthreads();   // s of all eight times is in A
    // ---- foreground model F f on the tensor pipe (3M), finished in the accumulator layout:
    //      lane (g, q) holds (F f)[time g][x = 8 ct + 2 q + e]; residual, chi^2, ln-posterior partials, masked signal
    {
        const double* Ft = a.Ft + 2 * (size_t)sys * m * n;
        const int nct = n / 8;
        const int g = lane >> 2, q = lane & 3;
        const bool tlive = t0 + g < a.T;
        const double* wrow = w + (size_t)g * a.w_ts;
        const double* nd = a.ninvd + (size_t)sys * a.ninv_bs + (size_t)(t0 + g) * a.ninv_ts;   // this lane's time
        double lnp = 0.0;
        // One group of global loads in flight per warp: the B fragments of all k-steps (mk <= 32: eight; more modes: the
        // first eight, the rest on demand) and the data of the NEXT tile are requested before this tile's products.
        constexpr int kBF = 8;
        double2 bnx[kBF], dnx[2];
        auto load_tile = [&](int ct, double2 (&b)[kBF], double2 (&d)[2]) {
            const int x = 8 * ct + g;
#pragma unroll
            for (int s8 = 0; s8 < kBF; ++s8) {
                const int k = 4 * s8 + q;
                b[s8] = (k < m && ct < nct) ? *reinterpret_cast<const double2*>(Ft + 2 * ((size_t)k * n + x)) : make_double2(0.0, 0.0);
            }
            d[0] = d[1] = make_double2(0.0, 0.0);
            if (tlive && ct < nct) {
                d[0] = *reinterpret_cast<const double2*>(wd + 2 * ((size_t)g * n + 8 * ct + 2 * q));
                d[1] = *reinterpret_cast<const double2*>(wd + 2 * ((size_t)g * n + 8 * ct + 2 * q + 1));
            }
        };
        load_tile(warp, bnx, dnx);
        for (int ct = warp; ct < nct; ct += kTP2) {
            double p1[2] = {0.0, 0.0}, p2[2] = {0.0, 0.0}, p3[2] = {0.0, 0.0};
            const int x0 = 8 * ct + 2 * q;
            double2 bc[kBF];
#pragma unroll
            for (int s8 = 0; s8 < kBF; ++s8) bc[s8] = bnx[s8];
            const double2 d0 = dnx[0], d1 = dnx[1];
            load_tile(ct + kTP2, bnx, dnx);
#pragma unroll
            for (int s8 = 0; s8 < kBF; ++s8) {
                const int k = 4 * s8 + q;
                if (4 * s8 < mk) {
                    const double2 af = fs[(size_t)g * ldf + k];
                    dmma884(p1[0], p1[1], af.x, bc[s8].x);
                    dmma884(p2[0], p2[1], af.y, bc[s8].y);
                    dmma884(p3[0], p3[1], af.x + af.y, bc[s8].x + bc[s8].y);
                }
            }
            for (int kc = 4 * kBF; kc < mk; kc += 4) {   // more than 32 foreground modes: remaining k-steps straight from L2
                const int k = kc + q;
                const double2 af = fs[(size_t)g * ldf + k];
                const double2 b = k < m ? *reinterpret_cast<const double2*>(Ft + 2 * ((size_t)k * n + 8 * ct + g)) : make_double2(0.0, 0.0);
                dmma884(p1[0], p1[1], af.x, b.x);
                dmma884(p2[0], p2[1], af.y, b.y);
                dmma884(p3[0], p3[1], af.x + af.y, b.x + b.y);
            }
            const double2 s0 = A[(size_t)g * ld + phys(x0)], s1 = A[(size_t)g * ld + phys(x0 + 1)];
            const double wx0 = (a.w_ts == 0 || tlive) ? wrow[x0] : 0.0, wx1 = (a.w_ts == 0 || tlive) ? wrow[x0 + 1] : 0.0;
            const double n0 = nd[x0], n1 = nd[x0 + 1];
            const double rr0 = d0.x - s0.x - (p1[0] - p2[0]), ri0 = d0.y - s0.y - (p3[0] - p1[0] - p2[0]);
            const double rr1 = d1.x - s1.x - (p1[1] - p2[1]), ri1 = d1.y - s1.y - (p3[1] - p1[1] - p2[1]);
            const double q0 = rr0 * rr0 + ri0 * ri0, q1 = rr1 * rr1 + ri1 * ri1;
            if (tlive) {
                if (a.chisq_out)
                    *reinterpret_cast<double2*>(a.chisq_out + (size_t)sys * a.chisq_bs + (size_t)(t0 + g) * n + x0) = make_double2(q0 * n0, q1 * n1);
                lnp += wx0 * n0 * q0 + wx1 * n1 * q1;
                if (a.Rm) {
                    double* rm = a.Rm + 2 * (((size_t)sys * a.Tp + t0 + g) * n + x0);
                    *reinterpret_cast<double2*>(rm) = make_double2(wx0 * rr0, wx0 * ri0);
                    *reinterpret_cast<double2*>(rm + 2) = make_double2(wx1 * rr1, wx1 * ri1);
                }
            }
            if (a.Empart) {
                // input of the second transform, in place: w s (-1)^x  (x0 is even)
                A[(size_t)g * ld + phys(x0)] = make_double2(wx0 * s0.x, wx0 * s0.y);
                A[(size_t)g * ld + phys(x0 + 1)] = make_double2(-wx1 * s1.x, -wx1 * s1.y);
            }
        }
        lnp += __shfl_xor_sync(0xffffffffu, lnp, 1);
        lnp += __shfl_xor_sync(0xffffffffu, lnp, 2);
        if (q == 0) red[warp * kTP2 + g] = lnp;
    }
    __syncthreads();
    if (tid < kTP2) {
        double s = 0.0;
        for (int wv = 0; wv < kTP2; ++wv) s += red[wv * kTP2 + tid];
        if (t0 + tid < a.Tp) a.lnp1[(size_t)sys * a.Tp + t0 + tid] = t0 + tid < a.T ? s : 0.0;
    }
    // ---- |U (w s)|^2 summed over the tile's times (second term of ln_post, pspec.py:479-483): reverse plan
    if (a.Empart) {
        if constexpr (P3 > 1) fft_run<E, P3, P2, P1, P0, false>(v, row, tw + n, lane);
        else fft_run<E, P2, P1, P0, 1, false>(v, row, tw + n, lane);
        constexpr int R = P0, Ns = n / P0;
        __syncwarp();   // the last pass has read the row: park |.|^2 in it (doubles, index k)
        double* erow = reinterpret_cast<double*>(row);
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int u = e / R, r = e - u * R;
            erow[lane + 32 * u + r * Ns] = live ? v[e].x * v[e].x + v[e].y * v[e].y : 0.0;
        }
        __syncthreads();
        double* Ep = a.Empart + ((size_t)sys * gridDim.x + tile) * n;
        for (int k = tid; k < n; k += kThreads) {
            double acc = 0.0;
#pragma unroll
            for (int tt = 0; tt < kTP2; ++tt) acc += reinterpret_cast<const double*>(A + (size_t)tt * ld)[k];
            Ep[k] = acc / (double)n;
        }
    }
}

namespace {
template <int E, int P0, int P1, int P2, int P3>
__global__ void __launch_bounds__(256) k_fft2_tables(double2* tw2, const double2* twg) {
    constexpr int n = 32 * E;
    for (int e = threadIdx.x; e < 2 * n; e += 256) tw2[e] = make_double2(0.0, 0.0);
    __syncthreads();
    build_twiddle_tables<E, P0, P1, P2, P3>(tw2, twg, threadIdx.x, 256);
    if constexpr (P3 > 1) build_twiddle_tables<E, P3, P2, P1, P0>(tw2 + n, twg, threadIdx.x, 256);
    else build_twiddle_tables<E, P2, P1, P0, 1>(tw2 + n, twg, threadIdx.x, 256);
}
}  // namespace

void launch_fft2_tables(double* tw2, const double* tw, int n, cudaStream_t st) {
    double2* o = reinterpret_cast<double2*>(tw2);
    const double2* t = reinterpret_cast<const double2*>(tw);
    if (n == 128) k_fft2_tables<4, 4, 4, 4, 2><<<1, 256, 0, st>>>(o, t);
    else if (n == 256) k_fft2_tables<8, 8, 8, 4, 1><<<1, 256, 0, st>>>(o, t);
    else if (n == 384) k_fft2_tables<12, 6, 4, 4, 4><<<1, 256, 0, st>>>(o, t);
    else if (n == 512) k_fft2_tables<16, 8, 8, 4, 2><<<1, 256, 0, st>>>(o, t);
    else if (n == 1024) k_fft2_tables<32, 8, 8, 4, 4><<<1, 256, 0, st>>>(o, t);
}

void launch_post_fft2(const PostFftArgs& a, cudaStream_t st) {
    const int n = a.plan.n;
    const size_t smem = postfft2_smem_bytes(n, a.m);
    static size_t attr_dev[kMaxDev][5] = {{0}};
    const int slot = n == 128 ? 0 : (n == 256 ? 1 : (n == 384 ? 2 : (n == 512 ? 3 : 4)));
    size_t& attr = attr_dev[current_device_slot()][slot];
    const dim3 grid((a.T + kTP2 - 1) / kTP2, a.nsys);
    if (n == 128) {
        if (smem > attr) { cudaFuncSetAttribute(k_post_fft2<4, 4, 4, 4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = smem; }
        k_post_fft2<4, 4, 4, 4, 2><<<grid, 32 * kTP2, smem, st>>>(a);
    } else if (n == 256) {
        if (smem > attr) { cudaFuncSetAttribute(k_post_fft2<8, 8, 8, 4, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = smem; }
        k_post_fft2<8, 8, 8, 4, 1><<<grid, 32 * kTP2, smem, st>>>(a);
    } else if (n == 384) {
        if (smem > attr) { cudaFuncSetAttribute(k_post_fft2<12, 6, 4, 4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = smem; }
        k_post_fft2<12, 6, 4, 4, 4><<<grid, 32 * kTP2, smem, st>>>(a);
    } else if (n == 512) {
        if (smem > attr) { cudaFuncSetAttribute(k_post_fft2<16, 8, 8, 4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = smem; }
        k_post_fft2<16, 8, 8, 4, 2><<<grid, 32 * kTP2, smem, st>>>(a);
    } else if (n == 1024) {
        if (smem > attr) { cudaFuncSetAttribute(k_post_fft2<32, 8, 8, 4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = smem; }
        k_post_fft2<32, 8, 8, 4, 4><<<grid, 32 * kTP2, smem, st>>>(a);
    }
}

}  // namespace hp
