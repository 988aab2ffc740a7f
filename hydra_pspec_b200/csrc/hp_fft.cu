// hp_fft.cu -- fused delay-transform kernel (shared-memory Stockham FFT + DMMA foreground products).
//
// The reference applies its shifted Fourier operator (utils.py:14-40) as dense matrices
// (pspec.py:91-95, 313-322).  On the device the operator is only ever applied to vectors, so it
// becomes an in-shared-memory mixed-radix FFT with pre/post twiddles for the two half-band shifts:
//
//     (U v)[k] = post[k] * sum_x exp(-2 pi i k x / n) (pre[x] v[x]),      h = n // 2
//     pre[x]  = exp(+2 pi i h x / n),   post[k] = exp(+2 pi i h k / n) exp(-2 pi i h^2 / n) / sqrt(n)
//
// and U^H v = conj(U conj(v)) because U is symmetric.
//
//   k_post_fft  : per (baseline, 8 times): s = U^H (lam * ytilde), model = s + F f (DMMA),
//                 residual, chi^2, ln-posterior partial sums, and |U (w s)|^2 partial sums
//                 (gibbs_step_fgmodes, pspec.py:442-485)
#include "hp_kernels.cuh"
#include "hp_math.h"
#include "hp_mma.cuh"

namespace hp {

namespace {

__device__ __forceinline__ double2 cmul2(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 cconj(double2 a) { return make_double2(a.x, -a.y); }
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
// multiply by -i / +i
__device__ __forceinline__ double2 cmul_mi(double2 a) { return make_double2(a.y, -a.x); }

// Forward DFT (kernel exp(-2 pi i k x / n)) of nvec vectors of length n, Stockham autosort,
// ping-pong between src and dst; returns the buffer that holds the result.  tw[j] = exp(-2 pi i j / n).
// All threads of the CTA must call it; it starts and ends with a barrier.
__device__ double2* fft_forward(double2* src, double2* dst, int nvec, const FftPlan& p, const double2* tw) {
    const int n = p.n;
    int Ns = 1;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int pass = 0; pass < p.nf; ++pass) {
        const int R = p.radix[pass];
        const int nb = n / R;
        const int tstep = n / (Ns * R);
        const uint32_t magic = p.magic[pass];  // ceil(2^32 / Ns): j / Ns = umulhi(j, magic) for j, Ns < 2^16
        // one warp per vector, lanes over the butterflies: no integer division in the index arithmetic
        for (int v = warp; v < nvec; v += nwarps) {
            const double2* sv = src + (size_t)v * n;
            double2* dv = dst + (size_t)v * n;
            for (int j = lane; j < nb; j += 32) {
                const int jq = Ns > 1 ? (int)__umulhi((uint32_t)j, magic) : j;   // j / Ns
                const int k = j - jq * Ns;                                        // j % Ns
                const double2* s = sv + j;
                double2* d = dv + jq * Ns * R + k;
                const int tk = k * tstep;  // twiddle index step: exp(-2 pi i r k / (Ns R)) = tw[r * tk]
                if (R == 4) {
                    double2 a0 = s[0], a1 = s[nb], a2 = s[2 * nb], a3 = s[3 * nb];
                    if (k) { a1 = cmul2(a1, tw[tk]); a2 = cmul2(a2, tw[2 * tk]); a3 = cmul2(a3, tw[3 * tk]); }
                    double2 b0 = cadd(a0, a2), b1 = csub(a0, a2), b2 = cadd(a1, a3), b3 = cmul_mi(csub(a1, a3));
                    d[0] = cadd(b0, b2); d[Ns] = cadd(b1, b3); d[2 * Ns] = csub(b0, b2); d[3 * Ns] = csub(b1, b3);
                } else if (R == 2) {
                    double2 a0 = s[0], a1 = s[nb];
                    if (k) a1 = cmul2(a1, tw[tk]);
                    d[0] = cadd(a0, a1); d[Ns] = csub(a0, a1);
                } else if (R == 3) {
                    double2 a0 = s[0], a1 = s[nb], a2 = s[2 * nb];
                    if (k) { a1 = cmul2(a1, tw[tk]); a2 = cmul2(a2, tw[2 * tk]); }
                    const double S3 = 0.86602540378443864676;
                    double2 t1 = cadd(a1, a2), t2 = make_double2(a0.x - 0.5 * t1.x, a0.y - 0.5 * t1.y);
                    double2 t3 = make_double2(S3 * (a1.y - a2.y), -S3 * (a1.x - a2.x));  // -i sqrt(3)/2 (a1 - a2)
                    d[0] = cadd(a0, t1); d[Ns] = cadd(t2, t3); d[2 * Ns] = csub(t2, t3);
                } else {
                    // generic radix (5, 7, 11, ...): O(R^2) with table twiddles
                    const int wstep = n / R;  // exp(-2 pi i q r / R) = tw[((q r) % R) * wstep]
                    for (int q = 0; q < R; ++q) {
                        double2 acc = make_double2(0.0, 0.0);
                        for (int r = 0; r < R; ++r) {
                            double2 a = s[r * nb];
                            int idx = r * tk + ((q * r) % R) * wstep;
                            idx %= n;
                            acc = cadd(acc, cmul2(a, tw[idx]));
                        }
                        d[q * Ns] = acc;
                    }
                }
            }
        }
        __syncthreads();
        double2* t = src; src = dst; dst = t;
        Ns *= R;
    }
    return src;
}

// exp(+2 pi i h x / n), h = n // 2: (-1)^x for even n (no table look-up, no integer division)
__device__ __forceinline__ double2 shift_pre(const double2* tw, int n, int x) {
    if ((n & 1) == 0) return make_double2((x & 1) ? -1.0 : 1.0, 0.0);
    return cconj(tw[(int)(((uint32_t)(n / 2) * (uint32_t)x) % (uint32_t)n)]);
}
// v * shift_pre(x)
__device__ __forceinline__ double2 mul_shift_pre(double2 v, const double2* tw, int n, int x) {
    if ((n & 1) == 0) return (x & 1) ? make_double2(-v.x, -v.y) : v;
    return cmul2(v, shift_pre(tw, n, x));
}

// one warp: C (8 x 8 complex) += A (8 x K, shared, interleaved, ld in complex) . B (K x 8, global interleaved)
//   B element (k, col) at Bg[k * sBk + col * sBj] (complex strides), conjugated if BC; rows k >= K zero.
template <bool BC>
__device__ __forceinline__ void warp_fg_product(double (&cr)[2], double (&ci)[2], const double2* As, int lda,
                                                const double* Bg, long long sBk, long long sBj, int col0, int ncols,
                                                int k0, int k1) {
    const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
    const bool colok = col0 + g < ncols;
    for (int kk = k0; kk < k1; kk += 4) {
        const int k = kk + q;
        double2 a = make_double2(0.0, 0.0), b = make_double2(0.0, 0.0);
        if (k < k1) {
            a = As[(size_t)g * lda + k];
            if (colok) b = *reinterpret_cast<const double2*>(Bg + 2 * ((long long)k * sBk + (long long)(col0 + g) * sBj));
        }
        if (BC) b.y = -b.y;
        dmma884(cr[0], cr[1], a.x, b.x);
        dmma884(ci[0], ci[1], a.x, b.y);
        dmma884(cr[0], cr[1], -a.y, b.y);
        dmma884(ci[0], ci[1], a.y, b.x);
    }
}

}  // namespace

bool make_fft_plan(int n, FftPlan* plan) {
    plan->n = n;
    plan->nf = 0;
    int rem = n;
    while (rem % 4 == 0 && plan->nf < 16) { plan->radix[plan->nf++] = 4; rem /= 4; }
    for (int p = 2; p <= 31 && rem > 1; ++p)
        while (rem % p == 0) {
            if (plan->nf >= 16) return false;
            plan->radix[plan->nf++] = p;
            rem /= p;
        }
    int Ns = 1;
    for (int i = 0; i < plan->nf; ++i) {
        plan->magic[i] = Ns > 1 ? (uint32_t)((0x100000000ull + (uint64_t)Ns - 1) / (uint64_t)Ns) : 0u;
        Ns *= plan->radix[i];
    }
    return rem == 1 && n >= 2 && n < 65536;
}

__global__ void k_twiddles(double* tw, int n) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    double s, c;
    sincospi(-2.0 * (double)j / (double)n, &s, &c);
    tw[2 * j] = c;
    tw[2 * j + 1] = s;
}
void launch_twiddles(double* tw, int n, cudaStream_t st) { k_twiddles<<<(n + 255) / 256, 256, 0, st>>>(tw, n); }

// ==========================================================================================
// kTP = times per CTA of the fused transform kernel = its warp count (one warp per time): 8 normally, 4 when the
// two ping-pong buffers of 8 times would not fit shared memory (Nfreqs = 1024)

size_t postfft_smem_bytes(int n, int m, int ktp) {
    int mk = ((m + 3) / 4) * 4;
    return sizeof(double2) * ((size_t)2 * ktp * n + n + (size_t)ktp * (mk + 1)) + 64 * sizeof(double);
}
int postfft_ktp(int n, int m, size_t max_smem) {
    for (int ktp = 8; ktp >= 4; ktp /= 2)
        if (postfft_smem_bytes(n, m, ktp) <= max_smem) return ktp;
    return 0;
}

template <int kTP>
__global__ void __launch_bounds__(32 * kTP, kTP == 8 ? 2 : 1) k_post_fft(PostFftArgs a) {
    constexpr int kThreads = 32 * kTP;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = a.plan.n, m = a.m, mk = ((m + 3) / 4) * 4, ldf = mk + 1;
    double2* buf0 = reinterpret_cast<double2*>(smem_raw);
    double2* buf1 = buf0 + (size_t)kTP * n;
    double2* tw = buf1 + (size_t)kTP * n;
    double2* fs = tw + n;
    double* red = reinterpret_cast<double*>(fs + (size_t)kTP * ldf);
    const int sys = blockIdx.y, tile = blockIdx.x, t0 = tile * kTP;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const double* X = a.X + 2 * ((size_t)sys * a.Tp + t0) * a.Np;
    const double* lam = a.lam + (size_t)sys * a.Np;
    const double* w = a.w + (size_t)sys * a.w_bs + (size_t)t0 * a.w_ts;
    const double* nd = a.ninvd + (size_t)sys * a.ninv_bs + (size_t)t0 * a.ninv_ts;
    double* Sf = a.Sf + 2 * ((size_t)sys * a.sf_bs + (size_t)t0 * n);
    const double2* twg = reinterpret_cast<const double2*>(a.tw);
    const double rsn = rsqrt((double)n);
    const double2 c0 = twg[(int)(((long long)(n / 2) * (n / 2)) % n)];  // exp(-2 pi i h^2 / n)

    {   // the data rows are consumed last: start them on their way from DRAM to L2 now
        const char* wdp = reinterpret_cast<const char*>(a.wd + 2 * ((size_t)sys * a.Tp + t0) * n);
        const size_t bytes = (size_t)min(kTP, a.T - t0) * n * 16;
        for (size_t off = (size_t)tid * 128; off < bytes; off += kThreads * 128)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(wdp + off));
    }
    for (int j = tid; j < n; j += kThreads) tw[j] = twg[j];
    for (int e = tid; e < kTP * ldf; e += kThreads) {
        int t = e / ldf, j = e - t * ldf;
        double2 v = make_double2(0.0, 0.0);
        if (j < m && t0 + t < a.T) v = *reinterpret_cast<const double2*>(X + 2 * ((size_t)t * a.Np + n + j));
        fs[e] = v;
        if (j < m && t0 + t < a.T && a.fg_out)
            *reinterpret_cast<double2*>(a.fg_out + (size_t)sys * a.fg_bs + 2 * ((size_t)(t0 + t) * m + j)) = v;
    }
    __syncthreads();
    double2* sbuf;
    if (a.do_inverse) {
        // s = U^H a = conj(U conj(a)),  a = lam * ytilde.   One warp per time (kTP == warps of the CTA).
        {
            const int t = warp;
            const bool live = t0 + t < a.T;
            // batches of four independent 16-byte loads per lane (the one-at-a-time loop exposed a full DRAM / L2
            // latency per element: 12 serialised round trips at Nfreqs = 384)
            for (int k0 = lane; k0 < n; k0 += 128) {
                double2 v[4];
                double l[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int k = k0 + 32 * u;
                    v[u] = make_double2(0.0, 0.0);
                    l[u] = 0.0;
                    if (live && k < n) {
                        v[u] = *reinterpret_cast<const double2*>(X + 2 * ((size_t)t * a.Np + k));
                        l[u] = lam[k];
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int k = k0 + 32 * u;
                    if (k < n) buf0[(size_t)t * n + k] = mul_shift_pre(make_double2(l[u] * v[u].x, -l[u] * v[u].y), tw, n, k);
                }
            }
        }
        __syncthreads();
        double2* res = fft_forward(buf0, buf1, kTP, a.plan, tw);
        {
            const int t = warp;
            const bool live = t0 + t < a.T;
            for (int x = lane; x < n; x += 32) {
                double2 v = cconj(cmul2(mul_shift_pre(res[(size_t)t * n + x], tw, n, x), c0));
                v.x *= rsn; v.y *= rsn;
                res[(size_t)t * n + x] = v;
                if (live) *reinterpret_cast<double2*>(Sf + 2 * ((size_t)t * n + x)) = v;
            }
        }
        sbuf = res;
    } else {
        {
            const int t = warp;
            const bool live = t0 + t < a.T;
            for (int x = lane; x < n; x += 32)
                buf0[(size_t)t * n + x] = live ? *reinterpret_cast<const double2*>(Sf + 2 * ((size_t)t * n + x)) : make_double2(0.0, 0.0);
        }
        sbuf = buf0;
    }
    double2* obuf = sbuf == buf0 ? buf1 : buf0;
    __syncthreads();
    // foreground model F f on the tensor pipe:  obuf[t][x] = sum_j f[t][j] Ft[j][x]
    // A = f tile (8 x m) stays in registers for all column tiles; the B fragments of a tile come
    // straight from global (L2-resident Ft) as one 16-byte load per k-step, issued as a batch and
    // prefetched one tile ahead.
    {
        const double* Ft = a.Ft + 2 * (size_t)sys * m * n;
        const int nct = (n + 7) / 8;
        const int g = lane >> 2, q = lane & 3;
        for (int kc = 0; kc < mk; kc += 32) {  // chunks of 8 k-steps
            double2 af[8], bcur[8], bnxt[8];
#pragma unroll
            for (int s8 = 0; s8 < 8; ++s8) {
                int k = kc + 4 * s8 + q;
                af[s8] = (k < mk && g < kTP) ? fs[(size_t)g * ldf + k] : make_double2(0.0, 0.0);
            }
            auto load_b = [&](int ct, double2 (&b)[8]) {
                const int x = 8 * ct + g;
#pragma unroll
                for (int s8 = 0; s8 < 8; ++s8) {
                    int k = kc + 4 * s8 + q;
                    b[s8] = (k < m && x < n && ct < nct) ? *reinterpret_cast<const double2*>(Ft + 2 * ((size_t)k * n + x))
                                                         : make_double2(0.0, 0.0);
                }
            };
            load_b(warp, bcur);
            for (int ct = warp; ct < nct; ct += kTP) {
                load_b(ct + kTP, bnxt);
                // three real DMMAs per complex MAC (3M):  P1 = Ar Br, P2 = Ai Bi, P3 = (Ar + Ai)(Br + Bi)
                double p1[2] = {0.0, 0.0}, p2[2] = {0.0, 0.0}, p3[2] = {0.0, 0.0};
#pragma unroll
                for (int s8 = 0; s8 < 8; ++s8) {
                    dmma884(p1[0], p1[1], af[s8].x, bcur[s8].x);
                    dmma884(p2[0], p2[1], af[s8].y, bcur[s8].y);
                    dmma884(p3[0], p3[1], af[s8].x + af[s8].y, bcur[s8].x + bcur[s8].y);
                }
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    int x = 8 * ct + 2 * q + e;
                    if (x < n && g < kTP) {
                        double2 v = make_double2(p1[e] - p2[e], p3[e] - p1[e] - p2[e]);
                        if (kc) { double2 o = obuf[(size_t)g * n + x]; v.x += o.x; v.y += o.y; }
                        obuf[(size_t)g * n + x] = v;
                    }
                }
#pragma unroll
                for (int s8 = 0; s8 < 8; ++s8) bcur[s8] = bnxt[s8];
            }
        }
        if (mk == 0)
            for (int e = tid; e < kTP * n; e += kThreads) obuf[e] = make_double2(0.0, 0.0);
    }
    __syncthreads();
    // residual, chi^2, ln-posterior partial, masked signal
    {
        const double* wd = a.wd + 2 * ((size_t)sys * a.Tp + t0) * n;
        double part[kTP];
#pragma unroll
        for (int t = 0; t < kTP; ++t) part[t] = 0.0;
        for (int x = tid; x < n; x += kThreads) {
            // all global loads of this channel first: the optional global stores below (chi^2, masked residual) would
            // otherwise keep the compiler from moving the next time's load above them (one exposed latency per time)
            double2 dv[kTP];
            double wv[kTP], nv[kTP];
#pragma unroll
            for (int t = 0; t < kTP; ++t) {
                dv[t] = make_double2(0.0, 0.0);
                if (t0 + t < a.T) dv[t] = *reinterpret_cast<const double2*>(wd + 2 * ((size_t)t * n + x));
                wv[t] = (a.w_ts == 0 || t0 + t < a.T) ? w[(size_t)t * a.w_ts + x] : 0.0;
                nv[t] = (a.ninv_ts == 0 || t0 + t < a.T) ? nd[(size_t)t * a.ninv_ts + x] : 0.0;
            }
#pragma unroll
            for (int t = 0; t < kTP; ++t) {
                const double wx = wv[t], ndx = nv[t];
                double2 s = sbuf[(size_t)t * n + x];
                double2 mf = obuf[(size_t)t * n + x];
                const double2 d = dv[t];
                double rr = d.x - s.x - mf.x, ri = d.y - s.y - mf.y;
                double r2 = rr * rr + ri * ri;
                if (t0 + t < a.T) {
                    if (a.chisq_out) a.chisq_out[(size_t)sys * a.chisq_bs + (size_t)(t0 + t) * n + x] = r2 * ndx;
                    part[t] += wx * ndx * r2;
                    if (a.Rm)
                        *reinterpret_cast<double2*>(a.Rm + 2 * (((size_t)sys * a.Tp + t0 + t) * n + x)) = make_double2(wx * rr, wx * ri);
                }
                obuf[(size_t)t * n + x] = mul_shift_pre(make_double2(wx * s.x, wx * s.y), tw, n, x);
            }
        }
#pragma unroll
        for (int t = 0; t < kTP; ++t) {
            double v = part[t];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) red[warp * kTP + t] = v;
        }
        __syncthreads();
        if (tid < kTP) {
            double s = 0.0;
            for (int wv = 0; wv < kTP; ++wv) s += red[wv * kTP + tid];
            if (t0 + tid < a.Tp) a.lnp1[(size_t)sys * a.Tp + t0 + tid] = t0 + tid < a.T ? s : 0.0;
        }
    }
    __syncthreads();
    // |U (w s)|^2 summed over the tile's times (second term of ln_post, pspec.py:479-483)
    if (a.Empart) {
        double2* res = fft_forward(obuf, sbuf, kTP, a.plan, tw);
        double* Ep = a.Empart + ((size_t)sys * gridDim.x + tile) * n;
        for (int k = tid; k < n; k += kThreads) {
            double acc = 0.0;
#pragma unroll
            for (int t = 0; t < kTP; ++t) { double2 v = res[(size_t)t * n + k]; acc += v.x * v.x + v.y * v.y; }
            Ep[k] = acc / (double)n;
        }
    }
    __syncthreads();
    // |U s|^2 (unmasked) for the general-basis iteration: reload s from global
    if (a.Eupart) {
        __syncthreads();
        {
            const int t = warp;
            const bool live = t0 + t < a.T;
            for (int x = lane; x < n; x += 32) {
                double2 v = make_double2(0.0, 0.0);
                if (live) v = mul_shift_pre(*reinterpret_cast<const double2*>(Sf + 2 * ((size_t)t * n + x)), tw, n, x);
                buf0[(size_t)t * n + x] = v;
            }
        }
        double2* res = fft_forward(buf0, buf1, kTP, a.plan, tw);
        double* Ep = a.Eupart + ((size_t)sys * gridDim.x + tile) * n;
        for (int k = tid; k < n; k += kThreads) {
            double acc = 0.0;
#pragma unroll
            for (int t = 0; t < kTP; ++t) { double2 v = res[(size_t)t * n + k]; acc += v.x * v.x + v.y * v.y; }
            Ep[k] = acc / (double)n;
        }
    }
}

int postfft_tiles(int T, int ktp) { return (T + ktp - 1) / ktp; }

void launch_post_fft(const PostFftArgs& a, cudaStream_t st) {
    const size_t smem = postfft_smem_bytes(a.plan.n, a.m, a.ktp);
    static size_t attr8_dev[kMaxDev] = {0}, attr4_dev[kMaxDev] = {0};
    size_t& attr8 = attr8_dev[current_device_slot()];
    size_t& attr4 = attr4_dev[current_device_slot()];
    if (a.ktp == 8) {
        if (smem > attr8) { cudaFuncSetAttribute(k_post_fft<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr8 = smem; }
        k_post_fft<8><<<dim3(postfft_tiles(a.T, 8), a.nsys), 256, smem, st>>>(a);
    } else {
        if (smem > attr4) { cudaFuncSetAttribute(k_post_fft<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr4 = smem; }
        k_post_fft<4><<<dim3(postfft_tiles(a.T, 4), a.nsys), 128, smem, st>>>(a);
    }
}

}  // namespace hp
