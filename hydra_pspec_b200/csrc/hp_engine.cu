// hp_engine.cu -- chain engine and C ABI (include/hydra_pspec_b200.h).
//
// One engine holds `nchains` independent baselines of identical shape resident in HBM and
// advances all of them one Gibbs iteration per step with a fixed sequence of batched kernels
// (hp_kernels.cu).  The host only enqueues launches; nothing is read back between iterations.
#include "../../include/hydra_pspec_b200.h"
#include "hp_kernels.cuh"
#include "hp_math.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CU_TRY(expr)                                                                              \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return fail(HP_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));        \
    } while (0)

template <typename T>
cudaError_t dalloc(T** p, size_t count) {
    *p = nullptr;
    if (count == 0) return cudaSuccess;
    cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
    if (e == cudaSuccess) e = cudaMemset(*p, 0, count * sizeof(T));
    return e;
}

// A[t][x] *= w[x]
__global__ void k_mask_cols(double* A, const double* w, int rows, int n) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)rows * n) return;
    int x = (int)(e % n);
    A[2 * e] *= w[x];
    A[2 * e + 1] *= w[x];
}

// A[e] *= W[e]  (A complex, W real, same shape): per-time flags
__global__ void k_mask_elem(double* A, const double* W, long long count) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= count) return;
    A[2 * e] *= W[e];
    A[2 * e + 1] *= W[e];
}
// out[t][x] = W[t][x] * v[x]
__global__ void k_rowscale(double* out, const double* W, const double* v, int rows, int n) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)rows * n) return;
    out[e] = W[e] * v[e % n];
}
// Bsel[x][0] = Bmat[x][0],  Bsel[x][1 + j] = Bmat[x][n + j]
__global__ void k_select_cols(double* Bsel, const double* Bmat, int n, int m, int Np) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)n * (1 + m)) return;
    int x = (int)(e / (1 + m)), j = (int)(e % (1 + m));
    size_t src = (size_t)x * Np + (j == 0 ? 0 : n + j - 1);
    Bsel[2 * e] = Bmat[2 * src];
    Bsel[2 * e + 1] = Bmat[2 * src + 1];
}
// dense Np x Np (interleaved complex, row-major) from the padded packed lower-block layout; zero above the diagonal blocks
__global__ void k_unpack_lower(const double* Wp, double* Wd, int nblk, size_t bsP) {
    const int Np = nblk * 32;
    const size_t sys = blockIdx.y;
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)Np * Np) return;
    const int i = (int)(e / Np), j = (int)(e % Np), bi = i >> 5, bj = j >> 5;
    double re = 0.0, im = 0.0;
    if (bj <= bi) {
        const double* blk = Wp + sys * bsP + hp::blk_index(bi, bj) * hp::kLBlkDoubles;
        re = blk[(i & 31) * hp::kLdBlk + (j & 31)];
        im = blk[hp::kLPlane + (i & 31) * hp::kLdBlk + (j & 31)];
    }
    double* o = Wd + 2 * (sys * (size_t)Np * Np + (size_t)e);
    o[0] = re; o[1] = im;
}
// r[t][row] = lam[row] Rfix[t][row] (+ wa[t][row], row < n); zero for padded times
__global__ void k_build_rhs(double* R, const double* Rfix, const double* wa, const double* lam, int n, int Np, int T, int Tp) {
    const size_t sys = blockIdx.y;
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)Tp * Np) return;
    const int t = (int)(e / Np), row = (int)(e % Np);
    const size_t off = 2 * (sys * (size_t)Tp * Np + (size_t)e);
    double vr = 0.0, vi = 0.0;
    if (t < T) {
        const double l = lam[sys * Np + row];
        vr = l * Rfix[off]; vi = l * Rfix[off + 1];
        if (wa && row < n) { vr += wa[off]; vi += wa[off + 1]; }
    }
    R[off] = vr; R[off + 1] = vi;
}
// y += xi, xi ~ CN(0, I): same Philox counter layout as k_solve
__global__ void k_add_noise(double* Y, int N, int Np, int T, int Tp, hp::DrawKey dk) {
    const size_t sys = blockIdx.y;
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)T * Np) return;
    const int t = (int)(e / Np), row = (int)(e % Np);
    if (row >= N) return;
    hp::u32x4 ctr; ctr.x = (uint32_t)row; ctr.y = (uint32_t)t; ctr.z = dk.iter; ctr.w = (uint32_t)__ldg(dk.chain_ids + sys);
    double n0, n1;
    hp::normal_pair_fast(hp::philox4x32_10(ctr, dk.key0, dk.key1 ^ 0xA5A5A5A5u), n0, n1);
    double* y = Y + 2 * (sys * (size_t)Tp * Np + (size_t)e);
    y[0] += n0 * 0.70710678118654752440; y[1] += n1 * 0.70710678118654752440;
}
// Ssc[t][k] = lam[k] X[t][k]  (k < n)
__global__ void k_make_ssc(double* Ssc, const double* X, const double* lam, int n, int Np, int T, int Tp) {
    const size_t sys = blockIdx.y;
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)T * n) return;
    const int t = (int)(e / n), k = (int)(e % n);
    const double l = lam[sys * Np + k];
    const double* x = X + 2 * ((sys * (size_t)Tp + t) * Np + k);
    double* o = Ssc + 2 * ((sys * (size_t)Tp + t) * n + k);
    o[0] = l * x[0]; o[1] = l * x[1];
}
__global__ void k_sqrt_vec(double* out, const double* in, int n) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = sqrt(in[k]);
}

// Bmat[x][k] (k < n) = conj(U[k][x])   (Q = U^H: delay eigenbasis of a stationary S)
__global__ void k_basis_fourier(double* Bmat, const double* U, int n, int Np) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)n * n) return;
    int x = (int)(e / n), k = (int)(e % n);
    Bmat[2 * ((size_t)x * Np + k)] = U[2 * ((size_t)k * n + x)];
    Bmat[2 * ((size_t)x * Np + k) + 1] = -U[2 * ((size_t)k * n + x) + 1];
}
// Bmat[x][k] = Q[x][k]
__global__ void k_basis_general(double* Bmat, const double* Q, int n, int Np) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)n * n) return;
    int x = (int)(e / n), k = (int)(e % n);
    Bmat[2 * ((size_t)x * Np + k)] = Q[2 * e];
    Bmat[2 * ((size_t)x * Np + k) + 1] = Q[2 * e + 1];
}
// Bmat[x][n + j] = F[x][j];  Ft[j][x] = F[x][j]
__global__ void k_basis_fg(double* Bmat, double* Ft, const double* F, int n, int m, int Np) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)n * m) return;
    int x = (int)(e / m), j = (int)(e % m);
    double fr = F[2 * e], fi = F[2 * e + 1];
    Bmat[2 * ((size_t)x * Np + n + j)] = fr;
    Bmat[2 * ((size_t)x * Np + n + j) + 1] = fi;
    if (Ft) { Ft[2 * ((size_t)j * n + x)] = fr; Ft[2 * ((size_t)j * n + x) + 1] = fi; }
}
// per-channel noise vectors:  ni = w * ninv,  nu = sqrt(ni)
__global__ void k_noise_vectors(const double* w, const double* ninv, double* ni, double* nu, int n) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n) return;
    double v = w[x] * ninv[x];
    ni[x] = v;
    nu[x] = sqrt(v);
}
// lam[k] = sqrt(lamsq[k]) (k<n), 1 (fg rows), 0 (padding);  ps[k] = n * lamsq[k]
__global__ void k_init_lam(double* lam, double* ps, const double* lamsq, int n, int N, int Np) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= Np) return;
    if (k < n) { lam[k] = sqrt(lamsq[k]); if (ps) ps[k] = (double)n * lamsq[k]; }
    else lam[k] = k < N ? 1.0 : 0.0;
}
__global__ void k_scale_vec(double* out, const double* in, double s, int n) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = in[k] * s;
}

// NiD[x][y] = w[x] w[y] Ninv[x][y]   (flags applied to rows and columns)
__global__ void k_mask_dense(double* NiD, const double* Ninv, const double* w, int n) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)n * n) return;
    int x = (int)(e / n), y = (int)(e % n);
    double s = w[x] * w[y];
    NiD[2 * e] = s * Ninv[2 * e];
    NiD[2 * e + 1] = s * Ninv[2 * e + 1];
}
// NiL = lower triangle of the Hermitian part of NiD with half its diagonal:  r^H Ni r = 2 Re(r^H NiL r)
__global__ void k_lower_half(double* NiL, const double* NiD, int n) {
    long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= (long long)n * n) return;
    int x = (int)(e / n), y = (int)(e % n);
    double re = 0.0, im = 0.0;
    if (y < x) {
        const long long f = (long long)y * n + x;
        re = 0.5 * (NiD[2 * e] + NiD[2 * f]);
        im = 0.5 * (NiD[2 * e + 1] - NiD[2 * f + 1]);
    } else if (y == x) {
        re = 0.5 * NiD[2 * e];
    }
    NiL[2 * e] = re; NiL[2 * e + 1] = im;
}
// out[t] = scale * Re sum_x conj(A[t][x]) B[t][x]
__global__ void k_rowdot(const double* A, const double* B, double* out, int T, int Tp, int n, double scale) {
    const int sys = blockIdx.y, t = blockIdx.x;
    const double* a = A + 2 * (((size_t)sys * Tp + t) * n);
    const double* b = B + 2 * (((size_t)sys * Tp + t) * n);
    double acc = 0.0;
    if (t < T)
        for (int x = threadIdx.x; x < n; x += blockDim.x) acc += a[2 * x] * b[2 * x] + a[2 * x + 1] * b[2 * x + 1];
    __shared__ double red[8];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s2 = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s2 += red[i];
        out[(size_t)sys * Tp + t] = scale * s2;
    }
}

inline unsigned nblocks(long long tot, int bs = 256) { return (unsigned)((tot + bs - 1) / bs); }

struct Basis {
    double* Bmat = nullptr;  // [C][n][Np]
    double* Gp = nullptr;    // [C][tri][2048]
    double* Rfix = nullptr;  // [C][Tp][Np]
    double* wa = nullptr;    // [C][Tp][Np]   injected mode: Q^H omega_a
    double* Rt = nullptr;    // [C][ntiles][nblk][2][32][16]  right-hand sides in k_solve3's tile layout (k_rhs_tile)
};

enum { CLS_CHOL = 0, CLS_SOLVE = 1, CLS_TRANSFORM = 2, CLS_POST = 3, CLS_SAMPLE = 4, CLS_LOWRANK = 5 };

// The paths an engine takes through the solve and the post-processing, chosen once by select_paths (DESIGN.md section 3)
enum class Solve { Solve3, Resident, Dense, PtLowRank, PtDirect };
enum class Post { Fft2, Fft, Dense };

}  // namespace

struct hp_engine {
    hp_config cfg;
    int C, T, n, m, N, nblk, Np, Tp, ntiles;
    cudaStream_t st = nullptr;
    cudaStream_t copy_st = nullptr;  // device-to-host streaming of the per-iteration outputs
    std::vector<cudaStream_t> sub_st;   // cfg.substreams > 1: one stream per sub-batch of chains
    cudaEvent_t fork_ev = nullptr;
    int active_subs = 1 << 30;          // runtime limit on the number of sub-batches (hp_engine_set_substreams)
    std::vector<cudaEvent_t> join_ev;
    bool own_stream = false;
    double *Fop = nullptr, *U = nullptr;
    Basis bF, b0;
    double *lam = nullptr, *ps = nullptr;
    double *wd = nullptr, *w = nullptr, *ninvd = nullptr, *ni = nullptr, *nu = nullptr, *Ft = nullptr, *prior = nullptr;
    double *Lp = nullptr, *Linvp = nullptr, *Wp = nullptr;
    double *wT = nullptr, *Hpt = nullptr, *niT = nullptr, *Bsel = nullptr, *ptScratch = nullptr;  // per-time flags
    int* ptSame = nullptr;   // [C][Tp]: flags of time t equal those of t - 1
    int pt_ctas = 0;
    Solve solve = Solve::Solve3;
    Post post = Post::Fft2;
    int ppart_tiles = 1;     // partial sums of beta per chain that the solve leaves in Ppart (k_sample adds them)
    bool uses_solve3() const { return solve == Solve::Solve3 || solve == Solve::PtLowRank; }
    // per-time flags in low-rank form (hp_ptlow.cu): the shared system of the channels unflagged at any time goes through
    // chol / trinv / k_solve3 with n extra right-hand sides (rows Tp0 .. of Rfix / X), k_pt_lowrank corrects every time
    int Tp0 = 0;             // padded number of times; Tp = Tp0 + padded Nfreqs when the engine was created as PtLowRank
    bool lowrank_rows() const { return Tp != Tp0; }   // the extra right-hand sides of the low-rank form exist
    int pt_kcap = 0;         // largest number of extra flagged channels of any loaded (chain, time)
    double* Pm = nullptr;    // [C][n][n] complex
    uint16_t* ptFidx = nullptr;   // [C][T][kPtLowMaxRank]
    int* ptFcnt = nullptr;   // [C][T]
    std::vector<int> pt_kmax;     // per chain: largest extra-flag count
    std::vector<uint8_t> hpt_built;   // per chain: the operands of k_pt_cholsolve (Hpt) are current
    std::vector<uint8_t> pt_loaded;   // per chain: loaded with per-time flags
    int gd_slots = 1;
    std::vector<uint8_t> pending;         // chains whose G / Rfix products are still to be built (flush_pending)
    double *Wf1 = nullptr, *Wf2 = nullptr;   // fragment-major W for k_solve3 (k_chol_w writes them)
    hp::Solve3Sched sched3{};
    double *Wd = nullptr, *Yb = nullptr;
    double *NiL = nullptr;   // dense noise: lower half of the Hermitian part of NiD (ln_post term as a triangular product)
    double *NiD = nullptr, *NihD = nullptr, *Td = nullptr, *Rm = nullptr, *Yd = nullptr;  // dense (non-diagonal) noise
    int* info = nullptr;
    int* chain_ids = nullptr;   // [C] Philox chain id of every chain (default: its index; hp_engine_set_chain_ids)
    double *X = nullptr, *Ssc = nullptr, *Ppart = nullptr, *Sf = nullptr, *Wm = nullptr, *Tmp = nullptr;
    double *Em = nullptr, *Eu = nullptr, *lnp1 = nullptr;
    double* sdraws = nullptr;
    double *ps_out = nullptr, *lnpost_out = nullptr, *cr_out = nullptr, *fg_out = nullptr, *chisq_out = nullptr;
    double *Gd = nullptr, *stage = nullptr, *vecn = nullptr;  // set-up scratch
    void* arena = nullptr;   // one device allocation holds every buffer below
    size_t arena_bytes = 0;
    hp::FftPlan plan{};
    int ntilesE = 0, ktp = 8;
    double *tw = nullptr, *tw2 = nullptr, *Empart = nullptr, *Eupart = nullptr;
    std::vector<uint8_t> flagged;  // per chain: any channel flagged
    bool any_omega = false;   // injected omega draws were set for some chain (hp_engine_set_draws)
    bool any_flagged = false;
    int ring = 1;     // device slots of the big per-iteration outputs (cfg.ring_iters, or max_iters)
    std::vector<cudaEvent_t> copy_done;   // run_to_host: the device-to-host copies out of ring slot s have completed
    std::vector<cudaEvent_t> sub_done;    // run_to_host: sub-batch i has finished the iteration being copied
    int iter = 0;     // Gibbs iterations since the chains were loaded (RNG counter, basis choice)
    int out_pos = 0;  // cursor in the per-iteration output buffers
    int ahead = 0;    // iterations computed beyond out_pos by hp_engine_run_to_host (sink.read_ahead), not yet delivered
    std::vector<cudaEvent_t> it_done;   // run_to_host: [ring slot][sub-batch] the iteration in that slot has been computed
    uint32_t draw_counter = 0;  // Philox counter of the GCR fluctuation draws (advances per GCR step)
    const double* last_sf = nullptr;  // where the last GCR solve's frequency-space signal lives
    long long last_sf_bs = 0;         // its batch stride (complex elements)
    long long launches = 0;
    // posterior moments (hp_engine_set_summary): own allocations, made when first asked for, so that an engine without the
    // summary pays nothing for it.  Accumulators [C][ld] with ld = T * n (T * m) rounded up to even (k_moments' pairs).
    // Batch means (batch > 0, hp_engine_set_summary_batched): snap (complex) and M2_bm (real) in the same layout, allocated
    // the first time batch means are asked for.
    struct Summary {
        int what = 0, burn_in = 0, thin = 1, batch = 0;
        long long seen = 0;   // iterations computed since the summary was (re)started
        int count = 0;        // iterations accumulated
        long long ld_cr = 0, ld_fg = 0;
        double *cr_mean = nullptr, *cr_m2 = nullptr, *fg_mean = nullptr, *fg_m2 = nullptr;
        double *cr_snap = nullptr, *cr_m2bm = nullptr, *fg_snap = nullptr, *fg_m2bm = nullptr;
    } sum;
    // profiling
    std::vector<cudaEvent_t> ev;
    std::vector<int> ev_cls;
    double ms_acc[HP_NUM_KERNEL_CLASSES] = {0};
    int launch_acc[HP_NUM_KERNEL_CLASSES] = {0};

    void prof_begin(int cls, cudaStream_t s) {
        if (!cfg.profile || ev_cls.size() >= 8192) return;
        cudaEvent_t a, b;
        cudaEventCreate(&a); cudaEventCreate(&b);
        cudaEventRecord(a, s);
        ev.push_back(a); ev.push_back(b); ev_cls.push_back(cls);
    }
    void prof_end(int cls, int nlaunch, cudaStream_t s) {
        launches += nlaunch;
        launch_acc[cls] += nlaunch;
        if (!cfg.profile || ev_cls.empty() || ev_cls.back() != cls) return;
        cudaEventRecord(ev.back(), s);
    }
};

namespace {
// One cached device arena per GPU.  The drop-in functions create and destroy an engine per call (the reference's
// driver calls gibbs_sample_with_fg once per baseline), and cudaMalloc / cudaFree of a multi-GB arena cost
// milliseconds to tens of milliseconds each: the arena of a destroyed engine is kept and handed to the next engine
// on that device if it is large enough.  hp_release_cached_memory() frees it; HP_NO_ARENA_CACHE=1 disables it.
constexpr int kMaxDevices = 64;
struct CachedArena { void* p = nullptr; size_t bytes = 0; };
CachedArena g_arena_cache[kMaxDevices];
std::mutex g_arena_mutex;
bool arena_cache_enabled() {
    static int on = -1;
    if (on < 0) { const char* e = getenv("HP_NO_ARENA_CACHE"); on = (e && e[0] == '1') ? 0 : 1; }
    return on == 1;
}
cudaError_t arena_acquire(void** base, size_t* bytes, int device) {
    if (arena_cache_enabled() && device >= 0 && device < kMaxDevices) {
        std::lock_guard<std::mutex> lk(g_arena_mutex);
        CachedArena& c = g_arena_cache[device];
        if (c.p && c.bytes >= *bytes) { *base = c.p; *bytes = c.bytes; c.p = nullptr; c.bytes = 0; return cudaSuccess; }
        if (c.p) { cudaFree(c.p); c.p = nullptr; c.bytes = 0; }   // too small: make room before the larger allocation
    }
    return cudaMalloc(base, *bytes);
}
void arena_release(void* p, size_t bytes, int device) {
    if (!p) return;
    if (arena_cache_enabled() && device >= 0 && device < kMaxDevices) {
        std::lock_guard<std::mutex> lk(g_arena_mutex);
        CachedArena& c = g_arena_cache[device];
        if (!c.p || c.bytes < bytes) {
            if (c.p) cudaFree(c.p);
            c.p = p; c.bytes = bytes;
            return;
        }
    }
    cudaFree(p);
}

// Collects buffer requests, then serves them all from one cudaMalloc (engine creation / teardown is
// part of the end-to-end path: one allocation and one free instead of ~45).
struct ArenaPlan {
    struct Req { void** p; size_t bytes; };
    std::vector<Req> reqs;
    template <typename T>
    void want(T** p, size_t count) { *p = nullptr; if (count) reqs.push_back({reinterpret_cast<void**>(p), count * sizeof(T)}); }
    cudaError_t commit(void** base, size_t* bytes_out, int device, cudaStream_t st) {
        size_t total = 0;
        for (auto& r : reqs) total += (r.bytes + 255) & ~size_t(255);
        if (!total) total = 256;
        *bytes_out = total;
        cudaError_t e = arena_acquire(base, bytes_out, device);
        if (e != cudaSuccess) return e;
        e = cudaMemsetAsync(*base, 0, total, st);
        if (e != cudaSuccess) return e;
        size_t off = 0;
        for (auto& r : reqs) { *r.p = static_cast<char*>(*base) + off; off += (r.bytes + 255) & ~size_t(255); }
        return cudaSuccess;
    }
};

void want_basis(hp_engine* e, ArenaPlan& ap, Basis& b) {
    size_t C = e->C;
    ap.want(&b.Bmat, 2 * C * e->n * e->Np);
    ap.want(&b.Gp, C * hp::tri_blocks(e->nblk) * hp::kBlkDoubles);
    ap.want(&b.Rfix, 2 * C * e->Tp * e->Np);
    if (e->cfg.rng_mode == HP_RNG_INJECTED) ap.want(&b.wa, 2 * C * e->Tp * e->Np);
    if (e->uses_solve3()) ap.want(&b.Rt, 2 * C * e->Tp * e->Np);
}

// Chooses the engine's solve and post-processing paths from its configuration and the device's shared memory, and what
// follows from them: the padded times of the low-rank form, k_solve3's schedule, the granularity of the beta partial sums
// and the FFT tiling.  Refuses the per-time-flag configurations that no path takes.
int select_paths(hp_engine* e, size_t max_smem) {
    const hp_config& cfg = e->cfg;
    e->ktp = hp::postfft_ktp(e->n, e->m, max_smem);
    if (!hp::make_fft_plan(e->n, &e->plan) || e->ktp == 0 || cfg.force_dense_transforms) {
        e->post = Post::Dense;
    } else if (hp::postfft2_ok(e->n) &&
               hp::postfft2_smem_bytes(e->n, e->m) <= max_smem / (e->n >= 512 ? 1 : 2)) {   // one CTA per SM from 512 channels on
        e->post = Post::Fft2;
        e->ktp = 8;   // k_post_fft2 handles eight times per CTA
    } else {
        e->post = Post::Fft;
    }
    e->ntilesE = hp::postfft_tiles(e->T, e->ktp > 0 ? e->ktp : 8);
    const bool s3 = hp::solve3_ok(e->nblk, max_smem);
    if (cfg.time_flags) {
        // low-rank form on top of k_solve3 unless HP_PT_DIRECT=1 (A/B runs, tests of k_pt_cholsolve)
        const char* pd = getenv("HP_PT_DIRECT");
        const bool low = !(pd && pd[0] == '1') && !cfg.force_dense_solve && s3 && e->n < 65536;
        e->solve = low ? Solve::PtLowRank : Solve::PtDirect;
        // a general (non-delay-diagonal) S_initial is possible in the low-rank form only: k_pt_cholsolve relies on the
        // circulant signal block of the delay basis
        if (cfg.dense_noise || cfg.cg_compat || cfg.force_dense_transforms || (cfg.general_basis0 && !low))
            return fail(HP_ERR_ARG, "per-time flags need diagonal noise, the exact solver and an FFT-able Nfreqs (and a delay-diagonal "
                                    "S_initial unless Nfreqs + Nmodes <= 448)");
        if (hp::pt_smem_bytes(e->nblk, e->n) > max_smem || e->post == Post::Dense)
            return fail(HP_ERR_SIZE, "per-time flags: Nfreqs too large for the shared-memory working set, or without an FFT plan");
    } else if (cfg.force_dense_solve || !hp::solve_resident_ok(e->nblk, max_smem)) {
        e->solve = Solve::Dense;
    } else {
        e->solve = s3 ? Solve::Solve3 : Solve::Resident;
    }
    if (e->solve == Solve::PtLowRank) {
        e->Tp += hp::kTT * ((e->n + hp::kTT - 1) / hp::kTT);
        e->ntiles = e->Tp / hp::kTT;
    }
    if (e->uses_solve3()) hp::solve3_make_schedule(e->nblk, &e->sched3, (e->N + 15) / 16);
    // k_solve and k_solve3 leave one partial sum per 16-time tile; the other paths, and k_solve3 followed by the reference-CG
    // scaling, one per chain (k_colsumsq)
    e->ppart_tiles = (e->solve == Solve::Resident || (e->solve == Solve::Solve3 && !cfg.cg_compat)) ? e->ntiles : 1;
    return HP_OK;
}
}  // namespace

static const char* kAheadMsg = "read-ahead iterations are pending (hp_host_sink.read_ahead): deliver them with hp_engine_run_to_host or "
                               "drop them with hp_engine_rewind first";

extern "C" {

const char* hp_last_error(void) { return g_err.c_str(); }
const char* hp_version(void) { return "hydra_pspec_b200 0.1 (sm_100a)"; }
void hp_release_cached_memory(void) {
    std::lock_guard<std::mutex> lk(g_arena_mutex);
    int cur = 0;
    cudaGetDevice(&cur);
    for (int d = 0; d < kMaxDevices; ++d)
        if (g_arena_cache[d].p) {
            cudaSetDevice(d);
            cudaFree(g_arena_cache[d].p);
            g_arena_cache[d] = CachedArena();
        }
    cudaSetDevice(cur);
}
const char* hp_kernel_class_name(int cls) {
    static const char* names[HP_NUM_KERNEL_CLASSES] = {"chol", "solve", "transform", "post", "sample", "lowrank"};
    return (cls >= 0 && cls < HP_NUM_KERNEL_CLASSES) ? names[cls] : "?";
}

int hp_engine_destroy(hp_engine* e) {
    if (!e) return HP_OK;
    cudaSetDevice(e->cfg.device);
    if (e->st) cudaStreamSynchronize(e->st);
    for (auto& x : e->ev) cudaEventDestroy(x);
    arena_release(e->arena, e->arena_bytes, e->cfg.device);
    for (double* p : {e->sum.cr_mean, e->sum.cr_m2, e->sum.fg_mean, e->sum.fg_m2, e->sum.cr_snap, e->sum.cr_m2bm, e->sum.fg_snap,
                      e->sum.fg_m2bm}) if (p) cudaFree(p);
    if (e->copy_st) cudaStreamDestroy(e->copy_st);
    for (auto x : e->sub_st) cudaStreamDestroy(x);
    if (e->fork_ev) cudaEventDestroy(e->fork_ev);
    for (auto x : e->join_ev) cudaEventDestroy(x);
    for (auto x : e->copy_done) cudaEventDestroy(x);
    for (auto x : e->it_done) cudaEventDestroy(x);
    for (auto x : e->sub_done) cudaEventDestroy(x);
    if (e->own_stream) cudaStreamDestroy(e->st);
    delete e;
    return HP_OK;
}

int hp_engine_create(const hp_config* cfg, hp_engine** out) {
    if (!cfg || !out) return fail(HP_ERR_ARG, "null argument");
    if (cfg->nchains < 1 || cfg->ntimes < 2 || cfg->nfreqs < 2 || cfg->nmodes < 0 || cfg->max_iters < 1)
        return fail(HP_ERR_ARG, "hp_engine_create: bad dimensions");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(HP_ERR_CUDA, "no CUDA device: hydra_pspec_b200 has no CPU fallback");
    CU_TRY(cudaSetDevice(cfg->device));
    hp_engine* e = new hp_engine();
    e->cfg = *cfg;
    e->C = cfg->nchains; e->T = cfg->ntimes; e->n = cfg->nfreqs; e->m = cfg->nmodes;
    e->N = e->n + e->m;
    e->nblk = (e->N + hp::kNB - 1) / hp::kNB;
    e->Np = e->nblk * hp::kNB;
    e->ntiles = (e->T + hp::kTT - 1) / hp::kTT;
    e->Tp = e->ntiles * hp::kTT;
    e->Tp0 = e->Tp;
    int max_smem = 0;
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device);
    if (const int rc = select_paths(e, (size_t)max_smem)) {
        delete e;
        return rc;
    }
    if (cfg->stream) e->st = (cudaStream_t)cfg->stream;
    else { CU_TRY(cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking)); e->own_stream = true; }
    const size_t C = e->C, n = e->n, m = e->m, Np = e->Np, Tp = e->Tp, T = e->T, I = cfg->max_iters;
    e->ring = (cfg->ring_iters > 0 && cfg->ring_iters < cfg->max_iters) ? cfg->ring_iters : cfg->max_iters;
    const size_t R = e->ring;
    const bool dense = e->post == Post::Dense;           // dense-transform scratch
    const bool need_ssc = dense || cfg->general_basis0;  // lam * ytilde as input of the dense back-transform
    ArenaPlan ap;
    ap.want(&e->Fop, 2 * n * n); ap.want(&e->U, 2 * n * n);
    want_basis(e, ap, e->bF);
    if (cfg->general_basis0) want_basis(e, ap, e->b0);
    ap.want(&e->lam, C * Np); ap.want(&e->ps, C * n);
    ap.want(&e->wd, 2 * C * Tp * n); ap.want(&e->w, C * n); ap.want(&e->ninvd, C * n);
    ap.want(&e->ni, C * n); ap.want(&e->nu, C * n); ap.want(&e->Ft, 2 * C * (m ? m : 1) * n);
    ap.want(&e->prior, C * 2 * n);
    ap.want(&e->Lp, C * hp::tri_blocks(e->nblk) * hp::kLBlkDoubles);
    ap.want(&e->Linvp, C * e->nblk * hp::kLBlkDoubles);
    ap.want(&e->Wp, C * hp::tri_blocks(e->nblk) * hp::kLBlkDoubles);
    if (e->uses_solve3()) { ap.want(&e->Wf1, C * hp::solve3_frag_doubles(e->nblk)); ap.want(&e->Wf2, C * hp::solve3_frag_doubles(e->nblk)); }
    ap.want(&e->info, C);
    ap.want(&e->chain_ids, C);
    ap.want(&e->X, 2 * C * Tp * Np);
    if (need_ssc) ap.want(&e->Ssc, 2 * C * Tp * n);   // (dense transforms / general first basis)
    ap.want(&e->Ppart, C * e->ntiles * n); ap.want(&e->Sf, 2 * C * Tp * n);
    if (dense) { ap.want(&e->Wm, 2 * C * Tp * n); ap.want(&e->Tmp, 2 * C * Tp * n); ap.want(&e->Em, C * n); ap.want(&e->Eu, C * n); }
    ap.want(&e->lnp1, C * Tp);
    if (e->solve == Solve::Dense) { ap.want(&e->Wd, 2 * C * Np * Np); ap.want(&e->Yb, 2 * C * Tp * Np); }
    if (cfg->time_flags) {
        e->pt_ctas = hp::pt_grid(e->C, e->T);
        ap.want(&e->wT, C * Tp * n);
        ap.want(&e->ptSame, C * Tp);
        ap.want(&e->Hpt, 2 * C * Tp * (1 + m) * Np);
        ap.want(&e->niT, Tp * n);
        ap.want(&e->Bsel, 2 * n * (1 + m));
        ap.want(&e->ptScratch, (size_t)e->pt_ctas * hp::pt_scratch_doubles_per_cta(e->nblk));
        if (e->solve == Solve::PtLowRank) {
            ap.want(&e->Pm, 2 * C * n * n);
            ap.want(&e->ptFidx, C * T * hp::kPtLowMaxRank);
            ap.want(&e->ptFcnt, C * T);
        }
    }
    if (cfg->dense_noise) {
        ap.want(&e->NiD, 2 * C * n * n);
        ap.want(&e->NiL, 2 * C * n * n);
        if (cfg->rng_mode == HP_RNG_INJECTED) ap.want(&e->NihD, 2 * C * n * n);
        ap.want(&e->Td, 2 * n * Np); ap.want(&e->Rm, 2 * C * Tp * n); ap.want(&e->Yd, 2 * C * Tp * n);
    }
    if (cfg->rng_mode != HP_RNG_PHILOX) ap.want(&e->sdraws, C * I * n);
    ap.want(&e->ps_out, C * I * n); ap.want(&e->lnpost_out, C * I);
    if (cfg->keep & HP_KEEP_CR) ap.want(&e->cr_out, 2 * C * R * T * n);
    if (cfg->keep & HP_KEEP_FG) ap.want(&e->fg_out, 2 * C * R * T * (m ? m : 1));
    if (cfg->keep & HP_KEEP_CHISQ) ap.want(&e->chisq_out, C * R * T * n);
    e->gd_slots = (int)(C < 16 ? C : 16);   // dense Gram scratch for a batch of chains (deferred set-up)
    ap.want(&e->Gd, 2 * (size_t)e->gd_slots * e->N * e->N);
    ap.want(&e->stage, 2 * (T * n > n * n ? T * n : n * n));
    ap.want(&e->vecn, 4 * n);
    ap.want(&e->tw, 2 * n);
    if (e->post == Post::Fft2) ap.want(&e->tw2, 4 * n);
    ap.want(&e->Empart, C * e->ntilesE * n); ap.want(&e->Eupart, C * e->ntilesE * n);
    {
        cudaError_t ce = ap.commit(&e->arena, &e->arena_bytes, cfg->device, e->st);
        if (ce != cudaSuccess) {
            std::string msg = std::string("device allocation failed: ") + cudaGetErrorString(ce);
            hp_engine_destroy(e);
            return fail(HP_ERR_CUDA, msg);
        }
    }
    e->flagged.assign(C, 0);
    e->pt_kmax.assign(C, 0);
    e->hpt_built.assign(C, 0);
    e->pt_loaded.assign(C, 0);
    e->pending.assign(C, 0);
    {
        int ns = cfg->substreams > 1 ? (cfg->substreams < (int)C ? cfg->substreams : (int)C) : 1;
        if (ns > 1) {
            for (int i = 0; i < ns; ++i) {
                cudaStream_t x; cudaEvent_t ev;
                cudaStreamCreateWithFlags(&x, cudaStreamNonBlocking); e->sub_st.push_back(x);
                cudaEventCreateWithFlags(&ev, cudaEventDisableTiming); e->join_ev.push_back(ev);
            }
            cudaEventCreateWithFlags(&e->fork_ev, cudaEventDisableTiming);
        }
    }
    {
        std::vector<int> ids(C);
        for (size_t c = 0; c < C; ++c) ids[c] = (int)c;
        cudaMemcpyAsync(e->chain_ids, ids.data(), C * sizeof(int), cudaMemcpyHostToDevice, e->st);   // pageable: staged before return
    }
    hp::launch_fourier_operator(e->Fop, e->n, 1.0, e->st);
    hp::launch_fourier_operator(e->U, e->n, 1.0 / std::sqrt((double)e->n), e->st);
    hp::launch_twiddles(e->tw, e->n, e->st);
    if (e->post == Post::Fft2) hp::launch_fft2_tables(e->tw2, e->tw, e->n, e->st);
    if (cudaStreamSynchronize(e->st) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
        hp_engine_destroy(e);
        return fail(HP_ERR_CUDA, "engine initialisation kernels failed");
    }
    *out = e;
    return HP_OK;
}

// Per-time flags, one factorisation per time (hp_pertime.cu): H_t = [Q|F]^H (w_t N^-1) [q_0 | F] for every time of chain c --
// column 0 is the generator chat_t of the circulant signal block, the rest are the foreground columns of G_t.  Built from what
// load_chain left on the device (Bmat, wT, ninvd), so it can be deferred until the direct form is actually needed.
static int build_hpt(hp_engine* e, int c) {
    const int n = e->n, m = e->m, N = e->N, Np = e->Np, T = e->T;
    const double* Bm = e->bF.Bmat + 2 * (size_t)c * n * Np;
    k_rowscale<<<nblocks((long long)T * n), 256, 0, e->st>>>(e->niT, e->wT + (size_t)c * e->Tp * n, e->ninvd + (size_t)c * n, T, n);
    k_select_cols<<<nblocks((long long)n * (1 + m)), 256, 0, e->st>>>(e->Bsel, Bm, n, m, Np);
    hp::ZgemmArgs h{};
    h.A = Bm; h.sAi = 1; h.sAk = Np; h.bsA = 0; h.conjA = 1;
    h.B = e->Bsel; h.sBk = 1 + m; h.sBj = 1; h.bsB = 0;
    h.C = e->Hpt + 2 * (size_t)c * e->Tp * (1 + m) * Np; h.sCi = 1; h.sCj = Np; h.bsC = (long long)(1 + m) * Np;
    h.dk = e->niT; h.bsD = n;
    h.M = N; h.N = 1 + m; h.K = n; h.accumulate = 0; h.alpha = 1.0; h.batch = T;
    hp::launch_zgemm(h, e->st);
    CU_TRY(cudaGetLastError());
    e->hpt_built[c] = 1;
    return HP_OK;
}

// G = B^H Ni B (packed), Rfix = B^H Ni (w d)^T  for chain c in basis b; Ni diagonal or dense
static int build_basis_products(hp_engine* e, Basis& b, int c) {
    const int n = e->n, N = e->N, Np = e->Np, T = e->T;
    double* Bm = b.Bmat + 2 * (size_t)c * n * Np;
    const bool dn = e->cfg.dense_noise != 0;
    const double* NiD = dn ? e->NiD + 2 * (size_t)c * n * n : nullptr;
    hp::ZgemmArgs g{};
    g.A = Bm; g.sAi = 1; g.sAk = Np; g.bsA = 0; g.conjA = 1;
    g.C = e->Gd; g.sCi = N; g.sCj = 1; g.bsC = 0;
    g.M = N; g.N = N; g.K = n; g.accumulate = 0; g.alpha = 1.0; g.batch = 1;
    if (dn) {
        hp::ZgemmArgs t1{};   // Td = Ni B
        t1.A = NiD; t1.sAi = n; t1.sAk = 1;
        t1.B = Bm; t1.sBk = Np; t1.sBj = 1;
        t1.C = e->Td; t1.sCi = Np; t1.sCj = 1;
        t1.M = n; t1.N = N; t1.K = n; t1.alpha = 1.0; t1.batch = 1;
        hp::launch_zgemm(t1, e->st);
        g.B = e->Td; g.sBk = Np; g.sBj = 1;
    } else {
        g.B = Bm; g.sBk = Np; g.sBj = 1; g.bsB = 0; g.conjB = 0;
        g.dk = e->ni + (size_t)c * n; g.bsD = 0;
    }
    hp::launch_zgemm(g, e->st);
    hp::launch_pack_lower(e->Gd, N, 0, b.Gp + (size_t)c * hp::tri_blocks(e->nblk) * hp::kBlkDoubles, N, e->nblk, 1, e->st);
    hp::ZgemmArgs r{};
    r.B = Bm; r.sBk = Np; r.sBj = 1; r.conjB = 1;
    r.C = b.Rfix + 2 * (size_t)c * e->Tp * Np; r.sCi = Np; r.sCj = 1;
    r.M = T; r.N = N; r.K = n; r.accumulate = 0; r.alpha = 1.0; r.batch = 1;
    if (dn) {
        hp::ZgemmArgs y{};    // Yd = (w d) Ni^T
        y.A = e->wd + 2 * (size_t)c * e->Tp * n; y.sAi = n; y.sAk = 1;
        y.B = NiD; y.sBk = 1; y.sBj = n;
        y.C = e->Yd + 2 * (size_t)c * e->Tp * n; y.sCi = n; y.sCj = 1;
        y.M = T; y.N = n; y.K = n; y.alpha = 1.0; y.batch = 1;
        hp::launch_zgemm(y, e->st);
        r.A = e->Yd + 2 * (size_t)c * e->Tp * n; r.sAi = n; r.sAk = 1;
    } else {
        r.A = e->wd + 2 * (size_t)c * e->Tp * n; r.sAi = n; r.sAk = 1; r.conjA = 0;
        // wd is already masked and w^2 = w: per-time flags use the unmasked diagonal
        r.dk = e->cfg.time_flags ? e->ninvd + (size_t)c * n : e->ni + (size_t)c * n;
    }
    hp::launch_zgemm(r, e->st);
    // low-rank form of per-time flags: the columns of A = D B^H sqrt(wbar N^-1) are n more right-hand sides (rows Tp0 + x)
    if (e->lowrank_rows()) hp::launch_pt_arows(b.Rfix + 2 * (size_t)c * e->Tp * Np, Bm, e->ni + (size_t)c * n, n, Np, e->Tp0, e->st);
    if (b.Rt && e->cfg.rng_mode == HP_RNG_PHILOX)
        hp::launch_rhs_tile(b.Rt + 2 * (size_t)c * e->Tp * Np, b.Rfix + 2 * (size_t)c * e->Tp * Np, nullptr, nullptr, e->nblk, e->n, e->N,
                            e->lowrank_rows() ? e->Tp : e->T, e->Tp, e->ntiles, 1, e->st);
    // the operands of k_pt_cholsolve are built only when the engine runs (or falls back to) one factorisation per time
    if (e->cfg.time_flags && &b == &e->bF) {
        e->hpt_built[c] = 0;
        if (e->solve == Solve::PtDirect) { const int rc = build_hpt(e, c); if (rc != HP_OK) return rc; }
    }
    CU_TRY(cudaGetLastError());
    return HP_OK;
}

// The same products for `nc` consecutive chains at once (diagonal noise, time-invariant flags): one batched launch
// fills the GPU where a single chain's 416 x 416 Gram product occupies a third of it.  Chain loading defers its
// products to the first call that needs them (flush_pending), so a batch of load_chain calls costs one set of launches.
static int build_basis_products_batch(hp_engine* e, Basis& b, int c0, int nc) {
    const int n = e->n, N = e->N, Np = e->Np, T = e->T;
    const size_t tri = hp::tri_blocks(e->nblk);
    for (int cc0 = c0; cc0 < c0 + nc; cc0 += e->gd_slots) {
        const int ncc = (c0 + nc - cc0) < e->gd_slots ? (c0 + nc - cc0) : e->gd_slots;
        double* Bm = b.Bmat + 2 * (size_t)cc0 * n * Np;
        hp::ZgemmArgs g{};
        g.A = Bm; g.sAi = 1; g.sAk = Np; g.bsA = (long long)n * Np; g.conjA = 1;
        g.B = Bm; g.sBk = Np; g.sBj = 1; g.bsB = (long long)n * Np;
        g.dk = e->ni + (size_t)cc0 * n; g.bsD = n;
        g.C = e->Gd; g.sCi = N; g.sCj = 1; g.bsC = (long long)N * N;
        g.M = N; g.N = N; g.K = n; g.accumulate = 0; g.alpha = 1.0; g.batch = ncc;
        hp::launch_zgemm(g, e->st);
        hp::launch_pack_lower(e->Gd, N, (long long)N * N, b.Gp + (size_t)cc0 * tri * hp::kBlkDoubles, N, e->nblk, ncc, e->st);
        hp::ZgemmArgs r{};
        r.A = e->wd + 2 * (size_t)cc0 * e->Tp * n; r.sAi = n; r.sAk = 1; r.bsA = (long long)e->Tp * n;
        r.dk = e->ni + (size_t)cc0 * n; r.bsD = n;
        r.B = Bm; r.sBk = Np; r.sBj = 1; r.bsB = (long long)n * Np; r.conjB = 1;
        r.C = b.Rfix + 2 * (size_t)cc0 * e->Tp * Np; r.sCi = Np; r.sCj = 1; r.bsC = (long long)e->Tp * Np;
        r.M = T; r.N = N; r.K = n; r.accumulate = 0; r.alpha = 1.0; r.batch = ncc;
        hp::launch_zgemm(r, e->st);
        if (b.Rt && e->cfg.rng_mode == HP_RNG_PHILOX)
            hp::launch_rhs_tile(b.Rt + 2 * (size_t)cc0 * e->Tp * Np, b.Rfix + 2 * (size_t)cc0 * e->Tp * Np, nullptr, nullptr, e->nblk,
                                e->n, e->N, e->T, e->Tp, e->ntiles, ncc, e->st);
    }
    CU_TRY(cudaGetLastError());
    return HP_OK;
}

static int flush_pending(hp_engine* e) {
    const int C = e->C;
    if (e->solve == Solve::PtDirect)   // fell back to one factorisation per time after some chains were loaded
        for (int c = 0; c < C; ++c)
            if (e->pt_loaded[c] && !e->hpt_built[c]) { const int rc = build_hpt(e, c); if (rc != HP_OK) return rc; }
    for (int c = 0; c < C;) {
        if (!e->pending[c]) { ++c; continue; }
        int c1 = c;
        while (c1 < C && e->pending[c1]) ++c1;
        int rc;
        if ((rc = build_basis_products_batch(e, e->bF, c, c1 - c)) != HP_OK) return rc;
        if (e->cfg.general_basis0 && (rc = build_basis_products_batch(e, e->b0, c, c1 - c)) != HP_OK) return rc;
        for (int k = c; k < c1; ++k) e->pending[k] = 0;
        c = c1;
    }
    return HP_OK;
}

static int load_chain_impl(hp_engine* e, int c, const double* vis, const uint8_t* flags, const double* fgmodes,
                           const double* ninv_diag, const double* ninv_dense, const double* nih_dense, const double* basis0,
                           const double* lam0sq, const double* ps_prior) {
    if (!e || !vis || !flags || !ninv_diag || !lam0sq || (e->m > 0 && !fgmodes))
        return fail(HP_ERR_ARG, "hp_engine_load_chain: null argument");
    if ((e->cfg.dense_noise != 0) != (ninv_dense != nullptr))
        return fail(HP_ERR_ARG, "hp_engine_load_chain: dense noise needs cfg.dense_noise and hp_engine_load_chain_dense");
    if (c < 0 || c >= e->C) return fail(HP_ERR_ARG, "hp_engine_load_chain: chain index out of range");
    if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);
    if (e->cfg.general_basis0 && !basis0) return fail(HP_ERR_ARG, "hp_engine_load_chain: general_basis0 set but basis0 is NULL");
    CU_TRY(cudaSetDevice(e->cfg.device));
    const int n = e->n, m = e->m, N = e->N, Np = e->Np, T = e->T, Tp = e->Tp;
    cudaStream_t st = e->st;
    const bool pt = e->cfg.time_flags != 0;   // flags: [Ntimes][Nfreqs]
    std::vector<double> wv(n);
    std::vector<double> wtv(pt ? (size_t)T * n : 0);
    bool anyf = false;
    if (pt) {
        for (size_t i = 0; i < (size_t)T * n; ++i) { wtv[i] = flags[i] ? 1.0 : 0.0; }
        // wbar: channels unflagged at any time (the shared system of the low-rank form; unused by k_pt_cholsolve)
        for (int x = 0; x < n; ++x) wv[x] = 0.0;
        for (int t = 0; t < T; ++t)
            for (int x = 0; x < n; ++x) if (flags[(size_t)t * n + x]) wv[x] = 1.0;
        anyf = true;  // the masked-signal term of ln_post is always evaluated with the per-time mask
        e->pt_loaded[c] = 1;
    } else {
        for (int x = 0; x < n; ++x) { wv[x] = flags[x] ? 1.0 : 0.0; anyf |= !flags[x]; }
    }
    e->flagged[c] = anyf;
    e->any_flagged = false;
    for (auto f : e->flagged) e->any_flagged |= (f != 0);
    double* wd = e->wd + 2 * (size_t)c * Tp * n;
    CU_TRY(cudaMemcpyAsync(e->w + (size_t)c * n, wv.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(e->ninvd + (size_t)c * n, ninv_diag, n * sizeof(double), cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(wd, vis, 2 * (size_t)T * n * sizeof(double), cudaMemcpyHostToDevice, st));
    if (pt) {
        CU_TRY(cudaMemcpyAsync(e->wT + (size_t)c * Tp * n, wtv.data(), (size_t)T * n * sizeof(double), cudaMemcpyHostToDevice, st));
        std::vector<int> same(Tp, 0);
        for (int t = 1; t < T; ++t) same[t] = std::memcmp(flags + (size_t)t * n, flags + (size_t)(t - 1) * n, n) == 0 ? 1 : 0;
        CU_TRY(cudaMemcpyAsync(e->ptSame + (size_t)c * Tp, same.data(), (size_t)Tp * sizeof(int), cudaMemcpyHostToDevice, st));
        if (e->lowrank_rows()) {
            // channels flagged at time t beyond the all-times mask
            std::vector<uint16_t> fidx((size_t)T * hp::kPtLowMaxRank, 0);
            std::vector<int> fcnt(T, 0);
            int kmax = 0;
            for (int t = 0; t < T; ++t) {
                int k = 0;
                for (int x = 0; x < n; ++x)
                    if (wv[x] != 0.0 && !flags[(size_t)t * n + x]) {
                        if (k < hp::kPtLowMaxRank) fidx[(size_t)t * hp::kPtLowMaxRank + k] = (uint16_t)x;
                        ++k;
                    }
                fcnt[t] = k;
                if (k > kmax) kmax = k;
            }
            e->pt_kmax[c] = kmax;
            CU_TRY(cudaMemcpyAsync(e->ptFidx + (size_t)c * T * hp::kPtLowMaxRank, fidx.data(), fidx.size() * sizeof(uint16_t),
                                   cudaMemcpyHostToDevice, st));
            CU_TRY(cudaMemcpyAsync(e->ptFcnt + (size_t)c * T, fcnt.data(), (size_t)T * sizeof(int), cudaMemcpyHostToDevice, st));
            e->pt_kcap = 0;
            for (int v : e->pt_kmax) if (v > e->pt_kcap) e->pt_kcap = v;
            // a time with more extra flags than the low-rank kernel takes: the whole engine uses k_pt_cholsolve
            e->solve = e->pt_kcap <= hp::kPtLowMaxRank ? Solve::PtLowRank : Solve::PtDirect;
            if (e->solve == Solve::PtDirect && e->cfg.general_basis0)
                return fail(HP_ERR_SIZE, "per-time flags with a general S_initial: a time has more than 64 channels flagged beyond the "
                                         "all-times mask (only the low-rank form of the per-time solve takes a general first basis)");
        }
    }
    // (wv / wtv are pageable locals: cudaMemcpyAsync has staged them before it returns; `vis` may be page-locked and is
    //  only guaranteed consumed by the stream synchronisation at the end of this function)
    if (pt) k_mask_elem<<<nblocks((long long)T * n), 256, 0, st>>>(wd, e->wT + (size_t)c * Tp * n, (long long)T * n);
    else k_mask_cols<<<nblocks((long long)T * n), 256, 0, st>>>(wd, e->w + (size_t)c * n, T, n);
    k_noise_vectors<<<nblocks(n), 256, 0, st>>>(e->w + (size_t)c * n, e->ninvd + (size_t)c * n, e->ni + (size_t)c * n,
                                               e->nu + (size_t)c * n, n);
    if (ps_prior) CU_TRY(cudaMemcpyAsync(e->prior + (size_t)c * 2 * n, ps_prior, 2 * n * sizeof(double), cudaMemcpyHostToDevice, st));
    else CU_TRY(cudaMemsetAsync(e->prior + (size_t)c * 2 * n, 0, 2 * n * sizeof(double), st));
    if (ninv_dense) {
        CU_TRY(cudaMemcpyAsync(e->stage, ninv_dense, 2 * (size_t)n * n * sizeof(double), cudaMemcpyHostToDevice, st));
        k_mask_dense<<<nblocks((long long)n * n), 256, 0, st>>>(e->NiD + 2 * (size_t)c * n * n, e->stage, e->w + (size_t)c * n, n);
        k_lower_half<<<nblocks((long long)n * n), 256, 0, st>>>(e->NiL + 2 * (size_t)c * n * n, e->NiD + 2 * (size_t)c * n * n, n);
        CU_TRY(cudaStreamSynchronize(st));
        if (e->NihD) {
            if (!nih_dense) return fail(HP_ERR_ARG, "injected-draw mode with dense noise needs the square root of the flagged N^-1");
            CU_TRY(cudaMemcpyAsync(e->NihD + 2 * (size_t)c * n * n, nih_dense, 2 * (size_t)n * n * sizeof(double),
                                   cudaMemcpyHostToDevice, st));
        }
    }
    // bases
    double* BF = e->bF.Bmat + 2 * (size_t)c * n * Np;
    k_basis_fourier<<<nblocks((long long)n * n), 256, 0, st>>>(BF, e->U, n, Np);
    if (m > 0) {
        CU_TRY(cudaMemcpyAsync(e->stage, fgmodes, 2 * (size_t)n * m * sizeof(double), cudaMemcpyHostToDevice, st));
        k_basis_fg<<<nblocks((long long)n * m), 256, 0, st>>>(BF, e->Ft + 2 * (size_t)c * m * n, e->stage, n, m, Np);
        if (e->cfg.general_basis0)
            k_basis_fg<<<nblocks((long long)n * m), 256, 0, st>>>(e->b0.Bmat + 2 * (size_t)c * n * Np, nullptr, e->stage, n, m, Np);
        // e->stage is reused below / by the next chain: stream order is enough, no host synchronisation
    }
    if (e->cfg.general_basis0) {
        CU_TRY(cudaMemcpyAsync(e->stage, basis0, 2 * (size_t)n * n * sizeof(double), cudaMemcpyHostToDevice, st));
        k_basis_general<<<nblocks((long long)n * n), 256, 0, st>>>(e->b0.Bmat + 2 * (size_t)c * n * Np, e->stage, n, Np);
    }
    if (!e->cfg.dense_noise && !e->cfg.time_flags) {
        e->pending[c] = 1;   // products built in one batched launch by the first call that needs them
    } else {
        int rc;
        if ((rc = build_basis_products(e, e->bF, c)) != HP_OK) return rc;
        if (e->cfg.general_basis0 && (rc = build_basis_products(e, e->b0, c)) != HP_OK) return rc;
    }
    // initial spectrum
    CU_TRY(cudaMemcpyAsync(e->vecn, lam0sq, n * sizeof(double), cudaMemcpyHostToDevice, st));
    k_init_lam<<<nblocks(Np), 256, 0, st>>>(e->lam + (size_t)c * Np, e->ps + (size_t)c * n, e->vecn, n, N, Np);
    CU_TRY(cudaStreamSynchronize(st));
    CU_TRY(cudaGetLastError());
    e->iter = 0;
    e->out_pos = 0;
    e->draw_counter = 0;
    return HP_OK;
}

int hp_engine_load_chain(hp_engine* e, int c, const double* vis, const uint8_t* flags, const double* fgmodes,
                         const double* ninv_diag, const double* basis0, const double* lam0sq, const double* ps_prior) {
    return load_chain_impl(e, c, vis, flags, fgmodes, ninv_diag, nullptr, nullptr, basis0, lam0sq, ps_prior);
}

int hp_engine_load_chain_dense(hp_engine* e, int c, const double* vis, const uint8_t* flags, const double* fgmodes,
                               const double* ninv_diag, const double* ninv_dense, const double* nih_dense,
                               const double* basis0, const double* lam0sq, const double* ps_prior) {
    if (!ninv_dense) return fail(HP_ERR_ARG, "hp_engine_load_chain_dense: ninv_dense is NULL");
    return load_chain_impl(e, c, vis, flags, fgmodes, ninv_diag, ninv_dense, nih_dense, basis0, lam0sq, ps_prior);
}

int hp_engine_set_draws(hp_engine* e, int c, const double* omega_a, const double* omega_b, const double* s_draws,
                        int n_draw_iters) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    if (e->cfg.rng_mode != HP_RNG_INJECTED) return fail(HP_ERR_ARG, "hp_engine_set_draws: engine is not in injected-draw mode");
    if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);
    if (c < 0 || c >= e->C) return fail(HP_ERR_ARG, "chain index out of range");
    if ((omega_a == nullptr) != (omega_b == nullptr)) return fail(HP_ERR_ARG, "omega_a and omega_b must both be given or both NULL");
    if (n_draw_iters > e->cfg.max_iters) return fail(HP_ERR_ARG, "more draw iterations than max_iters");
    CU_TRY(cudaSetDevice(e->cfg.device));
    { int rcf = flush_pending(e); if (rcf != HP_OK) return rcf; }
    const int n = e->n, Np = e->Np, T = e->T, Tp = e->Tp;
    cudaStream_t st = e->st;
    if (s_draws && n_draw_iters > 0)
        CU_TRY(cudaMemcpyAsync(e->sdraws + (size_t)c * e->cfg.max_iters * n, s_draws, (size_t)n_draw_iters * n * sizeof(double),
                               cudaMemcpyHostToDevice, st));
    if (omega_a) {
        for (int which = 0; which < (e->cfg.general_basis0 ? 2 : 1); ++which) {
            Basis& b = which ? e->b0 : e->bF;
            double* Bm = b.Bmat + 2 * (size_t)c * n * Np;
            // Rfix += B^H N^-1/2 omega_b
            CU_TRY(cudaMemcpyAsync(e->stage, omega_b, 2 * (size_t)T * n * sizeof(double), cudaMemcpyHostToDevice, st));
            hp::ZgemmArgs r{};
            r.A = e->stage; r.sAi = n; r.sAk = 1;
            r.B = Bm; r.sBk = Np; r.sBj = 1; r.conjB = 1;
            r.C = b.Rfix + 2 * (size_t)c * Tp * Np; r.sCi = Np; r.sCj = 1;
            if (e->cfg.dense_noise) {
                hp::ZgemmArgs y{};   // Yd = omega_b Nih^T
                y.A = e->stage; y.sAi = n; y.sAk = 1;
                y.B = e->NihD + 2 * (size_t)c * n * n; y.sBk = 1; y.sBj = n;
                y.C = e->Yd + 2 * (size_t)c * Tp * n; y.sCi = n; y.sCj = 1;
                y.M = T; y.N = n; y.K = n; y.alpha = 1.0; y.batch = 1;
                hp::launch_zgemm(y, st);
                r.A = e->Yd + 2 * (size_t)c * Tp * n;
            } else if (e->cfg.time_flags) {
                // N_t^-1/2 omega_b = sqrt(N^-1) (w_t omega_b)
                k_mask_elem<<<nblocks((long long)T * n), 256, 0, st>>>(e->stage, e->wT + (size_t)c * Tp * n, (long long)T * n);
                k_sqrt_vec<<<nblocks(n), 256, 0, st>>>(e->vecn, e->ninvd + (size_t)c * n, n);
                r.dk = e->vecn;
            } else {
                r.dk = e->nu + (size_t)c * n;
            }
            r.M = T; r.N = e->N; r.K = n; r.accumulate = 1; r.alpha = 1.0; r.batch = 1;
            hp::launch_zgemm(r, st);
            CU_TRY(cudaStreamSynchronize(st));
            // wa = Q^H omega_a
            CU_TRY(cudaMemcpyAsync(e->stage, omega_a, 2 * (size_t)T * n * sizeof(double), cudaMemcpyHostToDevice, st));
            hp::ZgemmArgs a{};
            a.A = e->stage; a.sAi = n; a.sAk = 1;
            a.B = Bm; a.sBk = Np; a.sBj = 1; a.conjB = 1;
            a.C = b.wa + 2 * (size_t)c * Tp * Np; a.sCi = Np; a.sCj = 1;
            a.M = T; a.N = n; a.K = n; a.accumulate = 0; a.alpha = 1.0; a.batch = 1;
            hp::launch_zgemm(a, st);
            CU_TRY(cudaStreamSynchronize(st));
        }
        e->any_omega = true;
    }
    CU_TRY(cudaStreamSynchronize(st));
    CU_TRY(cudaGetLastError());
    return HP_OK;
}

// rows x width bytes, device -> host: one strided copy when the pitches allow it (cudaMemcpy2D limits them to
// cudaDeviceProp::memPitch, 2^31 - 1), else row by row
static cudaError_t copy_rows_d2h(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t rows,
                                 cudaStream_t st) {
    if (rows == 0 || width == 0) return cudaSuccess;
    if (dpitch < (size_t)0x7fffffff && spitch < (size_t)0x7fffffff)
        return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaSuccess;
    for (size_t r = 0; r < rows && e == cudaSuccess; ++r)
        e = cudaMemcpyAsync((char*)dst + r * dpitch, (const char*)src + r * spitch, width, cudaMemcpyDeviceToHost, st);
    return e;
}

// Output slots of one Gibbs iteration (null = not kept).
struct IterOut {
    double* sf; long long sf_bs;            // frequency-space signal (scratch or signal_cr slot)
    double* fg; long long fg_bs;
    double* chisq; long long chisq_bs;
};

// A contiguous range of chains advanced on its own stream.  Chains are independent, so the engine
// splits its batch into `cfg.substreams` such ranges: one range's Cholesky / FFT kernels (low tensor
// occupancy) then overlap another range's k_solve instead of leaving the FP64 pipe idle.
struct Sub { int c0, nc; cudaStream_t st; };
#define OFFS(ptr, per_chain) ((ptr) ? (ptr) + (size_t)sb.c0 * (size_t)(per_chain) : nullptr)

// dense noise: first ln_post term  sum_x,y conj(wr_x) N^-1_xy wr_y  per time (pspec.py:474-478)
static void enqueue_dense_lnp1(hp_engine* e, const Sub& sb) {
    const size_t n = e->n, Tp = e->Tp;
    e->prof_begin(CLS_TRANSFORM, sb.st);
    hp::ZgemmArgs y{};
    y.A = OFFS(e->Rm, 2 * Tp * n); y.sAi = e->n; y.sAk = 1; y.bsA = (long long)e->Tp * e->n;
    // r^H Ni r = 2 Re(r^H NiL r) with NiL the lower half of the Hermitian part of Ni (k_lower_half): Y = R conj(NiL) is a
    // triangular product (B[k][j] = conj(NiL[k][j]) = 0 for k < j: k_zgemm2 skips that K range), half the flops of R Ni^T
    y.B = OFFS(e->NiL, 2 * n * n); y.sBk = e->n; y.sBj = 1; y.conjB = 1; y.bsB = (long long)e->n * e->n;
    y.C = OFFS(e->Yd, 2 * Tp * n); y.sCi = e->n; y.sCj = 1; y.bsC = (long long)e->Tp * e->n;
    y.M = e->T; y.N = e->n; y.K = e->n; y.alpha = 1.0; y.batch = sb.nc;
    y.tri = 2;
    hp::launch_zgemm(y, sb.st);
    k_rowdot<<<dim3(e->Tp, sb.nc), 128, 0, sb.st>>>(OFFS(e->Rm, 2 * Tp * n), OFFS(e->Yd, 2 * Tp * n), OFFS(e->lnp1, Tp), e->T,
                                                   e->Tp, e->n, 2.0);
    e->prof_end(CLS_TRANSFORM, 2, sb.st);
}

// Whether the next computed iteration is accumulated into the posterior moments: after hp_engine_set_summary the first
// burn_in iterations are skipped, then every thin-th one is taken.  Decided on the host once per iteration, for all
// sub-batches alike, and so is whether it closes a batch of the batch means (the count reaches j * batch).
struct SumStep {
    double invk = 0.0;   // 1 / (accumulated iterations including this one); 0: not accumulated
    double jj1 = -1.0;   // j (j - 1) when the iteration closes batch j; < 0: it closes none
};
static SumStep summary_step(hp_engine* e) {
    auto& s = e->sum;
    SumStep r;
    if (!s.what) return r;
    const long long k = s.seen++ - s.burn_in;
    if (k < 0 || k % s.thin != 0) return r;
    r.invk = 1.0 / (double)(++s.count);
    if (s.batch > 0 && s.count % s.batch == 0) {
        const double j = (double)(s.count / s.batch);
        r.jj1 = j * (j - 1.0);
    }
    return r;
}

// What one iteration (or GCR step) uses, decided on the host once for all sub-batches: the general first basis on the
// first iteration, the draw counter of the GCR fluctuations (fixed in Philox mode unless refresh_omega) and, with
// `summary`, the posterior-moment step (summary_step)
struct IterStep { bool general; uint32_t draw_iter; SumStep sum; };
static IterStep iter_step(hp_engine* e, bool summary) {
    IterStep r;
    r.general = e->cfg.general_basis0 && e->iter == 0;
    r.draw_iter = (e->cfg.rng_mode == HP_RNG_PHILOX && !e->cfg.refresh_omega) ? 0u : e->draw_counter++;
    if (summary) r.sum = summary_step(e);
    return r;
}

// the draw identity of sub-batch sb at draw counter `iter`
static hp::DrawKey draw_key(const hp_engine* e, const Sub& sb, uint32_t iter) {
    return hp::DrawKey{(uint32_t)e->cfg.seed, (uint32_t)(e->cfg.seed >> 32), iter, OFFS(e->chain_ids, 1)};
}

// Ppart[sys][0][k] = sum_t |ytilde_k|^2 from the solution X
static void launch_beta_sums(hp_engine* e, const Sub& sb) {
    hp::launch_colsumsq(OFFS(e->X, 2 * (size_t)e->Tp * e->Np), OFFS(e->Ppart, (size_t)e->ntiles * e->n), e->T, e->Tp, e->n, sb.nc,
                        sb.st, e->Np);
}
static void launch_make_ssc(hp_engine* e, const Sub& sb) {
    k_make_ssc<<<dim3(nblocks((long long)e->T * e->n), sb.nc), 256, 0, sb.st>>>(
        OFFS(e->Ssc, 2 * (size_t)e->Tp * e->n), OFFS(e->X, 2 * (size_t)e->Tp * e->Np), OFFS(e->lam, (size_t)e->Np), e->n, e->Np, e->T, e->Tp);
}

// The solve paths.  Each leaves the solution [ytilde ; f] in X, e->ppart_tiles partial sums of beta = sum_t |ytilde|^2 per
// chain in Ppart, and with `ssc` lam * ytilde in Ssc.  wa: Q^H omega_a of the injected draws, or null.
// x = W^H (W r + xi) as two dense products (W unpacked to a dense lower-triangular matrix): the path for Nfreqs + Nmodes
// beyond k_solve's shared-memory resident tile (BASELINE.json configs[4])
static void solve_dense(hp_engine* e, Basis& b, const Sub& sb, const hp::DrawKey& dk, const double* wa, bool ssc) {
    const size_t Np = e->Np, Tp = e->Tp, tri = hp::tri_blocks(e->nblk);
    e->prof_begin(CLS_SOLVE, sb.st);
    const long long NN = (long long)e->Np * e->Np, TN = (long long)e->Tp * e->Np;
    double* Wd = OFFS(e->Wd, 2 * Np * Np);
    double* Yb = OFFS(e->Yb, 2 * Tp * Np);
    double* X = OFFS(e->X, 2 * Tp * Np);
    k_unpack_lower<<<dim3(nblocks(NN), sb.nc), 256, 0, sb.st>>>(OFFS(e->Wp, tri * hp::kLBlkDoubles), Wd, e->nblk,
                                                               tri * hp::kLBlkDoubles);
    k_build_rhs<<<dim3(nblocks(TN), sb.nc), 256, 0, sb.st>>>(X, OFFS(b.Rfix, 2 * Tp * Np), wa, OFFS(e->lam, Np), e->n, e->Np, e->T,
                                                            e->Tp);
    hp::ZgemmArgs y{};   // Y[t][i] = sum_j r[t][j] W[i][j]
    y.A = X; y.sAi = e->Np; y.sAk = 1; y.bsA = TN;
    y.B = Wd; y.sBk = 1; y.sBj = e->Np; y.bsB = NN;
    y.C = Yb; y.sCi = e->Np; y.sCj = 1; y.bsC = TN;
    y.M = e->T; y.N = e->Np; y.K = e->Np; y.alpha = 1.0; y.batch = sb.nc;
    y.tri = 1;           // B[k = j][col = i] = W[i][j] = 0 for j > i
    hp::launch_zgemm(y, sb.st);
    const bool philox = e->cfg.rng_mode == HP_RNG_PHILOX;
    if (philox) k_add_noise<<<dim3(nblocks((long long)e->T * e->Np), sb.nc), 256, 0, sb.st>>>(Yb, e->N, e->Np, e->T, e->Tp, dk);
    hp::ZgemmArgs x{};   // X[t][i] = sum_j y[t][j] conj(W[j][i])
    x.A = Yb; x.sAi = e->Np; x.sAk = 1; x.bsA = TN;
    x.B = Wd; x.sBk = e->Np; x.sBj = 1; x.bsB = NN; x.conjB = 1;
    x.C = X; x.sCi = e->Np; x.sCj = 1; x.bsC = TN;
    x.M = e->T; x.N = e->Np; x.K = e->Np; x.alpha = 1.0; x.batch = sb.nc;
    x.tri = 2;           // B[k = j][col = i] = conj(W[j][i]) = 0 for j < i
    hp::launch_zgemm(x, sb.st);
    if (e->cfg.cg_compat) hp::launch_cg_scale(X, OFFS(b.Rfix, 2 * Tp * Np), wa, OFFS(e->lam, Np), e->n, e->N, e->Np, e->T, e->Tp, sb.nc, sb.st);
    launch_beta_sums(e, sb);
    if (ssc) launch_make_ssc(e, sb);
    // unpack, right-hand sides, two products, beta sums (+ noise, CG scaling, Ssc)
    e->prof_end(CLS_SOLVE, 5 + philox + (e->cfg.cg_compat != 0) + ssc, sb.st);
}

// k_solve3: right-hand sides in tile layout (Philox: the unscaled tiles built at load time, Wf1 = W diag(lam); injected draws:
// r = lam * Rfix + wa rebuilt per solve, Wf1 = W)
static void solve_solve3(hp_engine* e, Basis& b, const Sub& sb, const hp::DrawKey& dk, const double* wa, bool ssc) {
    const size_t n = e->n, Np = e->Np, Tp = e->Tp;
    const bool philox = e->cfg.rng_mode == HP_RNG_PHILOX;
    e->prof_begin(CLS_SOLVE, sb.st);
    if (!philox)
        hp::launch_rhs_tile(OFFS(b.Rt, 2 * Tp * Np), OFFS(b.Rfix, 2 * Tp * Np), wa, OFFS(e->lam, Np), e->nblk, e->n, e->N,
                            e->lowrank_rows() ? e->Tp : e->T, e->Tp, e->ntiles, sb.nc, sb.st);
    hp::Solve3Args sa{};
    sa.Wf1 = OFFS(e->Wf1, hp::solve3_frag_doubles(e->nblk)); sa.Wf2 = OFFS(e->Wf2, hp::solve3_frag_doubles(e->nblk));
    sa.Rt = OFFS(b.Rt, 2 * Tp * Np);
    sa.X = OFFS(e->X, 2 * Tp * Np);
    sa.Ppart = OFFS(e->Ppart, (size_t)e->ntiles * n);
    sa.nblk = e->nblk; sa.n = e->n; sa.N = e->N; sa.Tp = e->Tp; sa.ntiles = e->ntiles; sa.nsys = sb.nc; sa.T = e->T;
    sa.philox = philox ? 1 : 0;
    sa.dk = dk;
    sa.sched = e->sched3; sa.nstrip = (e->N + 15) / 16;
    hp::launch_solve3(sa, sb.st);
    if (e->cfg.cg_compat) {
        hp::launch_cg_scale(sa.X, OFFS(b.Rfix, 2 * Tp * Np), wa, OFFS(e->lam, Np), e->n, e->N, e->Np, e->T, e->Tp, sb.nc, sb.st);
        launch_beta_sums(e, sb);
    }
    if (ssc) launch_make_ssc(e, sb);
    e->prof_end(CLS_SOLVE, (philox ? 1 : 2) + 2 * (e->cfg.cg_compat != 0) + ssc, sb.st);
}

static void solve_resident(hp_engine* e, Basis& b, const Sub& sb, const hp::DrawKey& dk, const double* wa, bool ssc) {
    const size_t n = e->n, Np = e->Np, Tp = e->Tp, tri = hp::tri_blocks(e->nblk);
    e->prof_begin(CLS_SOLVE, sb.st);
    hp::SolveArgs sa{};
    sa.Wp = OFFS(e->Wp, tri * hp::kLBlkDoubles); sa.lam = OFFS(e->lam, Np);
    sa.Rfix = OFFS(b.Rfix, 2 * Tp * Np);
    sa.wa = wa;
    sa.X = OFFS(e->X, 2 * Tp * Np); sa.Ssc = ssc ? OFFS(e->Ssc, 2 * Tp * n) : nullptr;
    sa.Ppart = OFFS(e->Ppart, (size_t)e->ntiles * n);
    sa.nblk = e->nblk; sa.n = e->n; sa.N = e->N; sa.Tp = e->Tp; sa.ntiles = e->ntiles; sa.nsys = sb.nc; sa.T = e->T;
    sa.philox_wa = e->cfg.rng_mode == HP_RNG_PHILOX ? 1 : 0;
    sa.cg_compat = e->cfg.cg_compat;
    sa.dk = dk;
    hp::launch_solve(sa, sb.st);
    e->prof_end(CLS_SOLVE, 1, sb.st);
}

// per-time flags, low-rank form: k_solve3 leaves R = M_0^-1 A in rows Tp0 + x of X (no reference-CG mode with per-time
// flags).  P = A^H R, then the rank-k_t correction of every time
static void solve_pt_lowrank(hp_engine* e, Basis& b, const Sub& sb, const hp::DrawKey& dk, const double* wa, bool ssc) {
    const size_t n = e->n, Np = e->Np, Tp = e->Tp;
    solve_solve3(e, b, sb, dk, wa, false);
    e->prof_begin(CLS_LOWRANK, sb.st);
    double* X = OFFS(e->X, 2 * Tp * Np);
    hp::ZgemmArgs pz{};
    pz.A = OFFS(b.Rfix, 2 * Tp * Np) + 2 * (size_t)e->Tp0 * Np; pz.sAi = e->Np; pz.sAk = 1; pz.bsA = (long long)e->Tp * e->Np;
    pz.conjA = 1; pz.dk = OFFS(e->lam, Np); pz.bsD = e->Np;
    pz.B = X + 2 * (size_t)e->Tp0 * Np; pz.sBk = 1; pz.sBj = e->Np; pz.bsB = (long long)e->Tp * e->Np;
    pz.C = OFFS(e->Pm, 2 * n * n); pz.sCi = e->n; pz.sCj = 1; pz.bsC = (long long)e->n * e->n;
    pz.M = e->n; pz.N = e->n; pz.K = e->N; pz.alpha = 1.0; pz.batch = sb.nc;
    pz.lower_out = 1;   // k_pt_lowrank reads the lower triangle of P only
    hp::launch_zgemm(pz, sb.st);
    hp::PtLowArgs la{};
    la.Rfix = OFFS(b.Rfix, 2 * Tp * Np); la.wa = wa; la.lam = OFFS(e->lam, Np); la.X = X; la.Pm = OFFS(e->Pm, 2 * n * n);
    la.fidx = e->ptFidx + (size_t)sb.c0 * e->T * hp::kPtLowMaxRank; la.fcnt = e->ptFcnt + (size_t)sb.c0 * e->T;
    la.info = e->info + sb.c0;
    la.n = e->n; la.N = e->N; la.Np = e->Np; la.T = e->T; la.Tp = e->Tp; la.Tp0 = e->Tp0; la.nsys = sb.nc; la.nblk = e->nblk;
    la.kcap = e->pt_kcap; la.philox = e->cfg.rng_mode == HP_RNG_PHILOX ? 1 : 0;
    la.dk = dk;
    hp::launch_pt_lowrank(la, sb.st);
    launch_beta_sums(e, sb);
    e->prof_end(CLS_LOWRANK, 3, sb.st);
    e->prof_begin(CLS_SOLVE, sb.st);   // lam * ytilde for a general first basis, else empty
    if (ssc) launch_make_ssc(e, sb);
    e->prof_end(CLS_SOLVE, ssc ? 1 : 0, sb.st);
}

// per-time flags, one factorisation + solve per (chain, time); sub-batches share the SMs, each gets its share of the
// persistent grid and of the scratch slots.  Never asked for Ssc: a general first basis needs the low-rank form
// (select_paths, load_chain_impl refuse it here), and per-time flags always have an FFT plan
static void solve_pt_direct(hp_engine* e, Basis& b, const Sub& sb, const hp::DrawKey& dk, const double* wa) {
    const size_t m = e->m, Np = e->Np, Tp = e->Tp;
    const int nsub = e->C > 0 ? (e->C + sb.nc - 1) / sb.nc : 1;
    int grid = e->pt_ctas / (nsub > 0 ? nsub : 1);
    if (grid < 1) grid = 1;
    const int slot0 = (int)(((long long)sb.c0 * e->pt_ctas) / e->C);
    if (slot0 + grid > e->pt_ctas) grid = e->pt_ctas - slot0;
    e->prof_begin(CLS_SOLVE, sb.st);
    cudaMemsetAsync(e->info + sb.c0, 0, sizeof(int) * sb.nc, sb.st);
    hp::PtArgs pa{};
    pa.H = OFFS(e->Hpt, 2 * Tp * (1 + m) * Np); pa.lam = OFFS(e->lam, Np); pa.Rfix = OFFS(b.Rfix, 2 * Tp * Np);
    pa.wa = wa;
    pa.X = OFFS(e->X, 2 * Tp * Np);
    pa.same_prev = OFFS(e->ptSame, Tp);
    pa.scratch = e->ptScratch + (size_t)slot0 * hp::pt_scratch_doubles_per_cta(e->nblk);
    pa.info = e->info + sb.c0;
    pa.nblk = e->nblk; pa.n = e->n; pa.m = e->m; pa.N = e->N; pa.T = e->T; pa.Tp = e->Tp; pa.nsys = sb.nc;
    pa.philox_wa = e->cfg.rng_mode == HP_RNG_PHILOX ? 1 : 0;
    pa.dk = dk;
    hp::launch_pt_cholsolve(pa, grid, sb.st);
    launch_beta_sums(e, sb);
    e->prof_end(CLS_SOLVE, 2, sb.st);
}

// s = U^H (lam ytilde) (fused into k_post_fft / k_post_fft2, or with `ssc` a dense back-transform of Ssc), foreground
// amplitudes, residual statistics and the sums of |U s|^2, |U (w s)|^2 that k_sample reads (sample_energies)
static void enqueue_post(hp_engine* e, Basis& b, const IterOut& o, const Sub& sb, Post post, bool ssc) {
    const bool general = &b == &e->b0;
    const size_t n = e->n, m = e->m, Np = e->Np, Tp = e->Tp;
    double* sf = o.sf + 2 * (size_t)sb.c0 * (size_t)o.sf_bs;
    if (ssc) {
        // s = Q (lam * ytilde) as a dense product (general eigenbasis, or Nfreqs without an FFT plan)
        e->prof_begin(CLS_TRANSFORM, sb.st);
        hp::ZgemmArgs t{};
        t.A = OFFS(e->Ssc, 2 * Tp * n); t.sAi = e->n; t.sAk = 1; t.bsA = (long long)e->Tp * e->n;
        t.B = OFFS(b.Bmat, 2 * n * Np); t.sBk = 1; t.sBj = e->Np; t.bsB = (long long)e->n * e->Np;
        t.C = sf; t.sCi = e->n; t.sCj = 1; t.bsC = o.sf_bs;
        t.M = e->T; t.N = e->n; t.K = e->n; t.accumulate = 0; t.alpha = 1.0; t.batch = sb.nc;
        hp::launch_zgemm(t, sb.st);
        e->prof_end(CLS_TRANSFORM, 1, sb.st);
    }
    e->last_sf = o.sf;
    e->last_sf_bs = o.sf_bs;
    double* fg = o.fg ? o.fg + (size_t)sb.c0 * (size_t)o.fg_bs : nullptr;
    double* chisq = o.chisq ? o.chisq + (size_t)sb.c0 * (size_t)o.chisq_bs : nullptr;

    e->prof_begin(CLS_POST, sb.st);
    if (post == Post::Dense) {
        // dense fallback for Nfreqs with a large prime factor
        hp::PostArgs pa{};
        pa.Sf = sf; pa.sf_bs = o.sf_bs; pa.X = OFFS(e->X, 2 * Tp * Np); pa.Ft = OFFS(e->Ft, 2 * (m ? m : 1) * n);
        pa.wd = OFFS(e->wd, 2 * Tp * n); pa.w = OFFS(e->w, n); pa.ninvd = OFFS(e->ninvd, n);
        pa.fg_out = fg; pa.fg_bs = o.fg_bs; pa.chisq_out = chisq; pa.chisq_bs = o.chisq_bs;
        pa.Wm = e->any_flagged ? OFFS(e->Wm, 2 * Tp * n) : nullptr; pa.Rm = e->cfg.dense_noise ? OFFS(e->Rm, 2 * Tp * n) : nullptr;
        pa.lnp1 = OFFS(e->lnp1, Tp);
        pa.n = e->n; pa.m = e->m; pa.Np = e->Np; pa.T = e->T; pa.Tp = e->Tp; pa.nsys = sb.nc;
        hp::launch_post(pa, sb.st);
    } else {
        hp::PostFftArgs pa{};
        pa.plan = e->plan; pa.tw = e->tw; pa.tw2 = e->tw2; pa.X = OFFS(e->X, 2 * Tp * Np); pa.lam = OFFS(e->lam, Np); pa.Sf = sf; pa.sf_bs = o.sf_bs;
        pa.Ft = OFFS(e->Ft, 2 * (m ? m : 1) * n); pa.wd = OFFS(e->wd, 2 * Tp * n); pa.w = OFFS(e->w, n); pa.ninvd = OFFS(e->ninvd, n);
        pa.w_bs = e->n; pa.w_ts = 0;
        if (e->cfg.time_flags) { pa.w = OFFS(e->wT, Tp * n); pa.w_bs = (long long)e->Tp * e->n; pa.w_ts = e->n; }
        pa.fg_out = fg; pa.fg_bs = o.fg_bs; pa.chisq_out = chisq; pa.chisq_bs = o.chisq_bs;
        pa.lnp1 = OFFS(e->lnp1, Tp); pa.Rm = e->cfg.dense_noise ? OFFS(e->Rm, 2 * Tp * n) : nullptr;
        pa.Empart = e->any_flagged ? OFFS(e->Empart, (size_t)e->ntilesE * n) : nullptr;
        pa.Eupart = general ? OFFS(e->Eupart, (size_t)e->ntilesE * n) : nullptr;
        pa.m = e->m; pa.Np = e->Np; pa.T = e->T; pa.Tp = e->Tp; pa.nsys = sb.nc; pa.do_inverse = ssc ? 0 : 1; pa.ktp = e->ktp;
        if (post == Post::Fft2) hp::launch_post_fft2(pa, sb.st);
        else hp::launch_post_fft(pa, sb.st);
    }
    e->prof_end(CLS_POST, 1, sb.st);
    if (e->cfg.dense_noise) enqueue_dense_lnp1(e, sb);
    if (post == Post::Dense && (e->any_flagged || general)) {
        e->prof_begin(CLS_TRANSFORM, sb.st);
        int nl2 = 0;
        hp::ZgemmArgs t{};
        t.sAi = e->n; t.sAk = 1; t.bsA = (long long)e->Tp * e->n;
        t.B = e->U; t.sBk = 1; t.sBj = e->n; t.bsB = 0;
        t.C = OFFS(e->Tmp, 2 * Tp * n); t.sCi = e->n; t.sCj = 1; t.bsC = (long long)e->Tp * e->n;
        t.M = e->T; t.N = e->n; t.K = e->n; t.accumulate = 0; t.alpha = 1.0; t.batch = sb.nc;
        if (e->any_flagged) {
            t.A = OFFS(e->Wm, 2 * Tp * n);
            hp::launch_zgemm(t, sb.st);
            hp::launch_colsumsq(OFFS(e->Tmp, 2 * Tp * n), OFFS(e->Em, n), e->T, e->Tp, e->n, sb.nc, sb.st);
            nl2 += 2;
        }
        if (general) {
            t.A = sf; t.bsA = o.sf_bs;
            hp::launch_zgemm(t, sb.st);
            hp::launch_colsumsq(OFFS(e->Tmp, 2 * Tp * n), OFFS(e->Eu, n), e->T, e->Tp, e->n, sb.nc, sb.st);
            nl2 += 2;
        }
        e->prof_end(CLS_TRANSFORM, nl2, sb.st);
    }
}

// Where enqueue_post left sum_t |U s|^2 (Eu, general-basis iteration) and sum_t |U (w s)|^2 (Em, flagged channels) for
// k_sample: per-tile partial sums from k_post_fft / k_post_fft2, one sum per chain from the dense transforms
static void sample_energies(hp_engine* e, const Sub& sb, hp::SampleArgs& sp) {
    const size_t n = e->n;
    const bool tiles = e->post != Post::Dense;
    sp.ntilesE = tiles ? e->ntilesE : 0;
    sp.Eu = tiles ? OFFS(e->Eupart, (size_t)e->ntilesE * n) : OFFS(e->Eu, n);
    sp.Em = e->any_flagged ? (tiles ? OFFS(e->Empart, (size_t)e->ntilesE * n) : OFFS(e->Em, n)) : nullptr;
}

// GCR step (gcr_fgmodes) and everything of gibbs_step_fgmodes up to the power-spectrum draw:
// chol + solve + back-transform + residual statistics
static void enqueue_gcr(hp_engine* e, const IterOut& o, const Sub& sb, const IterStep& step) {
    Basis& b = step.general ? e->b0 : e->bF;
    const hp::DrawKey dk = draw_key(e, sb, step.draw_iter);
    // the general-basis first iteration needs Eupart, which k_post_fft2 does not write; the post-processing fuses the inverse
    // transform otherwise, and the solve leaves lam * ytilde in Ssc for a dense back-transform only when it does not
    const Post post = (step.general && e->post == Post::Fft2) ? Post::Fft : e->post;
    const bool ssc = post == Post::Dense || step.general;
    const bool philox = e->cfg.rng_mode == HP_RNG_PHILOX;
    const double* wa = (!philox && e->any_omega) ? OFFS(b.wa, 2 * (size_t)e->Tp * e->Np) : nullptr;
    if (e->solve != Solve::PtDirect) {
        const size_t Np = e->Np, tri = hp::tri_blocks(e->nblk);
        e->prof_begin(CLS_CHOL, sb.st);
        hp::CholArgs ca{};
        ca.Gp = OFFS(b.Gp, tri * hp::kBlkDoubles); ca.lam = OFFS(e->lam, Np); ca.Lp = OFFS(e->Lp, tri * hp::kLBlkDoubles);
        ca.Linvp = OFFS(e->Linvp, (size_t)e->nblk * hp::kLBlkDoubles); ca.info = e->info + sb.c0;
        ca.nblk = e->nblk; ca.n = e->n; ca.N = e->N; ca.nsys = sb.nc;
        // Philox mode: the stored right-hand-side tiles are the unscaled Rfix, so pass 1 multiplies by W diag(lam)
        const hp::TrinvExtra ex{OFFS(e->Wf1, hp::solve3_frag_doubles(e->nblk)), OFFS(e->Wf2, hp::solve3_frag_doubles(e->nblk)),
                                philox ? OFFS(e->lam, Np) : nullptr};
        e->prof_end(CLS_CHOL, hp::launch_chol_trinv(ca, OFFS(e->Wp, tri * hp::kLBlkDoubles), ex, sb.st), sb.st);
    }
    switch (e->solve) {
        case Solve::Solve3: solve_solve3(e, b, sb, dk, wa, ssc); break;
        case Solve::Resident: solve_resident(e, b, sb, dk, wa, ssc); break;
        case Solve::Dense: solve_dense(e, b, sb, dk, wa, ssc); break;
        case Solve::PtLowRank: solve_pt_lowrank(e, b, sb, dk, wa, ssc); break;
        case Solve::PtDirect: solve_pt_direct(e, b, sb, dk, wa); break;
    }
    enqueue_post(e, b, o, sb, post, ssc);
}

// sub-batches of the engine: [c0, c0 + nc) on stream st (the engine's own stream when there is one range)
static std::vector<Sub> make_subs(hp_engine* e) {
    std::vector<Sub> v;
    int ns = e->active_subs < (int)e->sub_st.size() ? e->active_subs : (int)e->sub_st.size();
    if (ns <= 1) { v.push_back({0, e->C, e->st}); return v; }
    int base = e->C / ns, rem = e->C % ns, c0 = 0;
    for (int i = 0; i < ns; ++i) {
        int nc = base + (i < rem ? 1 : 0);
        if (nc > 0) v.push_back({c0, nc, e->sub_st[i]});
        c0 += nc;
    }
    return v;
}
// fork: every sub-stream waits for what is already enqueued on the engine stream; join: the reverse
static void fork_subs(hp_engine* e, const std::vector<Sub>& subs) {
    if (subs.size() <= 1) return;
    cudaEventRecord(e->fork_ev, e->st);
    for (auto& sb : subs) cudaStreamWaitEvent(sb.st, e->fork_ev, 0);
}
static void join_subs(hp_engine* e, const std::vector<Sub>& subs) {
    if (subs.size() <= 1) return;
    for (size_t i = 0; i < subs.size(); ++i) {
        cudaEventRecord(e->join_ev[i], subs[i].st);
        cudaStreamWaitEvent(e->st, e->join_ev[i], 0);
    }
}

int hp_engine_gcr(hp_engine* e) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);
    CU_TRY(cudaSetDevice(e->cfg.device));
    { int rcf = flush_pending(e); if (rcf != HP_OK) return rcf; }
    const IterStep step = iter_step(e, false);
    IterOut o{e->Sf, (long long)e->Tp * e->n, nullptr, 0, nullptr, 0};
    auto subs = make_subs(e);
    fork_subs(e, subs);
    for (auto& sb : subs) enqueue_gcr(e, o, sb, step);
    join_subs(e, subs);
    CU_TRY(cudaGetLastError());
    return HP_OK;
}

// one Gibbs iteration (gibbs_step_fgmodes, pspec.py:377-490) of the chains of one sub-batch
// step.sum.invk > 0: accumulate the iteration into the posterior moments (SumStep)
static void enqueue_iteration_sub(hp_engine* e, const Sub& sb, int it, uint32_t iter, const IterStep& step) {
    const size_t n = e->n, m = e->m, T = e->T, Tp = e->Tp, I = e->cfg.max_iters, Np = e->Np;
    const bool philox = e->cfg.rng_mode == HP_RNG_PHILOX;
    IterOut o{};
    const size_t R = e->ring, slot = (size_t)it % R;   // big outputs: ring slot; signal_ps / ln_post: one entry per iteration
    // ring layout [slot][chain][...]: one iteration's array of all chains is contiguous (one plain copy to the host)
    const size_t Cn = (size_t)e->C;
    o.sf = e->cr_out ? e->cr_out + 2 * slot * Cn * T * n : e->Sf;
    o.sf_bs = e->cr_out ? (long long)(T * n) : (long long)(Tp * n);
    o.fg = e->fg_out ? e->fg_out + 2 * slot * Cn * T * m : nullptr; o.fg_bs = 2 * (long long)(T * m);
    o.chisq = e->chisq_out ? e->chisq_out + slot * Cn * T * n : nullptr; o.chisq_bs = (long long)(T * n);
    enqueue_gcr(e, o, sb, step);

    if (step.sum.invk > 0.0) {
        // signal_cr from the slot the iteration wrote; fg_amps straight from the solution X (rows t < T, columns n .. n + m),
        // where HP_BUF_LAST_FG reads it too, so that it needs no HP_KEEP_FG
        const auto& s = e->sum;
        hp::MomentsArr cr{}, fg{};
        hp::MomentsBatch crb{}, fgb{};
        if (s.what & HP_SUMMARY_CR) {
            cr.src = o.sf + 2 * (size_t)sb.c0 * (size_t)o.sf_bs; cr.src_cs = o.sf_bs; cr.w = e->n; cr.rs = e->n;
            cr.L = (int)(T * n); cr.nsys = sb.nc; cr.ld = s.ld_cr;
            cr.mean = s.cr_mean + 2 * (size_t)sb.c0 * s.ld_cr; cr.m2 = s.cr_m2 + (size_t)sb.c0 * s.ld_cr;
            if (s.batch > 0) { crb.snap = s.cr_snap + 2 * (size_t)sb.c0 * s.ld_cr; crb.m2 = s.cr_m2bm + (size_t)sb.c0 * s.ld_cr; }
        }
        if ((s.what & HP_SUMMARY_FG) && m > 0) {
            fg.src = OFFS(e->X, 2 * Tp * Np) + 2 * n; fg.src_cs = (long long)(Tp * Np); fg.w = e->m; fg.rs = e->Np;
            fg.L = (int)(T * m); fg.nsys = sb.nc; fg.ld = s.ld_fg;
            fg.mean = s.fg_mean + 2 * (size_t)sb.c0 * s.ld_fg; fg.m2 = s.fg_m2 + (size_t)sb.c0 * s.ld_fg;
            if (s.batch > 0) { fgb.snap = s.fg_snap + 2 * (size_t)sb.c0 * s.ld_fg; fgb.m2 = s.fg_m2bm + (size_t)sb.c0 * s.ld_fg; }
        }
        // only the iterations that close a batch run the longer k_moments_batch; the launch count is the same
        e->launches += step.sum.jj1 >= 0.0 ? hp::launch_moments_batch(cr, fg, crb, fgb, step.sum.invk, step.sum.jj1, sb.st)
                                           : hp::launch_moments(cr, fg, step.sum.invk, sb.st);
    }

    e->prof_begin(CLS_SAMPLE, sb.st);
    hp::SampleArgs sp{};
    sp.Ppart = OFFS(e->Ppart, (size_t)e->ntiles * n); sp.ntiles = e->ppart_tiles;
    sample_energies(e, sb, sp);
    sp.lnp1 = OFFS(e->lnp1, Tp); sp.lnp1_dense = nullptr; sp.prior = OFFS(e->prior, 2 * n);
    sp.draws = philox ? nullptr : OFFS(e->sdraws, I * n) + (size_t)it * n; sp.draws_bs = (long long)(I * n);
    sp.ps = OFFS(e->ps, n); sp.lam = OFFS(e->lam, Np);
    sp.ps_out = OFFS(e->ps_out, I * n) + (size_t)it * n; sp.ps_bs = (long long)(I * n);
    sp.lnpost_out = OFFS(e->lnpost_out, I) + it; sp.lnpost_bs = (long long)I;
    sp.n = e->n; sp.Np = e->Np; sp.T = e->T; sp.Tp = e->Tp; sp.nsys = sb.nc;
    sp.beta_mode = step.general ? 1 : 0; sp.philox = philox ? 1 : 0;
    sp.dk = draw_key(e, sb, iter);
    hp::launch_sample(sp, sb.st);
    e->prof_end(CLS_SAMPLE, 1, sb.st);
}

// `niter` Gibbs iterations of all chains.  Sub-batches run back to back on their own streams (no
// synchronisation between them: chains are independent); `after_iter(k)` is called on the host right
// after iteration k of every sub-batch has been enqueued, with the engine stream joined to it.
extern "C++" {
template <typename F>
static void enqueue_iterations(hp_engine* e, int niter, F&& after_iter) {
    auto subs = make_subs(e);
    fork_subs(e, subs);
    for (int k = 0; k < niter; ++k) {
        const IterStep step = iter_step(e, true);
        for (auto& sb : subs) enqueue_iteration_sub(e, sb, e->out_pos, (uint32_t)e->iter, step);
        e->iter++;
        e->out_pos++;
        if (after_iter(k)) { join_subs(e, subs); after_iter(-1 - k); if (k + 1 < niter) fork_subs(e, subs); }
    }
    join_subs(e, subs);
}
}  // extern "C++"

int hp_engine_run(hp_engine* e, int niter) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);
    if (niter < 0 || e->out_pos + niter > e->cfg.max_iters)
        return fail(HP_ERR_ARG, "hp_engine_run: would exceed max_iters (use hp_engine_rewind)");
    CU_TRY(cudaSetDevice(e->cfg.device));
    { int rcf = flush_pending(e); if (rcf != HP_OK) return rcf; }
    enqueue_iterations(e, niter, [](int) { return false; });
    CU_TRY(cudaGetLastError());
    return HP_OK;
}

int hp_engine_run_to_host(hp_engine* e, int niter, const hp_host_sink* sink) {
    if (!e || !sink) return fail(HP_ERR_ARG, "null argument");
    if (niter < 0 || e->out_pos + niter > e->cfg.max_iters || sink->first_iter < 0 || e->out_pos < sink->first_iter ||
        e->out_pos + niter - sink->first_iter > sink->iters)
        return fail(HP_ERR_ARG, "hp_engine_run_to_host: would exceed max_iters / sink capacity");
    if ((sink->signal_cr && !e->cr_out) || (sink->fg_amps && !e->fg_out) || (sink->chisq && !e->chisq_out))
        return fail(HP_ERR_ARG, "hp_engine_run_to_host: sink asks for an output that is not kept (cfg.keep)");
    CU_TRY(cudaSetDevice(e->cfg.device));
    { int rcf = flush_pending(e); if (rcf != HP_OK) return rcf; }
    if (!e->copy_st) CU_TRY(cudaStreamCreateWithFlags(&e->copy_st, cudaStreamNonBlocking));
    const size_t n = e->n, m = e->m, T = e->T, I = e->cfg.max_iters, HI = sink->iters, R = e->ring, C = (size_t)e->C;
    const int first = e->out_pos;
    const bool big = sink->signal_cr || (sink->fg_amps && m) || sink->chisq;
    auto subs = make_subs(e);
    const size_t nsub = subs.size();
    if (e->ahead > 0 && (!big || e->it_done.size() < R * nsub))
        return fail(HP_ERR_ARG, "hp_engine_run_to_host: read-ahead iterations are pending; deliver them with the same kind of sink");
    if (big) {
        while (e->copy_done.size() < R) {
            cudaEvent_t ev;
            CU_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            e->copy_done.push_back(ev);
        }
        while (e->it_done.size() < R * nsub) {
            cudaEvent_t ev;
            CU_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            e->it_done.push_back(ev);
        }
    }
    // Sub-batches never join between iterations: each records an event after its part of an iteration, the copy stream
    // waits for all of them and streams the iteration's ring slot to the host while the next iterations compute; a
    // sub-batch only waits (for the copies out of the slot it is about to overwrite) when it is R iterations ahead.
    fork_subs(e, subs);
    cudaError_t cerr = cudaSuccess;
    // compute iteration `it` (the next one of the chain) into its ring slot; records it_done[slot][*]
    auto compute_next = [&](size_t it) {
        const size_t slot = it % R;
        const IterStep step = iter_step(e, true);
        for (size_t i = 0; i < nsub; ++i) {
            // the slot was last used by iteration it - R: wait for its copies unless they completed in an earlier call
            if (big && it >= R + (size_t)first) cudaStreamWaitEvent(subs[i].st, e->copy_done[slot], 0);
            enqueue_iteration_sub(e, subs[i], (int)it, (uint32_t)e->iter, step);
            if (big) cudaEventRecord(e->it_done[slot * nsub + i], subs[i].st);
        }
        e->iter++;
    };
    for (int k = 0; k < niter && cerr == cudaSuccess; ++k) {
        const size_t it = (size_t)e->out_pos, slot = it % R, hs = it - (size_t)sink->first_iter;
        if (e->ahead > 0) --e->ahead;          // computed at the end of the previous call (read-ahead): only the copies are left
        else compute_next(it);
        e->out_pos++;
        if (!big) continue;
        for (size_t i = 0; i < nsub; ++i) cudaStreamWaitEvent(e->copy_st, e->it_done[slot * nsub + i], 0);
        // The ring is [slot][chain][...]: an iteration's array of all chains is one contiguous block.  iter_major sinks
        // ([iters][nchains][...]) take it with one plain copy per array; chain-major sinks ([nchains][iters][...]) with one
        // strided copy per array (rows = chains).
        if (sink->iter_major) {
            if (sink->signal_cr)
                cerr = cudaMemcpyAsync(sink->signal_cr + 2 * (hs * C * T * n), e->cr_out + 2 * (slot * C * T * n), C * T * n * 16,
                                       cudaMemcpyDeviceToHost, e->copy_st);
            if (sink->fg_amps && m && cerr == cudaSuccess)
                cerr = cudaMemcpyAsync(sink->fg_amps + 2 * (hs * C * T * m), e->fg_out + 2 * (slot * C * T * m), C * T * m * 16,
                                       cudaMemcpyDeviceToHost, e->copy_st);
            if (sink->chisq && cerr == cudaSuccess)
                cerr = cudaMemcpyAsync(sink->chisq + hs * C * T * n, e->chisq_out + slot * C * T * n, C * T * n * 8,
                                       cudaMemcpyDeviceToHost, e->copy_st);
        } else {
            if (sink->signal_cr)
                cerr = copy_rows_d2h(sink->signal_cr + 2 * (hs * T * n), HI * T * n * 16, e->cr_out + 2 * (slot * C * T * n), T * n * 16,
                                     T * n * 16, C, e->copy_st);
            if (sink->fg_amps && m && cerr == cudaSuccess)
                cerr = copy_rows_d2h(sink->fg_amps + 2 * (hs * T * m), HI * T * m * 16, e->fg_out + 2 * (slot * C * T * m), T * m * 16,
                                     T * m * 16, C, e->copy_st);
            if (sink->chisq && cerr == cudaSuccess)
                cerr = copy_rows_d2h(sink->chisq + hs * T * n, HI * T * n * 8, e->chisq_out + slot * C * T * n, T * n * 8, T * n * 8, C,
                                     e->copy_st);
        }
        cudaEventRecord(e->copy_done[slot], e->copy_st);
    }
    // Read-ahead: a call starts with one compute step during which the copy engine has nothing to do (a chunked chain pays it
    // once per chunk: 8 of 57 ms per two-iteration chunk at the headline shape).  With sink.read_ahead the next iterations of
    // the chain are computed into free ring slots now, under this call's last copies; the next call only copies them.
    if (big && cerr == cudaSuccess && sink->read_ahead > 0) {
        int want = sink->read_ahead < (int)R - 1 ? sink->read_ahead : (int)R - 1;
        while (e->ahead < want && e->out_pos + e->ahead < e->cfg.max_iters) {
            compute_next((size_t)(e->out_pos + e->ahead));
            ++e->ahead;
        }
    }
    join_subs(e, subs);
    if (cerr != cudaSuccess) return fail(HP_ERR_CUDA, std::string("hp_engine_run_to_host: ") + cudaGetErrorString(cerr));
    {
        cudaEvent_t ev;
        CU_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        CU_TRY(cudaEventRecord(ev, e->st));
        CU_TRY(cudaStreamWaitEvent(e->copy_st, ev, 0));
        cudaEventDestroy(ev);   // released once the wait has consumed it
    }
    if (niter > 0) {
        const size_t h0 = (size_t)(first - sink->first_iter);
        if (sink->signal_ps)
            CU_TRY(copy_rows_d2h(sink->signal_ps + h0 * n, HI * n * 8, e->ps_out + first * n, I * n * 8, (size_t)niter * n * 8, C,
                                 e->copy_st));
        if (sink->ln_post)
            CU_TRY(copy_rows_d2h(sink->ln_post + h0, HI * 8, e->lnpost_out + first, I * 8, (size_t)niter * 8, C, e->copy_st));
    }
    CU_TRY(cudaStreamSynchronize(e->copy_st));
    CU_TRY(cudaStreamSynchronize(e->st));
    CU_TRY(cudaGetLastError());
    return HP_OK;
}

int hp_engine_set_chain_ids(hp_engine* e, const int* ids) {
    if (!e || !ids) return fail(HP_ERR_ARG, "null argument");
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaMemcpyAsync(e->chain_ids, ids, (size_t)e->C * sizeof(int), cudaMemcpyHostToDevice, e->st));
    CU_TRY(cudaStreamSynchronize(e->st));
    return HP_OK;
}

int hp_engine_set_substreams(hp_engine* e, int n) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);
    e->active_subs = n < 1 ? 1 : n;
    return HP_OK;
}

int hp_engine_set_profile(hp_engine* e, int on) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    e->cfg.profile = on ? 1 : 0;
    return HP_OK;
}

int hp_engine_sync(hp_engine* e) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaStreamSynchronize(e->st));
    CU_TRY(cudaGetLastError());
    return HP_OK;
}
int hp_engine_iterations_done(const hp_engine* e) { return e ? e->iter : -1; }
int hp_engine_rewind(hp_engine* e) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    e->out_pos = 0;
    e->ahead = 0;     // read-ahead iterations stay part of the chain's history (the spectrum state is kept), undelivered
    return HP_OK;
}
long long hp_engine_launch_count(const hp_engine* e) { return e ? e->launches : -1; }
int hp_engine_pt_form(const hp_engine* e, int* low_rank, int* max_rank) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    if (low_rank) *low_rank = e->solve == Solve::PtLowRank ? 1 : 0;
    if (max_rank) *max_rank = e->pt_kcap;
    return HP_OK;
}

int hp_engine_read(hp_engine* e, int c, int buffer, int iter0, int niter, void* dst, size_t dst_bytes) {
    if (!e || !dst) return fail(HP_ERR_ARG, "null argument");
    if (c < 0 || c >= e->C) return fail(HP_ERR_ARG, "chain index out of range");
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaStreamSynchronize(e->st));
    const size_t n = e->n, m = e->m, T = e->T, Tp = e->Tp, Np = e->Np, I = e->cfg.max_iters;
    const bool per_iter = buffer <= HP_BUF_CHISQ;
    if (per_iter && (iter0 < 0 || niter < 0 || (size_t)(iter0 + niter) > I)) return fail(HP_ERR_ARG, "iteration range out of bounds");
    const double* src = nullptr;
    size_t bytes = 0;
    switch (buffer) {
        case HP_BUF_PS: src = e->ps_out + ((size_t)c * I + iter0) * n; bytes = (size_t)niter * n * 8; break;
        case HP_BUF_LNPOST: src = e->lnpost_out + (size_t)c * I + iter0; bytes = (size_t)niter * 8; break;
        case HP_BUF_CR:
        case HP_BUF_FG:
        case HP_BUF_CHISQ: {
            // ring [slot][chain][...]: iteration i lives in slot i % ring until iteration i + ring overwrites it
            const double* base = buffer == HP_BUF_CR ? e->cr_out : (buffer == HP_BUF_FG ? e->fg_out : e->chisq_out);
            if (!base) return fail(HP_ERR_ARG, "this output was not kept (cfg.keep)");
            const size_t R = e->ring;
            const size_t per = buffer == HP_BUF_CR ? 2 * T * n : (buffer == HP_BUF_FG ? 2 * T * m : T * n);   // doubles per iteration
            bytes = (size_t)niter * per * 8;
            if (dst_bytes < bytes) return fail(HP_ERR_ARG, "destination too small");
            if (niter > 0 && (size_t)iter0 + R < (size_t)(e->out_pos + e->ahead))
                return fail(HP_ERR_ARG, "iteration no longer in the device ring (cfg.ring_iters): stream it with hp_engine_run_to_host");
            for (int k = 0; k < niter; ++k) {
                const size_t slot = (size_t)(iter0 + k) % R;
                if (per) CU_TRY(cudaMemcpy((char*)dst + (size_t)k * per * 8, base + (slot * (size_t)e->C + (size_t)c) * per, per * 8, cudaMemcpyDeviceToHost));
            }
            return HP_OK;
        }
        case HP_BUF_LAST_CR:
            if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);
            if (!e->last_sf) return fail(HP_ERR_ARG, "no GCR solve has run yet");
            src = e->last_sf + 2 * (size_t)c * e->last_sf_bs; bytes = T * n * 16; break;
        case HP_BUF_PS_CUR:
            if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);
            src = e->ps + (size_t)c * n; bytes = n * 8; break;
        case HP_BUF_LAST_FG: {
            if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);
            bytes = T * m * 16;
            if (dst_bytes < bytes) return fail(HP_ERR_ARG, "destination too small");
            if (m == 0) return HP_OK;
            CU_TRY(cudaMemcpy2D(dst, m * 16, e->X + 2 * ((size_t)c * Tp * Np + n), Np * 16, m * 16, T, cudaMemcpyDeviceToHost));
            return HP_OK;
        }
        default: return fail(HP_ERR_ARG, "unknown buffer id");
    }
    if (dst_bytes < bytes) return fail(HP_ERR_ARG, "destination too small");
    if (bytes) CU_TRY(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return HP_OK;
}

int hp_engine_set_summary(hp_engine* e, int what, int burn_in, int thin) {
    return hp_engine_set_summary_batched(e, what, burn_in, thin, 0);
}

int hp_engine_set_summary_batched(hp_engine* e, int what, int burn_in, int thin, int batch) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    if (what < 0 || (what & ~(HP_SUMMARY_CR | HP_SUMMARY_FG))) return fail(HP_ERR_ARG, "hp_engine_set_summary: unknown quantity");
    if (burn_in < 0 || thin < 1) return fail(HP_ERR_ARG, "hp_engine_set_summary: needs burn_in >= 0 and thin >= 1");
    if (batch < 0) return fail(HP_ERR_ARG, "hp_engine_set_summary_batched: needs batch >= 0 (0: no batch means)");
    if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);   // read-ahead iterations were computed under the old settings
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaStreamSynchronize(e->st));   // no accumulation in flight
    auto& s = e->sum;
    const size_t C = e->C;
    s.ld_cr = ((long long)e->T * e->n + 1) & ~1LL;
    s.ld_fg = ((long long)e->T * e->m + 1) & ~1LL;
    bool grown = false;
    if ((what & HP_SUMMARY_CR) && !s.cr_mean) {
        CU_TRY(dalloc(&s.cr_mean, 2 * C * s.ld_cr)); CU_TRY(dalloc(&s.cr_m2, C * s.ld_cr));
        grown = true;
    }
    if ((what & HP_SUMMARY_FG) && !s.fg_mean && e->m > 0) {
        CU_TRY(dalloc(&s.fg_mean, 2 * C * s.ld_fg)); CU_TRY(dalloc(&s.fg_m2, C * s.ld_fg));
        grown = true;
    }
    if (batch > 0 && (what & HP_SUMMARY_CR) && !s.cr_snap) {
        CU_TRY(dalloc(&s.cr_snap, 2 * C * s.ld_cr)); CU_TRY(dalloc(&s.cr_m2bm, C * s.ld_cr));
        grown = true;
    }
    if (batch > 0 && (what & HP_SUMMARY_FG) && !s.fg_snap && e->m > 0) {
        CU_TRY(dalloc(&s.fg_snap, 2 * C * s.ld_fg)); CU_TRY(dalloc(&s.fg_m2bm, C * s.ld_fg));
        grown = true;
    }
    if (grown) CU_TRY(cudaStreamSynchronize(0));   // dalloc zeroes on the legacy stream, which the engine's streams do not wait for
    if (s.cr_mean) {
        CU_TRY(cudaMemsetAsync(s.cr_mean, 0, 2 * C * s.ld_cr * sizeof(double), e->st));
        CU_TRY(cudaMemsetAsync(s.cr_m2, 0, C * s.ld_cr * sizeof(double), e->st));
    }
    if (s.fg_mean) {
        CU_TRY(cudaMemsetAsync(s.fg_mean, 0, 2 * C * s.ld_fg * sizeof(double), e->st));
        CU_TRY(cudaMemsetAsync(s.fg_m2, 0, C * s.ld_fg * sizeof(double), e->st));
    }
    if (s.cr_snap) {
        CU_TRY(cudaMemsetAsync(s.cr_snap, 0, 2 * C * s.ld_cr * sizeof(double), e->st));
        CU_TRY(cudaMemsetAsync(s.cr_m2bm, 0, C * s.ld_cr * sizeof(double), e->st));
    }
    if (s.fg_snap) {
        CU_TRY(cudaMemsetAsync(s.fg_snap, 0, 2 * C * s.ld_fg * sizeof(double), e->st));
        CU_TRY(cudaMemsetAsync(s.fg_m2bm, 0, C * s.ld_fg * sizeof(double), e->st));
    }
    s.what = what; s.burn_in = burn_in; s.thin = thin; s.batch = batch; s.seen = 0; s.count = 0;
    return HP_OK;
}

// the refusals shared by hp_engine_read_summary and hp_engine_read_summary_mcse (fn: the caller's name for the messages)
static int check_summary_read(hp_engine* e, int c, int what, const char* fn) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    if (c < 0 || c >= e->C) return fail(HP_ERR_ARG, "chain index out of range");
    if (what != HP_SUMMARY_CR && what != HP_SUMMARY_FG)
        return fail(HP_ERR_ARG, std::string(fn) + ": what must be one HP_SUMMARY_* bit");
    if (!(e->sum.what & what))
        return fail(HP_ERR_ARG, std::string(fn) + ": this quantity is not being accumulated (hp_engine_set_summary)");
    if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);   // the moments include iterations not delivered yet
    return HP_OK;
}

int hp_engine_read_summary(hp_engine* e, int c, int what, double* mean, double* var, size_t bytes_each, int* count) {
    if (int rc = check_summary_read(e, c, what, "hp_engine_read_summary")) return rc;
    const auto& s = e->sum;
    const size_t L = (size_t)e->T * (what == HP_SUMMARY_CR ? e->n : e->m);
    if ((mean && bytes_each < L * 16) || (var && bytes_each < L * 8)) return fail(HP_ERR_ARG, "destination too small");
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaStreamSynchronize(e->st));
    if (count) *count = s.count;
    const double* dmean = what == HP_SUMMARY_CR ? s.cr_mean : s.fg_mean;
    const double* dm2 = what == HP_SUMMARY_CR ? s.cr_m2 : s.fg_m2;
    const size_t ld = what == HP_SUMMARY_CR ? s.ld_cr : s.ld_fg;
    if (L == 0) return HP_OK;
    if (mean) CU_TRY(cudaMemcpy(mean, dmean + 2 * (size_t)c * ld, L * 16, cudaMemcpyDeviceToHost));
    if (var) {
        // var = M2 / count (ddof = 0); zeros before anything was accumulated
        if (s.count == 0) { std::memset(var, 0, L * 8); return HP_OK; }
        CU_TRY(cudaMemcpy(var, dm2 + (size_t)c * ld, L * 8, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < L; ++i) var[i] /= (double)s.count;
    }
    return HP_OK;
}

int hp_engine_read_summary_mcse(hp_engine* e, int c, int what, double* mcse, double* ess, size_t bytes_each, int* nbatch) {
    if (int rc = check_summary_read(e, c, what, "hp_engine_read_summary_mcse")) return rc;
    const auto& s = e->sum;
    if (s.batch <= 0) return fail(HP_ERR_ARG, "hp_engine_read_summary_mcse: batch means are off (hp_engine_set_summary_batched)");
    const size_t L = (size_t)e->T * (what == HP_SUMMARY_CR ? e->n : e->m);
    if ((mcse || ess) && bytes_each < L * 8) return fail(HP_ERR_ARG, "destination too small");
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaStreamSynchronize(e->st));
    const int nb = s.count / s.batch;   // complete batches; a trailing partial batch counts in k and var only
    if (nbatch) *nbatch = nb;
    if (L == 0 || (!mcse && !ess)) return HP_OK;
    if (nb < 2) {
        const double nan = std::nan("");
        for (size_t i = 0; i < L; ++i) {
            if (mcse) mcse[i] = nan;
            if (ess) ess[i] = nan;
        }
        return HP_OK;
    }
    const size_t ld = what == HP_SUMMARY_CR ? s.ld_cr : s.ld_fg;
    std::vector<double> m2(L), m2bm(L);
    CU_TRY(cudaMemcpy(m2.data(), (what == HP_SUMMARY_CR ? s.cr_m2 : s.fg_m2) + (size_t)c * ld, L * 8, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(m2bm.data(), (what == HP_SUMMARY_CR ? s.cr_m2bm : s.fg_m2bm) + (size_t)c * ld, L * 8,
                      cudaMemcpyDeviceToHost));
    // s2_bm = M2_bm / (nb - 1);  mcse^2 = b s2_bm / k;  ess = var / mcse^2 with var = M2 / k as hp_engine_read_summary
    const double k = (double)s.count, b = (double)s.batch;
    for (size_t i = 0; i < L; ++i) {
        const double mcse2 = b * (m2bm[i] / (double)(nb - 1)) / k;
        if (mcse) mcse[i] = std::sqrt(mcse2);
        if (ess) ess[i] = (m2[i] / k) / mcse2;
    }
    return HP_OK;
}

int hp_engine_read_signal_S(hp_engine* e, int c, double* dst) {
    if (!e || !dst) return fail(HP_ERR_ARG, "null argument");
    if (c < 0 || c >= e->C) return fail(HP_ERR_ARG, "chain index out of range");
    if (e->ahead > 0) return fail(HP_ERR_ARG, kAheadMsg);   // the spectrum state is ahead of the delivered iterations
    CU_TRY(cudaSetDevice(e->cfg.device));
    const int n = e->n;
    // S = Fop^H diag(ps / n^2) Fop  (pspec.py:464, 313-322)
    k_scale_vec<<<nblocks(n), 256, 0, e->st>>>(e->vecn + n, e->ps + (size_t)c * n, 1.0 / ((double)n * n), n);
    hp::ZgemmArgs g{};
    g.A = e->Fop; g.sAi = 1; g.sAk = n; g.conjA = 1;
    g.B = e->Fop; g.sBk = n; g.sBj = 1;
    g.C = e->stage; g.sCi = n; g.sCj = 1;
    g.dk = e->vecn + n;
    g.M = n; g.N = n; g.K = n; g.alpha = 1.0; g.batch = 1;
    hp::launch_zgemm(g, e->st);
    CU_TRY(cudaStreamSynchronize(e->st));
    CU_TRY(cudaMemcpy(dst, e->stage, 2 * (size_t)n * n * sizeof(double), cudaMemcpyDeviceToHost));
    return HP_OK;
}

int hp_engine_info(hp_engine* e, int* info_host) {
    if (!e || !info_host) return fail(HP_ERR_ARG, "null argument");
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaStreamSynchronize(e->st));
    CU_TRY(cudaMemcpy(info_host, e->info, e->C * sizeof(int), cudaMemcpyDeviceToHost));
    return HP_OK;
}

int hp_engine_kernel_ms(hp_engine* e, double* ms, int* launches, int reset) {
    if (!e) return fail(HP_ERR_ARG, "null engine");
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaStreamSynchronize(e->st));
    for (size_t i = 0; i < e->ev_cls.size(); ++i) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, e->ev[2 * i], e->ev[2 * i + 1]) == cudaSuccess) e->ms_acc[e->ev_cls[i]] += t;
        cudaEventDestroy(e->ev[2 * i]); cudaEventDestroy(e->ev[2 * i + 1]);
    }
    e->ev.clear(); e->ev_cls.clear();
    for (int i = 0; i < HP_NUM_KERNEL_CLASSES; ++i) {
        if (ms) ms[i] = e->ms_acc[i];
        if (launches) launches[i] = e->launch_acc[i];
        if (reset) { e->ms_acc[i] = 0; e->launch_acc[i] = 0; }
    }
    return HP_OK;
}

int hp_sample_S(int device, int T, int n, const double* s, const double* prior, const double* draws, double* out) {
    if (!s || !draws || !out || T < 2 || n < 1) return fail(HP_ERR_ARG, "hp_sample_S: bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(HP_ERR_CUDA, "no CUDA device: hydra_pspec_b200 has no CPU fallback");
    CU_TRY(cudaSetDevice(device));
    double *U, *S, *Sk, *Eu, *pr, *dr, *ps, *lam, *lnp1, *psout, *lnp;
    CU_TRY(dalloc(&U, 2 * (size_t)n * n)); CU_TRY(dalloc(&S, 2 * (size_t)T * n)); CU_TRY(dalloc(&Sk, 2 * (size_t)T * n));
    CU_TRY(dalloc(&Eu, n)); CU_TRY(dalloc(&pr, 2 * (size_t)n)); CU_TRY(dalloc(&dr, n)); CU_TRY(dalloc(&ps, n));
    CU_TRY(dalloc(&lam, n + 64)); CU_TRY(dalloc(&lnp1, T)); CU_TRY(dalloc(&psout, n)); CU_TRY(dalloc(&lnp, 1));
    hp::launch_fourier_operator(U, n, 1.0 / std::sqrt((double)n), 0);
    CU_TRY(cudaMemcpy(S, s, 2 * (size_t)T * n * sizeof(double), cudaMemcpyHostToDevice));
    if (prior) CU_TRY(cudaMemcpy(pr, prior, 2 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(dr, draws, n * sizeof(double), cudaMemcpyHostToDevice));
    hp::ZgemmArgs t{};
    t.A = S; t.sAi = n; t.sAk = 1;
    t.B = U; t.sBk = 1; t.sBj = n;
    t.C = Sk; t.sCi = n; t.sCj = 1;
    t.M = T; t.N = n; t.K = n; t.alpha = 1.0; t.batch = 1;
    hp::launch_zgemm(t, 0);
    hp::launch_colsumsq(Sk, Eu, T, T, n, 1, 0);
    hp::SampleArgs sp{};
    sp.Eu = Eu; sp.lnp1 = lnp1; sp.prior = pr; sp.draws = dr; sp.draws_bs = n;
    sp.ps = ps; sp.lam = lam; sp.ps_out = psout; sp.ps_bs = n; sp.lnpost_out = lnp; sp.lnpost_bs = 1;
    sp.n = n; sp.Np = n; sp.T = T; sp.Tp = T; sp.ntiles = 0; sp.nsys = 1; sp.beta_mode = 1; sp.philox = 0;
    hp::launch_sample(sp, 0);
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpy(out, psout, n * sizeof(double), cudaMemcpyDeviceToHost));
    double* ptrs[] = {U, S, Sk, Eu, pr, dr, ps, lam, lnp1, psout, lnp};
    for (double* p : ptrs) cudaFree(p);
    return HP_OK;
}

int hp_fourier_operator(int device, int n, double* out) {
    if (!out || n < 1) return fail(HP_ERR_ARG, "hp_fourier_operator: bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(HP_ERR_CUDA, "no CUDA device: hydra_pspec_b200 has no CPU fallback");
    CU_TRY(cudaSetDevice(device));
    double* d;
    CU_TRY(dalloc(&d, 2 * (size_t)n * n));
    hp::launch_fourier_operator(d, n, 1.0, 0);
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpy(out, d, 2 * (size_t)n * n * sizeof(double), cudaMemcpyDeviceToHost));
    cudaFree(d);
    return HP_OK;
}

}  // extern "C"
