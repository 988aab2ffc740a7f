// hp_kernels.cuh -- launch interfaces of the sm_100a kernels (definitions in hp_kernels.cu).
//
// Conventions
//   * complex128 arrays in global memory are interleaved (re, im) doubles == numpy complex128.
//   * "packed lower-block" matrices (G, L): 32x32 blocks, block (i, j), j <= i, at block index
//     i (i+1)/2 + j; each block is 2048 doubles: a 32x32 row-major real plane followed by the
//     imaginary plane.  Diagonal blocks of G hold both triangles.  The factor L and the inverses of its
//     diagonal blocks use the same block order with rows padded to 36 doubles, so that one block is
//     one TMA bulk copy into its bank-conflict-free shared-memory layout.
//   * system vectors are padded to Np = 32 * nblk rows; times are padded to Tp = 16 * ntiles.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace hp {

constexpr int kNB = 32;                 // block edge of the packed format
constexpr int kBlkDoubles = 2 * 32 * 32;  // doubles per packed block of G (16 KiB)
constexpr int kLdBlk = 36;               // row stride (doubles) of a 32x32 plane of an L block, == 4 mod 16
constexpr int kLPlane = 32 * kLdBlk;     // doubles per plane of an L block
constexpr int kLBlkDoubles = 2 * kLPlane;  // L / L^-1 blocks are stored in the padded shared-memory layout (18 KiB)
constexpr int kTT = 16;                 // right-hand sides (times) per solve CTA
constexpr int kInvGrid = 1000;          // pspec.py:11 ngrid default

// cudaFuncSetAttribute is per device: the launch wrappers cache what they have set per device ordinal
constexpr int kMaxDev = 64;
inline int current_device_slot() {
    int d = 0;
    cudaGetDevice(&d);
    return (d < 0 || d >= kMaxDev) ? 0 : d;
}

__host__ __device__ inline size_t tri_blocks(int nblk) { return (size_t)nblk * (nblk + 1) / 2; }
__host__ __device__ inline size_t blk_index(int i, int j) { return (size_t)i * (i + 1) / 2 + j; }

// ---- generic strided batched complex GEMM:  C[b] (+)= alpha * opA(A[b]) * opB(B[b]) ----------
struct ZgemmArgs {
    const double* A; long long sAi, sAk, bsA;   // strides in complex elements
    const double* B; long long sBk, sBj, bsB;
    double* C;       long long sCi, sCj, bsC;
    const double* dk; long long bsD;            // optional real scale of index k (A side), or null
    int M, N, K;
    int conjA, conjB, accumulate;
    double alpha;
    int batch;
    int tri;   // 0: dense B;  1: B[k][j] = 0 for k > j;  2: B[k][j] = 0 for k < j  (the zero K range of a column tile is skipped)
    int lower_out;   // 1: only the 64 x 64 tiles of C that touch the lower triangle (j <= i) are computed (Hermitian result)
};
void launch_zgemm(const ZgemmArgs& a, cudaStream_t st);

// Fop[k][x] = exp(-2 pi i (k - n/2)(x - n/2) / n) * scale   (utils.py:14-40), n x n interleaved
void launch_fourier_operator(double* out, int n, double scale, cudaStream_t st);

// dense (N x N interleaved, leading dim ld, batch stride bs) -> packed lower blocks, zero padded
void launch_pack_lower(const double* dense, long long ld, long long bs, double* packed, int N, int nblk,
                       int batch, cudaStream_t st);

// ---- per-iteration kernels ---------------------------------------------------------------
// Identity of a launch's Philox draws: the key (the engine seed), the draw counter and the global chain id of every
// system, chain_ids[nsys] (read only when the kernel draws).  Each kernel builds its own counters from it.
struct DrawKey { uint32_t key0, key1, iter; const int* chain_ids; };

struct CholArgs {
    const double* Gp;      // [nsys][tri_blocks][2048]
    const double* lam;     // [nsys][Np]   (lambda for rows < n, 1 for fg rows, 0 for padding)
    double* Lp;            // [nsys][tri_blocks][2304]
    double* Linvp;         // [nsys][nblk][2304]
    int* info;             // [nsys]  0 ok, k+1 = non-positive pivot in block column k
    int nblk, n, N, nsys;
};
// Further copies of W = L^-1 that launch_chol_trinv writes besides Wp, each optional (null: not written):
//   ex.Wf1 / ex.Wf2: fragment-major copies for k_solve3 (hp_solve3.cu: Wf1 = pass-1 operand, scaled by lam when ex.lam is
//           given (lam: [nsys][Np]); Wf2 = W in pass-2 (transposed) fragment order), [nsys][solve3_frag_doubles]
struct TrinvExtra { double* Wf1; double* Wf2; const double* lam; };
// M = L L^H and W = L^-1 (Wp: the padded block layout of L, [nsys][tri_blocks][2304]) in one sequence of block-column
// launches of k_chol_w: the panel launch of column k also carries row k of W.  Returns the number of launches (1 for
// nblk = 1, otherwise nblk + 1).
int launch_chol_trinv(const CholArgs& a, double* Wp, const TrinvExtra& ex, cudaStream_t st);

struct SolveArgs {
    const double* Wp;      // [nsys][tri_blocks][2304]  W = L^-1 (launch_chol_trinv)
    const double* lam;     // [nsys][Np]
    const double* Rfix;    // [nsys][Tp][Np] complex: B^H N^-1 (w d)   (+ frozen noise term in numpy mode)
    const double* wa;      // [nsys][Tp][Np] complex or null: Q^H omega_a (rows < n)
    double* X;             // [nsys][Tp][Np] complex: solution [ytilde ; f]
    double* Ssc;           // [nsys][Tp][n]  complex: lambda * ytilde (signal in the S eigenbasis)
    double* Ppart;         // [nsys][ntiles][n] sum over the tile's times of |ytilde|^2
    int nblk, n, N, Tp, ntiles, nsys;
    int T;                 // valid times (t >= T are padding: zero RHS)
    int philox_wa;         // 1: add xi ~ CN(0, I) (Philox) to y = L^-1 r before the backward pass
    int stages;            // ring depth (set by launch_solve)
    int rows_per_round;    // times staged through the ring area per round (set by launch_solve)
    int cg_compat;         // 1: scale each column by the scalar CG model (hp_math.h:cg_theta)
    DrawKey dk;
};
void launch_solve(const SolveArgs& a, cudaStream_t st);
size_t solve_smem_bytes(int nblk);
bool solve_resident_ok(int nblk, size_t max_smem);   // false: use the dense-product solve (N > 576)

// ---- k_solve3 (hp_solve3.cu): independent warps, W fragments streamed from L2 into registers ------------------------
constexpr int kS3Warps = 16;         // warps of a k_solve3 CTA (all of them compute): four per scheduler hide the L2 latency
constexpr int kS3MaxStrips = 28;     // 16-row strips of the system (Np <= 448: two shared-memory tiles)
constexpr int kS3MaxPerWarp = 8;
struct Solve3Sched {                 // per pass and warp: the strips it owns, longest first (solve3_make_schedule)
    uint8_t n[2][kS3Warps];
    uint8_t strip[2][kS3Warps][kS3MaxPerWarp];
};
struct Solve3Args {
    const double* Wf1;     // [nsys][solve3_frag_doubles] pass-1 operand in fragment-major order (W, or W diag(lam))
    const double* Wf2;     // [nsys][solve3_frag_doubles] pass-2 operand (W, transposed fragment order)
    const double* Rt;      // [nsys][ntiles][nblk][2][32][16] right-hand sides in tile layout (k_rhs_tile)
    double* X;             // [nsys][Tp][Np] complex
    double* Ppart;         // [nsys][ntiles][n]
    int nblk, n, N, Tp, ntiles, nsys, T;
    int philox;
    DrawKey dk;
    int grid_limit;        // > 0: cap on the persistent grid (sub-batches sharing the GPU); 0 = one CTA per SM
    int nstrip;            // 16-row strips holding rows of the system, ceil(N / 16) (0: all 2 nblk); must match the schedule
    Solve3Sched sched;
};
void launch_solve3(const Solve3Args& a, cudaStream_t st);
bool solve3_ok(int nblk, size_t max_smem);
size_t solve3_frag_doubles(int nblk);               // doubles per system of Wf1 (and of Wf2)
void solve3_make_schedule(int nblk, Solve3Sched* sc, int nstrip = 0);
void launch_rhs_tile(double* Rt, const double* Rfix, const double* wa, const double* lam, int nblk, int n, int N, int T, int Tp,
                     int ntiles, int nsys, cudaStream_t st);
// scalar model of the reference's truncated CG applied to the global solution X (k_solve3, the dense-product solve)
void launch_cg_scale(double* X, const double* Rfix, const double* wa, const double* lam, int n, int N, int Np, int T, int Tp,
                     int nsys, cudaStream_t st);

struct PostArgs {
    const double* Sf;      // [nsys][>=T][n] complex: signal in frequency space (rows t < T are read)
    long long sf_bs;       // batch stride of Sf in complex elements
    const double* X;       // [nsys][Tp][Np]
    const double* Ft;      // [nsys][m][n] complex: fgmodes transposed
    const double* wd;      // [nsys][Tp][n] complex: flags * vis
    const double* w;       // [nsys][n] 0/1
    const double* ninvd;   // [nsys][n] diag(Ninv) (real part)
    double* fg_out;        // [nsys][T][m] complex or null
    double* chisq_out;     // [nsys][T][n] or null
    double* Wm;            // [nsys][Tp][n] complex: w * s   (or null when no channel is flagged)
    double* Rm;            // [nsys][Tp][n] complex: w * resid (dense-noise ln_post) or null
    double* lnp1;          // [nsys][Tp]: sum_x w ninv |resid|^2  (diagonal noise)
    int n, m, Np, T, Tp, nsys;
    long long fg_bs, chisq_bs;  // batch strides (doubles) of the output slots
};
void launch_post(const PostArgs& a, cudaStream_t st);

// out[sys][k] = sum_t |A[sys][t][k]|^2 over t < T   (rows of A are ld complex elements apart; ld = 0 -> n)
void launch_colsumsq(const double* A, double* out, int T, int Tp, int n, int nsys, cudaStream_t st, int ld = 0);

// ---- per-time flags (hp_pertime.cu): one factorisation + solve per (system, time) -------------
struct PtArgs {
    const double* H;       // [nsys][Tp][1 + m][Np] complex: column 0 = chat_t (first n entries), column 1 + j =
                           //   [Q|F]^H (w_t N^-1) F[:, j]
    const double* lam;     // [nsys][Np]
    const double* Rfix;    // [nsys][Tp][Np] complex
    const double* wa;      // [nsys][Tp][Np] complex or null
    double* X;             // [nsys][Tp][Np] complex: solution [ytilde ; f]
    double* scratch;       // [grid][pt_scratch_doubles_per_cta]: factor L and the inverses of its diagonal blocks
    const int* same_prev;  // [nsys][Tp] or null: 1 = the flags of time t equal those of t - 1 (the factor is re-used)
    int* info;             // [nsys], zeroed by the caller; atomicMax(k + 1) on a non-positive pivot in block column k
    int nblk, n, m, N, T, Tp, nsys;
    int philox_wa;
    DrawKey dk;
};
size_t pt_smem_bytes(int nblk, int n);
size_t pt_scratch_doubles_per_cta(int nblk);
int pt_grid(int nsys, int T);   // persistent grid: 2 CTAs per SM, at most one per (system, time) pair
void launch_pt_cholsolve(const PtArgs& a, int grid, cudaStream_t st);

// ---- per-time flags, low-rank form (hp_ptlow.cu): M_t = M_0 - V_t^H V_t with M_0 the system of the channels that are
// unflagged at any time (one shared factorisation, k_solve3) and V_t the k_t rows of the channels flagged at time t only.
//   x_t = x0_t + R_f K_t^-1 ((R^H b_t)_f [+ L_K zeta]),   K_t = I - P_ff = L_K L_K^H,   R = M_0^-1 A,   P = A^H R
// A = D [Q|F]^H sqrt(wbar N^-1) rides through k_solve3 as n extra right-hand sides (rows Tp0 .. Tp0 + n of Rfix / X).
constexpr int kPtLowMaxRank = 64;     // channels flagged at one time beyond the all-times mask; more -> k_pt_cholsolve
struct PtLowArgs {
    const double* Rfix;    // [nsys][Tp][Np] complex: rows t < T right-hand sides (unscaled), rows Tp0 + x the columns of A / D
    const double* wa;      // [nsys][Tp][Np] complex or null (injected draws)
    const double* lam;     // [nsys][Np]
    double* X;             // [nsys][Tp][Np] complex: rows t < T hold x0_t (in) / x_t (out); rows Tp0 + x hold R[:, x]
    const double* Pm;      // [nsys][n][n] complex, P = A^H R (lower triangle read)
    const uint16_t* fidx;  // [nsys][T][kPtLowMaxRank] channels flagged at time t only
    const int* fcnt;       // [nsys][T]
    int* info;             // [nsys]: atomicMax(nblk + 1) when a K_t is not positive definite
    int n, N, Np, T, Tp, Tp0, nsys, nblk, kcap;   // kcap: largest count in fcnt (shared-memory sizing)
    int philox;
    DrawKey dk;
};
size_t pt_lowrank_smem_bytes(int kcap, int warps);
void launch_pt_lowrank(const PtLowArgs& a, cudaStream_t st);
// Rfix rows Tp0 + x = sqrt(ni[x]) conj(Bmat[x][:]) for one system
void launch_pt_arows(double* Rfix_sys, const double* Bmat_sys, const double* ni_sys, int n, int Np, int Tp0, cudaStream_t st);

struct SampleArgs {
    const double* Ppart;   // [nsys][ntiles][n]  (beta_mode 0)
    const double* Eu;      // [nsys][n]: sum_t |U s|^2 (beta_mode 1: general-basis iteration)
    const double* Em;      // [nsys][n]: sum_t |U (w s)|^2, or null (no flags: = beta / n)
    const double* lnp1;    // [nsys][Tp]
    const double* lnp1_dense;  // [nsys][Tp] or null: dense-noise residual term (replaces lnp1)
    const double* prior;   // [nsys][2][n]  (pspec.py:84: [0]=upper, [1]=lower)
    const double* draws;   // [nsys][n] injected: uniform u for prior bins, 1/gammainccinv(alpha,u) otherwise
    double* ps;            // [nsys][n] in: current spectrum (beta_mode 0), out: new sample
    double* lam;           // [nsys][Np] out: sqrt(ps/n) for rows < n
    double* ps_out;        // [nsys][n] output slot
    double* lnpost_out;    // [nsys] output slot
    int n, Np, T, Tp, ntiles, nsys;
    int beta_mode, philox;
    int ntilesE;           // > 0: Em / Eu are per-tile partial sums [nsys][ntilesE][n]
    DrawKey dk;
    long long ps_bs, lnpost_bs, draws_bs;
};
void launch_sample(const SampleArgs& a, cudaStream_t st);

// ---- fused FFT kernels (hp_fft.cu) ----------------------------------------------------------
struct FftPlan { int n, nf; int radix[16]; uint32_t magic[16]; };  // magic[p] = ceil(2^32 / Ns_p)
bool make_fft_plan(int n, FftPlan* plan);          // false: n has a prime factor > 31 (dense fallback)
void launch_twiddles(double* tw, int n, cudaStream_t st);  // tw[j] = exp(-2 pi i j / n), interleaved
int postfft_ktp(int n, int m, size_t max_smem);   // times per CTA (8 or 4) that fit shared memory, 0 = none
int postfft_tiles(int T, int ktp);
size_t postfft_smem_bytes(int n, int m, int ktp);

struct PostFftArgs {
    FftPlan plan;
    const double* tw;
    const double* tw2;     // k_post_fft2: per-pass twiddle tables of the forward plan ([0, n)) and of the reverse plan ([n, 2 n)),
                           //   built once per engine (launch_fft2_tables)
    const double* X;       // [nsys][Tp][Np]
    const double* lam;     // [nsys][Np]
    double* Sf;            // [nsys][..][n] frequency-space signal: written (do_inverse) or read
    long long sf_bs;
    const double* Ft;      // [nsys][m][n]
    const double* wd; const double* w; const double* ninvd;
    long long w_bs, w_ts;  // w[sys * w_bs + t * w_ts + x]: (n, 0) time-invariant flags, (Tp n, n) per-time flags
    double* fg_out; double* chisq_out; long long fg_bs, chisq_bs;
    double* lnp1;          // [nsys][Tp]
    double* Rm;            // [nsys][Tp][n] complex or null: w * resid (dense noise: ln_post term via k_zgemm2)
    double* Empart;        // [nsys][tiles][n] or null
    double* Eupart;        // [nsys][tiles][n] or null
    int m, Np, T, Tp, nsys, do_inverse;
    int ktp;               // times per CTA (postfft_ktp)
};
void launch_post_fft(const PostFftArgs& a, cudaStream_t st);
// k_post_fft2 (hp_fft2.cu): register-resident FFTs, one shared-memory buffer; needs do_inverse = 1 and Eupart = NULL
bool postfft2_ok(int n);   // false: Nfreqs not covered (k_post_fft takes it)
size_t postfft2_smem_bytes(int n, int m);
void launch_post_fft2(const PostFftArgs& a, cudaStream_t st);   // a.plan.n: an Nfreqs of postfft2_ok
void launch_fft2_tables(double* tw2, const double* tw, int n, cudaStream_t st);   // tw2: 4 n doubles; n: an Nfreqs of postfft2_ok

// k_moments (hp_moments.cu): Welford update of per-chain posterior moments from one iteration's samples.
// Element i < L of chain c is src[c * src_cs + (i / w) * rs + i % w] (complex); its accumulators are mean[c * ld + i]
// (complex) and m2[c * ld + i] (real), ld even.  src = NULL or L = 0: nothing to update.
struct MomentsArr {
    const double* src; long long src_cs; int w, rs;
    int L, nsys; long long ld;
    double* mean; double* m2;
};
// one launch for both arrays (returns the number of launches, 0 or 1); invk = 1 / (accumulated iterations including this one)
int launch_moments(const MomentsArr& cr, const MomentsArr& fg, double invk, cudaStream_t st);
// k_moments_batch: the same update, then the close of batch j of the batch means.  snap[c * ld + i] (complex) is the mean at
// the previous batch boundary, m2[c * ld + i] (real) the batch means' sum of squared deviations; same layout as MomentsArr.
struct MomentsBatch {
    double* snap; double* m2;
};
// jj1 = j (j - 1); launches as launch_moments (0 or 1)
int launch_moments_batch(const MomentsArr& cr, const MomentsArr& fg, const MomentsBatch& crb, const MomentsBatch& fgb,
                         double invk, double jj1, cudaStream_t st);

}  // namespace hp
