/* hydra_pspec_b200.h -- C ABI of the B200 Gibbs hot path (libhydra_pspec_b200.so).
 *
 * This is the boundary a maintainer of HydraRadio/hydra-pspec would bind (ctypes stub in
 * INTEGRATION.md).  The reference is pure Python, so each entry point names the Python
 * function(s) whose work it takes over (paths relative to the reference checkout).
 *
 * Conventions: plain pointers and sizes only.  complex128 arrays are interleaved (re, im)
 * doubles in C order, i.e. exactly the memory of a numpy complex128 array.  All pointers are
 * HOST pointers unless the name ends in _dev.  Every function returns 0 on success or a
 * negative hp_status; hp_last_error() gives the message.  There is no CPU fallback: every
 * compute entry point needs a CUDA device and fails with HP_ERR_CUDA otherwise.
 */
#ifndef HYDRA_PSPEC_B200_H
#define HYDRA_PSPEC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hp_engine hp_engine;

enum hp_status { HP_OK = 0, HP_ERR_ARG = -1, HP_ERR_CUDA = -2, HP_ERR_SIZE = -3, HP_ERR_NUMERIC = -4 };

enum hp_rng_mode {
    HP_RNG_INJECTED = 0, /* draws supplied by the host: the reference's numpy streams */
    HP_RNG_PHILOX = 1    /* device counter-based Philox4x32-10 */
};

/* outputs kept per iteration (ps and ln_post are always kept) */
enum hp_keep { HP_KEEP_CR = 1, HP_KEEP_FG = 2, HP_KEEP_CHISQ = 4 };

/* buffers readable with hp_engine_read */
enum hp_buffer {
    HP_BUF_PS = 0,      /* [iters][Nfreqs]            double     signal_ps   (pspec.py:592) */
    HP_BUF_LNPOST = 1,  /* [iters]                    double     ln_post     (pspec.py:596) */
    HP_BUF_CR = 2,      /* [iters][Ntimes][Nfreqs]    complex128 signal_cr   (pspec.py:590) */
    HP_BUF_FG = 3,      /* [iters][Ntimes][Nmodes]    complex128 fg_amps     (pspec.py:593) */
    HP_BUF_CHISQ = 4,   /* [iters][Ntimes][Nfreqs]    double     chisq       (pspec.py:595) */
    HP_BUF_LAST_CR = 5, /* [Ntimes][Nfreqs]           complex128 signal part of the last GCR solve */
    HP_BUF_LAST_FG = 6, /* [Ntimes][Nmodes]           complex128 fg amplitudes of the last GCR solve */
    HP_BUF_PS_CUR = 7   /* [Nfreqs]                   double     current delay spectrum */
};

typedef struct hp_config {
    int device;          /* CUDA device ordinal */
    int nchains;         /* baselines resident in this engine (independent chains) */
    int ntimes, nfreqs, nmodes;
    int rng_mode;        /* hp_rng_mode */
    int cg_compat;       /* 1: reproduce the reference's truncated CG (pspec.py:228) through the
                            scalar model in csrc/hp_math.h; 0: exact solve */
    int refresh_omega;   /* Philox only. 1: new GCR fluctuation draws every iteration; 0: the same
                            white draws in every iteration (the reference re-uses its draws,
                            pspec.py:195-197) */
    int keep;            /* hp_keep bitmask */
    int max_iters;       /* capacity of the per-iteration output buffers */
    int general_basis0;  /* 1: S_initial is not delay-diagonal; hp_engine_load_chain gets its
                            eigenvectors (first iteration runs in that basis) */
    int profile;         /* 1: record per-kernel CUDA-event timings (hp_engine_kernel_ms) */
    int substreams;      /* > 1: advance the chains as this many independent sub-batches on separate streams
                            (overlaps one sub-batch's factorisation / FFT kernels with another's solve) */
    int dense_noise;     /* 1: chains are loaded with hp_engine_load_chain_dense (non-diagonal N^-1) */
    int force_dense_transforms; /* 1: apply the Fourier operator as dense products even when Nfreqs has
                            an FFT plan (the path used for Nfreqs with a prime factor > 31); tests */
    int force_dense_solve; /* 1: run the GCR solve as dense products with W = L^-1 even when the shared-memory
                            resident k_solve tile fits (the path Nfreqs + Nmodes > 576 takes in any case); with
                            time_flags = 1: one factorisation per time (csrc/hp_pertime.cu) instead of the
                            low-rank form; tests */
    int time_flags;      /* 1: flags are per time, [Ntimes][Nfreqs] (an extension: the reference collapses them to
                            "flagged at any time", run-hydra-pspec.py:520-526).  hp_engine_pt_form reports which
                            form of the per-time solve runs.  Needs diagonal noise, cg_compat = 0 */
    int ring_iters;      /* device slots of the big per-iteration outputs (signal_cr, fg_amps, chisq): 0 = max_iters
                            (every iteration stays readable with hp_engine_read); R > 0: a ring of R slots, iteration i
                            lives in slot i % R until iteration i + R overwrites it.  hp_engine_run_to_host streams
                            every iteration out before its slot is reused, so the device footprint does not grow with
                            the chain length (the reference holds one baseline's Niter samples in host RAM,
                            pspec.py:590-596, 625-636) */
    uint64_t seed;       /* Philox key */
    void* stream;        /* cudaStream_t to launch on, or NULL for an engine-owned stream */
} hp_config;

/* Number of kernel classes reported by hp_engine_kernel_ms and their names. */
#define HP_NUM_KERNEL_CLASSES 6
const char* hp_kernel_class_name(int cls);

int hp_engine_create(const hp_config* cfg, hp_engine** out);
int hp_engine_destroy(hp_engine* e);

/* Load one baseline (replaces the per-baseline set-up of gibbs_sample_with_fg, pspec.py:493-599,
 * and the iteration-independent half of build_matrices, pspec.py:325-374).
 *   vis        [Ntimes][Nfreqs] complex128  visibilities (NOT pre-multiplied by the flags)
 *   flags      [Nfreqs] uint8, 1 = unflagged (pspec.py:520-522); [Ntimes][Nfreqs] when cfg.time_flags = 1
 *   fgmodes    [Nfreqs][Nmodes] complex128
 *   ninv_diag  [Nfreqs] diagonal of the inverse noise covariance
 *   basis0     general_basis0 ? [Nfreqs][Nfreqs] complex128 eigenvectors (columns) of S_initial : NULL
 *   lam0sq     [Nfreqs] eigenvalues of S_initial in that basis; for a delay-diagonal S_initial
 *              these are diag(U S U^H) with U = fourier_operator(Nfreqs)/sqrt(Nfreqs)
 *   ps_prior   [2][Nfreqs] (pspec.py:84-86; [0] upper, [1] lower; 0 = no prior)
 * The host arrays may be reused as soon as the call returns.  With diagonal noise and time-invariant flags the Gram
 * matrix and right-hand-side products of the loaded chains are built lazily, for all pending chains in one batched
 * launch, by the first hp_engine_run / hp_engine_run_to_host / hp_engine_gcr / hp_engine_set_draws that follows.
 */
int hp_engine_load_chain(hp_engine* e, int chain, const double* vis, const uint8_t* flags, const double* fgmodes,
                         const double* ninv_diag, const double* basis0, const double* lam0sq,
                         const double* ps_prior);

/* Same with a non-diagonal inverse noise covariance (cfg.dense_noise = 1):
 *   ninv_diag  [Nfreqs] real diagonal of N^-1 (the reference's chi^2 weights, pspec.py:452)
 *   ninv_dense [Nfreqs][Nfreqs] complex128 Hermitian N^-1; the flags are applied to rows and columns
 *   nih_dense  [Nfreqs][Nfreqs] complex128 principal square root of the flagged N^-1 (pspec.py:362);
 *              only read in HP_RNG_INJECTED mode, NULL otherwise (the Philox path never needs it)
 */
int hp_engine_load_chain_dense(hp_engine* e, int chain, const double* vis, const uint8_t* flags, const double* fgmodes,
                               const double* ninv_diag, const double* ninv_dense, const double* nih_dense,
                               const double* basis0, const double* lam0sq, const double* ps_prior);

/* Same with a diagonal inverse noise covariance per time (an extension: the reference's build_matrices takes one N^-1,
 * pspec.py:361).  Needs cfg.time_flags = 1 and diagonal noise (cfg.dense_noise = 0), otherwise HP_ERR_ARG.
 *   flags      [Ntimes][Nfreqs] uint8, 1 = unflagged
 *   ninv_t     [Ntimes][Nfreqs] diag(N_t^-1) of every time, finite and >= 0 (HP_ERR_ARG otherwise); time t uses
 *              w_t N_t^-1 in the GCR system and N_t^-1 as its chi^2 / ln-posterior weight
 * A chain loaded this way runs one factorisation per time (csrc/hp_pertime.cu) and puts the whole engine on that form
 * (hp_engine_pt_form reports it); times whose flags and weights equal those of the time before re-use its factor.
 * Reloading the chain with hp_engine_load_chain removes the per-time noise; the engine returns to the low-rank form when no
 * chain has it and no time exceeds that form's rank.  A general basis0 (cfg.general_basis0) is refused with HP_ERR_SIZE.
 * The per-time weights of all chains (8 Ntimes Nfreqs bytes per chain, times padded to 16) are allocated, outside the
 * creation-time arena, when the first chain is loaded this way.
 */
int hp_engine_load_chain_time_noise(hp_engine* e, int chain, const double* vis, const uint8_t* flags, const double* fgmodes,
                                    const double* ninv_t, const double* basis0, const double* lam0sq,
                                    const double* ps_prior);

/* Injected draws (HP_RNG_INJECTED).
 *   omega_a, omega_b [Ntimes][Nfreqs] complex128: the unit complex Gaussians of pspec.py:215-217
 *                    (NULL, NULL = map_estimate, pspec.py:210-212)
 *   s_draws [max_iters][Nfreqs]: per iteration and delay bin, the uniform u of pspec.py:58 for
 *                    prior-bounded bins, or the invgamma(a = Ntimes-1) variate of pspec.py:125 otherwise
 */
int hp_engine_set_draws(hp_engine* e, int chain, const double* omega_a, const double* omega_b,
                        const double* s_draws, int n_draw_iters);

/* Run `niter` Gibbs iterations (gibbs_step_fgmodes, pspec.py:377-490) for all chains.
 * Asynchronous on the engine's stream. */
int hp_engine_run(hp_engine* e, int niter);
/* Host destinations of the sample arrays (page-locked memory recommended: hp_pinned_alloc).  Layout
 * [nchains][iters][...] with the shapes listed under enum hp_buffer -- or [iters][nchains][...] for the big arrays, see
 * iter_major; NULL = not wanted. */
typedef struct hp_host_sink {
    double* signal_ps; double* ln_post; double* signal_cr; double* fg_amps; double* chisq;
    int iters;           /* capacity (second dimension) of the host arrays */
    int first_iter;      /* iteration index stored in host slot 0: iteration i lands in slot i - first_iter.  A bounded
                            staging area is re-used chunk after chunk by advancing first_iter (0 = whole chain) */
    int iter_major;      /* 0: signal_cr / fg_amps / chisq host arrays are [nchains][iters][...] (one strided copy per array and
                            iteration); 1: [iters][nchains][...] -- an iteration's array of all chains is then one contiguous block
                            on both sides and leaves with one plain copy (full PCIe rate).  signal_ps / ln_post are always
                            [nchains][iters][...] */
    int read_ahead;      /* > 0: before returning, compute up to this many further iterations of the chain (at most ring_iters - 1)
                            into free device ring slots, under the call's last device-to-host copies; the next
                            hp_engine_run_to_host then starts copying at once instead of waiting for its first compute step.
                            The samples are unchanged (same draws, same order).  While read-ahead iterations are pending the
                            chain state is ahead of the delivered iterations: hp_engine_run / _gcr / _load_chain / _set_draws /
                            _read_signal_S refuse to run; pass read_ahead = 0 in the last call of a chain (or hp_engine_rewind) */
} hp_host_sink;
/* hp_engine_run + copy-out: every iteration's arrays are streamed to the host on a second stream
 * while the next iteration computes.  Returns when everything has landed. */
int hp_engine_run_to_host(hp_engine* e, int niter, const hp_host_sink* sink);
/* Only the GCR step (gcr_fgmodes, pspec.py:238-310) with the current spectrum; results in
 * HP_BUF_LAST_CR / HP_BUF_LAST_FG. */
int hp_engine_gcr(hp_engine* e);
int hp_engine_sync(hp_engine* e);
int hp_engine_iterations_done(const hp_engine* e);
/* Reset the iteration counter / output cursor (the spectrum state is kept). */
int hp_engine_rewind(hp_engine* e);

/* Copy results to the host.  iter0/niter select iterations for the per-iteration buffers. */
int hp_engine_read(hp_engine* e, int chain, int buffer, int iter0, int niter, void* dst, size_t dst_bytes);

/* Posterior moments accumulated on the device (csrc/hp_moments.cu).  Instead of streaming every sample of signal_cr /
 * fg_amps to the host and reducing it there, the engine keeps a running mean and variance per (chain, time, channel) and
 * (chain, time, mode), updated in FP64 in iteration order (Welford): the moments of a chain are bit-identical however its
 * iterations were split over hp_engine_run / hp_engine_run_to_host calls, sub-streams or read-ahead.  The accumulators
 * (24 bytes per complex element and chain) are allocated when first asked for, outside the creation-time arena.  Enabling
 * the summary changes no draw and no output of the chain; it needs no HP_KEEP_* bit.  hp_engine_gcr does not accumulate;
 * hp_engine_rewind keeps the accumulators.  Replaces the host-side reduction of the reference's sample arrays
 * (pspec.py:590-596).  Optional batch means add the Monte-Carlo standard error and effective sample size of each mean
 * (hp_engine_set_summary_batched, hp_engine_read_summary_mcse). */
enum hp_summary_what { HP_SUMMARY_CR = 1, HP_SUMMARY_FG = 2 };
/* (Re)start on-device posterior moments: accumulators zeroed; of the iterations computed from now on the first
 * burn_in are skipped, then every thin-th is accumulated (burn_in >= 0, thin >= 1).  what = 0 stops accumulating.
 * Refused while read-ahead iterations are pending. */
int hp_engine_set_summary(hp_engine* e, int what, int burn_in, int thin);
/* mean [T][n|m] complex128 and var [T][n|m] double (E|x - mean|^2 over the accumulated iterations, ddof = 0, i.e.
 * numpy.var of the complex samples); either may be NULL.  *count = accumulated iterations.  what = one HP_SUMMARY_* bit.
 * bytes_each: capacity of each destination (mean needs 16 T n|m bytes, var 8 T n|m).  With count = 0 both read as zeros.
 * Refused (HP_ERR_ARG) for a quantity that is not being accumulated and while read-ahead iterations are pending. */
int hp_engine_read_summary(hp_engine* e, int chain, int what, double* mean, double* var, size_t bytes_each, int* count);
/* hp_engine_set_summary with batch means: batch > 0 also keeps, per element, the spread of the means of consecutive
 * batches of `batch` accumulated (thinned) samples, for the Monte-Carlo standard error of the posterior mean
 * (hp_engine_read_summary_mcse); 24 more bytes per complex element and chain, allocated when first asked for.  batch = 0:
 * no batch means (hp_engine_set_summary); batch < 0 is refused.  Changes neither mean nor var. */
int hp_engine_set_summary_batched(hp_engine* e, int what, int burn_in, int thin, int batch);
/* Batch-means Monte-Carlo standard error of the mean and effective sample size, [T][n|m] doubles each (either may be NULL;
 * bytes_each: capacity of each, 8 T n|m bytes).  With k accumulated samples, b = batch, nb = floor(k / b) complete batches
 * (*nbatch) of means Ybar_j and their mean Ybar: s2_bm = sum_j |Ybar_j - Ybar|^2 / (nb - 1), mcse = sqrt(b s2_bm / k),
 * ess = var / mcse^2.  NaN while nb < 2.  Refused as hp_engine_read_summary, and when batch means are off. */
int hp_engine_read_summary_mcse(hp_engine* e, int chain, int what, double* mcse, double* ess, size_t bytes_each, int* nbatch);

/* signal_S of the reference's return value: F^H diag(ps / Nfreqs^2) F for the current spectrum
 * (covariance_from_pspec, pspec.py:313-322).  dst [Nfreqs][Nfreqs] complex128. */
int hp_engine_read_signal_S(hp_engine* e, int chain, double* dst);
/* Cholesky status per chain of the last iteration (0 = ok). */
int hp_engine_info(hp_engine* e, int* info_host);

/* Accumulated device time per kernel class since creation or the last call with reset=1 (needs cfg.profile). */
int hp_engine_kernel_ms(hp_engine* e, double* ms, int* launches, int reset);
/* Philox chain id of every chain, ids[nchains] (default: the chain's index in the engine).  The device draws of a chain
 * depend on (cfg.seed, id, iteration) only: a driver that shards baselines over GPUs passes the global baseline indices
 * and the same seed on every rank, and the samples do not depend on the number of GPUs
 * (reference: one numpy stream per baseline, run-hydra-pspec.py:487-557). */
int hp_engine_set_chain_ids(hp_engine* e, const int* ids);
/* Use at most n of the cfg.substreams sub-batches from now on (1 = everything on the engine stream). */
int hp_engine_set_substreams(hp_engine* e, int n);
/* Switch the per-kernel event timing on or off at run time. */
int hp_engine_set_profile(hp_engine* e, int on);
/* Per-time flags (cfg.time_flags): which form of the per-time solve the engine runs for the chains loaded so far.
 *   *low_rank = 1: one shared factorisation per chain + a rank-k_t correction per time (csrc/hp_ptlow.cu); 0: one
 *   factorisation per (chain, time) (csrc/hp_pertime.cu: a time has more than 64 channels flagged beyond the chain's
 *   all-times mask, a chain carries per-time noise (hp_engine_load_chain_time_noise), Nfreqs + Nmodes > 448, or
 *   cfg.force_dense_solve).  *max_rank = largest k_t of the loaded chains.
 * Replaces nothing in the reference (it has no per-time flags, pspec.py:428); either pointer may be NULL. */
int hp_engine_pt_form(const hp_engine* e, int* low_rank, int* max_rank);
/* Total kernel launches issued by hp_engine_run / hp_engine_gcr so far. */
long long hp_engine_launch_count(const hp_engine* e);

/* sample_S (pspec.py:67-127) on its own: s [Ntimes][Nfreqs] complex128 signal realisations,
 * prior [2][Nfreqs] or NULL, draws [Nfreqs] as in hp_engine_set_draws; out [Nfreqs]. */
int hp_sample_S(int device, int ntimes, int nfreqs, const double* s, const double* prior, const double* draws,
                double* out);

/* utils.fourier_operator (utils.py:14-40), computed on the device; out [n][n] complex128. */
int hp_fourier_operator(int device, int n, double* out);
/* Batched Hermitian eigendecomposition on the device (one-sided Jacobi, csrc/hp_eigh.cu): S [batch][n][n] complex128
 * Hermitian, V [batch][n][n] (eigenvectors as columns, numpy.linalg.eigh convention, unordered), w [batch][n] eigenvalues,
 * sweeps [batch] or NULL.  Used for a non-delay-diagonal S_initial, whose eigenbasis the first Gibbs iteration runs in; stands
 * in for the matrix square root the reference takes of the signal covariance (scipy sqrtm in build_matrices, pspec.py:355). */
int hp_eigh_batch(int device, int n, int batch, const double* S, double* V, double* w, int* sweeps);

/* ---- test hooks (tests/ only): single kernels with host buffers ------------------------------- */
int hp_test_zgemm(int M, int N, int K, const double* A, int transA, int conjA, const double* B, int transB, int conjB,
                  const double* dk, double* C);
int hp_test_chol_solve(int n, int m, int T, const double* G, const double* lam, const double* Rfix, const double* wa,
                       int cg_compat, double* Ldense, double* X, int* info);
/* chol + trinv + k_solve3 (hp_solve3.cu) for nsys systems sharing G and lam:
 * Rfix [nsys][T][N], wa [nsys][T][n] or NULL, X [nsys][T][N], psum [nsys][n] = sum_t |x_k|^2 or NULL; grid_limit > 0 caps
 * the persistent grid */
int hp_test_solve3(int n, int m, int T, int nsys, const double* G, const double* lam, const double* Rfix, const double* wa,
                   int cg_compat, int grid_limit, double* X, double* psum);

/* k_solve3's static strip schedule for a system of nblk 32-row blocks (host logic, no device needed):
 * n[2][nwarps] strips per pass and warp, strips[2][nwarps][max_per_warp] their 16-row strip indices */
int hp_test_solve3_schedule(int nblk, unsigned char* n, unsigned char* strips, int* nwarps, int* max_per_warp);

/* k_pt_lowrank (csrc/hp_ptlow.cu) alone, launched as the engine launches it, for nsys systems of N unknowns (n columns of A):
 * lam [nsys][N], Rfix [nsys][T][N], wa [nsys][T][n] or NULL, X0 [nsys][T][N] = M_0^-1 b_t, Rcols [nsys][n][N] = R^T (row x is
 * R[:, x]), P [nsys][n][n] (lower triangle read), fidx [nsys][T][64], fcnt [nsys][T], chain_ids [nsys] (philox only);
 * out X [nsys][T][N], info [nsys].  HP_ERR_SIZE for N > 448 or a count above 64. */
int hp_test_pt_lowrank(int n, int N, int T, int nsys, const double* lam, const double* Rfix, const double* wa, const double* X0,
                       const double* Rcols, const double* P, const uint16_t* fidx, const int* fcnt, int philox, uint32_t key0,
                       uint32_t key1, uint32_t iter, const int* chain_ids, double* X, int* info);
/* k_pt_cholsolve (csrc/hp_pertime.cu) alone for nsys systems of N = n + m unknowns: H [nsys][T][1 + m][N] (column 0 = chat_t,
 * first n entries), lam [nsys][N], Rfix [nsys][T][N], wa [nsys][T][n] or NULL, same_prev [nsys][T] or NULL, grid (0: the
 * engine's persistent grid), chain_ids [nsys] (philox only); out X [nsys][T][N], info [nsys].  HP_ERR_SIZE when the shared
 * working set exceeds the device's opt-in limit. */
int hp_test_pt_cholsolve(int n, int m, int T, int nsys, const double* H, const double* lam, const double* Rfix, const double* wa,
                         const int* same_prev, int grid, int philox, uint32_t key0, uint32_t key1, uint32_t iter,
                         const int* chain_ids, double* X, int* info);

/* ---- measurement helpers ---------------------------------------------------------------------- */
/* FP64 tensor-pipe (DMMA.8x8x4) peak of the device measured with an issue loop for ~`seconds`; TFLOP/s. */
double hp_fp64_peak_tflops(int device, double seconds);
/* page-locked host memory for the host<->device copies of the end-to-end path */
/* A destroyed engine's device arena is kept (one per GPU) for the next hp_engine_create on that device; this frees it.
 * HP_NO_ARENA_CACHE=1 in the environment disables the cache. */
void hp_release_cached_memory(void);
void* hp_pinned_alloc(size_t bytes);
void hp_pinned_free(void* p);

const char* hp_last_error(void);
const char* hp_version(void);

#ifdef __cplusplus
}
#endif
#endif
