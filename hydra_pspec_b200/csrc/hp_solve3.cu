// hp_solve3.cu -- k_solve3: the GCR solve  x = W^H (W r + xi)  with warps that never wait for each other inside a pass.
//
// Replaces the per-time preconditioned CG of the reference (gcr_fgmodes_1d, pspec.py:151-235).  k_solve (round 1) and
// round 2's k_solve2 (since retired) both reached ~62 % DMMA-pipe activity for the same reason
// (profiles/r2_solve2_v1_notes.md): all consumer warps walk one shared W-block ring and meet at a partial-sum exchange
// after every block row, so they issue DMMAs in lockstep and do their per-block / per-row housekeeping in lockstep too,
// with the pipe idle.  Here:
//
//   * one persistent CTA (16 warps) per SM walks the (baseline, 16-time tile) list;
//   * the tile of right-hand sides r (TMA bulk copy, tile-native layout of k_rhs_tile) and the tile of y = W1 r + xi live
//     in two separate shared-memory buffers: nothing is updated in place, so block rows carry no ordering constraint;
//   * a warp owns whole 16-row strips of the output (16 x 16 complex register tile, 3M DMMA products, full K range): no K
//     split, no partial-sum exchange, no ring.  Strips are dealt to the warps by a longest-first schedule computed on the
//     host so that every scheduler (warp pair) gets the same number of k-steps;
//   * the A operand never touches shared memory: k_chol_w writes W in fragment-major order (per strip and k-step 2 row groups
//     x 32 lanes x [re, im] = 1 KiB contiguous), and every warp streams its own fragments from L2 into registers one
//     k-step ahead, across strip, pass and tile boundaries (the schedule is static); four warps per scheduler hide the L2
//     latency (a deeper register queue does not: ptxas gives all prefetch sites one scoreboard);
//   * B fragments (r or y) come from shared memory one k-step ahead; per k-step a warp issues 2 LDG.128 + 4 LDS.64 + 4 DADD
//     for 12 DMMAs, all between its own DMMAs, so a single warp can keep the FP64 pipe of its scheduler busy;
//   * pass 2 writes x from the accumulators to global and sum_t |x|^2 with it; the next tile's right-hand sides land during
//     pass 2 (r is dead after pass 1).
//
// Synchronisation per tile: one consumer barrier (y complete), one split-phase mbarrier (y buffer free again) and the
// TMA mbarrier of the right-hand sides.
#include "hp_kernels.cuh"
#include "hp_math.h"
#include "hp_mma.cuh"
#include "hp_async.cuh"
#include <algorithm>
#include <cstdlib>
#include <vector>

namespace hp {

using namespace async;

namespace {

constexpr int kW3 = kS3Warps;                 // consumer warps (all warps of the CTA)
constexpr int kS3Threads = 32 * kW3;
constexpr int kRowDoubles3 = 2 * 32 * kTT;    // one block row of a tile: [plane][32 rows][16 columns, XOR-swizzled]
constexpr int kFragDoubles = 128;             // one k-step of one strip in fragment-major order: 32 lanes x 4 doubles
#ifndef HP_S3_L1_PREFETCH
#define HP_S3_L1_PREFETCH 2                   // k-steps of L1 prefetch distance (0: loads bypass L1, no prefetch)
#endif

__device__ __forceinline__ double4 ldg_frag(const double* p) {
    // streaming fragment ([row group][lane][re, im]: two 16-byte loads, each 512 contiguous bytes per warp); every byte is
    // used once per CTA, keep it out of L1.  Volatile asm: the load keeps its place between the (volatile) DMMAs, after the
    // first DMMA of a k-step has waited for the previous load -- one load group in flight per warp.
    double4 v;
#if HP_S3_L1_PREFETCH > 0
    // loads through L1: the group HP_S3_L1_PREFETCH k-steps ahead was requested into L1 by a prefetch (no destination
    // register, hence no scoreboard): more fragment data in flight without the scoreboard aliasing.  5.27 -> 5.15 ms.
    asm volatile("ld.global.ca.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    asm volatile("ld.global.ca.v2.f64 {%0, %1}, [%2];" : "=d"(v.z), "=d"(v.w) : "l"(p + 64));
#else
    asm volatile("ld.global.cg.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    asm volatile("ld.global.cg.v2.f64 {%0, %1}, [%2];" : "=d"(v.z), "=d"(v.w) : "l"(p + 64));
#endif
    return v;
}

struct BFrag { double br[2], bi[2]; };

__device__ __forceinline__ void load_b(BFrag& f, const double* __restrict__ tile, int kstep, int bo0, int bo1) {
    // rows 4 kstep + q of the tile: block row (4 kstep) / 32, local row (4 kstep) % 32 + q; bo* hold q * 16 + swizzled column
    const double* b = tile + (size_t)(kstep >> 3) * kRowDoubles3 + (kstep & 7) * 4 * kTT;
    f.br[0] = b[bo0]; f.bi[0] = b[bo0 + 32 * kTT];
    f.br[1] = b[bo1]; f.bi[1] = b[bo1 + 32 * kTT];
}

// 3M:  P0 += Ar.Br,  P1 += Ai.Bi,  P2 += (Ar +- Ai).(Br + Bi);  a = (ar0, ai0, ar1, ai1).  The k-step is issued in two
// parts so that the caller can place the next fragment load right after the first DMMA.
__device__ __forceinline__ void mma_first(double (&P)[3][2][2][2], const double4& a, const BFrag& f) {
    dmma884(P[0][0][0][0], P[0][0][0][1], a.x, f.br[0]);
}
template <bool kP2>
__device__ __forceinline__ void mma_rest(double (&P)[3][2][2][2], const double4& a, const BFrag& f) {
    const double as0 = kP2 ? a.x - a.y : a.x + a.y, as1 = kP2 ? a.z - a.w : a.z + a.w;
    const double bs0 = f.br[0] + f.bi[0], bs1 = f.br[1] + f.bi[1];
    dmma884(P[0][0][1][0], P[0][0][1][1], a.x, f.br[1]);
    dmma884(P[0][1][0][0], P[0][1][0][1], a.z, f.br[0]);
    dmma884(P[0][1][1][0], P[0][1][1][1], a.z, f.br[1]);
    dmma884(P[1][0][0][0], P[1][0][0][1], a.y, f.bi[0]);
    dmma884(P[1][0][1][0], P[1][0][1][1], a.y, f.bi[1]);
    dmma884(P[1][1][0][0], P[1][1][0][1], a.w, f.bi[0]);
    dmma884(P[1][1][1][0], P[1][1][1][1], a.w, f.bi[1]);
    dmma884(P[2][0][0][0], P[2][0][0][1], as0, bs0);
    dmma884(P[2][0][1][0], P[2][0][1][1], as0, bs1);
    dmma884(P[2][1][0][0], P[2][1][0][1], as1, bs0);
    dmma884(P[2][1][1][0], P[2][1][1][1], as1, bs1);
}

__device__ __forceinline__ void consumer_sync3() { asm volatile("bar.sync 1, %0;" ::"n"(kS3Threads) : "memory"); }

}  // namespace

// k-steps of strip s (16 output rows): pass 1 needs k < 16 (s + 1), pass 2 needs k >= 16 s
size_t solve3_frag_doubles(int nblk) { return (size_t)4 * nblk * (2 * nblk + 1) * kFragDoubles; }
static size_t solve3_smem_bytes(int nblk) { return sizeof(double) * 2 * (size_t)nblk * kRowDoubles3 + 64; }
bool solve3_ok(int nblk, size_t max_smem) { return nblk >= 1 && 2 * nblk <= kS3MaxStrips && solve3_smem_bytes(nblk) <= max_smem; }

// Longest-first schedule of the 2 nblk strips of each pass over the warps; the warps are then dealt to the four schedulers
// so that each carries the same number of k-steps.
void solve3_make_schedule(int nblk, Solve3Sched* sc, int nstrip) {
    // nstrip: 16-row strips that hold rows of the system (ceil(N / 16)); a trailing strip of pure padding (N mod 32 in 1..16)
    // is left out of both passes and of the k-range of pass 2 (272 rows in a 288-row layout: 10.5 % of the k-steps)
    const int ns = (nstrip > 0 && nstrip < 2 * nblk) ? nstrip : 2 * nblk;
    for (int pass = 0; pass < 2; ++pass) {
        for (int w = 0; w < kW3; ++w) sc->n[pass][w] = 0;
        std::vector<int> len(ns), order(ns);
        for (int s = 0; s < ns; ++s) { len[s] = pass == 0 ? 4 * (s + 1) : 4 * ns - 4 * s; order[s] = s; }
        std::sort(order.begin(), order.end(), [&](int a, int b) { return len[a] > len[b]; });
        std::vector<std::vector<int>> lists(kW3);
        std::vector<long long> load(kW3, 0);
        for (int s : order) {
            int best = 0;
            for (int w = 1; w < kW3; ++w) if (load[w] < load[best]) best = w;
            lists[best].push_back(s);
            load[best] += len[s];
        }
        std::vector<int> byload(kW3);
        for (int w = 0; w < kW3; ++w) byload[w] = w;
        std::sort(byload.begin(), byload.end(), [&](int a, int b) { return load[a] > load[b]; });
        // warps to schedulers (physical warp id mod 4) in snake order of decreasing load: every scheduler gets the same
        // number of warps and (nearly) the same number of k-steps
        int cnt[4] = {0, 0, 0, 0};
        for (int r = 0; r < kW3; ++r) {
            const int lap = r / 4, pos = r % 4, sched = (lap & 1) ? 3 - pos : pos;
            const int phys = sched + 4 * cnt[sched]++;
            const auto& L = lists[byload[r]];
            sc->n[pass][phys] = (uint8_t)L.size();
            for (size_t e = 0; e < L.size() && e < (size_t)kS3MaxPerWarp; ++e) sc->strip[pass][phys][e] = (uint8_t)L[e];
        }
    }
}

// Phase timers (HP_S3_TIMERS=1; profiles/scripts/solve3_timers.py), clock64 deltas of lane 0 of every warp:
//  [0] pass 1 strips  [1] Philox + y store  [2] barrier (y complete)  [3] pass 2 strips  [4] x store  [5] waiting for the
//  y buffer  [6] waiting for right-hand sides  [7] whole loop
__device__ unsigned long long g_solve3_cycles[8];

template <bool kTimers>
__global__ void __launch_bounds__(kS3Threads, 1) k_solve3(Solve3Args a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int nblk = a.nblk, Np = nblk * 32;
    const int nstrip = (a.nstrip > 0 && a.nstrip < 2 * nblk) ? a.nstrip : 2 * nblk;   // strips with rows of the system
    double* tileR = reinterpret_cast<double*>(smem_raw);                 // [nblk][2][32][16]  right-hand sides
    double* tileY = tileR + (size_t)nblk * kRowDoubles3;                 // [nblk][2][32][16]  y = W1 r + xi
    uint64_t* rhs_full = reinterpret_cast<uint64_t*>(tileY + (size_t)nblk * kRowDoubles3);
    uint64_t* yfree = rhs_full + 1;                                      // every warp is done reading y (pass 2 of a tile)

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, q = lane & 3;
    const int total = a.ntiles * a.nsys;
    const size_t wf = (size_t)4 * nblk * (2 * nblk + 1) * kFragDoubles;   // solve3_frag_doubles
    const uint32_t tile_bytes = (uint32_t)nblk * kRowDoubles3 * 8;

    if (tid == 0) {
        mbar_init(rhs_full, 1);
        mbar_init(yfree, kW3);
        mbar_fence_init();
        if ((int)blockIdx.x < total) {
            mbar_arrive_expect_tx(rhs_full, tile_bytes);
            bulk_g2s(tileR, a.Rt + (size_t)blockIdx.x * nblk * kRowDoubles3, tile_bytes, rhs_full);
        }
    }
    __syncthreads();

    const int n1 = a.sched.n[0][warp], n2 = a.sched.n[1][warp];
    const int nseq = n1 + n2;
    // B-fragment offsets inside a group of four tile rows: row q, column (8 wj + g) ^ 4 q
    const int bo0 = q * kTT + (g ^ (q << 2)), bo1 = q * kTT + ((8 + g) ^ (q << 2));

    // ---- prefetch iterator over this warp's fragment stream: (tile, entry of the per-tile sequence, k-step)
    int pf_w = blockIdx.x, pf_e = -1, pf_left = 0;
    const double* pf_p = a.Wf1;
    bool pf_valid = nseq > 0 && pf_w < total;
    auto pf_entry = [&]() {
        // position the iterator on entry pf_e of tile pf_w
        const int sys = pf_w / a.ntiles;
        if (pf_e < n1) {
            const int s = a.sched.strip[0][warp][pf_e];
            pf_p = a.Wf1 + (size_t)sys * wf + (size_t)(2 * s * (s + 1)) * kFragDoubles + lane * 2;
            pf_left = 4 * (s + 1);
        } else {
            const int s = a.sched.strip[1][warp][pf_e - n1];
            pf_p = a.Wf2 + (size_t)sys * wf + (size_t)(8 * nblk * s - 2 * s * (s - 1)) * kFragDoubles + lane * 2;
            pf_left = 4 * nstrip - 4 * s;
        }
    };
    auto pf_next = [&]() -> double4 {
        // fragment of the next k-step of the stream (zeros past the end of the warp's work)
        if (pf_left == 0) {
            if (pf_valid) {
                if (++pf_e == nseq) { pf_e = 0; pf_w += gridDim.x; pf_valid = pf_w < total; }
                if (pf_valid) pf_entry();
            }
            if (!pf_valid) return make_double4(0.0, 0.0, 0.0, 0.0);
        }
        const double4 v = ldg_frag(pf_p);
        pf_p += kFragDoubles;
        --pf_left;
#if HP_S3_L1_PREFETCH > 0
        if (pf_left >= HP_S3_L1_PREFETCH) {   // the group HP_S3_L1_PREFETCH k-steps after the one just requested
            asm volatile("prefetch.global.L1 [%0];" ::"l"(pf_p + (HP_S3_L1_PREFETCH - 1) * kFragDoubles));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(pf_p + (HP_S3_L1_PREFETCH - 1) * kFragDoubles + 64));
        }
#endif
        return v;
    };
    // Exactly one fragment load is in flight per warp (issued before the DMMAs of the current k-step, consumed by the next):
    // ptxas tracks all prefetch sites with one scoreboard, so a deeper register queue would be waited for as a whole
    // (profiles/r2_solve2_v1_notes.md); the L2 latency is hidden by the four warps of a scheduler instead.
    double4 acur = pf_next();

    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = 0;
    if (kTimers) tlast = clock64();
#define S3_T(idx) do { if (kTimers) { const long long now_ = clock64(); tacc[idx] += now_ - tlast; tlast = now_; } } while (0)
    const long long tloop0 = tlast;

    double P[3][2][2][2];
    uint32_t it = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x, ++it) {
        const int sys = w / a.ntiles, tile = w - sys * a.ntiles, t0 = tile * kTT;
        const uint32_t chain = a.philox ? (uint32_t)a.dk.chain_ids[sys] : 0u;
        mbar_wait(rhs_full, it & 1);
        S3_T(6);
        // ------------------------------------------------------------------ pass 1:  y = W1 r (+ xi)
        for (int e = 0; e < n1; ++e) {
            const int s = a.sched.strip[0][warp][e];
            const int nk = 4 * (s + 1);
#pragma unroll
            for (int p = 0; p < 3; ++p)
#pragma unroll
                for (int wi = 0; wi < 2; ++wi)
#pragma unroll
                    for (int wj = 0; wj < 2; ++wj) P[p][wi][wj][0] = P[p][wi][wj][1] = 0.0;
            BFrag bf[2];
            load_b(bf[0], tileR, 0, bo0, bo1);
            for (int t = 0; t < nk; t += 2) {
                // A and B fragments one k-step ahead (the k-step after the strip's last one reads a valid, unused row group)
                mma_first(P, acur, bf[0]);
                const double4 anx = pf_next();
                load_b(bf[1], tileR, t + 1, bo0, bo1);
                mma_rest<false>(P, acur, bf[0]);
                mma_first(P, anx, bf[1]);
                acur = pf_next();
                load_b(bf[0], tileR, (t + 2 < nk) ? t + 2 : 0, bo0, bo1);
                mma_rest<false>(P, anx, bf[1]);
            }
            S3_T(0);
            if (e == 0 && it > 0) { mbar_wait(yfree, (it - 1) & 1); S3_T(5); }   // the previous tile's pass 2 is done with y
            // y = (P0 - P1) + i (P2 - P0 - P1) + xi  ->  tile Y
#pragma unroll
            for (int wi = 0; wi < 2; ++wi) {
                const int rl = 16 * (s & 1) + 8 * wi + g, row = 16 * s + 8 * wi + g;
                double* trow = tileY + (size_t)(s >> 1) * kRowDoubles3 + rl * kTT;
#pragma unroll
                for (int wj = 0; wj < 2; ++wj)
#pragma unroll
                    for (int x = 0; x < 2; ++x) {
                        const int col = 8 * wj + 2 * q + x;
                        double vr = P[0][wi][wj][x] - P[1][wi][wj][x];
                        double vi = P[2][wi][wj][x] - P[0][wi][wj][x] - P[1][wi][wj][x];
#ifdef HP_S3_EXPERIMENT_NO_NOISE   // timing experiment only (wrong statistics): what the Philox draws cost
                        if (false) {
#else
                        if (a.philox && row < a.N && t0 + col < a.T) {
#endif
                            u32x4 ctr; ctr.x = (uint32_t)row; ctr.y = (uint32_t)(t0 + col); ctr.z = a.dk.iter; ctr.w = chain;
                            double x0, x1;
#ifdef HP_PHILOX_DOUBLE   // experiment (profiles/r2_summary.md): what full double-precision Box-Muller costs this kernel
                            normal_pair(philox4x32_10(ctr, a.dk.key0, a.dk.key1 ^ 0xA5A5A5A5u), x0, x1);
#else
                            normal_pair_fast(philox4x32_10(ctr, a.dk.key0, a.dk.key1 ^ 0xA5A5A5A5u), x0, x1);
#endif
                            vr += x0 * 0.70710678118654752440; vi += x1 * 0.70710678118654752440;
                        }
                        const int c = col ^ ((rl & 3) << 2);
                        trow[c] = vr;
                        trow[c + 32 * kTT] = vi;
                    }
            }
            S3_T(1);
        }
        if (n1 == 0 && it > 0) mbar_wait(yfree, (it - 1) & 1);   // keep the phase bookkeeping of idle warps in step
#ifndef HP_S3_EXPERIMENT_NO_BARRIER   // timing experiment only (wrong results): what the per-tile barrier costs
        consumer_sync3();   // y complete; r is dead
#endif
        S3_T(2);
        if (tid == 0 && w + (int)gridDim.x < total) {
            // the next tile's right-hand sides land while pass 2 runs
            mbar_arrive_expect_tx(rhs_full, tile_bytes);
            bulk_g2s(tileR, a.Rt + (size_t)(w + gridDim.x) * nblk * kRowDoubles3, tile_bytes, rhs_full);
        }
        // ------------------------------------------------------------------ pass 2:  x = W2^H y, straight to global
        double* Xg = a.X + 2 * ((size_t)sys * a.Tp + t0) * Np;
        double* Pp = a.Ppart + ((size_t)sys * a.ntiles + tile) * a.n;
        for (int e = 0; e < n2; ++e) {
            const int s = a.sched.strip[1][warp][e];
            const int k0 = 4 * s, nk = 4 * nstrip - 4 * s;
#pragma unroll
            for (int p = 0; p < 3; ++p)
#pragma unroll
                for (int wi = 0; wi < 2; ++wi)
#pragma unroll
                    for (int wj = 0; wj < 2; ++wj) P[p][wi][wj][0] = P[p][wi][wj][1] = 0.0;
            BFrag bf[2];
            load_b(bf[0], tileY, k0, bo0, bo1);
            for (int t = 0; t < nk; t += 2) {
                mma_first(P, acur, bf[0]);
                const double4 anx = pf_next();
                load_b(bf[1], tileY, k0 + t + 1, bo0, bo1);
                mma_rest<true>(P, acur, bf[0]);
                mma_first(P, anx, bf[1]);
                acur = pf_next();
                load_b(bf[0], tileY, (t + 2 < nk) ? k0 + t + 2 : 0, bo0, bo1);
                mma_rest<true>(P, anx, bf[1]);
            }
            S3_T(3);
            // x = (P0 + P1) + i (P2 - P0 + P1)   (conj(A) B)
#pragma unroll
            for (int wi = 0; wi < 2; ++wi) {
                const int row = 16 * s + 8 * wi + g;
                double psum = 0.0;
#pragma unroll
                for (int wj = 0; wj < 2; ++wj)
#pragma unroll
                    for (int x = 0; x < 2; ++x) {
                        const int col = 8 * wj + 2 * q + x;
                        const double vr = P[0][wi][wj][x] + P[1][wi][wj][x];
                        const double vi = P[2][wi][wj][x] - P[0][wi][wj][x] + P[1][wi][wj][x];
                        *reinterpret_cast<double2*>(Xg + 2 * ((size_t)col * Np + row)) = make_double2(vr, vi);
                        psum += vr * vr + vi * vi;
                    }
                psum += __shfl_xor_sync(0xffffffffu, psum, 1);
                psum += __shfl_xor_sync(0xffffffffu, psum, 2);
                if (q == 0 && row < a.n) Pp[row] = psum;
            }
            S3_T(4);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(yfree);
    }
    if (kTimers) {
        tacc[7] = clock64() - tloop0;
        if (lane == 0)
            for (int i = 0; i < 8; ++i) atomicAdd(&g_solve3_cycles[i], (unsigned long long)tacc[i]);
    }
#undef S3_T
}

extern "C" void hp_solve3_timers(unsigned long long* out, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_solve3_cycles, sizeof(unsigned long long) * 8);
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_solve3_cycles, z, sizeof(z)); }
}

void launch_solve3(const Solve3Args& a_in, cudaStream_t st) {
    Solve3Args a = a_in;
    static int num_sm = 0, timers = -1;
    if (!num_sm) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sm, cudaDevAttrMultiProcessorCount, dev);
        const char* ev = getenv("HP_S3_TIMERS");
        timers = (ev && ev[0] == '1') ? 1 : 0;
    }
    const size_t smem = solve3_smem_bytes(a.nblk);
    static size_t attr_dev[kMaxDev] = {0};
    size_t& attr_smem = attr_dev[current_device_slot()];
    if (smem > attr_smem) {
        cudaFuncSetAttribute(k_solve3<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_solve3<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_smem = smem;
    }
    const int total = a.ntiles * a.nsys;
    int grid = a.grid_limit > 0 ? a.grid_limit : num_sm;
    if (grid > total) grid = total;
    if (timers) k_solve3<true><<<grid, kS3Threads, smem, st>>>(a);
    else k_solve3<false><<<grid, kS3Threads, smem, st>>>(a);
}

// ---------------------------------------------------------------------------------------------------------------------
// k_rhs_tile: right-hand sides in the shared-memory layout of k_solve3's tile,
//     Rt[sys][tile][block row][plane][r][c ^ 4 (r & 3)] = (lam_row) Rfix[sys][16 tile + c][32 j + r] (+ wa)
// Built once per chain load when the chain runs unscaled right-hand sides (Philox mode), per iteration otherwise.
__global__ void __launch_bounds__(256) k_rhs_tile(double* __restrict__ Rt, const double* __restrict__ Rfix, const double* __restrict__ wa,
                                                  const double* __restrict__ lam, int nblk, int n, int N, int T, int Tp) {
    const int Np = nblk * 32;
    const int tile = blockIdx.x, sys = blockIdx.y, t0 = tile * kTT;
    const int ntiles = gridDim.x;
    const double* R = Rfix + 2 * ((size_t)sys * Tp + t0) * Np;
    const double* Wa = wa ? wa + 2 * ((size_t)sys * Tp + t0) * Np : nullptr;
    const double* lm = lam ? lam + (size_t)sys * Np : nullptr;
    double* out = Rt + ((size_t)sys * ntiles + tile) * nblk * kRowDoubles3;
    // thread -> (column c, row): consecutive threads read consecutive rows of one time (coalesced 16-byte loads)
    for (int e = threadIdx.x; e < Np * kTT; e += blockDim.x) {
        const int c = e / Np, row = e - c * Np;
        double vr = 0.0, vi = 0.0;
        if (t0 + c < T && row < N) {
            const double2 x = *reinterpret_cast<const double2*>(R + 2 * ((size_t)c * Np + row));
            const double l = lm ? lm[row] : 1.0;
            vr = l * x.x; vi = l * x.y;
            if (Wa && row < n) { const double2 y = *reinterpret_cast<const double2*>(Wa + 2 * ((size_t)c * Np + row)); vr += y.x; vi += y.y; }
        }
        const int j = row >> 5, r = row & 31;
        double* o = out + (size_t)j * kRowDoubles3 + r * kTT + (c ^ ((r & 3) << 2));
        o[0] = vr;
        o[32 * kTT] = vi;
    }
}
void launch_rhs_tile(double* Rt, const double* Rfix, const double* wa, const double* lam, int nblk, int n, int N, int T, int Tp,
                     int ntiles, int nsys, cudaStream_t st) {
    k_rhs_tile<<<dim3(ntiles, nsys), 256, 0, st>>>(Rt, Rfix, wa, lam, nblk, n, N, T, Tp);
}

// ---------------------------------------------------------------------------------------------------------------------
// k_cg_scale: the scalar model of the reference's truncated CG (pspec.py:228; DESIGN.md section 1, hp_math.h: cg_theta).
// Every column of the exact solution is multiplied by theta(c, ||b||) with
//     c = sum_k lam_k^2 conj(r_k) x_k + sum_j conj(r_j) x_j,   ||b||^2 = sum_k lam_k^2 |r_k|^2 + sum_j |r_j|^2
// in the whitened variables (r = lam * Rfix + wa).  One CTA per (time, baseline); works on the global solution, so it
// serves k_solve3 and the dense-product solve of large N (k_solve applies the model itself).
__global__ void __launch_bounds__(128) k_cg_scale(double* __restrict__ X, const double* __restrict__ Rfix, const double* __restrict__ wa,
                                                  const double* __restrict__ lam, int n, int N, int Np, int T, int Tp) {
    const int t = blockIdx.x, sys = blockIdx.y;
    if (t >= T) return;
    const size_t off = 2 * ((size_t)sys * Tp + t) * Np;
    double* x = X + off;
    const double* R = Rfix + off;
    const double* Wa = wa ? wa + off : nullptr;
    const double* lm = lam + (size_t)sys * Np;
    double sre = 0.0, sim = 0.0, sb = 0.0;
    for (int row = threadIdx.x; row < N; row += blockDim.x) {
        const double l = lm[row];
        double vr = l * R[2 * row], vi = l * R[2 * row + 1];
        if (Wa && row < n) { vr += Wa[2 * row]; vi += Wa[2 * row + 1]; }
        const double wgt = row < n ? l * l : 1.0;
        const double xr = x[2 * row], xim = x[2 * row + 1];
        sre += wgt * (vr * xr + vi * xim);   // conj(r) x
        sim += wgt * (vr * xim - vi * xr);
        sb += wgt * (vr * vr + vi * vi);
    }
    __shared__ double red[3][4];
    __shared__ double th[2];
    for (int o = 16; o > 0; o >>= 1) {
        sre += __shfl_down_sync(0xffffffffu, sre, o);
        sim += __shfl_down_sync(0xffffffffu, sim, o);
        sb += __shfl_down_sync(0xffffffffu, sb, o);
    }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = sre; red[1][threadIdx.x >> 5] = sim; red[2][threadIdx.x >> 5] = sb; }
    __syncthreads();
    if (threadIdx.x == 0) {
        cplx c; c.re = red[0][0] + red[0][1] + red[0][2] + red[0][3]; c.im = red[1][0] + red[1][1] + red[1][2] + red[1][3];
        const double b2 = red[2][0] + red[2][1] + red[2][2] + red[2][3];
        const cplx v = cg_theta(c, sqrt(b2), 1e-8, 1e-6, 100000);
        th[0] = v.re; th[1] = v.im;
    }
    __syncthreads();
    const double tr = th[0], ti = th[1];
    for (int row = threadIdx.x; row < Np; row += blockDim.x) {
        const double xr = x[2 * row], xim = x[2 * row + 1];
        x[2 * row] = tr * xr - ti * xim;
        x[2 * row + 1] = tr * xim + ti * xr;
    }
}
void launch_cg_scale(double* X, const double* Rfix, const double* wa, const double* lam, int n, int N, int Np, int T, int Tp,
                     int nsys, cudaStream_t st) {
    k_cg_scale<<<dim3(T, nsys), 128, 0, st>>>(X, Rfix, wa, lam, n, N, Np, T, Tp);
}

}  // namespace hp
