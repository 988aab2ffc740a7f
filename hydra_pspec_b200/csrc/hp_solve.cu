// hp_solve.cu -- k_solve: the GCR solve for all times of a baseline as two triangular block products.
//
// Replaces the per-time preconditioned CG of the reference (gcr_fgmodes_1d, pspec.py:151-235).
// With M = L L^H and W = L^-1 formed explicitly (k_chol_w), the solution for every time
// sample is  x = W^H (W r [+ xi]):  two block-triangular products without any dependency between
// block rows, instead of a substitution that serialises on every diagonal block.
//
// CTA = (tile of 16 times, baseline).  The 16-column tile (right-hand sides, then y = W r, then
// x = W^H y, all in place) stays in shared memory; the 32x32 blocks of W stream from L2 through a
// ring filled by TMA bulk copies (cp.async.bulk + mbarrier, one producer warp); sixteen consumer
// warps run the block products on the FP64 tensor pipe (DMMA.8x8x4), each on an 8x8 complex tile,
// three real products per complex one (3M scheme, see tile_mma).  In-place works because pass 1 walks the block rows downwards
// (y_i overwrites r_i after the column group's barrier that ends block row i) and pass 2 upwards.
//
// Right-hand sides are built on the fly (never stored):
//     injected draws :  r = lam * Rfix + wa                      (Rfix carries B^H N^-1/2 omega_b)
//     Philox         :  r = lam * Rfix, and xi ~ CN(0, I) is added to y = L^-1 r before the second
//                       product.  Since cov(lam B^H N^-1/2 omega_b + omega_a) = M = L L^H, this is the
//                       same distribution as drawing omega_a, omega_b (pspec.py:215-222) and needs no
//                       transform of the noise realisation.
#include "hp_kernels.cuh"
#include "hp_math.h"
#include "hp_mma.cuh"

namespace hp {

namespace {

constexpr int kLdX = 16;       // solution tile: 16 columns, no padding; XOR-swizzled (xs) instead
constexpr int kMaxStages = 6;
constexpr int kConsumers = 512;                      // 16 consumer warps: 8 tiles x 2 halves of K
constexpr int kScratchDoubles = 2 * 8 * 32 * 3;      // [K half][tile][lane][P1..P3]: the element handed to the other half

// Shared-memory index of element (row, col) of a 16-column tile.  The column is XORed with
// 4 (row & 3): a DMMA B-fragment load (4 consecutive rows x 8 columns per half-warp pair) then
// touches all 32 banks exactly once, with no padding columns.
__device__ __forceinline__ int xs(int row, int col) { return row * kLdX + (col ^ ((row & 3) << 2)); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "LAB_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra LAB_DONE_%=;\n\t"
        "bra LAB_WAIT_%=;\n\t"
        "LAB_DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// all eight consumer warps (the producer warp never takes part)
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 3, 512;" ::: "memory"); }
// the eight warps that own the same eight columns of the solution tile (ids 1 and 2)
__device__ __forceinline__ void group_sync(int tj) { asm volatile("bar.sync %0, 256;" ::"r"(1 + tj) : "memory"); }

// Complex block product with three real DMMAs per k-step instead of four (the "3M" scheme of
// zgemm3m):  P1 = Ar.Br,  P2 = Ai.Bi,  P3 = (Ar + s Ai).(Br + Bi)  with s = +1, or -1 for conj(A):
//      A  B :   re = P1 - P2,   im = P3 - P1 - P2
//   conj(A) B:  re = P1 + P2,   im = P3 - P1 + P2
// The operand sums cost two DADDs per k-step; the FP64 tensor pipe, which bounds this kernel, sees
// 25 % fewer instructions.  Normwise the rounding error is that of the ordinary product.
//   acc[0] = P1, acc[1] = P2, acc[2] = P3, over k in [k0, k1) (multiples of 4).
//   A element (row g, k): AT ? A[k * lda + g] : A[g * lda + k]   (pointers already offset to the warp's rows)
//   B element (k, col): swizzled 16-column tile, B[xs(k, col)]; Br/Bi point at row 0 of the k range's
//   block (a multiple of 4 rows), bcol = this lane's column already XORed with 4 q.
template <bool AT>
__device__ __forceinline__ void tile_mma(double (&acc)[3][2], const double* __restrict__ Ar, const double* __restrict__ Ai,
                                         int lda, const double* __restrict__ Br, const double* __restrict__ Bi, int bcol,
                                         int k0, int k1) {
    const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
    constexpr int ldb = kLdX;
    const int aoff = AT ? q * lda + g : g * lda + q;
    const int astep = AT ? 4 * lda : 4;
    const double* pa_r = Ar + aoff + (AT ? k0 * lda : k0);
    const double* pa_i = Ai + aoff + (AT ? k0 * lda : k0);
    const double* pb_r = Br + (k0 + q) * ldb + bcol;
    const double* pb_i = Bi + (k0 + q) * ldb + bcol;
    double ar = *pa_r, ai = *pa_i, br = *pb_r, bi = *pb_i;
#pragma unroll 4
    for (int kk = k0; kk < k1; kk += 4) {
        double nar = 0.0, nai = 0.0, nbr = 0.0, nbi = 0.0;
        if (kk + 4 < k1) {
            pa_r += astep; pa_i += astep; pb_r += 4 * ldb; pb_i += 4 * ldb;
            nar = *pa_r; nai = *pa_i; nbr = *pb_r; nbi = *pb_i;
        }
        const double as = AT ? ar - ai : ar + ai;  // AT is only used for conj(A)^T operands
        const double bs = br + bi;
        dmma884(acc[0][0], acc[0][1], ar, br);
        dmma884(acc[1][0], acc[1][1], ai, bi);
        dmma884(acc[2][0], acc[2][1], as, bs);
        ar = nar; ai = nai; br = nbr; bi = nbi;
    }
}

struct RhsCtx {
    const double* Rfix; const double* wa; const double* lam;
    int Np, n, N, T, t0;
};

// right-hand side element (system row `row`, tile column `col`)
__device__ __forceinline__ void rhs_elem(const RhsCtx& c, int row, int col, double& vr, double& vi) {
    int t = c.t0 + col;
    vr = 0.0; vi = 0.0;
    if (t >= c.T || row >= c.N) return;
    size_t off = 2 * ((size_t)t * c.Np + row);
    double2 x = *reinterpret_cast<const double2*>(c.Rfix + off);
    double l = c.lam[row];
    vr = l * x.x; vi = l * x.y;
    if (c.wa && row < c.n) { double2 wv = *reinterpret_cast<const double2*>(c.wa + off); vr += wv.x; vi += wv.y; }
}

}  // namespace

static size_t solve_smem_bytes_stages(int nblk, int stages) {
    size_t Np = (size_t)nblk * 32;
    size_t d = 2 * Np * kLdX                   // solution tile planes
             + (size_t)stages * kLBlkDoubles   // ring of W blocks (also the reduction scratch of the epilogue)
             + 2 * kScratchDoubles             // K-half exchange buffer, double buffered by block-row parity
             + 32                              // theta
             + 2 * kMaxStages + 6;             // mbarriers
    return d * sizeof(double);
}
size_t solve_smem_bytes(int nblk) { return solve_smem_bytes_stages(nblk, 2); }  // minimum configuration
// k_solve can take a system: the minimum configuration fits shared memory AND its two ring slots can stage four
// right-hand-side rows at a time (Np <= 576); larger systems go to the dense-product solve of the engine
bool solve_resident_ok(int nblk, size_t max_smem) {
    return solve_smem_bytes(nblk) <= max_smem && (size_t)2 * kLBlkDoubles * 8 >= (size_t)4 * nblk * 32 * 16;
}

__global__ void __launch_bounds__(544) k_solve(SolveArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int nblk = a.nblk, Np = nblk * 32;
    const int kStages = a.stages;
    double* ring = reinterpret_cast<double*>(smem_raw);          // [kStages][2304], 16-byte aligned for TMA
    double* Xr = ring + (size_t)kStages * kLBlkDoubles;
    double* Xi = Xr + (size_t)Np * kLdX;
    double* scratch = Xi + (size_t)Np * kLdX;                     // 2 * kScratchDoubles (double buffered by row parity)
    double* theta = scratch + 2 * kScratchDoubles;                // 32
    uint64_t* full = reinterpret_cast<uint64_t*>(theta + 32);     // [kMaxStages]
    uint64_t* empty = full + kMaxStages;                          // [kMaxStages]
    uint64_t* rowbar = empty + kMaxStages;                        // [2] one per column group
    uint64_t* stagebar = rowbar + 2;                              // right-hand-side rows landed in the ring area
    uint64_t* ringfree = rowbar + 3;                              // ... and have been moved into the tile
    double* red = ring;                                           // 16*16*3, epilogue only (ring idle by then)

    const int sys = blockIdx.y, tile = blockIdx.x;
    const double* Wp = a.Wp + (size_t)sys * tri_blocks(nblk) * kLBlkDoubles;
    const double* lam = a.lam + (size_t)sys * Np;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 16); }  // a.stages <= kMaxStages
        mbar_init(&rowbar[0], 4);
        mbar_init(&rowbar[1], 4);
        mbar_init(stagebar, 1);
        mbar_init(ringfree, 16);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == 16) {
        // ------------------------------------------------------------------ producer warp
        if (lane == 0) {
            // The ring area first receives the tile's right-hand-side rows (Rfix[t][0..Np), one bulk copy
            // per time, `a.rows_per_round` times per round); the consumers move them into the planar
            // tile and hand the ring back.
            {
                const int T0 = tile * kTT;
                uint32_t par = 0;
                for (int r0 = 0; r0 < kTT; r0 += a.rows_per_round) {
                    int nr = 0;
                    for (int t = r0; t < min(kTT, r0 + a.rows_per_round); ++t) nr += (T0 + t < a.T) ? 1 : 0;
                    mbar_arrive_expect_tx(stagebar, (uint32_t)nr * Np * 16);
                    for (int t = r0; t < min(kTT, r0 + a.rows_per_round); ++t)
                        if (T0 + t < a.T)
                            bulk_g2s(ring + (size_t)(t - r0) * Np * 2, a.Rfix + 2 * (((size_t)sys * a.Tp + T0 + t) * Np),
                                     (uint32_t)Np * 16, stagebar);
                    mbar_wait(ringfree, par);
                    par ^= 1;
                }
            }
            uint32_t s = 0, round = 0;  // ring slot and how many times the ring has wrapped
            auto push = [&](const double* src) {
                if (round > 0) mbar_wait(&empty[s], (round - 1) & 1);
                mbar_arrive_expect_tx(&full[s], kLBlkDoubles * 8);
                bulk_g2s(ring + (size_t)s * kLBlkDoubles, src, kLBlkDoubles * 8, &full[s]);
                if (++s == (uint32_t)kStages) { s = 0; ++round; }
            };
            // pass 1: block rows downwards, diagonal block first
            for (int i = nblk - 1; i >= 0; --i)
                for (int j = i; j >= 0; --j) push(Wp + blk_index(i, j) * kLBlkDoubles);
            // pass 2: block rows upwards; row i of W^H is column i of W, diagonal block first
            for (int i = 0; i < nblk; ++i)
                for (int j = i; j < nblk; ++j) push(Wp + blk_index(j, i) * kLBlkDoubles);
        }
        return;
    }

    // ---------------------------------------------------------------------- consumer warps
    RhsCtx rc;
    rc.Rfix = a.Rfix + 2 * (size_t)sys * a.Tp * Np;
    rc.wa = a.wa ? a.wa + 2 * (size_t)sys * a.Tp * Np : nullptr;
    rc.lam = lam; rc.Np = Np; rc.n = a.n; rc.N = a.N; rc.T = a.T; rc.t0 = tile * kTT;
    const uint32_t chain = a.philox_wa ? (uint32_t)a.dk.chain_ids[sys] : 0u;
    const int g = lane >> 2, q = lane & 3;
    // Warp tile: rows 8 ti.., columns 8 tj...  The two column groups (tj = 0, 1) never touch each
    // other's columns; they share only the ring.
    // Sixteen warps: tile (ti, tj) of the 32 x 16 block row and K half kh (k in [16 kh, 16 kh + 16) of
    // every block).  Two warps per tile double the warps per scheduler (the per-warp instruction stream
    // between DMMAs, not the tensor pipe or shared-memory bandwidth, limited the 8-warp version); the two
    // halves swap one element each at the end of a block row and finish one element apiece.
    const int wt = warp & 7, kh = warp >> 3;
    const int ti = wt >> 1, tj = wt & 1;
    const int bcol = (8 * tj + g) ^ (q << 2);  // this lane's B-fragment column in the swizzled tile

    // stage the right-hand sides:  tile[row][col] = lam_row Rfix[t0 + col][row] (+ wa).  The rows arrive
    // in the ring area by TMA (asynchronous, full DRAM burst instead of a load-use chain); a warp
    // instruction then moves 8 consecutive rows x 4 times: conflict-free 16-byte reads, at most 2-way
    // conflicts on the swizzled writes.
    {
        const int rl = lane & 7, cl = lane >> 3;
        const double2* stage = reinterpret_cast<const double2*>(ring);
        uint32_t par = 0;
        for (int r0 = 0; r0 < kTT; r0 += a.rows_per_round) {
            mbar_wait(stagebar, par);
            par ^= 1;
            const int ncg = a.rows_per_round / 4;  // column groups in this round
            const int ngrp = (Np / 8) * ncg;
            for (int grp = warp; grp < ngrp; grp += 16) {
                const int row = 8 * (grp / ncg) + rl, tl = 4 * (grp % ncg) + cl, col = r0 + tl;
                double vr = 0.0, vi = 0.0;
                if (rc.t0 + col < a.T && row < a.N) {
                    double2 x = stage[(size_t)tl * Np + row];
                    const double l = lam[row];
                    vr = l * x.x; vi = l * x.y;
                    if (rc.wa && row < a.n) {
                        double2 wv = *reinterpret_cast<const double2*>(rc.wa + 2 * ((size_t)(rc.t0 + col) * Np + row));
                        vr += wv.x; vi += wv.y;
                    }
                }
                Xr[xs(row, col)] = vr;
                Xi[xs(row, col)] = vi;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(ringfree);
        }
    }
    consumer_sync();

    uint32_t slot = 0, parity = 0;  // ring slot being consumed and its phase parity
    auto acquire = [&]() -> const double* {
        mbar_wait(&full[slot], parity);
        return ring + (size_t)slot * kLBlkDoubles;
    };
    auto release = [&]() {
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[slot]);
        if (++slot == (uint32_t)kStages) { slot = 0; parity ^= 1; }
    };
    // End of a block row: the two K halves of a tile exchange partial sums through shared memory (each
    // hands over the element of its lane pair that the other half finishes).  The exchange buffer
    // alternates with the row parity, so the only synchronisation is the column group's barrier between
    // writing and reading it; that barrier also guarantees that every warp of the group is done reading
    // block row i before it is overwritten in place (later rows of the pass never read it).
    uint32_t rowpar = 0;
    auto exchange = [&](double (&acc)[3][2], double (&P)[3]) {
        double* buf = scratch + (size_t)rowpar * kScratchDoubles;
        double* mine = buf + (((size_t)kh * 8 + wt) * 32 + lane) * 3;          // what I hand over
        const double* theirs = buf + (((size_t)(kh ^ 1) * 8 + wt) * 32 + lane) * 3;  // what my partner hands me
#pragma unroll
        for (int p = 0; p < 3; ++p) mine[p] = kh ? acc[p][0] : acc[p][1];  // half 0 keeps element 0, half 1 element 1
        group_sync(tj);
#pragma unroll
        for (int p = 0; p < 3; ++p) P[p] = (kh ? acc[p][1] : acc[p][0]) + theirs[p];
        rowpar ^= 1;
    };

    // ------------------------------------------------------------------ pass 1:  y = W r (+ xi)
    for (int i = nblk - 1; i >= 0; --i) {
        double acc[3][2] = {{0, 0}, {0, 0}, {0, 0}};
        // The fluctuation draw of the element this thread finishes does not depend on the products: issue it
        // first, so that its integer / MUFU instructions fill the issue slots between this row's DMMAs instead
        // of running after the row's barrier with the tensor pipe idle.
        double xi0 = 0.0, xi1 = 0.0;
        {
            const int row = 32 * i + 8 * ti + g, c = 8 * tj + 2 * q + kh;
            if (a.philox_wa && row < a.N && rc.t0 + c < a.T) {
                u32x4 ctr; ctr.x = (uint32_t)row; ctr.y = (uint32_t)(rc.t0 + c); ctr.z = a.dk.iter; ctr.w = chain;
                normal_pair_fast(philox4x32_10(ctr, a.dk.key0, a.dk.key1 ^ 0xA5A5A5A5u), xi0, xi1);
                xi0 *= 0.70710678118654752440; xi1 *= 0.70710678118654752440;
            }
        }
        {
            const double* blk = acquire();  // W_ii, lower triangular: k < 8 (ti + 1)
            const int k0 = 16 * kh, k1 = min(16 * kh + 16, 8 * (ti + 1));
            if (k0 < k1)
                tile_mma<false>(acc, blk + 8 * ti * kLdBlk, blk + kLPlane + 8 * ti * kLdBlk, kLdBlk, Xr + (size_t)32 * i * kLdX,
                                Xi + (size_t)32 * i * kLdX, bcol, k0, k1);
            release();
        }
        for (int j = i - 1; j >= 0; --j) {
            const double* blk = acquire();
            tile_mma<false>(acc, blk + 8 * ti * kLdBlk, blk + kLPlane + 8 * ti * kLdBlk, kLdBlk, Xr + (size_t)32 * j * kLdX,
                            Xi + (size_t)32 * j * kLdX, bcol, 16 * kh, 16 * kh + 16);
            release();
        }
        double P[3];
        exchange(acc, P);
        {
            const int row = 32 * i + 8 * ti + g, c = 8 * tj + 2 * q + kh;
            // y += xi, xi ~ CN(0, 1): fluctuation term of the constrained realisation
            const double vr = P[0] - P[1] + xi0, vi = P[2] - P[0] - P[1] + xi1;
            Xr[xs(row, c)] = vr;
            Xi[xs(row, c)] = vi;
        }
    }
    group_sync(tj);  // y complete and visible within the column group

    // ------------------------------------------------------------------ pass 2:  x = W^H y
    for (int i = 0; i < nblk; ++i) {
        double acc[3][2] = {{0, 0}, {0, 0}, {0, 0}};
        {
            const double* blk = acquire();  // W_ii^H, upper triangular: k >= 8 ti ; A element (r, k) = conj(W_ii[k][r])
            const int k0 = max(16 * kh, 8 * ti), k1 = 16 * kh + 16;
            if (k0 < k1)
                tile_mma<true>(acc, blk + 8 * ti, blk + kLPlane + 8 * ti, kLdBlk, Xr + (size_t)32 * i * kLdX,
                               Xi + (size_t)32 * i * kLdX, bcol, k0, k1);
            release();
        }
        for (int j = i + 1; j < nblk; ++j) {
            const double* blk = acquire();  // W_ji^H
            tile_mma<true>(acc, blk + 8 * ti, blk + kLPlane + 8 * ti, kLdBlk, Xr + (size_t)32 * j * kLdX,
                           Xi + (size_t)32 * j * kLdX, bcol, 16 * kh, 16 * kh + 16);
            release();
        }
        double P[3];
        exchange(acc, P);
        {
            const int row = 32 * i + 8 * ti + g, c = 8 * tj + 2 * q + kh;
            // conj(A) B:  re = P1 + P2, im = P3 - P1 + P2
            Xr[xs(row, c)] = P[0] + P[1];
            Xi[xs(row, c)] = P[2] - P[0] + P[1];
        }
    }
    consumer_sync();  // both column groups done; the ring is idle from here on

    // ------------------------------------------------------------------ epilogue
    if (a.cg_compat) {
        // c = b^H x*, ||b||^2 in the reference's (unwhitened) variables:
        //   weights lam^2 on the signal rows, 1 on the foreground rows (DESIGN.md, "CG model").
        int col = tid & 15, rg = tid >> 4;
        double sre = 0.0, sim = 0.0, sb = 0.0;
        for (int row = rg; row < a.N; row += kConsumers / 16) {
            double vr, vi;
            rhs_elem(rc, row, col, vr, vi);
            double w = row < a.n ? lam[row] * lam[row] : 1.0;
            double xr = Xr[xs(row, col)], xi = Xi[xs(row, col)];
            sre += w * (vr * xr + vi * xi);  // conj(R) X
            sim += w * (vr * xi - vi * xr);
            sb += w * (vr * vr + vi * vi);
        }
        red[(rg * 16 + col) * 3 + 0] = sre; red[(rg * 16 + col) * 3 + 1] = sim; red[(rg * 16 + col) * 3 + 2] = sb;
        consumer_sync();
        if (tid < 16) {
            double cre = 0.0, cim = 0.0, b2 = 0.0;
            for (int r2 = 0; r2 < kConsumers / 16; ++r2) {
                cre += red[(r2 * 16 + tid) * 3 + 0]; cim += red[(r2 * 16 + tid) * 3 + 1]; b2 += red[(r2 * 16 + tid) * 3 + 2];
            }
            cplx c; c.re = cre; c.im = cim;
            cplx th = cg_theta(c, sqrt(b2), 1e-8, 1e-6, 100000);
            theta[2 * tid] = th.re; theta[2 * tid + 1] = th.im;
        }
        consumer_sync();
        for (int e = tid; e < Np * 16; e += kConsumers) {
            int row = e >> 4, col2 = e & 15;
            double xr = Xr[xs(row, col2)], xi = Xi[xs(row, col2)];
            double tr = theta[2 * col2], tim = theta[2 * col2 + 1];
            Xr[xs(row, col2)] = tr * xr - tim * xi;
            Xi[xs(row, col2)] = tr * xi + tim * xr;
        }
        consumer_sync();
    }
    // write-out with the same 8 rows x 4 times mapping; sum_t |y|^2 per row reduced on the way
    {
        double* Xg = a.X + 2 * ((size_t)sys * a.Tp + (size_t)tile * kTT) * Np;
        double* Sg = a.Ssc ? a.Ssc + 2 * ((size_t)sys * a.Tp + (size_t)tile * kTT) * a.n : nullptr;
        double* Pp = a.Ppart + ((size_t)sys * a.ntiles + tile) * a.n;
        const int rl = lane & 7, cl = lane >> 3;
        for (int rg = warp; rg < Np / 8; rg += 16) {
            const int row = 8 * rg + rl;
            const double l = lam[row];
            double p = 0.0;
#pragma unroll
            for (int cg = 0; cg < 4; ++cg) {
                const int t = 4 * cg + cl;
                double xr = Xr[xs(row, t)], xi = Xi[xs(row, t)];
                *reinterpret_cast<double2*>(Xg + 2 * ((size_t)t * Np + row)) = make_double2(xr, xi);
                if (Sg && row < a.n) *reinterpret_cast<double2*>(Sg + 2 * ((size_t)t * a.n + row)) = make_double2(l * xr, l * xi);
                p += xr * xr + xi * xi;
            }
            p += __shfl_xor_sync(0xffffffffu, p, 8);
            p += __shfl_xor_sync(0xffffffffu, p, 16);
            if (cl == 0 && row < a.n) Pp[row] = p;
        }
    }
}

void launch_solve(const SolveArgs& a_in, cudaStream_t st) {
    SolveArgs a = a_in;
    static int max_smem = 0;
    if (!max_smem) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    }
    // deepest ring that fits: the ring hides the L2 latency of the L-block stream
    int stages = kMaxStages;
    while (stages > 2 && solve_smem_bytes_stages(a.nblk, stages) > (size_t)max_smem) --stages;
    a.stages = stages;
    // right-hand-side rows staged per round: as many times (multiple of 4) as fit into the ring area
    {
        size_t ring_bytes = (size_t)stages * kLBlkDoubles * 8, row_bytes = (size_t)a.nblk * 32 * 16;
        int rpr = (int)(ring_bytes / row_bytes) / 4 * 4;
        a.rows_per_round = rpr >= kTT ? kTT : (rpr >= 8 ? 8 : 4);
        if (ring_bytes < 4 * row_bytes) return;  // excluded by solve_resident_ok (the engine never launches this)
    }
    size_t smem = solve_smem_bytes_stages(a.nblk, stages);
    static size_t attr_dev[kMaxDev] = {0};
    size_t& attr_smem = attr_dev[current_device_slot()];
    if (smem > attr_smem) {
        cudaFuncSetAttribute(k_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_smem = smem;
    }
    k_solve<<<dim3(a.ntiles, a.nsys), 544, smem, st>>>(a);
}

}  // namespace hp
