// hp_zgemm.cu -- k_zgemm2: strided batched complex128 GEMM on the FP64 tensor pipe,  C (+)= alpha opA(A) diag(dk) opB(B).
//
// Carries every dense contraction that is not one of the resident solves: the Gram matrix and right-hand-side products
// of build_matrices (pspec.py:325-374) at chain load, the two triangular products of the N > 576 solve and the
// dense-noise ln-posterior term (pspec.py:474-478) per iteration (BASELINE.json configs[4]), and P = A^H R of the
// per-time low-rank form (hp_ptlow.cu, configs[2]).
//
// The round-1 kernel staged 64 x 64 x 16 tiles through registers into planar shared memory, 8 warps with 32 x 16 tiles and
// four real DMMAs per complex MAC: 0.60 of the DMMA peak at configs[4].  This one follows what k_solve3 showed to work
// (profiles/r2_dmma_mix.txt: 12 DMMA + 4 DADD + 8 LDS per k-step sustain 95 % of the pipe with four warps per scheduler):
//   * 16 warps, each a 16 x 16 complex tile with the 3M scheme (three real products per complex MAC, 48 accumulators);
//   * operands go global -> shared with cp.async (16 bytes = one complex element, any stride, zero-filled outside the
//     matrix or the triangular K range), three stages of 64 x 32 (A) and 32 x 64 (B), one barrier per 32-deep k-tile;
//   * interleaved (re, im) shared-memory tiles read as conflict-free LDS.128 fragments (leading dimensions 36 and 66
//     complex elements); conjugation and the diagonal scale are applied to the fragments.
// Tried and not kept: persistent CTAs (one per SM) with the cp.async pipeline running across output tiles -- the static
// tile assignment loses more to the uneven k-ranges of a triangular B than the hidden pipeline fills gain (configs[4] solve
// class 12.2 -> 12.5 ms, ln-posterior term 5.0 -> 5.2 ms even with a grid size coprime to the number of column tiles).
#include "hp_kernels.cuh"
#include "hp_mma.cuh"

namespace hp {
namespace {

constexpr int Z2_BM = 64, Z2_BN = 64, Z2_BK = 32, Z2_THREADS = 512, Z2_STAGES = 3;
constexpr int Z2_LDA = 36;   // complex elements per row of the A tile ([i][k]); == 4 (mod 8): conflict-free LDS.128 fragments
constexpr int Z2_LDB = 66;   // complex elements per row of the B tile ([k][j]); == 2 (mod 8)
constexpr int Z2_A_ELEMS = Z2_BM * Z2_LDA, Z2_B_ELEMS = Z2_BK * Z2_LDB;
constexpr size_t Z2_SMEM = (size_t)Z2_STAGES * (Z2_A_ELEMS + Z2_B_ELEMS) * sizeof(double2);

__device__ __forceinline__ void z2_cp16(void* smem_dst, const void* gmem_src, bool valid) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int bytes = valid ? 16 : 0;   // 0: nothing is read, the 16 bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem_src), "r"(bytes) : "memory");
}

__global__ void __launch_bounds__(Z2_THREADS, 1) k_zgemm2(ZgemmArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* As = reinterpret_cast<double2*>(smem_raw);                  // [stage][64][36]
    double2* Bs = As + Z2_STAGES * Z2_A_ELEMS;                           // [stage][32][66]
    const int i0 = blockIdx.y * Z2_BM, j0 = blockIdx.x * Z2_BN;
    if (a.lower_out && j0 > i0 + Z2_BM - 1) return;   // Hermitian result: only tiles that touch the lower triangle
    const int b = blockIdx.z;
    const double2* A = reinterpret_cast<const double2*>(a.A) + a.bsA * b;
    const double2* B = reinterpret_cast<const double2*>(a.B) + a.bsB * b;
    double* C = a.C + 2 * a.bsC * b;
    const double* dk = a.dk ? a.dk + a.bsD * b : nullptr;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, q = lane & 3;
    const int wr = warp >> 2, wc = warp & 3;          // warp tile: rows 16 wr .., columns 16 wc ..
    const bool a_kfast = a.sAk <= a.sAi, b_jfast = a.sBj <= a.sBk;
    const double sa = a.conjA ? -1.0 : 1.0, sb = a.conjB ? -1.0 : 1.0;
    // triangular B: skip the K range where this column tile of B is structurally zero
    //   tri = 1: B[k][j] = 0 for k > j  (k < j0 + BN suffices);   tri = 2: B[k][j] = 0 for k < j  (start at k = j0)
    const int kbeg = a.tri == 2 ? (j0 / Z2_BK) * Z2_BK : 0;
    const int kend = a.tri == 1 ? (a.K < j0 + Z2_BN ? a.K : j0 + Z2_BN) : a.K;
    const int ntile = kend > kbeg ? (kend - kbeg + Z2_BK - 1) / Z2_BK : 0;

    auto issue = [&](int kt) {
        const int k0 = kbeg + kt * Z2_BK, st = kt % Z2_STAGES;
        double2* as = As + st * Z2_A_ELEMS;
        double2* bs = Bs + st * Z2_B_ELEMS;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int e = tid + Z2_THREADS * r;
            int i, k;
            if (a_kfast) { i = e >> 5; k = e & 31; } else { i = e & 63; k = e >> 6; }
            const bool ok = i0 + i < a.M && k0 + k < kend;
            const double2* src = ok ? A + ((long long)(i0 + i) * a.sAi + (long long)(k0 + k) * a.sAk) : A;
            z2_cp16(as + i * Z2_LDA + k, src, ok);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int e = tid + Z2_THREADS * r;
            int k, j;
            if (b_jfast) { k = e >> 6; j = e & 63; } else { k = e & 31; j = e >> 5; }
            const bool ok = k0 + k < kend && j0 + j < a.N;
            const double2* src = ok ? B + ((long long)(k0 + k) * a.sBk + (long long)(j0 + j) * a.sBj) : B;
            z2_cp16(bs + k * Z2_LDB + j, src, ok);
        }
    };

    double P[3][2][2][2];
    warp_zero3m<2, 2>(P);
#pragma unroll
    for (int s = 0; s < Z2_STAGES - 1; ++s) {
        if (s < ntile) issue(s);
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (int kt = 0; kt < ntile; ++kt) {
        asm volatile("cp.async.wait_group %0;" ::"n"(Z2_STAGES - 2) : "memory");
        __syncthreads();   // tile kt has landed for every thread; the stage refilled below was read in iteration kt - 1
        if (kt + Z2_STAGES - 1 < ntile) issue(kt + Z2_STAGES - 1);
        asm volatile("cp.async.commit_group;" ::: "memory");
        const int st = kt % Z2_STAGES, k0 = kbeg + kt * Z2_BK;
        const double2* as = As + st * Z2_A_ELEMS + (16 * wr + g) * Z2_LDA + q;
        const double2* bs = Bs + st * Z2_B_ELEMS + q * Z2_LDB + 16 * wc + g;
#pragma unroll
        for (int kk = 0; kk < Z2_BK; kk += 4) {
            double ar[2], ai[2], as3[2], br[2], bi[2], bs3[2];
            double d = 1.0;
            if (dk) { const int kg = k0 + kk + q; d = kg < kend ? dk[kg] : 0.0; }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const double2 v = as[8 * i * Z2_LDA + kk];
                ar[i] = v.x * d; ai[i] = sa * v.y * d;
                as3[i] = ar[i] + ai[i];
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const double2 v = bs[kk * Z2_LDB + 8 * j];
                br[j] = v.x; bi[j] = sb * v.y;
                bs3[j] = br[j] + bi[j];
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    dmma884(P[0][i][j][0], P[0][i][j][1], ar[i], br[j]);
                    dmma884(P[1][i][j][0], P[1][i][j][1], ai[i], bi[j]);
                    dmma884(P[2][i][j][0], P[2][i][j][1], as3[i], bs3[j]);
                }
        }
    }
    // C = (P0 - P1) + i (P2 - P0 - P1)   (the conjugations are already in the signs of the imaginary fragments)
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int row = i0 + 16 * wr + 8 * i + g, col = j0 + 16 * wc + 8 * j + 2 * q + e;
                if (row < a.M && col < a.N) {
                    double* p = C + 2 * ((long long)row * a.sCi + (long long)col * a.sCj);
                    double vr = a.alpha * (P[0][i][j][e] - P[1][i][j][e]);
                    double vi = a.alpha * (P[2][i][j][e] - P[0][i][j][e] - P[1][i][j][e]);
                    if (a.accumulate) { vr += p[0]; vi += p[1]; }
                    p[0] = vr; p[1] = vi;
                }
            }
}

}  // namespace

void launch_zgemm(const ZgemmArgs& a, cudaStream_t st) {
    static bool attr_dev[kMaxDev] = {false};
    bool& done = attr_dev[current_device_slot()];
    if (!done) {
        cudaFuncSetAttribute(k_zgemm2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Z2_SMEM);
        done = true;
    }
    dim3 grid((a.N + Z2_BN - 1) / Z2_BN, (a.M + Z2_BM - 1) / Z2_BM, a.batch);
    k_zgemm2<<<grid, Z2_THREADS, Z2_SMEM, st>>>(a);
}

}  // namespace hp
