// hp_eigh.cu -- batched Hermitian eigendecomposition on the device (one-sided Jacobi), for a non-delay-diagonal S_initial.
//
// The reference takes scipy's sqrtm of whatever signal covariance it is given (build_matrices, pspec.py:355); the GPU path
// works in the eigenbasis of S (DESIGN.md section 2), which for a general S_initial (run-hydra-pspec.py --sigcov0) means one
// Hermitian eigendecomposition per baseline before the chain is loaded.  Round 1 did that with numpy on the host (30 - 50 ms
// per 384 x 384 matrix, one after the other); here a batch of matrices is decomposed on the device.
//
// One-sided (Hestenes) Jacobi on G = S: pairs of columns are rotated until all columns of G are mutually orthogonal, the
// same rotations are accumulated in V (starting from I).  At convergence G = S V with orthogonal columns, i.e. the columns
// of V are eigenvectors and lambda_j = v_j^H (S v_j) = v_j^H g_j (signed, so a slightly indefinite input is reported as
// such and clipped by the caller).  Rotations of disjoint pairs commute: a sweep is n - 1 rounds of n / 2 disjoint pairs
// (round-robin tournament), a warp per pair, one launch per round for the whole batch.  Columns are contiguous (column-major
// work arrays), so every access is coalesced; V stays unitary to round-off by construction.
#include "hp_kernels.cuh"
#include "../../include/hydra_pspec_b200.h"
#include <vector>

namespace hp {
namespace {

constexpr int kEighWarps = 8;   // pairs per CTA of a round

// G, V: [n][n] complex, column c at c * n (element r at c * n + r).  S: [n][n] row-major Hermitian.
__global__ void __launch_bounds__(256) k_eigh_init(const double2* __restrict__ S_all, double2* G_all, double2* V_all, int n) {
    const size_t nn = (size_t)n * n;
    const double2* S = S_all + blockIdx.y * nn;
    double2* G = G_all + blockIdx.y * nn;
    double2* V = V_all + blockIdx.y * nn;
    for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < nn; e += (size_t)gridDim.x * 256) {
        const int c = (int)(e / n), r = (int)(e - (size_t)c * n);
        const double2 s = S[e];                       // column c of S = conjugate of row c (Hermitian): contiguous reads
        G[e] = make_double2(s.x, -s.y);
        V[e] = make_double2(r == c ? 1.0 : 0.0, 0.0);
    }
}

// One round of the tournament: the ne / 2 disjoint column pairs of round `round`, a warp per pair, for every matrix of the
// batch (blockIdx.y).  rotated[matrix] is set when a pair was not yet orthogonal.  kNJ > 0: n <= 32 kNJ, the two columns of G
// stay in registers between the inner products and the rotation (one read instead of two, all loads issued up front).
template <int kNJ>
__global__ void __launch_bounds__(32 * kEighWarps) k_eigh_round(double2* G_all, double2* V_all, int n, int ne, int round, double tol,
                                                                 int* rotated) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * kEighWarps + (threadIdx.x >> 5);
    if (i >= ne / 2) return;
    int p, q;
    if (i == 0) { p = ne - 1; q = round; }
    else { p = (round + i) % (ne - 1); q = (round - i + (ne - 1)) % (ne - 1); }
    if (p >= n || q >= n) return;                     // the dummy player of an odd n
    if (p > q) { const int t = p; p = q; q = t; }
    const size_t nn = (size_t)n * n;
    double2* G = G_all + blockIdx.y * nn;
    double2* V = V_all + blockIdx.y * nn;
    double2* x = G + (size_t)p * n;
    double2* y = G + (size_t)q * n;
    constexpr int kR = kNJ > 0 ? kNJ : 1;
    double2 xa[kR], ya[kR];
    double al = 0.0, be = 0.0, gr = 0.0, gi = 0.0;
    if (kNJ > 0) {
#pragma unroll
        for (int u = 0; u < kR; ++u) {
            const int r = lane + 32 * u;
            xa[u] = r < n ? x[r] : make_double2(0.0, 0.0);
            ya[u] = r < n ? y[r] : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int u = 0; u < kR; ++u) {
            const double2 a = xa[u], b = ya[u];
            al += a.x * a.x + a.y * a.y;
            be += b.x * b.x + b.y * b.y;
            gr += a.x * b.x + a.y * b.y;              // conj(a) b
            gi += a.x * b.y - a.y * b.x;
        }
    } else {
        for (int r = lane; r < n; r += 32) {
            const double2 a = x[r], b = y[r];
            al += a.x * a.x + a.y * a.y;
            be += b.x * b.x + b.y * b.y;
            gr += a.x * b.x + a.y * b.y;
            gi += a.x * b.y - a.y * b.x;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        al += __shfl_xor_sync(0xffffffffu, al, o); be += __shfl_xor_sync(0xffffffffu, be, o);
        gr += __shfl_xor_sync(0xffffffffu, gr, o); gi += __shfl_xor_sync(0xffffffffu, gi, o);
    }
    const double g2 = gr * gr + gi * gi;
    if (!(g2 > tol * tol * al * be) || g2 == 0.0) return;
    const double ga = sqrt(g2);
    // y' = e^{-i phi} y makes x^H y' = |gamma| real; then the real Jacobi rotation that orthogonalises (x, y')
    const double er = gr / ga, ei = -gi / ga;         // e^{-i phi}
    const double zeta = (be - al) / (2.0 * ga);
    const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
    const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
    auto rot = [&](double2 a, double2 b0, double2& xo, double2& yo) {
        const double2 b = make_double2(b0.x * er - b0.y * ei, b0.x * ei + b0.y * er);
        xo = make_double2(c * a.x - s * b.x, c * a.y - s * b.y);
        yo = make_double2(s * a.x + c * b.x, s * a.y + c * b.y);
    };
    double2* vx = V + (size_t)p * n;
    double2* vy = V + (size_t)q * n;
    if (kNJ > 0) {
#pragma unroll
        for (int u = 0; u < kR; ++u) {
            const int r = lane + 32 * u;
            if (r < n) { double2 xo, yo; rot(xa[u], ya[u], xo, yo); x[r] = xo; y[r] = yo; }
        }
    } else {
        for (int r = lane; r < n; r += 32) { double2 xo, yo; rot(x[r], y[r], xo, yo); x[r] = xo; y[r] = yo; }
    }
#pragma unroll 4
    for (int r = lane; r < n; r += 32) { double2 xo, yo; rot(vx[r], vy[r], xo, yo); vx[r] = xo; vy[r] = yo; }
    if (lane == 0) rotated[blockIdx.y] = 1;
}

// Blocked round: a CTA takes a PAIR OF COLUMN BLOCKS (2 bw columns of G and of V) into shared memory, runs a full inner
// tournament over those columns there (a warp per pair, one CTA barrier per inner round) and writes them back.  A sweep over
// the blocks is nb - 1 launches instead of n - 1, and every column crosses L2 once per launch instead of once per pair: ~10x
// less L2 traffic at n = 384, bw = 8 (the unblocked rounds are L2-bandwidth bound for a batch of matrices).
__global__ void __launch_bounds__(256) k_eigh_block_round(double2* G_all, double2* V_all, int n, int nb, int nbe, int bw, int round,
                                                          double tol, int* rotated) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* gs = reinterpret_cast<double2*>(smem_raw);     // [2 bw][n]
    double2* vs = gs + (size_t)2 * bw * n;                  // [2 bw][n]
    const int i = blockIdx.x;
    int P, Q;
    if (i == 0) { P = nbe - 1; Q = round; }
    else { P = (round + i) % (nbe - 1); Q = (round - i + (nbe - 1)) % (nbe - 1); }
    if (P >= nb || Q >= nb) return;                         // the dummy block of an odd number of blocks
    if (P > Q) { const int t = P; P = Q; Q = t; }
    const int cP = min(bw, n - P * bw), cQ = min(bw, n - Q * bw), m = cP + cQ;
    const size_t nn = (size_t)n * n;
    double2* G = G_all + blockIdx.y * nn;
    double2* V = V_all + blockIdx.y * nn;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
    auto gcol = [&](int j) { return j < cP ? P * bw + j : Q * bw + (j - cP); };   // local column -> column of the matrix
    for (int j = 0; j < m; ++j) {
        const size_t src = (size_t)gcol(j) * n;
        for (int r = tid; r < n; r += nthr) { gs[(size_t)j * n + r] = G[src + r]; vs[(size_t)j * n + r] = V[src + r]; }
    }
    __syncthreads();
    const int me = m + (m & 1);
    bool any = false;
    for (int ir = 0; ir < me - 1; ++ir) {
        if (warp < me / 2) {
            int a, b;
            if (warp == 0) { a = me - 1; b = ir; }
            else { a = (ir + warp) % (me - 1); b = (ir - warp + (me - 1)) % (me - 1); }
            if (a < m && b < m) {
                if (a > b) { const int t = a; a = b; b = t; }
                double2* x = gs + (size_t)a * n;
                double2* y = gs + (size_t)b * n;
                double al = 0.0, be = 0.0, gr = 0.0, gi = 0.0;
                for (int r = lane; r < n; r += 32) {
                    const double2 u = x[r], v = y[r];
                    al += u.x * u.x + u.y * u.y;
                    be += v.x * v.x + v.y * v.y;
                    gr += u.x * v.x + u.y * v.y;
                    gi += u.x * v.y - u.y * v.x;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    al += __shfl_xor_sync(0xffffffffu, al, o); be += __shfl_xor_sync(0xffffffffu, be, o);
                    gr += __shfl_xor_sync(0xffffffffu, gr, o); gi += __shfl_xor_sync(0xffffffffu, gi, o);
                }
                const double g2 = gr * gr + gi * gi;
                if (g2 > tol * tol * al * be && g2 != 0.0) {
                    const double ga = sqrt(g2);
                    const double er = gr / ga, ei = -gi / ga;
                    const double zeta = (be - al) / (2.0 * ga);
                    const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                    const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
                    double2* vx = vs + (size_t)a * n;
                    double2* vy = vs + (size_t)b * n;
                    for (int r = lane; r < n; r += 32) {
                        {
                            const double2 u = x[r], w0 = y[r];
                            const double2 w = make_double2(w0.x * er - w0.y * ei, w0.x * ei + w0.y * er);
                            x[r] = make_double2(c * u.x - s * w.x, c * u.y - s * w.y);
                            y[r] = make_double2(s * u.x + c * w.x, s * u.y + c * w.y);
                        }
                        {
                            const double2 u = vx[r], w0 = vy[r];
                            const double2 w = make_double2(w0.x * er - w0.y * ei, w0.x * ei + w0.y * er);
                            vx[r] = make_double2(c * u.x - s * w.x, c * u.y - s * w.y);
                            vy[r] = make_double2(s * u.x + c * w.x, s * u.y + c * w.y);
                        }
                    }
                    any = true;
                }
            }
        }
        __syncthreads();
    }
    for (int j = 0; j < m; ++j) {
        const size_t dst = (size_t)gcol(j) * n;
        for (int r = tid; r < n; r += nthr) { G[dst + r] = gs[(size_t)j * n + r]; V[dst + r] = vs[(size_t)j * n + r]; }
    }
    if (any && lane == 0) rotated[blockIdx.y] = 1;
}

// lambda_j = Re(v_j^H g_j) (g_j = S v_j); eigenvectors as the columns of a row-major matrix (numpy.linalg.eigh convention)
__global__ void __launch_bounds__(256) k_eigh_finish(const double2* __restrict__ G_all, const double2* __restrict__ V_all, double* w_all,
                                                     double2* Vout_all, int n) {
    const size_t nn = (size_t)n * n;
    const double2* G = G_all + blockIdx.y * nn;
    const double2* V = V_all + blockIdx.y * nn;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int j = blockIdx.x * 8 + warp; j < n; j += gridDim.x * 8) {
        const double2* g = G + (size_t)j * n;
        const double2* v = V + (size_t)j * n;
        double acc = 0.0;
        for (int r = lane; r < n; r += 32) acc += v[r].x * g[r].x + v[r].y * g[r].y;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) w_all[blockIdx.y * (size_t)n + j] = acc;
    }
    double2* Vout = Vout_all + blockIdx.y * nn;
    for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < nn; e += (size_t)gridDim.x * 256) {
        const int r = (int)(e / n), j = (int)(e - (size_t)r * n);
        Vout[e] = V[(size_t)j * n + r];
    }
}

}  // namespace
}  // namespace hp

extern "C" int hp_eigh_batch(int device, int n, int batch, const double* S, double* V, double* w, int* sweeps) {
    if (!S || !V || !w || n < 1 || batch < 1) return HP_ERR_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return HP_ERR_CUDA;   // no CPU fallback
    if (cudaSetDevice(device) != cudaSuccess) return HP_ERR_CUDA;
    const size_t nn = (size_t)n * n;
    double2 *dS = nullptr, *dG = nullptr, *dV = nullptr, *dVo = nullptr;
    double* dw = nullptr;
    int* dsw = nullptr;
    cudaError_t e = cudaMalloc(&dS, 16 * nn * batch);
    if (e == cudaSuccess) e = cudaMalloc(&dG, 16 * nn * batch);
    if (e == cudaSuccess) e = cudaMalloc(&dV, 16 * nn * batch);
    if (e == cudaSuccess) e = cudaMalloc(&dVo, 16 * nn * batch);
    if (e == cudaSuccess) e = cudaMalloc(&dw, 8 * (size_t)n * batch);
    if (e == cudaSuccess) e = cudaMalloc(&dsw, sizeof(int) * batch);
    if (e == cudaSuccess) e = cudaMemcpy(dS, S, 16 * nn * batch, cudaMemcpyHostToDevice);
    int sweeps_used = 0;
    if (e == cudaSuccess) {
        // A sweep = ne - 1 rounds of ne / 2 disjoint pairs; one launch per round spreads a round over the whole GPU whatever
        // the batch size (one CTA per matrix was bound by a single SM's L2 bandwidth: 0.55 s for one 384 x 384 matrix).
        const int ne = n + (n & 1), max_sweeps = 30;
        const double tol = 1e-13;
        const dim3 grid((ne / 2 + hp::kEighWarps - 1) / hp::kEighWarps, batch);
        // blocked rounds when two blocks of >= 2 columns (G and V) fit the shared memory of a CTA
        int max_smem = 0;
        cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
        int bw = (int)((size_t)(max_smem > 8192 ? max_smem - 8192 : 0) / ((size_t)4 * n * 16));
        if (bw > 8) bw = 8;
        const int nb = bw >= 2 ? (n + bw - 1) / bw : 0, nbe = nb + (nb & 1);
        const size_t bsmem = (size_t)4 * bw * n * 16;
        if (bw >= 2) cudaFuncSetAttribute(hp::k_eigh_block_round, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem);
        hp::k_eigh_init<<<dim3(64, batch), 256>>>(dS, dG, dV, n);
        std::vector<int> flag(batch);
        for (; sweeps_used < max_sweeps && e == cudaSuccess;) {
            cudaMemsetAsync(dsw, 0, sizeof(int) * batch, 0);
            if (bw >= 2 && nb >= 2) {
                for (int round = 0; round < nbe - 1; ++round)
                    hp::k_eigh_block_round<<<dim3(nbe / 2, batch), 32 * bw, bsmem>>>(dG, dV, n, nb, nbe, bw, round, tol, dsw);
            } else {
                for (int round = 0; round < ne - 1; ++round) {
                    if (n <= 256) hp::k_eigh_round<8><<<grid, 32 * hp::kEighWarps>>>(dG, dV, n, ne, round, tol, dsw);
                    else if (n <= 512) hp::k_eigh_round<16><<<grid, 32 * hp::kEighWarps>>>(dG, dV, n, ne, round, tol, dsw);
                    else hp::k_eigh_round<0><<<grid, 32 * hp::kEighWarps>>>(dG, dV, n, ne, round, tol, dsw);
                }
            }
            ++sweeps_used;
            e = cudaMemcpy(flag.data(), dsw, sizeof(int) * batch, cudaMemcpyDeviceToHost);
            bool any = false;
            for (int f : flag) any |= (f != 0);
            if (!any) break;
        }
        if (e == cudaSuccess) {
            hp::k_eigh_finish<<<dim3(32, batch), 256>>>(dG, dV, dw, dVo, n);
            e = cudaDeviceSynchronize();
        }
    }
    if (e == cudaSuccess) e = cudaMemcpy(V, dVo, 16 * nn * batch, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(w, dw, 8 * (size_t)n * batch, cudaMemcpyDeviceToHost);
    if (sweeps) for (int b = 0; b < batch; ++b) sweeps[b] = sweeps_used;
    cudaFree(dS); cudaFree(dG); cudaFree(dV); cudaFree(dVo); cudaFree(dw); cudaFree(dsw);
    return e == cudaSuccess ? HP_OK : HP_ERR_CUDA;
}
