// hp_testhooks.cu -- host-in / host-out wrappers around single kernels, for tests/ only.
#include "../../include/hydra_pspec_b200.h"
#include "hp_kernels.cuh"

#include <string>
#include <vector>

extern "C" {

// C (M x N) = opA(A) (M x K) . opB(B) (K x N), all row-major complex128 host arrays.
//   transA: 0 = A is M x K, 1 = A is K x M (transposed storage);  conjA likewise; same for B.
int hp_test_zgemm(int M, int N, int K, const double* A, int transA, int conjA, const double* B, int transB, int conjB,
                  const double* dk, double* C) {
    double *dA, *dB, *dC, *dD = nullptr;
    if (cudaMalloc(&dA, 16ull * M * K) || cudaMalloc(&dB, 16ull * K * N) || cudaMalloc(&dC, 16ull * M * N)) return HP_ERR_CUDA;
    cudaMemcpy(dA, A, 16ull * M * K, cudaMemcpyHostToDevice);
    cudaMemcpy(dB, B, 16ull * K * N, cudaMemcpyHostToDevice);
    if (dk) { cudaMalloc(&dD, 8ull * K); cudaMemcpy(dD, dk, 8ull * K, cudaMemcpyHostToDevice); }
    hp::ZgemmArgs g{};
    g.A = dA; g.sAi = transA ? 1 : K; g.sAk = transA ? M : 1; g.conjA = conjA;
    g.B = dB; g.sBk = transB ? 1 : N; g.sBj = transB ? K : 1; g.conjB = conjB;
    g.C = dC; g.sCi = N; g.sCj = 1; g.dk = dD;
    g.M = M; g.N = N; g.K = K; g.alpha = 1.0; g.batch = 1;
    hp::launch_zgemm(g, 0);
    cudaError_t e = cudaDeviceSynchronize();
    cudaMemcpy(C, dC, 16ull * M * N, cudaMemcpyDeviceToHost);
    cudaFree(dA); cudaFree(dB); cudaFree(dC); cudaFree(dD);
    return e == cudaSuccess ? HP_OK : HP_ERR_CUDA;
}

// Factor M = J + D G D (G dense N x N Hermitian, lam[N] with lam = 1 on the rows >= n) and solve
// M X = R for T right-hand sides given as R[T][N] (already whitened: no lam scaling is applied
// by the caller -- the kernel multiplies Rfix by lam, so pass Rfix and lam separately).
//   Ldense [N][N] (lower triangle, optional), X [T][N].
int hp_test_chol_solve(int n, int m, int T, const double* G, const double* lam, const double* Rfix, const double* wa,
                       int cg_compat, double* Ldense, double* X, int* info) {
    const int N = n + m, nblk = (N + 31) / 32, Np = nblk * 32, ntiles = (T + 15) / 16, Tp = ntiles * 16;
    double *dG, *dGp, *dlam, *dLp, *dLinv, *dWp, *dR, *dW = nullptr, *dX, *dS, *dP;
    int* dinfo;
    size_t tri = hp::tri_blocks(nblk) * hp::kLBlkDoubles, trig = hp::tri_blocks(nblk) * hp::kBlkDoubles;
    cudaMalloc(&dG, 16ull * N * N); cudaMalloc(&dGp, 8 * trig); cudaMalloc(&dlam, 8ull * Np); cudaMalloc(&dLp, 8 * tri);
    cudaMalloc(&dLinv, 8ull * nblk * hp::kLBlkDoubles); cudaMalloc(&dWp, 8 * tri); cudaMalloc(&dR, 16ull * Tp * Np); cudaMalloc(&dX, 16ull * Tp * Np);
    cudaMalloc(&dS, 16ull * Tp * n); cudaMalloc(&dP, 8ull * ntiles * n); cudaMalloc(&dinfo, 4);
    cudaMemset(dR, 0, 16ull * Tp * Np); cudaMemset(dlam, 0, 8ull * Np);
    cudaMemcpy(dG, G, 16ull * N * N, cudaMemcpyHostToDevice);
    cudaMemcpy(dlam, lam, 8ull * N, cudaMemcpyHostToDevice);
    cudaMemcpy2D(dR, 16ull * Np, Rfix, 16ull * N, 16ull * N, T, cudaMemcpyHostToDevice);
    if (wa) {
        cudaMalloc(&dW, 16ull * Tp * Np); cudaMemset(dW, 0, 16ull * Tp * Np);
        cudaMemcpy2D(dW, 16ull * Np, wa, 16ull * n, 16ull * n, T, cudaMemcpyHostToDevice);
    }
    hp::launch_pack_lower(dG, N, 0, dGp, N, nblk, 1, 0);
    hp::CholArgs ca{};
    ca.Gp = dGp; ca.lam = dlam; ca.Lp = dLp; ca.Linvp = dLinv; ca.info = dinfo; ca.nblk = nblk; ca.n = n; ca.N = N; ca.nsys = 1;
    hp::launch_chol_trinv(ca, dWp, hp::TrinvExtra{nullptr, nullptr, nullptr}, 0);
    hp::SolveArgs sa{};
    sa.Wp = dWp; sa.lam = dlam; sa.Rfix = dR; sa.wa = dW; sa.X = dX; sa.Ssc = dS; sa.Ppart = dP;
    sa.nblk = nblk; sa.n = n; sa.N = N; sa.Tp = Tp; sa.ntiles = ntiles; sa.nsys = 1; sa.T = T; sa.cg_compat = cg_compat;
    hp::launch_solve(sa, 0);
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) {
        cudaMemcpy2D(X, 16ull * N, dX, 16ull * Np, 16ull * N, T, cudaMemcpyDeviceToHost);
        cudaMemcpy(info, dinfo, 4, cudaMemcpyDeviceToHost);
        if (Ldense) {
            std::vector<double> lp(tri);
            cudaMemcpy(lp.data(), dLp, 8 * tri, cudaMemcpyDeviceToHost);
            for (int i = 0; i < N; ++i)
                for (int j = 0; j < N; ++j) {
                    double re = 0, im = 0;
                    if (j <= i) {
                        const double* b = lp.data() + hp::blk_index(i / 32, j / 32) * hp::kLBlkDoubles;
                        re = b[(i % 32) * hp::kLdBlk + (j % 32)]; im = b[hp::kLPlane + (i % 32) * hp::kLdBlk + (j % 32)];
                    }
                    Ldense[2 * ((size_t)i * N + j)] = re; Ldense[2 * ((size_t)i * N + j) + 1] = im;
                }
        }
    }
    cudaFree(dG); cudaFree(dGp); cudaFree(dlam); cudaFree(dLp); cudaFree(dLinv); cudaFree(dWp); cudaFree(dR); cudaFree(dW); cudaFree(dX);
    cudaFree(dS); cudaFree(dP); cudaFree(dinfo);
    return e == cudaSuccess ? HP_OK : HP_ERR_CUDA;
}


// The same factorisation followed by k_solve3 (hp_solve3.cu) for `nsys` systems that share G and lam but have their own
// right-hand sides Rfix[nsys][T][N] (and wa[nsys][T][n]).  wa == NULL: unscaled right-hand sides in tile layout and
// Wf1 = W diag(lam) (the Philox-mode data flow, without the noise); wa != NULL: r = lam * Rfix + wa built by k_rhs_tile
// and Wf1 = W.  grid_limit > 0 caps the persistent grid (several tiles per CTA at test sizes).
// X [nsys][T][N]; psum [nsys][n] = sum_t |x_k|^2 from the kernel's partial sums (or NULL).
int hp_test_solve3(int n, int m, int T, int nsys, const double* G, const double* lam, const double* Rfix, const double* wa,
                   int cg_compat, int grid_limit, double* X, double* psum) {
    const int N = n + m, nblk = (N + 31) / 32, Np = nblk * 32, ntiles = (T + 15) / 16, Tp = ntiles * 16;
    int max_smem = 0, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (!hp::solve3_ok(nblk, (size_t)max_smem)) return HP_ERR_SIZE;
    const size_t wf = hp::solve3_frag_doubles(nblk);
    double *dG, *dGp, *dlam, *dLp, *dLinv, *dWp, *dR, *dW = nullptr, *dX, *dP, *dRt, *dWf1, *dWf2;
    int* dinfo;
    const size_t tri = hp::tri_blocks(nblk) * hp::kLBlkDoubles, trig = hp::tri_blocks(nblk) * hp::kBlkDoubles;
    const size_t rt_doubles = (size_t)nsys * ntiles * nblk * 2 * 32 * hp::kTT;
    cudaMalloc(&dG, 16ull * N * N); cudaMalloc(&dGp, 8 * trig); cudaMalloc(&dlam, 8ull * Np); cudaMalloc(&dLp, 8 * tri);
    cudaMalloc(&dLinv, 8ull * nblk * hp::kLBlkDoubles); cudaMalloc(&dWp, 8 * tri);
    cudaMalloc(&dR, 16ull * nsys * Tp * Np); cudaMalloc(&dX, 16ull * nsys * Tp * Np);
    cudaMalloc(&dP, 8ull * nsys * ntiles * n); cudaMalloc(&dinfo, 4); cudaMalloc(&dRt, 8 * rt_doubles);
    cudaMemset(dR, 0, 16ull * nsys * Tp * Np); cudaMemset(dlam, 0, 8ull * Np); cudaMemset(dX, 0xff, 16ull * nsys * Tp * Np);
    cudaMemcpy(dG, G, 16ull * N * N, cudaMemcpyHostToDevice);
    cudaMemcpy(dlam, lam, 8ull * N, cudaMemcpyHostToDevice);
    for (int s = 0; s < nsys; ++s)
        cudaMemcpy2D(dR + 2ull * s * Tp * Np, 16ull * Np, Rfix + 2ull * s * T * N, 16ull * N, 16ull * N, T, cudaMemcpyHostToDevice);
    if (wa) {
        cudaMalloc(&dW, 16ull * nsys * Tp * Np); cudaMemset(dW, 0, 16ull * nsys * Tp * Np);
        for (int s = 0; s < nsys; ++s)
            cudaMemcpy2D(dW + 2ull * s * Tp * Np, 16ull * Np, wa + 2ull * s * T * n, 16ull * n, 16ull * n, T, cudaMemcpyHostToDevice);
    }
    hp::launch_pack_lower(dG, N, 0, dGp, N, nblk, 1, 0);
    hp::CholArgs ca{};
    ca.Gp = dGp; ca.lam = dlam; ca.Lp = dLp; ca.Linvp = dLinv; ca.info = dinfo; ca.nblk = nblk; ca.n = n; ca.N = N; ca.nsys = 1;
    cudaMalloc(&dWf1, 8 * wf * nsys); cudaMalloc(&dWf2, 8 * wf * nsys);
    cudaMemset(dWf1, 0xff, 8 * wf * nsys); cudaMemset(dWf2, 0xff, 8 * wf * nsys);   // NaN: every fragment must be written
    // wa given: r = lam * Rfix + wa is built by k_rhs_tile and pass 1 uses the unscaled W
    hp::launch_chol_trinv(ca, dWp, hp::TrinvExtra{dWf1, dWf2, wa ? nullptr : dlam}, 0);
    for (int s = 0; s < nsys; ++s) {
        // lam is shared by the systems while k_rhs_tile indexes lam by system: build the tiles one system at a time
        hp::launch_rhs_tile(dRt + (size_t)s * ntiles * nblk * 2 * 32 * hp::kTT, dR + 2ull * s * Tp * Np,
                            dW ? dW + 2ull * s * Tp * Np : nullptr, wa ? dlam : nullptr, nblk, n, N, T, Tp, ntiles, 1, 0);
    }
    // one solve launch covers all systems and expects per-system W: replicate the one factor
    for (int s = 1; s < nsys; ++s) {
        cudaMemcpy(dWf1 + wf * s, dWf1, 8 * wf, cudaMemcpyDeviceToDevice);
        cudaMemcpy(dWf2 + wf * s, dWf2, 8 * wf, cudaMemcpyDeviceToDevice);
    }
    hp::Solve3Args s3{};
    s3.Wf1 = dWf1; s3.Wf2 = dWf2; s3.Rt = dRt; s3.X = dX; s3.Ppart = dP;
    s3.nblk = nblk; s3.n = n; s3.N = N; s3.Tp = Tp; s3.ntiles = ntiles; s3.nsys = nsys; s3.T = T;
    s3.philox = 0; s3.grid_limit = grid_limit;
    s3.nstrip = (N + 15) / 16;
    hp::solve3_make_schedule(nblk, &s3.sched, s3.nstrip);
    hp::launch_solve3(s3, 0);
    if (cg_compat)
        for (int s = 0; s < nsys; ++s)
            hp::launch_cg_scale(dX + 2ull * s * Tp * Np, dR + 2ull * s * Tp * Np, dW ? dW + 2ull * s * Tp * Np : nullptr, dlam, n, N,
                                Np, T, Tp, 1, 0);
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) {
        for (int s = 0; s < nsys; ++s)
            cudaMemcpy2D(X + 2ull * s * T * N, 16ull * N, dX + 2ull * s * Tp * Np, 16ull * Np, 16ull * N, T, cudaMemcpyDeviceToHost);
        if (psum) {
            std::vector<double> pp((size_t)nsys * ntiles * n);
            cudaMemcpy(pp.data(), dP, 8 * pp.size(), cudaMemcpyDeviceToHost);
            for (int s = 0; s < nsys; ++s)
                for (int k = 0; k < n; ++k) {
                    double acc = 0.0;
                    for (int tl = 0; tl < ntiles; ++tl) acc += pp[((size_t)s * ntiles + tl) * n + k];
                    psum[(size_t)s * n + k] = acc;
                }
        }
    }
    cudaFree(dG); cudaFree(dGp); cudaFree(dlam); cudaFree(dLp); cudaFree(dLinv); cudaFree(dWp); cudaFree(dR);
    cudaFree(dW); cudaFree(dX); cudaFree(dP); cudaFree(dinfo); cudaFree(dRt); cudaFree(dWf1); cudaFree(dWf2);
    return e == cudaSuccess ? HP_OK : HP_ERR_CUDA;
}

// k_solve3's static work schedule (host logic; no device needed): n[2][kS3Warps], strips[2][kS3Warps][kS3MaxPerWarp]
int hp_test_solve3_schedule(int nblk, unsigned char* n, unsigned char* strips, int* nwarps, int* max_per_warp) {
    if (nblk < 1 || 2 * nblk > hp::kS3MaxStrips) return HP_ERR_SIZE;
    hp::Solve3Sched sc{};
    hp::solve3_make_schedule(nblk, &sc);
    for (int p = 0; p < 2; ++p)
        for (int w = 0; w < hp::kS3Warps; ++w) {
            n[p * hp::kS3Warps + w] = sc.n[p][w];
            for (int e = 0; e < hp::kS3MaxPerWarp; ++e) strips[(p * hp::kS3Warps + w) * hp::kS3MaxPerWarp + e] = sc.strip[p][w][e];
        }
    *nwarps = hp::kS3Warps;
    *max_per_warp = hp::kS3MaxPerWarp;
    return HP_OK;
}

// k_pt_lowrank (hp_ptlow.cu) alone, launched as solve_pt_lowrank launches it, for nsys systems of N = Np - padding unknowns
// with n columns of A each.  In: lam [nsys][N], Rfix [nsys][T][N], wa [nsys][T][n] or NULL, X0 [nsys][T][N] (x0_t = M_0^-1 b_t),
// Rcols [nsys][n][N] (row x = R[:, x]), P [nsys][n][n], fidx [nsys][T][64], fcnt [nsys][T], chain_ids [nsys] (read with
// philox only).  Out: X [nsys][T][N], info [nsys].  Every device element the kernel must not read is NaN: the padding columns
// N .. Np of every row, the rows T .. Tp0 of X and all rows Tp0 + x of Rfix.
int hp_test_pt_lowrank(int n, int N, int T, int nsys, const double* lam, const double* Rfix, const double* wa, const double* X0,
                       const double* Rcols, const double* P, const uint16_t* fidx, const int* fcnt, int philox, uint32_t key0,
                       uint32_t key1, uint32_t iter, const int* chain_ids, double* X, int* info) {
    if (n < 1 || N < n || T < 1 || nsys < 1) return HP_ERR_ARG;
    const int nblk = (N + 31) / 32, Np = nblk * 32;
    if (nblk > 14) return HP_ERR_SIZE;   // k_pt_lowrank<14> holds at most 14 rows per lane
    int kcap = 0;
    for (size_t i = 0; i < (size_t)nsys * T; ++i) {
        if (fcnt[i] < 0) return HP_ERR_ARG;
        if (fcnt[i] > hp::kPtLowMaxRank) return HP_ERR_SIZE;
        for (int e = 0; e < fcnt[i]; ++e)
            if (fidx[i * hp::kPtLowMaxRank + e] >= n) return HP_ERR_ARG;
        if (fcnt[i] > kcap) kcap = fcnt[i];
    }
    const int Tp0 = 16 * ((T + 15) / 16), Tp = Tp0 + 16 * ((n + 15) / 16);
    const size_t rows = (size_t)nsys * Tp;
    double *dlam, *dR, *dW = nullptr, *dX, *dP;
    uint16_t* dF;
    int *dC, *dinfo, *dch;
    if (cudaMalloc(&dlam, 8ull * nsys * Np) || cudaMalloc(&dR, 16 * rows * Np) || cudaMalloc(&dX, 16 * rows * Np) ||
        cudaMalloc(&dP, 16ull * nsys * n * n) || cudaMalloc(&dF, 2ull * nsys * T * hp::kPtLowMaxRank) ||
        cudaMalloc(&dC, 4ull * nsys * T) || cudaMalloc(&dinfo, 4ull * nsys) || cudaMalloc(&dch, 4ull * nsys) ||
        (wa && cudaMalloc(&dW, 16 * rows * Np)))
        return HP_ERR_CUDA;
    cudaMemset(dlam, 0xff, 8ull * nsys * Np);   // 0xff..: NaN
    cudaMemset(dR, 0xff, 16 * rows * Np);
    cudaMemset(dX, 0xff, 16 * rows * Np);
    cudaMemset(dinfo, 0, 4ull * nsys);
    cudaMemcpy2D(dlam, 8ull * Np, lam, 8ull * N, 8ull * N, nsys, cudaMemcpyHostToDevice);
    for (int s = 0; s < nsys; ++s) {
        const size_t d0 = 2ull * s * Tp * Np;
        cudaMemcpy2D(dR + d0, 16ull * Np, Rfix + 2ull * s * T * N, 16ull * N, 16ull * N, T, cudaMemcpyHostToDevice);
        cudaMemcpy2D(dX + d0, 16ull * Np, X0 + 2ull * s * T * N, 16ull * N, 16ull * N, T, cudaMemcpyHostToDevice);
        cudaMemcpy2D(dX + d0 + 2ull * Tp0 * Np, 16ull * Np, Rcols + 2ull * s * n * N, 16ull * N, 16ull * N, n, cudaMemcpyHostToDevice);
    }
    if (wa) {
        cudaMemset(dW, 0xff, 16 * rows * Np);
        for (int s = 0; s < nsys; ++s)
            cudaMemcpy2D(dW + 2ull * s * Tp * Np, 16ull * Np, wa + 2ull * s * T * n, 16ull * n, 16ull * n, T, cudaMemcpyHostToDevice);
    }
    cudaMemcpy(dP, P, 16ull * nsys * n * n, cudaMemcpyHostToDevice);
    cudaMemcpy(dF, fidx, 2ull * nsys * T * hp::kPtLowMaxRank, cudaMemcpyHostToDevice);
    cudaMemcpy(dC, fcnt, 4ull * nsys * T, cudaMemcpyHostToDevice);
    if (philox) cudaMemcpy(dch, chain_ids, 4ull * nsys, cudaMemcpyHostToDevice);
    else cudaMemset(dch, 0xff, 4ull * nsys);
    hp::PtLowArgs la{};
    la.Rfix = dR; la.wa = dW; la.lam = dlam; la.X = dX; la.Pm = dP; la.fidx = dF; la.fcnt = dC; la.info = dinfo;
    la.n = n; la.N = N; la.Np = Np; la.T = T; la.Tp = Tp; la.Tp0 = Tp0; la.nsys = nsys; la.nblk = nblk; la.kcap = kcap;
    la.philox = philox ? 1 : 0;
    la.dk = hp::DrawKey{key0, key1, iter, dch};
    hp::launch_pt_lowrank(la, 0);
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) {
        for (int s = 0; s < nsys; ++s)
            cudaMemcpy2D(X + 2ull * s * T * N, 16ull * N, dX + 2ull * s * Tp * Np, 16ull * Np, 16ull * N, T, cudaMemcpyDeviceToHost);
        cudaMemcpy(info, dinfo, 4ull * nsys, cudaMemcpyDeviceToHost);
    }
    cudaFree(dlam); cudaFree(dR); cudaFree(dW); cudaFree(dX); cudaFree(dP); cudaFree(dF); cudaFree(dC); cudaFree(dinfo); cudaFree(dch);
    return e == cudaSuccess ? HP_OK : HP_ERR_CUDA;
}

// k_pt_cholsolve (hp_pertime.cu) alone for nsys systems of N = n + m unknowns and T times.  In: H [nsys][T][1 + m][N] (column 0:
// chat_t in its first n entries; column 1 + j: [Q|F]^H (w_t N^-1) F[:, j]), lam [nsys][N], Rfix [nsys][T][N], wa [nsys][T][n]
// or NULL, same_prev [nsys][T] or NULL, grid (0: pt_grid), chain_ids [nsys] (read with philox only).  Out: X [nsys][T][N],
// info [nsys].  The kernel reads the padding rows N .. Np of lam, Rfix and wa (zero in the engine): they are zero here; the
// padding rows of H and the entries n .. N of column 0 are NaN, and so is the scratch the factors live in, so that a
// factor re-used without having been computed poisons the result.
int hp_test_pt_cholsolve(int n, int m, int T, int nsys, const double* H, const double* lam, const double* Rfix, const double* wa,
                         const int* same_prev, int grid, int philox, uint32_t key0, uint32_t key1, uint32_t iter,
                         const int* chain_ids, double* X, int* info) {
    if (n < 1 || m < 0 || T < 1 || nsys < 1 || grid < 0) return HP_ERR_ARG;
    const int N = n + m, nblk = (N + 31) / 32, Np = nblk * 32, Tp = 16 * ((T + 15) / 16);
    int max_smem = 0, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (hp::pt_smem_bytes(nblk, n) > (size_t)max_smem) return HP_ERR_SIZE;
    if (grid == 0) grid = hp::pt_grid(nsys, T);
    const size_t rows = (size_t)nsys * Tp, hcols = (size_t)(1 + m), scr = (size_t)grid * hp::pt_scratch_doubles_per_cta(nblk);
    double *dH, *dlam, *dR, *dW = nullptr, *dX, *dS;
    int *dsame = nullptr, *dinfo, *dch;
    if (cudaMalloc(&dH, 16 * rows * hcols * Np) || cudaMalloc(&dlam, 8ull * nsys * Np) || cudaMalloc(&dR, 16 * rows * Np) ||
        cudaMalloc(&dX, 16 * rows * Np) || cudaMalloc(&dS, 8 * scr) || cudaMalloc(&dinfo, 4ull * nsys) ||
        cudaMalloc(&dch, 4ull * nsys) || (wa && cudaMalloc(&dW, 16 * rows * Np)) || (same_prev && cudaMalloc(&dsame, 4 * rows)))
        return HP_ERR_CUDA;
    cudaMemset(dH, 0xff, 16 * rows * hcols * Np);   // 0xff..: NaN
    cudaMemset(dX, 0xff, 16 * rows * Np);
    cudaMemset(dS, 0xff, 8 * scr);
    cudaMemset(dlam, 0, 8ull * nsys * Np);
    cudaMemset(dR, 0, 16 * rows * Np);
    cudaMemset(dinfo, 0, 4ull * nsys);
    cudaMemcpy2D(dlam, 8ull * Np, lam, 8ull * N, 8ull * N, nsys, cudaMemcpyHostToDevice);
    for (int s = 0; s < nsys; ++s) {
        double* h0 = dH + 2ull * s * Tp * hcols * Np;
        cudaMemcpy2D(h0, 16ull * Np, H + 2ull * s * T * hcols * N, 16ull * N, 16ull * N, T * hcols, cudaMemcpyHostToDevice);
        for (int t = 0; t < T; ++t)   // column 0 carries chat_t in its first n entries only
            if (N > n) cudaMemset(h0 + 2ull * t * hcols * Np + 2ull * n, 0xff, 16ull * (N - n));
        cudaMemcpy2D(dR + 2ull * s * Tp * Np, 16ull * Np, Rfix + 2ull * s * T * N, 16ull * N, 16ull * N, T, cudaMemcpyHostToDevice);
    }
    if (wa) {
        cudaMemset(dW, 0, 16 * rows * Np);
        for (int s = 0; s < nsys; ++s)
            cudaMemcpy2D(dW + 2ull * s * Tp * Np, 16ull * Np, wa + 2ull * s * T * n, 16ull * n, 16ull * n, T, cudaMemcpyHostToDevice);
    }
    if (same_prev) {
        cudaMemset(dsame, 0, 4 * rows);
        cudaMemcpy2D(dsame, 4ull * Tp, same_prev, 4ull * T, 4ull * T, nsys, cudaMemcpyHostToDevice);
    }
    if (philox) cudaMemcpy(dch, chain_ids, 4ull * nsys, cudaMemcpyHostToDevice);
    else cudaMemset(dch, 0xff, 4ull * nsys);
    hp::PtArgs pa{};
    pa.H = dH; pa.lam = dlam; pa.Rfix = dR; pa.wa = dW; pa.X = dX; pa.scratch = dS; pa.same_prev = dsame; pa.info = dinfo;
    pa.nblk = nblk; pa.n = n; pa.m = m; pa.N = N; pa.T = T; pa.Tp = Tp; pa.nsys = nsys;
    pa.philox_wa = philox ? 1 : 0;
    pa.dk = hp::DrawKey{key0, key1, iter, dch};
    hp::launch_pt_cholsolve(pa, grid, 0);
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) {
        for (int s = 0; s < nsys; ++s)
            cudaMemcpy2D(X + 2ull * s * T * N, 16ull * N, dX + 2ull * s * Tp * Np, 16ull * Np, 16ull * N, T, cudaMemcpyDeviceToHost);
        cudaMemcpy(info, dinfo, 4ull * nsys, cudaMemcpyDeviceToHost);
    }
    cudaFree(dH); cudaFree(dlam); cudaFree(dR); cudaFree(dW); cudaFree(dX); cudaFree(dS); cudaFree(dsame); cudaFree(dinfo);
    cudaFree(dch);
    return e == cudaSuccess ? HP_OK : HP_ERR_CUDA;
}

// ---- measurement helpers -----------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters, double a, double b) {
    double c[8][2];
#pragma unroll
    for (int i = 0; i < 8; ++i) { c[i][0] = threadIdx.x; c[i][1] = i; }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                         : "+d"(c[i][0]), "+d"(c[i][1]) : "d"(a), "d"(b));
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
    if (s == 12345.678) out[0] = s;
}
}  // namespace

// Measured FP64 tensor-pipe peak (DMMA.8x8x4 issue loop, all SMs), TFLOP/s.  Same loop as
// profiles/microbench/fp64_peak.cu; used by bench.py as the roofline denominator.
double hp_fp64_peak_tflops(int device, double seconds) {
    if (cudaSetDevice(device) != cudaSuccess) return -1.0;
    int nsm = 0;
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device);
    double* out;
    if (cudaMalloc(&out, 8) != cudaSuccess) return -1.0;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const int iters = 20000, bps = 4;
    k_fp64_peak<<<nsm * bps, 256>>>(out, iters / 10, 1.0000001, 1e-9);
    cudaDeviceSynchronize();
    double best = 0.0, spent = 0.0;
    while (spent < seconds * 1e3) {
        cudaEventRecord(e0);
        k_fp64_peak<<<nsm * bps, 256>>>(out, iters, 1.0000001, 1e-9);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1.0; break; }
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        double tf = 2.0 * 8 * 256 / 32.0 * iters * 256.0 * nsm * bps / ms * 1e-9;
        if (tf > best) best = tf;
        spent += ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    return best;
}

void* hp_pinned_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void hp_pinned_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
