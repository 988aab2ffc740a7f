// Host build of hp_math.h for CPU unit tests (tests/test_hp_math_cpu.py).  Not linked into
// the CUDA library: it exists so that the device math can be checked against scipy without a GPU.
#include "hp_math.h"
#include <vector>

extern "C" {

double hp_host_igamc(double a, double x) { return hp::igamc(a, x); }

double hp_host_invsamp(double alpha, double beta, double lo, double hi, double u, int ngrid) {
    std::vector<double> cdf(ngrid), xg(ngrid);
    double l0 = log10(lo), l1 = log10(hi);
    for (int j = 0; j < ngrid; ++j) {
        xg[j] = hp::invsamp_grid_x(l0, l1, j, ngrid);
        cdf[j] = hp::igamc(alpha, beta / xg[j]);
    }
    return hp::invsamp_from_cdf(cdf.data(), xg.data(), ngrid, u);
}

void hp_host_cg_theta(double cre, double cim, double bnorm, double* out) {
    hp::cplx c; c.re = cre; c.im = cim;
    hp::cplx t = hp::cg_theta(c, bnorm, 1e-8, 1e-6, 100000);
    out[0] = t.re; out[1] = t.im;
}

void hp_host_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
    hp::u32x4 c; c.x = c0; c.y = c1; c.z = c2; c.w = c3;
    hp::u32x4 r = hp::philox4x32_10(c, k0, k1);
    out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}

void hp_host_normals(uint32_t k0, uint32_t k1, int n, double* out) {
    for (int i = 0; i < n / 2; ++i) {
        hp::u32x4 c; c.x = (uint32_t)i; c.y = 0; c.z = 0; c.w = 0;
        hp::normal_pair(hp::philox4x32_10(c, k0, k1), out[2 * i], out[2 * i + 1]);
    }
}

void hp_host_normals_fast(uint32_t k0, uint32_t k1, int n, double* out) {
    for (int i = 0; i < n / 2; ++i) {
        hp::u32x4 c; c.x = (uint32_t)i; c.y = 0; c.z = 0; c.w = 0;
        hp::normal_pair_fast(hp::philox4x32_10(c, k0, k1), out[2 * i], out[2 * i + 1]);
    }
}

// One pair of normals from the Philox block of any counter: normal_pair (fast = 0) or normal_pair_fast (fast = 1).  Lets the
// GPU tests reproduce a kernel's draws from its counter layout.
void hp_host_normal_pair(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, int fast, double* out) {
    hp::u32x4 c; c.x = c0; c.y = c1; c.z = c2; c.w = c3;
    if (fast) hp::normal_pair_fast(hp::philox4x32_10(c, k0, k1), out[0], out[1]);
    else hp::normal_pair(hp::philox4x32_10(c, k0, k1), out[0], out[1]);
}

void hp_host_gammas(double alpha, uint32_t k0, uint32_t k1, int n, double* out) {
    for (int i = 0; i < n; ++i) out[i] = hp::gamma_mt(alpha, (uint32_t)i, 0, 7, k0, k1);
}

}  // extern "C"
