// Descriptor of the general (sum-of-products) Gram kernels, the per-factor core arithmetic and the staging of point
// tiles: shared by the Gram kernels of gram_iso.cu and the derivative-block kernels of gram_deriv.cu.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../include/lgp_b200.h"
#include "bessel_k.cuh"

namespace lgp {

constexpr int GT = 64;          // CTA tile (rows = cols)
constexpr int G_THREADS = 256;  // 16 x 16 threads, 4 x 4 entries each
constexpr int G_MAX_SLOTS = 96; // sum over factors of participating fields
constexpr int G_MAX_P = 8;

struct GramDesc {
    int nfactors;
    int nslots;
    int kind[LGP_MAX_FACTORS];
    int term[LGP_MAX_FACTORS];
    int ipar[LGP_MAX_FACTORS];
    int slot0[LGP_MAX_FACTORS];   // first slot of the factor
    int nslot[LGP_MAX_FACTORS];   // number of participating fields
    double scale_x[LGP_MAX_FACTORS], scale_y[LGP_MAX_FACTORS], loc_x[LGP_MAX_FACTORS], loc_y[LGP_MAX_FACTORS];
    double par0[LGP_MAX_FACTORS], par1[LGP_MAX_FACTORS], amp[LGP_MAX_FACTORS];
    double coef[LGP_MAX_FACTORS][G_MAX_P];  // Maternp Horner ratios c_{k+1}/c_k, k = 0..p-1
    double mat[LGP_MAX_FACTORS][MATERN_NPAR];  // Matern of real order: host-computed constants (bessel_k.cuh)
    unsigned char slot_dim[G_MAX_SLOTS];
    unsigned char slot_factor[G_MAX_SLOTS];
};

static int build_desc(const lgp_factor_t *f, int nf, int ndim, GramDesc &d) {
    if (nf < 1 || nf > LGP_MAX_FACTORS || ndim < 0 || ndim > LGP_MAX_DIMS) return LGP_ERR_BADARG;
    memset(&d, 0, sizeof(d));
    d.nfactors = nf;
    int slots = 0;
    for (int i = 0; i < nf; i++) {
        if (i > 0 && f[i].term < f[i - 1].term) return LGP_ERR_BADARG;  // factors must be grouped by term
        d.kind[i] = f[i].kind;
        d.term[i] = f[i].term;
        d.ipar[i] = f[i].ipar;
        d.scale_x[i] = f[i].scale_x; d.scale_y[i] = f[i].scale_y;
        d.loc_x[i] = f[i].loc_x; d.loc_y[i] = f[i].loc_y;
        d.par0[i] = f[i].par0; d.par1[i] = f[i].par1; d.amp[i] = f[i].amp;
        d.slot0[i] = slots;
        if (f[i].kind < 0 || f[i].kind > LGP_K_MATERN) return LGP_ERR_UNSUPPORTED;
        if (f[i].kind == LGP_K_MATERN && !matern_nu_setup(f[i].par0, d.mat[i])) return LGP_ERR_UNSUPPORTED;
        if (f[i].kind == LGP_K_MATERNP) {
            int p = f[i].ipar;
            if (p < 0 || p > G_MAX_P) return LGP_ERR_UNSUPPORTED;
            for (int k = 0; k < p; k++) d.coef[i][k] = (double)(p - k) / (double)((2 * p - k) * (k + 1));
        }
        if (f[i].kind != LGP_K_CONSTANT) {
            for (int dd = 0; dd < ndim; dd++)
                if (f[i].dimmask & (1u << dd)) {
                    if (slots >= G_MAX_SLOTS) return LGP_ERR_UNSUPPORTED;
                    d.slot_dim[slots] = (unsigned char)dd;
                    d.slot_factor[slots] = (unsigned char)i;
                    slots++;
                }
        }
        d.nslot[i] = slots - d.slot0[i];
    }
    d.nslots = slots;
    return LGP_OK;
}

// value of factor f (without amp) at squared distance r2
__device__ __forceinline__ double core_value(const GramDesc &d, int f, double r2) {
    switch (d.kind[f]) {
        case LGP_K_EXPQUAD:
            return exp(__dmul_rn(-0.5, r2));
        case LGP_K_MATERNP: {
            const int p = d.ipar[f];
            double z = __dadd_rn(__dmul_rn((double)(2 * p + 1), r2), d.par0[f]);
            double x = sqrt(z);
            double poly = 1.0;
            for (int k = p - 1; k >= 0; k--)
                poly = __dadd_rn(1.0, __dmul_rn(__dmul_rn(__dmul_rn(poly, d.coef[f][k]), 2.0), x));
            return __dmul_rn(exp(-x), poly);
        }
        case LGP_K_CAUCHY: {
            const double alpha = d.par0[f], beta = d.par1[f];
            double pw = (alpha == 2.0) ? r2 : pow(r2, alpha / 2.0);
            return pow(__dadd_rn(1.0, pw / beta), -beta / alpha);
        }
        case LGP_K_WHITE:
            return r2 == 0.0 ? 1.0 : 0.0;
        case LGP_K_MATERN: {
            double val, dr2;
            matern_nu_core(d.mat[f], r2, false, val, dr2);
            return val;
        }
        default:
            return 1.0;
    }
}

// d core / d r2 and d core / d par1 (Cauchy beta)
__device__ __forceinline__ void core_derivs(const GramDesc &d, int f, double r2, double &val, double &dr2,
                                            double &dpar1) {
    dpar1 = 0.0;
    switch (d.kind[f]) {
        case LGP_K_EXPQUAD:
            val = exp(-0.5 * r2);
            dr2 = -0.5 * val;
            return;
        case LGP_K_MATERNP: {
            const int p = d.ipar[f];
            const double nu2 = (double)(2 * p + 1);
            double z = nu2 * r2 + d.par0[f];
            double x = sqrt(z);
            double ex = exp(-x);
            double poly = 1.0;
            for (int k = p - 1; k >= 0; k--) poly = 1.0 + poly * d.coef[f][k] * 2.0 * x;
            val = ex * poly;
            if (p == 0) {
                dr2 = x > 0.0 ? -nu2 * ex / (2.0 * x) : 0.0;
            } else {
                // d/dz kvmodx2_hi(z, p) = -kvmodx2_hi(z, p-1) / (4 (p - 1/2))   (_bessel.py:112-122)
                const int pm = p - 1;
                double polym = 1.0;
                for (int k = pm - 1; k >= 0; k--)
                    polym = 1.0 + polym * ((double)(pm - k) / (double)((2 * pm - k) * (k + 1))) * 2.0 * x;
                dr2 = -nu2 * ex * polym / (4.0 * ((double)p - 0.5));
            }
            return;
        }
        case LGP_K_CAUCHY: {
            const double alpha = d.par0[f], beta = d.par1[f];
            double t = (alpha == 2.0) ? r2 : pow(r2, alpha / 2.0);
            double base = 1.0 + t / beta;
            val = pow(base, -beta / alpha);
            // d val / d t = -(1/alpha) base^(-beta/alpha - 1)
            double dvdt = -(1.0 / alpha) * val / base;
            double dtdr2 = (alpha == 2.0) ? 1.0 : (r2 > 0.0 ? (alpha / 2.0) * t / r2 : 0.0);
            dr2 = dvdt * dtdr2;
            dpar1 = val * (-(1.0 / alpha) * log(base) + (t / (alpha * beta)) / base);
            return;
        }
        case LGP_K_WHITE:
            val = r2 == 0.0 ? 1.0 : 0.0;
            dr2 = 0.0;
            return;
        case LGP_K_MATERN:
            matern_nu_core(d.mat[f], r2, true, val, dr2);
            return;
        default:
            val = 1.0;
            dr2 = 0.0;
            return;
    }
}

// tangent of the forward-mode kernels: 3 doubles per factor (d amp, d log scale, d par1)
struct GramTangent {
    double t[3 * LGP_MAX_FACTORS];
};

// stage transformed coordinates of a 64-point tile: su[slot][64]
__device__ __forceinline__ void stage_points(const GramDesc &d, double *s, const double *__restrict__ x, int64_t ldx,
                                             int64_t n, int64_t i0, bool is_y, int tid) {
    for (int idx = tid; idx < d.nslots * GT; idx += G_THREADS) {
        int slot = idx / GT, r = idx % GT;
        int f = d.slot_factor[slot];
        int64_t i = i0 + r;
        double v = 0.0;
        if (i < n) {
            double raw = x[(int64_t)d.slot_dim[slot] * ldx + i];
            double loc = is_y ? d.loc_y[f] : d.loc_x[f];
            double sc = is_y ? d.scale_y[f] : d.scale_x[f];
            v = __ddiv_rn(__dsub_rn(raw, loc), sc);
        }
        s[slot * GT + r] = v;
    }
}

}  // namespace lgp
