// Derivatives of the isotropic cores with respect to the scaled squared distance u, for the derivative-block kernels
// (gram_deriv.cu): c(u), c'(u), c''(u), c'''(u) and, for Cauchy, d/dbeta of c, c', c''.
//
//   ExpQuad           c(u) = exp(-u/2)                                   c^(j) = (-1/2)^j c
//   Cauchy, alpha = 2 c(u) = B^(-beta/2), B = 1 + u/beta                c^(j) = c^(j-1) * -(beta/2 + j - 1) / (beta B)
//   Maternp(p)        c(u) = kvmodx2_hi(z, p), z = (2p+1) u + par0       d/dz kvmodx2_hi(z, q) = -kvmodx2_hi(z, q-1) / (4q-2)
//                     (src/lsqfitgp/_special/_bessel.py:101-122); below q = 0: d/dz e^-x = -e^-x / (2x),
//                     d2/dz2 e^-x = e^-x (x + 1) / (4 x^3), x = sqrt(z).
//   Constant          c = 1.
//
// The derivatives that go below q = 0 diverge at x = 0 (c'' for p = 1, c''' for p = 1, 2).  They are returned as they
// are (possibly +-inf); the kernels only use them multiplied by products of coordinate differences that vanish at
// least as fast, through mul0(), which maps a zero product to 0 instead of 0 * inf.
//
// Plain C++ on the host, so that tests/test_deriv_cpu.py checks these numerics without a GPU.
#pragma once
#include <math.h>

#include "../../include/lgp_b200.h"

#ifdef __CUDACC__
#define LGP_DC_HD __host__ __device__ __forceinline__
#else
#define LGP_DC_HD static inline
#endif

namespace lgp {

// c * t with 0 when t == 0 (c may be infinite where t vanishes: the r = 0 singularities above)
LGP_DC_HD double mul0(double c, double t) { return t == 0.0 ? 0.0 : c * t; }

// kvmodx2_hi(z, q) = e^-x P_q(x) with the Horner ratios (q-k)/((2q-k)(k+1)) of _bessel.py:101-110
LGP_DC_HD double kvmodx2_hi_ex(double ex, double x, int q) {
    double poly = 1.0;
    for (int k = q - 1; k >= 0; k--) poly = 1.0 + poly * ((double)(q - k) / (double)((2 * q - k) * (k + 1))) * 2.0 * x;
    return ex * poly;
}

// c[0..3] = c, c', c'', c''' at u; db[0..2] = d/dbeta of c, c', c'' (Cauchy; 0 for the other kinds).
// kind: LGP_K_EXPQUAD, LGP_K_MATERNP (p >= 1), LGP_K_CAUCHY (alpha = par0 = 2, beta = par1), LGP_K_CONSTANT.
LGP_DC_HD void deriv_coefs(int kind, int p, double par0, double beta, double u, double c[4], double db[3]) {
    db[0] = db[1] = db[2] = 0.0;
    switch (kind) {
        case LGP_K_EXPQUAD: {
            c[0] = exp(-0.5 * u);
#pragma unroll
            for (int j = 1; j < 4; j++) c[j] = -0.5 * c[j - 1];
            return;
        }
        case LGP_K_CAUCHY: {
            const double B = 1.0 + u / beta;
            const double lb = log(B);
            c[0] = pow(B, -beta / 2.0);
            double hsum = 0.0;  // sum_{i<j} 1/(beta + 2i)
#pragma unroll
            for (int j = 0; j < 4; j++) {
                if (j > 0) c[j] = c[j - 1] * (-(0.5 * beta + (double)(j - 1))) / (beta * B);
                if (j < 3) db[j] = c[j] * (hsum - (double)j / beta - 0.5 * lb + (0.5 * beta + (double)j) * u / (beta * beta * B));
                hsum += 1.0 / (beta + 2.0 * (double)j);
            }
            return;
        }
        case LGP_K_MATERNP: {
            const double nu2 = (double)(2 * p + 1);
            const double z = nu2 * u + par0;
            const double x = sqrt(z);
            const double ex = exp(-x);
            double w = 1.0;  // nu2^j (-1)^j / prod_{i<j} (4(p-i) - 2), for j <= p
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int q = p - j;
                if (q >= 0) {
                    c[j] = w * kvmodx2_hi_ex(ex, x, q);
                    if (q > 0) w *= -nu2 / (double)(4 * q - 2);
                } else if (q == -1) {
                    c[j] = w * nu2 * (-ex / (2.0 * x));
                } else if (q == -2) {
                    c[j] = w * (nu2 * nu2) * (ex * (x + 1.0) / (4.0 * x * x * x));
                } else {
                    c[j] = NAN;  // not needed: kernels ask for at most c''' and reject p = 0
                }
            }
            return;
        }
        default:
            c[0] = 1.0;
            c[1] = c[2] = c[3] = 0.0;
            return;
    }
}

}  // namespace lgp
