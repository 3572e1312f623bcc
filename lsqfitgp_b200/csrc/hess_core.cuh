// Second hyperparameter derivatives of the isotropic cores, for the second-order Gram contraction (gram_hvp.cu).
//
// With u the scaled squared distance, lambda = log(scale) (du/dlambda = -2u) and beta = par1 (Cauchy):
//   h[0] = c                   h[1] = dc/dlambda = -2u c'          h[2] = d2c/dlambda2 = 4u c' + 4u^2 c''
//   h[3] = dc/dbeta            h[4] = d2c/dlambda dbeta            h[5] = d2c/dbeta2          (0 except Cauchy)
//
//   ExpQuad            c' = -c/2, c'' = c/4.
//   Maternp(p)         c, c', c'' of deriv_coefs; the products with u go through mul0 (c', c'' diverge at u = 0 for
//                      small p, u c' and u^2 c'' vanish there).
//   Matern(nu)         from the modified Bessel equation u^2 c'' = (nu u / 2) c + (nu - 1) u c', so that
//                      h[2] = 2 nu u (c + 2 c'): no K_{nu-2}, no downward recurrence; c and c' from matern_nu_core.
//   Cauchy(alpha)      with s = u^(alpha/2), B = 1 + s/beta, c = B^(-beta/alpha), the derivatives of log c:
//                        d_lambda = s/B, d_lambda^2 = -alpha s/B^2, d_beta = -log(B)/alpha + s/(alpha beta B),
//                        d_lambda d_beta = s^2/(beta^2 B^2), d_beta^2 = s^2/(alpha beta^3 B^2),
//                      and h = c times (second log-derivative + product of the first ones).
//   White, Constant    c only (they depend on the amplitude alone).
//
// Plain C++ on the host, so that tests/test_hess_cpu.py checks these numerics without a GPU.
#pragma once
#include <math.h>

#include "../../include/lgp_b200.h"
#include "bessel_k.cuh"
#include "deriv_core.cuh"

namespace lgp {

// `mat`: the Matern parameter block of matern_nu_setup (read for LGP_K_MATERN only).
LGP_DC_HD void hess_coefs(int kind, int p, double par0, double par1, const double *mat, double u, double h[6]) {
    h[3] = h[4] = h[5] = 0.0;
    switch (kind) {
        case LGP_K_EXPQUAD: {
            const double c = exp(-0.5 * u);
            h[0] = c;
            h[1] = u * c;
            h[2] = u * (u - 2.0) * c;
            return;
        }
        case LGP_K_MATERNP: {
            double c[4], db[3];
            deriv_coefs(kind, p, par0, 0.0, u, c, db);
            h[0] = c[0];
            h[1] = mul0(c[1], -2.0 * u);
            h[2] = mul0(c[1], 4.0 * u) + mul0(c[2], 4.0 * u * u);
            return;
        }
        case LGP_K_MATERN: {
            double c, c1;
            matern_nu_core(mat, u, true, c, c1);
            h[0] = c;
            h[1] = -2.0 * u * c1;
            h[2] = 2.0 * mat[MN_NU] * u * (c + 2.0 * c1);
            return;
        }
        case LGP_K_CAUCHY: {
            const double alpha = par0, beta = par1;
            const double s = (alpha == 2.0) ? u : pow(u, alpha / 2.0);
            const double B = 1.0 + s / beta;
            const double c = pow(B, -beta / alpha);
            const double sB = s / B;
            const double l1 = sB, l11 = -alpha * sB / B;
            const double lb = (sB / beta - log1p(s / beta)) / alpha;
            const double l1b = (sB / beta) * (sB / beta), lbb = l1b / (alpha * beta);
            h[0] = c;
            h[1] = c * l1;
            h[2] = c * (l11 + l1 * l1);
            h[3] = c * lb;
            h[4] = c * (l1b + l1 * lb);
            h[5] = c * (lbb + lb * lb);
            return;
        }
        case LGP_K_WHITE:
            h[0] = u == 0.0 ? 1.0 : 0.0;
            h[1] = h[2] = 0.0;
            return;
        default:
            h[0] = 1.0;
            h[1] = h[2] = 0.0;
            return;
    }
}

}  // namespace lgp
