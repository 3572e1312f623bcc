/* TEST INFRASTRUCTURE: host build of lsqfitgp_b200/csrc/hess_core.cuh (the per-factor second-derivative coefficients of
 * the second-order Gram contraction) so that tests/test_hess_cpu.py compares it with oracle/hess.py without a GPU.
 * The test compiles it as C++ into a temporary directory (g++ -x c++, -ffp-contract=off). */
#include "../lsqfitgp_b200/csrc/hess_core.cuh"

extern "C" {

/* h: n x 6 (c, dc/dlog scale, d2c/dlog scale2, dc/dbeta, d2c/dlog scale dbeta, d2c/dbeta2); par0 = nu for Matern.
 * Returns 0, or -1 if the Matern order is not supported. */
int lgp_host_hess_coefs(int kind, int p, double par0, double par1, const double *u, long n, double *h) {
    double mat[lgp::MATERN_NPAR] = {0};
    if (kind == LGP_K_MATERN && !lgp::matern_nu_setup(par0, mat)) return -1;
    for (long i = 0; i < n; i++) lgp::hess_coefs(kind, p, par0, par1, mat, u[i], h + 6 * i);
    return 0;
}
}
