/* TEST INFRASTRUCTURE: host build of lsqfitgp_b200/csrc/deriv_core.cuh (the per-factor derivative coefficients of the
 * derivative-block kernels) so that tests/test_deriv_cpu.py compares it with oracle/deriv.py without a GPU.
 * The test compiles it as C++ into a temporary directory (g++ -x c++, -ffp-contract=off). */
#include "../lsqfitgp_b200/csrc/deriv_core.cuh"

extern "C" {

/* c: n x 4 (c, c', c'', c'''), db: n x 3 (d/dbeta of c, c', c'') */
void lgp_host_deriv_coefs(int kind, int p, double par0, double beta, const double *u, long n, double *c, double *db) {
    for (long i = 0; i < n; i++) lgp::deriv_coefs(kind, p, par0, beta, u[i], c + 4 * i, db + 3 * i);
}

/* mul0 as the kernels use it */
void lgp_host_mul0(const double *c, const double *t, long n, double *out) {
    for (long i = 0; i < n; i++) out[i] = lgp::mul0(c[i], t[i]);
}
}
