// Derivatives of the Gram build with respect to the input points: the reverse-mode contraction (xvjp) and the
// forward-mode derivative (xjvp) that gradients of the marginal likelihood with respect to the points need.  The
// reference gets them from jax differentiating through `gpfactory` when the points depend on the hyperparameters
// (src/lsqfitgp/_fit.py:687-702: jax.vjp of the whole Gram build, points included).
//
// For a factor f with scaled coordinates u = (x - loc_x)/scale_x, v = (y - loc_y)/scale_y and a field d in its dimmask,
//   dK_f/dx_{d,i} =  amp_f c_f'(r2_f) 2 (u_{d,i} - v_{d,j}) / scale_x_f,
//   dK_f/dy_{d,j} = -amp_f c_f'(r2_f) 2 (u_{d,i} - v_{d,j}) / scale_y_f,
// with the product rule across the factors of a term (Q_f = product of the other factors, no division by factor
// values).  c' is the d/dr2 of core_derivs (gram_desc.cuh), the coefficient the hyperparameter VJP uses for
// d/d log(scale).  White and Constant contribute 0.
//
// r = 0: the product c' (u - v) goes through mul0 (deriv_core.cuh), which gives 0 where the difference is 0.  Where
// r2_f = 0 every difference of the factor is 0, so a c' that diverges there (Maternp p = 0 without offset, Matern of
// order <= 1/2, Cauchy alpha < 2) never produces NaN; on the diagonal K(x_i, x_i) is constant, so 0 is exact there.
// Same staging and 64 x 64 tiles as gram_iso_vjp_kernel / gram_iso_jvp_kernel (gram_iso.cu).
#include <math.h>
#include <string.h>

#include "../../include/lgp_b200.h"
#include "common.cuh"
#include "internal.h"
#include "gram_desc.cuh"
#include "deriv_core.cuh"

namespace lgp {

// gx[d][i] = sum_j G_ij dK_ij/dx_{d,i}, gy[d][j] = sum_i G_ij dK_ij/dy_{d,j}; symlower as in gram_iso_vjp_kernel, with
// both sides of every lower entry added to gx (gy == gx there).  Per slot s (factor f, field d) and entry, the term
// t = mul0(g Q_f amp_f c_f' 2, u_s - v_s) is summed over the 16 columns of a half-warp by shuffles into the row
// accumulator racc[s][row] (one writer per row), and over the two rows of a warp into the column accumulator
// cacc[s][col] (shared atomicAdd from the 8 warps).  Each tile then adds its accumulators to the outputs with atomicAdd.
__global__ void __launch_bounds__(G_THREADS) gram_iso_xvjp_kernel(const __grid_constant__ GramDesc d,
                                                                  const double *__restrict__ x, int64_t ldx, int64_t n,
                                                                  const double *__restrict__ y, int64_t ldy, int64_t m,
                                                                  const double *__restrict__ G, int64_t ldg,
                                                                  const double *__restrict__ bvec, int symlower,
                                                                  int tiles_n, double *gx, int64_t ldgx, double *gy,
                                                                  int64_t ldgy) {
    extern __shared__ __align__(16) double gsm[];
    double *su = gsm;
    double *sv = gsm + (size_t)d.nslots * GT;
    double *racc = sv + (size_t)d.nslots * GT;
    double *cacc = racc + (size_t)d.nslots * GT;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    int tm, tn;
    if (symlower) {
        int b = blockIdx.x;
        tm = (int)((sqrt(8.0 * b + 1.0) - 1.0) * 0.5);
        while ((tm + 1) * (tm + 2) / 2 <= b) tm++;
        while (tm * (tm + 1) / 2 > b) tm--;
        tn = b - tm * (tm + 1) / 2;
    } else {
        tm = blockIdx.x / tiles_n;
        tn = blockIdx.x % tiles_n;
    }
    const int64_t i0 = (int64_t)tm * GT, j0 = (int64_t)tn * GT;
    stage_points(d, su, x, ldx, n, i0, false, tid);
    stage_points(d, sv, y, ldy, m, j0, true, tid);
    for (int k = tid; k < 2 * d.nslots * GT; k += G_THREADS) racc[k] = 0.0;
    __syncthreads();

    const bool want_col = symlower || gy != nullptr;
#pragma unroll 1
    for (int a = 0; a < 4; a++) {
        const int r = ty + 16 * a;
        const int64_t i = i0 + r;
        const double bi = (bvec && i < n) ? bvec[i] : 0.0;
#pragma unroll 1
        for (int c = 0; c < 4; c++) {
            // every lane takes part in the shuffles below: entries outside the block (or above the diagonal) get g = 0
            const int cc = 2 * tx + 32 * (c >> 1) + (c & 1);
            const int64_t j = j0 + cc;
            double g = 0.0;
            if (i < n && j < m && !(symlower && j > i)) {
                g = G[i * ldg + j];
                if (bvec) g -= bi * bvec[j];
                if (symlower && j != i) g *= 2.0;
            }
            double val[LGP_MAX_FACTORS], dr2[LGP_MAX_FACTORS];
#pragma unroll
            for (int f = 0; f < LGP_MAX_FACTORS; f++) {
                if (f < d.nfactors) {
                    double r2 = 0.0;
                    for (int s = d.slot0[f]; s < d.slot0[f] + d.nslot[f]; s++) {
                        const double df = su[s * GT + r] - sv[s * GT + cc];
                        r2 += df * df;
                    }
                    double dp1;
                    core_derivs(d, f, r2, val[f], dr2[f], dp1);
                }
            }
#pragma unroll
            for (int f = 0; f < LGP_MAX_FACTORS; f++) {
                if (f < d.nfactors) {
                    double others = 1.0;
#pragma unroll
                    for (int h = 0; h < LGP_MAX_FACTORS; h++)
                        if (h < d.nfactors && h != f && d.term[h] == d.term[f]) others *= d.amp[h] * val[h];
                    // g == 0 (padding, upper triangle) must not meet a c' that diverges at a padded r2 = 0
                    const double coef = g == 0.0 ? 0.0 : 2.0 * g * others * d.amp[f] * dr2[f];
                    for (int s = d.slot0[f]; s < d.slot0[f] + d.nslot[f]; s++) {
                        const double t = mul0(coef, su[s * GT + r] - sv[s * GT + cc]);
                        double rs = t;
#pragma unroll
                        for (int o = 1; o < 16; o <<= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);
                        if (tx == 0) racc[s * GT + r] += rs;
                        if (want_col) {
                            const double cs = t + __shfl_xor_sync(0xffffffffu, t, 16);
                            if ((tid & 16) == 0) atomicAdd(&cacc[s * GT + cc], cs);
                        }
                    }
                }
            }
        }
    }
    __syncthreads();
    double *gcol = symlower ? gx : gy;
    const int64_t ldcol = symlower ? ldgx : ldgy;
    for (int k = tid; k < d.nslots * GT; k += G_THREADS) {
        const int s = k / GT, rr = k % GT;
        const int f = d.slot_factor[s], dim = d.slot_dim[s];
        if (gx && i0 + rr < n) atomicAdd(gx + dim * ldgx + i0 + rr, racc[k] / d.scale_x[f]);
        if (want_col && j0 + rr < m) atomicAdd(gcol + dim * ldcol + j0 + rr, -cacc[k] / d.scale_y[f]);
    }
}

// D_ij (+)= sum_d tx[d][i] dK_ij/dx_{d,i} + ty[d][j] dK_ij/dy_{d,j}: one pass over the tile, the tangents staged per slot
// already divided by the factor's scale, the product rule inside each term as in gram_iso_jvp_kernel.
__global__ void __launch_bounds__(G_THREADS) gram_iso_xjvp_kernel(const __grid_constant__ GramDesc d,
                                                                  const double *__restrict__ x, int64_t ldx, int64_t n,
                                                                  const double *__restrict__ y, int64_t ldy, int64_t m,
                                                                  const double *__restrict__ tanx, int64_t ldtx,
                                                                  const double *__restrict__ tany, int64_t ldty,
                                                                  double *__restrict__ D, int64_t ldd, int accumulate) {
    extern __shared__ __align__(16) double gsm[];
    double *su = gsm;
    double *sv = gsm + (size_t)d.nslots * GT;
    double *stx = sv + (size_t)d.nslots * GT;
    double *sty = stx + (size_t)d.nslots * GT;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t i0 = (int64_t)blockIdx.y * GT, j0 = (int64_t)blockIdx.x * GT;
    stage_points(d, su, x, ldx, n, i0, false, tid);
    stage_points(d, sv, y, ldy, m, j0, true, tid);
    for (int idx = tid; idx < d.nslots * GT; idx += G_THREADS) {
        const int s = idx / GT, rr = idx % GT;
        const int f = d.slot_factor[s], dim = d.slot_dim[s];
        stx[idx] = (tanx && i0 + rr < n) ? tanx[dim * ldtx + i0 + rr] / d.scale_x[f] : 0.0;
        sty[idx] = (tany && j0 + rr < m) ? tany[dim * ldty + j0 + rr] / d.scale_y[f] : 0.0;
    }
    __syncthreads();
#pragma unroll 1
    for (int a = 0; a < 4; a++) {
        const int r = ty + 16 * a;
        const int64_t i = i0 + r;
        if (i >= n) continue;
#pragma unroll 1
        for (int c = 0; c < 4; c++) {
            const int cc = 2 * tx + 32 * (c >> 1) + (c & 1);
            const int64_t j = j0 + cc;
            if (j >= m) continue;
            double total = 0.0;
            int f = 0;
            while (f < d.nfactors) {
                const int term = d.term[f];
                double prod = 1.0, dsum = 0.0;
                for (; f < d.nfactors && d.term[f] == term; f++) {
                    double r2 = 0.0, w = 0.0;   // w = sum_s 2 (u_s - v_s) (tx_s / scale_x - ty_s / scale_y)
                    for (int s = d.slot0[f]; s < d.slot0[f] + d.nslot[f]; s++) {
                        const double df = su[s * GT + r] - sv[s * GT + cc];
                        r2 += df * df;
                        w += 2.0 * df * (stx[s * GT + r] - sty[s * GT + cc]);
                    }
                    double val, dr2, dp1;
                    core_derivs(d, f, r2, val, dr2, dp1);
                    const double v = d.amp[f] * val;
                    const double dv = d.amp[f] * mul0(dr2, w);
                    dsum = dsum * v + prod * dv;
                    prod *= v;
                }
                total += dsum;
            }
            D[i * ldd + j] = accumulate ? D[i * ldd + j] + total : total;
        }
    }
}

}  // namespace lgp

using namespace lgp;

extern "C" {

int lgp_gram_iso_xvjp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                      int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *G, int64_t ldg,
                      const double *b, int symlower, double *gx, int64_t ldgx, double *gy, int64_t ldgy) {
    if (!factors || !G || !x || !y || n < 1 || m < 1 || ndim < 1 || ldx < n || ldy < m || ldg < m) return LGP_ERR_BADARG;
    if (symlower && (n != m || gy || !gx)) return LGP_ERR_BADARG;
    if (!symlower && !gx && !gy) return LGP_ERR_BADARG;
    if ((gx && ldgx < n) || (gy && ldgy < m)) return LGP_ERR_BADARG;
    GramDesc d;
    int rc = build_desc(factors, nfactors, ndim, d);
    if (rc) return rc;
    const int64_t tm = (n + GT - 1) / GT, tn = (m + GT - 1) / GT;
    const int64_t nblk = symlower ? tm * (tm + 1) / 2 : tm * tn;
    if (nblk > 2147483647LL) return LGP_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (gx && cudaMemset2DAsync(gx, sizeof(double) * ldgx, 0, sizeof(double) * n, ndim, st) != cudaSuccess)
        return LGP_ERR_CUDA;
    if (gy && cudaMemset2DAsync(gy, sizeof(double) * ldgy, 0, sizeof(double) * m, ndim, st) != cudaSuccess)
        return LGP_ERR_CUDA;
    if (d.nslots == 0) return LGP_OK;   // only Constant factors: no dependence on the points
    const size_t smem = (size_t)4 * d.nslots * GT * sizeof(double);
    if (smem_opt_in(gram_iso_xvjp_kernel, smem)) return LGP_ERR_CUDA;
    gram_iso_xvjp_kernel<<<(unsigned)nblk, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, G, ldg, b, symlower, (int)tn,
                                                                  gx, ldgx, gy, ldgy);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

int lgp_gram_iso_xjvp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                      int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *tx, int64_t ldtx,
                      const double *ty, int64_t ldty, double *D_out, int64_t ldd, int accumulate) {
    if (!factors || !D_out || !x || !y || n < 1 || m < 1 || ndim < 1 || ldx < n || ldy < m || ldd < m)
        return LGP_ERR_BADARG;
    if ((tx && ldtx < n) || (ty && ldty < m)) return LGP_ERR_BADARG;
    GramDesc d;
    int rc = build_desc(factors, nfactors, ndim, d);
    if (rc) return rc;
    dim3 grid((unsigned)((m + GT - 1) / GT), (unsigned)((n + GT - 1) / GT));
    if (grid.y > 65535) return LGP_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (d.nslots == 0 || (!tx && !ty)) {   // no dependence on the points, or a zero tangent
        if (accumulate) return LGP_OK;
        if (cudaMemset2DAsync(D_out, sizeof(double) * ldd, 0, sizeof(double) * m, n, st) != cudaSuccess)
            return LGP_ERR_CUDA;
        return LGP_OK;
    }
    const size_t smem = (size_t)4 * d.nslots * GT * sizeof(double);
    if (smem_opt_in(gram_iso_xjvp_kernel, smem)) return LGP_ERR_CUDA;
    gram_iso_xjvp_kernel<<<grid, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, tx, ldtx, ty, ldty, D_out, ldd,
                                                        accumulate);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

}  // extern "C"
