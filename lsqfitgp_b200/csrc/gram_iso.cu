// Gram-matrix build for sums of products of isotropic kernels, and its reverse-mode contraction.
//
// Reference arithmetic (one rounding per operation, field order, divide-before-difference):
//   src/lsqfitgp/_Kernel/_ops.py:292-326 (loc, scale applied per argument),
//   src/lsqfitgp/_Kernel/_isotropic.py:61-81 + _Kernel/_util.py:74-99 (r2 = sum_f (x_f-y_f)^2),
//   src/lsqfitgp/_kernels/_basic.py:46,59,75,339-343, _kernels/_matern.py:48-49,74-76,
//   src/lsqfitgp/_special/_bessel.py:101-122 (kvmodx2_hi and its derivative),
//   src/lsqfitgp/_Kernel/_alg.py:48-82 (sum / product / scalar multiple).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/lgp_b200.h"
#include "common.cuh"
#include "fastmath.cuh"
#include "bessel_k.cuh"
#include "internal.h"
#include "gram_desc.cuh"

namespace lgp {

// Device-resident hyperparameters (the XLA-FFI path: traced scalars live in device buffers, INTEGRATION.md section 3).
// `devpar` holds LGP_DEVPAR_STRIDE doubles per factor: scale_x, scale_y, loc_x, loc_y, par1, amp; the structural fields
// (kind, term, dimmask, ipar, par0) stay host-side attributes.  The DEV instantiations of the general kernels copy the
// descriptor into shared memory and overwrite the numeric fields from `devpar` before anything else.
template <bool DEV>
struct DevDescStore {
    char unused;
};
template <>
struct DevDescStore<true> {
    GramDesc d;
};
__device__ __forceinline__ void load_dev_desc(const GramDesc &d, const double *__restrict__ devpar, GramDesc &sd, int tid) {
    const int *src = reinterpret_cast<const int *>(&d);
    int *dst = reinterpret_cast<int *>(&sd);
    for (int i = tid; i < (int)(sizeof(GramDesc) / sizeof(int)); i += G_THREADS) dst[i] = src[i];
    __syncthreads();
    if (tid < d.nfactors) {
        const double *q = devpar + LGP_DEVPAR_STRIDE * tid;
        sd.scale_x[tid] = q[0];
        sd.scale_y[tid] = q[1];
        sd.loc_x[tid] = q[2];
        sd.loc_y[tid] = q[3];
        sd.par1[tid] = q[4];
        sd.amp[tid] = q[5];
    }
    __syncthreads();
}
template <bool DEV>
__global__ void __launch_bounds__(G_THREADS) gram_iso_kernel(const __grid_constant__ GramDesc d,
                                                             const double *__restrict__ x, int64_t ldx, int64_t n,
                                                             const double *__restrict__ y, int64_t ldy, int64_t m,
                                                             double *__restrict__ K, int64_t ldk, int vec_ok, const double *__restrict__ devpar) {
    __shared__ DevDescStore<DEV> sdesc;
    if constexpr (DEV) load_dev_desc(d, devpar, sdesc.d, threadIdx.x);
    const GramDesc &dd = [&]() -> const GramDesc & {
        if constexpr (DEV)
            return sdesc.d;
        else
            return d;
    }();
    extern __shared__ __align__(16) double gsm[];
    double *su = gsm;
    double *sv = gsm + (size_t)dd.nslots * GT;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t i0 = (int64_t)blockIdx.y * GT, j0 = (int64_t)blockIdx.x * GT;
    stage_points(dd, su, x, ldx, n, i0, false, tid);
    stage_points(dd, sv, y, ldy, m, j0, true, tid);
    __syncthreads();

    double sum[4][4];
    double prod[4][4];
    int cur_term = -1;
    bool first_term = true;
    for (int f = 0; f < dd.nfactors; f++) {
        double r2[4][4];
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) r2[a][c] = 0.0;
        for (int s = dd.slot0[f]; s < dd.slot0[f] + dd.nslot[f]; s++) {
            double uu[4], vv[4];
#pragma unroll
            for (int a = 0; a < 4; a++) uu[a] = su[s * GT + ty + 16 * a];
#pragma unroll
            for (int b = 0; b < 2; b++) {
                double2 t = *reinterpret_cast<const double2 *>(&sv[s * GT + 2 * tx + 32 * b]);
                vv[2 * b] = t.x;
                vv[2 * b + 1] = t.y;
            }
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    double df = __dsub_rn(uu[a], vv[c]);
                    double sq = __dmul_rn(df, df);
                    r2[a][c] = (s == dd.slot0[f]) ? sq : __dadd_rn(r2[a][c], sq);
                }
        }
        const bool new_term = dd.term[f] != cur_term;
        if (new_term && cur_term != -1) {
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) sum[a][c] = first_term ? prod[a][c] : __dadd_rn(sum[a][c], prod[a][c]);
            first_term = false;
        }
        cur_term = dd.term[f];
        const double amp = dd.amp[f];
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                double v = __dmul_rn(amp, core_value(dd, f, r2[a][c]));
                prod[a][c] = new_term ? v : __dmul_rn(prod[a][c], v);
            }
    }
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) sum[a][c] = first_term ? prod[a][c] : __dadd_rn(sum[a][c], prod[a][c]);

#pragma unroll
    for (int a = 0; a < 4; a++) {
        int64_t i = i0 + ty + 16 * a;
        if (i >= n) continue;
        double *krow = K + i * ldk;
#pragma unroll
        for (int b = 0; b < 2; b++) {
            int64_t j = j0 + 2 * tx + 32 * b;
            if (j >= m) continue;
            if (vec_ok && j + 1 < m) {
                *reinterpret_cast<double2 *>(krow + j) = make_double2(sum[a][2 * b], sum[a][2 * b + 1]);
            } else {
                krow[j] = sum[a][2 * b];
                if (j + 1 < m) krow[j + 1] = sum[a][2 * b + 1];
            }
        }
    }
}

// Reverse-mode contraction of the Gram build: out[f][.] += sum_ij G_ij dK_ij/d(param of factor f).
// symlower = 0: G is a dense n x m matrix, all pairs (i, j) are visited.
// symlower = 1: x == y, only j <= i is visited, G_ij = w_ij (Ginv[i][j] - b_i b_j) with w = 2 off the diagonal
//               (the collapsed dK_vjp(invK) - dK_vjp(outer(invKr, invKr)) of _decomp.py:505-509).
// acc layout per factor: [0] d/d amp, [1] d/d log(scale), [2] d/d par1
template <bool DEV>
__global__ void __launch_bounds__(G_THREADS) gram_iso_vjp_kernel(const __grid_constant__ GramDesc d,
                                                                 const double *__restrict__ x, int64_t ldx,
                                                                 int64_t n, const double *__restrict__ y, int64_t ldy,
                                                                 int64_t m, const double *__restrict__ G, int64_t ldg,
                                                                 const double *__restrict__ bvec, int symlower,
                                                                 int tiles_n, double *__restrict__ out, const double *__restrict__ devpar) {
    __shared__ DevDescStore<DEV> sdesc;
    if constexpr (DEV) load_dev_desc(d, devpar, sdesc.d, threadIdx.x);
    const GramDesc &dd = [&]() -> const GramDesc & {
        if constexpr (DEV)
            return sdesc.d;
        else
            return d;
    }();
    extern __shared__ __align__(16) double gsm[];
    double *su = gsm;
    double *sv = gsm + (size_t)dd.nslots * GT;
    __shared__ double red[G_THREADS / 32][3 * LGP_MAX_FACTORS];
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
    stage_points(dd, su, x, ldx, n, i0, false, tid);
    stage_points(dd, sv, y, ldy, m, j0, true, tid);
    __syncthreads();

    double acc[3 * LGP_MAX_FACTORS];
#pragma unroll
    for (int k = 0; k < 3 * LGP_MAX_FACTORS; k++) acc[k] = 0.0;

#pragma unroll 1
    for (int a = 0; a < 4; a++) {
        const int64_t i = i0 + ty + 16 * a;
        if (i >= n) continue;
        const double bi = bvec ? bvec[i] : 0.0;
#pragma unroll 1
        for (int c = 0; c < 4; c++) {
            const int cc = 2 * tx + 32 * (c >> 1) + (c & 1);
            const int64_t j = j0 + cc;
            if (j >= m || (symlower && j > i)) continue;
            double g = G[i * ldg + j];
            if (bvec) g -= bi * bvec[j];
            if (symlower && j != i) g *= 2.0;
            // evaluate all factors
            double val[LGP_MAX_FACTORS], dr2[LGP_MAX_FACTORS], dp1[LGP_MAX_FACTORS], r2s[LGP_MAX_FACTORS];
#pragma unroll
            for (int f = 0; f < LGP_MAX_FACTORS; f++) {
                if (f < dd.nfactors) {
                    double r2 = 0.0;
                    for (int s = dd.slot0[f]; s < dd.slot0[f] + dd.nslot[f]; s++) {
                        double df = su[s * GT + ty + 16 * a] - sv[s * GT + cc];
                        r2 += df * df;
                    }
                    r2s[f] = r2;
                    core_derivs(dd, f, r2, val[f], dr2[f], dp1[f]);
                }
            }
#pragma unroll
            for (int f = 0; f < LGP_MAX_FACTORS; f++) {
                if (f < dd.nfactors) {
                    // product of the other factors of the same term (with their amps)
                    double others = 1.0;
#pragma unroll
                    for (int h = 0; h < LGP_MAX_FACTORS; h++)
                        if (h < dd.nfactors && h != f && dd.term[h] == dd.term[f]) others *= dd.amp[h] * val[h];
                    const double go = g * others;
                    acc[3 * f + 0] += go * val[f];
                    acc[3 * f + 1] += go * dd.amp[f] * dr2[f] * (-2.0 * r2s[f]);
                    acc[3 * f + 2] += go * dd.amp[f] * dp1[f];
                }
            }
        }
    }
    const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
    for (int k = 0; k < 3 * LGP_MAX_FACTORS; k++) {
        double v = warp_sum(acc[k]);
        if (lane == 0) red[warp][k] = v;
    }
    __syncthreads();
    if (tid < 3 * dd.nfactors) {
        double v = 0.0;
        for (int w = 0; w < G_THREADS / 32; w++) v += red[w][tid];
        atomicAdd(out + tid, v);
    }
}

// Forward-mode derivative of the Gram build: D_ij = sum_f sum_c tan[3f+c] dK_ij/d(param c of factor f), c = amp, log scale,
// par1 (same layout as the VJP output).  One pass over the tile; every factor is evaluated once per entry with its
// derivatives, the product rule is applied inside each term.  Used by the Fisher-information path
// (src/lsqfitgp/_fit.py:676-683: jax.jacfwd of decomp.matrix(); _linalg/_decomp.py:535-558).
template <bool DEV>
__global__ void __launch_bounds__(G_THREADS) gram_iso_jvp_kernel(const __grid_constant__ GramDesc d,
                                                                 const __grid_constant__ GramTangent tan,
                                                                 const double *__restrict__ x, int64_t ldx, int64_t n,
                                                                 const double *__restrict__ y, int64_t ldy, int64_t m,
                                                                 double *__restrict__ D, int64_t ldd, const double *__restrict__ devpar, const double *__restrict__ devtan) {
    __shared__ DevDescStore<DEV> sdesc;
    if constexpr (DEV) load_dev_desc(d, devpar, sdesc.d, threadIdx.x);
    const GramDesc &dd = [&]() -> const GramDesc & {
        if constexpr (DEV)
            return sdesc.d;
        else
            return d;
    }();
    extern __shared__ __align__(16) double gsm[];
    double *su = gsm;
    double *sv = gsm + (size_t)dd.nslots * GT;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t i0 = (int64_t)blockIdx.y * GT, j0 = (int64_t)blockIdx.x * GT;
    stage_points(dd, su, x, ldx, n, i0, false, tid);
    stage_points(dd, sv, y, ldy, m, j0, true, tid);
    __syncthreads();
#pragma unroll 1
    for (int a = 0; a < 4; a++) {
        const int64_t i = i0 + ty + 16 * a;
        if (i >= n) continue;
#pragma unroll 1
        for (int c = 0; c < 4; c++) {
            const int cc = 2 * tx + 32 * (c >> 1) + (c & 1);
            const int64_t j = j0 + cc;
            if (j >= m) continue;
            double total = 0.0;
            // walk the terms: value of the term P = prod_f amp_f v_f, derivative sum_f (dlog-free product rule)
            int f = 0;
            while (f < dd.nfactors) {
                const int term = dd.term[f];
                double prod = 1.0;   // product of amp_h * val_h over the factors seen so far
                double dsum = 0.0;   // derivative of that product along the tangent
                for (; f < dd.nfactors && dd.term[f] == term; f++) {
                    double r2 = 0.0;
                    for (int s = dd.slot0[f]; s < dd.slot0[f] + dd.nslot[f]; s++) {
                        const double df = su[s * GT + ty + 16 * a] - sv[s * GT + cc];
                        r2 += df * df;
                    }
                    double val, dr2, dp1;
                    core_derivs(dd, f, r2, val, dr2, dp1);
                    const double v = dd.amp[f] * val;
                    const double t0 = DEV ? devtan[3 * f] : tan.t[3 * f], t1 = DEV ? devtan[3 * f + 1] : tan.t[3 * f + 1],
                                 t2 = DEV ? devtan[3 * f + 2] : tan.t[3 * f + 2];
                    const double dv = t0 * val + dd.amp[f] * (t1 * dr2 * (-2.0 * r2) + t2 * dp1);
                    dsum = dsum * v + prod * dv;
                    prod *= v;
                }
                total += dsum;
            }
            D[i * ldd + j] = total;
        }
    }
}

// out[0] += sum_{i<rows, j<cols} A[i*lda + j] * B[i*ldb + j]   (Frobenius inner product; the k x k Fisher contraction
// einsum('kij,qij->kq') of _decomp.py:553 is k(k+1)/2 of these)
__global__ void __launch_bounds__(256) frob_dot_kernel(const double *__restrict__ A, int64_t lda,
                                                       const double *__restrict__ B, int64_t ldb, int64_t rows,
                                                       int64_t cols, double *__restrict__ out) {
    __shared__ double red[8];
    double acc = 0.0;
    for (int64_t i = blockIdx.x; i < rows; i += gridDim.x) {
        const double *a = A + i * lda, *b = B + i * ldb;
        for (int64_t j = threadIdx.x; j < cols; j += 256) acc += a[j] * b[j];
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double v = 0.0;
        for (int w = 0; w < 8; w++) v += red[w];
        atomicAdd(out, v);
    }
}

// ------------------------------------------------------------------------------------------------
// Fast path: K = amp * core(r2 / scale^2) [+ amp_w * White] [+ const], one isotropic factor over the same fields
// for x and y.  Symmetric mode evaluates only tiles on or below the diagonal and mirrors them through shared
// memory so that both the tile and its transpose are written with full 512-byte row segments.
// The arithmetic (operation order, explicit roundings) is identical to the general kernel.
// ------------------------------------------------------------------------------------------------
struct FastDesc {
    int kind, p, nd;        // main factor
    int has_white, has_const, white_raw;
    double scale, loc, par0, par1, amp, amp_white, amp_const;
    double coef[G_MAX_P];
    double coef2[G_MAX_P];  // 2 * coef (exact), precomputed on the host for the fast path
    double mat[MATERN_NPAR];  // LGP_K_MATERN: host-computed constants of the order (bessel_k.cuh)
    double rpar1, cexp, r2max;  // rational quadratic fast path: RN(1/beta), -beta/2, largest r2 it accepts
    int cauchy_fast;
    double rscale;          // RN(1 / scale) for fm_div_recip
    int div_fast;           // scale inside the exponent range where fm_div_recip is exact
    unsigned char dims[LGP_MAX_DIMS];
};

// (x - loc) / scale, correctly rounded like the reference's division (_ops.py:292-326): with the host-computed
// reciprocal and two exact-residual corrections (fastmath.cuh) where that is proven exact, library division elsewhere
__device__ __forceinline__ double fast_scale_point(const FastDesc &d, double xr) {
    const double a = __dsub_rn(xr, d.loc);
    if (d.div_fast && fm_div_recip_ok(a)) return fm_div_recip(a, d.scale, d.rscale);
    return __ddiv_rn(a, d.scale);
}

template <int KIND>
__device__ __forceinline__ double fast_core(const FastDesc &d, double r2) {
    if (KIND == LGP_K_EXPQUAD) return exp(__dmul_rn(-0.5, r2));
    if (KIND == LGP_K_MATERNP) {
        double z = __dadd_rn(__dmul_rn((double)(2 * d.p + 1), r2), d.par0);
        double x = sqrt(z);
        double poly = 1.0;
        for (int k = d.p - 1; k >= 0; k--)
            poly = __dadd_rn(1.0, __dmul_rn(__dmul_rn(__dmul_rn(poly, d.coef[k]), 2.0), x));
        return __dmul_rn(exp(-x), poly);
    }
    if (KIND == LGP_K_MATERN) {
        double val, dr2;
        matern_nu_core(d.mat, r2, false, val, dr2);
        return val;
    }
    // Cauchy
    double pw = (d.par0 == 2.0) ? r2 : pow(r2, d.par0 / 2.0);
    return pow(__dadd_rn(1.0, pw / d.par1), -d.par1 / d.par0);
}

constexpr int FT = 64;

template <int KIND, bool SYM>
__global__ void __launch_bounds__(G_THREADS, 2) gram_fast_kernel(const __grid_constant__ FastDesc d,
                                                                 const double *__restrict__ x, int64_t ldx, int64_t n,
                                                                 const double *__restrict__ y, int64_t ldy, int64_t m,
                                                                 double *__restrict__ K, int64_t ldk, int vec_ok,
                                                                 int tiles_n) {
    extern __shared__ __align__(16) double fsm[];
    // layout: su[nd][64], sv[nd][64], (raw copies for White when the main factor rescales) ru[nd][64], rv[nd][64],
    // then the transpose buffer T[64][65] (version 1 kernel) in symmetric mode
    const int nd = d.nd;
    double *su = fsm, *sv = fsm + nd * FT;
    double *ru = sv + nd * FT, *rv = ru + (d.white_raw ? nd * FT : 0);
    double *T = rv + (d.white_raw ? nd * FT : 0);
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    int tm, tn;
    if (SYM) {
        long long b = blockIdx.x;
        tm = (int)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
        while ((long long)(tm + 1) * (tm + 2) / 2 <= b) tm++;
        while ((long long)tm * (tm + 1) / 2 > b) tm--;
        tn = (int)(b - (long long)tm * (tm + 1) / 2);
    } else {
        tm = blockIdx.x / tiles_n;
        tn = blockIdx.x % tiles_n;
    }
    const int64_t i0 = (int64_t)tm * FT, j0 = (int64_t)tn * FT;
    for (int idx = tid; idx < nd * FT; idx += G_THREADS) {
        const int s = idx / FT, r = idx % FT;
        const int64_t i = i0 + r, j = j0 + r;
        double xr = (i < n) ? x[(int64_t)d.dims[s] * ldx + i] : 0.0;
        double yr = (j < m) ? y[(int64_t)d.dims[s] * ldy + j] : 0.0;
        su[idx] = fast_scale_point(d, xr);
        sv[idx] = fast_scale_point(d, yr);
        if (d.white_raw) {
            ru[idx] = xr;
            rv[idx] = yr;
        }
    }
    __syncthreads();

    double r2[4][4];
    bool eq[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) {
            r2[a][c] = 0.0;
            eq[a][c] = true;
        }
    for (int s = 0; s < nd; s++) {
        double uu[4], vv[4];
#pragma unroll
        for (int a = 0; a < 4; a++) uu[a] = su[s * FT + ty + 16 * a];
#pragma unroll
        for (int b = 0; b < 2; b++) {
            double2 t = *reinterpret_cast<const double2 *>(&sv[s * FT + 2 * tx + 32 * b]);
            vv[2 * b] = t.x;
            vv[2 * b + 1] = t.y;
        }
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                double df = __dsub_rn(uu[a], vv[c]);
                r2[a][c] = __dadd_rn(r2[a][c], __dmul_rn(df, df));
            }
        if (d.has_white) {
            if (d.white_raw) {
#pragma unroll
                for (int a = 0; a < 4; a++) uu[a] = ru[s * FT + ty + 16 * a];
#pragma unroll
                for (int b = 0; b < 2; b++) {
                    double2 t = *reinterpret_cast<const double2 *>(&rv[s * FT + 2 * tx + 32 * b]);
                    vv[2 * b] = t.x;
                    vv[2 * b + 1] = t.y;
                }
            }
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) eq[a][c] = eq[a][c] && (uu[a] == vv[c]);
        }
    }
    double val[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) {
            double v = __dmul_rn(d.amp, fast_core<KIND>(d, r2[a][c]));
            if (d.has_white) v = __dadd_rn(v, eq[a][c] ? d.amp_white : 0.0);
            if (d.has_const) v = __dadd_rn(v, d.amp_const);
            val[a][c] = v;
        }
    // direct tile
#pragma unroll
    for (int a = 0; a < 4; a++) {
        int64_t i = i0 + ty + 16 * a;
        if (i >= n) continue;
        double *krow = K + i * ldk;
#pragma unroll
        for (int b = 0; b < 2; b++) {
            int64_t j = j0 + 2 * tx + 32 * b;
            if (j >= m) continue;
            if (vec_ok && j + 1 < m) {
                *reinterpret_cast<double2 *>(krow + j) = make_double2(val[a][2 * b], val[a][2 * b + 1]);
            } else {
                krow[j] = val[a][2 * b];
                if (j + 1 < m) krow[j + 1] = val[a][2 * b + 1];
            }
        }
    }
    if (SYM && tm != tn) {
        // mirrored tile: K[j][i] = K[i][j]
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) T[(2 * tx + 32 * (c >> 1) + (c & 1)) * (FT + 1) + ty + 16 * a] = val[a][c];
        __syncthreads();
        const int warp = tid >> 5, lane = tid & 31;
        for (int rr = warp; rr < FT; rr += G_THREADS / 32) {
            int64_t j = j0 + rr;  // row of the mirrored tile
            if (j >= m) break;
            double *krow = K + j * ldk + i0;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                int cidx = lane + 32 * h;
                if (i0 + cidx < n) krow[cidx] = T[rr * (FT + 1) + cidx];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Specialised fast path (ExpQuad, and Matern with nu = P + 1/2, P <= 3): same tiling and the same r2 arithmetic as
// gram_fast_kernel, but the core is evaluated with the short exp/sqrt of fastmath.cuh (11 + 7 DP instructions instead of
// libm's ~40 with slow-path calls), the Horner recurrence is unrolled at compile time, and the White term is only
// examined where r2 == 0.  With symmetry this brings the build from the FP64-ALU bound towards the HBM write bound
// (DESIGN.md section 3).  Error of the core <= 1 ulp (tests/test_fastmath_cpu.py); sqrt is correctly rounded.
// ------------------------------------------------------------------------------------------------
// Hot path: no branches, no range checks: the caller tracks the smallest and largest r2 of the thread (as unsigned high
// words, which order like the non-negative doubles) and redoes out-of-range entries on the slow path.
// Interleaved copies of the exp table in shared memory (see fm_exp_neg_fast).  Measured on B200, n = 20000, symmetric build:
// ExpQuad 0.632 -> 0.610 ms with 4 copies (the lookups' bank conflicts were on its critical path), Matern-5/2 0.740 -> 0.783 ms
// (issue-bound: the extra address arithmetic costs more than the conflicts), so only ExpQuad replicates.
template <int KIND>
struct FTabRep {
    static constexpr int value = KIND == LGP_K_EXPQUAD ? 4 : 1;
};

template <int KIND, int P>
__device__ __forceinline__ double fast2_core(double r2, double nu2, double par0, double c0, double c1, double c2,
                                             const ExpTab *tab, const LogTab *ltab) {
    if (KIND == LGP_K_EXPQUAD) return fm_exp_neg_fast<FTabRep<KIND>::value>(__dmul_rn(-0.5, r2), tab);
    if (KIND == LGP_K_CAUCHY) {
        // rational quadratic (alpha = 2): (1 + r2/beta)^(-beta/2) (_basic.py:339-343); here nu2 = beta, par0 = RN(1/beta),
        // c0 = -beta/2.  Division and sum rounded as in the reference, the power as exp(c0 log x) with the short log / exp
        const double x = __dadd_rn(1.0, fm_div_recip(r2, nu2, par0));
        return fm_exp_neg_fast<FTabRep<KIND>::value>(__dmul_rn(c0, fm_log_ge1_fast(x, ltab)), tab);
    }
    // Maternp: x = sqrt((2p+1) r2 + par0); exp(-x) * poly_p(2x)   (_matern.py:48-49, _bessel.py:103-110)
    const double z = __dadd_rn(__dmul_rn(nu2, r2), par0);
    const double x = fm_sqrt_fast(z);
    const double ex = fm_exp_neg_fast<FTabRep<KIND>::value>(-x, tab);
    if (P == 0) return ex;
    // Horner in the reference's order poly = 1 + ((poly*c_k)*2)*x, the last product-sum fused
    double poly = 1.0;
    // (c_k here = 2*coef_k, an exact doubling; the first step has poly == 1, so poly*c == c without a multiplication)
    if (P >= 3) poly = __fma_rn(c2, x, 1.0);
    if (P == 2) poly = __fma_rn(c1, x, 1.0);
    if (P >= 3) poly = __fma_rn(__dmul_rn(poly, c1), x, 1.0);
    if (P == 1) poly = __fma_rn(c0, x, 1.0);
    if (P >= 2) poly = __fma_rn(__dmul_rn(poly, c0), x, 1.0);
    return __dmul_rn(ex, poly);
}

// Is r2 outside the range where fast2_core is valid (or does it need the White comparison)?
//   ExpQuad: exp(-r2/2) leaves the normal range beyond r2 = 1416; r2 < 2^-1022 (high word 0, includes r2 == 0) matters
//            only for White but is always sent to the slow path.
//   Maternp: 2^-960 <= z = (2p+1) r2 + par0 <= 501264 (x <= 708; the lower end keeps the reciprocal-square-root estimate
//            in range and catches z == 0); with a White term also r2 == 0.
template <int KIND>
__device__ __forceinline__ bool fast2_out_of_range(double r2, double nu2, double par0, bool white) {
    const unsigned hr = (unsigned)__double2hiint(r2);
    if (KIND == LGP_K_EXPQUAD) return (hr - 1u) > (0x40962000u - 1u);
    if (KIND == LGP_K_CAUCHY)  // nu2 = largest accepted r2 (|exponent| <= 200); below 2^-500 (and r2 == 0): library path
        return (hr - 0x20b00000u) > ((unsigned)__double2hiint(nu2) - 0x20b00000u);
    const unsigned hz = (unsigned)__double2hiint(__dadd_rn(__dmul_rn(nu2, r2), par0));
    return ((hz - 0x03f00000u) > (0x411e9840u - 0x03f00000u)) || (white && hr == 0u);
}

// Slow path for one entry (rare: diagonal, duplicated points, underflowing tails): libm core + White comparison
template <int KIND>
__device__ __noinline__ double fast2_slow_entry(const FastDesc &d, double r2, const double *wu, const double *wv,
                                                int row, int col) {
    double v = __dmul_rn(d.amp, fast_core<KIND>(d, r2));
    if (d.has_white) {
        bool eq = (r2 == 0.0);
        for (int s = 0; s < d.nd && eq; s++) eq = (wu[s * FT + row] == wv[s * FT + col]);
        v = __dadd_rn(v, eq ? d.amp_white : 0.0);
    }
    return v;
}

// The same for the symmetric version-3 kernel, which does not stage raw coordinates: the White comparison of the (rare)
// entries with r2 == 0 reads them from global memory (keeps 3 KB of shared memory per CTA for the replicated exp table)
template <int KIND>
__device__ __noinline__ double fast3_slow_entry(const FastDesc &d, double r2, const double *su, const double *sv,
                                                const double *__restrict__ x, int64_t ldx, int64_t i, int64_t j, int row,
                                                int col) {
    double v = __dmul_rn(d.amp, fast_core<KIND>(d, r2));
    if (d.has_white) {
        bool eq = (r2 == 0.0);
        for (int s = 0; s < d.nd && eq; s++)
            eq = d.white_raw ? (x[(int64_t)d.dims[s] * ldx + i] == x[(int64_t)d.dims[s] * ldx + j])
                             : (su[s * FT + row] == sv[s * FT + col]);
        v = __dadd_rn(v, eq ? d.amp_white : 0.0);
    }
    return v;
}

constexpr int F2_TS = FT + 2;  // row stride of the transpose buffer: 16-byte aligned rows for the bulk stores

template <int KIND, int P, bool SYM>
__global__ void __launch_bounds__(G_THREADS, 3) gram_fast2_kernel(const __grid_constant__ FastDesc d,
                                                                  const double *__restrict__ x, int64_t ldx, int64_t n,
                                                                  const double *__restrict__ y, int64_t ldy, int64_t m,
                                                                  double *__restrict__ K, int64_t ldk, int vec_ok,
                                                                  int tiles_n) {
    extern __shared__ __align__(16) double fsm[];
    // layout: exp table (64 x 16 B), su[nd][64], sv[nd][64], raw copies ru, rv (White with a rescaled main factor),
    // transpose buffer T[64][66] in symmetric mode
    const int nd = d.nd;
    constexpr int F_TABREP = FTabRep<KIND>::value;
    ExpTab *tab0 = reinterpret_cast<ExpTab *>(fsm);      // F_TABREP interleaved copies: entry j of copy c at [j * F_TABREP + c]
    const ExpTab *tab = tab0 + (threadIdx.x & (F_TABREP - 1));  // this lane's copy
    const LogTab *ltab = reinterpret_cast<const LogTab *>(fsm + 128 * F_TABREP);  // rational quadratic only
    double *su = fsm + 128 * F_TABREP + (KIND == LGP_K_CAUCHY ? 256 : 0), *sv = su + nd * FT;
    double *ru = sv + nd * FT, *rv = ru + (d.white_raw ? nd * FT : 0);
    double *T = rv + (d.white_raw ? nd * FT : 0);
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    int tm, tn;
    if (SYM) {
        long long b = blockIdx.x;
        tm = (int)((sqrtf(8.0f * (float)b + 1.0f) - 1.0f) * 0.5f);  // single precision + exact integer fix-up
        while ((long long)(tm + 1) * (tm + 2) / 2 <= b) tm++;
        while ((long long)tm * (tm + 1) / 2 > b) tm--;
        tn = (int)(b - (long long)tm * (tm + 1) / 2);
    } else {
        tm = blockIdx.x / tiles_n;
        tn = blockIdx.x % tiles_n;
    }
    const int64_t i0 = (int64_t)tm * FT, j0 = (int64_t)tn * FT;
    if (tid < 64 * F_TABREP) tab0[tid] = EXP_TAB_DEV[tid / F_TABREP];
    if (KIND == LGP_K_CAUCHY && tid < 64) reinterpret_cast<LogTab *>(fsm + 128 * F_TABREP)[tid] = LOG_TAB_DEV[tid];
    for (int idx = tid; idx < nd * FT; idx += G_THREADS) {
        const int s = idx / FT, r = idx % FT;
        const int64_t i = i0 + r, j = j0 + r;
        double xr = (i < n) ? x[(int64_t)d.dims[s] * ldx + i] : 0.0;
        double yr = (j < m) ? y[(int64_t)d.dims[s] * ldy + j] : 0.0;
        su[idx] = fast_scale_point(d, xr);
        sv[idx] = fast_scale_point(d, yr);
        if (d.white_raw) {
            ru[idx] = xr;
            rv[idx] = yr;
        }
    }
    __syncthreads();

    // core parameters (Maternp: 2p+1, offset, doubled Horner ratios; rational quadratic: beta, 1/beta, -beta/2) and the
    // first argument of the range test (rational quadratic: the largest accepted r2)
    const double nu2 = KIND == LGP_K_CAUCHY ? d.par1 : (double)(2 * P + 1);
    const double par0 = KIND == LGP_K_CAUCHY ? d.rpar1 : d.par0, amp = d.amp;
    const double c0 = KIND == LGP_K_CAUCHY ? d.cexp : d.coef2[0], c1 = d.coef2[1], c2 = d.coef2[2];
    const double rng0 = KIND == LGP_K_CAUCHY ? d.r2max : nu2;
    const double *wu = d.white_raw ? ru : su, *wv = d.white_raw ? rv : sv;
    const bool white = d.has_white != 0;
    const bool mirror = SYM && tm != tn;
    const bool interior = vec_ok && i0 + FT <= n && j0 + FT <= m;  // whole tile inside the matrix: no bounds checks

    // The 4 x 4 entries of a thread are produced in two batches of 2 rows x 4 columns: half the live registers of a
    // full 16-entry batch (3 CTAs per SM without spills), still 8 independent dependency chains per thread.
#pragma unroll 1
    for (int a0 = 0; a0 < 4; a0 += 2) {
        double r2[2][4];
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) r2[a][c] = 0.0;
        for (int s = 0; s < nd; s++) {
            double uu[2], vv[4];
#pragma unroll
            for (int a = 0; a < 2; a++) uu[a] = su[s * FT + ty + 16 * (a0 + a)];
#pragma unroll
            for (int b = 0; b < 2; b++) {
                double2 t = *reinterpret_cast<const double2 *>(&sv[s * FT + 2 * tx + 32 * b]);
                vv[2 * b] = t.x;
                vv[2 * b + 1] = t.y;
            }
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    double df = __dsub_rn(uu[a], vv[c]);
                    r2[a][c] = __dadd_rn(r2[a][c], __dmul_rn(df, df));
                }
        }
        double val[2][4];
        unsigned hmin = 0xffffffffu, hmax = 0u;  // high words of the smallest / largest r2 (monotone for r2 >= 0)
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const unsigned hr = (unsigned)__double2hiint(r2[a][c]);
                hmin = min(hmin, hr);
                hmax = max(hmax, hr);
                val[a][c] = __dmul_rn(amp, fast2_core<KIND, P>(r2[a][c], nu2, par0, c0, c1, c2, tab, ltab));
            }
        // the range test is monotone in r2: test the two extremes (the high word rounds r2 down, which only makes the
        // test stricter at the low end; at the high end the bounds are far inside the true limits)
        if (fast2_out_of_range<KIND>(__hiloint2double((int)hmin, 0), rng0, par0, white) ||
            fast2_out_of_range<KIND>(__hiloint2double((int)hmax, 0xffffffff), rng0, par0, white)) {
            // some entry of this thread left the fast range: redo exactly those with the library path
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int c = 0; c < 4; c++)
                    if (fast2_out_of_range<KIND>(r2[a][c], rng0, par0, white))
                        val[a][c] = fast2_slow_entry<KIND>(d, r2[a][c], wu, wv, ty + 16 * (a0 + a),
                                                           2 * tx + 32 * (c >> 1) + (c & 1));
        }
        if (d.has_const) {
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) val[a][c] = __dadd_rn(val[a][c], d.amp_const);
        }
        // direct tile
        if (interior) {
            double *kp = K + (i0 + ty + 16 * a0) * ldk + j0 + 2 * tx;
#pragma unroll
            for (int a = 0; a < 2; a++) {
                *reinterpret_cast<double2 *>(kp) = make_double2(val[a][0], val[a][1]);
                *reinterpret_cast<double2 *>(kp + 32) = make_double2(val[a][2], val[a][3]);
                kp += 16 * ldk;
            }
        } else
#pragma unroll
        for (int a = 0; a < 2; a++) {
            int64_t i = i0 + ty + 16 * (a0 + a);
            if (i >= n) continue;
            double *krow = K + i * ldk;
#pragma unroll
            for (int b = 0; b < 2; b++) {
                int64_t j = j0 + 2 * tx + 32 * b;
                if (j >= m) continue;
                if (vec_ok && j + 1 < m) {
                    *reinterpret_cast<double2 *>(krow + j) = make_double2(val[a][2 * b], val[a][2 * b + 1]);
                } else {
                    krow[j] = val[a][2 * b];
                    if (j + 1 < m) krow[j + 1] = val[a][2 * b + 1];
                }
            }
        }
        if (mirror) {
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int c = 0; c < 4; c++)
                    T[(2 * tx + 32 * (c >> 1) + (c & 1)) * F2_TS + ty + 16 * (a0 + a)] = val[a][c];
        }
    }
    if (mirror) {
        // mirrored tile: K[j][i] = K[i][j]
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        const int warp = tid >> 5, lane = tid & 31;
        if (interior) {
            // TMA bulk stores: one 512-byte row of the transposed tile per copy, issued by 64 threads; the copies read
            // shared memory through the async proxy (made visible by the fence before the barrier above)
            if (tid < FT) {
                const uint32_t src = smem_u32(T + tid * F2_TS);
                double *dst = K + (j0 + tid) * ldk + i0;
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src),
                             "r"(FT * 8)
                             : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            }
        } else
        for (int rr = warp; rr < FT; rr += G_THREADS / 32) {
            int64_t j = j0 + rr;  // row of the mirrored tile
            if (j >= m) break;
            double *krow = K + j * ldk + i0;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                int cidx = lane + 32 * h;
                if (i0 + cidx < n) krow[cidx] = T[rr * F2_TS + cidx];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Symmetric fast path, version 3: same arithmetic as gram_fast2_kernel<.., true>, different data movement.
//   * lanes of a half-warp run along ROWS of the tile (ty = tid & 15), so that the transposed copy of the tile is
//     written to shared memory with consecutive addresses (conflict-free; the column-major lane order of version 2
//     put 8 wavefronts on every one of those stores);
//   * BOTH the tile and its mirror image are staged in shared memory (row stride 66 doubles: 16-byte aligned rows,
//     conflict-free 128-bit row stores) and leave through TMA bulk stores, one 512-byte row per copy: the SM issues
//     128 bulk copies per tile instead of 4096 scattered 16-byte stores, and no thread waits on a global store.
// Edge tiles (not fully inside the matrix) fall back to bounds-checked stores.
// ------------------------------------------------------------------------------------------------
// PREP (lgp_gram_iso_prepare): the factorisation's input instead of K.  Same tiles, but (a) every entry is multiplied by
// 1/s^2 (the power-of-two equilibration scale, uniform because the diagonal of a stationary kernel is constant: read from
// prep.sinv), (b) only tiles on or below the diagonal are stored (no mirror image), into the npad x npad factor storage
// whose rows / columns >= n are identity padding, (c) the sums of |entry| over the rows of the tile and, for the mirrored
// half of the matrix, over its columns go to prep.rowpart[other tile index][row]: every (slot, row) pair is written exactly
// once, so that the Gershgorin row sums (reference eigval_bound, _decomp.py:349-354) are reduced in a fixed order.
struct GramPrep {
    const double *sinv;  // aux + LGP_AUX_SINV: entry 0 = 1/s
    double *rowpart;     // [npad / 64][npad]
    int64_t npad;
};
// One lower tile per CTA, 3 CTAs per SM: at most 80 registers, and the launchers opt in to 77 400 bytes of shared memory
// (3 * (76800 + 1024 reserved) = 228 KB)
template <int KIND, int P, bool PREP>
__global__ void __launch_bounds__(G_THREADS, 3) gram_fast3_kernel(const __grid_constant__ FastDesc d,
                                                               const double *__restrict__ x, int64_t ldx, int64_t n,
                                                               double *__restrict__ K, int64_t ldk, int vec_ok,
                                                               const GramPrep prep) {
    extern __shared__ __align__(16) double fsm[];
    const int nd = d.nd;
    constexpr int F_TABREP = FTabRep<KIND>::value;
    ExpTab *tab0 = reinterpret_cast<ExpTab *>(fsm);      // F_TABREP interleaved copies: entry j of copy c at [j * F_TABREP + c]
    const ExpTab *tab = tab0 + (threadIdx.x & (F_TABREP - 1));  // this lane's copy
    const LogTab *ltab = reinterpret_cast<const LogTab *>(fsm + 128 * F_TABREP);  // rational quadratic only
    double *su = fsm + 128 * F_TABREP + (KIND == LGP_K_CAUCHY ? 256 : 0), *sv = su + nd * FT;
    // raw coordinates for the White comparison are staged only where the 1 KB table leaves room for them (3 CTAs per SM);
    // the ExpQuad instantiation, with its 4 KB replicated table, reads them from global memory on the rare slow path
    constexpr bool RAWSM = F_TABREP == 1;
    double *ru = sv + nd * FT, *rv = ru + ((RAWSM && d.white_raw) ? nd * FT : 0);
    double *D = rv + ((RAWSM && d.white_raw) ? nd * FT : 0);  // D[row][col], stride F2_TS
    double *T = D + FT * F2_TS;                    // T[col][row]
    const int tid = threadIdx.x, ty = tid & 15, tx = tid >> 4;
    if (tid < 64 * F_TABREP) tab0[tid] = EXP_TAB_DEV[tid / F_TABREP];
    if (KIND == LGP_K_CAUCHY && tid < 64) reinterpret_cast<LogTab *>(fsm + 128 * F_TABREP)[tid] = LOG_TAB_DEV[tid];
    const long long b = blockIdx.x;  // lower tile b: row tm, column tn <= tm
    int tm = (int)((sqrtf(8.0f * (float)b + 1.0f) - 1.0f) * 0.5f);  // single precision + exact integer fix-up
    while ((long long)(tm + 1) * (tm + 2) / 2 <= b) tm++;
    while ((long long)tm * (tm + 1) / 2 > b) tm--;
    const int tn = (int)(b - (long long)tm * (tm + 1) / 2);
    const int64_t i0 = (int64_t)tm * FT, j0 = (int64_t)tn * FT;
    for (int idx = tid; idx < nd * FT; idx += G_THREADS) {
        const int s = idx / FT, r = idx % FT;
        const int64_t i = i0 + r, j = j0 + r;
        double xr = (i < n) ? x[(int64_t)d.dims[s] * ldx + i] : 0.0;
        double yr = (j < n) ? x[(int64_t)d.dims[s] * ldx + j] : 0.0;
        su[idx] = fast_scale_point(d, xr);
        sv[idx] = fast_scale_point(d, yr);
        if (RAWSM && d.white_raw) {
            ru[idx] = xr;
            rv[idx] = yr;
        }
    }
    __syncthreads();

    // core parameters (Maternp: 2p+1, offset, doubled Horner ratios; rational quadratic: beta, 1/beta, -beta/2) and the
    // first argument of the range test (rational quadratic: the largest accepted r2)
    const double nu2 = KIND == LGP_K_CAUCHY ? d.par1 : (double)(2 * P + 1);
    const double par0 = KIND == LGP_K_CAUCHY ? d.rpar1 : d.par0, amp = d.amp;
    const double c0 = KIND == LGP_K_CAUCHY ? d.cexp : d.coef2[0], c1 = d.coef2[1], c2 = d.coef2[2];
    const double rng0 = KIND == LGP_K_CAUCHY ? d.r2max : nu2;
    const bool white = d.has_white != 0;
    const bool mirror = tm != tn;
    const bool interior = PREP || (vec_ok && i0 + FT <= n && j0 + FT <= n);
    double prep_scale = 1.0;
    if (PREP) {
        const double si = prep.sinv[0];
        prep_scale = si * si;
    }

#pragma unroll 1
    for (int a0 = 0; a0 < 4; a0 += 2) {
        double r2[2][4];
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) r2[a][c] = 0.0;
        for (int s = 0; s < nd; s++) {
            double uu[2], vv[4];
#pragma unroll
            for (int a = 0; a < 2; a++) uu[a] = su[s * FT + ty + 16 * (a0 + a)];
#pragma unroll
            for (int bb = 0; bb < 2; bb++) {
                double2 t = *reinterpret_cast<const double2 *>(&sv[s * FT + 2 * tx + 32 * bb]);
                vv[2 * bb] = t.x;
                vv[2 * bb + 1] = t.y;
            }
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    double df = __dsub_rn(uu[a], vv[c]);
                    r2[a][c] = __dadd_rn(r2[a][c], __dmul_rn(df, df));
                }
        }
        double val[2][4];
        unsigned hmin = 0xffffffffu, hmax = 0u;
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const unsigned hr = (unsigned)__double2hiint(r2[a][c]);
                hmin = min(hmin, hr);
                hmax = max(hmax, hr);
                val[a][c] = __dmul_rn(amp, fast2_core<KIND, P>(r2[a][c], nu2, par0, c0, c1, c2, tab, ltab));
            }
        if (fast2_out_of_range<KIND>(__hiloint2double((int)hmin, 0), rng0, par0, white) ||
            fast2_out_of_range<KIND>(__hiloint2double((int)hmax, 0xffffffff), rng0, par0, white)) {
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int c = 0; c < 4; c++)
                    if (fast2_out_of_range<KIND>(r2[a][c], rng0, par0, white) &&
                        !(PREP && (i0 + ty + 16 * (a0 + a) >= n || j0 + 2 * tx + 32 * (c >> 1) + (c & 1) >= n)))
                        val[a][c] = RAWSM ? fast2_slow_entry<KIND>(d, r2[a][c], d.white_raw ? ru : su, d.white_raw ? rv : sv,
                                                                   ty + 16 * (a0 + a), 2 * tx + 32 * (c >> 1) + (c & 1))
                                          : fast3_slow_entry<KIND>(d, r2[a][c], su, sv, x, ldx, i0 + ty + 16 * (a0 + a),
                                                                   j0 + 2 * tx + 32 * (c >> 1) + (c & 1),
                                                                   ty + 16 * (a0 + a), 2 * tx + 32 * (c >> 1) + (c & 1));
        }
        if (d.has_const) {
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) val[a][c] = __dadd_rn(val[a][c], d.amp_const);
        }
        if (PREP) {
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) val[a][c] *= prep_scale;  // exact: power of two
            if (i0 + FT > n) {  // last tile rows: identity padding beyond n
#pragma unroll
                for (int a = 0; a < 2; a++)
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        const int64_t i = i0 + ty + 16 * (a0 + a), j = j0 + 2 * tx + 32 * (c >> 1) + (c & 1);
                        if (i >= n || j >= n) val[a][c] = (i == j) ? 1.0 : 0.0;
                    }
            }
        }
        if (interior) {
#pragma unroll
            for (int a = 0; a < 2; a++) {
                double *dp = D + (ty + 16 * (a0 + a)) * F2_TS + 2 * tx;
                *reinterpret_cast<double2 *>(dp) = make_double2(val[a][0], val[a][1]);
                *reinterpret_cast<double2 *>(dp + 32) = make_double2(val[a][2], val[a][3]);
            }
        } else {
#pragma unroll
            for (int a = 0; a < 2; a++) {
                int64_t i = i0 + ty + 16 * (a0 + a);
                if (i >= n) continue;
                double *krow = K + i * ldk;
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    int64_t j = j0 + 2 * tx + 32 * (c >> 1) + (c & 1);
                    if (j < n) krow[j] = val[a][c];
                }
            }
        }
        if (mirror && !PREP) {
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int c = 0; c < 4; c++)
                    T[(2 * tx + 32 * (c >> 1) + (c & 1)) * F2_TS + ty + 16 * (a0 + a)] = val[a][c];
        }
    }
    if (interior) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (PREP) {
            // partial Gershgorin sums of the tile: threads 0..63 one row each (rotated start: conflict-free), threads
            // 64..127 one column each (the rows of the mirror image)
            const int q = tid & 63;
            if (tid < FT) {
                double sum = 0.0;
#pragma unroll 8
                for (int c = 0; c < FT; c++) sum += fabs(D[q * F2_TS + ((c + q) & (FT - 1))]);
                prep.rowpart[(int64_t)tn * prep.npad + i0 + q] = sum;
            } else if (mirror && tid < 2 * FT) {
                double sum = 0.0;
#pragma unroll 8
                for (int r2_ = 0; r2_ < FT; r2_++) sum += fabs(D[r2_ * F2_TS + q]);
                prep.rowpart[(int64_t)tm * prep.npad + j0 + q] = sum;
            }
        }
        // rows of the tile by threads 0..63, rows of its mirror image by threads 64..127
        const int r = tid & 63;
        if (tid < FT || (mirror && !PREP && tid < 2 * FT)) {
            const bool second = tid >= FT;
            const uint32_t src = smem_u32((second ? T : D) + r * F2_TS);
            double *dst = second ? K + (j0 + r) * ldk + i0 : K + (i0 + r) * ldk + j0;
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(FT * 8)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            // shared memory must stay valid until the bulk store has read it
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
    } else if (mirror && !PREP) {
        __syncthreads();
        const int warp = tid >> 5, lane = tid & 31;
        for (int rr = warp; rr < FT; rr += G_THREADS / 32) {
            int64_t j = j0 + rr;
            if (j >= n) break;
            double *krow = K + j * ldk + i0;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                int cidx = lane + 32 * h;
                if (i0 + cidx < n) krow[cidx] = T[rr * F2_TS + cidx];
            }
        }
    }
}

// d core / d r2 for the fast path (value returned through `val`)
template <int KIND>
__device__ __forceinline__ void fast_core_derivs(const FastDesc &d, double r2, double &val, double &dr2,
                                                 double &dpar1) {
    dpar1 = 0.0;
    if (KIND == LGP_K_MATERN) {
        matern_nu_core(d.mat, r2, true, val, dr2);
    } else if (KIND == LGP_K_EXPQUAD) {
        val = exp(-0.5 * r2);
        dr2 = -0.5 * val;
    } else if (KIND == LGP_K_MATERNP) {
        const double nu2 = (double)(2 * d.p + 1);
        double z = nu2 * r2 + d.par0;
        double x = sqrt(z);
        double ex = exp(-x);
        double poly = 1.0;
        for (int k = d.p - 1; k >= 0; k--) poly = 1.0 + poly * d.coef[k] * 2.0 * x;
        val = ex * poly;
        if (d.p == 0) {
            dr2 = x > 0.0 ? -nu2 * ex / (2.0 * x) : 0.0;
        } else {
            const int pm = d.p - 1;
            double polym = 1.0;
            for (int k = pm - 1; k >= 0; k--)
                polym = 1.0 + polym * ((double)(pm - k) / (double)((2 * pm - k) * (k + 1))) * 2.0 * x;
            dr2 = -nu2 * ex * polym / (4.0 * ((double)d.p - 0.5));
        }
    } else {
        const double alpha = d.par0, beta = d.par1;
        double t = (alpha == 2.0) ? r2 : pow(r2, alpha / 2.0);
        double base = 1.0 + t / beta;
        val = pow(base, -beta / alpha);
        double dvdt = -(1.0 / alpha) * val / base;
        double dtdr2 = (alpha == 2.0) ? 1.0 : (r2 > 0.0 ? (alpha / 2.0) * t / r2 : 0.0);
        dr2 = dvdt * dtdr2;
        dpar1 = val * (-(1.0 / alpha) * log(base) + (t / (alpha * beta)) / base);
    }
}

// Fast-math value and d core / d r2 (ExpQuad, Maternp with compile-time P), arguments inside the range accepted by
// fast2_out_of_range; same formulas as fast_core_derivs.
constexpr int V_TABREP = 1;  // replicated tables measured slower here (1.14 -> 1.18 ms with 8 copies): the kernel is issue-bound
template <int KIND, int P>
__device__ __forceinline__ void fast2_core_derivs(const FastDesc &d, double r2, const ExpTab *tab, double &val,
                                                  double &dr2) {
    if (KIND == LGP_K_EXPQUAD) {
        val = fm_exp_neg_fast<V_TABREP>(-0.5 * r2, tab);
        dr2 = -0.5 * val;
        return;
    }
    constexpr int PP = P < 0 ? 0 : P;
    constexpr double nu2 = (double)(2 * PP + 1);
    const double z = nu2 * r2 + d.par0;
    const double x = fm_sqrt_fast(z);
    const double ex = fm_exp_neg_fast<V_TABREP>(-x, tab);
    if (PP == 0) {
        val = ex;
        dr2 = -nu2 * ex / (2.0 * x);
        return;
    }
    double poly = 1.0;
#pragma unroll
    for (int k = PP - 1; k >= 0; k--) poly = fma(poly * d.coef2[k], x, 1.0);
    val = ex * poly;
    constexpr int pm = PP - 1;
    double polym = 1.0;
#pragma unroll
    for (int k = pm - 1; k >= 0; k--)
        polym = fma(polym * (2.0 * (double)(pm - k) / (double)((2 * pm - k) * (k + 1))), x, 1.0);
    dr2 = (-nu2 / (4.0 * ((double)PP - 0.5))) * ex * polym;
}

// Fast symmetric VJP over the lower triangle: out[0..2] main factor (d amp, d log scale, d par1),
// out[3] = d/d amp_white, out[4] = d/d amp_const.  G_ij = w_ij (Ginv_ij - b_i b_j).
// P >= 0 (ExpQuad: 0; Maternp: the order): short in-kernel exp/sqrt for in-range entries; P < 0: library path only.
template <int KIND, int P>
__global__ void __launch_bounds__(G_THREADS, 2) gram_fast_vjp_kernel(const __grid_constant__ FastDesc d,
                                                                     const double *__restrict__ x, int64_t ldx,
                                                                     int64_t n, const double *__restrict__ G,
                                                                     int64_t ldg, const double *__restrict__ bvec,
                                                                     double *__restrict__ out) {
    extern __shared__ __align__(16) double fsm[];
    const int nd = d.nd;
    double *su = fsm, *sv = fsm + nd * FT;
    double *ru = sv + nd * FT, *rv = ru + (d.white_raw ? nd * FT : 0);
    __shared__ double sbi[FT], sbj[FT];
    __shared__ double red[G_THREADS / 32][5];
    __shared__ ExpTab tab0[64 * V_TABREP];   // V_TABREP interleaved copies (bank-private lookups, see fm_exp_neg_fast)
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const ExpTab *tab = tab0 + (tid & (V_TABREP - 1));
    if (P >= 0)
        for (int i = tid; i < 64 * V_TABREP; i += G_THREADS) tab0[i] = EXP_TAB_DEV[i / V_TABREP];
    long long b = blockIdx.x;
    int tm = (int)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
    while ((long long)(tm + 1) * (tm + 2) / 2 <= b) tm++;
    while ((long long)tm * (tm + 1) / 2 > b) tm--;
    const int tn = (int)(b - (long long)tm * (tm + 1) / 2);
    const int64_t i0 = (int64_t)tm * FT, j0 = (int64_t)tn * FT;
    // Tiles strictly below the diagonal and fully inside the matrix (almost all of them): the 16 entries of G this thread
    // needs are requested FIRST, eight independent 16-byte loads in flight per thread while the points are staged and the
    // squared distances computed (issued one by one next to their use, the loads left the kernel latency-bound: 0.87 TB/s)
    const bool vec_ok = ((ldg & 1) == 0) && ((reinterpret_cast<uintptr_t>(G) & 15) == 0);
    const bool interior = vec_ok && tm > tn && i0 + FT <= n;
    double gpre[4][4];
    if (interior) {
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int bb = 0; bb < 2; bb++) {
                const double2 t = __ldcs(reinterpret_cast<const double2 *>(G + (i0 + ty + 16 * a) * ldg + j0 + 2 * tx + 32 * bb));
                gpre[a][2 * bb] = t.x;
                gpre[a][2 * bb + 1] = t.y;
            }
    }
    for (int idx = tid; idx < nd * FT; idx += G_THREADS) {
        const int s = idx / FT, r = idx % FT;
        const int64_t i = i0 + r, j = j0 + r;
        double xr = (i < n) ? x[(int64_t)d.dims[s] * ldx + i] : 0.0;
        double yr = (j < n) ? x[(int64_t)d.dims[s] * ldx + j] : 0.0;
        su[idx] = (xr - d.loc) / d.scale;
        sv[idx] = (yr - d.loc) / d.scale;
        if (d.white_raw) {
            ru[idx] = xr;
            rv[idx] = yr;
        }
    }
    if (tid < FT) {
        sbi[tid] = (bvec && i0 + tid < n) ? bvec[i0 + tid] : 0.0;
        sbj[tid] = (bvec && j0 + tid < n) ? bvec[j0 + tid] : 0.0;
    }
    __syncthreads();

    double r2[4][4];
    bool eq[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) {
            r2[a][c] = 0.0;
            eq[a][c] = true;
        }
    for (int s = 0; s < nd; s++) {
        double uu[4], vv[4];
#pragma unroll
        for (int a = 0; a < 4; a++) uu[a] = su[s * FT + ty + 16 * a];
#pragma unroll
        for (int bb = 0; bb < 2; bb++) {
            double2 t = *reinterpret_cast<const double2 *>(&sv[s * FT + 2 * tx + 32 * bb]);
            vv[2 * bb] = t.x;
            vv[2 * bb + 1] = t.y;
        }
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                double df = uu[a] - vv[c];
                r2[a][c] += df * df;
            }
        if (d.has_white) {
            if (d.white_raw) {
#pragma unroll
                for (int a = 0; a < 4; a++) uu[a] = ru[s * FT + ty + 16 * a];
#pragma unroll
                for (int bb = 0; bb < 2; bb++) {
                    double2 t = *reinterpret_cast<const double2 *>(&rv[s * FT + 2 * tx + 32 * bb]);
                    vv[2 * bb] = t.x;
                    vv[2 * bb + 1] = t.y;
                }
            }
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) eq[a][c] = eq[a][c] && (uu[a] == vv[c]);
        }
    }
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (interior) {
        // straight-line: every entry is valid, off the diagonal (weight 2); no White hits unless points are duplicated
#pragma unroll
        for (int a = 0; a < 4; a++) {
            const double bi = sbi[ty + 16 * a];
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int cc = 2 * tx + 32 * (c >> 1) + (c & 1);
                const double g = 2.0 * (gpre[a][c] - bi * sbj[cc]);
                double val, dr2, dp1 = 0.0;
                if (P >= 0 && !fast2_out_of_range<KIND>(r2[a][c], (double)(2 * P + 1), d.par0, false))
                    fast2_core_derivs<KIND, P>(d, r2[a][c], tab, val, dr2);
                else
                    fast_core_derivs<KIND>(d, r2[a][c], val, dr2, dp1);
                acc[0] += g * val;
                acc[1] += g * d.amp * dr2 * (-2.0 * r2[a][c]);
                acc[2] += g * d.amp * dp1;
                if (d.has_white && eq[a][c]) acc[3] += g;
                acc[4] += g;
            }
        }
    } else
#pragma unroll
    for (int a = 0; a < 4; a++) {
        const int64_t i = i0 + ty + 16 * a;
        if (i >= n) continue;
        const double bi = sbi[ty + 16 * a];
#pragma unroll
        for (int bb = 0; bb < 2; bb++) {
            const int cc = 2 * tx + 32 * bb;
            const int64_t j = j0 + cc;
            if (j > i) continue;
            double g0, g1 = 0.0;
            const bool second = (j + 1 <= i);  // j + 1 <= i < n
            if (vec_ok && second) {
                double2 t = *reinterpret_cast<const double2 *>(G + i * ldg + j);
                g0 = t.x;
                g1 = t.y;
            } else {
                g0 = G[i * ldg + j];
                if (second) g1 = G[i * ldg + j + 1];
            }
#pragma unroll
            for (int e = 0; e < 2; e++) {
                if (e == 1 && !second) continue;
                double g = (e ? g1 : g0) - bi * sbj[cc + e];
                if (j + e != i) g *= 2.0;
                double val, dr2, dp1 = 0.0;
                if (P >= 0 && !fast2_out_of_range<KIND>(r2[a][2 * bb + e], (double)(2 * P + 1), d.par0, false))
                    fast2_core_derivs<KIND, P>(d, r2[a][2 * bb + e], tab, val, dr2);
                else
                    fast_core_derivs<KIND>(d, r2[a][2 * bb + e], val, dr2, dp1);
                acc[0] += g * val;
                acc[1] += g * d.amp * dr2 * (-2.0 * r2[a][2 * bb + e]);
                acc[2] += g * d.amp * dp1;
                if (d.has_white && eq[a][2 * bb + e]) acc[3] += g;
                acc[4] += g;
            }
        }
    }
    const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
    for (int k = 0; k < 5; k++) {
        double v = warp_sum(acc[k]);
        if (lane == 0) red[warp][k] = v;
    }
    __syncthreads();
    if (tid < 5) {
        double v = 0.0;
        for (int w = 0; w < G_THREADS / 32; w++) v += red[w][tid];
        atomicAdd(out + tid, v);
    }
}

// scatter the 5 fast-path sums into the (nfactors x 3) layout of the public ABI
__global__ void fast_vjp_scatter_kernel(const double *__restrict__ tmp, double *__restrict__ out, int nfactors,
                                        int pos_white, int pos_const) {
    if (threadIdx.x == 0) {
        for (int i = 0; i < 3 * nfactors; i++) out[i] = 0.0;
        out[0] = tmp[0];
        out[1] = tmp[1];
        out[2] = tmp[2];
        if (pos_white >= 0) out[3 * pos_white] = tmp[3];
        if (pos_const >= 0) out[3 * pos_const] = tmp[4];
    }
}

static bool build_fast(const lgp_factor_t *f, int nf, int ndim, FastDesc &d) {
    // accepted shape: [main factor in its own term] [+ White term] [+ Constant term], each at most once
    if (nf < 1 || nf > 3) return false;
    memset(&d, 0, sizeof(d));
    int main_i = -1;
    for (int i = 0; i < nf; i++) {
        for (int j = 0; j < nf; j++)
            if (i != j && f[i].term == f[j].term) return false;  // products: general kernel
        if (f[i].kind == LGP_K_WHITE) {
            if (d.has_white) return false;
            d.has_white = 1;
            d.amp_white = f[i].amp;
            if (f[i].scale_x != 1.0 || f[i].scale_y != 1.0 || f[i].loc_x != 0.0 || f[i].loc_y != 0.0) return false;
        } else if (f[i].kind == LGP_K_CONSTANT) {
            if (d.has_const) return false;
            d.has_const = 1;
            d.amp_const = f[i].amp;
        } else {
            if (main_i >= 0) return false;
            main_i = i;
        }
    }
    if (main_i < 0) return false;
    // term order must be main, white, const so that the sums are rounded in the reference's order
    int pos_white = -1, pos_const = -1;
    for (int i = 0; i < nf; i++) {
        if (f[i].kind == LGP_K_WHITE) pos_white = i;
        if (f[i].kind == LGP_K_CONSTANT) pos_const = i;
    }
    if (main_i != 0) return false;
    if (pos_white >= 0 && pos_const >= 0 && pos_white > pos_const) return false;
    const lgp_factor_t &m = f[main_i];
    if (m.scale_x != m.scale_y || m.loc_x != m.loc_y) return false;
    if (m.kind != LGP_K_EXPQUAD && m.kind != LGP_K_MATERNP && m.kind != LGP_K_CAUCHY && m.kind != LGP_K_MATERN)
        return false;
    if (m.kind == LGP_K_MATERN && !matern_nu_setup(m.par0, d.mat)) return false;  // (general path reports the error)
    d.kind = m.kind;
    d.p = m.ipar;
    d.scale = m.scale_x;
    d.rscale = 1.0 / m.scale_x;
    if (m.kind == LGP_K_CAUCHY && m.par0 == 2.0 && m.par1 >= 0x1p-100 && m.par1 <= 0x1p100) {
        d.cauchy_fast = 1;
        d.rpar1 = 1.0 / m.par1;
        d.cexp = -0.5 * m.par1;
        // (beta/2) log(1 + r2/beta) <= 200 keeps the error of exp(c log x) below 1e-13; also r2 <= 2^500 for the division
        const double lim = 400.0 / m.par1;
        d.r2max = lim < 700.0 ? fmin(m.par1 * expm1(lim), 0x1p500) : 0x1p500;
    }
    d.div_fast = (fabs(m.scale_x) >= 0x1p-200 && fabs(m.scale_x) <= 0x1p200) ? 1 : 0;
    d.loc = m.loc_x;
    d.par0 = m.par0;
    d.par1 = m.par1;
    d.amp = m.amp;
    if (m.kind == LGP_K_MATERNP) {
        if (d.p < 0 || d.p > G_MAX_P) return false;
        for (int k = 0; k < d.p; k++) {
            d.coef[k] = (double)(d.p - k) / (double)((2 * d.p - k) * (k + 1));
            d.coef2[k] = 2.0 * d.coef[k];
        }
    }
    for (int dd = 0; dd < ndim; dd++)
        if (m.dimmask & (1u << dd)) d.dims[d.nd++] = (unsigned char)dd;
    if (d.nd == 0) return false;
    if (d.has_white) {
        if (f[pos_white].dimmask != m.dimmask) return false;
        d.white_raw = (d.scale != 1.0 || d.loc != 0.0);
    }
    return true;
}

template <int KIND>
static int launch_fast(cudaStream_t st, const FastDesc &d, const double *x, int64_t ldx, int64_t n, const double *y,
                       int64_t ldy, int64_t m, double *K, int64_t ldk, bool sym) {
    size_t smem = (size_t)(2 + (d.white_raw ? 2 : 0)) * d.nd * FT * sizeof(double) + (sym ? FT * (FT + 1) * 8 : 0);
    int64_t tm = (n + FT - 1) / FT, tn = (m + FT - 1) / FT;
    int64_t grid = sym ? tm * (tm + 1) / 2 : tm * tn;
    if (grid > 2147483647LL) return LGP_ERR_UNSUPPORTED;
    int vec_ok = ((ldk & 1) == 0) && ((reinterpret_cast<uintptr_t>(K) & 15) == 0);
    if (sym) {
        if (smem_opt_in(gram_fast_kernel<KIND, true>, smem)) return LGP_ERR_CUDA;
        gram_fast_kernel<KIND, true><<<(unsigned)grid, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, K, ldk, vec_ok,
                                                                             (int)tn);
    } else {
        if (smem_opt_in(gram_fast_kernel<KIND, false>, smem)) return LGP_ERR_CUDA;
        gram_fast_kernel<KIND, false><<<(unsigned)grid, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, K, ldk, vec_ok,
                                                                              (int)tn);
    }
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

template <int KIND, int P>
static int launch_fast2(cudaStream_t st, const FastDesc &d, const double *x, int64_t ldx, int64_t n, const double *y,
                        int64_t ldy, int64_t m, double *K, int64_t ldk, bool sym) {
    size_t smem = 1024 * FTabRep<KIND>::value + (KIND == LGP_K_CAUCHY ? 2048 : 0) + (size_t)(2 + (d.white_raw ? 2 : 0)) * d.nd * FT * sizeof(double) +
                  (sym ? FT * F2_TS * 8 : 0);
    int64_t tm = (n + FT - 1) / FT, tn = (m + FT - 1) / FT;
    int64_t grid = sym ? tm * (tm + 1) / 2 : tm * tn;
    if (grid > 2147483647LL) return LGP_ERR_UNSUPPORTED;
    int vec_ok = ((ldk & 1) == 0) && ((reinterpret_cast<uintptr_t>(K) & 15) == 0);
    // version 3 stages both the tile and its mirror image and no raw coordinates; it needs 3 CTAs per SM to pay off
    const size_t smem3 = smem + (size_t)FT * F2_TS * 8 -
                         ((d.white_raw && FTabRep<KIND>::value != 1) ? (size_t)2 * d.nd * FT * sizeof(double) : 0);
    if (sym && smem3 <= 77400) {
        smem = smem3;
        // 3 CTAs per SM (80 registers): measured 0.745 ms against 0.846 ms with 2 CTAs x 126 registers (Matern-5/2, n = 20k);
        // many-field inputs that need more shared memory go through version 2
        static DeviceOnce once;
        const int dev = current_device();
        if (dev < 0) return LGP_ERR_CUDA;
        if (!once.done(dev)) {
            if (cudaFuncSetAttribute(gram_fast3_kernel<KIND, P, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     77400) != cudaSuccess)
                return LGP_ERR_CUDA;
            once.set(dev);
        }
        gram_fast3_kernel<KIND, P, false><<<(unsigned)grid, G_THREADS, smem, st>>>(d, x, ldx, n, K, ldk, vec_ok,
                                                                                   GramPrep{nullptr, nullptr, 0});
    } else if (sym) {
        if (smem_opt_in(gram_fast2_kernel<KIND, P, true>, smem)) return LGP_ERR_CUDA;
        gram_fast2_kernel<KIND, P, true><<<(unsigned)grid, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, K, ldk,
                                                                                 vec_ok, (int)tn);
    } else {
        if (smem_opt_in(gram_fast2_kernel<KIND, P, false>, smem)) return LGP_ERR_CUDA;
        gram_fast2_kernel<KIND, P, false><<<(unsigned)grid, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, K, ldk,
                                                                                  vec_ok, (int)tn);
    }
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}


// ------------------------------------------------------------------------------------------------
// Gram build fused with the equilibration pass of the factorisation (lgp_gram_iso_prepare)
// ------------------------------------------------------------------------------------------------
// Diagonal value of the kernel matrix (the same for every point: stationary core at r2 = 0, plus White and Constant),
// rounded like the entries the Gram kernel writes there, and s = 2^rint(log2(d)/2) (reference diag_scale_pow2,
// _decomp.py:356-361): S / SINV of aux filled uniformly (1 for the padding rows), the 16 scalars zeroed.
template <int KIND>
__global__ void gram_prep_diag_kernel(const __grid_constant__ FastDesc d, int n, int npad, double *__restrict__ aux) {
    double v = __dmul_rn(d.amp, fast_core<KIND>(d, 0.0));
    if (d.has_white) v = __dadd_rn(v, d.amp_white);
    if (d.has_const) v = __dadd_rn(v, d.amp_const);
    double s = 1.0;
    if (v != 0.0) s = exp2(rint(0.5 * log2(v)));
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < npad; i += gridDim.x * blockDim.x) {
        aux[LGP_AUX_S(npad) + i] = (i < n) ? s : 1.0;
        aux[LGP_AUX_SINV(npad) + i] = (i < n) ? 1.0 / s : 1.0;
        if (i < 16) aux[LGP_AUX_SCALARS(npad) + i] = 0.0;
    }
}

// max_i sum_slots rowpart[slot][i] over the rows i < n, slots in a fixed order -> scalars[0] (the Gershgorin bound)
__global__ void __launch_bounds__(256) gram_prep_rowmax_kernel(const double *__restrict__ rowpart, int64_t npad, int slots,
                                                               int n, double *__restrict__ aux) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double sum = 0.0;
    if (i < n)
        for (int s = 0; s < slots; s++) sum += rowpart[(int64_t)s * npad + i];
    // max over the warp with NaN winning (a NaN row sum must reach eps like in the reference)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double u = __shfl_xor_sync(0xffffffffu, sum, o);
        sum = (u > sum || u != u) ? u : sum;
    }
    if ((threadIdx.x & 31) == 0)
        atomicMax(reinterpret_cast<unsigned long long *>(aux + LGP_AUX_SCALARS(npad)),
                  (unsigned long long)__double_as_longlong(sum));
}

// dynamic shared memory of the fused kernel (tables, staged points, tile + mirror staging)
static size_t prepare_smem(const FastDesc &d) {
    const int tabrep = d.kind == LGP_K_EXPQUAD ? FTabRep<LGP_K_EXPQUAD>::value : 1;
    return 1024 * tabrep + (d.kind == LGP_K_CAUCHY ? 2048 : 0) +
           (size_t)(2 + ((d.white_raw && tabrep == 1) ? 2 : 0)) * d.nd * FT * sizeof(double) + (size_t)2 * FT * F2_TS * 8;
}
// Does the fused Gram -> equilibration build apply?  Fast family only; the diagonal must take the library (slow) path of
// the Gram kernel, which gram_prep_diag_kernel reproduces; three CTAs per SM must fit.
static bool prepare_supported(const FastDesc &d) {
    const bool family = d.kind == LGP_K_EXPQUAD || (d.kind == LGP_K_MATERNP && d.p >= 0 && d.p <= 3) ||
                        (d.kind == LGP_K_CAUCHY && d.cauchy_fast);
    if (!family) return false;
    if (!(d.has_white || d.kind == LGP_K_EXPQUAD || d.kind == LGP_K_CAUCHY || d.par0 == 0.0)) return false;
    return prepare_smem(d) <= 77400;
}

template <int KIND, int P>
static int launch_prepare(cudaStream_t st, const FastDesc &d, const double *x, int64_t ldx, int64_t n, double *W,
                          int64_t ldw, double *aux, double *work) {
    const int64_t npad = lgp_chol_npad(n);
    if (!prepare_supported(d)) return LGP_ERR_UNSUPPORTED;
    const size_t smem = prepare_smem(d);
    static DeviceOnce once;
    const int dev = current_device();
    if (dev < 0) return LGP_ERR_CUDA;
    if (!once.done(dev)) {
        if (cudaFuncSetAttribute(gram_fast3_kernel<KIND, P, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 77400) !=
            cudaSuccess)
            return LGP_ERR_CUDA;
        once.set(dev);
    }
    const int64_t t = npad / FT, grid = t * (t + 1) / 2;
    if (grid > 2147483647LL) return LGP_ERR_UNSUPPORTED;
    gram_prep_diag_kernel<KIND><<<(unsigned)((npad + 255) / 256), 256, 0, st>>>(d, (int)n, (int)npad, aux);
    LGP_CUDA_CHECK_LAUNCH();
    gram_fast3_kernel<KIND, P, true><<<(unsigned)grid, G_THREADS, smem, st>>>(
        d, x, ldx, n, W, ldw, 1, GramPrep{aux + LGP_AUX_SINV(npad), work, npad});
    LGP_CUDA_CHECK_LAUNCH();
    gram_prep_rowmax_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(work, npad, (int)t, (int)n, aux);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

}  // namespace lgp

extern "C" {

int64_t lgp_gram_prepare_work_doubles(int64_t n) {
    const int64_t npad = lgp_chol_npad(n);
    return (npad / lgp::FT) * npad;
}

int lgp_gram_iso_prepare_supported(const lgp_factor_t *factors, int nfactors, int ndim) {
    using namespace lgp;
    if (!factors || !(nfactors >= 1 && nfactors <= LGP_MAX_FACTORS && ndim >= 1 && ndim <= LGP_MAX_DIMS)) return 0;
    FastDesc fd;
    return (build_fast(factors, nfactors, ndim, fd) && prepare_supported(fd)) ? 1 : 0;
}

int lgp_gram_iso_prepare(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                         int64_t ldx, int64_t n, double *W, int64_t ldw, double *aux, double *work) {
    using namespace lgp;
    if (!factors || !x || !W || !aux || !work || n < 1 || n > (1 << 30)) return LGP_ERR_BADARG;
    const int64_t npad = lgp_chol_npad(n);
    if (ldw < npad) return LGP_ERR_BADARG;
    if ((ldw & 1) || (reinterpret_cast<uintptr_t>(W) & 15) || (reinterpret_cast<uintptr_t>(aux) & 15)) return LGP_ERR_ALIGN;
    if (!(nfactors >= 1 && nfactors <= LGP_MAX_FACTORS && ndim >= 1 && ndim <= LGP_MAX_DIMS)) return LGP_ERR_UNSUPPORTED;
    FastDesc fd;
    if (!build_fast(factors, nfactors, ndim, fd)) return LGP_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (fd.kind == LGP_K_EXPQUAD) return launch_prepare<LGP_K_EXPQUAD, 0>(st, fd, x, ldx, n, W, ldw, aux, work);
    if (fd.kind == LGP_K_MATERNP && fd.p == 0) return launch_prepare<LGP_K_MATERNP, 0>(st, fd, x, ldx, n, W, ldw, aux, work);
    if (fd.kind == LGP_K_MATERNP && fd.p == 1) return launch_prepare<LGP_K_MATERNP, 1>(st, fd, x, ldx, n, W, ldw, aux, work);
    if (fd.kind == LGP_K_MATERNP && fd.p == 2) return launch_prepare<LGP_K_MATERNP, 2>(st, fd, x, ldx, n, W, ldw, aux, work);
    if (fd.kind == LGP_K_MATERNP && fd.p == 3) return launch_prepare<LGP_K_MATERNP, 3>(st, fd, x, ldx, n, W, ldw, aux, work);
    if (fd.kind == LGP_K_CAUCHY && fd.cauchy_fast) return launch_prepare<LGP_K_CAUCHY, 0>(st, fd, x, ldx, n, W, ldw, aux, work);
    return LGP_ERR_UNSUPPORTED;
}

}  // extern "C"

namespace lgp {

__global__ void zero_kernel(double *p, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = 0.0;
}


// ---- launchers of the general kernels: numeric descriptor fields from the host struct (devpar == nullptr) or from
// device memory (the *_dev entry points)

static int gram_general(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *devpar,
                        const double *x, int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, double *K_out,
                        int64_t ldk) {
    GramDesc d;
    int rc = build_desc(factors, nfactors, ndim, d);
    if (rc) return rc;
    const size_t smem = (size_t)2 * d.nslots * GT * sizeof(double);
    dim3 grid((unsigned)((m + GT - 1) / GT), (unsigned)((n + GT - 1) / GT));
    if (grid.y > 65535) return LGP_ERR_UNSUPPORTED;
    const int vec_ok = ((ldk & 1) == 0) && ((reinterpret_cast<uintptr_t>(K_out) & 15) == 0);
    cudaStream_t st = (cudaStream_t)stream;
    if (devpar) {
        if (smem_opt_in(gram_iso_kernel<true>, smem)) return LGP_ERR_CUDA;
        gram_iso_kernel<true><<<grid, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, K_out, ldk, vec_ok, devpar);
    } else {
        if (smem_opt_in(gram_iso_kernel<false>, smem)) return LGP_ERR_CUDA;
        gram_iso_kernel<false><<<grid, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, K_out, ldk, vec_ok, nullptr);
    }
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

static int vjp_general(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *devpar,
                       const double *x, int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *G,
                       int64_t ldg, const double *b, int symlower, double *out) {
    GramDesc d;
    int rc = build_desc(factors, nfactors, ndim, d);
    if (rc) return rc;
    const size_t smem = (size_t)2 * d.nslots * GT * sizeof(double);
    cudaStream_t st = (cudaStream_t)stream;
    zero_kernel<<<1, 32, 0, st>>>(out, 3 * nfactors);
    LGP_CUDA_CHECK_LAUNCH();
    const int64_t tm = (n + GT - 1) / GT, tn = (m + GT - 1) / GT;
    const int64_t nblk = symlower ? tm * (tm + 1) / 2 : tm * tn;
    if (nblk > 2147483647LL) return LGP_ERR_UNSUPPORTED;
    if (devpar) {
        if (smem_opt_in(gram_iso_vjp_kernel<true>, smem)) return LGP_ERR_CUDA;
        gram_iso_vjp_kernel<true><<<(unsigned)nblk, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, G, ldg, b, symlower,
                                                                           (int)tn, out, devpar);
    } else {
        if (smem_opt_in(gram_iso_vjp_kernel<false>, smem)) return LGP_ERR_CUDA;
        gram_iso_vjp_kernel<false><<<(unsigned)nblk, G_THREADS, smem, st>>>(d, x, ldx, n, y, ldy, m, G, ldg, b, symlower,
                                                                            (int)tn, out, nullptr);
    }
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

static int jvp_general(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *devpar,
                       const double *tangent_host, const double *tangent_dev, const double *x, int64_t ldx, int64_t n,
                       const double *y, int64_t ldy, int64_t m, double *D_out, int64_t ldd) {
    GramDesc d;
    int rc = build_desc(factors, nfactors, ndim, d);
    if (rc) return rc;
    GramTangent tan;
    memset(&tan, 0, sizeof(tan));
    if (tangent_host)
        for (int i = 0; i < 3 * nfactors; i++) tan.t[i] = tangent_host[i];
    const size_t smem = (size_t)2 * d.nslots * GT * sizeof(double);
    dim3 grid((unsigned)((m + GT - 1) / GT), (unsigned)((n + GT - 1) / GT));
    if (grid.y > 65535) return LGP_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (devpar) {
        if (smem_opt_in(gram_iso_jvp_kernel<true>, smem)) return LGP_ERR_CUDA;
        gram_iso_jvp_kernel<true><<<grid, G_THREADS, smem, st>>>(d, tan, x, ldx, n, y, ldy, m, D_out, ldd, devpar,
                                                                 tangent_dev);
    } else {
        if (smem_opt_in(gram_iso_jvp_kernel<false>, smem)) return LGP_ERR_CUDA;
        gram_iso_jvp_kernel<false><<<grid, G_THREADS, smem, st>>>(d, tan, x, ldx, n, y, ldy, m, D_out, ldd, nullptr,
                                                                  nullptr);
    }
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

}  // namespace lgp

using namespace lgp;

extern "C" {

int lgp_gram_iso(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                 int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, double *K_out, int64_t ldk,
                 int flags) {
    if (!factors || !K_out || n < 0 || m < 0) return LGP_ERR_BADARG;
    if (n == 0 || m == 0) return LGP_OK;
    if (ndim > 0 && (!x || !y)) return LGP_ERR_BADARG;
    if (ldk < m) return LGP_ERR_BADARG;
    if (nfactors >= 1 && nfactors <= LGP_MAX_FACTORS && ndim >= 1 && ndim <= LGP_MAX_DIMS &&
        !(flags & LGP_GRAM_GENERAL)) {
        FastDesc fd;
        if (build_fast(factors, nfactors, ndim, fd)) {
            const bool sym = (flags & LGP_GRAM_SYMMETRIC) && x == y && n == m && ldx == ldy;
            cudaStream_t st = (cudaStream_t)stream;
            if (!(flags & LGP_GRAM_LIBM)) {
                if (fd.kind == LGP_K_EXPQUAD)
                    return launch_fast2<LGP_K_EXPQUAD, 0>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
                if (fd.kind == LGP_K_MATERNP && fd.p == 0)
                    return launch_fast2<LGP_K_MATERNP, 0>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
                if (fd.kind == LGP_K_MATERNP && fd.p == 1)
                    return launch_fast2<LGP_K_MATERNP, 1>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
                if (fd.kind == LGP_K_MATERNP && fd.p == 2)
                    return launch_fast2<LGP_K_MATERNP, 2>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
                if (fd.kind == LGP_K_MATERNP && fd.p == 3)
                    return launch_fast2<LGP_K_MATERNP, 3>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
                if (fd.kind == LGP_K_CAUCHY && fd.cauchy_fast)
                    return launch_fast2<LGP_K_CAUCHY, 0>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
            }
            if (fd.kind == LGP_K_EXPQUAD) return launch_fast<LGP_K_EXPQUAD>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
            if (fd.kind == LGP_K_MATERNP) return launch_fast<LGP_K_MATERNP>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
            if (fd.kind == LGP_K_MATERN) return launch_fast<LGP_K_MATERN>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
            return launch_fast<LGP_K_CAUCHY>(st, fd, x, ldx, n, y, ldy, m, K_out, ldk, sym);
        }
    }
    return gram_general(stream, factors, nfactors, ndim, nullptr, x, ldx, n, y, ldy, m, K_out, ldk);
}

int lgp_gram_iso_dev(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *devpar,
                     const double *x, int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, double *K_out,
                     int64_t ldk, int flags) {
    (void)flags;
    if (!factors || !devpar || !K_out || n < 0 || m < 0) return LGP_ERR_BADARG;
    if (n == 0 || m == 0) return LGP_OK;
    if (ndim > 0 && (!x || !y)) return LGP_ERR_BADARG;
    if (ldk < m) return LGP_ERR_BADARG;
    return gram_general(stream, factors, nfactors, ndim, devpar, x, ldx, n, y, ldy, m, K_out, ldk);
}

int lgp_gram_iso_vjp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                     int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *G, int64_t ldg,
                     const double *b, int symlower, double *out) {
    if (!factors || !G || !out || n < 1 || m < 1) return LGP_ERR_BADARG;
    if (symlower && (n != m)) return LGP_ERR_BADARG;
    if (symlower && x == y && ldx == ldy && nfactors <= 3 && ndim >= 1 && ndim <= LGP_MAX_DIMS) {
        FastDesc fd;
        if (build_fast(factors, nfactors, ndim, fd)) {
            cudaStream_t st = (cudaStream_t)stream;
            int pos_white = -1, pos_const = -1;
            for (int i = 0; i < nfactors; i++) {
                if (factors[i].kind == LGP_K_WHITE) pos_white = i;
                if (factors[i].kind == LGP_K_CONSTANT) pos_const = i;
            }
            // the 5 partial sums live in out[0..4] only if nfactors >= 2; use a scratch tail otherwise is not
            // available (no allocation here), so accumulate in place when the layouts coincide
            double *tmp = out + 3 * nfactors;  // caller provides 3*nfactors + 8 doubles (see header)
            zero_kernel<<<1, 32, 0, st>>>(tmp, 8);
            LGP_CUDA_CHECK_LAUNCH();
            size_t smem = (size_t)(2 + (fd.white_raw ? 2 : 0)) * fd.nd * FT * sizeof(double);
            int64_t t = (n + FT - 1) / FT;
            int64_t nblk = t * (t + 1) / 2;
            if (nblk > 2147483647LL) return LGP_ERR_UNSUPPORTED;
#define LGP_VJP_LAUNCH(KIND, P)                                                                       \
    do {                                                                                              \
        if (smem_opt_in(gram_fast_vjp_kernel<KIND, P>, smem)) return LGP_ERR_CUDA;                     \
        gram_fast_vjp_kernel<KIND, P><<<(unsigned)nblk, G_THREADS, smem, st>>>(fd, x, ldx, n, G, ldg, b, tmp); \
    } while (0)
            if (fd.kind == LGP_K_EXPQUAD)
                LGP_VJP_LAUNCH(LGP_K_EXPQUAD, 0);
            else if (fd.kind == LGP_K_MATERNP && fd.p == 0)
                LGP_VJP_LAUNCH(LGP_K_MATERNP, 0);
            else if (fd.kind == LGP_K_MATERNP && fd.p == 1)
                LGP_VJP_LAUNCH(LGP_K_MATERNP, 1);
            else if (fd.kind == LGP_K_MATERNP && fd.p == 2)
                LGP_VJP_LAUNCH(LGP_K_MATERNP, 2);
            else if (fd.kind == LGP_K_MATERNP && fd.p == 3)
                LGP_VJP_LAUNCH(LGP_K_MATERNP, 3);
            else if (fd.kind == LGP_K_MATERNP)
                LGP_VJP_LAUNCH(LGP_K_MATERNP, -1);
            else if (fd.kind == LGP_K_MATERN)
                LGP_VJP_LAUNCH(LGP_K_MATERN, -1);
            else
                LGP_VJP_LAUNCH(LGP_K_CAUCHY, -1);
#undef LGP_VJP_LAUNCH
            LGP_CUDA_CHECK_LAUNCH();
            fast_vjp_scatter_kernel<<<1, 32, 0, st>>>(tmp, out, nfactors, pos_white, pos_const);
            LGP_CUDA_CHECK_LAUNCH();
            return LGP_OK;
        }
    }
    return vjp_general(stream, factors, nfactors, ndim, nullptr, x, ldx, n, y, ldy, m, G, ldg, b, symlower, out);
}

int lgp_gram_iso_vjp_dev(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *devpar,
                         const double *x, int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m,
                         const double *G, int64_t ldg, const double *b, int symlower, double *out) {
    if (!factors || !devpar || !G || !out || n < 1 || m < 1) return LGP_ERR_BADARG;
    if (symlower && (n != m)) return LGP_ERR_BADARG;
    return vjp_general(stream, factors, nfactors, ndim, devpar, x, ldx, n, y, ldy, m, G, ldg, b, symlower, out);
}

int lgp_gram_iso_jvp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                     int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *tangent,
                     double *D_out, int64_t ldd) {
    if (!factors || !tangent || !D_out || n < 1 || m < 1 || ldd < m) return LGP_ERR_BADARG;
    return jvp_general(stream, factors, nfactors, ndim, nullptr, tangent, nullptr, x, ldx, n, y, ldy, m, D_out, ldd);
}

int lgp_gram_iso_jvp_dev(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *devpar,
                         const double *x, int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m,
                         const double *tangent_dev, double *D_out, int64_t ldd) {
    if (!factors || !devpar || !tangent_dev || !D_out || n < 1 || m < 1 || ldd < m) return LGP_ERR_BADARG;
    return jvp_general(stream, factors, nfactors, ndim, devpar, nullptr, tangent_dev, x, ldx, n, y, ldy, m, D_out, ldd);
}

int lgp_frob_dot(lgp_stream_t stream, const double *A, int64_t lda, const double *B, int64_t ldb, int64_t rows,
                 int64_t cols, double *out) {
    if (!A || !B || !out || rows < 0 || cols < 0 || lda < cols || ldb < cols) return LGP_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    zero_kernel<<<1, 32, 0, st>>>(out, 1);
    LGP_CUDA_CHECK_LAUNCH();
    if (rows == 0 || cols == 0) return LGP_OK;
    const unsigned grid = (unsigned)(rows < 148 * 8 ? rows : 148 * 8);
    frob_dot_kernel<<<grid, 256, 0, st>>>(A, lda, B, ldb, rows, cols, out);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

}  // extern "C"
