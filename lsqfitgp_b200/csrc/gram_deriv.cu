// Derivative blocks of the Gram build: cov(d_a f(x), f(y)), cov(f(x), d_b f(y)) and cov(d_a f(x), d_b f(y)) for
// first derivatives with respect to one field a of x and / or one field b of y, with the VJP and JVP of these blocks
// with respect to the hyperparameters.  Replaces the reference's jax derivatives of the kernel core
// (src/lsqfitgp/_Kernel/_crosskernel.py linop('diff'), _Kernel/_ops.py:200-290, _GP/_elements.py:190-242).
//
// Every factor f of a term yields a hyper-dual number (v, gx, gy, h) of its value and its derivatives,
// with u = sum_{d in dims_f} D_d^2, D_d = (x_d - loc_x)/scale_x - (y_d - loc_y)/scale_y:
//   v = c(u),  gx = 2 c'(u) D_a / sx,  gy = -2 c'(u) D_b / sy,  h = -(4 c''(u) D_a D_b + 2 c'(u) delta_ab) / (sx sy)
// (D_a = 0 and delta_ab = 0 when a is not in dims_f), and a term is their product under the product rule, which has
// no divisions, so zero-valued factors are harmless.  The hyperparameter derivatives (amp, log scale, Cauchy beta)
// differentiate these four numbers once more (d u / d log s = -2u, d D / d log s = -D); they need c'''.
// Tiling and staging are those of gram_iso_kernel (gram_desc.cuh): 64 x 64 tiles, 256 threads, 4 x 4 entries each.
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../include/lgp_b200.h"
#include "common.cuh"
#include "internal.h"
#include "gram_desc.cuh"
#include "deriv_core.cuh"

namespace lgp {

// per factor: slot of the differentiated field of x (sa) and of y (sb) among the factor's slots, -1 if not there;
// sel: bit 0 = derivative on x, bit 1 = derivative on y (which component of the hyper-dual product is the block)
struct DerivSel {
    signed char sa[LGP_MAX_FACTORS], sb[LGP_MAX_FACTORS];
    int sel;
};

struct HD {
    double v, x, y, xy;
};

// product rule; explicitly rounded, and the two mixed products are added to each other first, so that swapping x and
// y (v, x, y, xy) -> (v, y, x, xy) in both operands swaps the result exactly (symmetric blocks are exactly symmetric)
__device__ __forceinline__ HD hd_mul(const HD &a, const HD &b) {
    HD r;
    r.v = __dmul_rn(a.v, b.v);
    r.x = __dadd_rn(__dmul_rn(a.x, b.v), __dmul_rn(a.v, b.x));
    r.y = __dadd_rn(__dmul_rn(a.y, b.v), __dmul_rn(a.v, b.y));
    r.xy = __dadd_rn(__dadd_rn(__dmul_rn(a.xy, b.v), __dadd_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x))),
                     __dmul_rn(a.v, b.xy));
    return r;
}

__device__ __forceinline__ double hd_sel(const HD &a, int sel) { return sel == 1 ? a.x : sel == 2 ? a.y : a.xy; }

__device__ __forceinline__ HD hd_axpy(double s, const HD &a, const HD &b) {  // s a + b
    return HD{s * a.v + b.v, s * a.x + b.x, s * a.y + b.y, s * a.xy + b.xy};
}

// hyper-dual value q of factor f (without amp) at the pair (r of the x tile, cc of the y tile); DOTS: also its
// derivatives ql along log(scale) (both scales together) and qb along par1 (Cauchy beta)
template <bool DOTS>
__device__ __forceinline__ void factor_hd(const GramDesc &d, const DerivSel &ds, int f, const double *su,
                                          const double *sv, int r, int cc, HD &q, HD &ql, HD &qb) {
    double u = 0.0, A = 0.0, B = 0.0;
    const int s0 = d.slot0[f];
    for (int s = s0; s < s0 + d.nslot[f]; s++) {
        const double df = __dsub_rn(su[s * GT + r], sv[s * GT + cc]);
        const double sq = __dmul_rn(df, df);
        u = (s == s0) ? sq : __dadd_rn(u, sq);
        if (s - s0 == ds.sa[f]) A = df;
        if (s - s0 == ds.sb[f]) B = df;
    }
    const bool ina = ds.sa[f] >= 0, inb = ds.sb[f] >= 0;
    if (!ina && !inb) {
        // the factor does not depend on the differentiated fields: value only, any kind
        if (DOTS) {
            double val, dr2, dp1;
            core_derivs(d, f, u, val, dr2, dp1);
            q = HD{val, 0.0, 0.0, 0.0};
            ql = HD{dr2 * (-2.0 * u), 0.0, 0.0, 0.0};
            qb = HD{dp1, 0.0, 0.0, 0.0};
        } else {
            q = HD{core_value(d, f, u), 0.0, 0.0, 0.0};
        }
        return;
    }
    double c[4], db[3];
    deriv_coefs(d.kind[f], d.ipar[f], d.par0[f], d.par1[f], u, c, db);
    const double sx = d.scale_x[f], sy = d.scale_y[f], W = __dmul_rn(sx, sy);
    const bool delta = ina && inb && ds.sa[f] == ds.sb[f];
    const double c1A = __dmul_rn(c[1], A), c1B = __dmul_rn(c[1], B), AB = __dmul_rn(A, B);
    const double t2 = mul0(c[2], AB);
    const double dl = delta ? c[1] : 0.0;
    q.v = c[0];
    q.x = __ddiv_rn(__dmul_rn(2.0, c1A), sx);
    q.y = -__ddiv_rn(__dmul_rn(2.0, c1B), sy);
    q.xy = -__ddiv_rn(__dadd_rn(__dmul_rn(4.0, t2), __dmul_rn(2.0, dl)), W);
    if (DOTS) {
        ql.v = c[1] * (-2.0 * u);
        ql.x = -4.0 * (mul0(c[2], u * A) + c1A) / sx;
        ql.y = 4.0 * (mul0(c[2], u * B) + c1B) / sy;
        ql.xy = (8.0 * mul0(c[3], u * AB) + 8.0 * t2 + 4.0 * (delta ? mul0(c[2], u) : 0.0)) / W - 2.0 * q.xy;
        qb.v = db[0];
        qb.x = 2.0 * db[1] * A / sx;
        qb.y = -(2.0 * db[1] * B / sy);
        qb.xy = -(4.0 * db[2] * AB + 2.0 * (delta ? db[1] : 0.0)) / W;
    }
}

__device__ __forceinline__ void tile_of_block(int symlower, int tiles_n, int &tm, int &tn) {
    if (symlower) {
        const int b = blockIdx.x;
        tm = (int)((sqrt(8.0 * b + 1.0) - 1.0) * 0.5);
        while ((tm + 1) * (tm + 2) / 2 <= b) tm++;
        while (tm * (tm + 1) / 2 > b) tm--;
        tn = b - tm * (tm + 1) / 2;
    } else {
        tm = blockIdx.x / tiles_n;
        tn = blockIdx.x % tiles_n;
    }
}

// JVP = false: K[i][j] = the block; sym: x == y, the block is symmetric: tiles tm >= tn only, the strictly lower ones
// mirrored through shared memory.  JVP = true: D[i][j] = its derivative along tan (layout of gram_iso_jvp_kernel).
template <bool JVP>
__global__ void __launch_bounds__(G_THREADS) gram_deriv_kernel(const __grid_constant__ GramDesc d,
                                                               const __grid_constant__ DerivSel ds,
                                                               const __grid_constant__ GramTangent tan,
                                                               const double *__restrict__ x, int64_t ldx, int64_t n,
                                                               const double *__restrict__ y, int64_t ldy, int64_t m,
                                                               double *__restrict__ K, int64_t ldk, int sym, int tiles_n) {
    extern __shared__ __align__(16) double gsm[];
    double *su = gsm;
    double *sv = gsm + (size_t)d.nslots * GT;
    double *mir = sv + (size_t)d.nslots * GT;  // sym: GT x (GT + 1)
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    int tm, tn;
    tile_of_block(sym, tiles_n, tm, tn);
    const int64_t i0 = (int64_t)tm * GT, j0 = (int64_t)tn * GT;
    stage_points(d, su, x, ldx, n, i0, false, tid);
    stage_points(d, sv, y, ldy, m, j0, true, tid);
    __syncthreads();
    const bool mirror = sym && tm != tn;
#pragma unroll 1
    for (int a = 0; a < 4; a++) {
        const int r = ty + 16 * a;
        const int64_t i = i0 + r;
#pragma unroll 1
        for (int c = 0; c < 4; c++) {
            const int cc = tx + 16 * c;
            const int64_t j = j0 + cc;
            if (i >= n || j >= m) continue;
            double total = 0.0;
            bool first = true;
            int f = 0;
            while (f < d.nfactors) {
                const int term = d.term[f];
                HD P{1.0, 0.0, 0.0, 0.0}, Pd{0.0, 0.0, 0.0, 0.0};
                for (; f < d.nfactors && d.term[f] == term; f++) {
                    HD q, ql, qb;
                    factor_hd<JVP>(d, ds, f, su, sv, r, cc, q, ql, qb);
                    const double amp = d.amp[f];
                    const HD Q{__dmul_rn(amp, q.v), __dmul_rn(amp, q.x), __dmul_rn(amp, q.y), __dmul_rn(amp, q.xy)};
                    if (JVP) {
                        const double t0 = tan.t[3 * f], t1 = tan.t[3 * f + 1], t2 = tan.t[3 * f + 2];
                        const HD Qd = hd_axpy(t0, q, hd_axpy(amp * t1, ql, hd_axpy(amp * t2, qb, HD{0.0, 0.0, 0.0, 0.0})));
                        const HD a1 = hd_mul(Pd, Q), a2 = hd_mul(P, Qd);
                        Pd = HD{a1.v + a2.v, a1.x + a2.x, a1.y + a2.y, a1.xy + a2.xy};
                    }
                    P = hd_mul(P, Q);
                }
                const double tv = hd_sel(JVP ? Pd : P, ds.sel);
                total = first ? tv : __dadd_rn(total, tv);
                first = false;
            }
            K[i * ldk + j] = total;
            if (mirror) mir[cc * (GT + 1) + r] = total;
        }
    }
    if (mirror) {
        __syncthreads();
        for (int idx = tid; idx < GT * GT; idx += G_THREADS) {
            const int rr = idx / GT, c2 = idx % GT;
            const int64_t i = j0 + rr, j = i0 + c2;
            if (i < m && j < n) K[i * ldk + j] = mir[rr * (GT + 1) + c2];
        }
    }
}

// out[3f + k] += sum_ij G_ij d block_ij / d(param k of factor f), k = amp, log scale, par1 (dense G; the layout of
// gram_iso_vjp_kernel).  One sweep of the tile per factor f: the product of the other factors of its term is
// recomputed (kernels have few factors), so that only the three accumulators of f are live.
__global__ void __launch_bounds__(G_THREADS) gram_deriv_vjp_kernel(const __grid_constant__ GramDesc d,
                                                                   const __grid_constant__ DerivSel ds,
                                                                   const double *__restrict__ x, int64_t ldx, int64_t n,
                                                                   const double *__restrict__ y, int64_t ldy, int64_t m,
                                                                   const double *__restrict__ G, int64_t ldg,
                                                                   int tiles_n, double *__restrict__ out) {
    extern __shared__ __align__(16) double gsm[];
    double *su = gsm;
    double *sv = gsm + (size_t)d.nslots * GT;
    __shared__ double red[G_THREADS / 32][3];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int warp = tid >> 5, lane = tid & 31;
    int tm, tn;
    tile_of_block(0, tiles_n, tm, tn);
    const int64_t i0 = (int64_t)tm * GT, j0 = (int64_t)tn * GT;
    stage_points(d, su, x, ldx, n, i0, false, tid);
    stage_points(d, sv, y, ldy, m, j0, true, tid);
    __syncthreads();
    const int sel = ds.sel;
#pragma unroll 1
    for (int f = 0; f < d.nfactors; f++) {
        double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0;
        const double amp = d.amp[f];
#pragma unroll 1
        for (int a = 0; a < 4; a++) {
            const int r = ty + 16 * a;
            const int64_t i = i0 + r;
#pragma unroll 1
            for (int c = 0; c < 4; c++) {
                const int cc = tx + 16 * c;
                const int64_t j = j0 + cc;
                if (i >= n || j >= m) continue;
                const double g = G[i * ldg + j];
                HD O{1.0, 0.0, 0.0, 0.0};
                HD q, ql, qb;
#pragma unroll 1
                for (int h = 0; h < d.nfactors; h++) {
                    if (h == f || d.term[h] != d.term[f]) continue;
                    factor_hd<false>(d, ds, h, su, sv, r, cc, q, ql, qb);
                    const double ah = d.amp[h];
                    O = hd_mul(O, HD{ah * q.v, ah * q.x, ah * q.y, ah * q.xy});
                }
                factor_hd<true>(d, ds, f, su, sv, r, cc, q, ql, qb);
                acc0 += g * hd_sel(hd_mul(O, q), sel);
                acc1 += g * amp * hd_sel(hd_mul(O, ql), sel);
                acc2 += g * amp * hd_sel(hd_mul(O, qb), sel);
            }
        }
        acc0 = warp_sum(acc0);
        acc1 = warp_sum(acc1);
        acc2 = warp_sum(acc2);
        if (lane == 0) {
            red[warp][0] = acc0;
            red[warp][1] = acc1;
            red[warp][2] = acc2;
        }
        __syncthreads();
        if (tid < 3) {
            double v = 0.0;
            for (int w = 0; w < G_THREADS / 32; w++) v += red[w][tid];
            atomicAdd(out + 3 * f + tid, v);
        }
        __syncthreads();
    }
}

__global__ void deriv_zero_kernel(double *p, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = 0.0;
}

// descriptor + derivative selection; LGP_ERR_UNSUPPORTED when a factor that depends on a differentiated field cannot
// be differentiated by the kernels (White, Matern of real order, Cauchy alpha != 2, Maternp p = 0)
static int build_deriv(const lgp_factor_t *f, int nf, int ndim, int dx_field, int dy_field, GramDesc &d, DerivSel &ds) {
    if (dx_field < -1 || dy_field < -1 || dx_field >= ndim || dy_field >= ndim) return LGP_ERR_BADARG;
    if (dx_field < 0 && dy_field < 0) return LGP_ERR_BADARG;
    int rc = build_desc(f, nf, ndim, d);
    if (rc) return rc;
    memset(&ds, 0, sizeof(ds));
    ds.sel = (dx_field >= 0 ? 1 : 0) | (dy_field >= 0 ? 2 : 0);
    for (int i = 0; i < nf; i++) {
        ds.sa[i] = ds.sb[i] = -1;
        for (int s = d.slot0[i]; s < d.slot0[i] + d.nslot[i]; s++) {
            if (d.slot_dim[s] == dx_field) ds.sa[i] = (signed char)(s - d.slot0[i]);
            if (d.slot_dim[s] == dy_field) ds.sb[i] = (signed char)(s - d.slot0[i]);
        }
        if (ds.sa[i] < 0 && ds.sb[i] < 0) continue;
        const bool ok = f[i].kind == LGP_K_EXPQUAD || (f[i].kind == LGP_K_MATERNP && f[i].ipar >= 1) ||
                        (f[i].kind == LGP_K_CAUCHY && f[i].par0 == 2.0);
        if (!ok) return LGP_ERR_UNSUPPORTED;
    }
    return LGP_OK;
}

static int deriv_launch(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                        int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, int dx_field, int dy_field,
                        const double *tangent, double *K_out, int64_t ldk, int flags) {
    if (!factors || !K_out || n < 0 || m < 0) return LGP_ERR_BADARG;
    if (ndim < 1 || !x || !y || ldk < m) return LGP_ERR_BADARG;
    GramDesc d;
    DerivSel ds;
    int rc = build_deriv(factors, nfactors, ndim, dx_field, dy_field, d, ds);
    if (rc) return rc;
    if (n == 0 || m == 0) return LGP_OK;
    GramTangent tan;
    memset(&tan, 0, sizeof(tan));
    if (tangent)
        for (int i = 0; i < 3 * nfactors; i++) tan.t[i] = tangent[i];
    bool sym = false;
    if (!tangent && (flags & LGP_GRAM_SYMMETRIC) && x == y && n == m && ldx == ldy && dx_field == dy_field) {
        sym = true;
        for (int i = 0; i < nfactors; i++)
            sym = sym && factors[i].scale_x == factors[i].scale_y && factors[i].loc_x == factors[i].loc_y;
    }
    const int64_t tm = (n + GT - 1) / GT, tn = (m + GT - 1) / GT;
    const int64_t nblk = sym ? tm * (tm + 1) / 2 : tm * tn;
    if (nblk > 2147483647LL) return LGP_ERR_UNSUPPORTED;
    const size_t smem = (size_t)2 * d.nslots * GT * sizeof(double) + (sym ? (size_t)GT * (GT + 1) * sizeof(double) : 0);
    cudaStream_t st = (cudaStream_t)stream;
    if (tangent) {
        if (smem_opt_in(gram_deriv_kernel<true>, smem)) return LGP_ERR_CUDA;
        gram_deriv_kernel<true><<<(unsigned)nblk, G_THREADS, smem, st>>>(d, ds, tan, x, ldx, n, y, ldy, m, K_out, ldk, 0,
                                                                         (int)tn);
    } else {
        if (smem_opt_in(gram_deriv_kernel<false>, smem)) return LGP_ERR_CUDA;
        gram_deriv_kernel<false><<<(unsigned)nblk, G_THREADS, smem, st>>>(d, ds, tan, x, ldx, n, y, ldy, m, K_out, ldk,
                                                                          sym ? 1 : 0, (int)tn);
    }
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

}  // namespace lgp

using namespace lgp;

extern "C" {

int lgp_gram_iso_deriv(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                       int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, int dx_field, int dy_field,
                       double *K_out, int64_t ldk, int flags) {
    return deriv_launch(stream, factors, nfactors, ndim, x, ldx, n, y, ldy, m, dx_field, dy_field, nullptr, K_out, ldk,
                        flags);
}

int lgp_gram_iso_deriv_jvp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                           int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, int dx_field, int dy_field,
                           const double *tangent, double *D_out, int64_t ldd) {
    if (!tangent) return LGP_ERR_BADARG;
    return deriv_launch(stream, factors, nfactors, ndim, x, ldx, n, y, ldy, m, dx_field, dy_field, tangent, D_out, ldd, 0);
}

int lgp_gram_iso_deriv_vjp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                           int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, int dx_field, int dy_field,
                           const double *G, int64_t ldg, double *out) {
    if (!factors || !G || !out || n < 1 || m < 1 || ldg < m) return LGP_ERR_BADARG;
    if (ndim < 1 || !x || !y) return LGP_ERR_BADARG;
    GramDesc d;
    DerivSel ds;
    int rc = build_deriv(factors, nfactors, ndim, dx_field, dy_field, d, ds);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    deriv_zero_kernel<<<1, 32, 0, st>>>(out, 3 * nfactors);
    LGP_CUDA_CHECK_LAUNCH();
    const int64_t tm = (n + GT - 1) / GT, tn = (m + GT - 1) / GT;
    if (tm * tn > 2147483647LL) return LGP_ERR_UNSUPPORTED;
    const size_t smem = (size_t)2 * d.nslots * GT * sizeof(double);
    if (smem_opt_in(gram_deriv_vjp_kernel, smem)) return LGP_ERR_CUDA;
    gram_deriv_vjp_kernel<<<(unsigned)(tm * tn), G_THREADS, smem, st>>>(d, ds, x, ldx, n, y, ldy, m, G, ldg, (int)tn, out);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

}  // extern "C"
