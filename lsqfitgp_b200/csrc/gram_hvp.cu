// Second-order contraction of the Gram build: the derivative, along a tangent of the hyperparameters, of the reverse-mode
// contraction of gram_iso_vjp_kernel (gram_iso.cu), which the second derivatives of the marginal likelihood need:
//   out[3f+k] = sum_ij G_ij d/dtheta_{f,k} ( sum_{g,l} tangent[3g+l] dK_ij/dtheta_{g,l} ),
//   theta_{f,.} = (amp_f, log scale_f, par1_f).
// Same staging, tiles and G modes as the VJP.  Inside a term P = prod_h v_h, v_h = amp_h c_h, the derivative along the
// tangent is D P = sum_h dv_h Q_h with Q_h = prod_{h' != h} v_h'; its derivative with respect to theta_{f,k} is
//   d_k(dv_f) Q_f + d_k(v_f) D(Q_f),
// where Q_f and D(Q_f) are accumulated over the other factors of the term (no division by factor values: a factor that
// vanishes is harmless, and the amplitude output is the product rule with amp_f left out, not D P / amp_f).
#include <math.h>
#include <string.h>

#include "../../include/lgp_b200.h"
#include "common.cuh"
#include "internal.h"
#include "gram_desc.cuh"
#include "hess_core.cuh"

namespace lgp {

__global__ void __launch_bounds__(G_THREADS) gram_iso_hvp_kernel(const __grid_constant__ GramDesc d,
                                                                 const __grid_constant__ GramTangent tan,
                                                                 const double *__restrict__ x, int64_t ldx, int64_t n,
                                                                 const double *__restrict__ y, int64_t ldy, int64_t m,
                                                                 const double *__restrict__ G, int64_t ldg,
                                                                 const double *__restrict__ bvec, int symlower,
                                                                 int tiles_n, double *__restrict__ out) {
    extern __shared__ __align__(16) double gsm[];
    double *su = gsm;
    double *sv = gsm + (size_t)d.nslots * GT;
    // per-thread accumulators in shared memory, acc[k * G_THREADS + tid]: in registers they would spill next to the
    // per-factor state of one entry
    double *acc = sv + (size_t)d.nslots * GT;
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
    stage_points(d, su, x, ldx, n, i0, false, tid);
    stage_points(d, sv, y, ldy, m, j0, true, tid);
    __syncthreads();

    for (int k = 0; k < 3 * d.nfactors; k++) acc[k * G_THREADS + tid] = 0.0;

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
            // per factor: value v, derivative dv along the tangent, first derivatives d[k] of v and the derivatives
            // e[k] = d_k(dv) of dv
            double v[LGP_MAX_FACTORS], dv[LGP_MAX_FACTORS], dk[LGP_MAX_FACTORS][3], ek[LGP_MAX_FACTORS][3];
#pragma unroll
            for (int f = 0; f < LGP_MAX_FACTORS; f++) {
                if (f < d.nfactors) {
                    double u = 0.0;
                    for (int s = d.slot0[f]; s < d.slot0[f] + d.nslot[f]; s++) {
                        const double df = su[s * GT + ty + 16 * a] - sv[s * GT + cc];
                        u += df * df;
                    }
                    double h[6];
                    hess_coefs(d.kind[f], d.ipar[f], d.par0[f], d.par1[f], d.mat[f], u, h);
                    const double A = d.amp[f];
                    const double t0 = tan.t[3 * f], t1 = tan.t[3 * f + 1], t2 = tan.t[3 * f + 2];
                    v[f] = A * h[0];
                    dk[f][0] = h[0];
                    dk[f][1] = A * h[1];
                    dk[f][2] = A * h[3];
                    dv[f] = t0 * dk[f][0] + t1 * dk[f][1] + t2 * dk[f][2];
                    ek[f][0] = t1 * h[1] + t2 * h[3];
                    ek[f][1] = t0 * h[1] + A * (t1 * h[2] + t2 * h[4]);
                    ek[f][2] = t0 * h[3] + A * (t1 * h[4] + t2 * h[5]);
                }
            }
#pragma unroll
            for (int f = 0; f < LGP_MAX_FACTORS; f++) {
                if (f < d.nfactors) {
                    double q = 1.0, dq = 0.0;  // Q_f and D(Q_f) over the other factors of the term
#pragma unroll
                    for (int h = 0; h < LGP_MAX_FACTORS; h++)
                        if (h < d.nfactors && h != f && d.term[h] == d.term[f]) {
                            dq = dq * v[h] + q * dv[h];
                            q *= v[h];
                        }
                    const double gq = g * q, gdq = g * dq;
#pragma unroll
                    for (int k = 0; k < 3; k++) acc[(3 * f + k) * G_THREADS + tid] += ek[f][k] * gq + dk[f][k] * gdq;
                }
            }
        }
    }
    const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
    for (int k = 0; k < 3 * LGP_MAX_FACTORS; k++) {
        double s = warp_sum(k < 3 * d.nfactors ? acc[k * G_THREADS + tid] : 0.0);
        if (lane == 0) red[warp][k] = s;
    }
    __syncthreads();
    if (tid < 3 * d.nfactors) {
        double s = 0.0;
        for (int w = 0; w < G_THREADS / 32; w++) s += red[w][tid];
        atomicAdd(out + tid, s);
    }
}

}  // namespace lgp

using namespace lgp;

extern "C" {

int lgp_gram_iso_hvp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                     int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *G, int64_t ldg,
                     const double *b, int symlower, const double *tangent, double *out) {
    if (!factors || !G || !tangent || !out || n < 1 || m < 1) return LGP_ERR_BADARG;
    if (symlower && (n != m)) return LGP_ERR_BADARG;
    GramDesc d;
    int rc = build_desc(factors, nfactors, ndim, d);
    if (rc) return rc;
    GramTangent tan;
    memset(&tan, 0, sizeof(tan));
    for (int i = 0; i < 3 * nfactors; i++) tan.t[i] = tangent[i];
    const size_t smem = ((size_t)2 * d.nslots * GT + (size_t)3 * nfactors * G_THREADS) * sizeof(double);
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(out, 0, sizeof(double) * 3 * nfactors, st) != cudaSuccess) return LGP_ERR_CUDA;
    const int64_t tm = (n + GT - 1) / GT, tn = (m + GT - 1) / GT;
    const int64_t nblk = symlower ? tm * (tm + 1) / 2 : tm * tn;
    if (nblk > 2147483647LL) return LGP_ERR_UNSUPPORTED;
    if (smem_opt_in(gram_iso_hvp_kernel, smem)) return LGP_ERR_CUDA;
    gram_iso_hvp_kernel<<<(unsigned)nblk, G_THREADS, smem, st>>>(d, tan, x, ldx, n, y, ldy, m, G, ldg, b, symlower,
                                                                 (int)tn, out);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

}  // extern "C"
