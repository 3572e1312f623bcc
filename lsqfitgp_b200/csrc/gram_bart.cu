// BART prior correlation Gram matrix (fast path with <= 3 levels per bracket), its alpha / beta derivatives and the
// fused reverse-mode contraction.
//
// Reference: BART._correlation, src/lsqfitgp/_kernels/_bart.py:628-757 (closed forms for bracket widths 1, 2, 3 and the
// `repeat` scan), called through BART.correlation :415-455 which folds `reset` brackets into stages of rows of
// non-termination probabilities (done by the caller of this ABI); several stages are chained per pair, gamma of one
// stage being the per-pair output of the previous one (:447-455).  Point equality is tested exactly (any(ix != iy))
// instead of through fasthash64 (:675-678).  The per-pair arithmetic lives in bart_core.cuh (also built for the host).
#include <math.h>
#include <string.h>

#include "../../include/lgp_b200.h"
#include "bart_core.cuh"
#include "common.cuh"
#include "internal.h"

namespace lgp {

constexpr int BT = 64;           // CTA tile
constexpr int B_THREADS = 512;   // 16 x 32 threads, 2 (rows ty, ty + 32) x 4 (columns 2tx + 32b + {0,1}) pairs each
constexpr int B_RA = 2;           // rows per thread
constexpr int B_MAX_P = 64;
constexpr int B_MAX_ROWS = LGP_BART_MAX_ROWS;
constexpr int B_MAX_STAGES = LGP_BART_MAX_STAGES;
constexpr int B_CHUNK = 8;       // dimensions staged in shared memory at a time
constexpr int B_TSTRIDE = BT + 1;

enum { BMODE_VALUE = 0, BMODE_DERIV = 1, BMODE_VJP = 2 };

struct BartDesc {
    int p;  // number of active (w != 0) covariates after compaction
    int nstages;
    int stage_width[B_MAX_STAGES], stage_nrows[B_MAX_STAGES];
    int dim[B_MAX_P];  // original column index of each active covariate
    int n[B_MAX_P];    // split counts
    double w[B_MAX_P];
    double rows[B_MAX_ROWS][3];   // all stages, in evaluation order
    double drows[2][B_MAX_ROWS][3];  // d rows / d alpha, d rows / d beta
    double Wn, inv_Wn, gamma, amp;
};

struct BartIO {
    const double *psi;
    const int32_t *ix, *iy;
    int64_t ldx, ldy, n, m;
    double *K;     // value (VALUE, DERIV; may be null in DERIV)
    int64_t ldk;
    double *dKa, *dKb;  // amp * d corr / d alpha, d beta (DERIV; each may be null)
    int64_t ldd;
    const double *G;  // VJP: cotangent
    int64_t ldg;
    const double *b;  // VJP, symlower: G_ij := G_ij - b_i b_j (may be null)
    double *out;      // VJP: out[0] += sum G corr, out[1] += sum G amp dcorr/dalpha, out[2] += ... dbeta
    int sym;          // x == y: only tiles with tile row >= tile column are evaluated (mirrored / weighted)
    int vec_ok;
};

// shared-memory layout of one staged chunk: per side (x, y), per dimension, per point: the 5 doubles of BartPoint as
// structure-of-arrays [field][dim][point]; then the per-dimension constants
struct BartSmem {
    double pt[2][5][B_CHUNK][BT];
    BartDim dim[B_CHUNK];
};
constexpr size_t B_SMEM_BYTES = sizeof(BartSmem) > sizeof(double) * BT * B_TSTRIDE ? sizeof(BartSmem)
                                                                                    : sizeof(double) * BT * B_TSTRIDE;

template <bool FULL>
__device__ __forceinline__ void bart_stage_chunk(const BartDesc &d, const BartIO &io, BartSmem &sm, int k0, int kc,
                                                 int64_t i0, int64_t j0, int tid) {
    if (tid < kc) {
        const int k = k0 + tid;
        sm.dim[tid] = bart_dim((double)d.n[k], d.w[k], d.Wn, d.inv_Wn, io.psi);
    }
    for (int idx = tid; idx < 2 * kc * BT; idx += B_THREADS) {
        const int side = idx / (kc * BT), rem = idx % (kc * BT), kk = rem / BT, r = rem % BT;
        const int k = k0 + kk, nk = d.n[k];
        int v = 0;
        if (side == 0) {
            const int64_t i = i0 + r;
            if (i < io.n) v = io.ix[(int64_t)d.dim[k] * io.ldx + i];
        } else {
            const int64_t j = j0 + r;
            if (j < io.m) v = io.iy[(int64_t)d.dim[k] * io.ldy + j];
        }
        v = min(max(v, 0), nk);  // indices outside [0, n] would index the digamma table out of bounds
        if (FULL) {
            const BartPoint p = bart_point(v, nk, io.psi);
            sm.pt[side][0][kk][r] = p.v;
            sm.pt[side][1][kk][r] = p.pa;
            sm.pt[side][2][kk][r] = p.pb;
            sm.pt[side][3][kk][r] = p.rm;
            sm.pt[side][4][kk][r] = p.rp;
        } else {
            sm.pt[side][0][kk][r] = (double)v;
        }
    }
}

template <int MODE, bool NEED2, bool NEED3>
__global__ void __launch_bounds__(B_THREADS, 1) gram_bart_kernel(const __grid_constant__ BartDesc d,
                                                                 const __grid_constant__ BartIO io) {
    extern __shared__ __align__(16) unsigned char bsm_raw[];
    BartSmem &sm = *reinterpret_cast<BartSmem *>(bsm_raw);
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    if (io.sym && blockIdx.x > blockIdx.y) return;
    const bool diag_tile = io.sym && blockIdx.x == blockIdx.y;
    const int64_t i0 = (int64_t)blockIdx.y * BT, j0 = (int64_t)blockIdx.x * BT;

    double S2[B_RA][4], S3[B_RA][4], sumi[B_RA][4];
    bool any0[B_RA][4];
#pragma unroll
    for (int a = 0; a < B_RA; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) {
            S2[a][c] = 0.0;
            S3[a][c] = 0.0;
            sumi[a][c] = 0.0;
            any0[a][c] = false;
        }

    // ---- pass 1: point equality, S2 / S3
    for (int k0 = 0; k0 < d.p; k0 += B_CHUNK) {
        const int kc = min(B_CHUNK, d.p - k0);
        __syncthreads();
        // a single chunk serves both passes when all dimensions fit
        if (NEED3 && d.p <= B_CHUNK)
            bart_stage_chunk<true>(d, io, sm, k0, kc, i0, j0, tid);
        else
            bart_stage_chunk<false>(d, io, sm, k0, kc, i0, j0, tid);
        __syncthreads();
        for (int kk = 0; kk < kc; kk++) {
            const BartDim dk = sm.dim[kk];
            double vx[B_RA], vy[4];
#pragma unroll
            for (int a = 0; a < B_RA; a++) vx[a] = sm.pt[0][0][kk][ty + 32 * a];
#pragma unroll
            for (int b = 0; b < 2; b++) {
                const double2 t = *reinterpret_cast<const double2 *>(&sm.pt[1][0][kk][2 * tx + 32 * b]);
                vy[2 * b] = t.x;
                vy[2 * b + 1] = t.y;
            }
#pragma unroll
            for (int a = 0; a < B_RA; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) bart_pass1<NEED2, NEED3>(dk, vx[a], vy[c], S2[a][c], S3[a][c], any0[a][c]);
        }
    }
    // ---- pass 2 (width-3 brackets need the complete S3 before the per-dimension terms)
    if (NEED3) {
        for (int k0 = 0; k0 < d.p; k0 += B_CHUNK) {
            const int kc = min(B_CHUNK, d.p - k0);
            if (d.p > B_CHUNK) {
                __syncthreads();
                bart_stage_chunk<true>(d, io, sm, k0, kc, i0, j0, tid);
                __syncthreads();
            }
            for (int kk = 0; kk < kc; kk++) {
                const BartDim dk = sm.dim[kk];
                BartPoint px[B_RA], py[4];
#pragma unroll
                for (int a = 0; a < B_RA; a++) {
                    const int r = ty + 32 * a;
                    px[a].v = sm.pt[0][0][kk][r];
                    px[a].pa = sm.pt[0][1][kk][r];
                    px[a].pb = sm.pt[0][2][kk][r];
                    px[a].rm = sm.pt[0][3][kk][r];
                    px[a].rp = sm.pt[0][4][kk][r];
                }
#pragma unroll
                for (int b = 0; b < 2; b++) {
                    const int r = 2 * tx + 32 * b;
                    const double2 t0 = *reinterpret_cast<const double2 *>(&sm.pt[1][0][kk][r]);
                    const double2 t1 = *reinterpret_cast<const double2 *>(&sm.pt[1][1][kk][r]);
                    const double2 t2 = *reinterpret_cast<const double2 *>(&sm.pt[1][2][kk][r]);
                    const double2 t3 = *reinterpret_cast<const double2 *>(&sm.pt[1][3][kk][r]);
                    const double2 t4 = *reinterpret_cast<const double2 *>(&sm.pt[1][4][kk][r]);
                    py[2 * b].v = t0.x, py[2 * b + 1].v = t0.y;
                    py[2 * b].pa = t1.x, py[2 * b + 1].pa = t1.y;
                    py[2 * b].pb = t2.x, py[2 * b + 1].pb = t2.y;
                    py[2 * b].rm = t3.x, py[2 * b + 1].rm = t3.y;
                    py[2 * b].rp = t4.x, py[2 * b + 1].rp = t4.y;
                }
#pragma unroll
                for (int a = 0; a < B_RA; a++)
#pragma unroll
                    for (int c = 0; c < 4; c++) bart_pass2(dk, d.inv_Wn, S3[a][c], px[a], py[c], sumi[a][c]);
            }
        }
    }

    // ---- `repeat` scans of all stages, value (and alpha / beta duals)
    constexpr bool DUAL = MODE != BMODE_VALUE;
    double ga[B_RA][4], gb[B_RA][4];
#pragma unroll
    for (int a = 0; a < B_RA; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) {
            double g = d.gamma, da_ = 0.0, db_ = 0.0;
            int r = 0;
            for (int s = 0; s < d.nstages; s++) {
                const int width = d.stage_width[s];
                for (int q = 0; q < d.stage_nrows[s]; q++, r++)
                    bart_row<DUAL>(width, any0[a][c], d.Wn, d.inv_Wn, S2[a][c], S3[a][c], sumi[a][c], d.rows[r],
                                   d.drows[0][r], d.drows[1][r], g, da_, db_);
            }
            S2[a][c] = g;  // reuse as the result
            ga[a][c] = da_;
            gb[a][c] = db_;
        }

    if (MODE == BMODE_VJP) {
        // sum_ij G_ij * {corr, amp dcorr/dalpha, amp dcorr/dbeta}; symlower: G read from the lower triangle, w = 2 off it
        double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0;
#pragma unroll
        for (int a = 0; a < B_RA; a++) {
            const int64_t i = i0 + ty + 32 * a;
            if (i >= io.n) continue;
            const double bi = io.b ? io.b[i] : 0.0;
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int64_t j = j0 + 2 * tx + 32 * (c >> 1) + (c & 1);
                if (j >= io.m) continue;
                double wgt = 1.0;
                if (io.sym) {
                    if (j > i) continue;
                    wgt = (j < i) ? 2.0 : 1.0;
                }
                double gij = io.G[i * io.ldg + j];
                if (io.b) gij -= bi * io.b[j];
                gij *= wgt;
                acc0 += gij * S2[a][c];
                acc1 += gij * ga[a][c];
                acc2 += gij * gb[a][c];
            }
        }
        acc1 *= d.amp;
        acc2 *= d.amp;
        acc0 = warp_sum(acc0);
        acc1 = warp_sum(acc1);
        acc2 = warp_sum(acc2);
        __syncthreads();
        double *red = reinterpret_cast<double *>(bsm_raw);
        if ((tid & 31) == 0) {
            red[3 * (tid >> 5) + 0] = acc0;
            red[3 * (tid >> 5) + 1] = acc1;
            red[3 * (tid >> 5) + 2] = acc2;
        }
        __syncthreads();
        if (tid < 3) {
            double t = 0.0;
#pragma unroll
            for (int w = 0; w < B_THREADS / 32; w++) t += red[3 * w + tid];
            atomicAdd(io.out + tid, t);
        }
        return;
    }

    // ---- stores: the tile, and (symmetric case, off-diagonal tiles) its transpose through shared memory
    double *tsm = reinterpret_cast<double *>(bsm_raw);
    const int nout = (MODE == BMODE_DERIV) ? 3 : 1;
    for (int o = 0; o < nout; o++) {
        double *dst = (o == 0) ? io.K : (o == 1 ? io.dKa : io.dKb);
        const int64_t ld = (o == 0) ? io.ldk : io.ldd;
        if (!dst) continue;
        double vals[B_RA][4];
#pragma unroll
        for (int a = 0; a < B_RA; a++)
#pragma unroll
            for (int c = 0; c < 4; c++)
                vals[a][c] = LGP_B_MUL(d.amp, o == 0 ? S2[a][c] : (o == 1 ? ga[a][c] : gb[a][c]));
#pragma unroll
        for (int a = 0; a < B_RA; a++) {
            const int64_t i = i0 + ty + 32 * a;
            if (i >= io.n) continue;
            double *krow = dst + i * ld;
#pragma unroll
            for (int b = 0; b < 2; b++) {
                const int64_t j = j0 + 2 * tx + 32 * b;
                if (j >= io.m) continue;
                if (io.vec_ok && j + 1 < io.m) {
                    *reinterpret_cast<double2 *>(krow + j) = make_double2(vals[a][2 * b], vals[a][2 * b + 1]);
                } else {
                    krow[j] = vals[a][2 * b];
                    if (j + 1 < io.m) krow[j + 1] = vals[a][2 * b + 1];
                }
            }
        }
        if (io.sym && !diag_tile) {
            __syncthreads();
#pragma unroll
            for (int a = 0; a < B_RA; a++)
#pragma unroll
                for (int c = 0; c < 4; c++)
                    tsm[(2 * tx + 32 * (c >> 1) + (c & 1)) * B_TSTRIDE + ty + 32 * a] = vals[a][c];
            __syncthreads();
            // row jj of the transposed tile = column jj of the tile; 64 consecutive entries per row
            for (int idx = tid; idx < BT * BT; idx += B_THREADS) {
                const int jj = idx / BT, ii = idx % BT;
                const int64_t j = j0 + jj, i = i0 + ii;
                if (j < io.m && i < io.n) dst[j * ld + i] = tsm[jj * B_TSTRIDE + ii];
            }
        }
    }
}

__global__ void fill_kernel(double *K, int64_t ldk, int64_t n, int64_t m, double v) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t i = blockIdx.y + (int64_t)65535 * blockIdx.z;
    if (j < m && i < n) K[i * ldk + j] = v;
}

__global__ void bart_sum_kernel(const double *G, int64_t ldg, const double *b, int64_t n, int64_t m, int sym, double scale,
                                double *out) {
    // p == 0: correlation identically 1: out[0] += sum w_ij (G_ij - b_i b_j)
    double acc = 0.0;
    for (int64_t i = blockIdx.x; i < n; i += gridDim.x)
        for (int64_t j = threadIdx.x; j < (sym ? i + 1 : m); j += blockDim.x) {
            double g = G[i * ldg + j];
            if (b) g -= b[i] * b[j];
            acc += (sym && j < i) ? 2.0 * g : g;
        }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, scale * acc);
}

template <int MODE>
static cudaError_t bart_launch(int need2, int need3, dim3 grid, cudaStream_t st, const BartDesc &d, const BartIO &io) {
#define LGP_BART_GO(N2, N3)                                                                                        \
    do {                                                                                                           \
        static DeviceOnce once;                                                                                    \
        const int dev = current_device();                                                                          \
        if (!once.done(dev)) {                                                                                     \
            cudaError_t e = cudaFuncSetAttribute(gram_bart_kernel<MODE, N2, N3>,                                   \
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B_SMEM_BYTES);  \
            if (e != cudaSuccess) return e;                                                                        \
            once.set(dev);                                                                                         \
        }                                                                                                          \
        gram_bart_kernel<MODE, N2, N3><<<grid, B_THREADS, B_SMEM_BYTES, st>>>(d, io);                              \
    } while (0)
    if (need2 && need3)
        LGP_BART_GO(true, true);
    else if (need3)
        LGP_BART_GO(false, true);
    else if (need2)
        LGP_BART_GO(true, false);
    else
        LGP_BART_GO(false, false);
#undef LGP_BART_GO
    return cudaGetLastError();
}

// fills the descriptor; returns LGP_OK, or 1 when no covariate is active (correlation identically 1), or an error
static int bart_build(BartDesc &d, int p, const int32_t *nsplits, const double *w, int nstages, const int32_t *stage_width,
                      const int32_t *stage_nrows, const double *rows, const double *drows, double gamma, double amp,
                      int *need2, int *need3) {
    memset(&d, 0, sizeof(d));
    if (p < 0 || (p && !nsplits) || nstages < 1 || !stage_width || !stage_nrows || !rows) return LGP_ERR_BADARG;
    if (nstages > B_MAX_STAGES) return LGP_ERR_UNSUPPORTED;
    int total = 0;
    *need2 = *need3 = 0;
    for (int s = 0; s < nstages; s++) {
        if (stage_width[s] < 1 || stage_width[s] > 3 || stage_nrows[s] < 1) return LGP_ERR_UNSUPPORTED;
        d.stage_width[s] = stage_width[s];
        d.stage_nrows[s] = stage_nrows[s];
        total += stage_nrows[s];
        if (stage_width[s] == 2) *need2 = 1;
        if (stage_width[s] == 3) *need3 = 1;
    }
    if (total > B_MAX_ROWS) return LGP_ERR_UNSUPPORTED;
    d.nstages = nstages;
    for (int r = 0; r < total; r++)
        for (int c = 0; c < 3; c++) {
            d.rows[r][c] = rows[3 * r + c];
            d.drows[0][r][c] = drows ? drows[3 * r + c] : 0.0;
            d.drows[1][r][c] = drows ? drows[3 * total + 3 * r + c] : 0.0;
        }
    // compact away zero-weight covariates (reference masks them: _bart.py:669-672)
    int pa = 0;
    double Wn = 0.0;
    for (int k = 0; k < p; k++) {
        double wk = w ? w[k] : 1.0;
        if (wk == 0.0) continue;
        if (pa >= B_MAX_P) return LGP_ERR_UNSUPPORTED;
        if (nsplits[k] < 0) return LGP_ERR_BADARG;
        d.dim[pa] = k;
        d.n[pa] = nsplits[k];
        d.w[pa] = wk;
        if (nsplits[k]) Wn += wk;  // Wn = sum(where(n, w, 0))   (_bart.py:694)
        pa++;
    }
    d.p = pa;
    d.Wn = Wn;
    d.inv_Wn = 1.0 / Wn;
    d.gamma = gamma;
    d.amp = amp;
    return pa == 0 ? 1 : LGP_OK;
}

}  // namespace lgp

using namespace lgp;

extern "C" {

// psi_out[k] = digamma(k) for k = 1..len-1 (psi_out[0] = -inf), HOST memory; extended precision recurrence.
int lgp_bart_digamma_table(double *psi_out, int64_t len) {
    if (!psi_out || len < 1) return LGP_ERR_BADARG;
    psi_out[0] = -INFINITY;
    long double v = -0.577215664901532860606512090082402431L;  // digamma(1) = -EulerGamma
    for (int64_t k = 1; k < len; k++) {
        psi_out[k] = (double)v;
        v += 1.0L / (long double)k;
    }
    return LGP_OK;
}

int lgp_gram_bart_stages(lgp_stream_t stream, int p, const int32_t *nsplits, const double *w, int nstages,
                         const int32_t *stage_width, const int32_t *stage_nrows, const double *rows, const double *drows,
                         double gamma, double amp, const double *psi, const int32_t *ix, int64_t ldx, int64_t n,
                         const int32_t *iy, int64_t ldy, int64_t m, double *K_out, int64_t ldk, double *dKa_out,
                         double *dKb_out, int64_t ldd, int flags) {
    if (n < 0 || m < 0 || (!K_out && !dKa_out && !dKb_out)) return LGP_ERR_BADARG;
    if (n == 0 || m == 0) return LGP_OK;
    if ((K_out && ldk < m) || ((dKa_out || dKb_out) && ldd < m)) return LGP_ERR_BADARG;
    const bool deriv = dKa_out || dKb_out;
    if (deriv && !drows) return LGP_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    BartDesc d;
    int need2, need3;
    int rc = bart_build(d, p, nsplits, w, nstages, stage_width, stage_nrows, rows, drows, gamma, amp, &need2, &need3);
    if (rc < 0) return rc;
    if (rc == 1) {
        // no covariates: correlation is identically 1 (_bart.py:659-661), derivatives 0
        dim3 g((unsigned)((m + 255) / 256), (unsigned)(n < 65535 ? n : 65535), (unsigned)((n + 65534) / 65535));
        if (K_out) fill_kernel<<<g, 256, 0, st>>>(K_out, ldk, n, m, amp);
        if (dKa_out) fill_kernel<<<g, 256, 0, st>>>(dKa_out, ldd, n, m, 0.0);
        if (dKb_out) fill_kernel<<<g, 256, 0, st>>>(dKb_out, ldd, n, m, 0.0);
        LGP_CUDA_CHECK_LAUNCH();
        return LGP_OK;
    }
    if (need3 && !psi) return LGP_ERR_BADARG;
    if (!ix || !iy) return LGP_ERR_BADARG;
    const bool sym = (flags & LGP_BART_SYMMETRIC) != 0;
    if (sym && (ix != iy || n != m)) return LGP_ERR_BADARG;
    BartIO io;
    memset(&io, 0, sizeof(io));
    io.psi = psi;
    io.ix = ix, io.iy = iy, io.ldx = ldx, io.ldy = ldy, io.n = n, io.m = m;
    io.K = K_out, io.ldk = ldk, io.dKa = dKa_out, io.dKb = dKb_out, io.ldd = ldd;
    io.sym = sym;
    auto aligned = [](const double *ptr, int64_t ld) { return !ptr || (((ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(ptr) & 15) == 0)); };
    io.vec_ok = aligned(K_out, ldk) && aligned(dKa_out, ldd) && aligned(dKb_out, ldd);
    dim3 grid((unsigned)((m + BT - 1) / BT), (unsigned)((n + BT - 1) / BT));
    if (grid.y > 65535) return LGP_ERR_UNSUPPORTED;
    cudaError_t e = deriv ? bart_launch<BMODE_DERIV>(need2, need3, grid, st, d, io)
                          : bart_launch<BMODE_VALUE>(need2, need3, grid, st, d, io);
    count_launch();
    return e == cudaSuccess ? LGP_OK : LGP_ERR_CUDA;
}

int lgp_gram_bart_vjp(lgp_stream_t stream, int p, const int32_t *nsplits, const double *w, int nstages,
                      const int32_t *stage_width, const int32_t *stage_nrows, const double *rows, const double *drows,
                      double gamma, double amp, const double *psi, const int32_t *ix, int64_t ldx, int64_t n,
                      const int32_t *iy, int64_t ldy, int64_t m, const double *G, int64_t ldg, const double *b,
                      int symlower, double *out) {
    if (n < 0 || m < 0 || !G || !out || !drows) return LGP_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(out, 0, 3 * sizeof(double), st) != cudaSuccess) return LGP_ERR_CUDA;
    if (n == 0 || m == 0) return LGP_OK;
    if (ldg < m) return LGP_ERR_BADARG;
    if (b && !symlower) return LGP_ERR_BADARG;
    BartDesc d;
    int need2, need3;
    int rc = bart_build(d, p, nsplits, w, nstages, stage_width, stage_nrows, rows, drows, gamma, amp, &need2, &need3);
    if (rc < 0) return rc;
    if (rc == 1) {
        bart_sum_kernel<<<1024, 256, 0, st>>>(G, ldg, b, n, m, symlower ? 1 : 0, 1.0, out);
        LGP_CUDA_CHECK_LAUNCH();
        return LGP_OK;
    }
    if (need3 && !psi) return LGP_ERR_BADARG;
    if (!ix || !iy) return LGP_ERR_BADARG;
    if (symlower && (ix != iy || n != m)) return LGP_ERR_BADARG;
    BartIO io;
    memset(&io, 0, sizeof(io));
    io.psi = psi;
    io.ix = ix, io.iy = iy, io.ldx = ldx, io.ldy = ldy, io.n = n, io.m = m;
    io.G = G, io.ldg = ldg, io.b = b, io.out = out;
    io.sym = symlower ? 1 : 0;
    dim3 grid((unsigned)((m + BT - 1) / BT), (unsigned)((n + BT - 1) / BT));
    if (grid.y > 65535) return LGP_ERR_UNSUPPORTED;
    cudaError_t e = bart_launch<BMODE_VJP>(need2, need3, grid, st, d, io);
    count_launch();
    return e == cudaSuccess ? LGP_OK : LGP_ERR_CUDA;
}

// single-bracket form kept for ABI compatibility (value only, one stage)
int lgp_gram_bart(lgp_stream_t stream, int p, const int32_t *nsplits, const double *w, const double *rows, int nrows,
                  int width, double gamma, double amp, const double *psi, const int32_t *ix, int64_t ldx, int64_t n,
                  const int32_t *iy, int64_t ldy, int64_t m, double *K_out, int64_t ldk, int flags) {
    if (!K_out || !rows || width < 1 || width > 3 || nrows < 1 || nrows > B_MAX_ROWS) return LGP_ERR_UNSUPPORTED;
    double r3[B_MAX_ROWS * 3];
    for (int r = 0; r < nrows; r++)
        for (int c = 0; c < 3; c++) r3[3 * r + c] = c < width ? rows[r * width + c] : 0.0;
    const int32_t sw = width, sn = nrows;
    return lgp_gram_bart_stages(stream, p, nsplits, w, 1, &sw, &sn, r3, nullptr, gamma, amp, psi, ix, ldx, n, iy, ldy, m,
                                K_out, ldk, nullptr, nullptr, 0, flags);
}

}  // extern "C"
