// Blocked recursive FP64 Cholesky with lsqfitgp's equilibration + Gershgorin jitter, triangular
// solves, triangular products, and inverse-from-factor, all built on the DMMA GEMM.
//
// Reference semantics: src/lsqfitgp/_linalg/_decomp.py:245-255 (_parseeps), :349-361
// (eigval_bound, diag_scale_pow2), :380-393 (Chol.__init__), :398-439 (solves), :466-472.
#include <limits.h>
#include <mutex>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../include/lgp_b200.h"
#include "common.cuh"
#include "gemm_dmma.cuh"
#include "internal.h"
#include "chol_leaf3.cuh"

namespace lgp {

// ------------------------------------------------------------------------------------------------
// 1. equilibration + jitter (one pass over K)
// ------------------------------------------------------------------------------------------------

// s_i = 2^rint(log2(K_ii)/2), 1 if K_ii == 0 (reference: diag_scale_pow2, _decomp.py:356-361)
__global__ void chol_diag_scale_kernel(const double *__restrict__ K, int64_t ldk, const double *__restrict__ addmat,
                                       int64_t ldadd, const double *__restrict__ adddiag, int n, int npad,
                                       double *__restrict__ aux) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npad) return;
    double s = 1.0;
    if (i < n) {
        double d = K[(int64_t)i * ldk + i];
        if (addmat) d = d + addmat[(int64_t)i * ldadd + i];
        if (adddiag) d = d + adddiag[i];
        if (d != 0.0) s = exp2(rint(0.5 * log2(d)));
    }
    aux[LGP_AUX_S(npad) + i] = s;
    aux[LGP_AUX_SINV(npad) + i] = 1.0 / s;
    if (i < 16) aux[LGP_AUX_SCALARS(npad) + i] = 0.0;
}

__device__ __forceinline__ void atomic_max_nonneg(double *addr, double v) {
    // non-negative doubles (and NaN, which compares above +inf as bits) order like their bit patterns
    atomicMax(reinterpret_cast<unsigned long long *>(addr), (unsigned long long)__double_as_longlong(v));
}

// One warp per row: Kt = (K + add)/s_i/s_j -> lower triangle of W, row abs-sums -> running max.
// Rows >= n are identity padding.
__global__ void __launch_bounds__(256) chol_prepare_kernel(const double *__restrict__ K, int64_t ldk,
                                                           const double *__restrict__ addmat, int64_t ldadd,
                                                           const double *__restrict__ adddiag, int n, int npad,
                                                           double *__restrict__ W, int64_t ldw,
                                                           double *__restrict__ aux) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + warp;
    if (i >= npad) return;
    double *wrow = W + (int64_t)i * ldw;
    if (i >= n) {
        for (int j = lane; j <= i; j += 32) wrow[j] = (j == i) ? 1.0 : 0.0;
        return;
    }
    const double *sinv = aux + LGP_AUX_SINV(npad);
    const double si = sinv[i];
    const double *krow = K + (int64_t)i * ldk;
    const double *arow = addmat ? addmat + (int64_t)i * ldadd : nullptr;
    double sum = 0.0;
    for (int j = lane; j < n; j += 32) {
        double v = krow[j];
        if (arow) v = v + arow[j];
        if (adddiag && j == i) v = v + adddiag[i];
        v = (v * sinv[j]) * si;  // exact: powers of two
        sum += fabs(v);
        if (j <= i) wrow[j] = v;
    }
    sum = warp_sum(sum);
    if (lane == 0) atomic_max_nonneg(aux + LGP_AUX_SCALARS(npad) + 0, sum);
}

// eps = epsrel * maxrowsum + epsabs; W_ii += eps (i < n); min s^2
__global__ void __launch_bounds__(1024) chol_jitter_kernel(int n, int npad, double epsrel, double epsabs,
                                                           double *__restrict__ W, int64_t ldw,
                                                           double *__restrict__ aux, int32_t *__restrict__ info) {
    double *sc = aux + LGP_AUX_SCALARS(npad);
    const double eps = epsrel * sc[0] + epsabs;
    const double *s = aux + LGP_AUX_S(npad);
    double mn = INFINITY;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        W[(int64_t)i * ldw + i] += eps;
        double v = s[i] * s[i];
        mn = (v < mn || v != v) ? v : mn;
    }
    __shared__ double red[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double u = __shfl_xor_sync(0xffffffffu, mn, o);
        mn = (u < mn || u != u) ? u : mn;
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mn;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); w++) {
            double u = red[w];
            mn = (u < mn || u != u) ? u : mn;
        }
        sc[1] = eps;
        sc[3] = mn;
        *info = INT_MAX;
    }
}

// ------------------------------------------------------------------------------------------------
// 2. small elementwise / reduction kernels
// ------------------------------------------------------------------------------------------------
constexpr int GRID_Y_MAX = 65535;
// grid covering `cols` columns (256 per CTA) x `rows` rows, rows folded over (y, z) to respect the gridDim.y limit
static inline dim3 rows_grid(int cols, int rows) {
    return dim3((unsigned)((cols + 255) / 256), (unsigned)(rows < GRID_Y_MAX ? rows : GRID_Y_MAX),
                (unsigned)((rows + GRID_Y_MAX - 1) / GRID_Y_MAX));
}

__global__ void row_scale_kernel(double *__restrict__ B, int64_t ldb, int n, int m, const double *__restrict__ f) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)n * m) return;
    int i = (int)(idx / m), j = (int)(idx % m);
    B[(int64_t)i * ldb + j] *= f[i];
}

__global__ void row_scale_copy_kernel(const double *__restrict__ X, int64_t ldx, double *__restrict__ Y, int64_t ldy,
                                      int n, int m, const double *__restrict__ f) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)n * m) return;
    int i = (int)(idx / m), j = (int)(idx % m);
    Y[(int64_t)i * ldy + j] = X[(int64_t)i * ldx + j] * (f ? f[i] : 1.0);
}

__global__ void get_factor_kernel(const double *__restrict__ W, int64_t ldw, const double *__restrict__ s, int n,
                                  double *__restrict__ L, int64_t ldl) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y + GRID_Y_MAX * blockIdx.z;  // gridDim.y is limited to 65535: rows continue along z
    if (j >= n || i >= n) return;
    L[(int64_t)i * ldl + j] = (j <= i) ? W[(int64_t)i * ldw + j] * s[i] : 0.0;
}

// Kinv_ij *= sinv_i * sinv_j on the lower triangle (undo the equilibration of the inverse)
__global__ void copy_block_kernel(const double *__restrict__ src, int64_t lds, double *__restrict__ dst, int64_t ldd,
                                  int rows, int cols) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j >= cols || i >= rows) return;
    dst[(int64_t)i * ldd + j] = src[(int64_t)i * lds + j];
}

// out[0] = sum_i log(d_i * s_i), out[1] = sum_i a_i^2 ; single CTA, fixed summation order (deterministic)
__global__ void __launch_bounds__(1024) logdet_quad_kernel(const double *__restrict__ d, const double *__restrict__ s,
                                                           const double *__restrict__ a, int n,
                                                           double *__restrict__ out) {
    double ld = 0.0, q = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        ld += log(d[i] * s[i]);
        if (a) q += a[i] * a[i];
    }
    __shared__ double r0[32], r1[32];
    ld = warp_sum(ld);
    q = warp_sum(q);
    if ((threadIdx.x & 31) == 0) {
        r0[threadIdx.x >> 5] = ld;
        r1[threadIdx.x >> 5] = q;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        int nw = blockDim.x >> 5;
        ld = threadIdx.x < nw ? r0[threadIdx.x] : 0.0;
        q = threadIdx.x < nw ? r1[threadIdx.x] : 0.0;
        ld = warp_sum(ld);
        q = warp_sum(q);
        if (threadIdx.x == 0) {
            out[0] = ld;
            out[1] = q;
        }
    }
}

__global__ void finalize_info_kernel(int32_t *info, int n) {
    int v = *info;
    if (v == INT_MAX || v > n) *info = 0;  // pivots in the identity padding cannot fail first
}

// ------------------------------------------------------------------------------------------------
// 3. host-side recursion (all sizes in 128-blocks of the padded matrix)
// ------------------------------------------------------------------------------------------------
// the > 48 KB shared-memory opt-in is a per-device attribute: once per device, not once per process
static int leaf_attr() {
    static DeviceOnce once;
    const int dev = current_device();
    if (dev < 0) return LGP_ERR_CUDA;
    if (!once.done(dev)) {
        if (cudaFuncSetAttribute(potrf_leaf3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L3_SMEM_BYTES) !=
            cudaSuccess)
            return LGP_ERR_CUDA;
        once.set(dev);
    }
    return LGP_OK;
}
// experiment switches are read once per process
static bool trace_enabled() {
    static const bool v = getenv("LGP_TRACE") != nullptr;
    return v;
}
static int panel_blocks() {
    static const int v = [] {
        const char *e = getenv("LGP_PANEL_BLOCKS");
        return (e && atoi(e) > 0) ? atoi(e) : 4;
    }();
    return v;
}
static void leaf_launch(cudaStream_t st, double *Wblk, int64_t ld, double *invd, double *dvec, int32_t *info, int j0) {
    potrf_leaf3_kernel<<<1, L3_THREADS, L3_SMEM_BYTES, st>>>(Wblk, ld, invd, dvec, info, j0);
}

struct CholCtx {
    cudaStream_t st;
    double *W;
    int64_t ldw;
    double *invd;  // per-block 128x128 inverses
    double *dvec;
    int32_t *info;
    int rc;
    int j0base = 0;  // global index of row 0 of W (tile-wise use: pivots and dvec are indexed globally)
    GemmMirror mir = {};  // extra destinations of the solved panel (lgp_tile_trsm_right_bcast); column 0 = column 0 of B
};

struct FlagPtrs {
    int n;
    unsigned long long *p[LGP_MAX_FLAGS];
};

#define RC(x)                   \
    do {                        \
        int r__ = (x);          \
        if (r__ != LGP_OK) {    \
            c.rc = r__;         \
            return;             \
        }                       \
    } while (0)

static inline double *Wp(const CholCtx &c, int rb, int cb) { return c.W + (int64_t)rb * NB * c.ldw + (int64_t)cb * NB; }

// X * Lt^T = B in place for the nb-block triangle Lt (pointer to its top-left, ld ldl; inverted 128x128 diagonal
// blocks in invd); B points at the `rows` x nb*128 block to be solved (ld ldb)
// `col0`: column of B relative to the panel origin (offset of the mirror destinations, which receive the final value of
// every 128-column block from the epilogue of its last product)
static void trsm_right_ptr(CholCtx &c, double *B, int64_t ldb, int rows, const double *Lt, int64_t ldl,
                           const double *invd, int nb, int col0 = 0) {
    if (c.rc) return;
    if (nb == 1) {
        if (c.mir.n) {
            GemmMirror m = c.mir;
            for (int i = 0; i < m.n; i++) m.dst[i] += col0;
            RC(gemm_launch(c.st, true, true, rows, NB, NB, 1.0, B, ldb, invd, NB, B, ldb,
                           GEMM_BETA0 | GEMM_B_LOWER_K | GEMM_INPLACE_A, &m));
            return;
        }
        RC(gemm_launch(c.st, true, true, rows, NB, NB, 1.0, B, ldb, invd, NB, B, ldb,
                       GEMM_BETA0 | GEMM_B_LOWER_K | GEMM_INPLACE_A));
        return;
    }
    int n1 = nb / 2, n2 = nb - n1;
    trsm_right_ptr(c, B, ldb, rows, Lt, ldl, invd, n1, col0);
    if (c.rc) return;
    // B2 -= B1 * L21^T
    RC(gemm_launch(c.st, true, true, rows, n2 * NB, n1 * NB, -1.0, B, ldb, Lt + (int64_t)n1 * NB * ldl, ldl,
                   B + (int64_t)n1 * NB, ldb, 0));
    trsm_right_ptr(c, B + (int64_t)n1 * NB, ldb, rows, Lt + (int64_t)n1 * NB * ldl + (int64_t)n1 * NB, ldl,
                   invd + (int64_t)n1 * NB * NB, n2, col0 + n1 * NB);
}

// X * Lt[jb..jb+nb, jb..jb+nb]^T = B in place; B = W[rb.., jb..] with `rows` rows
static void trsm_right_rec(CholCtx &c, int rb, int rows, int jb, int nb) {
    trsm_right_ptr(c, Wp(c, rb, jb), c.ldw, rows, Wp(c, jb, jb), c.ldw, c.invd + (int64_t)jb * NB * NB, nb);
}

static void potrf_rec(CholCtx &c, int jb, int nb) {
    if (c.rc) return;
    if (nb == 1) {
        leaf_launch(c.st, Wp(c, jb, jb), c.ldw, c.invd + (int64_t)jb * NB * NB, c.dvec, c.info, c.j0base + jb * NB);
        count_launch();
        if (cudaGetLastError() != cudaSuccess) c.rc = LGP_ERR_CUDA;
        return;
    }
    int n1 = nb / 2, n2 = nb - n1;
    potrf_rec(c, jb, n1);
    trsm_right_rec(c, jb + n1, n2 * NB, jb, n1);
    if (c.rc) return;
    RC(gemm_launch(c.st, true, true, n2 * NB, n2 * NB, n1 * NB, -1.0, Wp(c, jb + n1, jb), c.ldw, Wp(c, jb + n1, jb),
                   c.ldw, Wp(c, jb + n1, jb + n1), c.ldw, GEMM_LOWER));
    potrf_rec(c, jb + n1, n2);
}

// Right-looking blocked factorisation with one-panel look-ahead on two streams:
//   panel stream (high priority): diagonal-block potrf + TRSM of the block column below it;
//   main stream: trailing SYRK, split into "next block column" (releases the next panel) and "rest".
// The panel chain of small launches overlaps the big trailing update of the previous panel.
// One panel stream per caller stream (up to 8; concurrent factorisations issued from different streams / host threads, e.g.
// a batch of hyperparameter points in flight, must not serialise their panel chains behind each other).
// The pool is per device: stream handles are only meaningful on the device they were created on, and the default
// stream handle (0) is the same on every device.
static cudaStream_t panel_stream(cudaStream_t caller) {
    static std::mutex mu;
    struct Slot {
        cudaStream_t caller, s;
        bool used;
    };
    static Slot pools[MAX_DEVICES][8];
    const int dev = current_device();
    if (dev < 0) return nullptr;
    Slot *pool = pools[dev];
    std::lock_guard<std::mutex> lock(mu);
    int free_slot = -1;
    for (int i = 0; i < 8; i++) {
        if (pool[i].used && pool[i].caller == caller) return pool[i].s;
        if (!pool[i].used && free_slot < 0) free_slot = i;
    }
    if (free_slot < 0) return pool[0].s;  // more than 8 caller streams: share (still correct, ordered by events)
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    cudaStream_t s = nullptr;
    if (cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, hi) != cudaSuccess) return nullptr;
    pool[free_slot].caller = caller;
    pool[free_slot].s = s;
    pool[free_slot].used = true;
    return s;
}

// cross-stream ordering helpers: a failed record / wait would silently drop an ordering constraint, so every return
// code is checked and turned into LGP_ERR_CUDA
static inline bool ev_record(cudaEvent_t e, cudaStream_t s) { return e && cudaEventRecord(e, s) == cudaSuccess; }
static inline bool ev_wait(cudaStream_t s, cudaEvent_t e) { return e && cudaStreamWaitEvent(s, e, 0) == cudaSuccess; }

// Panel width (in 128-blocks) for a trailing matrix of `left` blocks.  Wide panels make the trailing rank-k updates
// efficient while they dominate; once the trailing matrix is small the factorisation is bound by the chain of dependent
// panel kernels, whose length per 128 columns grows with the recursion depth of the panel (4-block panel: 4 leaves + 17
// small GEMMs per 512 columns; 1-block panels: 4 leaves + 8), so the tail switches to narrower panels.
static int panel_width(int left, int pb) {
    static int t0 = -1, t1 = -1, t2 = -1;
    if (t0 < 0) {
        // thresholds in blocks of remaining rows: above a -> 2 * pb (rank-1024 trailing updates run at 35.4 instead of
        // 34.4 TFLOP/s), above b -> pb, above c -> 2 blocks, else 1 block.  Tuned on B200 (see DESIGN.md section 3).
        int a = 96, b = 64, c = 32;
        const char *e = getenv("LGP_TAIL_BLOCKS");
        if (e) {
            int x = 0, y = 0, z = 0;
            const int got = sscanf(e, "%d,%d,%d", &x, &y, &z);
            if (got == 3) a = x, b = y, c = z;
            if (got == 2) b = x, c = y;
        }
        t1 = b;
        t2 = c;
        t0 = a;
    }
    int w = pb;
    if (left > t0) w = 2 * pb;
    if (left <= t1 && w > 2) w = 2;
    if (left <= t2) w = 1;
    return w < left ? w : left;
}

static int chain_blocks() {
    static const int v = [] {
        const char *e = getenv("LGP_CHAIN_BLOCKS");
        return e ? atoi(e) : 32;
    }();
    return v;
}
static int first_blocks() {
    static const int v = [] {
        const char *e = getenv("LGP_FIRST_BLOCKS");
        return (e && atoi(e) > 0) ? atoi(e) : 2;
    }();
    return v;
}

static int potrf_lookahead(CholCtx &cm, int nblk, int pb) {
    cudaStream_t ps = (nblk > pb) ? panel_stream(cm.st) : nullptr;
    if (!ps) {
        potrf_rec(cm, 0, nblk);
        return cm.rc;
    }
    const bool trace = trace_enabled();  // debug only: synchronises and prints a per-panel timeline
    CholCtx cp = cm;
    cp.st = ps;
    const int np = nblk;  // upper bound on the number of panels (the tail uses narrower ones)
    cudaEvent_t e_fork = nullptr, e_last = nullptr;
    cudaEvent_t *t_pstart = nullptr, *t_restend = nullptr, *t_panel = nullptr, *t_col = nullptr;
    if (trace) {
        t_pstart = new cudaEvent_t[4 * np + 1];
        t_restend = t_pstart + np;
        t_panel = t_restend + np;
        t_col = t_panel + np;
        for (int i = 0; i < 4 * np + 1; i++) cudaEventCreate(&t_pstart[i]);
        e_fork = t_pstart[4 * np];
    } else {
        e_fork = ring_event();
    }
    bool ok = ev_record(e_fork, cm.st) && ev_wait(ps, e_fork);
    int rc = LGP_OK;
    int last = -1;
    cudaEvent_t e_colnext = nullptr;  // recorded on the main stream when the next panel's block column is updated
    cudaEvent_t e_rest = nullptr;     // recorded on the main stream behind the rest of the previous trailing update
    int jb = 0;
    for (int j = 0; jb < nblk && rc == LGP_OK && ok; j++) {
        int w = panel_width(nblk - jb, pb);
        // nothing overlaps the very first panel: keep it narrow (the second one hides behind its trailing update)
        if (j == 0 && w > first_blocks()) w = first_blocks();
        const int rest = nblk - jb - w;
        // ---- panel stream
        if (e_colnext) ok = ok && ev_wait(ps, e_colnext);
        e_colnext = nullptr;
        if (trace) cudaEventRecord(t_pstart[j], ps);
        potrf_rec(cp, jb, w);
        if (rest > 0) trsm_right_rec(cp, jb + w, rest * NB, jb, w);
        cudaEvent_t e_panel = trace ? t_panel[j] : ring_event();
        ok = ok && ev_record(e_panel, ps);
        e_last = e_panel;
        last = j;
        if ((rc = cp.rc) != LGP_OK || rest == 0 || !ok) break;
        const int w2 = panel_width(rest, pb);  // width of the next panel
        const int rest2 = rest - w2;
        const int K = w * NB;
        // Update of the next block column (rows jb+w.., cols jb+w..jb+w+w2): one full GEMM; the part above the block
        // diagonal is scratch (never read: leaves and LOWER kernels only touch r >= c).  While the trailing matrix is
        // large it runs on the main stream, in order behind the rest of the previous update.  In the chain-bound tail it
        // stays on the panel stream: leaf -> TRSM -> column update -> next leaf then are launches of ONE stream, without
        // the two cross-stream event hops per panel (it still waits for the previous rest update, which has long
        // finished there).
        // (measured on B200: at n <= 12 800 the whole factorisation is faster this way, 14.06 -> 13.68 ms at n = 10 000; at
        // n = 20 000 only the last 32 blocks are)
        const bool chain_on_ps = rest <= (nblk <= 100 ? nblk : chain_blocks());
        if (chain_on_ps) {
            if (e_rest) ok = ok && ev_wait(ps, e_rest);
            rc = gemm_launch(ps, true, true, rest * NB, w2 * NB, K, -1.0, Wp(cm, jb + w, jb), cm.ldw, Wp(cm, jb + w, jb),
                             cm.ldw, Wp(cm, jb + w, jb + w), cm.ldw, 0);
            if (trace) cudaEventRecord(t_col[j], ps);
            ok = ok && ev_wait(cm.st, e_panel);
        } else {
            ok = ok && ev_wait(cm.st, e_panel);
            rc = gemm_launch(cm.st, true, true, rest * NB, w2 * NB, K, -1.0, Wp(cm, jb + w, jb), cm.ldw,
                             Wp(cm, jb + w, jb), cm.ldw, Wp(cm, jb + w, jb + w), cm.ldw, 0);
            e_colnext = trace ? t_col[j] : ring_event();
            ok = ok && ev_record(e_colnext, cm.st);
        }
        // rest of the trailing matrix
        if (rc == LGP_OK && rest2 > 0)
            rc = gemm_launch(cm.st, true, true, rest2 * NB, rest2 * NB, K, -1.0, Wp(cm, jb + w + w2, jb), cm.ldw,
                             Wp(cm, jb + w + w2, jb), cm.ldw, Wp(cm, jb + w + w2, jb + w + w2), cm.ldw, GEMM_LOWER);
        if (trace) {
            cudaEventRecord(t_restend[j], cm.st);
            e_rest = t_restend[j];
        } else {
            e_rest = ring_event();
            ok = ok && ev_record(e_rest, cm.st);
        }
        if (chain_on_ps) {
            // the join below must see the column update as well
            e_last = ring_event();
            ok = ok && ev_record(e_last, ps);
        }
        jb += w;
    }
    if (e_last) ok = ev_wait(cm.st, e_last) && ok;  // join
    if (!ok) {
        // an ordering constraint could not be enqueued: drain both streams so that nothing runs out of order, and fail
        cudaStreamSynchronize(ps);
        cudaStreamSynchronize(cm.st);
        if (rc == LGP_OK) rc = LGP_ERR_CUDA;
    }
    if (trace) {
        cudaStreamSynchronize(cm.st);
        cudaStreamSynchronize(ps);
        for (int j = 0; j <= last; j++) {
            float a = 0, b = 0, c2 = 0, d = 0;
            cudaEventElapsedTime(&a, e_fork, t_pstart[j]);
            cudaEventElapsedTime(&b, e_fork, t_panel[j]);
            if (j < last) {
                cudaEventElapsedTime(&c2, e_fork, t_col[j]);
                cudaEventElapsedTime(&d, e_fork, t_restend[j]);
            }
            fprintf(stderr, "[lgp trace] panel %3d: start %8.3f done %8.3f (%.3f ms) | colupd done %8.3f rest done %8.3f\n", j,
                    a, b, b - a, c2, d);
        }
        for (int i = 0; i < 4 * np + 1; i++) cudaEventDestroy(t_pstart[i]);
        delete[] t_pstart;
    }
    if (rc == LGP_OK && cudaGetLastError() != cudaSuccess) rc = LGP_ERR_CUDA;
    return rc;
}

struct SolveCtx {
    cudaStream_t st;
    const double *W;
    int64_t ldw;
    const double *invd;
    int n;  // true size (rows of B)
    double *B;
    int64_t ldb;
    int m;
    int rc;
};
static inline const double *Wc(const SolveCtx &c, int rb, int cb) {
    return c.W + (int64_t)rb * NB * c.ldw + (int64_t)cb * NB;
}
static inline int rows_in(const SolveCtx &c, int jb, int nb) {
    int lo = jb * NB, hi = (jb + nb) * NB;
    if (hi > c.n) hi = c.n;
    return hi > lo ? hi - lo : 0;
}

// Lt X = B (forward), blocks [jb, jb+nb)
static void solve_lower_rec(SolveCtx &c, int jb, int nb) {
    if (c.rc) return;
    int rows = rows_in(c, jb, nb);
    if (rows == 0) return;
    double *Bj = c.B + (int64_t)jb * NB * c.ldb;
    if (nb == 1) {
        RC(gemm_launch(c.st, true, false, rows, c.m, rows, 1.0, c.invd + (int64_t)jb * NB * NB, NB, Bj, c.ldb, Bj,
                       c.ldb, GEMM_BETA0 | GEMM_A_LOWER_K | GEMM_INPLACE_B));
        return;
    }
    int n1 = nb / 2, n2 = nb - n1;
    solve_lower_rec(c, jb, n1);
    if (c.rc) return;
    int rows2 = rows_in(c, jb + n1, n2);
    if (rows2 > 0) {
        RC(gemm_launch(c.st, true, false, rows2, c.m, n1 * NB, -1.0, Wc(c, jb + n1, jb), c.ldw, Bj, c.ldb,
                       Bj + (int64_t)n1 * NB * c.ldb, c.ldb, 0));
        solve_lower_rec(c, jb + n1, n2);
    }
}

// Lt^T X = B (backward)
static void solve_upper_rec(SolveCtx &c, int jb, int nb) {
    if (c.rc) return;
    int rows = rows_in(c, jb, nb);
    if (rows == 0) return;
    double *Bj = c.B + (int64_t)jb * NB * c.ldb;
    if (nb == 1) {
        RC(gemm_launch(c.st, false, false, rows, c.m, rows, 1.0, c.invd + (int64_t)jb * NB * NB, NB, Bj, c.ldb, Bj,
                       c.ldb, GEMM_BETA0 | GEMM_A_UPPER_K | GEMM_INPLACE_B));
        return;
    }
    int n1 = nb / 2, n2 = nb - n1;
    int rows2 = rows_in(c, jb + n1, n2);
    if (rows2 > 0) {
        solve_upper_rec(c, jb + n1, n2);
        if (c.rc) return;
        // B1 -= L21^T X2 : Aop[i][k] = L21[k][i]
        RC(gemm_launch(c.st, false, false, n1 * NB, c.m, rows2, -1.0, Wc(c, jb + n1, jb), c.ldw,
                       Bj + (int64_t)n1 * NB * c.ldb, c.ldb, Bj, c.ldb, 0));
    }
    solve_upper_rec(c, jb, n1);
}

// ------------------------------------------------------------------------------------------------
// vector triangular solves (m == 1): ONE kernel per sweep, block rows chained by flags (decoupled look-back)
// ------------------------------------------------------------------------------------------------
// In-place blocked TRSV.  Round 1 used two launches per 128-block (628 dependent launches for the two sweeps at n =
// 20 000: 4.2 ms for 3.2 GB of traffic).  Here a sweep is one kernel of one CTA per 128-block row:
//   forward  (L x = b):   CTA i:  x_i = invd_i (b_i / s_i - sum_{j < i} L_ij x_j)
//   backward (L^T x = y): CTA i:  x_i = invd_i^T (y_i - sum_{j > i} L_ji^T x_j) / s_i
// CTA i streams its block row (column) of L as the x_j become available, so that when x_{i-1} (x_{i+1}) is published
// only one 128 x 128 product, prefetched into shared memory, and the product with the inverted diagonal block, prefetched
// into registers, remain on the chain.  Block rows are handed out through an atomic ticket in dependency order, so a CTA
// only ever waits for CTAs that are already running: no co-residency requirement, no cooperative launch.  Flags carry
// the epoch of the launch and the ticket counter is never reset: nothing to clear between launches.
// `stride` is the element stride of the vector (a column of a row-major n x m matrix).
constexpr int TRSV_THREADS = 256;
constexpr int TRSV_SMEM_BYTES = NB * NB * 8 + (8 * NB + 2 * NB + 8) * 8;

__device__ __forceinline__ unsigned trsv_ld_acquire(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void trsv_st_release(unsigned *p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

struct TrsvArgs {
    const double *W;
    int64_t ldw;
    const double *invd;
    const double *sinv;  // 1/s (nullptr: no scaling)
    const double *svec;  // s: the backward sweep publishes x = z / s and its consumers need z = x s (exact: powers of two)
    double *b;
    int64_t stride;
    int n, nblk;
    unsigned long long *counter;
    unsigned long long base;
    unsigned *flags;
    unsigned epoch;
};

template <bool TRANS>
__global__ void __launch_bounds__(TRSV_THREADS, 1) trsv_sweep_kernel(const TrsvArgs a) {
    extern __shared__ __align__(16) double tsm[];
    double *Lbuf = tsm;                 // the last block of the chain: L_{i,i-1} (forward) / L_{i+1,i} (backward)
    double *part = Lbuf + NB * NB;      // [8][128] partial sums
    double *rhs = part + 8 * NB;        // [128]
    double *xs = rhs + NB;              // [128]
    int *ish = reinterpret_cast<int *>(xs + NB);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) ish[0] = (int)(atomicAdd(a.counter, 1ULL) - a.base);
    __syncthreads();
    const int ticket = ish[0];
    const int i = TRANS ? a.nblk - 1 - ticket : ticket;
    const int i0 = i * NB;
    const double *invd = a.invd + (int64_t)i * NB * NB;
    const int nchain = TRANS ? a.nblk - 1 - i : i;  // number of blocks x_j this CTA consumes

    // ---- prefetch: the chain's last block into shared memory, the inverted diagonal block into registers
    if (nchain > 0) {
        const double *Lp = TRANS ? a.W + (int64_t)(i0 + NB) * a.ldw + i0 : a.W + (int64_t)i0 * a.ldw + (i0 - NB);
        for (int ch = tid; ch < NB * NB / 2; ch += TRSV_THREADS) {
            const int r = ch >> 6, c2 = ch & 63;
            cp_async16(smem_u32(Lbuf + r * NB + 2 * c2), Lp + (int64_t)r * a.ldw + 2 * c2, 16);
        }
    }
    cp_async_commit();
    // forward: warp w owns rows 16w..16w+15, lanes along k (k = lane + 32 q); backward: thread (c4 = 4 lane, g = warp)
    // owns columns c4..c4+3 and rows 16g..16g+15 of every block
    double dv[16][4];
    if (!TRANS) {
#pragma unroll
        for (int r = 0; r < 16; r++)
#pragma unroll
            for (int q = 0; q < 4; q++) dv[r][q] = invd[(16 * warp + r) * NB + lane + 32 * q];
    } else {
#pragma unroll
        for (int r = 0; r < 16; r++) {
            const double4 v = *reinterpret_cast<const double4 *>(invd + (16 * warp + r) * NB + 4 * lane);
            dv[r][0] = v.x, dv[r][1] = v.y, dv[r][2] = v.z, dv[r][3] = v.w;
        }
    }
    // own right-hand side (forward: scaled by 1/s)
    if (tid < NB) {
        const int g = i0 + tid;
        double v = (g < a.n) ? a.b[(int64_t)g * a.stride] : 0.0;
        if (!TRANS && a.sinv && g < a.n) v *= a.sinv[g];
        rhs[tid] = v;
    }

    double acc[16];
#pragma unroll
    for (int r = 0; r < 16; r++) acc[r] = 0.0;
    // one block of the chain: forward acc[r] (row 16 warp + r, partial over this lane's 4 columns) += L[r][4 lane..] . x;
    // backward acc[0..3] (columns 4 lane.., partial over rows 16 warp..) += L[r][c] x[r]
    auto block_product = [&](const double *Lp, int64_t ldl, int j0) {
        if (!TRANS) {
            double xv[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int g = j0 + 4 * lane + q;
                xv[q] = (g < a.n) ? __ldcg(a.b + (int64_t)g * a.stride) : 0.0;
            }
#pragma unroll
            for (int h = 0; h < 2; h++) {  // eight 32-byte loads in flight
                double4 l[8];
#pragma unroll
                for (int r = 0; r < 8; r++)
                    l[r] = *reinterpret_cast<const double4 *>(Lp + (int64_t)(16 * warp + 8 * h + r) * ldl + 4 * lane);
#pragma unroll
                for (int r = 0; r < 8; r++)
                    acc[8 * h + r] += l[r].x * xv[0] + l[r].y * xv[1] + l[r].z * xv[2] + l[r].w * xv[3];
            }
        } else {
            double xv[16];
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const int g = j0 + 16 * warp + r;
                xv[r] = (g < a.n) ? __ldcg(a.b + (int64_t)g * a.stride) : 0.0;
                if (a.svec && g < a.n) xv[r] *= a.svec[g];
            }
#pragma unroll
            for (int h = 0; h < 2; h++) {
                double4 l[8];
#pragma unroll
                for (int r = 0; r < 8; r++)
                    l[r] = *reinterpret_cast<const double4 *>(Lp + (int64_t)(16 * warp + 8 * h + r) * ldl + 4 * lane);
#pragma unroll
                for (int r = 0; r < 8; r++) {
                    acc[0] += l[r].x * xv[8 * h + r];
                    acc[1] += l[r].y * xv[8 * h + r];
                    acc[2] += l[r].z * xv[8 * h + r];
                    acc[3] += l[r].w * xv[8 * h + r];
                }
            }
        }
    };

    // ---- the chain: blocks in dependency order (forward j = 0..i-1, backward j = nblk-1..i+1), the last one from Lbuf
    int done = 0;  // blocks consumed; `ready` of them are known to be published
    int ready = 0;
    while (done < nchain) {
        if (ready == done) {
            if (tid == 0) {
                int k = done;
                // wait for the next one, then take every further one that is already there
                while (trsv_ld_acquire(a.flags + (TRANS ? a.nblk - 1 - k : k)) != a.epoch) __nanosleep(32);
                k++;
                while (k < nchain && trsv_ld_acquire(a.flags + (TRANS ? a.nblk - 1 - k : k)) == a.epoch) k++;
                ish[1] = k;
            }
            __syncthreads();
            ready = ish[1];
            __syncthreads();
        }
        for (; done < ready; done++) {
            const int j = TRANS ? a.nblk - 1 - done : done;
            if (done == nchain - 1) {
                cp_async_wait<0>();
                __syncthreads();
                block_product(Lbuf, NB, j * NB);
            } else {
                const double *Lp = TRANS ? a.W + (int64_t)j * NB * a.ldw + i0 : a.W + (int64_t)i0 * a.ldw + (int64_t)j * NB;
                block_product(Lp, a.ldw, j * NB);
            }
        }
    }

    // ---- rhs - sum, then the product with the inverted diagonal block
    if (!TRANS) {
        double mine = 0.0;  // lane r keeps the sum of row 16 warp + r
#pragma unroll
        for (int r = 0; r < 16; r++) {
            const double s = warp_sum(acc[r]);
            if (lane == r) mine = s;
        }
        __syncthreads();  // rhs is complete
        if (lane < 16) rhs[16 * warp + lane] -= mine;
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 16; r++) {
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < 4; q++) s += dv[r][q] * rhs[lane + 32 * q];  // invd is zero above the diagonal
            s = warp_sum(s);
            if (lane == r) mine = s;
        }
        if (lane < 16) {
            const int g = i0 + 16 * warp + lane;
            if (g < a.n) a.b[(int64_t)g * a.stride] = mine;
        }
    } else {
#pragma unroll
        for (int q = 0; q < 4; q++) part[warp * NB + 4 * lane + q] = acc[q];
        __syncthreads();
        if (tid < NB) {
            double s = 0.0;
#pragma unroll
            for (int g = 0; g < 8; g++) s += part[g * NB + tid];
            rhs[tid] -= s;
        }
        __syncthreads();
        // x[c] = sum_k invd[k][c] rhs[k]  (invd is zero above the diagonal)
        double s4[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int r = 0; r < 16; r++) {
            const double y = rhs[16 * warp + r];
#pragma unroll
            for (int q = 0; q < 4; q++) s4[q] += dv[r][q] * y;
        }
#pragma unroll
        for (int q = 0; q < 4; q++) part[warp * NB + 4 * lane + q] = s4[q];
        __syncthreads();
        if (tid < NB) {
            double s = 0.0;
#pragma unroll
            for (int g = 0; g < 8; g++) s += part[g * NB + tid];
            const int g = i0 + tid;
            if (g < a.n) a.b[(int64_t)g * a.stride] = a.sinv ? s * a.sinv[g] : s;
        }
    }
    __syncthreads();
    // (st.release.gpu orders the stores of the whole CTA, which thread 0 has observed through the barrier, before the flag)
    if (tid == 0) trsv_st_release(a.flags + i, a.epoch);
}

// Flag workspace of the sweeps: one slot per (device, caller stream), allocated once; the host side hands out epochs and
// ticket bases under the lock that also covers the launch, so that they follow the stream order of the launches.
struct TrsvSlot {
    cudaStream_t caller;
    bool used;
    unsigned long long *counter;
    unsigned *flags;
    unsigned long long base;
    unsigned epoch;
};
constexpr int TRSV_SLOTS = 128;  // (torch hands out at most 65 stream handles per device: default + 2 pools of 32)
constexpr int TRSV_MAX_BLOCKS = 1 << 16;  // n up to 8.4 million

static int trsv_inplace(cudaStream_t st, const double *W, int64_t ldw, const double *invd, const double *sinv,
                        const double *svec, int n, double *b, int64_t stride, int trans) {
    static std::mutex mu;
    static TrsvSlot pools[MAX_DEVICES][TRSV_SLOTS];
    static DeviceOnce attr;
    const int nblk = (n + NB - 1) / NB;
    if (nblk > TRSV_MAX_BLOCKS) return LGP_ERR_UNSUPPORTED;
    if ((ldw & 1) || (reinterpret_cast<uintptr_t>(W) & 15) || (reinterpret_cast<uintptr_t>(invd) & 15)) return LGP_ERR_ALIGN;
    const int dev = current_device();
    if (dev < 0 || dev >= MAX_DEVICES) return LGP_ERR_CUDA;
    std::lock_guard<std::mutex> lock(mu);
    if (!attr.done(dev)) {
        if (cudaFuncSetAttribute(trsv_sweep_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TRSV_SMEM_BYTES) !=
                cudaSuccess ||
            cudaFuncSetAttribute(trsv_sweep_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TRSV_SMEM_BYTES) !=
                cudaSuccess)
            return LGP_ERR_CUDA;
        attr.set(dev);
    }
    TrsvSlot *slot = nullptr, *free_slot = nullptr;
    for (int k = 0; k < TRSV_SLOTS; k++) {
        TrsvSlot &s = pools[dev][k];
        if (s.used && s.caller == st) {
            slot = &s;
            break;
        }
        if (!s.used && !free_slot) free_slot = &s;
    }
    if (!slot) {
        if (!free_slot) return LGP_ERR_UNSUPPORTED;  // more than 128 distinct caller streams on one device
        void *p = nullptr;
        const size_t bytes = 256 + (size_t)TRSV_MAX_BLOCKS * sizeof(unsigned);
        if (cudaMalloc(&p, bytes) != cudaSuccess) return LGP_ERR_CUDA;
        // cleared in stream order: cudaMemset runs on the NULL stream, which a non-blocking caller stream does not wait for
        if (cudaMemsetAsync(p, 0, bytes, st) != cudaSuccess) return LGP_ERR_CUDA;
        slot = free_slot;
        slot->caller = st;
        slot->used = true;
        slot->counter = static_cast<unsigned long long *>(p);
        slot->flags = reinterpret_cast<unsigned *>(static_cast<char *>(p) + 256);
        slot->base = 0;
        slot->epoch = 0;
    }
    if (++slot->epoch == 0) {
        // the 32-bit epoch wrapped: flags of 2^32 launches ago could alias; clear them (stream-ordered)
        if (cudaMemsetAsync(slot->flags, 0, (size_t)TRSV_MAX_BLOCKS * sizeof(unsigned), st) != cudaSuccess) return LGP_ERR_CUDA;
        slot->epoch = 1;
    }
    TrsvArgs a{W, ldw, invd, sinv, svec, b, stride, n, nblk, slot->counter, slot->base, slot->flags, slot->epoch};
    slot->base += (unsigned long long)nblk;
    if (trans)
        trsv_sweep_kernel<true><<<nblk, TRSV_THREADS, TRSV_SMEM_BYTES, st>>>(a);
    else
        trsv_sweep_kernel<false><<<nblk, TRSV_THREADS, TRSV_SMEM_BYTES, st>>>(a);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

__global__ void vec_scale_copy_kernel(const double *__restrict__ src, int64_t stride, double *__restrict__ dst, int n,
                                      const double *__restrict__ f) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[(int64_t)i * stride] * (f ? f[i] : 1.0);
}

// X = Lt^-1 (lower) out of place into X (ld = ldx); the strict upper triangle of X is scratch.
struct InvCtx {
    cudaStream_t st;
    const double *W;
    int64_t ldw;
    const double *invd;
    double *X;
    int64_t ldx;
    int rc;
};
// The two halves of a node are independent until its two combining products: down to TRTRI_FORK_DEPTH the right half
// runs on a side stream, so that the small, latency-bound products near the leaves of different subtrees overlap and
// fill the GPU (the recursion issues ~3 launches per 128-block, strictly ordered on a single stream otherwise).
constexpr int TRTRI_FORK_DEPTH = 4;
static cudaStream_t trtri_side_stream(int idx) {
    static std::mutex mu;
    static cudaStream_t pools[MAX_DEVICES][1 << TRTRI_FORK_DEPTH];
    static bool inits[MAX_DEVICES][1 << TRTRI_FORK_DEPTH];
    const int dev = current_device();
    if (dev < 0) return nullptr;
    std::lock_guard<std::mutex> lock(mu);
    if (!inits[dev][idx]) {
        if (cudaStreamCreateWithFlags(&pools[dev][idx], cudaStreamNonBlocking) != cudaSuccess) pools[dev][idx] = nullptr;
        inits[dev][idx] = true;
    }
    return pools[dev][idx];
}

static void trtri_rec(InvCtx &c, int jb, int nb, int depth = 0, int path = 1) {
    if (c.rc) return;
    if (nb == 1) {
        dim3 g((NB + 127) / 128, NB);
        copy_block_kernel<<<g, 128, 0, c.st>>>(c.invd + (int64_t)jb * NB * NB, NB,
                                               c.X + (int64_t)jb * NB * c.ldx + (int64_t)jb * NB, c.ldx, NB, NB);
        count_launch();
        if (cudaGetLastError() != cudaSuccess) c.rc = LGP_ERR_CUDA;
        return;
    }
    int n1 = nb / 2, n2 = nb - n1;
    cudaStream_t side = (depth < TRTRI_FORK_DEPTH && nb >= 4) ? trtri_side_stream(path) : nullptr;
    if (side) {
        // fork: if the ordering cannot be enqueued, the right half simply stays on this stream
        cudaEvent_t fork = ring_event();
        if (!(ev_record(fork, c.st) && ev_wait(side, fork))) side = nullptr;
    }
    if (side) {
        InvCtx cs = c;
        cs.st = side;
        trtri_rec(c, jb, n1, depth + 1, 2 * path);
        trtri_rec(cs, jb + n1, n2, depth + 1, 2 * path + 1);
        cudaEvent_t join = ring_event();
        if (!(ev_record(join, side) && ev_wait(c.st, join))) {
            cudaStreamSynchronize(side);  // never let the combining products overtake the side stream
            c.rc = LGP_ERR_CUDA;
        }
        if (cs.rc) c.rc = cs.rc;
    } else {
        trtri_rec(c, jb, n1, depth + 1, 2 * path);
        trtri_rec(c, jb + n1, n2, depth + 1, 2 * path + 1);
    }
    if (c.rc) return;
    const double *L21 = c.W + (int64_t)(jb + n1) * NB * c.ldw + (int64_t)jb * NB;
    double *X11 = c.X + (int64_t)jb * NB * c.ldx + (int64_t)jb * NB;
    double *X22 = c.X + (int64_t)(jb + n1) * NB * c.ldx + (int64_t)(jb + n1) * NB;
    double *X21 = c.X + (int64_t)(jb + n1) * NB * c.ldx + (int64_t)jb * NB;
    double *Tt = c.X + (int64_t)jb * NB * c.ldx + (int64_t)(jb + n1) * NB;  // n1 x n2 scratch (upper block)
    // Tt[j][i] = sum_k X11[k][j] * L21[i][k]   (k >= j)
    RC(gemm_launch(c.st, false, true, n1 * NB, n2 * NB, n1 * NB, 1.0, X11, c.ldx, L21, c.ldw, Tt, c.ldx,
                   GEMM_BETA0 | GEMM_A_UPPER_K));
    // X21[i][j] = - sum_k X22[i][k] * Tt[j][k]  (k <= i)
    RC(gemm_launch(c.st, true, true, n2 * NB, n1 * NB, n2 * NB, -1.0, X22, c.ldx, Tt, c.ldx, X21, c.ldx,
                   GEMM_BETA0 | GEMM_A_LOWER_K));
}

}  // namespace lgp

using namespace lgp;

extern "C" {

int64_t lgp_chol_npad(int64_t n) { return (n + NB - 1) / NB * NB; }
int64_t lgp_chol_aux_doubles(int64_t n) {
    int64_t npad = lgp_chol_npad(n);
    return 3 * npad + 16 + (npad / NB) * (int64_t)NB * NB;
}

// `prepared`: W already holds the equilibrated lower triangle with identity padding, aux the scales and, in scalar 0, the
// Gershgorin bound (lgp_gram_iso_prepare): the two passes over K are skipped
static int chol_factor_impl(lgp_stream_t stream, bool prepared, const double *K, int64_t ldk, const double *addmat,
                            int64_t ldadd, const double *adddiag, int64_t n64, double epsrel, double epsabs, double *W,
                            int64_t ldw, double *aux, int32_t *info) {
    if (n64 < 1 || n64 > (1 << 30) || (!prepared && !K) || !W || !aux || !info) return LGP_ERR_BADARG;
    const int n = (int)n64, npad = (int)lgp_chol_npad(n);
    if (ldw < npad || (!prepared && (ldk < n || (addmat && ldadd < n)))) return LGP_ERR_BADARG;
    if ((ldw & 1) || (reinterpret_cast<uintptr_t>(W) & 15) || (reinterpret_cast<uintptr_t>(aux) & 15))
        return LGP_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    if (leaf_attr()) return LGP_ERR_CUDA;
    if (epsrel < 0) epsrel = (double)n * 2.220446049250313e-16;
    if (!prepared) {
        chol_diag_scale_kernel<<<(npad + 255) / 256, 256, 0, st>>>(K, ldk, addmat, ldadd, adddiag, n, npad, aux);
        LGP_CUDA_CHECK_LAUNCH();
        chol_prepare_kernel<<<(npad + 7) / 8, 256, 0, st>>>(K, ldk, addmat, ldadd, adddiag, n, npad, W, ldw, aux);
        LGP_CUDA_CHECK_LAUNCH();
    }
    chol_jitter_kernel<<<1, 1024, 0, st>>>(n, npad, epsrel, epsabs, W, ldw, aux, info);
    LGP_CUDA_CHECK_LAUNCH();
    CholCtx c{st, W, ldw, aux + LGP_AUX_INVDIAG(npad), aux + LGP_AUX_DIAG(npad), info, LGP_OK};
    {
        int rc = potrf_lookahead(c, npad / NB, panel_blocks());
        if (rc) return rc;
    }
    finalize_info_kernel<<<1, 1, 0, st>>>(info, n);
    LGP_CUDA_CHECK_LAUNCH();
    logdet_quad_kernel<<<1, 1024, 0, st>>>(aux + LGP_AUX_DIAG(npad), aux + LGP_AUX_S(npad), nullptr, n,
                                           aux + LGP_AUX_SCALARS(npad) + 4);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

int lgp_chol_factor(lgp_stream_t stream, const double *K, int64_t ldk, const double *addmat, int64_t ldadd,
                    const double *adddiag, int64_t n, double epsrel, double epsabs, double *W, int64_t ldw, double *aux,
                    int32_t *info) {
    return chol_factor_impl(stream, false, K, ldk, addmat, ldadd, adddiag, n, epsrel, epsabs, W, ldw, aux, info);
}
int lgp_chol_factor_prepared(lgp_stream_t stream, int64_t n, double epsrel, double epsabs, double *W, int64_t ldw,
                             double *aux, int32_t *info) {
    return chol_factor_impl(stream, true, nullptr, 0, nullptr, 0, nullptr, n, epsrel, epsabs, W, ldw, aux, info);
}

// debug/benchmark hook (not in the public header): run the 128x128 leaf `reps` times back to back
int lgp_debug_leaf(lgp_stream_t stream, double *Wblk, int64_t ld, double *invd, double *dvec, int32_t *info, int reps) {
    if (leaf_attr()) return LGP_ERR_CUDA;
    for (int i = 0; i < reps; i++) leaf_launch((cudaStream_t)stream, Wblk, ld, invd, dvec, info, 0);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

// debug hook: phase timestamps (SM clock cycles) of the last leaf-3 launch
int lgp_debug_leaf3_clocks(long long *out32) {
    return cudaMemcpyFromSymbol(out32, l3_dbg, 32 * sizeof(long long)) == cudaSuccess ? LGP_OK : LGP_ERR_CUDA;
}

int lgp_chol_solve(lgp_stream_t stream, const double *W, int64_t ldw, const double *aux, int64_t n64, double *B,
                   int64_t ldb, int64_t m64, int trans) {
    if (n64 < 1 || m64 < 1 || !W || !aux || !B) return LGP_ERR_BADARG;
    const int n = (int)n64, m = (int)m64, npad = (int)lgp_chol_npad(n);
    if ((ldb & 1) || (reinterpret_cast<uintptr_t>(B) & 15)) return LGP_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    const double *sinv = aux + LGP_AUX_SINV(npad);
    int64_t total = (int64_t)n * m;
    if (m == 1) return trsv_inplace(st, W, ldw, aux + LGP_AUX_INVDIAG(npad), sinv, aux + LGP_AUX_S(npad), n, B, ldb, trans);
    SolveCtx c{st, W, ldw, aux + LGP_AUX_INVDIAG(npad), n, B, ldb, m, LGP_OK};
    if (!trans) {
        row_scale_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(B, ldb, n, m, sinv);
        LGP_CUDA_CHECK_LAUNCH();
        solve_lower_rec(c, 0, npad / NB);
    } else {
        solve_upper_rec(c, 0, npad / NB);
        if (c.rc) return c.rc;
        row_scale_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(B, ldb, n, m, sinv);
        LGP_CUDA_CHECK_LAUNCH();
    }
    return c.rc;
}

int lgp_chol_mult(lgp_stream_t stream, const double *W, int64_t ldw, const double *aux, int64_t n64, const double *X,
                  int64_t ldx, int64_t m64, double *Y, int64_t ldy, double *tmp, int64_t ldt, int trans) {
    if (n64 < 1 || m64 < 1 || !W || !aux || !X || !Y) return LGP_ERR_BADARG;
    const int n = (int)n64, m = (int)m64, npad = (int)lgp_chol_npad(n);
    cudaStream_t st = (cudaStream_t)stream;
    const double *s = aux + LGP_AUX_S(npad);
    int64_t total = (int64_t)n * m;
    int rc;
    if (!trans) {
        // Y = S (Lt X): Aop[i][k] = Lt[i][k] (k <= i), Bop[j][k] = X[k][j]
        rc = gemm_launch(st, true, false, n, m, n, 1.0, W, ldw, X, ldx, Y, ldy, GEMM_BETA0 | GEMM_A_LOWER_K);
        if (rc) return rc;
        row_scale_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(Y, ldy, n, m, s);
        LGP_CUDA_CHECK_LAUNCH();
    } else {
        // Y = Lt^T (S X): tmp = S X, then Aop[i][k] = Lt[k][i] (k >= i)
        if (!tmp) return LGP_ERR_BADARG;
        row_scale_copy_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(X, ldx, tmp, ldt, n, m, s);
        LGP_CUDA_CHECK_LAUNCH();
        rc = gemm_launch(st, false, false, n, m, n, 1.0, W, ldw, tmp, ldt, Y, ldy, GEMM_BETA0 | GEMM_A_UPPER_K);
        if (rc) return rc;
    }
    return LGP_OK;
}

int lgp_chol_get_factor(lgp_stream_t stream, const double *W, int64_t ldw, const double *aux, int64_t n64,
                        double *Lout, int64_t ldl) {
    if (n64 < 1 || !W || !aux || !Lout) return LGP_ERR_BADARG;
    const int n = (int)n64, npad = (int)lgp_chol_npad(n);
    dim3 g = rows_grid(n, n);
    get_factor_kernel<<<g, 256, 0, (cudaStream_t)stream>>>(W, ldw, aux + LGP_AUX_S(npad), n, Lout, ldl);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

// X = Lt^-1 into scratch (TRTRI), then Kinv = X^T X with the equilibration undone (LAUUM), on `st`
static int chol_inverse_impl(cudaStream_t st, const double *W, int64_t ldw, const double *aux, int npad, double *scratch,
                             double *Kinv, int64_t ldk) {
    InvCtx c{st, W, ldw, aux + LGP_AUX_INVDIAG(npad), scratch, (int64_t)npad, LGP_OK};
    const bool trace = trace_enabled();
    cudaEvent_t t0, t1, t2;
    if (trace) {
        cudaEventCreate(&t0); cudaEventCreate(&t1); cudaEventCreate(&t2);
        cudaEventRecord(t0, st);
    }
    trtri_rec(c, 0, npad / NB);
    if (c.rc) return c.rc;
    if (trace) cudaEventRecord(t1, st);
    // Kinv[i][j] = sum_{k >= i} X[k][i] X[k][j] / (s_i s_j), j <= i   (LAUUM as one triangular-K SYRK launch; the
    // equilibration scales are applied in its epilogue: exact, powers of two)
    int rc = gemm_launch(st, false, false, npad, npad, npad, 1.0, scratch, npad, scratch, npad, Kinv, ldk,
                         GEMM_BETA0 | GEMM_LOWER | GEMM_A_UPPER_K, nullptr, aux + LGP_AUX_SINV(npad));
    if (rc) return rc;
    if (trace) {
        cudaEventRecord(t2, st);
        cudaEventSynchronize(t2);
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, t0, t1);
        cudaEventElapsedTime(&b, t1, t2);
        fprintf(stderr, "[lgp trace] inverse: trtri %.3f ms, lauum+scale %.3f ms\n", a, b);
        cudaEventDestroy(t0); cudaEventDestroy(t1); cudaEventDestroy(t2);
    }
    return LGP_OK;
}

int lgp_chol_inverse(lgp_stream_t stream, const double *W, int64_t ldw, const double *aux, int64_t n64,
                     double *scratch, double *Kinv, int64_t ldk) {
    if (n64 < 1 || !W || !aux || !scratch || !Kinv) return LGP_ERR_BADARG;
    const int n = (int)n64, npad = (int)lgp_chol_npad(n);
    if (ldk < npad) return LGP_ERR_BADARG;
    if ((ldk & 1) || (reinterpret_cast<uintptr_t>(Kinv) & 15) || (reinterpret_cast<uintptr_t>(scratch) & 15))
        return LGP_ERR_ALIGN;
    return chol_inverse_impl((cudaStream_t)stream, W, ldw, aux, npad, scratch, Kinv, ldk);
}

// ---- factorisation and inverse-from-factor in one call: the inverse runs on `inv_stream` behind the complete factor
static int chol_factor_inverse_impl(lgp_stream_t stream, lgp_stream_t inv_stream, bool prepared, const double *K,
                                    int64_t ldk, const double *addmat, int64_t ldadd, const double *adddiag, int64_t n64,
                                    double epsrel, double epsabs, double *W, int64_t ldw, double *aux, int32_t *info,
                                    double *scratch, double *Kinv, int64_t ldkinv) {
    const int64_t npad = lgp_chol_npad(n64);
    if (!scratch || !Kinv || ldkinv < npad) return LGP_ERR_BADARG;
    if ((ldkinv & 1) || (reinterpret_cast<uintptr_t>(Kinv) & 15) || (reinterpret_cast<uintptr_t>(scratch) & 15))
        return LGP_ERR_ALIGN;
    int rc = chol_factor_impl(stream, prepared, K, ldk, addmat, ldadd, adddiag, n64, epsrel, epsabs, W, ldw, aux, info);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream, si = (cudaStream_t)inv_stream;
    if (si != st) {
        cudaEvent_t e = ring_event();
        if (!(ev_record(e, st) && ev_wait(si, e))) {
            cudaStreamSynchronize(st);  // ordering could not be enqueued: fall back to a host-side join
        }
    }
    return chol_inverse_impl(si, W, ldw, aux, (int)npad, scratch, Kinv, ldkinv);
}

int lgp_chol_factor_inverse(lgp_stream_t stream, lgp_stream_t inv_stream, const double *K, int64_t ldk,
                            const double *addmat, int64_t ldadd, const double *adddiag, int64_t n, double epsrel,
                            double epsabs, double *W, int64_t ldw, double *aux, int32_t *info, double *scratch,
                            double *Kinv, int64_t ldkinv) {
    return chol_factor_inverse_impl(stream, inv_stream, false, K, ldk, addmat, ldadd, adddiag, n, epsrel, epsabs, W, ldw,
                                    aux, info, scratch, Kinv, ldkinv);
}
int lgp_chol_factor_inverse_prepared(lgp_stream_t stream, lgp_stream_t inv_stream, int64_t n, double epsrel, double epsabs,
                                     double *W, int64_t ldw, double *aux, int32_t *info, double *scratch, double *Kinv,
                                     int64_t ldkinv) {
    return chol_factor_inverse_impl(stream, inv_stream, true, nullptr, 0, nullptr, 0, nullptr, n, epsrel, epsabs, W, ldw,
                                    aux, info, scratch, Kinv, ldkinv);
}

// ---- tile-level entry points: building blocks of the block-cyclic multi-GPU factorisation (lsqfitgp_b200/_dist.py)
int lgp_tile_potrf(lgp_stream_t stream, double *A, int64_t lda, int64_t t, double *invd, double *dvec, int32_t *info,
                   int64_t j0) {
    if (t < NB || t % NB || t > (1 << 20) || !A || !invd || !dvec || !info || j0 < 0) return LGP_ERR_BADARG;
    if ((lda & 1) || (reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(invd) & 15))
        return LGP_ERR_ALIGN;
    if (leaf_attr()) return LGP_ERR_CUDA;
    CholCtx c{(cudaStream_t)stream, A, lda, invd, dvec, info, LGP_OK};
    c.j0base = (int)j0;
    potrf_rec(c, 0, (int)(t / NB));
    return c.rc;
}

int lgp_tile_trsm_right(lgp_stream_t stream, const double *L, int64_t ldl, const double *invd, int64_t t, double *B,
                        int64_t ldb, int64_t rows) {
    if (t < NB || t % NB || rows < 0 || rows > (1 << 30) || !L || !invd || !B) return LGP_ERR_BADARG;
    if (rows == 0) return LGP_OK;
    CholCtx c{(cudaStream_t)stream, nullptr, 0, nullptr, nullptr, nullptr, LGP_OK};
    trsm_right_ptr(c, B, ldb, (int)rows, L, ldl, invd, (int)(t / NB));
    return c.rc;
}

int lgp_tile_trsm_right_bcast(lgp_stream_t stream, const double *L, int64_t ldl, const double *invd, int64_t t, double *B,
                              int64_t ldb, int64_t rows, int n_dst, void *const *dst, int64_t ld_dst, int multimem) {
    if (t < NB || t % NB || rows < 0 || rows > (1 << 30) || !L || !invd || !B) return LGP_ERR_BADARG;
    if (n_dst < 0 || n_dst > GEMM_MAX_MIRRORS || (n_dst && (!dst || ld_dst < t)) || (multimem && n_dst != 1))
        return LGP_ERR_BADARG;
    if (rows == 0) return LGP_OK;
    CholCtx c{(cudaStream_t)stream, nullptr, 0, nullptr, nullptr, nullptr, LGP_OK};
    c.mir.n = n_dst;
    c.mir.multimem = multimem ? 1 : 0;
    c.mir.ld = ld_dst;
    for (int i = 0; i < n_dst; i++) {
        if (!dst[i]) return LGP_ERR_BADARG;
        c.mir.dst[i] = (double *)dst[i];
    }
    trsm_right_ptr(c, B, ldb, (int)rows, L, ldl, invd, (int)(t / NB));
    return c.rc;
}

// ---- cross-GPU flags (monotone counters in peer-mapped memory) ordering the peer stores above against their readers
__global__ void flag_signal_kernel(FlagPtrs f, unsigned long long value) {
    const int i = threadIdx.x;
    if (i < f.n) {
        __threadfence_system();  // stores of the preceding kernels of this stream (kernel boundary) before the flag
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(f.p[i]), "l"(value) : "memory");
    }
}

__global__ void flag_wait_kernel(const unsigned long long *flags, int n, unsigned long long value,
                                 unsigned long long timeout_ns, int *err) {
    const int i = threadIdx.x;
    if (i >= n) return;
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + i) : "memory");
        if (v >= value) break;
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > timeout_ns) {
            atomicExch(err, 1);  // the caller checks this flag: never spin forever on a peer that will not arrive
            break;
        }
        __nanosleep(200);
    }
}

int lgp_flag_signal(lgp_stream_t stream, void *const *flag_ptrs, int n, uint64_t value) {
    if (n < 0 || n > LGP_MAX_FLAGS || (n && !flag_ptrs)) return LGP_ERR_BADARG;
    if (n == 0) return LGP_OK;
    FlagPtrs f;
    f.n = n;
    for (int i = 0; i < n; i++) {
        if (!flag_ptrs[i] || (reinterpret_cast<uintptr_t>(flag_ptrs[i]) & 7)) return LGP_ERR_BADARG;
        f.p[i] = (unsigned long long *)flag_ptrs[i];
    }
    flag_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(f, (unsigned long long)value);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

int lgp_flag_wait(lgp_stream_t stream, const uint64_t *flags, int n, uint64_t value, int64_t timeout_ms, int32_t *err) {
    if (n < 0 || n > LGP_MAX_FLAGS || (n && !flags) || !err || timeout_ms < 0) return LGP_ERR_BADARG;
    if (n == 0) return LGP_OK;
    flag_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const unsigned long long *)flags, n, (unsigned long long)value,
                                                         (unsigned long long)timeout_ms * 1000000ull, err);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

int lgp_tile_trsv(lgp_stream_t stream, const double *L, int64_t ldl, const double *invd, int64_t t, double *b,
                  int trans) {
    if (t < NB || t % NB || !L || !invd || !b) return LGP_ERR_BADARG;
    return trsv_inplace((cudaStream_t)stream, L, ldl, invd, nullptr, nullptr, (int)t, b, 1, trans);
}

int lgp_chol_logdet_quad(lgp_stream_t stream, const double *aux, int64_t n64, const double *a, double *out) {
    if (n64 < 1 || !aux || !out) return LGP_ERR_BADARG;
    const int n = (int)n64, npad = (int)lgp_chol_npad(n);
    logdet_quad_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(aux + LGP_AUX_DIAG(npad), aux + LGP_AUX_S(npad), a, n,
                                                             out);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

}  // extern "C"
