// 128x128 Cholesky leaf, version 3: Cholesky factor AND its inverse of one diagonal block in one CTA.
//
// Reads the lower triangle of Wblk, writes L into the lower triangle
// (zeros above), X = L^-1 into invd (row-major 128 x 128, zeros above the diagonal), dvec[j0 + k] = L_kk, and
// atomicMin(info, j0 + k + 1) at the first non-positive / non-finite pivot (NaNs then propagate like a failed
// LAPACK/JAX factorisation, reference _linalg/_decomp.py:388-391).
//
// Versions 1 (unblocked, 128 CTA-wide rank-1 steps of ~1040 cycles) and 2 (blocked 4 x 32, one warp factoring the
// diagonal blocks with ~385 cycles per column while seven warps wait) both take 67-68 us.  What bounds a leaf is the
// chain of 128 dependent column steps, so version 3 is built around the chain:
//
//  * Augmented elimination: the combined array S holds A/L on and below the diagonal and Y = L^-T above it
//    (S[r][c] = X[c][r] for r < c).  Eliminating the columns of [A; I] turns the bottom block into L^-T, so one sweep of
//    four 32-column panels produces the factor and its inverse, and every row block of a panel is treated alike.
//  * Inside a panel the column steps run in LDL^T form: a step needs 1/pivot (hardware estimate + one third-order
//    step, 3 dependent DFMAs), not 1/sqrt(pivot) (~12); the square roots of the 32 pivots are taken once, in
//    parallel, after the last step, and every row is scaled then.  Step j of the chain warp (lane r = row r of the
//    diagonal block): publish a_rj to shared memory, read column j back (broadcast 16-byte loads), t_r = a_rj / a_jj,
//    a_rc -= t_r a_cj.  The entry of the next column is updated and published FIRST, the other 30 - j FMAs follow.
//  * The other four row blocks of the panel (the three off-diagonal blocks and the identity rows that become
//    L_JJ^-T) are four FOLLOWER warps, one row per lane, in lockstep with the chain warp: the chain warp publishes
//    t_cj = a_cj / a_jj per step behind a shared-memory mbarrier, a follower does p_rc -= p_rj t_cj.  The triangular
//    solves of the panel therefore cost nothing after the last column step.
//  * Rank-32 updates on the FP64 tensor pipe (DMMA 8x8x4 from shared memory, 16 independent accumulator tiles per warp).
//    Only the next panel's block column (4 blocks) is updated between two panels; the remaining blocks are done by the
//    three spare warps WHILE the next panel's chain runs.
//  * Measured on B200 (phase clocks, tools/bench_leaf.py): load 3.5k cycles, panels 7.0-8.7k each (~220 cycles per
//    column step), block-column updates 3.3k each (DMMA issue bound is 2k), stores 10k: 55k cycles = 28 us + launch.
#pragma once
#include "common.cuh"

namespace lgp {

constexpr int L3_B = 32;        // panel width
constexpr int L3_S = 133;       // row stride of S (odd: one row per lane is conflict-free)
constexpr int L3_XS = 33;       // row stride of the L_JJ^-T scratch blocks
constexpr int L3_THREADS = 256;
constexpr int L3_NSPARE = 3;    // warps 5..7
// S[128][133] | RAW[32][32] (column j of the diagonal block, unscaled) | TS[32][32] (column j / pivot) |
// XD[2][32][33] (L_JJ^-T, double-buffered) | RL[128] (1 / L_kk) | 32 mbarriers
constexpr int L3_OFF_RAW = 128 * L3_S;
constexpr int L3_OFF_TS = L3_OFF_RAW + L3_B * L3_B;
constexpr int L3_OFF_XD = L3_OFF_TS + L3_B * L3_B;
constexpr int L3_OFF_RL = L3_OFF_XD + 2 * L3_B * L3_XS;
constexpr int L3_OFF_BAR = L3_OFF_RL + 128;
constexpr int L3_SMEM_BYTES = (L3_OFF_BAR + 32) * 8;
static_assert(L3_OFF_RAW % 2 == 0 && L3_OFF_TS % 2 == 0, "16-byte alignment of the broadcast buffers");

__device__ __forceinline__ void l3_mbar_init(uint32_t a, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory");
}
__device__ __forceinline__ void l3_mbar_arrive(uint32_t a) {
    asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}" ::"r"(a) : "memory");
}
__device__ __forceinline__ void l3_mbar_wait(uint32_t a, uint32_t parity) {
    asm volatile(
        "{\n.reg .pred P1;\nL3_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra L3_DONE;\nbra "
        "L3_WAIT;\nL3_DONE:\n}" ::"r"(a),
        "r"(parity)
        : "memory");
}

// explicit shared-space accesses with a 32-bit address kept in a register (generic pointers made the compiler
// rematerialise the shared window base with an S2R in every column step)
__device__ __forceinline__ void l3_lds2(double &x, double &y, uint32_t a) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x), "=d"(y) : "r"(a) : "memory");
}
__device__ __forceinline__ void l3_sts(uint32_t a, double v) {
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory");
}

// 1/x from the hardware estimate (MUFU.RCP64H, ~2^-20) and one third-order step: y0 (1 + e + e^2), e = 1 - x y0, three
// dependent DFMAs, relative error ~2^-58.  No range test on the critical path: pivots of an equilibrated matrix are
// O(1); a pivot that is zero, negative or not finite is reported through `info` by its owner lane, a positive pivot
// below ~1e-300 (numerically singular beyond anything the jitter allows) turns the following columns into NaN and is
// reported at the next column.
__device__ __forceinline__ double l3_rcp(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x, y, 1.0);
    e = fma(e, e, e);
    return fma(y, e, y);
}

// sqrt(pv) and 1/sqrt(pv) to ~1 ulp from the hardware estimate: two Goldschmidt iterations and a Newton correction
// with the exact residual (cf. fastmath.cuh).  NaN for pv < 0, inf for pv == 0 through the library path.
__device__ __forceinline__ void l3_sqrt_rsqrt(double pv, double &l, double &rl) {
    if (pv >= 1e-280 && pv <= 1e280) {
        double y0;
        asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(pv));
        double g = pv * y0, h = 0.5 * y0;
        double r = fma(-h, g, 0.5);
        g = fma(g, r, g);
        h = fma(h, r, h);
        r = fma(-h, g, 0.5);
        g = fma(g, r, g);
        h = fma(h, r, h);
        l = fma(fma(-g, g, pv), h, g);
        rl = h + h;
        rl = fma(fma(-l, rl, 1.0), rl, rl);
    } else {
        rl = rsqrt(pv);
        l = pv * rl;
    }
}

// ---- chain warp: the 32 column steps of the diagonal block, lane r = row r (entries c <= r are meaningful) -----------
// One basic block per step (between two __syncwarp): mbarrier arrive for the followers, the broadcast loads of the next
// column, the 30 - j FMAs of the previous step, then pivot -> reciprocal -> t -> next-column entry -> the two stores.
// The compiler interleaves the independent FMAs with the dependent chain.
__device__ __forceinline__ void l3_chain(double (&a)[L3_B], uint32_t raw, uint32_t ts, double *__restrict__ rlbuf,
                                         uint32_t bar0, double *__restrict__ dvec, int32_t *__restrict__ info, int jglob,
                                         int lane, double &ldiag) {
    double mypv = 0.0;
    double u[L3_B];
    l3_sts(raw + 8 * lane, a[0]);
    __syncwarp();
#pragma unroll
    for (int c2 = 0; c2 < L3_B / 2; c2++) l3_lds2(u[2 * c2], u[2 * c2 + 1], raw + 16 * c2);
#pragma unroll
    for (int j = 0; j < L3_B; j++) {
        const double pv = u[j];
        if (lane == j) mypv = pv;
        if (j + 1 < L3_B) {
            const double rinv = l3_rcp(pv);
            const double t = a[j] * rinv;
            a[j + 1] = fma(-t, u[j + 1], a[j + 1]);
            l3_sts(raw + 8 * ((j + 1) * L3_B + lane), a[j + 1]);
            l3_sts(ts + 8 * (j * L3_B + lane), t);
            __syncwarp();
            if (lane == 0) l3_mbar_arrive(bar0 + 8 * j);  // TS row j is complete
            double un[L3_B];
#pragma unroll
            for (int c2 = (j + 1) / 2; c2 < L3_B / 2; c2++)
                l3_lds2(un[2 * c2], un[2 * c2 + 1], raw + 8 * ((j + 1) * L3_B + 2 * c2));
#pragma unroll
            for (int c = j + 2; c < L3_B; c++) a[c] = fma(-t, u[c], a[c]);
#pragma unroll
            for (int c = j + 1; c < L3_B; c++) u[c] = un[c];
        }
    }
    double rl;
    l3_sqrt_rsqrt(mypv, ldiag, rl);
    if (!(mypv > 0.0) || !(ldiag < INFINITY)) atomicMin(info, jglob + lane + 1);
    dvec[jglob + lane] = ldiag;
    rlbuf[lane] = rl;
    __syncwarp();
    if (lane == 0) l3_mbar_arrive(bar0 + 8 * (L3_B - 1));  // RL is complete
}

// ---- follower warp: one row of the panel per lane, p_c -= p_j t_cj behind the chain warp ---------------------------------
__device__ __forceinline__ void l3_follow(double (&p)[L3_B], uint32_t ts, uint32_t rlbuf, uint32_t bar0, uint32_t parity) {
#pragma unroll
    for (int j = 0; j + 1 < L3_B; j++) {
        l3_mbar_wait(bar0 + 8 * j, parity);
        const double pj = p[j];
#pragma unroll
        for (int c2 = (j + 1) / 2; c2 < L3_B / 2; c2++) {
            double vx, vy;
            l3_lds2(vx, vy, ts + 8 * (j * L3_B + 2 * c2));
            if (2 * c2 > j) p[2 * c2] = fma(-pj, vx, p[2 * c2]);
            p[2 * c2 + 1] = fma(-pj, vy, p[2 * c2 + 1]);
        }
    }
    l3_mbar_wait(bar0 + 8 * (L3_B - 1), parity);
#pragma unroll
    for (int c2 = 0; c2 < L3_B / 2; c2++) {
        double vx, vy;
        l3_lds2(vx, vy, rlbuf + 16 * c2);
        p[2 * c2] *= vx;
        p[2 * c2 + 1] *= vy;
    }
}

// ---- rank-32 update of a 32 x 16 half block on the FP64 tensor pipe:  C(r, c) -= sum_k A(r, k) B(c, k), k contiguous ----
// 16 independent accumulator tiles (4 row tiles x 2 column tiles x 2 halves of k): the warp is bound by the DMMA issue
// rate (64 DMMAs = 1024 cycles on its scheduler), not by the DMMA latency.
__device__ __forceinline__ void l3_unit(const double *__restrict__ pa, int sar, const double *__restrict__ pb, int sbr,
                                        double *__restrict__ pc, int scr, int lane) {
    const int lr = lane >> 2, q = lane & 3;
    double acc[2][4][2][2];
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int n = 0; n < 2; n++) acc[h][i][n][0] = acc[h][i][n][1] = 0.0;
#pragma unroll
    for (int s = 0; s < 4; s++) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int k0 = 16 * h + 4 * s;
            double af[4], bf[2];
#pragma unroll
            for (int n = 0; n < 2; n++) bf[n] = pb[(8 * n + lr) * sbr + k0 + q];
#pragma unroll
            for (int i = 0; i < 4; i++) af[i] = pa[(8 * i + lr) * sar + k0 + q];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int n = 0; n < 2; n++) dmma884(acc[h][i][n][0], acc[h][i][n][1], af[i], bf[n]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int n = 0; n < 2; n++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
                double *p = pc + (8 * i + lr) * scr + 8 * n + 2 * q + e;
                *p -= acc[0][i][n][e] + acc[1][i][n][e];
            }
}

// update of block (I, K), column half hf, from panel Js
__device__ __forceinline__ void l3_update_unit(double *__restrict__ S, const double *__restrict__ XD, int I, int K, int hf,
                                               int Js, int lane) {
    const double *pb = S + (K * L3_B + 16 * hf) * L3_S + Js * L3_B;
    double *pc = S + (I * L3_B) * L3_S + K * L3_B + 16 * hf;
    if (I == Js)
        l3_unit(XD + (Js & 1) * L3_B * L3_XS, L3_XS, pb, L3_S, pc, L3_S, lane);
    else
        l3_unit(S + (I * L3_B) * L3_S + Js * L3_B, L3_S, pb, L3_S, pc, L3_S, lane);
}

// Global stores of block column Jp: L[:, Jp] (zeros above the diagonal) and rows Jp of X = L^-1.  16-byte stores, two
// adjacent output entries per thread read from S with two 8-byte loads (odd row stride), eight in flight.  One SM moves
// ~25 bytes per cycle towards L2, so the 256 KB of output cost ~10 000 cycles whatever the instruction mix, and stores
// issued EARLY (block column J-1 during panel J, by the spare warps or by the bulk-copy engine) slowed the shared-memory
// traffic of the following update phase by more than they saved (measured: 39.7 / 45.3 us per leaf against 31.0): all
// outputs leave at the end.
template <int NT, bool VEC>
__device__ __forceinline__ void l3_store_colblock(const double *__restrict__ S, const double *__restrict__ RL,
                                                     double *__restrict__ Wblk, int64_t ld, double *__restrict__ invd,
                                                     int Jp, int t) {
    const int c0 = Jp * L3_B;
    constexpr int NEL2 = 128 * L3_B / 2;
    for (int base = t; base < NEL2; base += 8 * NT) {
        double2 v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int idx = base + k * NT;
            const int r = idx >> 4, c = c0 + 2 * (idx & 15);
            v[k].x = (idx < NEL2 && r >= c) ? S[r * L3_S + c] : 0.0;
            v[k].y = (idx < NEL2 && r >= c + 1) ? S[r * L3_S + c + 1] : 0.0;
        }
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int idx = base + k * NT;
            if (idx < NEL2) {
                double *dst = Wblk + (int64_t)(idx >> 4) * ld + c0 + 2 * (idx & 15);
                if (VEC) {
                    *reinterpret_cast<double2 *>(dst) = v[k];
                } else {
                    dst[0] = v[k].x;
                    dst[1] = v[k].y;
                }
            }
        }
    }
    for (int base = t; base < NEL2; base += 8 * NT) {
        double2 v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int idx = base + k * NT;
            const int i = c0 + (idx >> 6), r = 2 * (idx & 63);  // X[i][r], X[i][r + 1]
            v[k].x = (idx < NEL2) ? ((r < i) ? S[r * L3_S + i] : ((r == i) ? RL[i] : 0.0)) : 0.0;
            v[k].y = (idx < NEL2) ? ((r + 1 < i) ? S[(r + 1) * L3_S + i] : ((r + 1 == i) ? RL[i] : 0.0)) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int idx = base + k * NT;
            if (idx < NEL2) {
                double *dst = invd + (c0 + (idx >> 6)) * 128 + 2 * (idx & 63);
                if (VEC) {
                    *reinterpret_cast<double2 *>(dst) = v[k];
                } else {
                    dst[0] = v[k].x;
                    dst[1] = v[k].y;
                }
            }
        }
    }
}

__device__ long long l3_dbg[32];  // phase timestamps of the last launch (clock64 of thread 0): lgp_debug_leaf3_clocks
#define L3_STAMP(i)                          \
    do {                                     \
        if (tid == 0) l3_dbg[i] = clock64(); \
    } while (0)

__global__ void __launch_bounds__(L3_THREADS, 1) potrf_leaf3_kernel(double *__restrict__ Wblk, int64_t ld,
                                                                   double *__restrict__ invd,
                                                                   double *__restrict__ dvec,
                                                                   int32_t *__restrict__ info, int j0) {
    extern __shared__ __align__(16) double l3sm[];
    double *S = l3sm;
    double *RAW = S + L3_OFF_RAW;
    double *TS = S + L3_OFF_TS;
    double *XD = S + L3_OFF_XD;
    double *RL = S + L3_OFF_RL;
    const uint32_t bar0 = smem_u32(S + L3_OFF_BAR);
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;

    L3_STAMP(0);
    if (tid < 32) l3_mbar_init(bar0 + 8 * tid, 1);
    // lower triangle in, 16-byte loads with eight in flight per thread: block column 0 by everybody (the panel-0 chain
    // starts on it), the other three block columns by the spare warps while panel 0 runs
    const bool vec = !((ld & 1) | (int64_t)((reinterpret_cast<uintptr_t>(Wblk) | reinterpret_cast<uintptr_t>(invd)) & 15));
    {
        double2 v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int idx = tid + k * L3_THREADS, r = idx >> 4, c = 2 * (idx & 15);
            v[k] = make_double2(0.0, 0.0);
            if (vec) {
                if (r >= c) v[k] = *reinterpret_cast<const double2 *>(Wblk + (int64_t)r * ld + c);
            } else {
                if (r >= c) v[k].x = Wblk[(int64_t)r * ld + c];
                if (r >= c + 1) v[k].y = Wblk[(int64_t)r * ld + c + 1];
            }
        }
        // block columns 1..3 (rows 32..127): asynchronous copies queued behind the loads above, waited for after panel 0
        for (int idx = tid; idx < 96 * 96; idx += L3_THREADS) {
            const int r = 32 + idx / 96, c = 32 + idx % 96;
            if (r >= c) cp_async8(smem_u32(S + r * L3_S + c), Wblk + (int64_t)r * ld + c);
        }
        cp_async_commit();
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int idx = tid + k * L3_THREADS, r = idx >> 4, c = 2 * (idx & 15);
            S[r * L3_S + c] = v[k].x;
            S[r * L3_S + c + 1] = (r >= c + 1) ? v[k].y : 0.0;
        }
    }
    __syncthreads();
    L3_STAMP(1);

    const uint32_t raw_s = smem_u32(RAW), ts_s = smem_u32(TS);
#pragma unroll 1
    for (int J = 0; J < 4; J++) {
        const int c0 = J * L3_B;
        const uint32_t parity = J & 1;
        const uint32_t rl_s = smem_u32(RL + c0);
        // warp roles: 0 chain, 4 identity rows (both on scheduler 0, which gets no DMMA work during a panel), 1..3 the
        // off-diagonal row blocks, 5..7 spare
        if (w == 0) {
            double a[L3_B];
            double *row = S + (c0 + lane) * L3_S + c0;
#pragma unroll
            for (int c = 0; c < L3_B; c++) a[c] = row[c];
            double ldiag;
            l3_chain(a, raw_s, ts_s, RL + c0, bar0, dvec, info, j0 + c0, lane, ldiag);
            // every lane of this warp already sees RL (written before the last __syncwarp of l3_chain)
#pragma unroll
            for (int c = 0; c < L3_B; c++) {
                const double v = (c == lane) ? ldiag : a[c] * RL[c0 + c];
                if (c <= lane) row[c] = v;
            }
        } else if (w == 4) {
            // identity rows: become L_JJ^-T (upper triangular); strict upper part to S, whole block to XD
            double p[L3_B];
#pragma unroll
            for (int c = 0; c < L3_B; c++) p[c] = (c == lane) ? 1.0 : 0.0;
            l3_follow(p, ts_s, rl_s, bar0, parity);
            double *row = S + (c0 + lane) * L3_S + c0;
            double *xrow = XD + (J & 1) * L3_B * L3_XS + lane * L3_XS;
#pragma unroll
            for (int c = 0; c < L3_B; c++) {
                xrow[c] = p[c];
                if (c > lane) row[c] = p[c];
            }
        } else if (w <= 3) {
            // the three off-diagonal row blocks of the panel (below: L_IJ; above: Y_IJ)
            const int I = (w - 1 < J) ? (w - 1) : w;
            double p[L3_B];
            double *row = S + (I * L3_B + lane) * L3_S + c0;
#pragma unroll
            for (int c = 0; c < L3_B; c++) p[c] = row[c];
            l3_follow(p, ts_s, rl_s, bar0, parity);
#pragma unroll
            for (int c = 0; c < L3_B; c++) row[c] = p[c];
        } else if (J == 0) {
            // spare warps during panel 0: zeros into the blocks above the block diagonal (Y starts as the identity, whose
            // diagonal blocks the identity-row warp supplies)
            const int t = (w - 5) * 32 + lane;
            for (int idx = t; idx < 96 * 96; idx += L3_NSPARE * 32) {
                const int r = idx / 96, c = 32 + idx % 96;
                if ((r >> 5) < (c >> 5)) S[r * L3_S + c] = 0.0;
            }
        } else {
            // spare warps: blocks of the previous panel's update that the current panel does not touch, then the global
            // stores of the previous block column
            const int sw = w - 5, Js = J - 1;
            int cnt = 0;
            for (int K = J + 1; K < 4; K++)
                for (int I = 0; I < 4; I++) {
                    if (!(I <= Js || I >= K)) continue;
                    for (int hf = 0; hf < 2; hf++, cnt++)
                        if (cnt % L3_NSPARE == sw) l3_update_unit(S, XD, I, K, hf, Js, lane);
                }
        }
        if (J == 0) cp_async_wait<0>();
        __syncthreads();
        L3_STAMP(2 + 2 * J);
        if (J == 3) break;
        // block column J+1 from panel J: 8 half blocks, one per warp
        l3_update_unit(S, XD, w >> 1, J + 1, w & 1, J, lane);
        __syncthreads();
        L3_STAMP(3 + 2 * J);
    }
    if (vec)
        for (int Jp = 0; Jp < 4; Jp++) l3_store_colblock<L3_THREADS, true>(S, RL, Wblk, ld, invd, Jp, tid);
    else
        for (int Jp = 0; Jp < 4; Jp++) l3_store_colblock<L3_THREADS, false>(S, RL, Wblk, ld, invd, Jp, tid);
    L3_STAMP(9);
}

}  // namespace lgp
