// Launcher for the FP64 DMMA GEMM (see gemm_dmma.cuh).
#include "gemm_dmma.cuh"
#include "internal.h"
#include <math.h>
#include <string.h>

namespace lgp {

template <class Cfg, bool AK, bool BK_>
static int launch_cfg(cudaStream_t stream, GemmParams &p) {
    p.tiles_m = (p.M + Cfg::BM - 1) / Cfg::BM;
    p.tiles_n = (p.N + Cfg::BN - 1) / Cfg::BN;
    int64_t grid = (p.flags & GEMM_LOWER) ? (int64_t)(Cfg::BM >= Cfg::BN ? Cfg::BM / Cfg::BN : 1) * p.tiles_m * (p.tiles_m + 1) / 2
                                          : (int64_t)p.tiles_m * p.tiles_n;
    if (grid > 2147483647LL) return LGP_ERR_UNSUPPORTED;
    static DeviceOnce attr_set;  // one flag per template instantiation and device
    const int dev = current_device();
    if (!attr_set.done(dev)) {
        if (cudaFuncSetAttribute(gemm_dmma_kernel<Cfg, AK, BK_>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 Cfg::SMEM_BYTES) != cudaSuccess)
            return LGP_ERR_CUDA;
        attr_set.set(dev);
    }
    gemm_dmma_kernel<Cfg, AK, BK_><<<(unsigned)grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(p);
    LGP_CUDA_CHECK_LAUNCH();
    return LGP_OK;
}

// number of SMs of the current device (cached per device)
static int sm_count() {
    static int cached[MAX_DEVICES];
    const int dev = current_device();
    if (dev < 0 || dev >= MAX_DEVICES) return 148;
    if (!cached[dev]) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        cached[dev] = v;
    }
    return cached[dev];
}

template <class Cfg>
static int launch_layout(cudaStream_t stream, bool a_kmaj, bool b_kmaj, GemmParams &p) {
    if (a_kmaj && b_kmaj) return launch_cfg<Cfg, true, true>(stream, p);
    if (a_kmaj && !b_kmaj) return launch_cfg<Cfg, true, false>(stream, p);
    if (!a_kmaj && b_kmaj) return launch_cfg<Cfg, false, true>(stream, p);
    return launch_cfg<Cfg, false, false>(stream, p);
}

// Host-side launcher (internal; the C ABI wrapper is lgp_dgemm in capi.cu).
int gemm_launch(cudaStream_t stream, bool a_kmaj, bool b_kmaj, int M, int N, int K, double alpha, const double *A,
                int64_t lda, const double *B, int64_t ldb, double *C, int64_t ldc, int flags, const GemmMirror *mir,
                const double *scale) {
    if (M <= 0 || N <= 0) return LGP_OK;
    if (mir && (mir->n < 0 || mir->n > GEMM_MAX_MIRRORS || (mir->multimem && mir->n != 1))) return LGP_ERR_BADARG;
    if (mir)
        for (int i = 0; i < mir->n; i++)
            if (reinterpret_cast<uintptr_t>(mir->dst[i]) & 15) return LGP_ERR_ALIGN;
    if ((lda & 1) || (ldb & 1) || (reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(B) & 15))
        return LGP_ERR_ALIGN;
    if ((flags & GEMM_LOWER) && M != N) return LGP_ERR_BADARG;
    if ((flags & GEMM_INPLACE_A) && N > 128) return LGP_ERR_BADARG;
    if ((flags & GEMM_INPLACE_B) && M > 128) return LGP_ERR_BADARG;
    GemmParams p;
    p.A = A; p.B = B; p.C = C;
    p.M = M; p.N = N; p.K = K;
    p.lda = lda; p.ldb = ldb; p.ldc = ldc;
    p.alpha = alpha;
    p.flags = flags;
    p.scale = scale;
    if (mir)
        p.mir = *mir;
    else
        memset(&p.mir, 0, sizeof(p.mir));
    // tile configuration: the in-place products need the aliased dimension inside one tile; grids that would leave SMs
    // idle with the throughput tiles use the latency tiles (4x the CTAs)
    const int sms = sm_count();
    if (flags & GEMM_INPLACE_B) {
        const bool small = (N + 63) / 64 < sms;
        if (a_kmaj && !b_kmaj)
            return small ? launch_cfg<GemmWideSmall, true, false>(stream, p) : launch_cfg<GemmWide, true, false>(stream, p);
        if (!a_kmaj && !b_kmaj)
            return small ? launch_cfg<GemmWideSmall, false, false>(stream, p)
                         : launch_cfg<GemmWide, false, false>(stream, p);
        return LGP_ERR_UNSUPPORTED;
    }
    if (flags & GEMM_INPLACE_A) {
        const bool small = (M + 63) / 64 < sms;
        if (a_kmaj && b_kmaj)
            return small ? launch_cfg<GemmTallSmall, true, true>(stream, p) : launch_cfg<GemmTall, true, true>(stream, p);
        return LGP_ERR_UNSUPPORTED;
    }
    const int64_t tm = (M + 63) / 64, tn = (N + 63) / 64;
    const int64_t tiles = (flags & GEMM_LOWER) ? tm * (tm + 1) / 2 : tm * tn;
    if (tiles < sms) return launch_layout<GemmSmall>(stream, a_kmaj, b_kmaj, p);
    return launch_layout<GemmBig>(stream, a_kmaj, b_kmaj, p);
}

}  // namespace lgp

// debug hook (not in the public header; host code, no GPU needed): tile (tm, tn) that CTA `b` of a lower-triangular launch
// with `tiles_m` tile rows works on: the host-side twin of the index arithmetic at the top of gemm_dmma_kernel
extern "C" int lgp_debug_lower_tile(long long b, int tiles_m, int *out2) {
    if (b < 0 || tiles_m < 1 || b >= (long long)tiles_m * (tiles_m + 1) / 2 || !out2) return LGP_ERR_BADARG;
    int tm = (int)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
    while ((long long)(tm + 1) * (tm + 2) / 2 <= b) tm++;
    while ((long long)tm * (tm + 1) / 2 > b) tm--;
    int tn = (int)(b - (long long)tm * (tm + 1) / 2);
    lgp::gemm_lower_grouped_tile(b, tm, tiles_m, tm, tn);
    out2[0] = tm;
    out2[1] = tn;
    return LGP_OK;
}
