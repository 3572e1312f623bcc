// Shared device helpers for the lsqfitgp-b200 CUDA kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define LGP_OK 0
#define LGP_ERR_BADARG (-1)
#define LGP_ERR_ALIGN (-2)
#define LGP_ERR_CUDA (-3)
#define LGP_ERR_UNSUPPORTED (-4)

#define LGP_STR_(x) #x
#define LGP_STR(x) LGP_STR_(x)

// number of kernel launches issued by this library since it was loaded (bench.py reports it as gpu_launches)
extern "C" long long lgp_launch_count(void);
namespace lgp { void count_launch(); }

#define LGP_CUDA_CHECK_LAUNCH()                          \
    do {                                                 \
        lgp::count_launch();                             \
        cudaError_t e__ = cudaGetLastError();            \
        if (e__ != cudaSuccess) return LGP_ERR_CUDA;     \
    } while (0)

namespace lgp {

// Opt `kernel` in to `dyn` bytes of dynamic shared memory before a launch.  Without the opt-in a launch may use 48 KiB
// of static plus dynamic shared memory in all; so the kernel's static size counts against that limit too.  A failed
// query or opt-in is cleared from cudaGetLastError so that it does not surface at a later, unrelated launch check.
template <class F>
static int smem_opt_in(F *kernel, size_t dyn) {
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, (const void *)kernel) != cudaSuccess) {
        cudaGetLastError();
        return LGP_ERR_CUDA;
    }
    if (fa.sharedSizeBytes + dyn <= 48 * 1024) return LGP_OK;
    if (cudaFuncSetAttribute((const void *)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn) != cudaSuccess) {
        cudaGetLastError();
        return LGP_ERR_CUDA;
    }
    return LGP_OK;
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// 16-byte async copy global -> shared, zero-filling bytes beyond src_bytes.
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(src), "r"(src_bytes));
}
// 8-byte async copy global -> shared (for rows whose shared-memory stride is not a multiple of 16 bytes)
__device__ __forceinline__ void cp_async8(uint32_t dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

// FP64 tensor-core MMA: D(8x8) += A(8x4, row) * B(4x8, col). SASS: DMMA.8x8x4.
// lane l holds A[l/4][l%4], B[k=l%4][n=l/4], C[l/4][2*(l%4)+{0,1}].
__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace lgp
