// common.cuh -- shared helpers of libcdfgpu (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/cdfgpu.h"

namespace cdfgpu {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// ---- error plumbing -------------------------------------------------------------------------------------------
extern char g_errbuf[512];
inline int set_error(int code, const char *fmt, const char *a = "", const char *b = "")
{
    snprintf(g_errbuf, sizeof(g_errbuf), fmt, a, b);
    return code;
}
// A failed runtime call also records its error as the thread's "last error"; it is consumed here, so that a later
// CDF_CUDA(cudaGetLastError()) after a good launch does not report it again (a sticky error stays in the context).
#define CDF_CUDA(call)                                                                                       \
    do {                                                                                                     \
        cudaError_t e__ = (call);                                                                            \
        if (e__ != cudaSuccess) {                                                                            \
            (void)cudaGetLastError();                                                                        \
            snprintf(cdfgpu::g_errbuf, sizeof(cdfgpu::g_errbuf), "%s failed: %s (%s:%d)", #call,             \
                     cudaGetErrorString(e__), __FILE__, __LINE__);                                           \
            return (e__ == cudaErrorMemoryAllocation) ? CDFGPU_ERR_NOMEM                                     \
                   : (e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver) ? CDFGPU_ERR_NODEVICE  \
                                                                                      : CDFGPU_ERR_CUDA;     \
        }                                                                                                    \
    } while (0)

// ---- device helpers -------------------------------------------------------------------------------------------
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// L2 policy for data that is read exactly once (the record and the resident area field): evict first, so the
// small mask planes that every level re-reads stay in L2.
__device__ __forceinline__ uint64_t make_evict_first_policy()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// streaming 16-byte load: read-only path, no L1 allocation, L2 evict-first
__device__ __forceinline__ float4 ld_stream_f4(const float4 *p, uint64_t pol)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}

// asynchronous global -> shared copies (LDGSTS): no registers are held while the data are in flight
__device__ __forceinline__ void cp_async16(void *dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(void *dst, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait()
{
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// K3: in-place 32-bit byte swap of a record (big-endian NetCDF-3 REAL(4) -> host order).  HBM-bound, 8 B per value.
__global__ void bswap32_kernel(uint32_t *__restrict__ p, size_t n)
{
    const size_t n4 = n >> 2;
    uint4 *p4 = reinterpret_cast<uint4 *>(p);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        uint4 v = p4[i];
        v.x = __byte_perm(v.x, 0, 0x0123); v.y = __byte_perm(v.y, 0, 0x0123);
        v.z = __byte_perm(v.z, 0, 0x0123); v.w = __byte_perm(v.w, 0, 0x0123);
        p4[i] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const size_t i = (n4 << 2) + threadIdx.x;
        p[i] = __byte_perm(p[i], 0, 0x0123);
    }
}

}  // namespace cdfgpu
