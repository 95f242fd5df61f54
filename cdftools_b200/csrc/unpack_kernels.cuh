// unpack_kernels.cuh -- K3b: NC_SHORT records (cdf16bit output) unpacked on the device.
//
// A packed variable stores int16 values with scale_factor / add_offset; getvar decodes them after NF90_GET_VAR as three
// masked passes (src/cdfio.F90:1599-1605): x*sf where x /= spval, then x+ao where x /= spval (the comparison sees the
// scaled value).  The host reader does the same (nc3::Reader::read_f32).  This kernel reproduces that bit for bit: the
// int16 -> float conversion is exact, and the product and sum are rounded separately (__fmul_rn / __fadd_rn: never
// contracted into an FFMA, which would round once and differ).  HBM-bound: 2 B read and 4 B written per value.
#pragma once
#include "common.cuh"

namespace cdfgpu {

__device__ __forceinline__ float unpack_i16_one(uint32_t v16, float sf, float ao, float sp)
{
    float x = (float)(int16_t)(uint16_t)v16;
    if (sf != 1.f && x != sp) x = __fmul_rn(x, sf);
    if (ao != 0.f && x != sp) x = __fadd_rn(x, ao);
    return x;
}

// raw: n int16 values (big-endian file order when swap != 0, else host order); out: n floats.  Both 16-byte aligned.
__global__ void __launch_bounds__(256) unpack_i16_kernel(const uint16_t *__restrict__ raw, float *__restrict__ out, size_t n,
                                                         int swap, float sf, float ao, float sp)
{
    const size_t n8 = n >> 3;
    const uint4 *r8 = reinterpret_cast<const uint4 *>(raw);
    float4 *o4 = reinterpret_cast<float4 *>(out);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
        uint4 w = __ldcs(r8 + i);
        if (swap) {
            w.x = __byte_perm(w.x, 0, 0x2301); w.y = __byte_perm(w.y, 0, 0x2301);
            w.z = __byte_perm(w.z, 0, 0x2301); w.w = __byte_perm(w.w, 0, 0x2301);
        }
        float4 a, b;
        a.x = unpack_i16_one(w.x & 0xffffu, sf, ao, sp); a.y = unpack_i16_one(w.x >> 16, sf, ao, sp);
        a.z = unpack_i16_one(w.y & 0xffffu, sf, ao, sp); a.w = unpack_i16_one(w.y >> 16, sf, ao, sp);
        b.x = unpack_i16_one(w.z & 0xffffu, sf, ao, sp); b.y = unpack_i16_one(w.z >> 16, sf, ao, sp);
        b.z = unpack_i16_one(w.w & 0xffffu, sf, ao, sp); b.w = unpack_i16_one(w.w >> 16, sf, ao, sp);
        o4[2 * i] = a;
        o4[2 * i + 1] = b;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 7)) {
        const size_t i = (n8 << 3) + threadIdx.x;
        uint32_t v = raw[i];
        if (swap) v = __byte_perm(v, 0, 0x3201);
        out[i] = unpack_i16_one(v, sf, ao, sp);
    }
}

}  // namespace cdfgpu
