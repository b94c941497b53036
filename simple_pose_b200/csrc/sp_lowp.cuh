// float16 / bfloat16 / float32 element access for the loss kernels that read `pred` in its own dtype: one
// 16-byte group (4 floats or 8 halves) per load / store, conversions with round-to-nearest-even exactly as
// torch's .to(dtype).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "sp_common.cuh"

namespace sp_lowp {

__device__ __forceinline__ float to_float(float v) { return v; }
__device__ __forceinline__ float to_float(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ float from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_float<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ float4 ldg_stream4(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// the 16 bytes at a 16-byte aligned address -> float[16 / sizeof(T)]
__device__ __forceinline__ void load_group(const float* p, float (&out)[4]) {
    const uint4 a = ldg_stream16(p);
    out[0] = __uint_as_float(a.x); out[1] = __uint_as_float(a.y); out[2] = __uint_as_float(a.z); out[3] = __uint_as_float(a.w);
}
__device__ __forceinline__ void load_group(const __half* p, float (&out)[8]) {
    const uint4 a = ldg_stream16(p);
    const unsigned w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
        const float2 f = __half22float2(h);
        out[2 * i] = f.x;
        out[2 * i + 1] = f.y;
    }
}
__device__ __forceinline__ void load_group(const __nv_bfloat16* p, float (&out)[8]) {
    const uint4 a = ldg_stream16(p);
    const unsigned w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {             // bfloat16 -> float32 is a 16-bit shift
        out[2 * i] = __uint_as_float(w[i] << 16);
        out[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}

__device__ __forceinline__ void store_group(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void store_group(__half* p, const float (&v)[8]) {
    uint4 r;
    unsigned* w = reinterpret_cast<unsigned*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
        w[i] = *reinterpret_cast<const unsigned*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = r;
}
__device__ __forceinline__ void store_group(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 r;
    unsigned* w = reinterpret_cast<unsigned*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        w[i] = *reinterpret_cast<const unsigned*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = r;
}

}  // namespace sp_lowp
