// Raw feature rows stored as fp32, fp16 or bf16 (CONE_DTYPE_*): loads that convert to fp32, and the host-side dispatch
// from a dtype code to the element type.  fp16 and bf16 convert to fp32 exactly, so a kernel that loads through these
// helpers and keeps its fp32 arithmetic and reduction order gives the bits of its fp32 instantiation on the upcast rows.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace cone {

// 4 consecutive elements at p: one 16-byte load for fp32, one 8-byte load for the 16-bit types (p aligned to that size)
__device__ __forceinline__ float4 load_feat4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ldg_feat4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

__device__ __forceinline__ float4 feat4_from_bits(uint2 u, const __half*) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float4 feat4_from_bits(uint2 u, const __nv_bfloat16*) {
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
template <class T>
__device__ __forceinline__ float4 load_feat4(const T* p) {
    return feat4_from_bits(*reinterpret_cast<const uint2*>(p), p);
}
template <class T>
__device__ __forceinline__ float4 ldg_feat4(const T* p) {
    return feat4_from_bits(__ldg(reinterpret_cast<const uint2*>(p)), p);
}

// f(const T* tag) with T the element type of `dtype`; an unknown code is CONE_ERR_INVALID
template <class F>
int dispatch_feature(int dtype, F&& f) {
    switch (dtype) {
        case CONE_DTYPE_F32: return f(static_cast<const float*>(nullptr));
        case CONE_DTYPE_F16: return f(static_cast<const __half*>(nullptr));
        case CONE_DTYPE_BF16: return f(static_cast<const __nv_bfloat16*>(nullptr));
        default: set_error("unknown feature dtype %d", dtype); return CONE_ERR_INVALID;
    }
}

}  // namespace cone
