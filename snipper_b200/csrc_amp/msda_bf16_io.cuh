// bf16 row I/O of the mixed-precision layer tails (csrc_amp/msda_amp_tail.cu, csrc_amp_train/msda_amp_train_tail.cu):
// 4 channels per lane and step, 8 bytes, converted to and from float4.  bf16 -> fp32 is exact; fp32 -> bf16 rounds to
// nearest even, as torch's .to(torch.bfloat16) does.
#pragma once

#include <cuda_bf16.h>
#include <stdint.h>

namespace msda {

namespace {

__device__ __forceinline__ float4 load4(const __nv_bfloat16 *p, int c4)
{
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(p) + c4);
    const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&u.x));
    const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&u.y));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

__device__ __forceinline__ void store4_bf16(__nv_bfloat16 *p, int c4, float4 v)
{
    const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<const uint32_t *>(&lo);
    u.y = *reinterpret_cast<const uint32_t *>(&hi);
    reinterpret_cast<uint2 *>(p)[c4] = u;
}

}  // namespace

}  // namespace msda
