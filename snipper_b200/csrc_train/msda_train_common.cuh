// What the training tails of libmsda_b200_train.so (msda_train_tail.cu) and libmsda_b200_amp_train.so
// (csrc_amp_train/msda_amp_train_tail.cu) share: the warp reduction, the keep-mask load, the backward's partial-row grid
// and CTA reduction, the ordered parameter-gradient sum and the host-side validation helpers.  The partial-row grid and
// the summation order are defined here once, so both libraries reduce the parameter gradients in the same order.
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace msda {

namespace {

constexpr int kWarps = 8;              // rows per CTA step, forward and backward
constexpr int kMaxBwdBlocks = 296;     // backward CTAs: 2 per SM of a B200; the grid is min(ceil(rows / 8), this)

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float4 load4(const float *p, int c4) { return __ldg(reinterpret_cast<const float4 *>(p) + c4); }

__device__ __forceinline__ float4 load_mask4(const uint8_t *m, int c4)
{
    const uchar4 u = __ldg(reinterpret_cast<const uchar4 *>(m) + c4);
    return make_float4((float)u.x, (float)u.y, (float)u.z, (float)u.w);
}

__device__ __forceinline__ void add4(float4 &acc, float4 v)
{
    acc.x += v.x;
    acc.y += v.y;
    acc.z += v.z;
    acc.w += v.w;
}

// dst[c] = sum over the CTA's warps w in order of p (of warp w) at channel c
template <int VPL>
__device__ __forceinline__ void cta_partial(float4 (*red)[32 * VPL], const float4 (&p)[VPL], float *__restrict__ dst)
{
    constexpr int C = 128 * VPL;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < VPL; ++k) red[warp][lane + 32 * k] = p[k];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const float *col = reinterpret_cast<const float *>(&red[0][0]) + c;
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += col[w * C];
        dst[c] = s;
    }
    __syncthreads();
}

// out[i] = sum over CTAs b in order of partials[b][i], i < 3 C
__global__ void __launch_bounds__(256)
layer_tail_param_sum_kernel(const float *__restrict__ partials, float *__restrict__ out, int blocks, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = 0.f;
#pragma unroll 8
    for (int b = 0; b < blocks; ++b) s += __ldg(partials + (size_t)b * n + i);
    out[i] = s;
}

bool cols_ok(int cols) { return cols > 0 && cols % 128 == 0 && cols <= 1024; }

// the backward's grid: a function of rows only, so the partial rows and their sum do not depend on the device
int bwd_blocks(int64_t rows)
{
    const int64_t b = (rows + kWarps - 1) / kWarps;
    return (int)(b < kMaxBwdBlocks ? b : kMaxBwdBlocks);
}

bool scale_ok(float s) { return isfinite(s) && s >= 1.f; }

// false for NULL: optional pointers pass; required ones are checked for NULL separately
bool misaligned(const void *p) { return reinterpret_cast<uintptr_t>(p) % 16 != 0; }

}  // namespace

}  // namespace msda
