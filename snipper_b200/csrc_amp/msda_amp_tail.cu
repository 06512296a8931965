// Layer tail under bf16 autocast (include/msda_b200_amp.h), sm_100a.
//
// Under torch.autocast(bfloat16) the Linear in front of a tail returns bf16 while the residual stream stays fp32
// (autocast runs layer_norm in fp32), and autocast casts the fp32 stream to bf16 again in front of every following
// GEMM.  This kernel reads the bf16 GEMM output, writes the fp32 stream and, in the same pass, the bf16 copies the
// next GEMMs take:
//
//     out          = LayerNorm(residual + (float(y) + bias)) * gamma + beta     fp32
//     out_bf16     = bf16_rn(out)                                               optional: linear1 / value_proj input
//     out_pos_bf16 = bf16_rn(out + pos)                                         optional: the next block's query
//
// The layout and the arithmetic are those of layer_tail_kernel (snipper_b200/csrc/msda_tail.cu), operation for
// operation: one warp per row, VPL groups of 4 channels per lane (channel 4 * (lane + 32 k)), bias added to y before
// the residual, mean and variance in two passes over the registers.  bf16 -> fp32 is exact, so `out` has the bits of
// the fp32 kernel run on float(y), float(residual), and the float32 validation of that kernel carries over.  The bf16
// loads and stores are 8 bytes per lane and step.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/msda_b200_amp.h"
#include "msda_bf16_io.cuh"

namespace msda {

namespace {

thread_local int g_last_cuda_error = 0;

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float4 load4(const float *p, int c4) { return __ldg(reinterpret_cast<const float4 *>(p) + c4); }

template <int VPL, typename Residual>
__global__ void __launch_bounds__(256)
layer_tail_amp_kernel(const __nv_bfloat16 *__restrict__ y, const float *__restrict__ bias,
                      const Residual *__restrict__ residual, const float *__restrict__ gamma,
                      const float *__restrict__ beta, const float *__restrict__ pos, float *__restrict__ out,
                      __nv_bfloat16 *__restrict__ out_bf16, __nv_bfloat16 *__restrict__ out_pos_bf16, int64_t rows,
                      float eps)
{
    constexpr int C = 128 * VPL;
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    float4 x[VPL];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
        const int c4 = lane + 32 * k;
        const float4 a = load4(y + row * C, c4), r = load4(residual + row * C, c4);
        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
        if (bias != nullptr) b = load4(bias, c4);
        // layer_tail_kernel's order: (Linear output incl. bias) first, then the residual add
        x[k] = make_float4(r.x + (a.x + b.x), r.y + (a.y + b.y), r.z + (a.z + b.z), r.w + (a.w + b.w));
        sum += (x[k].x + x[k].y) + (x[k].z + x[k].w);
    }
    const float mean = warp_sum(sum) * (1.f / C);
    float sq = 0.f;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
        const float dx = x[k].x - mean, dy = x[k].y - mean, dz = x[k].z - mean, dw = x[k].w - mean;
        sq += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
    const float rstd = 1.f / sqrtf(warp_sum(sq) * (1.f / C) + eps);
    float4 *o4 = reinterpret_cast<float4 *>(out + row * C);
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
        const int c4 = lane + 32 * k;
        const float4 g = load4(gamma, c4);
        const float4 b = load4(beta, c4);
        float4 o;
        o.x = (x[k].x - mean) * rstd * g.x + b.x;
        o.y = (x[k].y - mean) * rstd * g.y + b.y;
        o.z = (x[k].z - mean) * rstd * g.z + b.z;
        o.w = (x[k].w - mean) * rstd * g.w + b.w;
        o4[c4] = o;
        if (out_bf16 != nullptr) store4_bf16(out_bf16 + row * C, c4, o);
        if (out_pos_bf16 != nullptr) {
            const float4 p = load4(pos + row * C, c4);
            store4_bf16(out_pos_bf16 + row * C, c4, make_float4(o.x + p.x, o.y + p.y, o.z + p.z, o.w + p.w));
        }
    }
}

template <typename Residual>
cudaError_t launch(const __nv_bfloat16 *y, const float *bias, const Residual *residual, const float *gamma,
                   const float *beta, const float *pos, float *out, __nv_bfloat16 *out_bf16,
                   __nv_bfloat16 *out_pos_bf16, int64_t rows, int cols, float eps, cudaStream_t stream)
{
    constexpr int kWarps = 8;
    const int64_t blocks = (rows + kWarps - 1) / kWarps;
    if (blocks > 0x7fffffff) return cudaErrorInvalidValue;
#define MSDA_AMP_TAIL(V)                                                                                             \
    case V:                                                                                                          \
        layer_tail_amp_kernel<V, Residual><<<(unsigned)blocks, 32 * kWarps, 0, stream>>>(                             \
            y, bias, residual, gamma, beta, pos, out, out_bf16, out_pos_bf16, rows, eps);                            \
        break;
    switch (cols / 128) {
        MSDA_AMP_TAIL(1) MSDA_AMP_TAIL(2) MSDA_AMP_TAIL(3) MSDA_AMP_TAIL(4)
        MSDA_AMP_TAIL(5) MSDA_AMP_TAIL(6) MSDA_AMP_TAIL(7) MSDA_AMP_TAIL(8)
        default: return cudaErrorInvalidValue;
    }
#undef MSDA_AMP_TAIL
    return cudaGetLastError();
}

// false for NULL: optional pointers pass; required ones are checked for NULL separately
bool misaligned(const void *p) { return reinterpret_cast<uintptr_t>(p) % 16 != 0; }

}  // namespace

}  // namespace msda

extern "C" {

int msda_amp_abi_version(void) { return MSDA_AMP_ABI_VERSION; }

int msda_amp_last_cuda_error(void) { return msda::g_last_cuda_error; }

int msda_amp_layer_tail(const void *y, const void *bias, const void *residual, int residual_dtype, const void *gamma,
                        const void *beta, const void *pos, void *out, void *out_bf16, void *out_plus_pos_bf16,
                        int64_t rows, int cols, float eps, void *stream)
{
    if (residual_dtype != MSDA_DTYPE_F32 && residual_dtype != MSDA_DTYPE_BF16) return MSDA_ERR_UNSUPPORTED_DTYPE;
    if (rows < 0 || cols <= 0 || cols % 128 != 0 || cols > 1024 || !(eps >= 0.f)) return MSDA_ERR_INVALID_ARGUMENT;
    if ((pos == nullptr) != (out_plus_pos_bf16 == nullptr)) return MSDA_ERR_INVALID_ARGUMENT;
    if (rows == 0) return MSDA_OK;
    const void *ptrs[] = {y, residual, gamma, beta, out};
    for (const void *p : ptrs)
        if (p == nullptr || msda::misaligned(p)) return MSDA_ERR_INVALID_ARGUMENT;
    if (msda::misaligned(bias) || msda::misaligned(pos) || msda::misaligned(out_bf16) ||
        msda::misaligned(out_plus_pos_bf16))
        return MSDA_ERR_INVALID_ARGUMENT;
    const auto *y16 = static_cast<const __nv_bfloat16 *>(y);
    const auto *b = static_cast<const float *>(bias), *g = static_cast<const float *>(gamma);
    const auto *be = static_cast<const float *>(beta), *p = static_cast<const float *>(pos);
    auto *o = static_cast<float *>(out);
    auto *o16 = static_cast<__nv_bfloat16 *>(out_bf16), *op16 = static_cast<__nv_bfloat16 *>(out_plus_pos_bf16);
    const auto s = static_cast<cudaStream_t>(stream);
    const cudaError_t e =
        residual_dtype == MSDA_DTYPE_F32
            ? msda::launch(y16, b, static_cast<const float *>(residual), g, be, p, o, o16, op16, rows, cols, eps, s)
            : msda::launch(y16, b, static_cast<const __nv_bfloat16 *>(residual), g, be, p, o, o16, op16, rows, cols,
                           eps, s);
    if (e == cudaSuccess) return MSDA_OK;
    msda::g_last_cuda_error = (int)e;
    return MSDA_ERR_CUDA;
}

}  // extern "C"
