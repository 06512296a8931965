// Layer tail for training under bf16 autocast (include/msda_b200_amp_train.h), sm_100a.
//
// In a bf16 autocast training step the reference's x = norm(x + dropout(Linear(..))) is, in stock PyTorch, a bf16 GEMM
// with a bias epilogue, a bf16 dropout, a type-promoting add into the fp32 residual, an fp32 LayerNorm and a cast to
// bf16 in front of every following GEMM, and the matching backward passes.  These kernels are the training tails of
// csrc_train/msda_train_tail.cu with the amp tail's I/O (csrc_amp/msda_amp_tail.cu): bf16 GEMM output and fp32 or
// bf16 residual in, the fp32 stream plus the next GEMMs' bf16 copies out.
//
// Forward: layer_tail_train_fwd_kernel's layout and arithmetic, operation for operation, on float(y) and
// float(residual) (bf16 -> fp32 is exact), so out, h and (mean, rstd) have its bits.
//
// Backward: layer_tail_train_bwd_kernel with g = (grad_out + float(grad_out_bf16)) + float(grad_out_pos_bf16), the
// residual gradient written in the residual's dtype and the GEMM-output gradient in bf16, each rounded once from the
// fp32 value.  The grad_y partial (the Linear-bias gradient) is taken before that rounding.  The partial-row grid,
// the CTA reduction and layer_tail_param_sum_kernel are csrc_train's (msda_train_common.cuh): no atomics, the result
// is bit-reproducible.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/msda_b200_amp_train.h"
#include "../csrc_amp/msda_bf16_io.cuh"
#include "../csrc_train/msda_train_common.cuh"

namespace msda {

namespace {

thread_local int g_last_cuda_error = 0;

__device__ __forceinline__ void store4(float *p, int c4, float4 v) { reinterpret_cast<float4 *>(p)[c4] = v; }

__device__ __forceinline__ void store4(__nv_bfloat16 *p, int c4, float4 v) { store4_bf16(p, c4, v); }

template <int VPL, typename Residual>
__global__ void __launch_bounds__(256)
layer_tail_amp_train_fwd_kernel(const __nv_bfloat16 *__restrict__ y, const float *__restrict__ bias,
                                const Residual *__restrict__ residual, const uint8_t *__restrict__ keep_mask,
                                float keep_scale, const float *__restrict__ gamma, const float *__restrict__ beta,
                                const float *__restrict__ pos, float *__restrict__ out,
                                __nv_bfloat16 *__restrict__ out_bf16, __nv_bfloat16 *__restrict__ out_pos_bf16,
                                float *__restrict__ h, float2 *__restrict__ mean_rstd, int64_t rows, float eps)
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
        float4 d = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
        if (keep_mask != nullptr) {
            // + 0.f as in layer_tail_train_fwd_kernel (a dropped -0 becomes +0)
            const float4 m = load_mask4(keep_mask + row * C, c4);
            d = make_float4((d.x * keep_scale) * m.x + 0.f, (d.y * keep_scale) * m.y + 0.f,
                            (d.z * keep_scale) * m.z + 0.f, (d.w * keep_scale) * m.w + 0.f);
        }
        x[k] = make_float4(r.x + d.x, r.y + d.y, r.z + d.z, r.w + d.w);
        reinterpret_cast<float4 *>(h + row * C)[c4] = x[k];
        sum += (x[k].x + x[k].y) + (x[k].z + x[k].w);
    }
    const float total = warp_sum(sum);
    const float mean = total * (1.f / C);
    float sq = 0.f;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
        const float dx = x[k].x - mean, dy = x[k].y - mean, dz = x[k].z - mean, dw = x[k].w - mean;
        sq += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
    const float rstd = 1.f / sqrtf(warp_sum(sq) * (1.f / C) + eps);
    // the stored mean is rounded as layer_tail_train_fwd_kernel rounds it (see there): `mean` itself stays fused
    // into x - mean
    if (lane == 0) mean_rstd[row] = make_float2(__fmul_rn(total, 1.f / C), rstd);
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

// partials: one row of 3 C floats per CTA, [g xhat | g | grad_y], as layer_tail_train_bwd_kernel writes them
template <int VPL, typename Residual>
__global__ void __launch_bounds__(256, VPL <= 3 ? 2 : 1)
layer_tail_amp_train_bwd_kernel(const float *__restrict__ grad_out, const __nv_bfloat16 *__restrict__ grad_out_bf16,
                                const __nv_bfloat16 *__restrict__ grad_out_pos_bf16, const float *__restrict__ h,
                                const float2 *__restrict__ mean_rstd, const uint8_t *__restrict__ keep_mask,
                                float keep_scale, const float *__restrict__ gamma,
                                Residual *__restrict__ grad_residual, __nv_bfloat16 *__restrict__ grad_y,
                                float *__restrict__ partials, int64_t rows)
{
    constexpr int C = 128 * VPL;
    __shared__ float4 red[kWarps][C / 4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float4 p_gx[VPL], p_g[VPL], p_gy[VPL];
#pragma unroll
    for (int k = 0; k < VPL; ++k) p_gx[k] = p_g[k] = p_gy[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t row = (int64_t)blockIdx.x * kWarps + warp; row < rows; row += (int64_t)gridDim.x * kWarps) {
        const float2 mr = __ldg(mean_rstd + row);
        const size_t off = (size_t)row * C;
        float4 g[VPL], xh[VPL];
        float s_gg = 0.f, s_ggx = 0.f;
#pragma unroll
        for (int k = 0; k < VPL; ++k) {
            const int c4 = lane + 32 * k;
            g[k] = load4(grad_out + off, c4);
            if (grad_out_bf16 != nullptr) {
                const float4 q = load4(grad_out_bf16 + off, c4);
                g[k] = make_float4(g[k].x + q.x, g[k].y + q.y, g[k].z + q.z, g[k].w + q.w);
            }
            if (grad_out_pos_bf16 != nullptr) {
                const float4 q = load4(grad_out_pos_bf16 + off, c4);
                g[k] = make_float4(g[k].x + q.x, g[k].y + q.y, g[k].z + q.z, g[k].w + q.w);
            }
            const float4 hv = load4(h + off, c4), ga = load4(gamma, c4);
            xh[k] = make_float4((hv.x - mr.x) * mr.y, (hv.y - mr.x) * mr.y, (hv.z - mr.x) * mr.y, (hv.w - mr.x) * mr.y);
            const float4 gg = make_float4(ga.x * g[k].x, ga.y * g[k].y, ga.z * g[k].z, ga.w * g[k].w);
            s_gg += (gg.x + gg.y) + (gg.z + gg.w);
            s_ggx += (gg.x * xh[k].x + gg.y * xh[k].y) + (gg.z * xh[k].z + gg.w * xh[k].w);
            add4(p_gx[k], make_float4(g[k].x * xh[k].x, g[k].y * xh[k].y, g[k].z * xh[k].z, g[k].w * xh[k].w));
            add4(p_g[k], g[k]);
        }
        const float m1 = warp_sum(s_gg) * (1.f / C), m2 = warp_sum(s_ggx) * (1.f / C);
#pragma unroll
        for (int k = 0; k < VPL; ++k) {
            const int c4 = lane + 32 * k;
            const float4 ga = load4(gamma, c4);
            float4 gh;
            gh.x = mr.y * ((ga.x * g[k].x - m1) - xh[k].x * m2);
            gh.y = mr.y * ((ga.y * g[k].y - m1) - xh[k].y * m2);
            gh.z = mr.y * ((ga.z * g[k].z - m1) - xh[k].z * m2);
            gh.w = mr.y * ((ga.w * g[k].w - m1) - xh[k].w * m2);
            store4(grad_residual + off, c4, gh);
            if (keep_mask != nullptr) {
                const float4 m = load_mask4(keep_mask + off, c4);
                gh = make_float4(gh.x * keep_scale * m.x, gh.y * keep_scale * m.y, gh.z * keep_scale * m.z,
                                 gh.w * keep_scale * m.w);
            }
            store4_bf16(grad_y + off, c4, gh);
            add4(p_gy[k], gh);                              // fp32: grad_bias is summed before the bf16 rounding
        }
    }
    float *prow = partials + (size_t)blockIdx.x * 3 * C;
    cta_partial<VPL>(red, p_gx, prow);
    cta_partial<VPL>(red, p_g, prow + C);
    cta_partial<VPL>(red, p_gy, prow + 2 * C);
}

template <typename Residual>
cudaError_t launch_forward(const __nv_bfloat16 *y, const float *bias, const Residual *residual,
                           const uint8_t *keep_mask, float keep_scale, const float *gamma, const float *beta,
                           const float *pos, float *out, __nv_bfloat16 *out_bf16, __nv_bfloat16 *out_pos_bf16,
                           float *h, float2 *mean_rstd, int64_t rows, int cols, float eps, cudaStream_t s)
{
    const int64_t blocks = (rows + kWarps - 1) / kWarps;
#define MSDA_AMP_TRAIN_FWD(V)                                                                                        \
    case V:                                                                                                          \
        layer_tail_amp_train_fwd_kernel<V, Residual><<<(unsigned)blocks, 32 * kWarps, 0, s>>>(                      \
            y, bias, residual, keep_mask, keep_scale, gamma, beta, pos, out, out_bf16, out_pos_bf16, h, mean_rstd,   \
            rows, eps);                                                                                              \
        break;
    switch (cols / 128) {
        MSDA_AMP_TRAIN_FWD(1) MSDA_AMP_TRAIN_FWD(2) MSDA_AMP_TRAIN_FWD(3) MSDA_AMP_TRAIN_FWD(4)
        MSDA_AMP_TRAIN_FWD(5) MSDA_AMP_TRAIN_FWD(6) MSDA_AMP_TRAIN_FWD(7) MSDA_AMP_TRAIN_FWD(8)
    }
#undef MSDA_AMP_TRAIN_FWD
    return cudaGetLastError();
}

template <typename Residual>
cudaError_t launch_backward(const float *grad_out, const __nv_bfloat16 *grad_out_bf16,
                            const __nv_bfloat16 *grad_out_pos_bf16, const float *h, const float2 *mean_rstd,
                            const uint8_t *keep_mask, float keep_scale, const float *gamma, Residual *grad_residual,
                            __nv_bfloat16 *grad_y, float *param_grads, float *partials, int64_t rows, int cols,
                            cudaStream_t s)
{
    const int blocks = bwd_blocks(rows), n = 3 * cols;
#define MSDA_AMP_TRAIN_BWD(V)                                                                                        \
    case V:                                                                                                          \
        layer_tail_amp_train_bwd_kernel<V, Residual><<<blocks, 32 * kWarps, 0, s>>>(                                \
            grad_out, grad_out_bf16, grad_out_pos_bf16, h, mean_rstd, keep_mask, keep_scale, gamma, grad_residual,   \
            grad_y, partials, rows);                                                                                 \
        break;
    switch (cols / 128) {
        MSDA_AMP_TRAIN_BWD(1) MSDA_AMP_TRAIN_BWD(2) MSDA_AMP_TRAIN_BWD(3) MSDA_AMP_TRAIN_BWD(4)
        MSDA_AMP_TRAIN_BWD(5) MSDA_AMP_TRAIN_BWD(6) MSDA_AMP_TRAIN_BWD(7) MSDA_AMP_TRAIN_BWD(8)
    }
#undef MSDA_AMP_TRAIN_BWD
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    layer_tail_param_sum_kernel<<<(n + 255) / 256, 256, 0, s>>>(partials, param_grads, blocks, n);
    return cudaGetLastError();
}

int status_of(cudaError_t e)
{
    if (e == cudaSuccess) return MSDA_OK;
    g_last_cuda_error = (int)e;
    return MSDA_ERR_CUDA;
}

bool dtype_ok(int residual_dtype) { return residual_dtype == MSDA_DTYPE_F32 || residual_dtype == MSDA_DTYPE_BF16; }

}  // namespace

}  // namespace msda

extern "C" {

int msda_amp_train_abi_version(void) { return MSDA_AMP_TRAIN_ABI_VERSION; }

int msda_amp_train_last_cuda_error(void) { return msda::g_last_cuda_error; }

int msda_amp_train_layer_tail_forward(const void *y, const float *bias, const void *residual, int residual_dtype,
                                      const uint8_t *keep_mask, float keep_scale, const float *gamma,
                                      const float *beta, const float *pos, float *out, void *out_bf16,
                                      void *out_plus_pos_bf16, float *h, float *mean_rstd, int64_t rows, int cols,
                                      float eps, void *stream)
{
    if (!msda::dtype_ok(residual_dtype)) return MSDA_ERR_UNSUPPORTED_DTYPE;
    if (rows < 0 || !msda::cols_ok(cols) || !(eps >= 0.f) || !msda::scale_ok(keep_scale))
        return MSDA_ERR_INVALID_ARGUMENT;
    if ((pos == nullptr) != (out_plus_pos_bf16 == nullptr)) return MSDA_ERR_INVALID_ARGUMENT;
    if (rows == 0) return MSDA_OK;
    const void *required[] = {y, residual, gamma, beta, out, h, mean_rstd};
    for (const void *p : required)
        if (p == nullptr || msda::misaligned(p)) return MSDA_ERR_INVALID_ARGUMENT;
    if (msda::misaligned(bias) || msda::misaligned(keep_mask) || msda::misaligned(pos) || msda::misaligned(out_bf16) ||
        msda::misaligned(out_plus_pos_bf16))
        return MSDA_ERR_INVALID_ARGUMENT;
    if ((rows + msda::kWarps - 1) / msda::kWarps > 0x7fffffff) return MSDA_ERR_INVALID_ARGUMENT;
    const auto *y16 = static_cast<const __nv_bfloat16 *>(y);
    auto *o16 = static_cast<__nv_bfloat16 *>(out_bf16), *op16 = static_cast<__nv_bfloat16 *>(out_plus_pos_bf16);
    auto *mr = reinterpret_cast<float2 *>(mean_rstd);
    const auto s = static_cast<cudaStream_t>(stream);
    const cudaError_t e =
        residual_dtype == MSDA_DTYPE_F32
            ? msda::launch_forward(y16, bias, static_cast<const float *>(residual), keep_mask, keep_scale, gamma, beta,
                                   pos, out, o16, op16, h, mr, rows, cols, eps, s)
            : msda::launch_forward(y16, bias, static_cast<const __nv_bfloat16 *>(residual), keep_mask, keep_scale,
                                   gamma, beta, pos, out, o16, op16, h, mr, rows, cols, eps, s);
    return msda::status_of(e);
}

size_t msda_amp_train_layer_tail_workspace_bytes(int64_t rows, int cols)
{
    if (rows <= 0 || !msda::cols_ok(cols)) return 0;
    // one partial row of 3 C per CTA
    return (size_t)msda::bwd_blocks(rows) * 3 * cols * sizeof(float);
}

int msda_amp_train_layer_tail_backward(const float *grad_out, const void *grad_out_bf16,
                                       const void *grad_out_plus_pos_bf16, const float *h, const float *mean_rstd,
                                       const uint8_t *keep_mask, float keep_scale, const float *gamma,
                                       void *grad_residual, int residual_dtype, void *grad_y, float *param_grads,
                                       float *partials, int64_t rows, int cols, void *stream)
{
    if (!msda::dtype_ok(residual_dtype)) return MSDA_ERR_UNSUPPORTED_DTYPE;
    if (rows < 0 || !msda::cols_ok(cols) || !msda::scale_ok(keep_scale)) return MSDA_ERR_INVALID_ARGUMENT;
    if (rows == 0) return MSDA_OK;
    const void *required[] = {grad_out, h, mean_rstd, gamma, grad_residual, grad_y, param_grads, partials};
    for (const void *p : required)
        if (p == nullptr || msda::misaligned(p)) return MSDA_ERR_INVALID_ARGUMENT;
    if (msda::misaligned(grad_out_bf16) || msda::misaligned(grad_out_plus_pos_bf16) || msda::misaligned(keep_mask))
        return MSDA_ERR_INVALID_ARGUMENT;
    const auto *g16 = static_cast<const __nv_bfloat16 *>(grad_out_bf16);
    const auto *gp16 = static_cast<const __nv_bfloat16 *>(grad_out_plus_pos_bf16);
    const auto *mr = reinterpret_cast<const float2 *>(mean_rstd);
    auto *gy = static_cast<__nv_bfloat16 *>(grad_y);
    const auto s = static_cast<cudaStream_t>(stream);
    const cudaError_t e =
        residual_dtype == MSDA_DTYPE_F32
            ? msda::launch_backward(grad_out, g16, gp16, h, mr, keep_mask, keep_scale, gamma,
                                    static_cast<float *>(grad_residual), gy, param_grads, partials, rows, cols, s)
            : msda::launch_backward(grad_out, g16, gp16, h, mr, keep_mask, keep_scale, gamma,
                                    static_cast<__nv_bfloat16 *>(grad_residual), gy, param_grads, partials, rows,
                                    cols, s);
    return msda::status_of(e);
}

}  // extern "C"
