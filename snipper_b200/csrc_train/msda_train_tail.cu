// Layer tail for training (include/msda_b200_train.h), sm_100a.
//
// In training the reference's x = norm(x + dropout(Linear(..))) is, in stock PyTorch, a bias epilogue, a dropout, an
// add and a LayerNorm forward, and the matching backward passes.  These kernels do the forward in one pass and the
// backward in one pass plus a small ordered reduction of the parameter gradients.  The dropout keep-mask is an input
// (drawn by torch's generator), so the result can be checked exactly and runs repeat under a fixed seed.
//
// Forward: layer_tail_kernel's layout and arithmetic (snipper_b200/csrc/msda_tail.cu), operation for operation: one
// warp per row, VPL float4 per lane (channel 4 (lane + 32 k)), the row in registers, two-pass mean and variance.  It
// also writes h = residual + d (the LayerNorm input) and (mean, rstd) per row for the backward.
//
// Backward: a grid whose size depends on rows only; warp w of CTA b takes rows (b + gridDim k) * 8 + w in order,
// keeps its per-lane column partials of (g xhat, g, grad_y) in registers, and the CTA adds its 8 warps' partials in
// shared memory in warp order into one partial row.  layer_tail_param_sum_kernel adds the CTA rows in CTA order.  No
// atomics anywhere: the result is bit-reproducible.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/msda_b200_train.h"
#include "msda_train_common.cuh"

namespace msda {

namespace {

thread_local int g_last_cuda_error = 0;

template <int VPL>
__global__ void __launch_bounds__(256)
layer_tail_train_fwd_kernel(const float *__restrict__ y, const float *__restrict__ bias,
                            const float *__restrict__ residual, const uint8_t *__restrict__ keep_mask,
                            float keep_scale, const float *__restrict__ gamma, const float *__restrict__ beta,
                            const float *__restrict__ pos, float *__restrict__ out, float *__restrict__ out_pos,
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
            // layer_tail_kernel on the pre-dropped input with bias = NULL adds its zero bias: + 0.f keeps its bits
            // (it turns a dropped -0 into +0)
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
    // `mean` keeps layer_tail_kernel's only use, x - mean, which the compiler fuses into fma(total, -1/C, x) as it
    // does there; storing `mean` itself would make it round the product once and change the bits of `out`.  The
    // stored mean is that product rounded, by an operation the compiler neither fuses nor merges with `mean`.
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
        if (out_pos != nullptr) {
            const float4 p = load4(pos + row * C, c4);
            reinterpret_cast<float4 *>(out_pos + row * C)[c4] = make_float4(o.x + p.x, o.y + p.y, o.z + p.z, o.w + p.w);
        }
    }
}

// partials: one row of 3 C floats per CTA, [g xhat | g | grad_y]
template <int VPL>
__global__ void __launch_bounds__(256, VPL <= 3 ? 2 : 1)
layer_tail_train_bwd_kernel(const float *__restrict__ grad_out, const float *__restrict__ grad_out_pos,
                            const float *__restrict__ h, const float2 *__restrict__ mean_rstd,
                            const uint8_t *__restrict__ keep_mask, float keep_scale, const float *__restrict__ gamma,
                            float *__restrict__ grad_residual, float *__restrict__ grad_y,
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
            if (grad_out_pos != nullptr) {
                const float4 q = load4(grad_out_pos + off, c4);
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
            reinterpret_cast<float4 *>(grad_residual + off)[c4] = gh;
            if (keep_mask != nullptr) {
                const float4 m = load_mask4(keep_mask + off, c4);
                gh = make_float4(gh.x * keep_scale * m.x, gh.y * keep_scale * m.y, gh.z * keep_scale * m.z,
                                 gh.w * keep_scale * m.w);
            }
            reinterpret_cast<float4 *>(grad_y + off)[c4] = gh;
            add4(p_gy[k], gh);
        }
    }
    // the CTA's partial row: the 8 warps' partials added in warp order, one quantity at a time
    float *prow = partials + (size_t)blockIdx.x * 3 * C;
    cta_partial<VPL>(red, p_gx, prow);
    cta_partial<VPL>(red, p_g, prow + C);
    cta_partial<VPL>(red, p_gy, prow + 2 * C);
}

int status_of(cudaError_t e)
{
    if (e == cudaSuccess) return MSDA_OK;
    g_last_cuda_error = (int)e;
    return MSDA_ERR_CUDA;
}

}  // namespace

}  // namespace msda

extern "C" {

int msda_train_abi_version(void) { return MSDA_TRAIN_ABI_VERSION; }

int msda_train_last_cuda_error(void) { return msda::g_last_cuda_error; }

int msda_train_layer_tail_forward(const float *y, const float *bias, const float *residual, const uint8_t *keep_mask,
                                  float keep_scale, const float *gamma, const float *beta, const float *pos,
                                  float *out, float *out_plus_pos, float *h, float *mean_rstd, int64_t rows, int cols,
                                  float eps, void *stream)
{
    if (rows < 0 || !msda::cols_ok(cols) || !(eps >= 0.f) || !msda::scale_ok(keep_scale))
        return MSDA_ERR_INVALID_ARGUMENT;
    if ((pos == nullptr) != (out_plus_pos == nullptr)) return MSDA_ERR_INVALID_ARGUMENT;
    if (rows == 0) return MSDA_OK;
    const void *required[] = {y, residual, gamma, beta, out, h, mean_rstd};
    for (const void *p : required)
        if (p == nullptr || msda::misaligned(p)) return MSDA_ERR_INVALID_ARGUMENT;
    if (msda::misaligned(bias) || msda::misaligned(keep_mask) || msda::misaligned(pos) ||
        msda::misaligned(out_plus_pos))
        return MSDA_ERR_INVALID_ARGUMENT;
    const int64_t blocks = (rows + msda::kWarps - 1) / msda::kWarps;
    if (blocks > 0x7fffffff) return MSDA_ERR_INVALID_ARGUMENT;
    const auto s = static_cast<cudaStream_t>(stream);
    auto *mr = reinterpret_cast<float2 *>(mean_rstd);
#define MSDA_TRAIN_FWD(V)                                                                                            \
    case V:                                                                                                          \
        msda::layer_tail_train_fwd_kernel<V><<<(unsigned)blocks, 32 * msda::kWarps, 0, s>>>(                         \
            y, bias, residual, keep_mask, keep_scale, gamma, beta, pos, out, out_plus_pos, h, mr, rows, eps);        \
        break;
    switch (cols / 128) {
        MSDA_TRAIN_FWD(1) MSDA_TRAIN_FWD(2) MSDA_TRAIN_FWD(3) MSDA_TRAIN_FWD(4)
        MSDA_TRAIN_FWD(5) MSDA_TRAIN_FWD(6) MSDA_TRAIN_FWD(7) MSDA_TRAIN_FWD(8)
    }
#undef MSDA_TRAIN_FWD
    return msda::status_of(cudaGetLastError());
}

size_t msda_train_layer_tail_workspace_bytes(int64_t rows, int cols)
{
    if (rows <= 0 || !msda::cols_ok(cols)) return 0;
    // one partial row of 3 C per CTA
    return (size_t)msda::bwd_blocks(rows) * 3 * cols * sizeof(float);
}

int msda_train_layer_tail_backward(const float *grad_out, const float *grad_out_plus_pos, const float *h,
                                   const float *mean_rstd, const uint8_t *keep_mask, float keep_scale,
                                   const float *gamma, float *grad_residual, float *grad_y, float *param_grads,
                                   float *partials, int64_t rows, int cols, void *stream)
{
    if (rows < 0 || !msda::cols_ok(cols) || !msda::scale_ok(keep_scale)) return MSDA_ERR_INVALID_ARGUMENT;
    if (rows == 0) return MSDA_OK;
    const void *required[] = {grad_out, h, mean_rstd, gamma, grad_residual, grad_y, param_grads, partials};
    for (const void *p : required)
        if (p == nullptr || msda::misaligned(p)) return MSDA_ERR_INVALID_ARGUMENT;
    if (msda::misaligned(grad_out_plus_pos) || msda::misaligned(keep_mask)) return MSDA_ERR_INVALID_ARGUMENT;
    const auto s = static_cast<cudaStream_t>(stream);
    const auto *mr = reinterpret_cast<const float2 *>(mean_rstd);
    const int blocks = msda::bwd_blocks(rows), n = 3 * cols;
#define MSDA_TRAIN_BWD(V)                                                                                            \
    case V:                                                                                                          \
        msda::layer_tail_train_bwd_kernel<V><<<blocks, 32 * msda::kWarps, 0, s>>>(                                   \
            grad_out, grad_out_plus_pos, h, mr, keep_mask, keep_scale, gamma, grad_residual, grad_y, partials, rows);    \
        break;
    switch (cols / 128) {
        MSDA_TRAIN_BWD(1) MSDA_TRAIN_BWD(2) MSDA_TRAIN_BWD(3) MSDA_TRAIN_BWD(4)
        MSDA_TRAIN_BWD(5) MSDA_TRAIN_BWD(6) MSDA_TRAIN_BWD(7) MSDA_TRAIN_BWD(8)
    }
#undef MSDA_TRAIN_BWD
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return msda::status_of(e);
    msda::layer_tail_param_sum_kernel<<<(n + 255) / 256, 256, 0, s>>>(partials, param_grads, blocks, n);
    return msda::status_of(cudaGetLastError());
}

}  // extern "C"
