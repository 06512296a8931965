// Kernels of the neighbour-frame pre-summation (see msda_frames.cu), shared by libmsda_b200.so (fp32 and bf16) and
// libmsda_b200_f16.so (fp16, csrc_f16/): each library instantiates them for its own element types.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "msda_internal.h"

namespace msda {

namespace {

constexpr int kMaxRegFrames = 8;  // frames / slots held in registers; more falls back to re-reading

template <typename ET> struct Vec16;

template <> struct Vec16<float> {
    static constexpr int N = 4;
    float x[4];
    static __device__ __forceinline__ Vec16 load(const float *p)
    {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(p));
        Vec16 r;
        r.x[0] = v.x; r.x[1] = v.y; r.x[2] = v.z; r.x[3] = v.w;
        return r;
    }
    __device__ __forceinline__ void store(float *p) const
    {
        *reinterpret_cast<float4 *>(p) = make_float4(x[0], x[1], x[2], x[3]);
    }
};

template <> struct Vec16<__nv_bfloat16> {
    static constexpr int N = 8;
    float x[8];
    static __device__ __forceinline__ Vec16 load(const __nv_bfloat16 *p)
    {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p));
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
        Vec16 r;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            r.x[2 * i] = __uint_as_float(w[i] << 16);
            r.x[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
        return r;
    }
    __device__ __forceinline__ void store(__nv_bfloat16 *p) const
    {
        unsigned w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const __nv_bfloat162 t = __floats2bfloat162_rn(x[2 * i], x[2 * i + 1]);
            w[i] = *reinterpret_cast<const unsigned *>(&t);
        }
        *reinterpret_cast<uint4 *>(p) = make_uint4(w[0], w[1], w[2], w[3]);
    }
};

template <> struct Vec16<__half> {
    static constexpr int N = 8;
    float x[8];
    static __device__ __forceinline__ Vec16 load(const __half *p)
    {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p));
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
        Vec16 r;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&w[i]));
            r.x[2 * i] = f.x;
            r.x[2 * i + 1] = f.y;
        }
        return r;
    }
    __device__ __forceinline__ void store(__half *p) const
    {
        unsigned w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const __half2 t = __floats2half2_rn(x[2 * i], x[2 * i + 1]);
            w[i] = *reinterpret_cast<const unsigned *>(&t);
        }
        *reinterpret_cast<uint4 *>(p) = make_uint4(w[0], w[1], w[2], w[3]);
    }
};

// four fp32 channels rounded once to nearest even into 8 bytes of a 16-bit type (overflow gives +-inf)
__device__ __forceinline__ uint2 pack4(const float4 &g, const __nv_bfloat16 *)
{
    const __nv_bfloat162 lo = __floats2bfloat162_rn(g.x, g.y), hi = __floats2bfloat162_rn(g.z, g.w);
    return make_uint2(*reinterpret_cast<const unsigned *>(&lo), *reinterpret_cast<const unsigned *>(&hi));
}

__device__ __forceinline__ uint2 pack4(const float4 &g, const __half *)
{
    const __half2 lo = __floats2half2_rn(g.x, g.y), hi = __floats2half2_rn(g.z, g.w);
    return make_uint2(*reinterpret_cast<const unsigned *>(&lo), *reinterpret_cast<const unsigned *>(&hi));
}

// bit i set <=> channel i of this thread's chunk is masked
template <int N>
__device__ __forceinline__ unsigned mask_bits(const uint8_t *__restrict__ mp, int col_stride)
{
    if (col_stride == 0) return __ldg(mp) ? (1u << N) - 1u : 0u;
    unsigned bits = 0u;
#pragma unroll
    for (int w = 0; w < N / 4; ++w) {
        const unsigned mk = __ldg(reinterpret_cast<const unsigned *>(mp) + w);
#pragma unroll
        for (int b = 0; b < 4; ++b)
            if ((mk >> (8 * b)) & 0xffu) bits |= 1u << (4 * w + b);
    }
    return bits;
}

struct FrameArgs {
    int N, T2, T1, n_frame, S, C;   // C = M * D elements per row
    int n_local, has_all, NS;       // slot structure
    int64_t value_stride_n, value_stride_t;  // elements
    int64_t mask_row_stride;
    int mask_col_stride;
    int chunks_per_row;             // C / Vec16::N
    int64_t total;                  // N * S * chunks_per_row threads
};

__device__ __forceinline__ void slot_range(int j, const FrameArgs &a, int &lo, int &hi)
{
    if (j < a.n_local) { lo = max(j - 1, 0); hi = min(j + 1, a.n_frame - 1); }
    else { lo = 0; hi = a.T2 - 1; }
}

template <typename ET>
__global__ void __launch_bounds__(256)
frame_sum_kernel(const ET *__restrict__ value, const uint8_t *__restrict__ mask, ET *__restrict__ vsum,
                 const FrameArgs a)
{
    using V = Vec16<ET>;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.total) return;
    const int64_t row = i / a.chunks_per_row;
    const int c0 = (int)(i - row * a.chunks_per_row) * V::N;
    const int n = (int)(row / a.S);
    const int s = (int)(row - (int64_t)n * a.S);
    const ET *vp = value + n * a.value_stride_n + (int64_t)s * a.C + c0;
    const uint8_t *mp = mask ? mask + ((int64_t)n * a.T2 * a.S + s) * a.mask_row_stride + (int64_t)c0 * a.mask_col_stride
                             : nullptr;
    const int64_t mask_frame = (int64_t)a.S * a.mask_row_stride;
    ET *op = vsum + (((int64_t)n * a.NS) * a.S + s) * a.C + c0;
    const int64_t out_frame = (int64_t)a.S * a.C;

    auto load_frame = [&](int t) {
        V v = V::load(vp + t * a.value_stride_t);
        if (mp != nullptr) {
            const unsigned bits = mask_bits<V::N>(mp + t * mask_frame, a.mask_col_stride);
#pragma unroll
            for (int k = 0; k < V::N; ++k)
                if (bits & (1u << k)) v.x[k] = 0.f;
        }
        return v;
    };

    if (a.T2 <= kMaxRegFrames) {
        V f[kMaxRegFrames];
#pragma unroll
        for (int t = 0; t < kMaxRegFrames; ++t)
            if (t < a.T2) f[t] = load_frame(t);
        for (int j = 0; j < a.NS; ++j) {
            int lo, hi;
            slot_range(j, a, lo, hi);
            V acc;
#pragma unroll
            for (int k = 0; k < V::N; ++k) acc.x[k] = 0.f;
#pragma unroll
            for (int t = 0; t < kMaxRegFrames; ++t)
                if (t >= lo && t <= hi) {
#pragma unroll
                    for (int k = 0; k < V::N; ++k) acc.x[k] += f[t].x[k];
                }
            acc.store(op + j * out_frame);
        }
    } else {
        for (int j = 0; j < a.NS; ++j) {
            int lo, hi;
            slot_range(j, a, lo, hi);
            V acc = load_frame(lo);
            for (int t = lo + 1; t <= hi; ++t) {
                const V v = load_frame(t);
#pragma unroll
                for (int k = 0; k < V::N; ++k) acc.x[k] += v.x[k];
            }
            acc.store(op + j * out_frame);
        }
    }
}

// grad_vsum is fp32 (the backward kernels accumulate in fp32 whatever the value type is); OT = element
// type of grad_value.  One thread per 4 channels (16 bytes of fp32).
template <typename OT>
__global__ void __launch_bounds__(256)
frame_unsum_kernel(const float *__restrict__ gsum, const uint8_t *__restrict__ mask, OT *__restrict__ grad_value,
                   const FrameArgs a)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.total) return;
    const int64_t row = i / a.chunks_per_row;
    const int c0 = (int)(i - row * a.chunks_per_row) * 4;
    const int n = (int)(row / a.S);
    const int s = (int)(row - (int64_t)n * a.S);
    const int64_t frame = (int64_t)a.S * a.C;
    const float *gp = gsum + (((int64_t)n * a.NS) * a.S + s) * a.C + c0;
    OT *op = grad_value + (((int64_t)n * a.T2) * a.S + s) * a.C + c0;
    const uint8_t *mp = mask ? mask + ((int64_t)n * a.T2 * a.S + s) * a.mask_row_stride + (int64_t)c0 * a.mask_col_stride
                             : nullptr;
    const int64_t mask_frame = (int64_t)a.S * a.mask_row_stride;

    auto store = [&](int t, float4 g) {
        if (mp != nullptr) {
            const unsigned bits = mask_bits<4>(mp + t * mask_frame, a.mask_col_stride);
            if (bits & 1u) g.x = 0.f;
            if (bits & 2u) g.y = 0.f;
            if (bits & 4u) g.z = 0.f;
            if (bits & 8u) g.w = 0.f;
        }
        if constexpr (sizeof(OT) == 4)
            *reinterpret_cast<float4 *>(op + t * frame) = g;
        else
            *reinterpret_cast<uint2 *>(op + t * frame) = pack4(g, op);
    };
    auto add = [](float4 &acc, const float4 &v) { acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; };

    if (a.NS <= kMaxRegFrames) {
        float4 g[kMaxRegFrames];
#pragma unroll
        for (int j = 0; j < kMaxRegFrames; ++j)
            if (j < a.NS) g[j] = __ldg(reinterpret_cast<const float4 *>(gp + j * frame));
        for (int t = 0; t < a.T2; ++t) {
            // slots whose frame range contains t: local slots t-1, t, t+1 (t < n_frame) and the all-frames slot
            const int lo = t < a.n_frame ? max(t - 1, 0) : a.n_local;
            const int hi = t < a.n_frame ? min(t + 1, a.n_local - 1) : a.n_local - 1;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int j = 0; j < kMaxRegFrames; ++j)
                if ((j >= lo && j <= hi) || (a.has_all && j == a.n_local)) add(acc, g[j]);
            store(t, acc);
        }
    } else {
        for (int t = 0; t < a.T2; ++t) {
            const int lo = t < a.n_frame ? max(t - 1, 0) : a.n_local;
            const int hi = t < a.n_frame ? min(t + 1, a.n_local - 1) : a.n_local - 1;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int j = lo; j <= hi; ++j) add(acc, __ldg(reinterpret_cast<const float4 *>(gp + j * frame)));
            if (a.has_all) add(acc, __ldg(reinterpret_cast<const float4 *>(gp + a.n_local * frame)));
            store(t, acc);
        }
    }
}

FrameArgs make_frame_args(const FrameDims &d, int vec)
{
    FrameArgs a;
    a.N = d.N; a.T2 = d.T2; a.T1 = d.T1; a.n_frame = d.n_frame; a.S = d.S; a.C = d.C;
    a.n_local = d.T1 < d.n_frame ? d.T1 : d.n_frame;
    a.has_all = d.T1 > d.n_frame ? 1 : 0;
    a.NS = a.n_local + a.has_all;
    a.value_stride_n = d.value_stride_n;
    a.value_stride_t = d.value_stride_t;
    a.mask_row_stride = d.mask_row_stride;
    a.mask_col_stride = d.mask_col_stride;
    a.chunks_per_row = d.C / vec;
    a.total = (int64_t)d.N * d.S * a.chunks_per_row;
    return a;
}


// ET = float (16-byte rows of 4 channels) or a 16-bit type (8 channels)
template <typename ET>
cudaError_t launch_frame_sum_typed(const ET *value, const uint8_t *mask, ET *vsum, const FrameDims &d, cudaStream_t stream)
{
    const FrameArgs a = make_frame_args(d, 16 / (int)sizeof(ET));
    if (a.total == 0) return cudaSuccess;
    const int64_t blocks = (a.total + 255) / 256;
    if (blocks > 0x7fffffff) return cudaErrorInvalidValue;
    frame_sum_kernel<ET><<<(unsigned)blocks, 256, 0, stream>>>(value, mask, vsum, a);
    return cudaGetLastError();
}

// OT = element type of grad_value (float or a 16-bit type, each rounded once from the fp32 sum)
template <typename OT>
cudaError_t launch_frame_unsum_typed(const float *grad_vsum, const uint8_t *mask, OT *grad_value, const FrameDims &d,
                                     cudaStream_t stream)
{
    const FrameArgs a = make_frame_args(d, 4);
    if (a.total == 0) return cudaSuccess;
    const int64_t blocks = (a.total + 255) / 256;
    if (blocks > 0x7fffffff) return cudaErrorInvalidValue;
    frame_unsum_kernel<OT><<<(unsigned)blocks, 256, 0, stream>>>(grad_vsum, mask, grad_value, a);
    return cudaGetLastError();
}

}  // namespace

}  // namespace msda
