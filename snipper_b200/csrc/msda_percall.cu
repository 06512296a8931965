// Per-call multi-scale deformable attention, forward + backward, sm_100a.
//
// Replaces the reference launchers ms_deformable_im2col_cuda / ms_deformable_col2im_cuda
// (models/ops/src/cuda/ms_deform_im2col_cuda.cuh:923-954, :956-1327) and the seven
// __global__ kernels behind them with two designs:
//
//  * FAST (fp32, D % 16 == 0, D <= 128 -- Snipper's D = 48 is the tuned case)
//      CTA = PAIRS (n,q,m) pairs x LANES (= D/4) lanes, "flat" mapping: consecutive lanes own
//      consecutive 16-byte channel chunks, so one warp-wide LDG.128 covers whole 192-byte
//      head slices (2.67 of them) and every gathered cell is read as full 32-byte sectors.
//      Phase 1: one thread per SAMPLE computes the bilinear set-up once (4 cell offsets +
//      weights) and parks it in shared memory -- the reference redoes this per channel.
//      Phase 2: each lane walks the samples of its pair: broadcast LDS of the record,
//      4 x predicated LDG.128 gathers, FFMA.  Backward additionally issues one
//      red.global.add.v4.f32 per corner per lane (4x fewer L2 atomics than scalar REDs),
//      reduces the three per-sample scalars over channels with 2 shuffles inside 4-lane
//      sub-groups + a tiny smem hop (no serial thread-0 tail, no __syncthreads per point).
//  * GENERIC (float / double, any D): straightforward one-thread-per-output-element forward
//      and one-warp-per-pair backward; used for fp64 parity tests and odd channel counts
//      (the reference's test list 30, 71, 1025, ... models/ops/test.py:85).
#include "msda_percall.cuh"

namespace msda {

cudaError_t launch_forward_fast_f32(const float *value, const int64_t *shapes, const int64_t *lsi,
                                    const float *loc, const float *attn, float *out,
                                    const OpDims &d, cudaStream_t stream)
{
    if (d.N * d.Lq * d.M == 0) return cudaSuccess;
    if (launch_fwd_split<float>(value, shapes, lsi, loc, attn, out, d, stream)) return cudaGetLastError();
#define CALL(VT, LN, PR) launch_fwd_fast<VT, LN, PR>(value, shapes, lsi, loc, attn, out, d, stream)
    MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
}

cudaError_t launch_backward_fast_f32(const float *value, const int64_t *shapes, const int64_t *lsi,
                                     const float *loc, const float *attn, const float *grad_out,
                                     float *grad_value, float *grad_loc, float *grad_attn,
                                     const OpDims &d, cudaStream_t stream)
{
    if (d.N * d.Lq * d.M == 0) return cudaSuccess;
#define CALL(VT, LN, PR) \
    launch_bwd_fast<VT, LN, PR>(value, shapes, lsi, loc, attn, grad_out, grad_value, grad_loc, grad_attn, d, stream)
    MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
}

cudaError_t launch_forward_fast_bf16(const void *value, const int64_t *shapes, const int64_t *lsi,
                                     const float *loc, const float *attn, void *out,
                                     const OpDims &d, cudaStream_t stream)
{
    return launch_forward_fast_half<__nv_bfloat16, bf16q>(value, shapes, lsi, loc, attn, out, d, stream);
}

cudaError_t launch_backward_fast_bf16(const void *value, const int64_t *shapes, const int64_t *lsi,
                                      const float *loc, const float *attn, const void *grad_out,
                                      float *grad_value, float *grad_loc, float *grad_attn,
                                      const OpDims &d, cudaStream_t stream)
{
    return launch_backward_fast_half<__nv_bfloat16, bf16q>(value, shapes, lsi, loc, attn, grad_out, grad_value,
                                                           grad_loc, grad_attn, d, stream);
}

// ------------------------------------------------------------------------------------------
// GENERIC path (float / double, any D)
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
msda_fwd_generic_kernel(const T *__restrict__ value, const int64_t *__restrict__ shapes,
                        const int64_t *__restrict__ lsi, const T *__restrict__ loc,
                        const T *__restrict__ attn, T *__restrict__ out,
                        int S, int M, int D, int L, int P, int Lq, int64_t total, int64_t value_batch_stride)
{
    __shared__ LevelTable lv;
    load_level_table(lv, shapes, lsi, L, S);
    __syncthreads();
    const int LP = L * P;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % D);
        const int64_t pair = idx / D;
        const int m = (int)(pair % M);
        const int64_t b = pair / ((int64_t)Lq * M);
        const T *vb = value + b * value_batch_stride + (int64_t)m * D + c;
        const int64_t cs = (int64_t)M * D;
        T acc = (T)0;
        for (int lp = 0; lp < LP; ++lp) {
            const int l = lp / P;
            const int64_t si = pair * LP + lp;
            const Sample<T> s = make_sample<T>(loc[2 * si], loc[2 * si + 1], lv.H[l], lv.W[l], lv.start[l]);
            const T hx = (T)1 - s.lx, hy = (T)1 - s.ly;
            T val = (T)0;
            if (s.cell[0] >= 0) val += hy * hx * vb[s.cell[0] * cs];
            if (s.cell[1] >= 0) val += hy * s.lx * vb[s.cell[1] * cs];
            if (s.cell[2] >= 0) val += s.ly * hx * vb[s.cell[2] * cs];
            if (s.cell[3] >= 0) val += s.ly * s.lx * vb[s.cell[3] * cs];
            acc += attn[si] * val;
        }
        out[idx] = acc;
    }
}

// one warp per (n,q,m) pair; lanes stride over channels
template <typename T>
__global__ void __launch_bounds__(256)
msda_bwd_generic_kernel(const T *__restrict__ value, const int64_t *__restrict__ shapes,
                        const int64_t *__restrict__ lsi, const T *__restrict__ loc,
                        const T *__restrict__ attn, const T *__restrict__ grad_out,
                        T *__restrict__ grad_value, T *__restrict__ grad_loc,
                        T *__restrict__ grad_attn,
                        int S, int M, int D, int L, int P, int Lq, int64_t total_pairs,
                        int64_t value_batch_stride, bool scatter)
{
    __shared__ LevelTable lv;
    load_level_table(lv, shapes, lsi, L, S);
    __syncthreads();
    const int LP = L * P;
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t cs = (int64_t)M * D;
    for (int64_t pair = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5); pair < total_pairs;
         pair += (int64_t)gridDim.x * warps_per_block) {
        const int m = (int)(pair % M);
        const int64_t b = pair / ((int64_t)Lq * M);
        const T *vb = value + b * value_batch_stride + (int64_t)m * D;
        T *gvb = grad_value + b * (int64_t)S * M * D + (int64_t)m * D;
        const T *g = grad_out + pair * D;
        for (int lp = 0; lp < LP; ++lp) {
            const int l = lp / P;
            const int64_t si = pair * LP + lp;
            const Sample<T> s = make_sample<T>(loc[2 * si], loc[2 * si + 1], lv.H[l], lv.W[l], lv.start[l]);
            const T a = attn[si];
            const T hx = (T)1 - s.lx, hy = (T)1 - s.ly;
            const T w0 = hy * hx, w1 = hy * s.lx, w2 = s.ly * hx, w3 = s.ly * s.lx;
            T pa = (T)0, px = (T)0, py = (T)0;
            for (int c = lane; c < D; c += 32) {
                const T gc = g[c];
                const T v0 = s.cell[0] >= 0 ? vb[s.cell[0] * cs + c] : (T)0;
                const T v1 = s.cell[1] >= 0 ? vb[s.cell[1] * cs + c] : (T)0;
                const T v2 = s.cell[2] >= 0 ? vb[s.cell[2] * cs + c] : (T)0;
                const T v3 = s.cell[3] >= 0 ? vb[s.cell[3] * cs + c] : (T)0;
                const T ga = gc * a;
                if (scatter) {
                    if (s.cell[0] >= 0) atomicAdd(gvb + s.cell[0] * cs + c, w0 * ga);
                    if (s.cell[1] >= 0) atomicAdd(gvb + s.cell[1] * cs + c, w1 * ga);
                    if (s.cell[2] >= 0) atomicAdd(gvb + s.cell[2] * cs + c, w2 * ga);
                    if (s.cell[3] >= 0) atomicAdd(gvb + s.cell[3] * cs + c, w3 * ga);
                }
                pa += gc * (w0 * v0 + w1 * v1 + w2 * v2 + w3 * v3);
                px += gc * (hy * (v1 - v0) + s.ly * (v3 - v2));
                py += gc * (hx * (v2 - v0) + s.lx * (v3 - v1));
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                pa += __shfl_xor_sync(0xffffffffu, pa, o);
                px += __shfl_xor_sync(0xffffffffu, px, o);
                py += __shfl_xor_sync(0xffffffffu, py, o);
            }
            if (lane == 0) {
                grad_attn[si] = pa;
                grad_loc[2 * si] = (T)lv.W[l] * a * px;
                grad_loc[2 * si + 1] = (T)lv.H[l] * a * py;
            }
        }
    }
}

template <typename T>
cudaError_t launch_forward_generic(const T *value, const int64_t *shapes, const int64_t *lsi,
                                   const T *loc, const T *attn, T *out, const OpDims &d,
                                   cudaStream_t stream)
{
    const int64_t total = (int64_t)d.N * d.Lq * d.M * d.D;
    if (total == 0) return cudaSuccess;
    const int64_t blocks = (total + 255) / 256;
    const int grid = (int)(blocks < 148 * 64 ? blocks : 148 * 64);
    msda_fwd_generic_kernel<T><<<grid, 256, 0, stream>>>(value, shapes, lsi, loc, attn, out, d.S, d.M, d.D,
                                                         d.L, d.P, d.Lq, total, d.value_batch_stride);
    return cudaGetLastError();
}

template <typename T>
static cudaError_t launch_backward_generic_impl(const T *value, const int64_t *shapes, const int64_t *lsi,
                                                const T *loc, const T *attn, const T *grad_out,
                                                T *grad_value, T *grad_loc, T *grad_attn, const OpDims &d,
                                                cudaStream_t stream, bool scatter)
{
    const int64_t total_pairs = (int64_t)d.N * d.Lq * d.M;
    if (total_pairs == 0) return cudaSuccess;
    const int64_t blocks = (total_pairs + 7) / 8;
    const int grid = (int)(blocks < 148 * 64 ? blocks : 148 * 64);
    msda_bwd_generic_kernel<T><<<grid, 256, 0, stream>>>(value, shapes, lsi, loc, attn, grad_out,
                                                         grad_value, grad_loc, grad_attn, d.S, d.M,
                                                         d.D, d.L, d.P, d.Lq, total_pairs,
                                                         d.value_batch_stride, scatter);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_backward_generic(const T *value, const int64_t *shapes, const int64_t *lsi,
                                    const T *loc, const T *attn, const T *grad_out,
                                    T *grad_value, T *grad_loc, T *grad_attn, const OpDims &d,
                                    cudaStream_t stream)
{
    return launch_backward_generic_impl<T>(value, shapes, lsi, loc, attn, grad_out, grad_value, grad_loc,
                                           grad_attn, d, stream, true);
}

// grad_sampling_loc / grad_attn_weight only (used by the deterministic mode)
cudaError_t launch_backward_no_scatter_f32(const float *value, const int64_t *shapes, const int64_t *lsi,
                                           const float *loc, const float *attn, const float *grad_out,
                                           float *grad_loc, float *grad_attn, const OpDims &d,
                                           cudaStream_t stream)
{
    if (d.N * d.Lq * d.M == 0) return cudaSuccess;
    const bool vec_ok = (reinterpret_cast<uintptr_t>(value) & 15u) == 0 && (reinterpret_cast<uintptr_t>(grad_out) & 15u) == 0;
    if (fast_path_ok(d) && vec_ok) {
        float *none = nullptr;
#define CALL(VT, LN, PR) \
    launch_bwd_fast<VT, LN, PR, false>(value, shapes, lsi, loc, attn, grad_out, none, grad_loc, grad_attn, d, stream)
        MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
    }
    return launch_backward_generic_impl<float>(value, shapes, lsi, loc, attn, grad_out, nullptr, grad_loc,
                                               grad_attn, d, stream, false);
}

template cudaError_t launch_forward_generic<float>(const float *, const int64_t *, const int64_t *,
                                                   const float *, const float *, float *,
                                                   const OpDims &, cudaStream_t);
template cudaError_t launch_forward_generic<double>(const double *, const int64_t *, const int64_t *,
                                                    const double *, const double *, double *,
                                                    const OpDims &, cudaStream_t);
template cudaError_t launch_backward_generic<float>(const float *, const int64_t *, const int64_t *,
                                                    const float *, const float *, const float *,
                                                    float *, float *, float *, const OpDims &,
                                                    cudaStream_t);
template cudaError_t launch_backward_generic<double>(const double *, const int64_t *, const int64_t *,
                                                     const double *, const double *, const double *,
                                                     double *, double *, double *, const OpDims &,
                                                     cudaStream_t);

}  // namespace msda
