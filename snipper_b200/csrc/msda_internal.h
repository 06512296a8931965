// Internal launcher interface between the C ABI (msda_capi.cu) and the kernel files.
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace msda {

constexpr int kMaxLevels = 64;
constexpr int kSnippetMaxLP = 32;   // L * P of the fused snippet kernels
constexpr int kPlanarD = 48;        // fp32 head channels the planar slot layout is built for: 128-byte plane + 64-byte plane

// Dynamic shared memory above which a launcher opts in with cudaFuncAttributeMaxDynamicSharedMemorySize: the 48 KB
// default limit covers STATIC + dynamic shared memory, and every kernel here also holds a static level table (~1 KB).
constexpr size_t kSmemOptIn = 44 * 1024;

struct OpDims {
    int N, S, M, D, L, Lq, P;
    int64_t value_batch_stride;  // elements
    // deterministic grad_value only: batch item b scatters into frame
    //     (b / frame_q) * frame_slots + min(b % frame_q, frame_local)
    // of grad_value -- the per-query-frame slots of the fused layer (msda_frames.cu); frame_q == 0: frame b
    int frame_q = 0, frame_local = 0, frame_slots = 0;
};

struct SnippetDims {
    int N, T2, T1, n_frame, S, M, D, L, Lq, P;
    int64_t value_stride_n, value_stride_t;  // elements
    int64_t ref_stride_n, ref_stride_t;      // elements
    // offsets / logits (and their gradients) may be column blocks of ONE projection output
    // (the module runs both Linear layers as a single GEMM): floats between consecutive (n,t1,q) rows
    int64_t off_row_stride, logit_row_stride;
    // optional biases of the two Linear layers, added here instead of in a GEMM epilogue kernel
    const float *off_bias;    // (M, L, P, 2) or nullptr
    const float *logit_bias;  // (M, L, P) or nullptr
    // encoder self-attention only (Lq == S, query q IS pixel q of the pyramid): when non-null the reference points are
    // computed in-kernel from the query index instead of being read -- (N, L, 2) valid ratios (w, h) as built by
    // DeformableTransformer.get_valid_ratio; reproduces get_reference_points (deformable_transformer.py:219-232) bit for bit
    const float *valid_ratios;
    // presummed: `value` (and grad_value) hold one frame per SLOT (msda_frames.cu) instead of one per
    // source frame: (N, n_slots, S, M, D) with the strides above; each query frame gathers exactly one
    int presummed;
    // optional padding mask applied to the gathered value / the scattered grad_value (direct mode only):
    // element (n,t,s,c) at mask[((n*T2+t)*S+s)*mask_row_stride + c*mask_col_stride], col stride 0 or 1
    const uint8_t *mask;
    int64_t mask_row_stride;
    int mask_col_stride;
};

// neighbour-frame pre-summation (msda_frames.cu)
struct FrameDims {
    int N, T2, T1, n_frame, S, C;            // C = M * D
    int64_t value_stride_n, value_stride_t;  // elements (frame_sum input only)
    int64_t mask_row_stride;
    int mask_col_stride;
};

// ---- per-call op (msda_percall.cu) ----
// fast = vectorised fp32 path (D % 16 == 0, D <= 256); generic = any D, float or double.
// esize = sizeof(VT): 4 (float) or 2 (bf16 / fp16)
inline bool fast_path_ok(const OpDims &d, int esize)
{
    const int epl = 16 / esize;                    // channels per 16-byte lane
    if (d.D % epl != 0) return false;
    const int lanes = d.D / epl;
    if (lanes % 2 != 0 || lanes > 32) return false;
    if (esize == 4 && lanes % 4 != 0) return false;  // fp32 instantiations: LANES in {4,8,...,32}
    if (esize == 2 && lanes != 2 && lanes != 4 && lanes != 6 && lanes != 8 && lanes != 12 && lanes != 16) return false;
    if (d.L > kMaxLevels) return false;
    if ((d.value_batch_stride * esize) % 16 != 0) return false;
    // 28-bit row stride / 31-bit cell offsets in bytes (SampleMeta)
    if ((int64_t)d.S * d.M * d.D * esize >= ((int64_t)1 << 28)) return false;
    // grid dimensions (y: query tiles, z: batch) and the 24-bit fast_div range
    if (d.N > 65535 || (d.Lq + 7) / 8 > 65535) return false;
    if ((int64_t)d.L * d.P >= 4096) return false;
    return true;
}

inline bool fast_path_ok(const OpDims &d) { return fast_path_ok(d, 4); }

// bf16 value / output / grad_output, fp32 everything else (grad_value accumulates in fp32)
cudaError_t launch_forward_fast_bf16(const void *value, const int64_t *shapes, const int64_t *lsi,
                                     const float *loc, const float *attn, void *out,
                                     const OpDims &d, cudaStream_t stream);
cudaError_t launch_backward_fast_bf16(const void *value, const int64_t *shapes, const int64_t *lsi,
                                      const float *loc, const float *attn, const void *grad_out,
                                      float *grad_value, float *grad_loc, float *grad_attn,
                                      const OpDims &d, cudaStream_t stream);

cudaError_t launch_forward_fast_f32(const float *value, const int64_t *shapes, const int64_t *lsi,
                                    const float *loc, const float *attn, float *out,
                                    const OpDims &d, cudaStream_t stream);
cudaError_t launch_backward_fast_f32(const float *value, const int64_t *shapes, const int64_t *lsi,
                                     const float *loc, const float *attn, const float *grad_out,
                                     float *grad_value, float *grad_loc, float *grad_attn,
                                     const OpDims &d, cudaStream_t stream);

template <typename T>
cudaError_t launch_forward_generic(const T *value, const int64_t *shapes, const int64_t *lsi,
                                   const T *loc, const T *attn, T *out, const OpDims &d,
                                   cudaStream_t stream);
template <typename T>
cudaError_t launch_backward_generic(const T *value, const int64_t *shapes, const int64_t *lsi,
                                    const T *loc, const T *attn, const T *grad_out,
                                    T *grad_value, T *grad_loc, T *grad_attn, const OpDims &d,
                                    cudaStream_t stream);

// ---- deterministic backward (msda_deterministic.cu) ----
size_t deterministic_workspace_bytes(const OpDims &d);
cudaError_t launch_backward_deterministic_f32(const float *value, const int64_t *shapes,
                                              const int64_t *lsi, const float *loc,
                                              const float *attn, const float *grad_out,
                                              float *grad_value, float *grad_loc, float *grad_attn,
                                              const OpDims &d, void *workspace, cudaStream_t stream,
                                              bool accumulate);

// grad_value part of the above alone (count / scan / fill / ordered reduce); loc / attn per sample, (N,Lq,M,L,P[,2])
cudaError_t launch_deterministic_grad_value_f32(const int64_t *shapes, const int64_t *lsi, const float *loc,
                                                const float *attn, const float *grad_out, float *grad_value,
                                                const OpDims &d, void *workspace, cudaStream_t stream,
                                                bool accumulate);

// ---- in-place masked zero-fill (msda_mask.cu) ----
cudaError_t launch_masked_zero(void *data, const uint8_t *mask, int64_t n, int elem_bytes, cudaStream_t stream);

// ---- layer tail: bias + residual + LayerNorm (+ pos) in one pass (msda_tail.cu) ----
bool layer_tail_ok(int cols);
cudaError_t launch_layer_tail(const float *y, const float *bias, const float *residual, const float *gamma,
                              const float *beta, const float *pos, float *out, float *out_pos, int64_t rows,
                              int cols, float eps, cudaStream_t stream);

// ---- neighbour-frame pre-summation (msda_frames.cu) ----
inline int snippet_num_slots(int T1, int n_frame) { return (T1 < n_frame ? T1 : n_frame) + (T1 > n_frame ? 1 : 0); }

inline bool frame_dims_ok(const FrameDims &d, int esize)
{
    const int vec = 16 / esize;
    if (d.N < 0 || d.T2 <= 0 || d.T1 <= 0 || d.n_frame <= 0 || d.n_frame > d.T2 || d.S <= 0 || d.C <= 0) return false;
    if (d.C % vec != 0 || d.C % 4 != 0) return false;
    if ((d.value_stride_n * esize) % 16 != 0 || (d.value_stride_t * esize) % 16 != 0) return false;
    if (d.mask_col_stride != 0 && d.mask_col_stride != 1) return false;
    // per-channel masks are read as 32-bit words: rows must start on a 4-byte boundary
    if (d.mask_col_stride == 1 && d.mask_row_stride % 4 != 0) return false;
    if ((int64_t)d.N * d.S * (d.C / 4) >= ((int64_t)1 << 40)) return false;
    return true;
}

cudaError_t launch_frame_sum(const void *value, const uint8_t *mask, void *vsum, const FrameDims &d, int esize,
                             cudaStream_t stream);
cudaError_t launch_frame_unsum(const float *grad_vsum, const uint8_t *mask, void *grad_value, const FrameDims &d,
                               int out_esize, cudaStream_t stream);

// ---- planar neighbour-frame slots (msda_planar.cu): fp32, D = 48 ----
// bytes of one (n, slot) of the planar layout, 0 when it does not apply
inline size_t planar_slot_bytes(int S, int M, int D, int esize)
{
    if (esize != 4 || D != kPlanarD || S <= 0 || M <= 0) return 0;
    const int64_t bytes = (int64_t)M * (S * (int64_t)128 + (int64_t)((S + 3) & ~1) * 128);
    if (bytes >= ((int64_t)1 << 31) - 256 || (int64_t)S * 16 >= ((int64_t)1 << 27)) return 0;
    return (size_t)bytes;
}
cudaError_t launch_frame_sum_planar(const float *value, const uint8_t *mask, void *vsum, const FrameDims &d, int M,
                                    cudaStream_t stream);
cudaError_t launch_frame_unsum_planar(const void *grad_vsum, const uint8_t *mask, float *grad_value, const FrameDims &d,
                                      int M, cudaStream_t stream);
cudaError_t launch_planar_forward_f32(const void *vsum, const int64_t *shapes, const int64_t *lsi, const float *offsets,
                                      const float *logits, const float *ref, float *out, const SnippetDims &d,
                                      cudaStream_t stream);
cudaError_t launch_planar_backward_f32(const void *vsum, const int64_t *shapes, const int64_t *lsi, const float *offsets,
                                       const float *logits, const float *ref, const float *grad_out, void *gsum,
                                       float *grad_offsets, float *grad_logits, const SnippetDims &d, cudaStream_t stream);

// ---- fused snippet op (msda_snippet.cu) ----
inline bool snippet_ok(const SnippetDims &d, int esize)
{
    const int epl = 16 / esize;
    if (d.D % epl != 0) return false;
    const int lanes = d.D / epl;
    if (esize == 4 && (lanes % 4 != 0 || lanes > 32)) return false;
    if (esize == 2 && lanes != 2 && lanes != 4 && lanes != 6 && lanes != 8 && lanes != 12 && lanes != 16) return false;
    if (d.L > kMaxLevels || d.L * d.P > kSnippetMaxLP) return false;
    if ((d.value_stride_n * esize) % 16 != 0 || (d.value_stride_t * esize) % 16 != 0) return false;
    if ((int64_t)d.S * d.M * d.D * esize >= ((int64_t)1 << 28)) return false;  // SampleMeta bit budget
    if ((int64_t)d.N * d.T1 > 65535 || (d.Lq + 7) / 8 > 65535) return false;
    return true;
}

inline bool snippet_ok(const SnippetDims &d) { return snippet_ok(d, 4); }
cudaError_t launch_snippet_forward_bf16(const void *value, const int64_t *shapes,
                                        const int64_t *lsi, const float *offsets,
                                        const float *logits, const float *ref, void *out,
                                        const SnippetDims &d, cudaStream_t stream);
cudaError_t launch_snippet_backward_bf16(const void *value, const int64_t *shapes,
                                         const int64_t *lsi, const float *offsets,
                                         const float *logits, const float *ref,
                                         const void *grad_out, float *grad_value,
                                         float *grad_offsets, float *grad_logits,
                                         const SnippetDims &d, cudaStream_t stream);
cudaError_t launch_snippet_forward_f32(const float *value, const int64_t *shapes,
                                       const int64_t *lsi, const float *offsets,
                                       const float *logits, const float *ref, float *out,
                                       const SnippetDims &d, cudaStream_t stream);
cudaError_t launch_snippet_backward_f32(const float *value, const int64_t *shapes,
                                        const int64_t *lsi, const float *offsets,
                                        const float *logits, const float *ref,
                                        const float *grad_out, float *grad_value,
                                        float *grad_offsets, float *grad_logits,
                                        const SnippetDims &d, cudaStream_t stream);

// deterministic mode of the fused layer (presummed, fp32): everything but grad_value, no atomics anywhere ...
cudaError_t launch_snippet_backward_noscatter_f32(const float *value, const int64_t *shapes, const int64_t *lsi,
                                                  const float *offsets, const float *logits, const float *ref,
                                                  const float *grad_out, float *grad_offsets, float *grad_logits,
                                                  const SnippetDims &d, cudaStream_t stream);
// ... and the per-sample locations / weights the two-pass grad_value needs: loc (N*T1,Lq,M,L,P,2), attn (N*T1,Lq,M,L,P)
cudaError_t launch_snippet_loc_attn(const int64_t *shapes, const int64_t *lsi, const float *offsets,
                                    const float *logits, const float *ref, float *loc, float *attn,
                                    const SnippetDims &d, cudaStream_t stream);

}  // namespace msda
