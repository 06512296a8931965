/*
 * msda_b200.h -- C ABI of the B200-native multi-scale deformable attention library
 * (libmsda_b200.so, hand-written sm_100a CUDA, no ATen / pybind / torch types).
 *
 * This is the drop-in boundary for the hot path of JimmyZou/Snipper.  Each entry point
 * names the reference interface it replaces (paths relative to the reference repo):
 *
 *   msda_forward            <- ms_deform_attn_forward / ms_deform_attn_cuda_forward
 *                              models/ops/src/ms_deform_attn.h:20-39,
 *                              models/ops/src/cuda/ms_deform_attn_cuda.cu:20-80,
 *                              launcher ms_deformable_im2col_cuda  ms_deform_im2col_cuda.cuh:923-954
 *   msda_backward           <- ms_deform_attn_backward / ms_deform_attn_cuda_backward
 *                              models/ops/src/ms_deform_attn.h:41-61,
 *                              models/ops/src/cuda/ms_deform_attn_cuda.cu:83-153,
 *                              launcher ms_deformable_col2im_cuda  ms_deform_im2col_cuda.cuh:956-1327
 *   msda_snippet_forward /  <- the per-frame loop of MSDeformAttn.forward
 *   msda_snippet_backward      models/ops/modules/ms_deform_attn.py:126-225 (offset normalisation,
 *                              softmax over levels x points x neighbour frames, one op call per
 *                              (t1,t2) pair, sum over t2) fused into one launch per layer
 *   msda_layer_tail         <- `x = x + dropout(Linear(..)); x = norm(x)` + `with_pos_embed` of the calling layers
 *                              models/deformable_transformer.py:188-205,270-295 (opt-in, SURVEY 8f rank 3)
 *   msda_frame_sum /        <- value.masked_fill(input_padding_mask, 0) (ms_deform_attn.py:116-117) and
 *   msda_frame_unsum           the stack(-1).sum(-1) over neighbour frames (:225), moved IN FRONT of the
 *                              gather by linearity of the op in `value` (one gather per query frame)
 *
 * Conventions
 *   - every pointer is a DEVICE pointer; the caller owns every buffer; the library allocates
 *     nothing, never synchronises and only enqueues work on `stream` (a cudaStream_t).
 *   - spatial_shapes (L,2) = (H_l, W_l) and level_start_index (L) are int64 ON THE DEVICE
 *     (the reference builds them there, models/deformable_transformer.py:100-101); they are
 *     read inside the kernels -- no host sync.
 *   - layouts as in the reference: value (N,S,M,D); sampling_loc (N,Lq,M,L,P,2) as (x,y) in
 *     [0,1] incl. padding; attn_weight (N,Lq,M,L,P); output (N,Lq,M*D).
 *   - every function returns an msda_status_t (0 = ok).  Launch failures are returned, not
 *     printed (the reference only printf()s them, ms_deform_im2col_cuda.cuh:948-952).
 *   - re-entrant and stateless: no entry point writes process state.  (Benchmark knobs are READ from the
 *     environment once, at the first launch; they change speed, not results beyond rounding: MSDA_PAIRS_D48 /
 *     MSDA_SNIP_PAIRS_D48 = 8|16|32 and MSDA_PLANAR_PAIRS = 16|32|64, queries per CTA tile, and
 *     MSDA_PLANAR_TILE2D=0, row-segment tiles in the planar kernels, keep each output's summation order, so
 *     forwards are bit-identical; MSDA_FWD_SPLIT=0 keeps the tile kernels for few-queries launches, which sum in
 *     another order than the split kernels.)
 *   - padding masks: one byte per element, != 0 = padding; element (n,t,s,c) of a mask over value
 *     (N,T2,S,M*D) lives at mask[((n*T2+t)*S+s)*mask_row_stride + c*mask_col_stride] with
 *     mask_col_stride 1 (the reference's materialised (N,T,S,C) bool tensor, models/model.py:156-157;
 *     needs mask 4-byte aligned and mask_row_stride % 4 == 0) or 0 (one byte per pixel).
 */
#ifndef MSDA_B200_H_
#define MSDA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_ABI_VERSION 4

#if defined(__GNUC__)
#define MSDA_API __attribute__((visibility("default")))
#else
#define MSDA_API
#endif

typedef enum {
    MSDA_OK = 0,
    MSDA_ERR_INVALID_ARGUMENT = 1, /* null pointer, non-positive size, bad stride/alignment   */
    MSDA_ERR_IM2COL_STEP = 2,      /* batch % min(batch, im2col_step) != 0 (cu:50-52)        */
    MSDA_ERR_UNSUPPORTED_DTYPE = 3,
    MSDA_ERR_WORKSPACE = 4,        /* deterministic mode: workspace missing or too small     */
    MSDA_ERR_TOO_LARGE = 5,        /* a 32-bit in-kernel index would overflow                */
    MSDA_ERR_CUDA = 6              /* cudaGetLastError() != cudaSuccess after a launch       */
} msda_status_t;

typedef enum {
    MSDA_DTYPE_F32 = 0,
    MSDA_DTYPE_F64 = 1,
    MSDA_DTYPE_BF16 = 2 /* value / output / grad_output are bf16; sampling_loc, attn_weight (offsets,
                           logits, reference_points) and EVERY gradient buffer -- grad_value too --
                           are fp32; all arithmetic and accumulation is fp32.  D % 16 == 0 only
                           (MSDA_ERR_UNSUPPORTED_DTYPE otherwise); no deterministic mode. */
} msda_dtype_t;

/* flags of msda_backward / msda_snippet_forward / msda_snippet_backward */
#define MSDA_FLAG_DETERMINISTIC 1u   /* two-pass, atomics-free grad_value (needs workspace)   */
#define MSDA_FLAG_ACCUMULATE_VALUE 2u /* add into grad_value instead of zero-filling it first */
#define MSDA_FLAG_PRESUMMED 4u       /* snippet entries: `value` / `grad_value` hold one neighbour-frame
                                        SUM per query-frame slot, (N, msda_snippet_num_slots(), S, M, D),
                                        as written by msda_frame_sum / consumed by msda_frame_unsum    */

#define MSDA_FLAG_PLANAR 8u          /* with MSDA_FLAG_PRESUMMED: the slots are in the library's PLANAR layout
                                        (msda_planar_slot_bytes() bytes per (n, slot), 128-byte aligned), as
                                        written by msda_frame_sum_planar / consumed by msda_frame_unsum_planar.
                                        The slots are a buffer the library defines, so it lays them out for the
                                        gather: every L1 wavefront of the encoder kernels is a full 128-byte line
                                        (6 per sample instead of 8.4, csrc/msda_planar.cu).  MSDA_DTYPE_F32,
                                        channels == 48; not with MSDA_FLAG_DETERMINISTIC                        */

MSDA_API int msda_abi_version(void);
MSDA_API const char *msda_error_string(int status);
/* cudaError_t of the last failed launch seen by this thread (0 if none). */
MSDA_API int msda_last_cuda_error(void);

/*
 * Forward.  output[n,q,m*D+c] = sum_{l,p} attn[n,q,m,l,p] * bilinear(value_l[n,:,m,c], loc[n,q,m,l,p])
 * value_batch_stride: elements between consecutive batch items of `value`
 *                     (0 means S*M*D, i.e. contiguous) -- lets a caller pass value[:, t2]
 *                     without the copy the reference makes (ms_deform_attn.py:179).
 * im2col_step: validated like the reference (MSDA_ERR_IM2COL_STEP); the whole batch is then
 *              processed by one launch -- results do not depend on the chunking.
 */
MSDA_API int msda_forward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                 const void *sampling_loc, const void *attn_weight, void *output,
                 int batch, int spatial_size, int num_heads, int channels, int num_levels,
                 int num_query, int num_point, int64_t value_batch_stride, int im2col_step,
                 int dtype, void *stream);

/*
 * Backward.  Writes grad_sampling_loc (N,Lq,M,L,P,2) and grad_attn_weight (N,Lq,M,L,P) in full;
 * grad_value (N,S,M,D, contiguous) is zero-filled first unless MSDA_FLAG_ACCUMULATE_VALUE.
 * With MSDA_FLAG_DETERMINISTIC the result is bit-reproducible run to run; pass a workspace of
 * at least msda_backward_workspace_bytes(...) bytes (256-byte aligned).
 */
MSDA_API int msda_backward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                  const void *sampling_loc, const void *attn_weight, const void *grad_output,
                  void *grad_value, void *grad_sampling_loc, void *grad_attn_weight,
                  int batch, int spatial_size, int num_heads, int channels, int num_levels,
                  int num_query, int num_point, int64_t value_batch_stride, int im2col_step,
                  int dtype, unsigned flags, void *workspace, size_t workspace_bytes, void *stream);

MSDA_API size_t msda_backward_workspace_bytes(int batch, int spatial_size, int num_heads, int channels,
                                     int num_levels, int num_query, int num_point, int dtype,
                                     unsigned flags);

/*
 * In-place masked zero-fill: data[i] = 0 where mask[i] != 0, i < n_elements (data: MSDA_DTYPE_F32 or
 * MSDA_DTYPE_BF16, contiguous; mask: one byte per element, 16-byte aligned).  Replaces the out-of-place
 * `value.masked_fill(input_padding_mask, 0)` of the reference module (ms_deform_attn.py:116-117) and its
 * mirror on grad_value: only the mask is read and only masked elements are written.
 */
MSDA_API int msda_masked_zero(void *data, const unsigned char *mask, int64_t n_elements, int dtype, void *stream);

/*
 * Fused Snipper snippet attention (one launch per transformer layer).
 *   value            (N,T2,S,M,D)       element strides value_stride_n / value_stride_t
 *                                       [MSDA_FLAG_PRESUMMED: (N,slots,S,M,D), see msda_frame_sum;
 *                                        with MSDA_FLAG_PLANAR the planar slots of msda_frame_sum_planar]
 *   offsets          (N,T1,Lq,M,L,P,2)  raw sampling_offsets Linear output, in pixels
 *   logits           (N,T1,Lq,M,L,P)    raw attention_weights Linear output
 *                                       both dense per (n,t1,q) row; offsets_row_stride / logits_row_stride =
 *                                       floats between consecutive rows (0 = dense), so the two may be column
 *                                       blocks of ONE projection output (one GEMM instead of two)
 *   offsets_bias     (M,L,P,2) or NULL  biases of the two Linear layers, added in-kernel (saves the GEMM
 *   logits_bias      (M,L,P)   or NULL  epilogue pass over the projection output)
 *   reference_points (N,T1,Lq,L,2)      element strides ref_stride_n / ref_stride_t (0 allowed:
 *                                       the encoder expands one frame over T1); may be NULL with:
 *   encoder_valid_ratios (N,L,2) or NULL  encoder self-attention (Lq == S: query q is pixel q of the pyramid): the
 *                                       reference points are computed in-kernel from the query index and these
 *                                       (w,h) valid ratios, bit-identical to get_reference_points
 *                                       (models/deformable_transformer.py:219-232), instead of being materialised
 *                                       once per forward and re-read by every layer
 *   value_mask       NULL, or the padding mask over value (N,T2,S,M*D) (layout: see Conventions): masked
 *                                       elements are gathered as zero and receive no gradient -- the
 *                                       reference's value.masked_fill(mask, 0) (ms_deform_attn.py:116-117)
 *                                       without a pass over the value tensor.  Not with MSDA_FLAG_PRESUMMED
 *                                       (msda_frame_sum / msda_frame_unsum apply the mask there).
 *   output           (N,T1,Lq,M*D)      contiguous
 * Per (n,t1,q,m): A = softmax_{l,p}(logits) / k,  loc = ref + offsets / (W_l,H_l),
 * out = sum over the k neighbour frames t2 of msda(value[:,t2], loc, A); neighbour frames are
 * {t1-1,t1,t1+1} clipped to [0,n_frame) for t1 < n_frame, all T2 frames otherwise
 * (ms_deform_attn.py:137-140,189,201).  Requires the frame slots to share one Linear
 * (ms_deform_attn.py:68-71), which makes logits/offsets identical across t2.
 * MSDA_DTYPE_F32 or MSDA_DTYPE_BF16 (bf16 value / output, fp32 offsets / logits / reference
 * points); L*P <= 32; D % 16 == 0; D <= 128.
 */
MSDA_API int msda_snippet_forward(const void *value, const int64_t *spatial_shapes,
                         const int64_t *level_start_index, const void *offsets, const void *logits,
                         const void *reference_points, void *output,
                         int batch, int n_src_frames, int n_query_frames, int n_frame,
                         int spatial_size, int num_heads, int channels, int num_levels,
                         int num_query, int num_point,
                         int64_t value_stride_n, int64_t value_stride_t,
                         int64_t ref_stride_n, int64_t ref_stride_t,
                         int64_t offsets_row_stride, int64_t logits_row_stride,
                         const void *offsets_bias, const void *logits_bias, const void *encoder_valid_ratios,
                         const unsigned char *value_mask, int64_t mask_row_stride, int mask_col_stride,
                         int dtype, unsigned flags, void *stream);

/*
 * grad_value (N,T2,S,M,D contiguous fp32 [MSDA_FLAG_PRESUMMED: (N,slots,S,M,D); + MSDA_FLAG_PLANAR: planar
 * fp32 slots, batch * slots * msda_planar_slot_bytes() bytes]; zero-filled unless
 * MSDA_FLAG_ACCUMULATE_VALUE), grad_offsets like offsets, grad_logits like logits (same row strides).
 * The gradient w.r.t. reference_points is sum_{m,p} grad_offsets * (W_l,H_l), the gradients of the biases
 * are the sums of grad_offsets / grad_logits over rows; both are left to the caller.
 * MSDA_FLAG_DETERMINISTIC (with MSDA_FLAG_PRESUMMED, MSDA_DTYPE_F32): bit-reproducible run to run -- grad_offsets /
 * grad_logits come from the same kernel with its scatter compiled out (no atomics), grad_value from the two-pass
 * count / fill / ordered-reduce of msda_backward's deterministic mode run over the slots; needs a workspace of
 * msda_snippet_backward_workspace_bytes(...) bytes.  msda_frame_sum / msda_frame_unsum are deterministic by
 * construction, so the whole fused layer is.
 */
MSDA_API int msda_snippet_backward(const void *value, const int64_t *spatial_shapes,
                          const int64_t *level_start_index, const void *offsets, const void *logits,
                          const void *reference_points, const void *grad_output,
                          void *grad_value, void *grad_offsets, void *grad_logits,
                          int batch, int n_src_frames, int n_query_frames, int n_frame,
                          int spatial_size, int num_heads, int channels, int num_levels,
                          int num_query, int num_point,
                          int64_t value_stride_n, int64_t value_stride_t,
                          int64_t ref_stride_n, int64_t ref_stride_t,
                          int64_t offsets_row_stride, int64_t logits_row_stride,
                          const void *offsets_bias, const void *logits_bias, const void *encoder_valid_ratios,
                          const unsigned char *value_mask, int64_t mask_row_stride, int mask_col_stride,
                          int dtype, unsigned flags, void *workspace, size_t workspace_bytes, void *stream);

/* Bytes of (256-byte aligned) workspace msda_snippet_backward needs: 0 unless MSDA_FLAG_DETERMINISTIC. */
MSDA_API size_t msda_snippet_backward_workspace_bytes(int batch, int n_query_frames, int n_frame, int spatial_size,
                                                      int num_heads, int channels, int num_levels, int num_query,
                                                      int num_point, int dtype, unsigned flags);

/*
 * Neighbour-frame pre-summation.  The op is linear in `value` and the reference uses the same sampling
 * locations and weights for every neighbour frame, so the sum over t2 (ms_deform_attn.py:225) can be taken
 * BEFORE the gather:  slots = msda_snippet_num_slots(n_query_frames, n_frame);
 *   slot j <  min(T1, n_frame):  frames max(j-1,0) .. min(j+1, n_frame-1);
 *   slot j == min(T1, n_frame) (only if T1 > n_frame): all T2 frames (future query frames).
 * msda_frame_sum    vsum (N,slots,S,C) [dtype]   = per-slot sums of mask ? 0 : value (N,T2,S,C)
 * msda_frame_unsum  grad_value (N,T2,S,C) [dtype] = mask ? 0 : sum of the fp32 grad_vsum slots covering t2
 * C = M*D (C % 4 == 0; bf16: C % 8 == 0).  Then call the snippet entries with MSDA_FLAG_PRESUMMED.
 * msda_snippet_prefers_presum: 1 when the streaming pass costs less than the neighbour-frame gathers it
 * removes (encoder-sized query sets), 0 for few queries (decoder) or a single frame.
 */
MSDA_API int msda_snippet_num_slots(int n_query_frames, int n_frame);
MSDA_API int msda_snippet_prefers_presum(int n_src_frames, int n_query_frames, int n_frame, int spatial_size,
                                         int num_levels, int num_query, int num_point);
MSDA_API int msda_frame_sum(const void *value, const unsigned char *value_mask, void *vsum,
                            int batch, int n_src_frames, int n_query_frames, int n_frame,
                            int spatial_size, int row_elems,
                            int64_t value_stride_n, int64_t value_stride_t,
                            int64_t mask_row_stride, int mask_col_stride, int dtype, void *stream);
MSDA_API int msda_frame_unsum(const void *grad_vsum, const unsigned char *value_mask, void *grad_value,
                              int batch, int n_src_frames, int n_query_frames, int n_frame,
                              int spatial_size, int row_elems,
                              int64_t mask_row_stride, int mask_col_stride, int dtype, void *stream);

/*
 * Planar slots (MSDA_FLAG_PLANAR).  msda_planar_slot_bytes: bytes of one (n, slot) -- allocate
 * batch * msda_snippet_num_slots() * that, 128-byte aligned -- or 0 when the layout does not apply (then use
 * msda_frame_sum / msda_frame_unsum and MSDA_FLAG_PRESUMMED alone).  The two passes mirror msda_frame_sum /
 * msda_frame_unsum (same slots, same mask semantics, same fixed summation order); value and grad_value keep the
 * reference layout (N,T2,S,M,D), fp32.
 */
MSDA_API size_t msda_planar_slot_bytes(int spatial_size, int num_heads, int channels, int dtype);
MSDA_API int msda_frame_sum_planar(const void *value, const unsigned char *value_mask, void *vsum_planar,
                                   int batch, int n_src_frames, int n_query_frames, int n_frame,
                                   int spatial_size, int num_heads, int channels,
                                   int64_t value_stride_n, int64_t value_stride_t,
                                   int64_t mask_row_stride, int mask_col_stride, int dtype, void *stream);
MSDA_API int msda_frame_unsum_planar(const void *grad_vsum_planar, const unsigned char *value_mask, void *grad_value,
                                     int batch, int n_src_frames, int n_query_frames, int n_frame,
                                     int spatial_size, int num_heads, int channels,
                                     int64_t mask_row_stride, int mask_col_stride, int dtype, void *stream);

/*
 * Layer tail (SURVEY.md section 8f rank 3): what follows every attention / FFN block of the reference's encoder and
 * decoder layers (models/deformable_transformer.py:204-205,194-198,294-295,270-274) and precedes the next attention
 * block (with_pos_embed, :188-190,:202,:292), in ONE pass over the activations instead of five:
 *     out          = LayerNorm(residual + (y + bias)) * gamma + beta        (rows, cols)
 *     out_plus_pos = out + pos                                              (optional, both or neither)
 * y = raw GEMM output of the block's last Linear (bias not added yet; bias may be NULL), every row dense.
 * MSDA_DTYPE_F32; cols % 128 == 0, cols <= 1024; inference only (no gradient formula is provided).
 */
MSDA_API int msda_layer_tail(const void *y, const void *bias, const void *residual, const void *gamma, const void *beta,
                             const void *pos, void *out, void *out_plus_pos, int64_t rows, int cols, float eps,
                             int dtype, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_H_ */
