/*
 * libmsda_b200_f16.so -- the attention op of libmsda_b200.so with float16 storage, for torch.autocast's default
 * dtype.  It returns the status codes of msda_b200.h and has an ABI version of its own.
 *
 * Semantics are those of MSDA_DTYPE_BF16 with fp16 storage:
 *   - fp16: value, output, grad_output and the pre-summed slots of msda_f16_frame_sum;
 *   - fp32: sampling locations, attention weights, offsets, logits, reference points and the gradients
 *     grad_sampling_loc / grad_attn_weight / grad_offsets / grad_logits;
 *   - all arithmetic and accumulation is fp32.  grad_value is accumulated in fp32: msda_f16_backward and
 *     msda_f16_snippet_backward write an fp32 grad_value buffer (rounding it is left to the caller), and
 *     msda_f16_frame_unsum rounds the fp32 slot gradients once, to nearest even, into fp16.  Values beyond the fp16
 *     range round to +-inf, exactly as a float -> half cast of the fp32 result does (loss scalers rely on it to skip
 *     overflowing steps).
 *   - shapes: D % 16 == 0, D <= 128; L * P <= 32 on the fused entries.
 *   - no deterministic mode and no planar slots: MSDA_FLAG_DETERMINISTIC / MSDA_FLAG_PLANAR get the status
 *     libmsda_b200.so returns for them with MSDA_DTYPE_BF16.
 * Each entry point takes the arguments of its msda_* twin in msda_b200.h without `dtype` (and, for the backward
 * entries, without the deterministic workspace), and returns, for any arguments, what its twin returns for the same
 * arguments with MSDA_DTYPE_BF16.
 *
 * Known range limit: a pre-summed slot holds the SUM of up to 3 neighbour frames (all T2 frames for the slot of the
 * future query frames) and is stored in fp16, so it overflows where the per-(t1,t2) composition would not when value
 * elements exceed about 65504 / 3 (65504 / T2 for the future-frame slot).  The bf16 slots have the same structure.
 */
#ifndef MSDA_B200_F16_H_
#define MSDA_B200_F16_H_

#include "msda_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_F16_ABI_VERSION 1

MSDA_API int msda_f16_abi_version(void);
/* cudaError_t of the last failed launch of this library seen by this thread (0 if none). */
MSDA_API int msda_f16_last_cuda_error(void);

MSDA_API int msda_f16_forward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                              const void *sampling_loc, const void *attn_weight, void *output,
                              int batch, int spatial_size, int num_heads, int channels, int num_levels,
                              int num_query, int num_point, int64_t value_batch_stride, int im2col_step, void *stream);

/* grad_value: fp32 (N,S,M,D), zero-filled first unless MSDA_FLAG_ACCUMULATE_VALUE. */
MSDA_API int msda_f16_backward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                               const void *sampling_loc, const void *attn_weight, const void *grad_output,
                               void *grad_value, void *grad_sampling_loc, void *grad_attn_weight,
                               int batch, int spatial_size, int num_heads, int channels, int num_levels,
                               int num_query, int num_point, int64_t value_batch_stride, int im2col_step,
                               unsigned flags, void *stream);

MSDA_API int msda_f16_snippet_forward(const void *value, const int64_t *spatial_shapes,
                                      const int64_t *level_start_index, const void *offsets, const void *logits,
                                      const void *reference_points, void *output,
                                      int batch, int n_src_frames, int n_query_frames, int n_frame,
                                      int spatial_size, int num_heads, int channels, int num_levels,
                                      int num_query, int num_point,
                                      int64_t value_stride_n, int64_t value_stride_t,
                                      int64_t ref_stride_n, int64_t ref_stride_t,
                                      int64_t offsets_row_stride, int64_t logits_row_stride,
                                      const void *offsets_bias, const void *logits_bias,
                                      const void *encoder_valid_ratios,
                                      const unsigned char *value_mask, int64_t mask_row_stride, int mask_col_stride,
                                      unsigned flags, void *stream);

/* grad_value: fp32, (N,T2,S,M,D) or, with MSDA_FLAG_PRESUMMED, (N,slots,S,M,D). */
MSDA_API int msda_f16_snippet_backward(const void *value, const int64_t *spatial_shapes,
                                       const int64_t *level_start_index, const void *offsets, const void *logits,
                                       const void *reference_points, const void *grad_output,
                                       void *grad_value, void *grad_offsets, void *grad_logits,
                                       int batch, int n_src_frames, int n_query_frames, int n_frame,
                                       int spatial_size, int num_heads, int channels, int num_levels,
                                       int num_query, int num_point,
                                       int64_t value_stride_n, int64_t value_stride_t,
                                       int64_t ref_stride_n, int64_t ref_stride_t,
                                       int64_t offsets_row_stride, int64_t logits_row_stride,
                                       const void *offsets_bias, const void *logits_bias,
                                       const void *encoder_valid_ratios,
                                       const unsigned char *value_mask, int64_t mask_row_stride, int mask_col_stride,
                                       unsigned flags, void *stream);

/* vsum: fp16 (N,slots,S,C) from fp16 value (N,T2,S,C).  grad_value: fp16 (N,T2,S,C) from fp32 grad_vsum. */
MSDA_API int msda_f16_frame_sum(const void *value, const unsigned char *value_mask, void *vsum,
                                int batch, int n_src_frames, int n_query_frames, int n_frame,
                                int spatial_size, int row_elems,
                                int64_t value_stride_n, int64_t value_stride_t,
                                int64_t mask_row_stride, int mask_col_stride, void *stream);
MSDA_API int msda_f16_frame_unsum(const void *grad_vsum, const unsigned char *value_mask, void *grad_value,
                                  int batch, int n_src_frames, int n_query_frames, int n_frame,
                                  int spatial_size, int row_elems,
                                  int64_t mask_row_stride, int mask_col_stride, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_F16_H_ */
