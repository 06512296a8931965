// extern "C" entry points of libmsda_b200_f16.so (include/msda_b200_f16.h).  Each one runs the validation of its
// msda_* twin in csrc/msda_capi.cu (the helpers of csrc/msda_validate.h, called with MSDA_DTYPE_BF16) in the same order,
// so that it returns the twin's status for any arguments; only the launch differs.
#include "../../include/msda_b200_f16.h"
#include "../csrc/msda_validate.h"
#include "msda_f16_internal.h"

namespace {

thread_local int g_last_cuda_error = 0;

int cuda_status(cudaError_t e)
{
    if (e == cudaSuccess) return MSDA_OK;
    g_last_cuda_error = (int)e;
    return MSDA_ERR_CUDA;
}

constexpr int kAs = MSDA_DTYPE_BF16;   // the dtype whose validation rules the fp16 entries share

}  // namespace

extern "C" {

int msda_f16_abi_version(void) { return MSDA_F16_ABI_VERSION; }

int msda_f16_last_cuda_error(void) { return g_last_cuda_error; }

int msda_f16_forward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                     const void *sampling_loc, const void *attn_weight, void *output,
                     int batch, int spatial_size, int num_heads, int channels, int num_levels,
                     int num_query, int num_point, int64_t value_batch_stride, int im2col_step, void *stream)
{
    const void *ptrs[] = {value, spatial_shapes, level_start_index, sampling_loc, attn_weight, output};
    int st = check_common(ptrs, 6, batch, spatial_size, num_heads, channels, num_levels, num_query, num_point);
    if (st != MSDA_OK) return st;
    st = check_im2col_step(batch, im2col_step);
    if (st != MSDA_OK) return st;
    if (batch == 0 || num_query == 0) return MSDA_OK;
    if (value_batch_stride == 0) value_batch_stride = (int64_t)spatial_size * num_heads * channels;
    if (value_batch_stride < 0) return MSDA_ERR_INVALID_ARGUMENT;
    msda::OpDims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point, value_batch_stride};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (spatial_size == 0)  // nothing to sample: every corner is invalid
        return cuda_status(cudaMemsetAsync(output, 0, (size_t)2 * batch * num_query * num_heads * channels, s));
    // vectorised path only: D % 16 == 0 (16-byte lanes of 8 channels, an even number of lanes)
    if (!(msda::fast_path_ok(d, 2) && !misaligned(value, 16) && !misaligned(output, 16))) return MSDA_ERR_UNSUPPORTED_DTYPE;
    return cuda_status(msda::launch_forward_fast_f16(value, spatial_shapes, level_start_index, (const float *)sampling_loc,
                                                     (const float *)attn_weight, output, d, s));
}

int msda_f16_backward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                      const void *sampling_loc, const void *attn_weight, const void *grad_output,
                      void *grad_value, void *grad_sampling_loc, void *grad_attn_weight,
                      int batch, int spatial_size, int num_heads, int channels, int num_levels,
                      int num_query, int num_point, int64_t value_batch_stride, int im2col_step,
                      unsigned flags, void *stream)
{
    const void *ptrs[] = {value, spatial_shapes, level_start_index, sampling_loc, attn_weight,
                          grad_output, grad_value, grad_sampling_loc, grad_attn_weight};
    int st = check_common(ptrs, 9, batch, spatial_size, num_heads, channels, num_levels, num_query, num_point);
    if (st != MSDA_OK) return st;
    st = check_im2col_step(batch, im2col_step);
    if (st != MSDA_OK) return st;
    // the bounds msda_backward checks before refusing the deterministic mode for 16-bit storage
    if ((flags & MSDA_FLAG_DETERMINISTIC) &&
        ((int64_t)batch * num_query * num_heads * num_levels * num_point * 4 >= (int64_t)INT32_MAX ||
         (int64_t)batch * spatial_size * num_heads >= (int64_t)INT32_MAX))
        return MSDA_ERR_TOO_LARGE;
    if (value_batch_stride == 0) value_batch_stride = (int64_t)spatial_size * num_heads * channels;
    if (value_batch_stride < 0) return MSDA_ERR_INVALID_ARGUMENT;
    msda::OpDims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point, value_batch_stride};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t value_elems = (size_t)batch * spatial_size * num_heads * channels;   // every gradient buffer is fp32
    if (!(flags & MSDA_FLAG_ACCUMULATE_VALUE) && value_elems > 0 && grad_value != nullptr) {
        st = cuda_status(cudaMemsetAsync(grad_value, 0, sizeof(float) * value_elems, s));
        if (st != MSDA_OK) return st;
    }
    if (batch == 0 || num_query == 0) return MSDA_OK;
    if (spatial_size == 0) {
        const size_t n = (size_t)batch * num_query * num_heads * num_levels * num_point;
        st = cuda_status(cudaMemsetAsync(grad_sampling_loc, 0, sizeof(float) * 2 * n, s));
        if (st != MSDA_OK) return st;
        return cuda_status(cudaMemsetAsync(grad_attn_weight, 0, sizeof(float) * n, s));
    }
    if (flags & MSDA_FLAG_DETERMINISTIC) return MSDA_ERR_UNSUPPORTED_DTYPE;
    if (!(msda::fast_path_ok(d, 2) && !misaligned(value, 16) && !misaligned(grad_output, 16) && !misaligned(grad_value, 16)))
        return MSDA_ERR_UNSUPPORTED_DTYPE;
    return cuda_status(msda::launch_backward_fast_f16(value, spatial_shapes, level_start_index, (const float *)sampling_loc,
                                                      (const float *)attn_weight, grad_output, (float *)grad_value,
                                                      (float *)grad_sampling_loc, (float *)grad_attn_weight, d, s));
}

int msda_f16_snippet_forward(const void *value, const int64_t *spatial_shapes,
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
                             unsigned flags, void *stream)
{
    // MSDA_FLAG_PLANAR is refused here (the planar slots are float32 only)
    int st = snippet_flags_ok(flags, MSDA_FLAG_PRESUMMED | MSDA_FLAG_PLANAR, kAs, spatial_size, num_heads, channels);
    if (st != MSDA_OK) return st;
    msda::SnippetDims d;
    st = snippet_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, num_heads,
                      channels, num_levels, num_query, num_point, value_stride_n,
                      value_stride_t, ref_stride_n, ref_stride_t, offsets_row_stride, logits_row_stride,
                      offsets_bias, logits_bias, encoder_valid_ratios, value_mask, mask_row_stride, mask_col_stride,
                      kAs, flags);
    if (st != MSDA_OK) return st;
    if (batch == 0 || num_query == 0) return MSDA_OK;
    if (!snippet_pointers_ok(d, value, spatial_shapes, level_start_index, offsets, logits, reference_points, output, false,
                             nullptr))
        return MSDA_ERR_INVALID_ARGUMENT;
    return cuda_status(msda::launch_snippet_forward_f16(value, spatial_shapes, level_start_index, (const float *)offsets,
                                                        (const float *)logits, (const float *)reference_points, output,
                                                        d, static_cast<cudaStream_t>(stream)));
}

int msda_f16_snippet_backward(const void *value, const int64_t *spatial_shapes,
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
                              unsigned flags, void *stream)
{
    // MSDA_FLAG_DETERMINISTIC and MSDA_FLAG_PLANAR are refused here (both are float32 only)
    int st = snippet_flags_ok(flags, MSDA_FLAG_PRESUMMED | MSDA_FLAG_ACCUMULATE_VALUE | MSDA_FLAG_DETERMINISTIC |
                              MSDA_FLAG_PLANAR, kAs, spatial_size, num_heads, channels);
    if (st != MSDA_OK) return st;
    msda::SnippetDims d;
    st = snippet_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, num_heads,
                      channels, num_levels, num_query, num_point, value_stride_n,
                      value_stride_t, ref_stride_n, ref_stride_t, offsets_row_stride, logits_row_stride,
                      offsets_bias, logits_bias, encoder_valid_ratios, value_mask, mask_row_stride, mask_col_stride,
                      kAs, flags);
    if (st != MSDA_OK) return st;
    const bool accumulate = (flags & MSDA_FLAG_ACCUMULATE_VALUE) != 0, work = batch > 0 && num_query > 0;
    const int gframes = (flags & MSDA_FLAG_PRESUMMED) ? msda::snippet_num_slots(n_query_frames, n_frame) : n_src_frames;
    if (batch == 0) return MSDA_OK;
    if (!accumulate && !grad_value) return MSDA_ERR_INVALID_ARGUMENT;
    void *const grads[] = {grad_value, grad_offsets, grad_logits};
    if (work && !snippet_pointers_ok(d, value, spatial_shapes, level_start_index, offsets, logits, reference_points,
                                     grad_output, false, grads))
        return MSDA_ERR_INVALID_ARGUMENT;
    // everything is validated: from here on work is enqueued
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!accumulate) {
        st = cuda_status(cudaMemsetAsync(grad_value, 0, sizeof(float) * batch * gframes * ((size_t)spatial_size * num_heads * channels), s));
        if (st != MSDA_OK) return st;
    }
    if (!work) return MSDA_OK;
    return cuda_status(msda::launch_snippet_backward_f16(value, spatial_shapes, level_start_index, (const float *)offsets,
                                                         (const float *)logits, (const float *)reference_points,
                                                         grad_output, (float *)grad_value, (float *)grad_offsets,
                                                         (float *)grad_logits, d, s));
}

int msda_f16_frame_sum(const void *value, const unsigned char *value_mask, void *vsum,
                       int batch, int n_src_frames, int n_query_frames, int n_frame,
                       int spatial_size, int row_elems, int64_t value_stride_n, int64_t value_stride_t,
                       int64_t mask_row_stride, int mask_col_stride, void *stream)
{
    msda::FrameDims d;
    int st = frame_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, row_elems, value_stride_n,
                        value_stride_t, value_mask, mask_row_stride, mask_col_stride, kAs, 2);
    if (st != MSDA_OK) return st;
    if (batch == 0) return MSDA_OK;
    if (!value || !vsum || misaligned(value, 16) || misaligned(vsum, 16)) return MSDA_ERR_INVALID_ARGUMENT;
    return cuda_status(msda::launch_frame_sum_f16(value, value_mask, vsum, d, static_cast<cudaStream_t>(stream)));
}

int msda_f16_frame_unsum(const void *grad_vsum, const unsigned char *value_mask, void *grad_value,
                         int batch, int n_src_frames, int n_query_frames, int n_frame,
                         int spatial_size, int row_elems, int64_t mask_row_stride, int mask_col_stride, void *stream)
{
    msda::FrameDims d;
    int st = frame_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, row_elems, 0, 0,
                        value_mask, mask_row_stride, mask_col_stride, kAs, 4);   // one thread per 4 fp32 channels
    if (st != MSDA_OK) return st;
    if (batch == 0) return MSDA_OK;
    // each thread stores 4 fp16 channels: 8 bytes
    if (!grad_vsum || !grad_value || misaligned(grad_vsum, 16) || misaligned(grad_value, 8))
        return MSDA_ERR_INVALID_ARGUMENT;
    return cuda_status(msda::launch_frame_unsum_f16(static_cast<const float *>(grad_vsum), value_mask, grad_value, d,
                                                    static_cast<cudaStream_t>(stream)));
}

}  // extern "C"
