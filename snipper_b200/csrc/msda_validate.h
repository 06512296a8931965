// Argument validation of the C entry points, shared by libmsda_b200.so (msda_capi.cu) and libmsda_b200_f16.so
// (csrc_f16/msda_f16_capi.cu) so that both libraries reject the same arguments with the same status.  Host code only.
#pragma once

#include <stdint.h>

#include "../../include/msda_b200.h"
#include "msda_internal.h"

namespace {

int check_common(const void *const *ptrs, int nptrs, int batch, int spatial_size, int num_heads,
                 int channels, int num_levels, int num_query, int num_point)
{
    if (batch < 0 || spatial_size < 0 || num_query < 0) return MSDA_ERR_INVALID_ARGUMENT;
    if (num_heads <= 0 || channels <= 0 || num_levels <= 0 || num_point <= 0) return MSDA_ERR_INVALID_ARGUMENT;
    if (num_levels > msda::kMaxLevels) return MSDA_ERR_INVALID_ARGUMENT;
    const bool empty = (batch == 0 || num_query == 0);
    if (!empty)
        for (int i = 0; i < nptrs; ++i)
            if (ptrs[i] == nullptr) return MSDA_ERR_INVALID_ARGUMENT;
    return MSDA_OK;
}

// reference ms_deform_attn_cuda.cu:50-52
int check_im2col_step(int batch, int im2col_step)
{
    if (batch == 0) return MSDA_OK;
    if (im2col_step <= 0) return MSDA_ERR_IM2COL_STEP;
    const int step = batch < im2col_step ? batch : im2col_step;
    return (batch % step == 0) ? MSDA_OK : MSDA_ERR_IM2COL_STEP;
}

// false for NULL: optional pointers pass; required ones are checked for NULL separately
bool misaligned(const void *p, uintptr_t bytes) { return reinterpret_cast<uintptr_t>(p) % bytes != 0; }

// the planar slot layout exists for float32 heads of 48 channels (msda_planar.cu)
bool planar_ok(int spatial_size, int num_heads, int channels, int dtype)
{
    return dtype == MSDA_DTYPE_F32 && msda::planar_slot_bytes(spatial_size, num_heads, channels, 4) != 0;
}

int check_mask(const unsigned char *mask, int64_t row_stride, int col_stride)
{
    if (mask == nullptr) return MSDA_OK;
    if (row_stride < 0 || (col_stride != 0 && col_stride != 1)) return MSDA_ERR_INVALID_ARGUMENT;
    // per-channel masks are read as 32-bit words
    if (col_stride == 1 && (misaligned(mask, 4) || (row_stride & 3))) return MSDA_ERR_INVALID_ARGUMENT;
    return MSDA_OK;
}

int snippet_dims(msda::SnippetDims &d, int batch, int n_src_frames, int n_query_frames,
                        int n_frame, int spatial_size, int num_heads, int channels, int num_levels,
                        int num_query, int num_point, int64_t value_stride_n, int64_t value_stride_t,
                        int64_t ref_stride_n, int64_t ref_stride_t, int64_t offsets_row_stride,
                        int64_t logits_row_stride, const void *offsets_bias, const void *logits_bias,
                        const void *encoder_valid_ratios,
                        const unsigned char *value_mask, int64_t mask_row_stride, int mask_col_stride,
                        int dtype, unsigned flags)
{
    if (dtype != MSDA_DTYPE_F32 && dtype != MSDA_DTYPE_BF16) return MSDA_ERR_UNSUPPORTED_DTYPE;
    if (batch < 0 || num_query < 0 || n_src_frames <= 0 || n_query_frames <= 0 || n_frame <= 0 ||
        n_frame > n_src_frames || spatial_size <= 0 || num_heads <= 0 || channels <= 0 ||
        num_levels <= 0 || num_point <= 0)
        return MSDA_ERR_INVALID_ARGUMENT;
    const bool presummed = (flags & MSDA_FLAG_PRESUMMED) != 0;
    if (presummed && value_mask != nullptr) return MSDA_ERR_INVALID_ARGUMENT;  // the mask belongs to msda_frame_sum / _unsum
    int st = check_mask(value_mask, mask_row_stride, mask_col_stride);
    if (st != MSDA_OK) return st;
    const int frames = presummed ? msda::snippet_num_slots(n_query_frames, n_frame) : n_src_frames;
    if (value_stride_t == 0) value_stride_t = (int64_t)spatial_size * num_heads * channels;
    if (value_stride_n == 0) value_stride_n = value_stride_t * frames;
    if (value_stride_n < 0 || value_stride_t < 0 || ref_stride_n < 0 || ref_stride_t < 0)
        return MSDA_ERR_INVALID_ARGUMENT;
    const int64_t mlp = (int64_t)num_heads * num_levels * num_point;
    if (offsets_row_stride == 0) offsets_row_stride = 2 * mlp;
    if (logits_row_stride == 0) logits_row_stride = mlp;
    // float2 loads of the offsets need even row strides; rows must not overlap
    if (offsets_row_stride < 2 * mlp || logits_row_stride < mlp || (offsets_row_stride & 1)) return MSDA_ERR_INVALID_ARGUMENT;
    d = msda::SnippetDims{batch, n_src_frames, n_query_frames, n_frame, spatial_size, num_heads,
                          channels, num_levels, num_query, num_point, value_stride_n,
                          value_stride_t, ref_stride_n, ref_stride_t, offsets_row_stride, logits_row_stride,
                          static_cast<const float *>(offsets_bias), static_cast<const float *>(logits_bias),
                          static_cast<const float *>(encoder_valid_ratios),
                          presummed ? 1 : 0, value_mask, mask_row_stride, mask_col_stride};
    // analytic reference points: the queries ARE the pixels of the pyramid
    if (encoder_valid_ratios != nullptr && num_query != spatial_size) return MSDA_ERR_INVALID_ARGUMENT;
    if (!msda::snippet_ok(d, dtype == MSDA_DTYPE_BF16 ? 2 : 4)) return MSDA_ERR_INVALID_ARGUMENT;
    return MSDA_OK;
}

// flag combinations of the snippet entries: planar slots and the deterministic mode both ride on the pre-summed
// path, and they exclude each other (the deterministic mode walks cell-major float32 slots)
int snippet_flags_ok(unsigned flags, unsigned allowed, int dtype, int spatial_size, int num_heads, int channels)
{
    const bool presummed = (flags & MSDA_FLAG_PRESUMMED) != 0, deterministic = (flags & MSDA_FLAG_DETERMINISTIC) != 0,
               planar = (flags & MSDA_FLAG_PLANAR) != 0;
    if ((flags & ~allowed) || ((planar || deterministic) && !presummed) || (planar && deterministic))
        return MSDA_ERR_INVALID_ARGUMENT;
    if ((planar && !planar_ok(spatial_size, num_heads, channels, dtype)) || (deterministic && dtype != MSDA_DTYPE_F32))
        return MSDA_ERR_UNSUPPORTED_DTYPE;
    return MSDA_OK;
}

// the pointers a snippet launch dereferences, checked when there is work to do: none NULL, each aligned for its widest
// access.  `out`: the forward's output or the backward's grad_output; `grads`: the backward's three outputs or NULL.
bool snippet_pointers_ok(const msda::SnippetDims &d, const void *value, const int64_t *spatial_shapes,
                                const int64_t *level_start_index, const void *offsets, const void *logits,
                                const void *reference_points, const void *out, bool planar, void *const *grads)
{
    const uintptr_t slot_align = planar ? 128 : 16;
    if (grads && (!grads[0] || !grads[1] || !grads[2] || misaligned(grads[0], slot_align) || misaligned(grads[1], 8) ||
                  misaligned(grads[2], 4)))
        return false;
    return value && spatial_shapes && level_start_index && offsets && logits && (reference_points || d.valid_ratios) &&
           out && !misaligned(value, slot_align) && !misaligned(out, 16) && !misaligned(offsets, 8) &&
           !misaligned(logits, 4) && !misaligned(d.off_bias, 8);
}

int frame_dims(msda::FrameDims &d, int batch, int n_src_frames, int n_query_frames, int n_frame,
                      int spatial_size, int row_elems, int64_t value_stride_n, int64_t value_stride_t,
                      const unsigned char *mask, int64_t mask_row_stride, int mask_col_stride, int dtype, int esize)
{
    if (dtype != MSDA_DTYPE_F32 && dtype != MSDA_DTYPE_BF16) return MSDA_ERR_UNSUPPORTED_DTYPE;
    if (batch < 0 || n_src_frames <= 0 || n_query_frames <= 0 || n_frame <= 0 || n_frame > n_src_frames ||
        spatial_size <= 0 || row_elems <= 0)
        return MSDA_ERR_INVALID_ARGUMENT;
    int st = check_mask(mask, mask_row_stride, mask_col_stride);
    if (st != MSDA_OK) return st;
    if (value_stride_t == 0) value_stride_t = (int64_t)spatial_size * row_elems;
    if (value_stride_n == 0) value_stride_n = value_stride_t * n_src_frames;
    if (value_stride_n < 0 || value_stride_t < 0) return MSDA_ERR_INVALID_ARGUMENT;
    d = msda::FrameDims{batch, n_src_frames, n_query_frames, n_frame, spatial_size, row_elems, value_stride_n,
                        value_stride_t, mask ? mask_row_stride : 0, mask ? mask_col_stride : 0};
    return msda::frame_dims_ok(d, esize) ? MSDA_OK : MSDA_ERR_INVALID_ARGUMENT;
}

}  // namespace
