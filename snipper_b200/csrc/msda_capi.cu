// extern "C" entry points of libmsda_b200.so (see include/msda_b200.h for the contract and
// the reference interfaces each one replaces).  Argument validation mirrors the reference host
// code (models/ops/src/cuda/ms_deform_attn_cuda.cu:28-52) but reports through return codes.
#include "../../include/msda_b200.h"
#include "msda_internal.h"

#include <stdint.h>
#include <string.h>

namespace {

thread_local int g_last_cuda_error = 0;

int cuda_status(cudaError_t e)
{
    if (e == cudaSuccess) return MSDA_OK;
    g_last_cuda_error = (int)e;
    return MSDA_ERR_CUDA;
}

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

}  // namespace

extern "C" {

int msda_abi_version(void) { return MSDA_ABI_VERSION; }

int msda_last_cuda_error(void) { return g_last_cuda_error; }

const char *msda_error_string(int status)
{
    switch (status) {
        case MSDA_OK: return "ok";
        case MSDA_ERR_INVALID_ARGUMENT: return "invalid argument (null pointer, bad size, stride or alignment)";
        case MSDA_ERR_IM2COL_STEP: return "batch must divide im2col_step";
        case MSDA_ERR_UNSUPPORTED_DTYPE: return "unsupported dtype for this entry point";
        case MSDA_ERR_WORKSPACE: return "deterministic mode needs a workspace of msda_backward_workspace_bytes()";
        case MSDA_ERR_TOO_LARGE: return "problem too large for 32-bit in-kernel indices";
        case MSDA_ERR_CUDA: return "CUDA launch failed (see msda_last_cuda_error)";
        default: return "unknown msda status";
    }
}

int msda_forward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                 const void *sampling_loc, const void *attn_weight, void *output,
                 int batch, int spatial_size, int num_heads, int channels, int num_levels,
                 int num_query, int num_point, int64_t value_batch_stride, int im2col_step,
                 int dtype, void *stream)
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
    if (spatial_size == 0) {  // nothing to sample: every corner is invalid
        const size_t esz = dtype == MSDA_DTYPE_F64 ? 8 : (dtype == MSDA_DTYPE_BF16 ? 2 : 4);
        if (dtype != MSDA_DTYPE_F32 && dtype != MSDA_DTYPE_F64 && dtype != MSDA_DTYPE_BF16) return MSDA_ERR_UNSUPPORTED_DTYPE;
        return cuda_status(cudaMemsetAsync(output, 0, esz * batch * num_query * num_heads * channels, s));
    }
    switch (dtype) {
        case MSDA_DTYPE_F32:
            if (msda::fast_path_ok(d) && !misaligned(value, 16) && !misaligned(output, 16))
                return cuda_status(msda::launch_forward_fast_f32(
                    (const float *)value, spatial_shapes, level_start_index, (const float *)sampling_loc,
                    (const float *)attn_weight, (float *)output, d, s));
            return cuda_status(msda::launch_forward_generic<float>(
                (const float *)value, spatial_shapes, level_start_index, (const float *)sampling_loc,
                (const float *)attn_weight, (float *)output, d, s));
        case MSDA_DTYPE_F64:
            return cuda_status(msda::launch_forward_generic<double>(
                (const double *)value, spatial_shapes, level_start_index, (const double *)sampling_loc,
                (const double *)attn_weight, (double *)output, d, s));
        case MSDA_DTYPE_BF16:
            // vectorised path only: D % 16 == 0 (16-byte lanes of 8 channels, an even number of lanes)
            if (!(msda::fast_path_ok(d, 2) && !misaligned(value, 16) && !misaligned(output, 16))) return MSDA_ERR_UNSUPPORTED_DTYPE;
            return cuda_status(msda::launch_forward_fast_bf16(
                value, spatial_shapes, level_start_index, (const float *)sampling_loc,
                (const float *)attn_weight, output, d, s));
        default:
            return MSDA_ERR_UNSUPPORTED_DTYPE;
    }
}

size_t msda_backward_workspace_bytes(int batch, int spatial_size, int num_heads, int channels,
                                     int num_levels, int num_query, int num_point, int dtype,
                                     unsigned flags)
{
    if (!(flags & MSDA_FLAG_DETERMINISTIC) || dtype != MSDA_DTYPE_F32) return 0;
    msda::OpDims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point, 0};
    return msda::deterministic_workspace_bytes(d);
}

int msda_backward(const void *value, const int64_t *spatial_shapes, const int64_t *level_start_index,
                  const void *sampling_loc, const void *attn_weight, const void *grad_output,
                  void *grad_value, void *grad_sampling_loc, void *grad_attn_weight,
                  int batch, int spatial_size, int num_heads, int channels, int num_levels,
                  int num_query, int num_point, int64_t value_batch_stride, int im2col_step,
                  int dtype, unsigned flags, void *workspace, size_t workspace_bytes, void *stream)
{
    const void *ptrs[] = {value, spatial_shapes, level_start_index, sampling_loc, attn_weight,
                          grad_output, grad_value, grad_sampling_loc, grad_attn_weight};
    int st = check_common(ptrs, 9, batch, spatial_size, num_heads, channels, num_levels, num_query, num_point);
    if (st != MSDA_OK) return st;
    st = check_im2col_step(batch, im2col_step);
    if (st != MSDA_OK) return st;
    if (dtype != MSDA_DTYPE_F32 && dtype != MSDA_DTYPE_F64 && dtype != MSDA_DTYPE_BF16) return MSDA_ERR_UNSUPPORTED_DTYPE;
    // corner ids / cell ids of the deterministic two-pass mode are 32-bit (checked before anything is enqueued)
    if ((flags & MSDA_FLAG_DETERMINISTIC) &&
        ((int64_t)batch * num_query * num_heads * num_levels * num_point * 4 >= (int64_t)INT32_MAX ||
         (int64_t)batch * spatial_size * num_heads >= (int64_t)INT32_MAX))
        return MSDA_ERR_TOO_LARGE;
    if (value_batch_stride == 0) value_batch_stride = (int64_t)spatial_size * num_heads * channels;
    if (value_batch_stride < 0) return MSDA_ERR_INVALID_ARGUMENT;
    msda::OpDims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point, value_batch_stride};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t esz = dtype == MSDA_DTYPE_F64 ? 8 : 4;  // bf16 mode: every gradient buffer is fp32
    const size_t value_elems = (size_t)batch * spatial_size * num_heads * channels;
    if (!(flags & MSDA_FLAG_ACCUMULATE_VALUE) && value_elems > 0 && grad_value != nullptr) {
        st = cuda_status(cudaMemsetAsync(grad_value, 0, esz * value_elems, s));
        if (st != MSDA_OK) return st;
    }
    if (batch == 0 || num_query == 0) return MSDA_OK;
    if (spatial_size == 0) {
        const size_t n = (size_t)batch * num_query * num_heads * num_levels * num_point;
        st = cuda_status(cudaMemsetAsync(grad_sampling_loc, 0, esz * 2 * n, s));
        if (st != MSDA_OK) return st;
        return cuda_status(cudaMemsetAsync(grad_attn_weight, 0, esz * n, s));
    }
    if (dtype == MSDA_DTYPE_F64) {
        if (flags & MSDA_FLAG_DETERMINISTIC) return MSDA_ERR_UNSUPPORTED_DTYPE;
        return cuda_status(msda::launch_backward_generic<double>(
            (const double *)value, spatial_shapes, level_start_index, (const double *)sampling_loc,
            (const double *)attn_weight, (const double *)grad_output, (double *)grad_value,
            (double *)grad_sampling_loc, (double *)grad_attn_weight, d, s));
    }
    if (dtype == MSDA_DTYPE_BF16) {
        if (flags & MSDA_FLAG_DETERMINISTIC) return MSDA_ERR_UNSUPPORTED_DTYPE;
        if (!(msda::fast_path_ok(d, 2) && !misaligned(value, 16) && !misaligned(grad_output, 16) && !misaligned(grad_value, 16)))
            return MSDA_ERR_UNSUPPORTED_DTYPE;
        return cuda_status(msda::launch_backward_fast_bf16(
            value, spatial_shapes, level_start_index, (const float *)sampling_loc,
            (const float *)attn_weight, grad_output, (float *)grad_value,
            (float *)grad_sampling_loc, (float *)grad_attn_weight, d, s));
    }
    if (flags & MSDA_FLAG_DETERMINISTIC) {
        const size_t need = msda::deterministic_workspace_bytes(d);
        if (workspace == nullptr || workspace_bytes < need || misaligned(workspace, 256))
            return MSDA_ERR_WORKSPACE;
        return cuda_status(msda::launch_backward_deterministic_f32(
            (const float *)value, spatial_shapes, level_start_index, (const float *)sampling_loc,
            (const float *)attn_weight, (const float *)grad_output, (float *)grad_value,
            (float *)grad_sampling_loc, (float *)grad_attn_weight, d, workspace, s,
            (flags & MSDA_FLAG_ACCUMULATE_VALUE) != 0));
    }
    if (msda::fast_path_ok(d) && !misaligned(value, 16) && !misaligned(grad_output, 16) && !misaligned(grad_value, 16))
        return cuda_status(msda::launch_backward_fast_f32(
            (const float *)value, spatial_shapes, level_start_index, (const float *)sampling_loc,
            (const float *)attn_weight, (const float *)grad_output, (float *)grad_value,
            (float *)grad_sampling_loc, (float *)grad_attn_weight, d, s));
    return cuda_status(msda::launch_backward_generic<float>(
        (const float *)value, spatial_shapes, level_start_index, (const float *)sampling_loc,
        (const float *)attn_weight, (const float *)grad_output, (float *)grad_value,
        (float *)grad_sampling_loc, (float *)grad_attn_weight, d, s));
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// the fused layer's backward as a per-call problem over N*T1 batch items whose grad_value frames are the slots
static msda::OpDims snippet_det_dims(int batch, int n_query_frames, int n_frame, int spatial_size, int num_heads,
                                     int channels, int num_levels, int num_query, int num_point)
{
    msda::OpDims od{batch * n_query_frames, spatial_size, num_heads, channels, num_levels, num_query, num_point, 0};
    od.frame_q = n_query_frames;
    od.frame_local = n_query_frames < n_frame ? n_query_frames : n_frame;
    od.frame_slots = msda::snippet_num_slots(n_query_frames, n_frame);
    return od;
}

// the deterministic workspace starts with the sampling locations (2 floats per sample) and attention weights (1),
// each block 256-byte aligned; the two-pass state of msda_backward follows
static size_t det_sample_bytes(const msda::OpDims &od, int floats)
{
    return align256(sizeof(float) * floats * (size_t)od.N * od.Lq * od.M * od.L * od.P);
}

static int check_mask(const unsigned char *mask, int64_t row_stride, int col_stride)
{
    if (mask == nullptr) return MSDA_OK;
    if (row_stride < 0 || (col_stride != 0 && col_stride != 1)) return MSDA_ERR_INVALID_ARGUMENT;
    // per-channel masks are read as 32-bit words
    if (col_stride == 1 && (misaligned(mask, 4) || (row_stride & 3))) return MSDA_ERR_INVALID_ARGUMENT;
    return MSDA_OK;
}

static int snippet_dims(msda::SnippetDims &d, int batch, int n_src_frames, int n_query_frames,
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
static int snippet_flags_ok(unsigned flags, unsigned allowed, int dtype, int spatial_size, int num_heads, int channels)
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
static bool snippet_pointers_ok(const msda::SnippetDims &d, const void *value, const int64_t *spatial_shapes,
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

int msda_masked_zero(void *data, const unsigned char *mask, int64_t n_elements, int dtype, void *stream)
{
    if (n_elements < 0) return MSDA_ERR_INVALID_ARGUMENT;
    if (n_elements == 0) return MSDA_OK;
    if (!data || !mask) return MSDA_ERR_INVALID_ARGUMENT;
    if (dtype != MSDA_DTYPE_F32 && dtype != MSDA_DTYPE_BF16) return MSDA_ERR_UNSUPPORTED_DTYPE;
    if (misaligned(mask, 16)) return MSDA_ERR_INVALID_ARGUMENT;
    return cuda_status(msda::launch_masked_zero(data, mask, n_elements, dtype == MSDA_DTYPE_BF16 ? 2 : 4,
                                                static_cast<cudaStream_t>(stream)));
}

int msda_snippet_forward(const void *value, const int64_t *spatial_shapes,
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
                         int dtype, unsigned flags, void *stream)
{
    int st = snippet_flags_ok(flags, MSDA_FLAG_PRESUMMED | MSDA_FLAG_PLANAR, dtype, spatial_size, num_heads, channels);
    if (st != MSDA_OK) return st;
    const bool planar = (flags & MSDA_FLAG_PLANAR) != 0;
    msda::SnippetDims d;
    st = snippet_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, num_heads,
                      channels, num_levels, num_query, num_point, value_stride_n,
                      value_stride_t, ref_stride_n, ref_stride_t, offsets_row_stride, logits_row_stride,
                      offsets_bias, logits_bias, encoder_valid_ratios, value_mask, mask_row_stride, mask_col_stride,
                      dtype, flags);
    if (st != MSDA_OK) return st;
    if (batch == 0 || num_query == 0) return MSDA_OK;
    if (!snippet_pointers_ok(d, value, spatial_shapes, level_start_index, offsets, logits, reference_points, output, planar,
                             nullptr))
        return MSDA_ERR_INVALID_ARGUMENT;
    const float *off = (const float *)offsets, *lg = (const float *)logits, *ref = (const float *)reference_points;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (planar)
        return cuda_status(msda::launch_planar_forward_f32(value, spatial_shapes, level_start_index, off, lg, ref,
                                                           (float *)output, d, s));
    if (dtype == MSDA_DTYPE_BF16)
        return cuda_status(msda::launch_snippet_forward_bf16(value, spatial_shapes, level_start_index, off, lg, ref,
                                                             output, d, s));
    return cuda_status(msda::launch_snippet_forward_f32((const float *)value, spatial_shapes, level_start_index, off,
                                                        lg, ref, (float *)output, d, s));
}

// bit-reproducible backward (MSDA_FLAG_DETERMINISTIC, pre-summed float32 slots, validated): the fused kernel with
// its scatter compiled out for grad_offsets / grad_logits, then msda_backward's two-pass grad_value over the slots
static int snippet_backward_deterministic(const msda::SnippetDims &d, const float *value, const int64_t *spatial_shapes,
                                          const int64_t *level_start_index, const float *offsets, const float *logits,
                                          const float *reference_points, const float *grad_output, float *grad_value,
                                          float *grad_offsets, float *grad_logits, bool accumulate, void *workspace,
                                          cudaStream_t s)
{
    const msda::OpDims od = snippet_det_dims(d.N, d.T1, d.n_frame, d.S, d.M, d.D, d.L, d.Lq, d.P);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    float *loc = reinterpret_cast<float *>(ws), *attn = reinterpret_cast<float *>(ws + det_sample_bytes(od, 2));
    int st = cuda_status(msda::launch_snippet_backward_noscatter_f32(
        value, spatial_shapes, level_start_index, offsets, logits, reference_points, grad_output, grad_offsets,
        grad_logits, d, s));
    if (st != MSDA_OK) return st;
    st = cuda_status(msda::launch_snippet_loc_attn(spatial_shapes, level_start_index, offsets, logits, reference_points,
                                                   loc, attn, d, s));
    if (st != MSDA_OK) return st;
    // grad_value: count / scan / fill / ordered reduce; every slot cell is written exactly once
    return cuda_status(msda::launch_deterministic_grad_value_f32(spatial_shapes, level_start_index, loc, attn, grad_output,
        grad_value, od, ws + det_sample_bytes(od, 2) + det_sample_bytes(od, 1), s, accumulate));
}

int msda_snippet_backward(const void *value, const int64_t *spatial_shapes,
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
                          int dtype, unsigned flags, void *workspace, size_t workspace_bytes, void *stream)
{
    int st = snippet_flags_ok(flags, MSDA_FLAG_PRESUMMED | MSDA_FLAG_ACCUMULATE_VALUE | MSDA_FLAG_DETERMINISTIC |
                              MSDA_FLAG_PLANAR, dtype, spatial_size, num_heads, channels);
    if (st != MSDA_OK) return st;
    msda::SnippetDims d;
    st = snippet_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, num_heads,
                      channels, num_levels, num_query, num_point, value_stride_n,
                      value_stride_t, ref_stride_n, ref_stride_t, offsets_row_stride, logits_row_stride,
                      offsets_bias, logits_bias, encoder_valid_ratios, value_mask, mask_row_stride, mask_col_stride,
                      dtype, flags);
    if (st != MSDA_OK) return st;
    const bool planar = (flags & MSDA_FLAG_PLANAR) != 0, accumulate = (flags & MSDA_FLAG_ACCUMULATE_VALUE) != 0,
               deterministic = (flags & MSDA_FLAG_DETERMINISTIC) != 0, work = batch > 0 && num_query > 0;
    const int gframes = (flags & MSDA_FLAG_PRESUMMED) ? msda::snippet_num_slots(n_query_frames, n_frame) : n_src_frames;
    if (deterministic) {
        // 32-bit corner / cell ids
        if ((int64_t)batch * n_query_frames * num_query * num_heads * num_levels * num_point * 4 >= (int64_t)INT32_MAX ||
            (int64_t)batch * gframes * spatial_size * num_heads >= (int64_t)INT32_MAX)
            return MSDA_ERR_TOO_LARGE;
        const size_t need = msda_snippet_backward_workspace_bytes(batch, n_query_frames, n_frame, spatial_size, num_heads,
                                                                  channels, num_levels, num_query, num_point, dtype, flags);
        if (work && (workspace == nullptr || workspace_bytes < need || misaligned(workspace, 256)))
            return MSDA_ERR_WORKSPACE;
    }
    if (batch == 0) return MSDA_OK;
    // grad_value is zero-filled unless accumulated into or written in full by the deterministic ordered reduce
    const bool zero_fill = !accumulate && !(deterministic && work);
    if (((zero_fill || deterministic) && !grad_value) || (deterministic && misaligned(grad_value, 16)))
        return MSDA_ERR_INVALID_ARGUMENT;
    void *const grads[] = {grad_value, grad_offsets, grad_logits};
    if (work && !snippet_pointers_ok(d, value, spatial_shapes, level_start_index, offsets, logits, reference_points,
                                     grad_output, planar, grads))
        return MSDA_ERR_INVALID_ARGUMENT;
    // everything is validated: from here on work is enqueued
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (zero_fill) {
        const size_t slot_elems = planar ? msda::planar_slot_bytes(spatial_size, num_heads, channels, 4) / 4
                                         : (size_t)spatial_size * num_heads * channels;
        st = cuda_status(cudaMemsetAsync(grad_value, 0, sizeof(float) * batch * gframes * slot_elems, s));
        if (st != MSDA_OK) return st;
    }
    if (!work) return MSDA_OK;
    const float *off = (const float *)offsets, *lg = (const float *)logits, *ref = (const float *)reference_points;
    float *goff = (float *)grad_offsets, *glg = (float *)grad_logits;
    if (deterministic)
        return snippet_backward_deterministic(d, (const float *)value, spatial_shapes, level_start_index, off, lg, ref,
                                              (const float *)grad_output, (float *)grad_value, goff, glg, accumulate,
                                              workspace, s);
    if (planar)
        return cuda_status(msda::launch_planar_backward_f32(value, spatial_shapes, level_start_index, off, lg, ref,
                                                            (const float *)grad_output, grad_value, goff, glg, d, s));
    if (dtype == MSDA_DTYPE_BF16)
        return cuda_status(msda::launch_snippet_backward_bf16(value, spatial_shapes, level_start_index, off, lg, ref,
                                                              grad_output, (float *)grad_value, goff, glg, d, s));
    return cuda_status(msda::launch_snippet_backward_f32((const float *)value, spatial_shapes, level_start_index, off,
                                                         lg, ref, (const float *)grad_output, (float *)grad_value, goff,
                                                         glg, d, s));
}

size_t msda_snippet_backward_workspace_bytes(int batch, int n_query_frames, int n_frame, int spatial_size,
                                             int num_heads, int channels, int num_levels, int num_query,
                                             int num_point, int dtype, unsigned flags)
{
    if (!(flags & MSDA_FLAG_DETERMINISTIC) || dtype != MSDA_DTYPE_F32) return 0;
    if (batch <= 0 || n_query_frames <= 0 || n_frame <= 0 || num_query <= 0) return 0;
    const msda::OpDims od = snippet_det_dims(batch, n_query_frames, n_frame, spatial_size, num_heads, channels,
                                             num_levels, num_query, num_point);
    return det_sample_bytes(od, 2) + det_sample_bytes(od, 1) + msda::deterministic_workspace_bytes(od);
}

int msda_snippet_num_slots(int n_query_frames, int n_frame)
{
    if (n_query_frames <= 0 || n_frame <= 0) return 0;
    return msda::snippet_num_slots(n_query_frames, n_frame);
}

int msda_snippet_prefers_presum(int n_src_frames, int n_query_frames, int n_frame, int spatial_size,
                                int num_levels, int num_query, int num_point)
{
    if (n_src_frames <= 0 || n_query_frames <= 0 || n_frame <= 0 || n_frame > n_src_frames) return 0;
    // (t1,t2) pairs the direct gather walks (reference ms_deform_attn.py:137-140,189,201)
    int64_t pairs = 0;
    for (int t1 = 0; t1 < n_query_frames; ++t1) {
        if (t1 < n_frame) {
            const int lo = t1 > 0 ? t1 - 1 : 0, hi = t1 + 1 < n_frame ? t1 + 1 : n_frame - 1;
            pairs += hi - lo + 1;
        } else {
            pairs += n_src_frames;
        }
    }
    // cells gathered by the neighbour-frame loop that the presummed gather does not touch (per head) ...
    const int64_t saved = (pairs - n_query_frames) * (int64_t)num_query * num_levels * num_point * 4;
    // ... against the cells the streaming pass reads and writes (forward; the backward mirrors it)
    const int64_t slots = msda::snippet_num_slots(n_query_frames, n_frame);
    const int64_t streamed = ((int64_t)n_src_frames + slots) * spatial_size;
    return saved >= 4 * streamed ? 1 : 0;
}

static int frame_dims(msda::FrameDims &d, int batch, int n_src_frames, int n_query_frames, int n_frame,
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

int msda_frame_sum(const void *value, const unsigned char *value_mask, void *vsum,
                   int batch, int n_src_frames, int n_query_frames, int n_frame,
                   int spatial_size, int row_elems, int64_t value_stride_n, int64_t value_stride_t,
                   int64_t mask_row_stride, int mask_col_stride, int dtype, void *stream)
{
    msda::FrameDims d;
    const int esize = dtype == MSDA_DTYPE_BF16 ? 2 : 4;
    int st = frame_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, row_elems, value_stride_n,
                        value_stride_t, value_mask, mask_row_stride, mask_col_stride, dtype, esize);
    if (st != MSDA_OK) return st;
    if (batch == 0) return MSDA_OK;
    if (!value || !vsum || misaligned(value, 16) || misaligned(vsum, 16)) return MSDA_ERR_INVALID_ARGUMENT;
    return cuda_status(msda::launch_frame_sum(value, value_mask, vsum, d, esize, static_cast<cudaStream_t>(stream)));
}

int msda_frame_unsum(const void *grad_vsum, const unsigned char *value_mask, void *grad_value,
                     int batch, int n_src_frames, int n_query_frames, int n_frame,
                     int spatial_size, int row_elems, int64_t mask_row_stride, int mask_col_stride,
                     int dtype, void *stream)
{
    msda::FrameDims d;
    int st = frame_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, row_elems, 0, 0,
                        value_mask, mask_row_stride, mask_col_stride, dtype, 4);   // one thread per 4 fp32 channels
    if (st != MSDA_OK) return st;
    if (batch == 0) return MSDA_OK;
    // each thread stores 4 channels: 16 bytes of float32, 8 of bfloat16
    if (!grad_vsum || !grad_value || misaligned(grad_vsum, 16) || misaligned(grad_value, dtype == MSDA_DTYPE_F32 ? 16 : 8))
        return MSDA_ERR_INVALID_ARGUMENT;
    return cuda_status(msda::launch_frame_unsum(static_cast<const float *>(grad_vsum), value_mask, grad_value, d,
                                                dtype == MSDA_DTYPE_BF16 ? 2 : 4, static_cast<cudaStream_t>(stream)));
}

size_t msda_planar_slot_bytes(int spatial_size, int num_heads, int channels, int dtype)
{
    if (dtype != MSDA_DTYPE_F32) return 0;
    return msda::planar_slot_bytes(spatial_size, num_heads, channels, 4);
}

int msda_frame_sum_planar(const void *value, const unsigned char *value_mask, void *vsum_planar,
                          int batch, int n_src_frames, int n_query_frames, int n_frame,
                          int spatial_size, int num_heads, int channels, int64_t value_stride_n, int64_t value_stride_t,
                          int64_t mask_row_stride, int mask_col_stride, int dtype, void *stream)
{
    if (!planar_ok(spatial_size, num_heads, channels, dtype)) return MSDA_ERR_UNSUPPORTED_DTYPE;
    msda::FrameDims d;
    int st = frame_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, num_heads * channels,
                        value_stride_n, value_stride_t, value_mask, mask_row_stride, mask_col_stride, dtype, 4);
    if (st != MSDA_OK) return st;
    if (batch == 0) return MSDA_OK;
    if (!value || !vsum_planar || misaligned(value, 16) || misaligned(vsum_planar, 128))
        return MSDA_ERR_INVALID_ARGUMENT;
    return cuda_status(msda::launch_frame_sum_planar(static_cast<const float *>(value), value_mask, vsum_planar, d,
                                                     num_heads, static_cast<cudaStream_t>(stream)));
}

int msda_frame_unsum_planar(const void *grad_vsum_planar, const unsigned char *value_mask, void *grad_value,
                            int batch, int n_src_frames, int n_query_frames, int n_frame,
                            int spatial_size, int num_heads, int channels, int64_t mask_row_stride, int mask_col_stride,
                            int dtype, void *stream)
{
    if (!planar_ok(spatial_size, num_heads, channels, dtype)) return MSDA_ERR_UNSUPPORTED_DTYPE;
    msda::FrameDims d;
    int st = frame_dims(d, batch, n_src_frames, n_query_frames, n_frame, spatial_size, num_heads * channels, 0, 0,
                        value_mask, mask_row_stride, mask_col_stride, dtype, 4);
    if (st != MSDA_OK) return st;
    if (batch == 0) return MSDA_OK;
    if (!grad_vsum_planar || !grad_value || misaligned(grad_vsum_planar, 128) || misaligned(grad_value, 16))
        return MSDA_ERR_INVALID_ARGUMENT;
    return cuda_status(msda::launch_frame_unsum_planar(grad_vsum_planar, value_mask, static_cast<float *>(grad_value), d,
                                                       num_heads, static_cast<cudaStream_t>(stream)));
}

int msda_layer_tail(const void *y, const void *bias, const void *residual, const void *gamma, const void *beta,
                    const void *pos, void *out, void *out_plus_pos, int64_t rows, int cols, float eps, int dtype,
                    void *stream)
{
    if (dtype != MSDA_DTYPE_F32) return MSDA_ERR_UNSUPPORTED_DTYPE;
    if (rows < 0 || !msda::layer_tail_ok(cols) || !(eps >= 0.f)) return MSDA_ERR_INVALID_ARGUMENT;
    if ((pos == nullptr) != (out_plus_pos == nullptr)) return MSDA_ERR_INVALID_ARGUMENT;
    if (rows == 0) return MSDA_OK;
    const void *ptrs[] = {y, residual, gamma, beta, out};
    for (const void *p : ptrs)
        if (p == nullptr || misaligned(p, 16)) return MSDA_ERR_INVALID_ARGUMENT;
    if (misaligned(bias, 16) || misaligned(pos, 16) || misaligned(out_plus_pos, 16)) return MSDA_ERR_INVALID_ARGUMENT;
    return cuda_status(msda::launch_layer_tail((const float *)y, (const float *)bias, (const float *)residual,
                                               (const float *)gamma, (const float *)beta, (const float *)pos,
                                               (float *)out, (float *)out_plus_pos, rows, cols, eps,
                                               static_cast<cudaStream_t>(stream)));
}

}  // extern "C"
