// Launchers of libmsda_b200_f16.so: the templates of csrc/ instantiated for fp16 lanes (__half, halfq).
#pragma once

#include "../csrc/msda_internal.h"

namespace msda {

cudaError_t launch_forward_fast_f16(const void *value, const int64_t *shapes, const int64_t *lsi, const float *loc,
                                    const float *attn, void *out, const OpDims &d, cudaStream_t stream);
cudaError_t launch_backward_fast_f16(const void *value, const int64_t *shapes, const int64_t *lsi, const float *loc,
                                     const float *attn, const void *grad_out, float *grad_value, float *grad_loc,
                                     float *grad_attn, const OpDims &d, cudaStream_t stream);
cudaError_t launch_snippet_forward_f16(const void *value, const int64_t *shapes, const int64_t *lsi,
                                       const float *offsets, const float *logits, const float *ref, void *out,
                                       const SnippetDims &d, cudaStream_t stream);
cudaError_t launch_snippet_backward_f16(const void *value, const int64_t *shapes, const int64_t *lsi,
                                        const float *offsets, const float *logits, const float *ref,
                                        const void *grad_out, float *grad_value, float *grad_offsets,
                                        float *grad_logits, const SnippetDims &d, cudaStream_t stream);
cudaError_t launch_frame_sum_f16(const void *value, const uint8_t *mask, void *vsum, const FrameDims &d,
                                 cudaStream_t stream);
cudaError_t launch_frame_unsum_f16(const float *grad_vsum, const uint8_t *mask, void *grad_value, const FrameDims &d,
                                   cudaStream_t stream);

}  // namespace msda
