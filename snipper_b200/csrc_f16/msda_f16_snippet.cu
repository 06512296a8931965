// Fused snippet op with fp16 value (or fp16 pre-summed slots) / output / grad_output: the kernels of
// csrc/msda_snippet.cuh on fp16 lanes, with the bf16 mode's dispatch.
#include "../csrc/msda_snippet.cuh"
#include "msda_f16_internal.h"

namespace msda {

cudaError_t launch_snippet_forward_f16(const void *value, const int64_t *shapes, const int64_t *lsi,
                                       const float *offsets, const float *logits, const float *ref, void *out,
                                       const SnippetDims &d, cudaStream_t stream)
{
    return launch_snippet_forward_half<__half, halfq>(value, shapes, lsi, offsets, logits, ref, out, d, stream);
}

cudaError_t launch_snippet_backward_f16(const void *value, const int64_t *shapes, const int64_t *lsi,
                                        const float *offsets, const float *logits, const float *ref,
                                        const void *grad_out, float *grad_value, float *grad_offsets,
                                        float *grad_logits, const SnippetDims &d, cudaStream_t stream)
{
    return launch_snippet_backward_half<__half, halfq>(value, shapes, lsi, offsets, logits, ref, grad_out, grad_value,
                                                       grad_offsets, grad_logits, d, stream);
}

}  // namespace msda
