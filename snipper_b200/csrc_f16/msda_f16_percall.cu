// Per-call op with fp16 value / output / grad_output: the fast kernels of csrc/msda_percall.cuh on fp16 lanes, with the
// bf16 mode's dispatch (16-byte lanes forward, 8-byte lanes backward and for few-CTA or split forwards).
#include "../csrc/msda_percall.cuh"
#include "msda_f16_internal.h"

namespace msda {

cudaError_t launch_forward_fast_f16(const void *value, const int64_t *shapes, const int64_t *lsi, const float *loc,
                                    const float *attn, void *out, const OpDims &d, cudaStream_t stream)
{
    return launch_forward_fast_half<__half, halfq>(value, shapes, lsi, loc, attn, out, d, stream);
}

cudaError_t launch_backward_fast_f16(const void *value, const int64_t *shapes, const int64_t *lsi, const float *loc,
                                     const float *attn, const void *grad_out, float *grad_value, float *grad_loc,
                                     float *grad_attn, const OpDims &d, cudaStream_t stream)
{
    return launch_backward_fast_half<__half, halfq>(value, shapes, lsi, loc, attn, grad_out, grad_value, grad_loc,
                                                    grad_attn, d, stream);
}

}  // namespace msda
