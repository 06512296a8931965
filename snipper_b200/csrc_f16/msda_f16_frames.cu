// Neighbour-frame pre-summation with fp16 slots: the kernels of csrc/msda_frames.cuh for __half.
#include "../csrc/msda_frames.cuh"
#include "msda_f16_internal.h"

namespace msda {

cudaError_t launch_frame_sum_f16(const void *value, const uint8_t *mask, void *vsum, const FrameDims &d,
                                 cudaStream_t stream)
{
    return launch_frame_sum_typed(static_cast<const __half *>(value), mask, static_cast<__half *>(vsum), d, stream);
}

cudaError_t launch_frame_unsum_f16(const float *grad_vsum, const uint8_t *mask, void *grad_value, const FrameDims &d,
                                   cudaStream_t stream)
{
    return launch_frame_unsum_typed(grad_vsum, mask, static_cast<__half *>(grad_value), d, stream);
}

}  // namespace msda
