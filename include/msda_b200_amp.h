/*
 * libmsda_b200_amp.so -- the mixed-precision companion of libmsda_b200.so for inference under
 * torch.autocast(bfloat16).  It returns the status codes of msda_b200.h and has an ABI version of its own.
 *
 * Layer tail with a bf16 GEMM output in front and bf16 GEMM inputs behind (snipper_b200/csrc_amp/msda_amp_tail.cu):
 *     x                 = residual + (float(y) + bias)                       (rows, cols)
 *     out               = LayerNorm(x) * gamma + beta                        fp32, always written
 *     out_bf16          = bf16_rn(out)                                       optional
 *     out_plus_pos_bf16 = bf16_rn(out + pos)                                 optional, given together with pos
 * y: bf16, the raw output of the block's last Linear (bias not added; bias may be NULL).  residual: fp32
 * (residual_dtype MSDA_DTYPE_F32) or bf16 (MSDA_DTYPE_BF16).  bias, gamma, beta, pos: fp32.  The arithmetic is
 * msda_layer_tail's, in its order, so `out` has the bits msda_layer_tail gives for float(y), float(residual); the
 * two bf16 outputs have the bits of rounding out and out + pos to nearest even, which is what autocast's own cast
 * of those tensors in front of the next GEMM makes.
 * cols % 128 == 0, cols <= 1024; every row dense, every pointer 16-byte aligned; rows == 0 is a no-op.
 * Inference only (no gradient formula is provided).
 */
#ifndef MSDA_B200_AMP_H_
#define MSDA_B200_AMP_H_

#include "msda_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_AMP_ABI_VERSION 1

MSDA_API int msda_amp_abi_version(void);
/* cudaError_t of the last failed launch of this library seen by this thread (0 if none). */
MSDA_API int msda_amp_last_cuda_error(void);

MSDA_API int msda_amp_layer_tail(const void *y, const void *bias, const void *residual, int residual_dtype,
                                 const void *gamma, const void *beta, const void *pos, void *out, void *out_bf16,
                                 void *out_plus_pos_bf16, int64_t rows, int cols, float eps, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_AMP_H_ */
