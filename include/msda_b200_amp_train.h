/*
 * libmsda_b200_amp_train.so -- the companion of libmsda_b200.so for training under torch.autocast(bfloat16): the layer
 * tail with dropout on a bf16 GEMM output, and its backward.  It returns the status codes of msda_b200.h and has an
 * ABI version of its own.
 *
 * Forward (snipper_b200/csrc_amp_train/msda_amp_train_tail.cu), on float(y) and float(residual):
 *     d                 = keep_mask ? ((y + bias) * keep_scale) * m : (y + bias)     m = keep_mask[i] in {0, 1}
 *     h                 = residual + d                                              fp32, saved for the backward
 *     out               = (h - mean) * rstd * gamma + beta                          fp32, the residual stream
 *     out_bf16          = bf16_rn(out)                                              optional: the next GEMM's input
 *     out_plus_pos_bf16 = bf16_rn(out + pos)                                        optional, given together with pos
 *     mean_rstd         = (mean, rstd) per row                                      rows x 2 fp32
 * y: bf16, the raw output of the block's last Linear.  residual: fp32 (residual_dtype MSDA_DTYPE_F32) or bf16
 * (MSDA_DTYPE_BF16).  bias, gamma, beta, pos: fp32; bias may be NULL.  The arithmetic is msda_train_layer_tail_forward's,
 * operation for operation, so out, h and mean_rstd have the bits it gives for float(y), float(residual) and the same
 * mask, and the bf16 outputs the bits of rounding its out and out_plus_pos to nearest even.
 *
 * Backward:
 *     g             = (grad_out + float(grad_out_bf16)) + float(grad_out_plus_pos_bf16)     each bf16 term optional
 *     grad_residual = grad_h                                        in the residual's dtype (residual_dtype)
 *     grad_y        = bf16_rn(keep_mask ? grad_h * keep_scale * m : grad_h)                  bf16, rounded once
 * with grad_h as in msda_train_layer_tail_backward.  (grad_gamma, grad_beta, grad_bias) = sum over rows of
 * (g xhat, g, grad_y before rounding) go to `param_grads` (3 * cols fp32), reduced without atomics through the same
 * fixed grid of per-CTA partial rows and the same ordered sum as libmsda_b200_train.so, so the backward is
 * bit-reproducible, and given the same g its fp32 outputs have that library's bits.  grad_bias is thus summed from fp32
 * values; stock autocast sums the bf16 GEMM-output gradient instead.  `partials` is a caller-owned workspace of
 * msda_amp_train_layer_tail_workspace_bytes(rows, cols) bytes, which only the call itself reads.
 *
 * cols % 128 == 0, cols <= 1024; keep_scale finite and >= 1 (0 <= p < 1); eps >= 0; every row dense; every pointer
 * 16-byte aligned, the required ones not NULL; rows == 0 is a no-op.
 */
#ifndef MSDA_B200_AMP_TRAIN_H_
#define MSDA_B200_AMP_TRAIN_H_

#include "msda_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_AMP_TRAIN_ABI_VERSION 1

MSDA_API int msda_amp_train_abi_version(void);
/* cudaError_t of the last failed launch of this library seen by this thread (0 if none). */
MSDA_API int msda_amp_train_last_cuda_error(void);

MSDA_API int msda_amp_train_layer_tail_forward(const void *y, const float *bias, const void *residual,
                                               int residual_dtype, const uint8_t *keep_mask, float keep_scale,
                                               const float *gamma, const float *beta, const float *pos, float *out,
                                               void *out_bf16, void *out_plus_pos_bf16, float *h, float *mean_rstd,
                                               int64_t rows, int cols, float eps, void *stream);

/* Bytes of the backward's `partials` workspace (0 when rows == 0 or cols is not supported). */
MSDA_API size_t msda_amp_train_layer_tail_workspace_bytes(int64_t rows, int cols);

MSDA_API int msda_amp_train_layer_tail_backward(const float *grad_out, const void *grad_out_bf16,
                                                const void *grad_out_plus_pos_bf16, const float *h,
                                                const float *mean_rstd, const uint8_t *keep_mask, float keep_scale,
                                                const float *gamma, void *grad_residual, int residual_dtype,
                                                void *grad_y, float *param_grads, float *partials, int64_t rows,
                                                int cols, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_AMP_TRAIN_H_ */
