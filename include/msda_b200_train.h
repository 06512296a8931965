/*
 * libmsda_b200_train.so -- the training companion of libmsda_b200.so: the layer tail with dropout and its backward.
 * It returns the status codes of msda_b200.h and has an ABI version of its own.  fp32 only.
 *
 * Forward (snipper_b200/csrc_train/msda_train_tail.cu):
 *     d            = keep_mask ? ((y + bias) * keep_scale) * m : (y + bias)        m = keep_mask[i] in {0, 1}
 *     h            = residual + d                                                  saved for the backward
 *     out          = (h - mean) * rstd * gamma + beta                              two-pass mean / variance
 *     out_plus_pos = out + pos                                                     optional, given together with pos
 *     mean_rstd    = (mean, rstd) per row                                          rows x 2 fp32
 * keep_mask is one byte per element (dense rows of cols bytes), drawn by the caller; keep_scale = 1 / (1 - p) in
 * float.  Without keep_mask the arithmetic is msda_layer_tail's, in its order, so `out` has its bits; with it, `out`
 * has the bits msda_layer_tail gives for the pre-dropped input ((y + bias) * keep_scale) * m and bias = NULL.
 *
 * Backward:
 *     g             = grad_out (+ grad_out_plus_pos)
 *     xhat          = (h - mean) * rstd
 *     grad_h        = rstd * (gamma g - mean_c(gamma g) - xhat * mean_c(gamma g xhat))
 *     grad_residual = grad_h
 *     grad_y        = keep_mask ? grad_h * keep_scale * m : grad_h                 also the gradient of y + bias
 * and, without atomics, (grad_gamma, grad_beta, grad_bias) = sum over rows of (g xhat, g, grad_y): a fixed grid (a
 * function of rows only) writes one partial row per CTA into `partials`, which a second kernel sums in a fixed order.
 * The result is bit-reproducible run to run.  `param_grads` (3 * cols floats) receives
 * (grad_gamma, grad_beta, grad_bias), each cols long; `partials` is a caller-owned workspace of
 * msda_train_layer_tail_workspace_bytes(rows, cols) bytes, which only the call itself reads.
 *
 * cols % 128 == 0, cols <= 1024; keep_scale finite and >= 1 (0 <= p < 1); eps >= 0; every row dense; every pointer
 * 16-byte aligned, the required ones not NULL; rows == 0 is a no-op.
 */
#ifndef MSDA_B200_TRAIN_H_
#define MSDA_B200_TRAIN_H_

#include "msda_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_TRAIN_ABI_VERSION 1

MSDA_API int msda_train_abi_version(void);
/* cudaError_t of the last failed launch of this library seen by this thread (0 if none). */
MSDA_API int msda_train_last_cuda_error(void);

MSDA_API int msda_train_layer_tail_forward(const float *y, const float *bias, const float *residual,
                                           const uint8_t *keep_mask, float keep_scale, const float *gamma,
                                           const float *beta, const float *pos, float *out, float *out_plus_pos,
                                           float *h, float *mean_rstd, int64_t rows, int cols, float eps,
                                           void *stream);

/* Bytes of the backward's `partials` workspace (0 when rows == 0 or cols is not supported). */
MSDA_API size_t msda_train_layer_tail_workspace_bytes(int64_t rows, int cols);

MSDA_API int msda_train_layer_tail_backward(const float *grad_out, const float *grad_out_plus_pos, const float *h,
                                            const float *mean_rstd, const uint8_t *keep_mask, float keep_scale,
                                            const float *gamma, float *grad_residual, float *grad_y,
                                            float *param_grads, float *partials, int64_t rows, int cols,
                                            void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_TRAIN_H_ */
