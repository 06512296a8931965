// Neighbour-frame pre-summation for the fused snippet attention (sm_100a).
//
// The reference module (models/ops/modules/ms_deform_attn.py:130-225) calls the op once per
// (query frame t1, neighbour frame t2) with the SAME sampling locations and the SAME attention
// weights for every t2 (the frame slots alias one Linear, :68-71) and sums the results (:225).
// The op is linear in `value`, so
//
//     sum_{t2 in nb(t1)} msda(value[:, t2], loc, A)  ==  msda( sum_{t2 in nb(t1)} value[:, t2], loc, A )
//
// and one streaming pass that builds the per-query-frame sums ("slots") lets the gather kernel read ONE
// frame per query frame instead of |nb(t1)| (10 frame pairs -> 4 gathers at T = 4: 2.5 x fewer bytes
// through the L1 data pipe, which is what bounds the gather; the same factor on the vector reductions of
// the backward).  This pass also applies the padding mask (`value.masked_fill(mask, 0)`, :116-117), so no
// separate masking pass over the value tensor exists any more.
//
//   slots:  j <  n_local = min(T1, n_frame):  frames max(j-1,0) .. min(j+1, n_frame-1)   (:137-140)
//           j == n_local (only if T1 > n_frame, "future" query frames): all T2 frames    (:189,201)
//
//   frame_sum    vsum[n, j, s, :]       = sum_{t2 in slot j} (mask[n,t2,s,:] ? 0 : value[n,t2,s,:])
//   frame_unsum  grad_value[n, t2, s, :] = mask ? 0 : sum_{j : t2 in slot j} grad_vsum[n, j, s, :]
//
// Both are plain HBM/L2 streaming kernels: one thread per 16-byte chunk of a (n, s) row, every source
// frame loaded once into registers, sums formed in a fixed (ascending frame / slot) order, so the
// results are bit-reproducible.  mask element (n,t,s,c) lives at mask[((n*T2+t)*S+s)*mask_row_stride +
// c*mask_col_stride]: col stride 1 = the reference's materialised (N,T,S,C) bool tensor
// (models/model.py:156-157), col stride 0 = a per-pixel predicate (1 byte per pixel instead of C).
#include "msda_frames.cuh"

namespace msda {

cudaError_t launch_frame_sum(const void *value, const uint8_t *mask, void *vsum, const FrameDims &d, int esize,
                             cudaStream_t stream)
{
    if (esize == 4)
        return launch_frame_sum_typed(static_cast<const float *>(value), mask, static_cast<float *>(vsum), d, stream);
    return launch_frame_sum_typed(static_cast<const __nv_bfloat16 *>(value), mask, static_cast<__nv_bfloat16 *>(vsum), d,
                                  stream);
}

cudaError_t launch_frame_unsum(const float *grad_vsum, const uint8_t *mask, void *grad_value, const FrameDims &d,
                               int out_esize, cudaStream_t stream)
{
    if (out_esize == 4)
        return launch_frame_unsum_typed(grad_vsum, mask, static_cast<float *>(grad_value), d, stream);
    return launch_frame_unsum_typed(grad_vsum, mask, static_cast<__nv_bfloat16 *>(grad_value), d, stream);
}

}  // namespace msda
