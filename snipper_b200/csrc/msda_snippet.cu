// Fused Snipper snippet attention: one launch per transformer layer (sm_100a, fp32).
//
// Replaces the Python per-frame loop of the reference module
// (models/ops/modules/ms_deform_attn.py:126-225): for every query frame t1 the reference
// re-runs the sampling_offsets / attention_weights GEMMs per neighbour frame t2, a softmax over
// (levels, points, neighbour frames), two .contiguous() copies and one op launch per (t1,t2)
// pair (10 pairs at T=4), then stacks and sums.  Because every frame slot holds the SAME Linear
// (ms_deform_attn.py:68-71) the logits/offsets do not depend on t2, so
//     softmax_{l,p,k}(logits)[.., j] = softmax_{l,p}(logits) / k      (k = #neighbour frames)
// and the whole loop collapses to: per (n,t1,q,m) set up L*P samples ONCE
// (loc = ref + offset/(W,H); A = softmax/k) and gather them from each of the k neighbour
// frames of `value`, accumulating in registers.
//
// Same CTA organisation as the per-call fast path (msda_percall.cu): PAIRS pairs x LANES lanes,
// phase 1 = one thread per sample (here it also does the softmax and the offset normalisation),
// phase 2 = lanes gather 128-bit channel chunks; backward adds vector reductions into
// grad_value, 4-lane shuffles for the per-sample scalars and the softmax backward in phase 3.
#include "msda_snippet.cuh"

namespace msda {

// Few-queries forward (the decoder's cross-attention: 60 queries per frame).  With 16 or 8 queries per CTA such a launch
// is a few hundred CTAs whose lanes walk L*P samples x |nb(t1)| frames one after the other -- a chain of ~24 dependent
// round trips to L2 / HBM (58-66 us per launch for 53 MB of traffic, profiles/r02_run9_launch_list_summary.txt).  Here
// ONE (query, head) pair owns a CTA and thread = (sample, 16-byte chunk): every thread issues the loads of its
// sample's neighbour frames at once (one round trip), the L*P partial sums meet in shared memory.
template <int LANES, int BLOCK, int MODE>
__global__ void __launch_bounds__(BLOCK)
msda_snippet_fwd_split_kernel(const float *__restrict__ value, const int64_t *__restrict__ shapes,
                              const int64_t *__restrict__ lsi, const float *__restrict__ offsets,
                              const float *__restrict__ logits, const float *__restrict__ ref,
                              float *__restrict__ out, const SnipArgs a)
{
    using C = Chunk<float>;
    const SnippetDims &d = a.d;
    __shared__ LevelTable lv;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int LP = d.L * d.P;
    float4 *rec = reinterpret_cast<float4 *>(smem_raw);                    // LP + 1 records
    float4 *red = rec + (LP + 1);                                          // [sample][chunk] partial sums
    float *zs = reinterpret_cast<float *>(red + LP * LANES);

    const int tid = threadIdx.x;
    const int m = blockIdx.x, q = blockIdx.y;
    const int n = blockIdx.z / d.T1, t1 = blockIdx.z - n * d.T1;
    int lo, hi;
    frame_range(t1, d.n_frame, d.T2, lo, hi);
    const int nf = hi - lo + 1;
    const size_t qbase = ((size_t)n * d.T1 + t1) * d.Lq;

    snippet_phase1<BLOCK, 1>(rec, zs, lv, shapes, lsi, a, n, t1, q, m, qbase, offsets, logits, ref, 1.f / (float)nf);

    const int sidx = tid / LANES, lane = tid - sidx * LANES;
    if (sidx < LP) {
        const char *pf = reinterpret_cast<const char *>(value + n * d.value_stride_n + lo * d.value_stride_t) +
                         (size_t)(m * LANES + lane) * C::BYTES;
        const int64_t fstride = d.value_stride_t * (int64_t)sizeof(float);
        const int level_w = lv.W[fast_div(sidx, a.magic_P)];
        const float4 r = rec[sidx];
        C acc = zero_chunk<C>();
        if (MODE == kDirectMasked) {
            MaskView mv;
            mv.row = d.mask_row_stride;
            mv.frame = (int64_t)d.S * d.mask_row_stride;
            mv.col = d.mask_col_stride;
            mv.inv_cell_bytes = 1.f / (float)a.cell_bytes;
            mv.p = d.mask + ((int64_t)n * d.T2 + lo) * mv.frame + (int64_t)((m * LANES + lane) * C::N) * mv.col;
            gather_fma_frames_masked<float>(acc, record_meta(r, (unsigned)(level_w * a.cell_bytes)), record_weights(r), pf,
                                            fstride, nf, a.cell_bytes, level_w, mv);
        } else {
            gather_fma_frames<float, 0>(acc, record_meta(r, (unsigned)(level_w * a.cell_bytes)), record_weights(r), pf,
                                        fstride, nf, a.cell_bytes);
        }
        red[sidx * LANES + lane] = make_float4(acc.x[0], acc.x[1], acc.x[2], acc.x[3]);
    }
    __syncthreads();
    if (tid < LANES) {
        float4 sum = red[tid];
        for (int j = 1; j < LP; ++j) {       // fixed order: bit-reproducible
            const float4 v = red[j * LANES + tid];
            sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
        }
        const size_t pair = (qbase + q) * d.M + m;
        *reinterpret_cast<float4 *>(reinterpret_cast<char *>(out) + (pair * LANES + tid) * C::BYTES) = sum;
    }
}

// MSDA_FWD_SPLIT=0 in the environment keeps the tile kernels for few-queries launches (benchmark knob, read once)
static bool fwd_split_on()
{
    static const bool v = [] { const char *e = getenv("MSDA_FWD_SPLIT"); return !(e && e[0] == '0'); }();
    return v;
}

template <int LANES>
static cudaError_t launch_snip_fwd_split(const float *value, const int64_t *shapes, const int64_t *lsi,
                                         const float *offsets, const float *logits, const float *ref, float *out,
                                         const SnippetDims &d, cudaStream_t stream)
{
    const SnipArgs a = make_snip_args<float>(d);
    const int LP = d.L * d.P;
    const dim3 grid(d.M, d.Lq, d.N * d.T1);
    const size_t smem = sizeof(float4) * (LP + 1 + LP * LANES) + sizeof(float) * LP;
    const bool masked = d.mask != nullptr;
#define MSDA_LAUNCH_SPLIT(BLOCK_)                                                                                         \
    do {                                                                                                                  \
        if (masked)                                                                                                       \
            msda_snippet_fwd_split_kernel<LANES, BLOCK_, kDirectMasked><<<grid, BLOCK_, smem, stream>>>(                  \
                value, shapes, lsi, offsets, logits, ref, out, a);                                                        \
        else                                                                                                              \
            msda_snippet_fwd_split_kernel<LANES, BLOCK_, kDirect><<<grid, BLOCK_, smem, stream>>>(                        \
                value, shapes, lsi, offsets, logits, ref, out, a);                                                        \
    } while (0)
    if (LP * LANES <= 160) MSDA_LAUNCH_SPLIT(160);
    else MSDA_LAUNCH_SPLIT(kSnippetMaxLP * LANES);
#undef MSDA_LAUNCH_SPLIT
    return cudaGetLastError();
}

template <typename VT, int LANES, int PAIRS>
static cudaError_t launch_snip_bwd_noscatter(const typename Chunk<VT>::elem *value, const int64_t *shapes,
                                             const int64_t *lsi, const float *offsets, const float *logits,
                                             const float *ref, const typename Chunk<VT>::elem *grad_out,
                                             float *grad_offsets, float *grad_logits, const SnippetDims &d,
                                             cudaStream_t stream)
{
    using Cfg = SnipCfg<LANES, PAIRS>;
    const SnipArgs a = make_snip_args<VT>(d);
    const dim3 grid(d.M, (d.Lq + PAIRS - 1) / PAIRS, d.N * d.T1);
    const size_t smem = sizeof(float4) * Cfg::PAIRS * (d.L * d.P + 1) + sizeof(float) * 3 * Cfg::SUBS * Cfg::PAIRS * d.L * d.P;
    auto kernel = msda_snippet_bwd_kernel<VT, LANES, PAIRS, 0, kPresummed, false>;
    if (smem > kSmemOptIn) {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    kernel<<<grid, Cfg::THREADS, smem, stream>>>(value, shapes, lsi, offsets, logits, ref, grad_out, nullptr,
                                                grad_offsets, grad_logits, a);
    return cudaGetLastError();
}

// Per-sample sampling locations and attention weights written out (deterministic mode only: the two-pass
// grad_value of msda_deterministic.cu consumes the per-call layout).  One thread per (n,t1,q,m); same
// operation order as snippet_phase1, so floor() picks the cells the forward gathered.
__global__ void __launch_bounds__(128)
snippet_loc_attn_kernel(const int64_t *__restrict__ shapes, const int64_t *__restrict__ lsi,
                        const float *__restrict__ offsets, const float *__restrict__ logits,
                        const float *__restrict__ ref, float *__restrict__ loc, float *__restrict__ attn,
                        const SnippetDims d, int64_t total)
{
    __shared__ LevelTable lv;
    load_level_table(lv, shapes, lsi, d.L, d.S);
    __syncthreads();
    const int LP = d.L * d.P;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int m = (int)(i % d.M);
        const int64_t row = i / d.M;                       // (n*T1 + t1)*Lq + q
        const int q = (int)(row % d.Lq);
        const int64_t nt = row / d.Lq;
        const int t1 = (int)(nt % d.T1), n = (int)(nt / d.T1);
        int lo, hi;
        frame_range(t1, d.n_frame, d.T2, lo, hi);
        const float inv_k = 1.f / (float)(hi - lo + 1);
        const float *zrow = logits + row * d.logit_row_stride + m * LP;
        const float *zb = d.logit_bias ? d.logit_bias + m * LP : nullptr;
        float mx = -INFINITY;
        for (int j = 0; j < LP; ++j) mx = fmaxf(mx, __ldg(zrow + j) + (zb ? __ldg(zb + j) : 0.f));
        float sum = 0.f;
        for (int j = 0; j < LP; ++j) sum += expf(__ldg(zrow + j) + (zb ? __ldg(zb + j) : 0.f) - mx);
        const float2 *orow = reinterpret_cast<const float2 *>(offsets + row * d.off_row_stride) + m * LP;
        const float2 *ob = d.off_bias ? reinterpret_cast<const float2 *>(d.off_bias) + m * LP : nullptr;
        for (int j = 0; j < LP; ++j) {
            const int l = j / d.P;
            float2 o = __ldg(orow + j);
            if (ob) { const float2 b = __ldg(ob + j); o.x += b.x; o.y += b.y; }
            float2 r2;
            if (d.valid_ratios != nullptr) {
                r2 = analytic_reference_point(lv, d.valid_ratios + (size_t)n * d.L * 2, d.L, q, l);
            } else {
                const float *rp = ref + n * d.ref_stride_n + t1 * d.ref_stride_t + ((int64_t)q * d.L + l) * 2;
                r2 = make_float2(__ldg(rp), __ldg(rp + 1));
            }
            const int64_t si = i * LP + j;
            loc[2 * si] = r2.x + o.x / (float)lv.W[l];
            loc[2 * si + 1] = r2.y + o.y / (float)lv.H[l];
            attn[si] = expf(__ldg(zrow + j) + (zb ? __ldg(zb + j) : 0.f) - mx) / sum * inv_k;
        }
    }
}

cudaError_t launch_snippet_forward_f32(const float *value, const int64_t *shapes,
                                       const int64_t *lsi, const float *offsets,
                                       const float *logits, const float *ref, float *out,
                                       const SnippetDims &d, cudaStream_t stream)
{
    // few queries (decoder): latency-bound -- one CTA per (query, head), samples spread over the threads
    if (!d.presummed && d.D == 48 && d.Lq <= 65535 && fwd_split_on() &&
        pick_pairs_d48(snip_pairs_d48(), d.Lq, d.M, d.N * d.T1) == 8)
        return launch_snip_fwd_split<12>(value, shapes, lsi, offsets, logits, ref, out, d, stream);
#define CALL(VT, LN, PR) launch_snip_fwd<VT, LN, PR>(value, shapes, lsi, offsets, logits, ref, out, d, stream)
    MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
}

cudaError_t launch_snippet_backward_f32(const float *value, const int64_t *shapes,
                                        const int64_t *lsi, const float *offsets,
                                        const float *logits, const float *ref,
                                        const float *grad_out, float *grad_value,
                                        float *grad_offsets, float *grad_logits,
                                        const SnippetDims &d, cudaStream_t stream)
{
#define CALL(VT, LN, PR) \
    launch_snip_bwd<VT, LN, PR>(value, shapes, lsi, offsets, logits, ref, grad_out, grad_value, grad_offsets, grad_logits, d, stream)
    MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
}

cudaError_t launch_snippet_backward_noscatter_f32(const float *value, const int64_t *shapes, const int64_t *lsi,
                                                  const float *offsets, const float *logits, const float *ref,
                                                  const float *grad_out, float *grad_offsets, float *grad_logits,
                                                  const SnippetDims &d, cudaStream_t stream)
{
    if (!d.presummed) return cudaErrorInvalidValue;
#define CALL(VT, LN, PR) \
    launch_snip_bwd_noscatter<VT, LN, PR>(value, shapes, lsi, offsets, logits, ref, grad_out, grad_offsets, grad_logits, d, stream)
    MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
}

cudaError_t launch_snippet_loc_attn(const int64_t *shapes, const int64_t *lsi, const float *offsets,
                                    const float *logits, const float *ref, float *loc, float *attn,
                                    const SnippetDims &d, cudaStream_t stream)
{
    const int64_t total = (int64_t)d.N * d.T1 * d.Lq * d.M;
    if (total == 0) return cudaSuccess;
    const int64_t blocks = (total + 127) / 128;
    snippet_loc_attn_kernel<<<(int)(blocks < 148 * 32 ? blocks : 148 * 32), 128, 0, stream>>>(shapes, lsi, offsets, logits,
                                                                                           ref, loc, attn, d, total);
    return cudaGetLastError();
}

cudaError_t launch_snippet_forward_bf16(const void *value, const int64_t *shapes,
                                        const int64_t *lsi, const float *offsets,
                                        const float *logits, const float *ref, void *out,
                                        const SnippetDims &d, cudaStream_t stream)
{
    return launch_snippet_forward_half<__nv_bfloat16, bf16q>(value, shapes, lsi, offsets, logits, ref, out, d, stream);
}

cudaError_t launch_snippet_backward_bf16(const void *value, const int64_t *shapes,
                                         const int64_t *lsi, const float *offsets,
                                         const float *logits, const float *ref,
                                         const void *grad_out, float *grad_value,
                                         float *grad_offsets, float *grad_logits,
                                         const SnippetDims &d, cudaStream_t stream)
{
    return launch_snippet_backward_half<__nv_bfloat16, bf16q>(value, shapes, lsi, offsets, logits, ref, grad_out,
                                                              grad_value, grad_offsets, grad_logits, d, stream);
}

}  // namespace msda
