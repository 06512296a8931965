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
#include "msda_snippet_common.cuh"

namespace msda {

#ifndef MSDA_BWD_PRESUM_THREADS
#define MSDA_BWD_PRESUM_THREADS 960   // resident threads per SM the presummed backward is compiled for (5 x 192)
#endif

// How phase 2 reaches `value` (a template constant: the three bodies share phase 1 and the epilogues)
//   kDirect        gather every neighbour frame of value (N,T2,S,M,D)            -- few queries (decoder)
//   kDirectMasked  same, with the padding mask applied to every gathered chunk / scattered reduction
//   kPresummed     `value` holds the neighbour-frame SUMS, one slot per query frame (msda_frames.cu):
//                  one gather per sample instead of |nb(t1)|                      -- encoder
enum { kDirect = 0, kDirectMasked = 1, kPresummed = 2 };

// grid = (M, query tiles, N*T1): a CTA owns PAIRS consecutive queries of ONE head of one
// (batch item, query frame); neighbouring encoder queries gather overlapping cells (L1 hits).
template <int LANES, int PAIRS_>
struct SnipCfg {
    static constexpr int PAIRS = PAIRS_;
    static constexpr int THREADS = PAIRS * LANES;
    static constexpr int SUBG = sub_group(LANES);
    static constexpr int SUBS = LANES / SUBG;
    static constexpr int BWD_MIN_BLOCKS = 768 / THREADS < 1 ? 1 : (768 / THREADS > 16 ? 16 : 768 / THREADS);  // <= 80 regs
    // presummed backward: no neighbour-frame loop to keep in flight, so a tighter register budget costs nothing
    static constexpr int BWD_MIN_BLOCKS_PRESUM = MSDA_BWD_PRESUM_THREADS / THREADS < 1 ? 1 : (MSDA_BWD_PRESUM_THREADS / THREADS > 16 ? 16 : MSDA_BWD_PRESUM_THREADS / THREADS);
    static_assert(LANES % 2 == 0 && THREADS % 32 == 0 && THREADS <= 1024, "lane groups must tile warps");
};

// ---- padding mask applied in the gather (kDirectMasked) ----
// bit i set <=> channel i of the lane's chunk is masked (col stride 0: one byte per pixel)
template <int N>
__device__ __forceinline__ unsigned lane_mask_bits(const uint8_t *__restrict__ mp, int col_stride)
{
    if (col_stride == 0) return __ldg(mp) ? (1u << N) - 1u : 0u;
    unsigned bits = 0u;
#pragma unroll
    for (int w = 0; w < N / 4; ++w) {
        const unsigned mk = __ldg(reinterpret_cast<const unsigned *>(mp) + w);
#pragma unroll
        for (int b = 0; b < 4; ++b)
            if ((mk >> (8 * b)) & 0xffu) bits |= 1u << (4 * w + b);
    }
    return bits;
}

struct MaskView {
    const uint8_t *p;      // mask element of (n, first gathered frame, cell 0, this lane's first channel)
    int64_t row, frame;    // bytes between consecutive cells / frames
    int col;
    float inv_cell_bytes;  // 1 / (M * D * sizeof(VT))
};

// cell index of a sample's (y0,x0) corner from its byte offset: off is a multiple of 16 below 2^28, hence exact in
// fp32, and the quotient (< 2^24) survives the reciprocal's rounding -- no integer division in the gather loop
__device__ __forceinline__ int cell_of(int off, float inv_cell_bytes)
{
    return __float2int_rn(__int2float_rn(off) * inv_cell_bytes);
}

// != 0 <=> some channel of the lane's chunk is masked (the cheap test; lane_mask_bits says which)
template <int N>
__device__ __forceinline__ unsigned lane_mask_any(const uint8_t *__restrict__ mp, int col_stride)
{
    if (col_stride == 0) return __ldg(mp);
    unsigned any = 0u;
#pragma unroll
    for (int w = 0; w < N / 4; ++w) any |= __ldg(reinterpret_cast<const unsigned *>(mp) + w);
    return any;
}

// forward, all neighbour frames, every gathered chunk masked (value.masked_fill(mask, 0), ms_deform_attn.py:116-117).
// The four mask reads and the four value reads of a frame are issued together (corners outside the level are
// predicated off); padding is rare, so the common case -- no masked channel under any corner -- runs the plain
// 16 FMAs and only samples next to padding take the per-channel path.
template <typename VT>
__device__ __forceinline__ void gather_fma_frames_masked(Chunk<VT> &acc, const SampleMeta mt, const float4 w,
                                                         const char *__restrict__ pf, int64_t frame_bytes, int nf,
                                                         int csb, int level_w, const MaskView &mv)
{
    using C = Chunk<VT>;
    const unsigned cm = mt.wm >> 28;
    if (cm == 0u) return;
    const ptrdiff_t row = (ptrdiff_t)(mt.wm & 0x0fffffffu);
    const char *a0 = pf + (ptrdiff_t)mt.off;
    const uint8_t *m0 = mv.p + (int64_t)cell_of(mt.off, mv.inv_cell_bytes) * mv.row;
    const int64_t mrow = (int64_t)level_w * mv.row;
    const ptrdiff_t vo[4] = {0, csb, row, row + csb};
    const int64_t mo[4] = {0, mv.row, mrow, mrow + mv.row};
    const float wk[4] = {w.x, w.y, w.z, w.w};
#pragma unroll 2
    for (int f = 0; f < nf; ++f, a0 += frame_bytes, m0 += mv.frame) {
        unsigned any = 0u;
        C v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            v[k] = zero_chunk<C>();             // a corner outside the level contributes nothing
            if (cm & (1u << k)) {
                any |= lane_mask_any<C::N>(m0 + mo[k], mv.col);
                v[k] = C::load(a0 + vo[k]);
            }
        }
        if (any == 0u) {
#pragma unroll
            for (int k = 0; k < 4; ++k) fma_chunk(acc, wk[k], v[k]);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (!(cm & (1u << k))) continue;
                const unsigned bits = lane_mask_bits<C::N>(m0 + mo[k], mv.col);
#pragma unroll
                for (int i = 0; i < C::N; ++i)
                    if (!(bits & (1u << i))) acc.x[i] = fmaf(wk[k], v[k].x[i], acc.x[i]);
            }
        }
    }
}

// backward of one sample on one frame with the mask: masked channels of value read as zero and receive no gradient
template <typename VT>
__device__ __forceinline__ void gather_scatter_masked(const SampleMeta mt, const BwdWeights &b, const Chunk<VT> &g,
                                                      const RedView<VT> &gr, const char *__restrict__ p0, char *gp0,
                                                      int csb, int level_w, const uint8_t *__restrict__ m0,
                                                      int64_t mrow, int mcol, float inv_cell_bytes,
                                                      float &pa, float &px, float &py)
{
    using C = Chunk<VT>;
    static_assert(C::N == 4, "backward lanes own four channels");
    constexpr int GS = 4 / (int)sizeof(typename C::elem);
    const unsigned cm = mt.wm >> 28;
    if (cm == 0u) return;
    const ptrdiff_t row = (ptrdiff_t)(mt.wm & 0x0fffffffu);
    const int64_t cell0 = cell_of(mt.off, inv_cell_bytes);
    const ptrdiff_t o[4] = {(ptrdiff_t)mt.off, (ptrdiff_t)mt.off + csb, (ptrdiff_t)mt.off + row, (ptrdiff_t)mt.off + row + csb};
    const int64_t mc[4] = {cell0, cell0 + 1, cell0 + level_w, cell0 + level_w + 1};
    const float aw[4] = {b.a0, b.a1, b.a2, b.a3};
    unsigned any = 0u;
    C v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        v[k] = zero_chunk<C>();
        if (cm & (1u << k)) {
            any |= lane_mask_any<4>(m0 + mc[k] * mrow, mcol);
            v[k] = C::load(p0 + o[k]);
        }
    }
    float dk[4];
    if (any == 0u) {   // the common case: no padding under any corner
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            dk[k] = dot_chunk(g, v[k]);
            if (cm & (1u << k)) gr.red(gp0 + GS * o[k], aw[k]);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            dk[k] = 0.f;
            if (!(cm & (1u << k))) continue;
            const unsigned bits = lane_mask_bits<4>(m0 + mc[k] * mrow, mcol);
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (bits & (1u << i)) v[k].x[i] = 0.f;
            dk[k] = dot_chunk(g, v[k]);
            if (bits != 0xfu) {
                RedView<VT> gm = gr;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (bits & (1u << i)) gm.x[i] = 0.f;
                gm.red(gp0 + GS * o[k], aw[k]);
            }
        }
    }
    pa = fmaf(b.w0, dk[0], fmaf(b.w1, dk[1], fmaf(b.w2, dk[2], fmaf(b.w3, dk[3], pa))));
    px = fmaf(b.hy, dk[1] - dk[0], fmaf(b.ly, dk[3] - dk[2], px));
    py = fmaf(b.hx, dk[2] - dk[0], fmaf(b.lx, dk[3] - dk[1], py));
}

// No occupancy floor in the launch bounds on purpose: given a register budget ptxas hoists loads
// until it is used up (56 registers + spills at a 6-CTA floor, 64 at 5, 80 at 4) and the kernel gets
// SLOWER -- left alone it needs 40 registers, 8 CTAs per SM fit, and the gather is 10-13 % faster
// (profiles/r01_run21_*): this kernel wants warps in flight, not loads per warp.
template <typename VT, int LANES, int PAIRS, int CSB, int MODE>
__global__ void __launch_bounds__(SnipCfg<LANES, PAIRS>::THREADS)
msda_snippet_fwd_kernel(const typename Chunk<VT>::elem *__restrict__ value, const int64_t *__restrict__ shapes,
                        const int64_t *__restrict__ lsi, const float *__restrict__ offsets,
                        const float *__restrict__ logits, const float *__restrict__ ref,
                        typename Chunk<VT>::elem *__restrict__ out, const SnipArgs a)
{
    using Cfg = SnipCfg<LANES, PAIRS>;
    using C = Chunk<VT>;
    using ET = typename C::elem;
    const SnippetDims &d = a.d;
    __shared__ LevelTable lv;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int LP = d.L * d.P;
    float4 *rec = reinterpret_cast<float4 *>(smem_raw);
    float *zs = reinterpret_cast<float *>(smem_raw + sizeof(float4) * Cfg::PAIRS * (LP + 1));

    const int tid = threadIdx.x;
    const int m = blockIdx.x, q0 = blockIdx.y * Cfg::PAIRS;
    const int n = blockIdx.z / d.T1, t1 = blockIdx.z - n * d.T1;
    int lo, hi;
    frame_range(t1, d.n_frame, d.T2, lo, hi);
    const int nf = hi - lo + 1;
    const size_t qbase = ((size_t)n * d.T1 + t1) * d.Lq;  // first query row of this (n, t1)

    snippet_phase1<Cfg::THREADS, Cfg::PAIRS>(rec, zs, lv, shapes, lsi, a, n, t1, q0, m, qbase, offsets, logits, ref,
                                            1.f / (float)nf);

    // ---- phase 2: gather from every neighbour frame ----
    const int pl = tid / LANES;
    const int lane = tid - pl * LANES;
    if (q0 + pl >= d.Lq) return;
    const int chunk = lane_chunk<VT, LANES>(tid, lane, m);
    const size_t pair = (qbase + q0 + pl) * d.M + m;
    // first frame this query frame gathers from: its slot (presummed) or its first neighbour frame
    const int first = MODE == kPresummed ? (t1 < d.n_frame ? t1 : a.n_local) : lo;
    const char *pf = reinterpret_cast<const char *>(value + n * d.value_stride_n + first * d.value_stride_t) +
                     (size_t)(m * LANES + chunk) * C::BYTES;
    const int64_t fstride = d.value_stride_t * (int64_t)sizeof(ET);  // bytes between frames
    MaskView mv{nullptr, 0, 0, 0, 0.f};
    if (MODE == kDirectMasked) {
        mv.row = d.mask_row_stride;
        mv.frame = (int64_t)d.S * d.mask_row_stride;
        mv.col = d.mask_col_stride;
        mv.inv_cell_bytes = 1.f / (float)a.cell_bytes;
        mv.p = d.mask + ((int64_t)n * d.T2 + lo) * mv.frame + (int64_t)((m * LANES + chunk) * C::N) * mv.col;
    }
    const float4 *rr = rec + pl * (LP + 1);
    C acc = zero_chunk<C>();
    for (int l = 0; l < d.L; ++l) {
        const unsigned row = (unsigned)(lv.W[l] * a.cell_bytes);
        for (int p = 0; p < d.P; ++p) {
            const float4 r = rr[l * d.P + p];
            if (MODE == kPresummed)
                gather_fma<VT, CSB>(acc, record_meta(r, row), record_weights(r), pf, a.cell_bytes);
            else if (MODE == kDirect)
                gather_fma_frames<VT, CSB>(acc, record_meta(r, row), record_weights(r), pf, fstride, nf, a.cell_bytes);
            else
                gather_fma_frames_masked<VT>(acc, record_meta(r, row), record_weights(r), pf, fstride, nf,
                                             a.cell_bytes, lv.W[l], mv);
        }
    }
    acc.store(reinterpret_cast<char *>(out) + (pair * LANES + chunk) * C::BYTES);
}

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

// SCATTER == false (presummed only): grad_offsets / grad_logits alone, no atomics anywhere -- the deterministic
// mode computes grad_value with the two-pass gather of msda_deterministic.cu.
template <typename VT, int LANES, int PAIRS, int CSB, int MODE, bool SCATTER = true>
__global__ void __launch_bounds__(SnipCfg<LANES, PAIRS>::THREADS,
                                  MODE == kPresummed ? SnipCfg<LANES, PAIRS>::BWD_MIN_BLOCKS_PRESUM
                                                     : SnipCfg<LANES, PAIRS>::BWD_MIN_BLOCKS)
msda_snippet_bwd_kernel(const typename Chunk<VT>::elem *__restrict__ value, const int64_t *__restrict__ shapes,
                        const int64_t *__restrict__ lsi, const float *__restrict__ offsets,
                        const float *__restrict__ logits, const float *__restrict__ ref,
                        const typename Chunk<VT>::elem *__restrict__ grad_out, float *__restrict__ grad_value,
                        float *__restrict__ grad_offsets, float *__restrict__ grad_logits,
                        const SnipArgs a)
{
    using Cfg = SnipCfg<LANES, PAIRS>;
    using C = Chunk<VT>;
    using ET = typename C::elem;
    constexpr int GS = 4 / (int)sizeof(ET);
    const SnippetDims &d = a.d;
    __shared__ LevelTable lv;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int LP = d.L * d.P;
    float4 *frac = reinterpret_cast<float4 *>(smem_raw);  // {lx, ly, A, off | mask}
    float *part = reinterpret_cast<float *>(smem_raw + sizeof(float4) * Cfg::PAIRS * (LP + 1));
    float *zs = part;  // phase-1 scratch aliases `part` ([rec][SUBS][3] >= 1 float per record)

    const int tid = threadIdx.x;
    const int m = blockIdx.x, q0 = blockIdx.y * Cfg::PAIRS;
    const int n = blockIdx.z / d.T1, t1 = blockIdx.z - n * d.T1;
    int lo, hi;
    frame_range(t1, d.n_frame, d.T2, lo, hi);
    const int nf = hi - lo + 1;
    const size_t qbase = ((size_t)n * d.T1 + t1) * d.Lq;

    snippet_phase1<Cfg::THREADS, Cfg::PAIRS>(frac, zs, lv, shapes, lsi, a, n, t1, q0, m, qbase, offsets, logits, ref,
                                            1.f / (float)nf);

    // ---- phase 2: every thread participates (full-mask shuffles) ----
    {
        const int pl = tid / LANES;
        const int lane = tid - pl * LANES;
        const int sub = lane / Cfg::SUBG;
        const int chunk = lane_chunk<VT, LANES>(tid, lane, m);
        const bool live = q0 + pl < d.Lq;
        const size_t pair = (qbase + q0 + pl) * d.M + m;
        const int first = MODE == kPresummed ? (t1 < d.n_frame ? t1 : a.n_local) : lo;
        const int gframes = MODE == kPresummed ? a.n_slots : d.T2;  // frames per batch item of grad_value
        const char *pf = reinterpret_cast<const char *>(value + n * d.value_stride_n + first * d.value_stride_t) +
                         (size_t)(m * LANES + chunk) * C::BYTES;
        // grad_value is a dense fp32 (N,T2 | slots,S,M,D) buffer: GS x the value byte offsets
        char *gpf = reinterpret_cast<char *>(grad_value) +
                    (((size_t)n * gframes + first) * d.S * a.cell_bytes + (size_t)m * LANES * C::BYTES) * GS +
                    RedView<VT>::lane_offset(chunk);
        const int64_t mframe = (int64_t)d.S * d.mask_row_stride;
        const uint8_t *mpf = MODE == kDirectMasked
                                 ? d.mask + ((int64_t)n * d.T2 + lo) * mframe + (int64_t)((m * LANES + chunk) * C::N) * d.mask_col_stride
                                 : nullptr;
        C g = zero_chunk<C>();
        if (live) g = C::load(reinterpret_cast<const char *>(grad_out) + (pair * LANES + chunk) * C::BYTES);
        const RedView<VT> gr = RedView<VT>::make(g);
        const int64_t fstride = d.value_stride_t * (int64_t)sizeof(ET);
        const int64_t gfstride = (int64_t)d.S * a.cell_bytes * GS;
        const float4 *ff = frac + pl * (LP + 1);
        float *mypart = part + (size_t)(pl * LP) * (Cfg::SUBS * 3) + sub * 3;
        for (int j = 0; j < LP; ++j) {
            const float4 f = ff[j];
            const int level_w = lv.W[fast_div(j, a.magic_P)];
            const SampleMeta mt = record_meta(f, (unsigned)(level_w * a.cell_bytes));
            const BwdWeights bw = make_bwd_weights(f.x, f.y, f.z);
            float pa = 0.f, px = 0.f, py = 0.f;
            const char *p0 = pf;
            char *gp0 = gpf;
            // (the backward, unlike the forward, prefers loads in flight over occupancy: not unrolling
            //  this loop -- 64 registers, 5 CTAs per SM -- measured 4-7 % slower, profiles/r01_run24_*)
            if (MODE == kPresummed) {
                gather_scatter<VT, CSB, SCATTER>(mt, bw, g, gr, p0, gp0, a.cell_bytes, pa, px, py);
            } else if (MODE == kDirect) {
                for (int fr = 0; fr < nf; ++fr, p0 += fstride, gp0 += gfstride)
                    gather_scatter<VT, CSB, true>(mt, bw, g, gr, p0, gp0, a.cell_bytes, pa, px, py);
            } else {
                const uint8_t *mp = mpf;
                for (int fr = 0; fr < nf; ++fr, p0 += fstride, gp0 += gfstride, mp += mframe)
                    gather_scatter_masked<VT>(mt, bw, g, gr, p0, gp0, a.cell_bytes, level_w, mp, d.mask_row_stride,
                                              d.mask_col_stride, 1.f / (float)a.cell_bytes, pa, px, py);
            }
            subgroup_sum3<Cfg::SUBG>(pa, px, py);
            // zs/es alias `part`: all phase-1 reads finished at the barrier that ends phase 1
            if ((lane & (Cfg::SUBG - 1)) == 0) {
                float *dst = mypart + j * (Cfg::SUBS * 3);
                dst[0] = pa; dst[1] = px; dst[2] = py;
            }
        }
    }
    __syncthreads();

    // ---- phase 3: per-sample finish + softmax backward ----
    // dL/dz_i = A_i * (gA_i - k * sum_j gA_j A_j)   with A = softmax/k, gA_i = <G, val_i> summed over frames
    for (int i = tid; i < Cfg::PAIRS * LP; i += Cfg::THREADS) {
        const float *p = part + (size_t)i * (Cfg::SUBS * 3);
        float pa = 0.f, px = 0.f, py = 0.f;
#pragma unroll
        for (int s = 0; s < Cfg::SUBS; ++s) { pa += p[3 * s]; px += p[3 * s + 1]; py += p[3 * s + 2]; }
        const int spl = fast_div(i, a.magic_LP);
        const float at = frac[i + spl].z;
        if (q0 + spl < d.Lq) {
            // loc = ref + off/(W,H) and x = loc*W - 0.5  =>  dx/doff_x = 1: the W factor of the
            // per-call grad_loc (W*A*px) cancels against the 1/W of the normalisation.
            reinterpret_cast<float2 *>(grad_offsets + (qbase + q0 + spl) * d.off_row_stride)[m * LP + (i - spl * LP)] =
                make_float2(at * px, at * py);
        }
        part[(size_t)i * (Cfg::SUBS * 3)] = pa * at;  // own slots only ([0] = gA_i A_i, [1] = gA_i)
        part[(size_t)i * (Cfg::SUBS * 3) + 1] = pa;
    }
    __syncthreads();
    for (int i = tid; i < Cfg::PAIRS * LP; i += Cfg::THREADS) {
        const int spl = fast_div(i, a.magic_LP);
        if (q0 + spl < d.Lq) {
            float dot = 0.f;
            for (int j = 0; j < LP; ++j) dot += part[(size_t)(spl * LP + j) * (Cfg::SUBS * 3)];
            grad_logits[(qbase + q0 + spl) * d.logit_row_stride + m * LP + (i - spl * LP)] =
                frac[i + spl].z * (part[(size_t)i * (Cfg::SUBS * 3) + 1] - (float)nf * dot);
        }
    }
}

bool snippet_ok(const SnippetDims &d, int esize)
{
    const int epl = 16 / esize;
    if (d.D % epl != 0) return false;
    const int lanes = d.D / epl;
    if (esize == 4 && (lanes % 4 != 0 || lanes > 32)) return false;
    if (esize == 2 && lanes != 2 && lanes != 4 && lanes != 6 && lanes != 8 && lanes != 12 && lanes != 16) return false;
    if (d.L > kMaxLevels || d.L * d.P > kSnippetMaxLP) return false;
    if ((d.value_stride_n * esize) % 16 != 0 || (d.value_stride_t * esize) % 16 != 0) return false;
    if ((int64_t)d.S * d.M * d.D * esize >= ((int64_t)1 << 28)) return false;  // SampleMeta bit budget
    if ((int64_t)d.N * d.T1 > 65535 || (d.Lq + 7) / 8 > 65535) return false;
    return true;
}

bool snippet_ok(const SnippetDims &d) { return snippet_ok(d, 4); }

// queries per CTA tile for D = 48: 16 unless MSDA_SNIP_PAIRS_D48 = 8 | 16 | 32 is set in the environment
// (benchmark knob, read once; every tile length sums each output in the same order)
int snip_pairs_d48()
{
    static const int v = env_tile_pairs("MSDA_SNIP_PAIRS_D48");
    return v;
}


static int snip_mode(const SnippetDims &d) { return d.presummed ? kPresummed : (d.mask ? kDirectMasked : kDirect); }

// Snipper's cell stride (M*D = 384 elements) as an immediate offset
template <typename VT, int LANES>
constexpr int snip_csb() { return (LANES * Chunk<VT>::N == 48) ? 384 * (int)sizeof(typename Chunk<VT>::elem) : 0; }

template <typename VT, int LANES, int PAIRS>
static cudaError_t launch_snip_fwd(const typename Chunk<VT>::elem *value, const int64_t *shapes, const int64_t *lsi,
                                   const float *offsets, const float *logits, const float *ref,
                                   typename Chunk<VT>::elem *out, const SnippetDims &d, cudaStream_t stream)
{
    using Cfg = SnipCfg<LANES, PAIRS>;
    const SnipArgs a = make_snip_args<VT>(d);
    const dim3 grid(d.M, (d.Lq + PAIRS - 1) / PAIRS, d.N * d.T1);
    const size_t smem = sizeof(float4) * Cfg::PAIRS * (d.L * d.P + 1) + sizeof(float) * Cfg::PAIRS * d.L * d.P;
    constexpr int C = snip_csb<VT, LANES>();
    const bool imm = C != 0 && d.M * d.D == 384;
#define MSDA_LAUNCH_FWD(CSB_, MODE_)                                                                   \
    msda_snippet_fwd_kernel<VT, LANES, PAIRS, CSB_, MODE_><<<grid, Cfg::THREADS, smem, stream>>>(     \
        value, shapes, lsi, offsets, logits, ref, out, a)
    switch (snip_mode(d)) {
        case kPresummed:
            if (imm) MSDA_LAUNCH_FWD(C, kPresummed); else MSDA_LAUNCH_FWD(0, kPresummed);
            break;
        case kDirectMasked:   // runtime cell stride only: the masked gather is the few-queries path
            MSDA_LAUNCH_FWD(0, kDirectMasked);
            break;
        default:
            if (imm) MSDA_LAUNCH_FWD(C, kDirect); else MSDA_LAUNCH_FWD(0, kDirect);
    }
#undef MSDA_LAUNCH_FWD
    return cudaGetLastError();
}

template <typename VT, int LANES, int PAIRS, int CSB, int MODE>
static cudaError_t launch_snip_bwd_impl(const typename Chunk<VT>::elem *value, const int64_t *shapes, const int64_t *lsi,
                                        const float *offsets, const float *logits, const float *ref,
                                        const typename Chunk<VT>::elem *grad_out, float *grad_value, float *grad_offsets,
                                        float *grad_logits, const SnippetDims &d, cudaStream_t stream)
{
    using Cfg = SnipCfg<LANES, PAIRS>;
    const SnipArgs a = make_snip_args<VT>(d);
    const dim3 grid(d.M, (d.Lq + PAIRS - 1) / PAIRS, d.N * d.T1);
    const size_t smem = sizeof(float4) * Cfg::PAIRS * (d.L * d.P + 1) + sizeof(float) * 3 * Cfg::SUBS * Cfg::PAIRS * d.L * d.P;
    if (smem > kSmemOptIn) {
        const cudaError_t e = cudaFuncSetAttribute(msda_snippet_bwd_kernel<VT, LANES, PAIRS, CSB, MODE>,
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    msda_snippet_bwd_kernel<VT, LANES, PAIRS, CSB, MODE><<<grid, Cfg::THREADS, smem, stream>>>(
        value, shapes, lsi, offsets, logits, ref, grad_out, grad_value, grad_offsets, grad_logits, a);
    return cudaGetLastError();
}

template <typename VT, int LANES, int PAIRS>
static cudaError_t launch_snip_bwd(const typename Chunk<VT>::elem *value, const int64_t *shapes, const int64_t *lsi,
                                   const float *offsets, const float *logits, const float *ref,
                                   const typename Chunk<VT>::elem *grad_out, float *grad_value, float *grad_offsets,
                                   float *grad_logits, const SnippetDims &d, cudaStream_t stream)
{
    constexpr int C = snip_csb<VT, LANES>();
    const bool imm = C != 0 && d.M * d.D == 384;
#define MSDA_LAUNCH_BWD(CSB_, MODE_)                                                                             \
    launch_snip_bwd_impl<VT, LANES, PAIRS, CSB_, MODE_>(value, shapes, lsi, offsets, logits, ref, grad_out,     \
                                                        grad_value, grad_offsets, grad_logits, d, stream)
    switch (snip_mode(d)) {
        case kPresummed: return imm ? MSDA_LAUNCH_BWD(C, kPresummed) : MSDA_LAUNCH_BWD(0, kPresummed);
        case kDirectMasked: return MSDA_LAUNCH_BWD(0, kDirectMasked);
        default: return imm ? MSDA_LAUNCH_BWD(C, kDirect) : MSDA_LAUNCH_BWD(0, kDirect);
    }
#undef MSDA_LAUNCH_BWD
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

#define MSDA_DISPATCH_LANES(D, CALL)                                  \
    switch ((D) / 4) {                                                \
        case 4: return CALL(float, 4, 16);                            \
        case 8: return CALL(float, 8, 16);                            \
        case 12: {                                                    \
            const int pairs_ = pick_pairs_d48(snip_pairs_d48(), d.Lq, d.M, d.N * d.T1); \
            if (pairs_ == 8) return CALL(float, 12, 8);               \
            if (pairs_ == 32) return CALL(float, 12, 32);             \
            return CALL(float, 12, 16);                               \
        }                                                             \
        case 16: return CALL(float, 16, 16);                          \
        case 20: return CALL(float, 20, 8);                           \
        case 24: return CALL(float, 24, 8);                           \
        case 28: return CALL(float, 28, 8);                           \
        case 32: return CALL(float, 32, 8);                           \
        default: return cudaErrorInvalidValue;                        \
    }

#define MSDA_DISPATCH_LANES_BF16(D, CALL)                             \
    switch ((D) / 8) {                                                \
        case 2: return CALL(__nv_bfloat16, 2, 16);                    \
        case 4: return CALL(__nv_bfloat16, 4, 16);                    \
        case 6: return CALL(__nv_bfloat16, 6, 16);                    \
        case 8: return CALL(__nv_bfloat16, 8, 16);                    \
        case 12: return CALL(__nv_bfloat16, 12, 16);                  \
        case 16: return CALL(__nv_bfloat16, 16, 8);                   \
        default: return cudaErrorInvalidValue;                        \
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

cudaError_t launch_snippet_forward_bf16(const void *value_, const int64_t *shapes,
                                        const int64_t *lsi, const float *offsets,
                                        const float *logits, const float *ref, void *out_,
                                        const SnippetDims &d, cudaStream_t stream)
{
    const __nv_bfloat16 *value = static_cast<const __nv_bfloat16 *>(value_);
    __nv_bfloat16 *out = static_cast<__nv_bfloat16 *>(out_);
    // few CTAs (decoder layers): latency-bound -- 8-byte lanes give twice the threads per query
    if ((long long)((d.Lq + 15) / 16) * d.M * d.N * d.T1 < 148 * 3) {
#define CALL(VT, LN, PR) launch_snip_fwd<bf16q, LN, PR>(value, shapes, lsi, offsets, logits, ref, out, d, stream)
        MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
    }
#define CALL(VT, LN, PR) launch_snip_fwd<VT, LN, PR>(value, shapes, lsi, offsets, logits, ref, out, d, stream)
    MSDA_DISPATCH_LANES_BF16(d.D, CALL)
#undef CALL
}

cudaError_t launch_snippet_backward_bf16(const void *value_, const int64_t *shapes,
                                         const int64_t *lsi, const float *offsets,
                                         const float *logits, const float *ref,
                                         const void *grad_out_, float *grad_value,
                                         float *grad_offsets, float *grad_logits,
                                         const SnippetDims &d, cudaStream_t stream)
{
    const __nv_bfloat16 *value = static_cast<const __nv_bfloat16 *>(value_);
    const __nv_bfloat16 *grad_out = static_cast<const __nv_bfloat16 *>(grad_out_);
    // backward lanes are 8 bytes = 4 channels (bf16q): same lane count and reduction pattern as fp32
#define CALL(VT, LN, PR) \
    launch_snip_bwd<bf16q, LN, PR>(value, shapes, lsi, offsets, logits, ref, grad_out, grad_value, grad_offsets, grad_logits, d, stream)
    MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
}

}  // namespace msda
