// Kernels and launchers of the fast per-call path (see msda_percall.cu), shared by libmsda_b200.so (fp32 and bf16
// lanes) and libmsda_b200_f16.so (fp16 lanes, csrc_f16/): each library instantiates the templates for its own lane
// types.
#pragma once

#include "msda_fast.cuh"
#include "msda_internal.h"

namespace msda {

// ------------------------------------------------------------------------------------------
// FAST path (see msda_fast.cuh for the CTA organisation).  VT = element type of value / output /
// grad_output (float or __nv_bfloat16); loc / attn / grad_loc / grad_attn / grad_value are fp32.
// ------------------------------------------------------------------------------------------
// grid = (M, query tiles, N): a CTA owns PAIRS consecutive queries of ONE head.  Consecutive
// queries are neighbouring pixels in the encoder, so the cells they gather overlap and hit in L1.
template <int LANES, int PAIRS_>
struct FastCfg {
    static constexpr int PAIRS = PAIRS_;
    static constexpr int THREADS = PAIRS * LANES;
    static constexpr int SUBG = sub_group(LANES);                          // lanes per shuffle group
    static constexpr int SUBS = LANES / SUBG;                              // shuffle groups per pair
    static constexpr int CHUNK = (512 / PAIRS) < 32 ? (512 / PAIRS) : 32;  // samples per query per pass
    static_assert(LANES % 2 == 0 && THREADS % 32 == 0 && THREADS <= 1024, "lane groups must tile warps");
};

struct FastArgs {
    int M, L, P, Lq, S;
    int cell_bytes;            // M * D * sizeof(VT): bytes between consecutive cells of `value`
    int cl;                    // samples per query per pass (<= CHUNK)
    unsigned magic_cl, magic_P;
    int64_t value_batch_stride;  // elements
};

// No occupancy floor in the launch bounds: left alone ptxas needs 40 registers (8 CTAs of 192 threads per
// SM).  Variants that trade occupancy for loads in flight (two samples per step at 64 registers, a
// 32-register build) measured equal or slower once the chunk rotation was in (profiles/r01_run9_*,
// r01_run22_*).
template <typename VT, int LANES, int PAIRS, int CSB>
__global__ void __launch_bounds__(FastCfg<LANES, PAIRS>::THREADS)
msda_fwd_fast_kernel(const typename Chunk<VT>::elem *__restrict__ value, const int64_t *__restrict__ shapes,
                     const int64_t *__restrict__ lsi, const float *__restrict__ loc,
                     const float *__restrict__ attn, typename Chunk<VT>::elem *__restrict__ out, const FastArgs a)
{
    using Cfg = FastCfg<LANES, PAIRS>;
    using C = Chunk<VT>;
    using ET = typename C::elem;
    __shared__ LevelTable lv;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4 *rec = reinterpret_cast<float4 *>(smem_raw);  // {lx, ly, A, off | mask}, stride cl + 1 per query

    const int tid = threadIdx.x;
    const int m = blockIdx.x, q0 = blockIdx.y * Cfg::PAIRS, nb = blockIdx.z;
    const int LP = a.L * a.P;

    load_level_table(lv, shapes, lsi, a.L, a.S);
    __syncthreads();

    const int pl = tid / LANES;
    const int lane = tid - pl * LANES;
    const bool live = q0 + pl < a.Lq;
    const int chunk = lane_chunk<VT, LANES>(tid, lane, m);
    const size_t pair = ((size_t)nb * a.Lq + q0 + pl) * a.M + m;
    const char *p0 = reinterpret_cast<const char *>(value + (int64_t)nb * a.value_batch_stride) +
                     (size_t)(m * LANES + chunk) * C::BYTES;
    C acc = zero_chunk<C>();

    for (int lp0 = 0; lp0 < LP; lp0 += a.cl) {
        const int n = min(a.cl, LP - lp0);
        const unsigned magic_n = n == a.cl ? a.magic_cl : fast_magic_dev(n);
        // ---- phase 1: one thread per sample ----
        for (int i = tid; i < Cfg::PAIRS * n; i += Cfg::THREADS) {
            const int spl = fast_div(i, magic_n);
            const int lp = lp0 + (i - spl * n);
            float4 r = empty_record();
            if (q0 + spl < a.Lq) {
                const size_t si = (((size_t)nb * a.Lq + q0 + spl) * a.M + m) * LP + lp;
                const float2 uv = __ldg(reinterpret_cast<const float2 *>(loc) + si);
                const int l = fast_div(lp, a.magic_P);
                const Sample<float> s = make_sample<float>(uv.x, uv.y, lv.H[l], lv.W[l], lv.start[l]);
                r = make_record(s, __ldg(attn + si), a.cell_bytes);
            }
            rec[i + spl] = r;
        }
        __syncthreads();
        // ---- phase 2: gather ----
        if (live) {
            const float4 *rr = rec + pl * (n + 1);
            // fp32 lanes: unroll 2 = 40 registers / 8 CTAs per SM (unroll 4 takes 54 and loses two resident
            // CTAs: 3 % slower at N = 8); the bf16 lane types measured better with 4 (profiles/r01_run44_*)
#pragma unroll (sizeof(ET) == 4 ? 2 : 4)
            for (int j = 0; j < n; ++j) {
                const float4 r = rr[j];
                const unsigned row = (unsigned)(lv.W[fast_div(lp0 + j, a.magic_P)] * a.cell_bytes);
                gather_fma<VT, CSB>(acc, record_meta(r, row), record_weights(r), p0, a.cell_bytes);
            }
        }
        if (lp0 + a.cl < LP) __syncthreads();  // staging buffers are reused by the next pass
    }
    if (live) acc.store(reinterpret_cast<char *>(out) + (pair * LANES + chunk) * C::BYTES);
}

// Few-queries forward (decoder-sized Lq): with 8 or 16 queries per CTA such a launch is a handful of CTAs whose
// lanes walk the L*P samples one after the other -- a chain of dependent round trips to L2 / HBM that the reference's
// thread-per-output-element kernel does not have (cold L2: 24.6 us against its 19.5 us,
// profiles/r02_run9_opbench_l2_flushed.jsonl).  Here ONE (query, head) pair owns a CTA and thread = (sample, 16-byte
// chunk): the location / weight loads are one round trip, the four corner loads a second, and the L*P partial sums
// meet in shared memory (summed in a fixed order).
template <typename VT, int LANES, int BLOCK>   // VT = float (16-byte lanes) or bf16q / halfq (8-byte lanes): 4 channels per lane
__global__ void __launch_bounds__(BLOCK)
msda_fwd_split_kernel(const typename Chunk<VT>::elem *__restrict__ value, const int64_t *__restrict__ shapes,
                      const int64_t *__restrict__ lsi, const float *__restrict__ loc, const float *__restrict__ attn,
                      typename Chunk<VT>::elem *__restrict__ out, const FastArgs a)
{
    using C = Chunk<VT>;
    static_assert(C::N == 4, "one float4 of partial sums per lane");
    __shared__ LevelTable lv;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4 *red = reinterpret_cast<float4 *>(smem_raw);   // [sample][chunk]
    const int tid = threadIdx.x;
    const int m = blockIdx.x, q = blockIdx.y, nb = blockIdx.z;
    const int LP = a.L * a.P;
    constexpr int SLOTS = BLOCK / LANES;          // samples in flight per pass; thread = (slot, chunk)
    const int sidx = tid / LANES, lane = tid - sidx * LANES;
    const size_t pair = ((size_t)nb * a.Lq + q) * a.M + m;
    // issued before the level table is staged: the first sample's own loads do not depend on it
    float2 uv = make_float2(0.f, 0.f);
    float at = 0.f;
    if (sidx < LP && sidx < SLOTS) {
        uv = __ldg(reinterpret_cast<const float2 *>(loc) + pair * LP + sidx);
        at = __ldg(attn + pair * LP + sidx);
    }
    load_level_table(lv, shapes, lsi, a.L, a.S);
    __syncthreads();
    if (sidx < SLOTS) {
        const char *p0 = reinterpret_cast<const char *>(value + (int64_t)nb * a.value_batch_stride) +
                         (size_t)(m * LANES + lane) * C::BYTES;
        C acc = zero_chunk<C>();
        for (int sp = sidx; sp < LP; sp += SLOTS) {   // more than SLOTS samples (frames presented as levels): a few passes
            if (sp != sidx) {
                uv = __ldg(reinterpret_cast<const float2 *>(loc) + pair * LP + sp);
                at = __ldg(attn + pair * LP + sp);
            }
            const int l = fast_div(sp, a.magic_P);
            const Sample<float> s = make_sample<float>(uv.x, uv.y, lv.H[l], lv.W[l], lv.start[l]);
            const float4 r = make_record(s, at, a.cell_bytes);
            gather_fma<VT, 0>(acc, record_meta(r, (unsigned)(lv.W[l] * a.cell_bytes)), record_weights(r), p0, a.cell_bytes);
        }
        red[sidx * LANES + lane] = make_float4(acc.x[0], acc.x[1], acc.x[2], acc.x[3]);
    }
    __syncthreads();
    if (tid < LANES) {
        float4 sum = red[tid];
        const int used = LP < SLOTS ? LP : SLOTS;
        for (int j = 1; j < used; ++j) {
            const float4 v = red[j * LANES + tid];
            sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
        }
        C o;
        o.x[0] = sum.x; o.x[1] = sum.y; o.x[2] = sum.z; o.x[3] = sum.w;
        o.store(reinterpret_cast<char *>(out) + (pair * LANES + tid) * C::BYTES);
    }
}

// few queries (decoder-sized launches): one CTA per (query, head), samples spread over the threads
// (MSDA_FWD_SPLIT=0 in the environment keeps the tile kernel: benchmark knob, read once)
template <typename VT>
static bool launch_fwd_split(const typename Chunk<VT>::elem *value, const int64_t *shapes, const int64_t *lsi,
                             const float *loc, const float *attn, typename Chunk<VT>::elem *out, const OpDims &d,
                             cudaStream_t stream)
{
    static const bool split_on = [] { const char *e = getenv("MSDA_FWD_SPLIT"); return !(e && e[0] == '0'); }();
    if (!(split_on && d.D == 48 && d.L * d.P <= (1 << 20) && d.Lq <= 65535 && d.N <= 65535 &&
          (long long)((d.Lq + 15) / 16) * d.M * d.N < 148 * 3))
        return false;
    FastArgs a;
    a.M = d.M; a.L = d.L; a.P = d.P; a.Lq = d.Lq; a.S = d.S;
    a.cell_bytes = d.M * d.D * (int)sizeof(typename Chunk<VT>::elem);
    a.cl = d.L * d.P;
    a.magic_cl = fast_magic(a.cl);
    a.magic_P = fast_magic(d.P);
    a.value_batch_stride = d.value_batch_stride;
    const dim3 grid(d.M, d.Lq, d.N);
    const size_t smem = sizeof(float4) * 32 * 12;   // one partial sum per (sample slot, chunk)
    if (d.L * d.P * 12 <= 160)
        msda_fwd_split_kernel<VT, 12, 160><<<grid, 160, smem, stream>>>(value, shapes, lsi, loc, attn, out, a);
    else
        msda_fwd_split_kernel<VT, 12, 384><<<grid, 384, smem, stream>>>(value, shapes, lsi, loc, attn, out, a);
    return true;
}

// SCATTER == false: grad_sampling_loc / grad_attn_weight only (deterministic mode computes
// grad_value separately, msda_deterministic.cu).  grad_value is fp32 for every VT.
template <typename VT, int LANES, int PAIRS, int CSB, bool SCATTER>
__global__ void __launch_bounds__(FastCfg<LANES, PAIRS>::THREADS)
msda_bwd_fast_kernel(const typename Chunk<VT>::elem *__restrict__ value, const int64_t *__restrict__ shapes,
                     const int64_t *__restrict__ lsi, const float *__restrict__ loc,
                     const float *__restrict__ attn, const typename Chunk<VT>::elem *__restrict__ grad_out,
                     float *__restrict__ grad_value, float *__restrict__ grad_loc,
                     float *__restrict__ grad_attn, const FastArgs a)
{
    using Cfg = FastCfg<LANES, PAIRS>;
    using C = Chunk<VT>;
    using ET = typename C::elem;
    constexpr int GS = 4 / (int)sizeof(ET);
    __shared__ LevelTable lv;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4 *frac = reinterpret_cast<float4 *>(smem_raw);  // {lx, ly, A, off | mask}, stride cl + 1 per query
    float *part = reinterpret_cast<float *>(smem_raw + sizeof(float4) * Cfg::PAIRS * (a.cl + 1));

    const int tid = threadIdx.x;
    const int m = blockIdx.x, q0 = blockIdx.y * Cfg::PAIRS, nb = blockIdx.z;
    const int LP = a.L * a.P;

    load_level_table(lv, shapes, lsi, a.L, a.S);
    __syncthreads();

    const int pl = tid / LANES;
    const int lane = tid - pl * LANES;
    const int sub = lane / Cfg::SUBG;
    const int chunk = lane_chunk<VT, LANES>(tid, lane, m);
    const bool live = q0 + pl < a.Lq;
    const size_t pair = ((size_t)nb * a.Lq + q0 + pl) * a.M + m;
    const char *p0 = reinterpret_cast<const char *>(value + (int64_t)nb * a.value_batch_stride) +
                     (size_t)(m * LANES + chunk) * C::BYTES;
    char *gp0 = reinterpret_cast<char *>(grad_value) + ((size_t)nb * a.S * a.cell_bytes + (size_t)m * LANES * C::BYTES) * GS +
                RedView<VT>::lane_offset(chunk);
    C g = zero_chunk<C>();
    if (live) g = C::load(reinterpret_cast<const char *>(grad_out) + (pair * LANES + chunk) * C::BYTES);
    const RedView<VT> gr = RedView<VT>::make(g);

    for (int lp0 = 0; lp0 < LP; lp0 += a.cl) {
        const int n = min(a.cl, LP - lp0);
        const unsigned magic_n = n == a.cl ? a.magic_cl : fast_magic_dev(n);
        // ---- phase 1: one thread per sample ----
        for (int i = tid; i < Cfg::PAIRS * n; i += Cfg::THREADS) {
            const int spl = fast_div(i, magic_n);
            const int lp = lp0 + (i - spl * n);
            float4 f = empty_record();
            if (q0 + spl < a.Lq) {
                const size_t si = (((size_t)nb * a.Lq + q0 + spl) * a.M + m) * LP + lp;
                const float2 uv = __ldg(reinterpret_cast<const float2 *>(loc) + si);
                const int l = fast_div(lp, a.magic_P);
                const Sample<float> s = make_sample<float>(uv.x, uv.y, lv.H[l], lv.W[l], lv.start[l]);
                f = make_record(s, __ldg(attn + si), a.cell_bytes);
            }
            frac[i + spl] = f;
        }
        __syncthreads();
        // ---- phase 2: gather + scatter; every thread runs it (full-mask shuffles) ----
        {
            const float4 *ff = frac + pl * (n + 1);
            float *mypart = part + (size_t)(pl * n) * (Cfg::SUBS * 3) + sub * 3;
#pragma unroll 2
            for (int j = 0; j < n; ++j) {
                const float4 f = ff[j];
                const SampleMeta mt = record_meta(f, (unsigned)(lv.W[fast_div(lp0 + j, a.magic_P)] * a.cell_bytes));
                const BwdWeights bw = make_bwd_weights(f.x, f.y, f.z);
                float pa = 0.f, px = 0.f, py = 0.f;
                gather_scatter<VT, CSB, SCATTER>(mt, bw, g, gr, p0, gp0, a.cell_bytes, pa, px, py);
                subgroup_sum3<Cfg::SUBG>(pa, px, py);
                if ((lane & (Cfg::SUBG - 1)) == 0) {
                    float *dst = mypart + j * (Cfg::SUBS * 3);
                    dst[0] = pa; dst[1] = px; dst[2] = py;
                }
            }
        }
        __syncthreads();
        // ---- phase 3: one thread per sample finishes grad_attn / grad_loc ----
        for (int i = tid; i < Cfg::PAIRS * n; i += Cfg::THREADS) {
            const int spl = fast_div(i, magic_n);
            const int lp = lp0 + (i - spl * n);
            if (q0 + spl < a.Lq) {
                const float *p = part + (size_t)i * (Cfg::SUBS * 3);
                float pa = 0.f, px = 0.f, py = 0.f;
#pragma unroll
                for (int s = 0; s < Cfg::SUBS; ++s) { pa += p[3 * s]; px += p[3 * s + 1]; py += p[3 * s + 2]; }
                const float at = frac[i + spl].z;
                const int l = fast_div(lp, a.magic_P);
                const size_t si = (((size_t)nb * a.Lq + q0 + spl) * a.M + m) * LP + lp;
                grad_attn[si] = pa;
                reinterpret_cast<float2 *>(grad_loc)[si] =
                    make_float2((float)lv.W[l] * at * px, (float)lv.H[l] * at * py);
            }
        }
        if (lp0 + a.cl < LP) __syncthreads();
    }
}

// queries per CTA tile for LANES == 12: 16 unless MSDA_PAIRS_D48 = 8 | 16 | 32 is set in the environment
// (benchmark knob, read once; every tile length sums each output in the same order)
static int pairs_d48()
{
    static const int v = env_tile_pairs("MSDA_PAIRS_D48");
    return v;
}

template <typename VT, int LANES, int PAIRS>
static FastArgs make_fast_args(const OpDims &d)  // VT = lane type (float, __nv_bfloat16, bf16q, __half, halfq)
{
    using Cfg = FastCfg<LANES, PAIRS>;
    const int LP = d.L * d.P;
    FastArgs a;
    a.M = d.M; a.L = d.L; a.P = d.P; a.Lq = d.Lq; a.S = d.S;
    a.cell_bytes = d.M * d.D * (int)sizeof(typename Chunk<VT>::elem);
    a.cl = LP < Cfg::CHUNK ? LP : Cfg::CHUNK;
    a.magic_cl = fast_magic(a.cl);
    a.magic_P = fast_magic(d.P);
    a.value_batch_stride = d.value_batch_stride;
    return a;
}

// Snipper's cell stride (M*D = 384 elements) becomes an immediate offset in the gather
template <typename VT, int LANES>
constexpr int snipper_csb() { return (LANES * Chunk<VT>::N == 48) ? 384 * (int)sizeof(typename Chunk<VT>::elem) : 0; }

template <typename VT, int LANES, int PAIRS>
static cudaError_t launch_fwd_fast(const typename Chunk<VT>::elem *value, const int64_t *shapes, const int64_t *lsi,
                                   const float *loc, const float *attn, typename Chunk<VT>::elem *out,
                                   const OpDims &d, cudaStream_t stream)
{
    using Cfg = FastCfg<LANES, PAIRS>;
    const FastArgs a = make_fast_args<VT, LANES, PAIRS>(d);
    const dim3 grid(d.M, (d.Lq + PAIRS - 1) / PAIRS, d.N);
    const size_t smem = sizeof(float4) * Cfg::PAIRS * (a.cl + 1);
    constexpr int C = snipper_csb<VT, LANES>();
    if (C != 0 && d.M * d.D == 384)
        msda_fwd_fast_kernel<VT, LANES, PAIRS, C><<<grid, Cfg::THREADS, smem, stream>>>(value, shapes, lsi, loc, attn, out, a);
    else
        msda_fwd_fast_kernel<VT, LANES, PAIRS, 0><<<grid, Cfg::THREADS, smem, stream>>>(value, shapes, lsi, loc, attn, out, a);
    return cudaGetLastError();
}

template <typename VT, int LANES, int PAIRS, bool SCATTER = true>
static cudaError_t launch_bwd_fast(const typename Chunk<VT>::elem *value, const int64_t *shapes, const int64_t *lsi,
                                   const float *loc, const float *attn, const typename Chunk<VT>::elem *grad_out,
                                   float *grad_value, float *grad_loc, float *grad_attn,
                                   const OpDims &d, cudaStream_t stream)
{
    using Cfg = FastCfg<LANES, PAIRS>;
    const FastArgs a = make_fast_args<VT, LANES, PAIRS>(d);
    const dim3 grid(d.M, (d.Lq + PAIRS - 1) / PAIRS, d.N);
    const size_t smem = sizeof(float4) * Cfg::PAIRS * (a.cl + 1) + sizeof(float) * 3 * Cfg::SUBS * Cfg::PAIRS * a.cl;
    constexpr int C = snipper_csb<VT, LANES>();
    if (C != 0 && d.M * d.D == 384) {
        msda_bwd_fast_kernel<VT, LANES, PAIRS, C, SCATTER><<<grid, Cfg::THREADS, smem, stream>>>(
            value, shapes, lsi, loc, attn, grad_out, grad_value, grad_loc, grad_attn, a);
    } else {
        if (smem > kSmemOptIn) {  // wide heads x many samples per pass (D = 128, L*P = 32: 57.6 KB)
            const cudaError_t e = cudaFuncSetAttribute(msda_bwd_fast_kernel<VT, LANES, PAIRS, 0, SCATTER>,
                                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        msda_bwd_fast_kernel<VT, LANES, PAIRS, 0, SCATTER><<<grid, Cfg::THREADS, smem, stream>>>(
            value, shapes, lsi, loc, attn, grad_out, grad_value, grad_loc, grad_attn, a);
    }
    return cudaGetLastError();
}

// fp32: LANES = D/4 in {4,...,32}; Snipper's D = 48 (12 lanes) has a tunable tile length
#define MSDA_DISPATCH_LANES(D, CALL)                                  \
    switch ((D) / 4) {                                                \
        case 4: return CALL(float, 4, 16);                            \
        case 8: return CALL(float, 8, 16);                            \
        case 12: {                                                    \
            const int pairs_ = pick_pairs_d48(pairs_d48(), d.Lq, d.M, d.N); \
            if (pairs_ == 8) return CALL(float, 12, 8);               \
            if (pairs_ == 32) return CALL(float, 12, 32);             \
            return CALL(float, 12, 16);                               \
        }                                                             \
        case 16: return CALL(float, 16, 16);                          \
        case 20: return CALL(float, 20, 16);                          \
        case 24: return CALL(float, 24, 16);                          \
        case 28: return CALL(float, 28, 16);                          \
        case 32: return CALL(float, 32, 16);                          \
        default: return cudaErrorInvalidValue;                        \
    }

// 16-bit: LANES = D/8 lanes of type H16 (the template parameter of the launcher it expands in); 16 queries x 6 lanes
// = 96 threads for Snipper's D = 48
#define MSDA_DISPATCH_LANES_HALF(D, CALL)                             \
    switch ((D) / 8) {                                                \
        case 2: return CALL(H16, 2, 16);                              \
        case 4: return CALL(H16, 4, 16);                              \
        case 6: return CALL(H16, 6, 16);                              \
        case 8: return CALL(H16, 8, 16);                              \
        case 12: return CALL(H16, 12, 16);                            \
        case 16: return CALL(H16, 16, 16);                            \
        default: return cudaErrorInvalidValue;                        \
    }

// 16-bit storage (bf16 or fp16): H16 is the 16-byte lane of 8 channels (__nv_bfloat16 / __half), H8 the 8-byte lane of
// 4 channels (bf16q / halfq).  value / output / grad_output are 16-bit, everything else fp32.
template <typename H16, typename H8>
cudaError_t launch_forward_fast_half(const void *value_, const int64_t *shapes, const int64_t *lsi,
                                     const float *loc, const float *attn, void *out_,
                                     const OpDims &d, cudaStream_t stream)
{
    using ET = typename Chunk<H16>::elem;
    if (d.N * d.Lq * d.M == 0) return cudaSuccess;
    const ET *value = static_cast<const ET *>(value_);
    ET *out = static_cast<ET *>(out_);
    if (launch_fwd_split<H8>(value, shapes, lsi, loc, attn, out, d, stream)) return cudaGetLastError();
    // few CTAs (decoder-sized Lq): latency-bound -- 8-byte lanes give twice the threads per query
    // (measured 20-45 % faster there, profiles/r01_run14_*); large grids keep the 16-byte lanes.
    if ((long long)((d.Lq + 15) / 16) * d.M * d.N < 148 * 3) {
#define CALL(VT, LN, PR) launch_fwd_fast<H8, LN, PR>(value, shapes, lsi, loc, attn, out, d, stream)
        MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
    }
#define CALL(VT, LN, PR) launch_fwd_fast<VT, LN, PR>(value, shapes, lsi, loc, attn, out, d, stream)
    MSDA_DISPATCH_LANES_HALF(d.D, CALL)
#undef CALL
}

template <typename H16, typename H8>
cudaError_t launch_backward_fast_half(const void *value_, const int64_t *shapes, const int64_t *lsi,
                                      const float *loc, const float *attn, const void *grad_out_,
                                      float *grad_value, float *grad_loc, float *grad_attn,
                                      const OpDims &d, cudaStream_t stream)
{
    using ET = typename Chunk<H16>::elem;
    if (d.N * d.Lq * d.M == 0) return cudaSuccess;
    const ET *value = static_cast<const ET *>(value_);
    const ET *grad_out = static_cast<const ET *>(grad_out_);
    // backward lanes are 8 bytes = 4 channels (H8): same lane count and reduction pattern as fp32
#define CALL(VT, LN, PR) \
    launch_bwd_fast<H8, LN, PR>(value, shapes, lsi, loc, attn, grad_out, grad_value, grad_loc, grad_attn, d, stream)
    MSDA_DISPATCH_LANES(d.D, CALL)
#undef CALL
}

}  // namespace msda
