// Planar neighbour-frame slots (opt-in, MSDA_FLAG_PLANAR): the encoder's gather / scatter with every L1 wavefront a full
// 128-byte line (sm_100a, fp32, D = 48).
//
// In the reference layout (.., S, M, D) a head's 48 fp32 channels are a 192-byte slice at a 64-byte-aligned offset of a
// 1536-byte cell: every corner costs two L1 wavefronts that carry 192 of 256 bytes, and 12 lanes per query leave the
// quarter warps straddling queries (measured 2.1 wavefronts per corner, 8.4 per sample).  The gather cannot choose the
// layout of `value` -- but the pre-summed slots (msda_frames.cu: sum over neighbour frames, taken before the gather by
// linearity) are a buffer of OUR OWN, written once per layer by a streaming pass.  So that pass can write them PLANAR,
// per (n, slot):
//
//   plane A   [m][s]    channels  0..31 of head m at pixel s: one 128-byte line per cell
//   plane Be  [m][s]    channels 32..47, 64-byte cells: x-adjacent cells (s, s+1) share a line when s is even
//   plane Bo  [m][s+1]  the same data shifted by one cell: (s, s+1) share a line when s is odd
//
// and a query is served by ONE QUARTER WARP (8 lanes): per sample 4 x LDG.128 on plane A (one line each) and
// 2 x LDG.128 on plane B (lanes 0-3 the (y,x0) cell, lanes 4-7 the (y,x0+1) cell of row y0 / y0+1, from whichever copy
// has the pair line-aligned) -- 6 wavefronts per sample, every one a full line.  The backward scatters the same way
// (6 full-line vector reductions per sample) into planar fp32 slots that msda_frame_unsum_planar folds back into
// grad_value (N,T2,S,M,D).  Cost: the slots take 4/3 of the bytes (Be and Bo hold the same 16 channels).
//
// MEASURED (DESIGN.md section 3, profiles/r02_run6_* .. r02_run8_*): 20 % fewer global-load wavefronts and, with the
// quarter-warp-local set-up below, 30 % fewer instructions than the cell-major kernels -- at the SAME speed (166 vs
// 164 us per encoder layer): both layouts run at the rate of the L1 global-load path, which does not depend on line
// utilisation.  Hence opt-in, not the default.  The layout is kept because a window of a planar slot is a set of
// contiguous row segments, which is what a shared-memory staged gather needs.
//
// Pad cells (Bo cell 0 of each head, the tail of each B plane) are never read with a live lane and never written by
// the scatter: a pair is only loaded / reduced as a whole when all four corners of the sample are inside the level
// (then s and s+1 are pixels of one row); border samples take the per-corner predicated path.
//
// Math and operation order per sample are those of msda_snippet.cu; the softmax denominator and the sums over
// channels / corners inside one output element are taken in a different order, as between any two lane mappings.
#include "msda_snippet_common.cuh"

namespace msda {

namespace {

constexpr int kALanes = 8;          // 16-byte chunks of a cell in plane A
constexpr int kBLanes = 4;          // 16-byte chunks of a cell in plane B

struct PlanarGeom {
    int S, M, SB;                   // SB = cells per head in each B plane (S + pad, even)
    int a_head, b_head;             // bytes of one head's plane A / plane B
    int a_bytes, b_bytes;           // bytes of plane A / of ONE B plane, all heads
    int slot_bytes;                 // a_bytes + 2 * b_bytes
    int odd_delta;                  // from a Be cell address to the same pair in Bo: b_bytes + 64
};

PlanarGeom make_geom(int S, int M)
{
    PlanarGeom g;
    g.S = S; g.M = M;
    g.SB = (S + 3) & ~1;
    g.a_head = S * 128;
    g.b_head = g.SB * 64;
    g.a_bytes = M * g.a_head;
    g.b_bytes = M * g.b_head;
    g.slot_bytes = g.a_bytes + 2 * g.b_bytes;
    g.odd_delta = g.b_bytes + 64;
    return g;
}

__device__ __forceinline__ float4 ld16(const char *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }

__device__ __forceinline__ void red16(char *p, float a, const float4 &g)
{
    red_add_v4(reinterpret_cast<float *>(p), a * g.x, a * g.y, a * g.z, a * g.w);
}

// ------------------------------------------------------------------------------------------
// streaming passes: value (N,T2,S,M,D) -> planar slots, planar fp32 gradient slots -> grad_value
// ------------------------------------------------------------------------------------------
constexpr int kMaxRegFrames = 8;

struct PlanarFrameArgs {
    int N, T2, T1, n_frame, S, M;
    int n_local, has_all, NS;
    int64_t value_stride_n, value_stride_t;   // elements
    int64_t mask_row_stride;
    int mask_col_stride;
    int64_t total;                            // N * S * M * 12 threads
};

__device__ __forceinline__ unsigned mask_bits4(const uint8_t *__restrict__ mp, int col_stride)
{
    if (col_stride == 0) return __ldg(mp) ? 0xfu : 0u;
    const unsigned mk = __ldg(reinterpret_cast<const unsigned *>(mp));
    return ((mk & 0xffu) ? 1u : 0u) | ((mk & 0xff00u) ? 2u : 0u) | ((mk & 0xff0000u) ? 4u : 0u) | ((mk & 0xff000000u) ? 8u : 0u);
}

__device__ __forceinline__ void slot_range(int j, const PlanarFrameArgs &a, int &lo, int &hi)
{
    if (j < a.n_local) { lo = max(j - 1, 0); hi = min(j + 1, a.n_frame - 1); }
    else { lo = 0; hi = a.T2 - 1; }
}

// one thread per 16-byte chunk of a (n, s) row of value: every source frame is read once (coalesced), every slot is
// written as whole 128-byte (plane A) / 64-byte (planes Be, Bo) segments
__global__ void __launch_bounds__(256)
frame_sum_planar_kernel(const float *__restrict__ value, const uint8_t *__restrict__ mask, char *__restrict__ vsum,
                        const PlanarFrameArgs a, const PlanarGeom g)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.total) return;
    const int cpr = a.M * 12;
    const int64_t row = i / cpr;
    const int c = (int)(i - row * cpr);
    const int m = c / 12, k = c - m * 12;
    const int n = (int)(row / a.S);
    const int s = (int)(row - (int64_t)n * a.S);
    const float *vp = value + n * a.value_stride_n + (int64_t)s * (a.M * kPlanarD) + 4 * c;
    const uint8_t *mp = mask ? mask + ((int64_t)n * a.T2 * a.S + s) * a.mask_row_stride + (int64_t)(4 * c) * a.mask_col_stride
                             : nullptr;
    const int64_t mask_frame = (int64_t)a.S * a.mask_row_stride;
    char *op = vsum + (int64_t)n * a.NS * g.slot_bytes;
    int o0, o1 = -1;     // byte offsets inside a slot (o1: the shifted copy of a plane-B chunk)
    if (k < kALanes) {
        o0 = m * g.a_head + s * 128 + 16 * k;
    } else {
        o0 = g.a_bytes + m * g.b_head + s * 64 + 16 * (k - kALanes);
        o1 = o0 + g.odd_delta;
    }

    auto load_frame = [&](int t) {
        float4 v = __ldg(reinterpret_cast<const float4 *>(vp + t * a.value_stride_t));
        if (mp != nullptr) {
            const unsigned bits = mask_bits4(mp + t * mask_frame, a.mask_col_stride);
            if (bits & 1u) v.x = 0.f;
            if (bits & 2u) v.y = 0.f;
            if (bits & 4u) v.z = 0.f;
            if (bits & 8u) v.w = 0.f;
        }
        return v;
    };
    auto add = [](float4 &acc, const float4 &v) { acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; };
    auto store = [&](int j, const float4 &v) {
        char *sp = op + (int64_t)j * g.slot_bytes;
        *reinterpret_cast<float4 *>(sp + o0) = v;
        if (o1 >= 0) *reinterpret_cast<float4 *>(sp + o1) = v;
    };

    if (a.T2 <= kMaxRegFrames) {
        float4 f[kMaxRegFrames];
#pragma unroll
        for (int t = 0; t < kMaxRegFrames; ++t)
            if (t < a.T2) f[t] = load_frame(t);
        for (int j = 0; j < a.NS; ++j) {
            int lo, hi;
            slot_range(j, a, lo, hi);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int t = 0; t < kMaxRegFrames; ++t)
                if (t >= lo && t <= hi) add(acc, f[t]);   // ascending frame order, as frame_sum_kernel
            store(j, acc);
        }
    } else {
        for (int j = 0; j < a.NS; ++j) {
            int lo, hi;
            slot_range(j, a, lo, hi);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int t = lo; t <= hi; ++t) add(acc, load_frame(t));
            store(j, acc);
        }
    }
}

__global__ void __launch_bounds__(256)
frame_unsum_planar_kernel(const char *__restrict__ gsum, const uint8_t *__restrict__ mask, float *__restrict__ grad_value,
                          const PlanarFrameArgs a, const PlanarGeom g)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.total) return;
    const int cpr = a.M * 12;
    const int64_t row = i / cpr;
    const int c = (int)(i - row * cpr);
    const int m = c / 12, k = c - m * 12;
    const int n = (int)(row / a.S);
    const int s = (int)(row - (int64_t)n * a.S);
    const int64_t frame = (int64_t)a.S * a.M * kPlanarD;
    float *op = grad_value + ((int64_t)n * a.T2 * a.S + s) * (a.M * kPlanarD) + 4 * c;
    const uint8_t *mp = mask ? mask + ((int64_t)n * a.T2 * a.S + s) * a.mask_row_stride + (int64_t)(4 * c) * a.mask_col_stride
                             : nullptr;
    const int64_t mask_frame = (int64_t)a.S * a.mask_row_stride;
    const char *gp = gsum + (int64_t)n * a.NS * g.slot_bytes;
    int o0, o1 = -1;
    if (k < kALanes) {
        o0 = m * g.a_head + s * 128 + 16 * k;
    } else {
        o0 = g.a_bytes + m * g.b_head + s * 64 + 16 * (k - kALanes);
        o1 = o0 + g.odd_delta;
    }
    auto add = [](float4 &acc, const float4 &v) { acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; };
    // gradient of one slot: plane A chunk, or the sum of the two plane-B copies (fixed order: even copy first)
    auto load_slot = [&](int j) {
        const char *sp = gp + (int64_t)j * g.slot_bytes;
        float4 v = ld16(sp + o0);
        if (o1 >= 0) add(v, ld16(sp + o1));
        return v;
    };
    auto store = [&](int t, float4 v) {
        if (mp != nullptr) {
            const unsigned bits = mask_bits4(mp + t * mask_frame, a.mask_col_stride);
            if (bits & 1u) v.x = 0.f;
            if (bits & 2u) v.y = 0.f;
            if (bits & 4u) v.z = 0.f;
            if (bits & 8u) v.w = 0.f;
        }
        *reinterpret_cast<float4 *>(op + t * frame) = v;
    };
    if (a.NS <= kMaxRegFrames) {
        float4 gs[kMaxRegFrames];
#pragma unroll
        for (int j = 0; j < kMaxRegFrames; ++j)
            if (j < a.NS) gs[j] = load_slot(j);
        for (int t = 0; t < a.T2; ++t) {
            const int lo = t < a.n_frame ? max(t - 1, 0) : a.n_local;
            const int hi = t < a.n_frame ? min(t + 1, a.n_local - 1) : a.n_local - 1;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int j = 0; j < kMaxRegFrames; ++j)
                if ((j >= lo && j <= hi) || (a.has_all && j == a.n_local)) add(acc, gs[j]);
            store(t, acc);
        }
    } else {
        for (int t = 0; t < a.T2; ++t) {
            const int lo = t < a.n_frame ? max(t - 1, 0) : a.n_local;
            const int hi = t < a.n_frame ? min(t + 1, a.n_local - 1) : a.n_local - 1;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int j = lo; j <= hi; ++j) add(acc, load_slot(j));
            if (a.has_all) add(acc, load_slot(a.n_local));
            store(t, acc);
        }
    }
}

PlanarFrameArgs make_planar_frame_args(const FrameDims &d, int M)
{
    PlanarFrameArgs a;
    a.N = d.N; a.T2 = d.T2; a.T1 = d.T1; a.n_frame = d.n_frame; a.S = d.S; a.M = M;
    a.n_local = d.T1 < d.n_frame ? d.T1 : d.n_frame;
    a.has_all = d.T1 > d.n_frame ? 1 : 0;
    a.NS = a.n_local + a.has_all;
    a.value_stride_n = d.value_stride_n;
    a.value_stride_t = d.value_stride_t;
    a.mask_row_stride = d.mask_row_stride;
    a.mask_col_stride = d.mask_col_stride;
    a.total = (int64_t)d.N * d.S * M * 12;
    return a;
}

// ------------------------------------------------------------------------------------------
// gather / scatter kernels: grid = (M, query tiles, N*T1); CTA = PAIRS queries x 8 lanes, one head
//
// A query belongs to ONE QUARTER WARP from its first load to its last store, so the kernels need no block-wide
// barrier after the level table is staged: warps of a CTA drift apart and the set-up loads of one overlap the
// gathers of another.
//   phase 1  lane j sets up samples j, j+8, ..: biases, softmax over the query's L*P logits (quarter-warp
//            shuffles: one expf per sample instead of L*P+1), loc = ref + offset / (W_l, H_l) in the reference's
//            operation order (ms_deform_attn.py:164-165), bilinear set-up, and parks TWO 16-byte records per sample:
//              weights  forward: the four corner weights x A;   backward: {lx, ly, A, -}
//              offsets  {plane-A byte offset of (y0,x0) | corner mask, the same one row down, plane-B offsets of the
//                        row-y0 / row-y0+1 pairs (already pointing into the even or the odd copy)}
//            -- everything a lane would otherwise recompute per sample (8 lanes x ~35 instructions) is done once.
//   phase 2  per sample two broadcast LDS.128, then the loads / reductions.  When all four corners are inside the level
//            (mask 15, the common case) every offset is non-negative and goes into the address as an unsigned 32-bit
//            add; the mask bits ride in the low bits of the first offset and are folded into the base pointer.
// ------------------------------------------------------------------------------------------
template <int PAIRS>
struct PlanarCfg {
    static constexpr int THREADS = PAIRS * 8;
    static_assert(THREADS % 32 == 0 && THREADS <= 1024, "quarter warps must tile warps");
};

__device__ __forceinline__ float quarter_max(float v)
{
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
    return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 4));
}

__device__ __forceinline__ float quarter_sum(float v)
{
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v + __shfl_xor_sync(0xffffffffu, v, 4);
}

// Encoder self-attention (Lq == S): the queries ARE the pixels of the pyramid, row-major per level.  A CTA's PAIRS
// consecutive query slots are mapped to a 2-D patch of ONE level (8 wide x PAIRS/8 tall) instead of a row segment,
// so that the cells its samples touch overlap more and stay in L1 (row segment of 32 pixels, offsets within +-4 px:
// ~720 cells per head over the three levels; 8 x 4 patch: ~400).  A bijection of [0, S) onto itself per level (bands of
// TH rows, walked tile by tile; the last tile of a band may be narrower, the last band lower); slots outside every
// level map to themselves.  Results do not depend on it.
template <int TH>
__device__ __forceinline__ int tile_query(int q, const LevelTable &lv, int L)
{
    constexpr int TW = 8;
    int l = 0;
    while (l + 1 < L && q >= lv.start[l + 1]) ++l;
    const int W = lv.W[l], H = lv.H[l], r = q - lv.start[l];
    if (W <= 0 || r < 0 || r >= W * H) return q;
    const int band = r / (TH * W), k = r - band * TH * W;
    const int rb = min(TH, H - band * TH);              // rows of this band
    const int tile = rb * TW, full = (W / TW) * tile;   // pixels of a full-width tile / of all of them
    int tx, inner, wt;
    if (k < full) { tx = k / tile; inner = k - tx * tile; wt = TW; }
    else { tx = W / TW; inner = k - full; wt = W - tx * TW; }
    const int dy = inner / wt, dx = inner - dy * wt;
    return lv.start[l] + (band * TH + dy) * W + tx * TW + dx;
}

// Phase 1 (see above).  Every lane of the warp calls it (full-mask shuffles); `live` = the quarter warp's query exists.
// recw / reco / zs point at the query's own LP entries.  BWD selects the weight record.
template <bool BWD>
__device__ __forceinline__ void planar_phase1(float4 *recw, uint4 *reco, float *zs, const LevelTable &lv,
                                              const SnipArgs &a, const PlanarGeom &g, int n, int t1, int q, bool live,
                                              int j, int m, size_t row, const float *__restrict__ offsets,
                                              const float *__restrict__ logits, const float *__restrict__ ref, float inv_k)
{
    const SnippetDims &d = a.d;
    const int LP = d.L * d.P;
    float mx = -INFINITY;
    if (live) {
        const float *zrow = logits + row * d.logit_row_stride + m * LP;
        for (int i = j; i < LP; i += 8) {
            float z = __ldg(zrow + i);
            if (d.logit_bias != nullptr) z += __ldg(d.logit_bias + m * LP + i);
            zs[i] = z;
            mx = fmaxf(mx, z);
        }
    }
    mx = quarter_max(mx);
    float sum = 0.f;
    if (live)
        for (int i = j; i < LP; i += 8) {
            const float e = expf(zs[i] - mx);
            zs[i] = e;
            sum += e;
        }
    sum = quarter_sum(sum);
    if (!live) {   // empty records: the quarter warp walks them and does nothing (the backward's phase 3 reads A = 0)
        for (int i = j; i < LP; i += 8) { recw[i] = make_float4(0.f, 0.f, 0.f, 0.f); reco[i] = make_uint4(0u, 0u, 0u, 0u); }
        return;
    }
    // encoder: the query is pixel (y, x) of level lq; its reference point on level l is this times vr[l]
    // (analytic_reference_point, same operations in the same order)
    float rxb = 0.f, ryb = 0.f;
    const float *vr = d.valid_ratios ? d.valid_ratios + (size_t)n * d.L * 2 : nullptr;
    if (vr != nullptr) {
        int lq = 0;
        while (lq + 1 < d.L && q >= lv.start[lq + 1]) ++lq;
        const int Wq = max(lv.W[lq], 1);
        const int r = q - lv.start[lq];
        const int y = r / Wq, x = r - y * Wq;
        rxb = ((float)x + 0.5f) / (__ldg(vr + 2 * lq) * (float)lv.W[lq]);
        ryb = ((float)y + 0.5f) / (__ldg(vr + 2 * lq + 1) * (float)lv.H[lq]);
    }
    const float2 *orow = reinterpret_cast<const float2 *>(offsets + row * d.off_row_stride) + m * LP;
    for (int i = j; i < LP; i += 8) {
        const int l = fast_div(i, a.magic_P);
        float2 o = __ldg(orow + i);
        if (d.off_bias != nullptr) {
            const float2 b = __ldg(reinterpret_cast<const float2 *>(d.off_bias) + m * LP + i);
            o.x += b.x; o.y += b.y;
        }
        float2 rp;
        if (vr != nullptr) {
            rp = make_float2(rxb * __ldg(vr + 2 * l), ryb * __ldg(vr + 2 * l + 1));
        } else {
            const float *p = ref + n * d.ref_stride_n + t1 * d.ref_stride_t + ((int64_t)q * d.L + l) * 2;
            rp = make_float2(__ldg(p), __ldg(p + 1));
        }
        const int W = lv.W[l], H = lv.H[l];
        const float u = rp.x + o.x / (float)W;
        const float v = rp.y + o.y / (float)H;
        const Sample<float> s = make_sample<float>(u, v, H, W, lv.start[l]);
        const float at = zs[i] / sum * inv_k;
        if (BWD) {
            recw[i] = make_float4(s.lx, s.ly, at, 0.f);
        } else {
            const float hx = 1.f - s.lx, hy = 1.f - s.ly;
            const float ah = hy * at, al = s.ly * at;
            recw[i] = make_float4(ah * hx, ah * s.lx, al * hx, al * s.lx);
        }
        const int base = s.base, below = s.base + W;
        uint4 o4;
        o4.x = (unsigned)(base * 128) | (unsigned)s.mask;
        o4.y = (unsigned)(below * 128);
        o4.z = (unsigned)(base * 64 + ((base & 1) ? g.odd_delta : 0));
        o4.w = (unsigned)(below * 64 + ((below & 1) ? g.odd_delta : 0));
        if (s.mask == 0) o4 = make_uint4(0u, 0u, 0u, 0u);
        reco[i] = o4;
    }
}

#ifndef MSDA_PLANAR_FWD_MIN_BLOCKS
#define MSDA_PLANAR_FWD_MIN_BLOCKS 4     // x 256 threads: register budget 64
#endif

template <int PAIRS>
__global__ void __launch_bounds__(PlanarCfg<PAIRS>::THREADS, (MSDA_PLANAR_FWD_MIN_BLOCKS * 256) / PlanarCfg<PAIRS>::THREADS)
msda_planar_fwd_kernel(const char *__restrict__ vsum, const int64_t *__restrict__ shapes, const int64_t *__restrict__ lsi,
                       const float *__restrict__ offsets, const float *__restrict__ logits, const float *__restrict__ ref,
                       float *__restrict__ out, const SnipArgs a, const PlanarGeom g)
{
    const SnippetDims &d = a.d;
    __shared__ LevelTable lv;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int LP = d.L * d.P;
    float4 *recw = reinterpret_cast<float4 *>(smem_raw);
    uint4 *reco = reinterpret_cast<uint4 *>(smem_raw + sizeof(float4) * PAIRS * LP);
    float *zs = reinterpret_cast<float *>(smem_raw + 2 * sizeof(float4) * PAIRS * LP);

    const int tid = threadIdx.x;
    const int m = blockIdx.x, q0 = blockIdx.y * PAIRS;
    const int n = blockIdx.z / d.T1, t1 = blockIdx.z - n * d.T1;
    int lo, hi;
    frame_range(t1, d.n_frame, d.T2, lo, hi);
    const size_t qbase = ((size_t)n * d.T1 + t1) * d.Lq;
    const int pl = tid >> 3, j = tid & 7;
    const bool live = q0 + pl < d.Lq;
    recw += pl * LP; reco += pl * LP; zs += pl * LP;

    load_level_table(lv, shapes, lsi, d.L, d.S);
    __syncthreads();
    const int q = (a.tile2d && live) ? tile_query<PAIRS / 8>(q0 + pl, lv, d.L) : q0 + pl;
    planar_phase1<false>(recw, reco, zs, lv, a, g, n, t1, q, live, j, m, qbase + q, offsets, logits, ref,
                         1.f / (float)(hi - lo + 1));
    __syncwarp();

    // ---- phase 2 ----
    const bool left = j < kBLanes;                 // plane B: lanes 0-3 hold the x0 cell, lanes 4-7 the x0+1 cell
    const int slot = t1 < d.n_frame ? t1 : a.n_local;
    const char *sp = vsum + ((int64_t)n * a.n_slots + slot) * g.slot_bytes;
    const char *pa = sp + m * g.a_head + 16 * j;
    const char *pb = sp + g.a_bytes + m * g.b_head + 16 * j;
    const char *pa15 = pa - 15;                    // fast path: offset | 15 == offset + 15
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), accb = make_float4(0.f, 0.f, 0.f, 0.f);
    const int nsamp = live ? LP : 0;
#pragma unroll 2
    for (int i = 0; i < nsamp; ++i) {
        const float4 w = recw[i];
        const uint4 o = reco[i];
        const float wt = left ? w.x : w.y, wb = left ? w.z : w.w;
        const unsigned mask = o.x & 15u;
        if (mask == 0xfu) {
            const char *a0 = pa15 + o.x, *a1 = pa + o.y;
            const float4 v0 = ld16(a0), v1 = ld16(a0 + 128), v2 = ld16(a1), v3 = ld16(a1 + 128);
            const float4 u0 = ld16(pb + o.z), u1 = ld16(pb + o.w);
            fma4(acc, w.x, v0); fma4(acc, w.y, v1); fma4(acc, w.z, v2); fma4(acc, w.w, v3);
            fma4(accb, wt, u0); fma4(accb, wb, u1);
        } else if (mask != 0u) {
            const char *a0 = pa + (ptrdiff_t)(int)(o.x & ~15u), *a1 = pa + (ptrdiff_t)(int)o.y;
            if (mask & 1u) fma4(acc, w.x, ld16(a0));
            if (mask & 2u) fma4(acc, w.y, ld16(a0 + 128));
            if (mask & 4u) fma4(acc, w.z, ld16(a1));
            if (mask & 8u) fma4(acc, w.w, ld16(a1 + 128));
            if (mask & (left ? 1u : 2u)) fma4(accb, wt, ld16(pb + (ptrdiff_t)(int)o.z));
            if (mask & (left ? 4u : 8u)) fma4(accb, wb, ld16(pb + (ptrdiff_t)(int)o.w));
        }
    }
    // the two halves of the quarter warp hold the same 16 channels of plane B (left / right cells)
    accb.x += __shfl_xor_sync(0xffffffffu, accb.x, 4);
    accb.y += __shfl_xor_sync(0xffffffffu, accb.y, 4);
    accb.z += __shfl_xor_sync(0xffffffffu, accb.z, 4);
    accb.w += __shfl_xor_sync(0xffffffffu, accb.w, 4);
    if (live) {
        char *op = reinterpret_cast<char *>(out) + ((qbase + q) * d.M + m) * (size_t)(kPlanarD * 4);
        *reinterpret_cast<float4 *>(op + 16 * j) = acc;
        if (left) *reinterpret_cast<float4 *>(op + 128 + 16 * j) = accb;
    }
}

// sum pa / px / py over the 8 lanes of a quarter warp with 6 shuffles instead of 9: the halves first trade pa
// against px, so after the xor-4 step lanes 0-3 carry pa and lanes 4-7 px.  Result: lane 0 -> pa, lane 4 -> px,
// every lane -> py.
__device__ __forceinline__ void quarter_sum3(float &pax, float &py, float pa, float px, bool left)
{
    const float send = left ? px : pa;
    pax = (left ? pa : px) + __shfl_xor_sync(0xffffffffu, send, 4);
    py += __shfl_xor_sync(0xffffffffu, py, 4);
    pax += __shfl_xor_sync(0xffffffffu, pax, 2);
    py += __shfl_xor_sync(0xffffffffu, py, 2);
    pax += __shfl_xor_sync(0xffffffffu, pax, 1);
    py += __shfl_xor_sync(0xffffffffu, py, 1);
}

#ifndef MSDA_PLANAR_BWD_MIN_BLOCKS
#define MSDA_PLANAR_BWD_MIN_BLOCKS 4
#endif

template <int PAIRS>
__global__ void __launch_bounds__(PlanarCfg<PAIRS>::THREADS, (MSDA_PLANAR_BWD_MIN_BLOCKS * 256) / PlanarCfg<PAIRS>::THREADS)
msda_planar_bwd_kernel(const char *__restrict__ vsum, const int64_t *__restrict__ shapes, const int64_t *__restrict__ lsi,
                       const float *__restrict__ offsets, const float *__restrict__ logits, const float *__restrict__ ref,
                       const float *__restrict__ grad_out, char *__restrict__ gsum, float *__restrict__ grad_offsets,
                       float *__restrict__ grad_logits, const SnipArgs a, const PlanarGeom g)
{
    using Cfg = PlanarCfg<PAIRS>;
    const SnippetDims &d = a.d;
    __shared__ LevelTable lv;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int LP = d.L * d.P;
    float4 *recw_all = reinterpret_cast<float4 *>(smem_raw);                                  // {lx, ly, A, -}
    uint4 *reco_all = reinterpret_cast<uint4 *>(smem_raw + sizeof(float4) * PAIRS * LP);
    float *zs_all = reinterpret_cast<float *>(smem_raw + 2 * sizeof(float4) * PAIRS * LP);
    float *part = zs_all + PAIRS * LP;                                                        // [sample][3]
    __shared__ int qmap[PAIRS];                                                               // query of each slot of the tile

    const int tid = threadIdx.x;
    const int m = blockIdx.x, q0 = blockIdx.y * PAIRS;
    const int n = blockIdx.z / d.T1, t1 = blockIdx.z - n * d.T1;
    int lo, hi;
    frame_range(t1, d.n_frame, d.T2, lo, hi);
    const int nf = hi - lo + 1;
    const size_t qbase = ((size_t)n * d.T1 + t1) * d.Lq;

    load_level_table(lv, shapes, lsi, d.L, d.S);
    __syncthreads();
    {
        const int pl = tid >> 3, j = tid & 7;
        const bool live = q0 + pl < d.Lq;
        const int q = (a.tile2d && live) ? tile_query<PAIRS / 8>(q0 + pl, lv, d.L) : q0 + pl;
        if (j == 0) qmap[pl] = q;
        const bool left = j < kBLanes;
        float4 *recw = recw_all + pl * LP;
        uint4 *reco = reco_all + pl * LP;
        planar_phase1<true>(recw, reco, zs_all + pl * LP, lv, a, g, n, t1, q, live, j, m, qbase + q, offsets, logits, ref,
                            1.f / (float)nf);
        __syncwarp();

        // ---- phase 2: every thread participates (full-mask shuffles) ----
        const int slot = t1 < d.n_frame ? t1 : a.n_local;
        const int64_t slot_off = ((int64_t)n * a.n_slots + slot) * g.slot_bytes;
        const char *pa = vsum + slot_off + m * g.a_head + 16 * j;
        const char *pb = vsum + slot_off + g.a_bytes + m * g.b_head + 16 * j;
        char *ga = gsum + slot_off + m * g.a_head + 16 * j;
        char *gb = gsum + slot_off + g.a_bytes + m * g.b_head + 16 * j;
        float4 gA = make_float4(0.f, 0.f, 0.f, 0.f), gB = gA;
        if (live) {
            const char *gp = reinterpret_cast<const char *>(grad_out) + ((qbase + q) * d.M + m) * (size_t)(kPlanarD * 4);
            gA = ld16(gp + 16 * j);
            gB = ld16(gp + 128 + 16 * (j & 3));
        }
        float *mypart = part + (size_t)(pl * LP) * 3;
        for (int i = 0; i < LP; ++i) {
            const float4 f = recw[i];
            const uint4 o = reco[i];
            const unsigned mask = o.x & 15u;
            const BwdWeights bw = make_bwd_weights(f.x, f.y, f.z);
            const float at = left ? bw.a0 : bw.a1, ab = left ? bw.a2 : bw.a3;
            float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f, et = 0.f, eb = 0.f;
            if (mask == 0xfu) {
                const size_t o0 = (size_t)o.x - 15u, o1 = o.y;
                const float4 v0 = ld16(pa + o0), v1 = ld16(pa + o0 + 128), v2 = ld16(pa + o1), v3 = ld16(pa + o1 + 128);
                const float4 u0 = ld16(pb + o.z), u1 = ld16(pb + o.w);
                red16(ga + o0, bw.a0, gA); red16(ga + o0 + 128, bw.a1, gA); red16(ga + o1, bw.a2, gA); red16(ga + o1 + 128, bw.a3, gA);
                red16(gb + o.z, at, gB); red16(gb + o.w, ab, gB);
                d0 = dot4(gA, v0); d1 = dot4(gA, v1); d2 = dot4(gA, v2); d3 = dot4(gA, v3);
                et = dot4(gB, u0); eb = dot4(gB, u1);
            } else if (mask != 0u) {
                const ptrdiff_t o0 = (ptrdiff_t)(int)(o.x & ~15u), o1 = (ptrdiff_t)(int)o.y;
                const ptrdiff_t b0 = (ptrdiff_t)(int)o.z, b1 = (ptrdiff_t)(int)o.w;
                if (mask & 1u) { d0 = dot4(gA, ld16(pa + o0)); red16(ga + o0, bw.a0, gA); }
                if (mask & 2u) { d1 = dot4(gA, ld16(pa + o0 + 128)); red16(ga + o0 + 128, bw.a1, gA); }
                if (mask & 4u) { d2 = dot4(gA, ld16(pa + o1)); red16(ga + o1, bw.a2, gA); }
                if (mask & 8u) { d3 = dot4(gA, ld16(pa + o1 + 128)); red16(ga + o1 + 128, bw.a3, gA); }
                if (mask & (left ? 1u : 2u)) { et = dot4(gB, ld16(pb + b0)); red16(gb + b0, at, gB); }
                if (mask & (left ? 4u : 8u)) { eb = dot4(gB, ld16(pb + b1)); red16(gb + b1, ab, gB); }
            }
            // this lane's share of d_k = <G, V_k>: its 4 channels of plane A for every corner + its plane-B cell
            if (left) { d0 += et; d2 += eb; } else { d1 += et; d3 += eb; }
            float pa_ = fmaf(bw.w0, d0, fmaf(bw.w1, d1, fmaf(bw.w2, d2, bw.w3 * d3)));
            float px_ = fmaf(bw.hy, d1 - d0, bw.ly * (d3 - d2));
            float py_ = fmaf(bw.hx, d2 - d0, bw.lx * (d3 - d1));
            float pax;
            quarter_sum3(pax, py_, pa_, px_, left);
            if (j == 0) { mypart[i * 3] = pax; mypart[i * 3 + 2] = py_; }
            if (j == 4) mypart[i * 3 + 1] = pax;
        }
    }
    __syncthreads();

    // ---- phase 3: per-sample finish + softmax backward (as msda_snippet_bwd_kernel) ----
    // dL/dz_i = A_i * (gA_i - k * sum_j gA_j A_j)   with A = softmax/k, gA_i = <G, val_i>
    for (int i = tid; i < PAIRS * LP; i += Cfg::THREADS) {
        const float pa_ = part[i * 3], px_ = part[i * 3 + 1], py_ = part[i * 3 + 2];
        const int spl = fast_div(i, a.magic_LP);
        const float at = recw_all[i].z;
        if (q0 + spl < d.Lq)
            reinterpret_cast<float2 *>(grad_offsets + (qbase + qmap[spl]) * d.off_row_stride)[m * LP + (i - spl * LP)] =
                make_float2(at * px_, at * py_);
        part[i * 3] = pa_ * at;   // own slots only ([0] = gA_i A_i, [1] = gA_i)
        part[i * 3 + 1] = pa_;
    }
    __syncthreads();
    for (int i = tid; i < PAIRS * LP; i += Cfg::THREADS) {
        const int spl = fast_div(i, a.magic_LP);
        if (q0 + spl < d.Lq) {
            float dot = 0.f;
            for (int jj = 0; jj < LP; ++jj) dot += part[(spl * LP + jj) * 3];
            grad_logits[(qbase + qmap[spl]) * d.logit_row_stride + m * LP + (i - spl * LP)] =
                recw_all[i].z * (part[i * 3 + 1] - (float)nf * dot);
        }
    }
}

SnipArgs make_planar_args(const SnippetDims &d)
{
    SnipArgs a = make_snip_args<float>(d);
    a.cell_bytes = 16;   // (unused by the planar kernels)
    // encoder self-attention: the query slots of a CTA walk 2-D pixel patches (MSDA_PLANAR_TILE2D=0 in the environment
    // keeps row segments: benchmark knob, read once; results do not depend on it)
    static const bool tile2d_on = [] { const char *e = getenv("MSDA_PLANAR_TILE2D"); return !(e && e[0] == '0'); }();
    a.tile2d = (tile2d_on && d.Lq == d.S) ? 1 : 0;
    return a;
}

// queries per CTA: 32 unless MSDA_PLANAR_PAIRS = 16 | 32 | 64 is set in the environment (benchmark knob, read once)
int planar_pairs()
{
    static const int v = [] {
        const char *e = getenv("MSDA_PLANAR_PAIRS");
        const int x = e ? atoi(e) : 32;
        return (x == 16 || x == 32 || x == 64) ? x : 32;
    }();
    return v;
}

template <int PAIRS>
cudaError_t launch_fwd(const void *vsum, const int64_t *shapes, const int64_t *lsi, const float *offsets,
                       const float *logits, const float *ref, float *out, const SnippetDims &d, cudaStream_t stream)
{
    const SnipArgs a = make_planar_args(d);
    const PlanarGeom g = make_geom(d.S, d.M);
    const dim3 grid(d.M, (d.Lq + PAIRS - 1) / PAIRS, d.N * d.T1);
    const size_t smem = (2 * sizeof(float4) + sizeof(float)) * PAIRS * d.L * d.P;
    if (smem > kSmemOptIn) {
        const cudaError_t e =
            cudaFuncSetAttribute(msda_planar_fwd_kernel<PAIRS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    msda_planar_fwd_kernel<PAIRS><<<grid, PlanarCfg<PAIRS>::THREADS, smem, stream>>>(
        static_cast<const char *>(vsum), shapes, lsi, offsets, logits, ref, out, a, g);
    return cudaGetLastError();
}

template <int PAIRS>
cudaError_t launch_bwd(const void *vsum, const int64_t *shapes, const int64_t *lsi, const float *offsets,
                       const float *logits, const float *ref, const float *grad_out, void *gsum, float *grad_offsets,
                       float *grad_logits, const SnippetDims &d, cudaStream_t stream)
{
    const SnipArgs a = make_planar_args(d);
    const PlanarGeom g = make_geom(d.S, d.M);
    const dim3 grid(d.M, (d.Lq + PAIRS - 1) / PAIRS, d.N * d.T1);
    const size_t smem = (2 * sizeof(float4) + 4 * sizeof(float)) * PAIRS * d.L * d.P;
    if (smem > kSmemOptIn) {
        const cudaError_t e =
            cudaFuncSetAttribute(msda_planar_bwd_kernel<PAIRS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    msda_planar_bwd_kernel<PAIRS><<<grid, PlanarCfg<PAIRS>::THREADS, smem, stream>>>(
        static_cast<const char *>(vsum), shapes, lsi, offsets, logits, ref, grad_out, static_cast<char *>(gsum),
        grad_offsets, grad_logits, a, g);
    return cudaGetLastError();
}

}  // namespace

// 0 when the planar layout does not apply (it is built for fp32 heads of 48 channels, 32-bit slot offsets)
cudaError_t launch_frame_sum_planar(const float *value, const uint8_t *mask, void *vsum, const FrameDims &d, int M,
                                    cudaStream_t stream)
{
    const PlanarFrameArgs a = make_planar_frame_args(d, M);
    if (a.total == 0) return cudaSuccess;
    const int64_t blocks = (a.total + 255) / 256;
    if (blocks > 0x7fffffff) return cudaErrorInvalidValue;
    frame_sum_planar_kernel<<<(unsigned)blocks, 256, 0, stream>>>(value, mask, static_cast<char *>(vsum), a,
                                                                  make_geom(d.S, M));
    return cudaGetLastError();
}

cudaError_t launch_frame_unsum_planar(const void *grad_vsum, const uint8_t *mask, float *grad_value, const FrameDims &d,
                                      int M, cudaStream_t stream)
{
    const PlanarFrameArgs a = make_planar_frame_args(d, M);
    if (a.total == 0) return cudaSuccess;
    const int64_t blocks = (a.total + 255) / 256;
    if (blocks > 0x7fffffff) return cudaErrorInvalidValue;
    frame_unsum_planar_kernel<<<(unsigned)blocks, 256, 0, stream>>>(static_cast<const char *>(grad_vsum), mask, grad_value,
                                                                    a, make_geom(d.S, M));
    return cudaGetLastError();
}

cudaError_t launch_planar_forward_f32(const void *vsum, const int64_t *shapes, const int64_t *lsi, const float *offsets,
                                      const float *logits, const float *ref, float *out, const SnippetDims &d,
                                      cudaStream_t stream)
{
    switch (planar_pairs()) {
        case 16: return launch_fwd<16>(vsum, shapes, lsi, offsets, logits, ref, out, d, stream);
        case 64: return launch_fwd<64>(vsum, shapes, lsi, offsets, logits, ref, out, d, stream);
        default: return launch_fwd<32>(vsum, shapes, lsi, offsets, logits, ref, out, d, stream);
    }
}

cudaError_t launch_planar_backward_f32(const void *vsum, const int64_t *shapes, const int64_t *lsi, const float *offsets,
                                       const float *logits, const float *ref, const float *grad_out, void *gsum,
                                       float *grad_offsets, float *grad_logits, const SnippetDims &d, cudaStream_t stream)
{
    switch (planar_pairs()) {
        case 16: return launch_bwd<16>(vsum, shapes, lsi, offsets, logits, ref, grad_out, gsum, grad_offsets, grad_logits, d, stream);
        case 64: return launch_bwd<64>(vsum, shapes, lsi, offsets, logits, ref, grad_out, gsum, grad_offsets, grad_logits, d, stream);
        default: return launch_bwd<32>(vsum, shapes, lsi, offsets, logits, ref, grad_out, gsum, grad_offsets, grad_logits, d, stream);
    }
}

}  // namespace msda
