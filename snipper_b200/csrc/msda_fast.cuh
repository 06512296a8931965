// Shared machinery of the fast fp32 kernels (per-call and fused snippet), sm_100a.
//
// CTA = TILE of PAIRS consecutive queries x ONE head; thread = (query-in-tile, 16-byte channel
// chunk) -- LANES = D/4 lanes per query, so one warp-wide LDG.128 covers whole 4*D-byte head
// slices and every gathered cell is consumed as full 32-byte sectors.
//
//   phase 1  one thread per SAMPLE (query, level, point): bilinear set-up done once and parked
//            in shared memory as ONE 16-byte record {lx, ly, A, byte offset of the (y0,x0) cell | corner mask}
//            (the reference redoes this set-up in every one of the D channel threads)
//   phase 2  each lane walks its query's samples: one broadcast LDS.128, 8 FP instructions for the
//            four corner weights, then -- when all four corners are valid, the common case -- 4
//            unpredicated LDG.128 whose "+1 cell" addresses are immediate offsets (the cell stride is
//            a template constant for Snipper's M*D = 384), 16 FFMA.  Border samples take a predicated
//            slow path.
//
// Why this shape: ncu on the first versions (profiles/r01_run3_*, r01_run6_*) showed the gather
// limited first by INSTRUCTION ISSUE (64-bit address arithmetic, zero-filling registers for
// predicated loads, per-corner predicate tests: ~93 instructions per lane-point for 16 useful
// FFMA + 4 LDG); once that was gone, by the L1 DATA PIPE (two 128-byte wavefronts per 192-byte head
// slice, plus one per quarter warp for every wide shared load): the fused forward now runs at the
// measured L1 gather ceiling (tools/micro/l1_tex_vs_ldg.cu).  HBM traffic is only the compulsory one.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include "msda_common.cuh"

namespace msda {

// register form of a sample (unpacked from its record by record_meta)
struct __align__(8) SampleMeta {
    int off;        // byte offset of cell (y0,x0) relative to (batch base + head slice), may be "virtual"
    unsigned wm;    // (row stride in bytes) | corner mask << 28
};

constexpr unsigned kAllCorners = 0xF0000000u;

// exact i / d for 0 <= i*d < 2^24 with magic = ceil(2^24 / d)  (host: fast_magic)
__device__ __forceinline__ int fast_div(int i, unsigned magic) { return (int)(((unsigned)i * magic) >> 24); }
inline unsigned fast_magic(int d) { return (unsigned)(((1u << 24) + (unsigned)d - 1u) / (unsigned)d); }
__device__ __forceinline__ unsigned fast_magic_dev(int d) { return ((1u << 24) + (unsigned)d - 1u) / (unsigned)d; }

// A sample is parked in shared memory as ONE 16-byte record {lx, ly, A, off | mask}: `off` is the byte
// offset of the (y0,x0) cell -- a multiple of 16, so its low four bits carry the corner mask.  One
// LDS.128 per sample and lane in the gather loop (wide shared loads cost an L1 wavefront per quarter
// warp, and the L1 data pipe is what bounds these kernels); the row stride comes from the level table
// and the four corner weights are recomputed per lane (8 FP instructions on otherwise idle issue slots).
__device__ __forceinline__ float4 make_record(const Sample<float> &s, float at, int cell_bytes)
{
    return make_float4(s.lx, s.ly, at, __int_as_float((s.base * cell_bytes) | s.mask));
}

__device__ __forceinline__ float4 empty_record() { return make_float4(0.f, 0.f, 0.f, __int_as_float(0)); }

// Unpack a record into the SampleMeta the gather helpers take (row = W_l * cell_bytes).
__device__ __forceinline__ SampleMeta record_meta(const float4 &r, unsigned row)
{
    const int om = __float_as_int(r.w);
    SampleMeta mt;
    mt.off = om & ~15;
    mt.wm = row | ((unsigned)(om & 15) << 28);
    return mt;
}

// forward corner weights (bilinear x A) from a record
__device__ __forceinline__ float4 record_weights(const float4 &r)
{
    const float hx = 1.f - r.x, hy = 1.f - r.y;
    const float ah = hy * r.z, al = r.y * r.z;
    return make_float4(ah * hx, ah * r.x, al * hx, al * r.x);
}

template <int CSB>
__device__ __forceinline__ int cell_stride_bytes(int runtime_csb) { return CSB > 0 ? CSB : runtime_csb; }

// ------------------------------------------------------------------------------------------
// 16-byte channel chunk of the value / output / grad_output element type VT, widened to fp32:
//   float          4 channels  (LDG.E.128 -> 4 registers used as they are)
//   __nv_bfloat16  8 channels  (LDG.E.128 -> 4 registers, each split with one shift / one mask)
//   __half         8 channels  (LDG.E.128 -> 4 registers, each widened by two half -> float conversions)
// All arithmetic is fp32 whatever VT is.
// ------------------------------------------------------------------------------------------
template <typename VT> struct Chunk;

template <> struct Chunk<float> {
    using elem = float;
    static constexpr int N = 4;
    static constexpr int BYTES = 16;
    float x[4];
    static __device__ __forceinline__ Chunk load(const char *p)
    {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(p));
        Chunk c;
        c.x[0] = v.x; c.x[1] = v.y; c.x[2] = v.z; c.x[3] = v.w;
        return c;
    }
    __device__ __forceinline__ void store(char *p) const
    {
        *reinterpret_cast<float4 *>(p) = make_float4(x[0], x[1], x[2], x[3]);
    }
};

template <> struct Chunk<__nv_bfloat16> {
    using elem = __nv_bfloat16;
    static constexpr int N = 8;
    static constexpr int BYTES = 16;
    float x[8];
    static __device__ __forceinline__ Chunk load(const char *p)
    {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p));
        Chunk c;
        c.x[0] = __uint_as_float(v.x << 16); c.x[1] = __uint_as_float(v.x & 0xffff0000u);
        c.x[2] = __uint_as_float(v.y << 16); c.x[3] = __uint_as_float(v.y & 0xffff0000u);
        c.x[4] = __uint_as_float(v.z << 16); c.x[5] = __uint_as_float(v.z & 0xffff0000u);
        c.x[6] = __uint_as_float(v.w << 16); c.x[7] = __uint_as_float(v.w & 0xffff0000u);
        return c;
    }
    __device__ __forceinline__ void store(char *p) const
    {
        uint4 v;
        __nv_bfloat162 t;
        t = __floats2bfloat162_rn(x[0], x[1]); v.x = *reinterpret_cast<unsigned *>(&t);
        t = __floats2bfloat162_rn(x[2], x[3]); v.y = *reinterpret_cast<unsigned *>(&t);
        t = __floats2bfloat162_rn(x[4], x[5]); v.z = *reinterpret_cast<unsigned *>(&t);
        t = __floats2bfloat162_rn(x[6], x[7]); v.w = *reinterpret_cast<unsigned *>(&t);
        *reinterpret_cast<uint4 *>(p) = v;
    }
};

// 8-byte lane of 4 bf16 channels: the BACKWARD lane type for bf16.  With 4 channels per lane the
// fp32 grad_value bytes a lane owns are one contiguous 16-byte vector reduction, exactly as in the
// fp32 kernels; the 16-byte lane of 8 channels would need two half-filled reductions per corner
// (measured 25 % slower, profiles/r01_run12_*).
struct bf16q {};

template <> struct Chunk<bf16q> {
    using elem = __nv_bfloat16;
    static constexpr int N = 4;
    static constexpr int BYTES = 8;
    float x[4];
    static __device__ __forceinline__ Chunk load(const char *p)
    {
        const uint2 v = __ldg(reinterpret_cast<const uint2 *>(p));
        Chunk c;
        c.x[0] = __uint_as_float(v.x << 16); c.x[1] = __uint_as_float(v.x & 0xffff0000u);
        c.x[2] = __uint_as_float(v.y << 16); c.x[3] = __uint_as_float(v.y & 0xffff0000u);
        return c;
    }
    __device__ __forceinline__ void store(char *p) const
    {
        uint2 v;
        __nv_bfloat162 t;
        t = __floats2bfloat162_rn(x[0], x[1]); v.x = *reinterpret_cast<unsigned *>(&t);
        t = __floats2bfloat162_rn(x[2], x[3]); v.y = *reinterpret_cast<unsigned *>(&t);
        *reinterpret_cast<uint2 *>(p) = v;
    }
};

// fp16 twins of the two bf16 lane types (libmsda_b200_f16.so): same lanes, same bytes, only the widening and the
// rounding differ -- one conversion per channel on load (as the bf16 shift / mask), one packing conversion per two
// channels on store, round to nearest even with overflow to +-inf.
__device__ __forceinline__ float2 widen_half2(unsigned w) { return __half22float2(*reinterpret_cast<const __half2 *>(&w)); }

__device__ __forceinline__ unsigned narrow_half2(float a, float b)
{
    const __half2 t = __floats2half2_rn(a, b);
    return *reinterpret_cast<const unsigned *>(&t);
}

template <> struct Chunk<__half> {
    using elem = __half;
    static constexpr int N = 8;
    static constexpr int BYTES = 16;
    float x[8];
    static __device__ __forceinline__ Chunk load(const char *p)
    {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p));
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
        Chunk c;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 f = widen_half2(w[i]);
            c.x[2 * i] = f.x; c.x[2 * i + 1] = f.y;
        }
        return c;
    }
    __device__ __forceinline__ void store(char *p) const
    {
        *reinterpret_cast<uint4 *>(p) = make_uint4(narrow_half2(x[0], x[1]), narrow_half2(x[2], x[3]),
                                                   narrow_half2(x[4], x[5]), narrow_half2(x[6], x[7]));
    }
};

// 8-byte lane of 4 fp16 channels: the twin of bf16q
struct halfq {};

template <> struct Chunk<halfq> {
    using elem = __half;
    static constexpr int N = 4;
    static constexpr int BYTES = 8;
    float x[4];
    static __device__ __forceinline__ Chunk load(const char *p)
    {
        const uint2 v = __ldg(reinterpret_cast<const uint2 *>(p));
        const float2 lo = widen_half2(v.x), hi = widen_half2(v.y);
        Chunk c;
        c.x[0] = lo.x; c.x[1] = lo.y; c.x[2] = hi.x; c.x[3] = hi.y;
        return c;
    }
    __device__ __forceinline__ void store(char *p) const
    {
        *reinterpret_cast<uint2 *>(p) = make_uint2(narrow_half2(x[0], x[1]), narrow_half2(x[2], x[3]));
    }
};

template <typename C>
__device__ __forceinline__ C zero_chunk()
{
    C c;
#pragma unroll
    for (int i = 0; i < C::N; ++i) c.x[i] = 0.f;
    return c;
}

template <typename C>
__device__ __forceinline__ void fma_chunk(C &acc, float w, const C &v)
{
#pragma unroll
    for (int i = 0; i < C::N; ++i) acc.x[i] = fmaf(w, v.x[i], acc.x[i]);
}

template <typename C>
__device__ __forceinline__ float dot_chunk(const C &a, const C &b)
{
    float d = a.x[C::N - 1] * b.x[C::N - 1];
#pragma unroll
    for (int i = C::N - 2; i >= 0; --i) d = fmaf(a.x[i], b.x[i], d);
    return d;
}

// grad_value is accumulated in fp32 whatever VT is.  A lane that gathers C::N channels owns
// C::N * 4 bytes of the fp32 slice.  fp32: one 128-bit vector reduction at byte 16 * lane.
// bf16: two, and they must not be the lane's own 32 contiguous bytes -- each instruction would
// then touch every 32-byte sector of the slice half-filled and double the L2 request count.
// Instead lanes pair up (2j, 2j+1) over 64 bytes: instruction A writes bytes [0,32) of the pair
// (16 each), instruction B bytes [32,64).  `RedView` holds G's channels in that arrangement
// (swapped once per pair of lanes with four shuffles), `red_lane_offset` the matching address.
// Lanes of 4 channels (float, bf16q, halfq) and lanes of 8 (__nv_bfloat16, __half) each have one view.
template <typename VT, int N = Chunk<VT>::N> struct RedView;

template <typename VT> struct RedView<VT, 4> {
    float x[4];
    static __device__ __forceinline__ RedView make(const Chunk<VT> &g)
    {
        RedView r;
#pragma unroll
        for (int i = 0; i < 4; ++i) r.x[i] = g.x[i];
        return r;
    }
    static __device__ __forceinline__ int lane_offset(int lane) { return lane * 16; }
    __device__ __forceinline__ void red(char *gp, float a) const
    {
        red_add_v4(reinterpret_cast<float *>(gp), a * x[0], a * x[1], a * x[2], a * x[3]);
    }
};

template <typename VT> struct RedView<VT, 8> {
    float x[8];  // [0,4): what instruction A writes, [4,8): instruction B
    // every lane of the warp must call this (full-mask shuffles); LANES is even, so (2j, 2j+1) never
    // straddles a query
    static __device__ __forceinline__ RedView make(const Chunk<VT> &g)
    {
        const bool odd = threadIdx.x & 1;
        RedView r;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float send = odd ? g.x[i] : g.x[4 + i];          // the half the partner writes
            const float recv = __shfl_xor_sync(0xffffffffu, send, 1);
            r.x[i] = odd ? recv : g.x[i];                          // A: channels 16j + 4*(lane&1) + i
            r.x[4 + i] = odd ? g.x[4 + i] : recv;                  // B: channels 16j + 8 + 4*(lane&1) + i
        }
        return r;
    }
    static __device__ __forceinline__ int lane_offset(int lane) { return (lane >> 1) * 64 + (lane & 1) * 16; }
    __device__ __forceinline__ void red(char *gp, float a) const
    {
        red_add_v4(reinterpret_cast<float *>(gp), a * x[0], a * x[1], a * x[2], a * x[3]);
        red_add_v4(reinterpret_cast<float *>(gp + 32), a * x[4], a * x[5], a * x[6], a * x[7]);
    }
};

// Forward gather of one sample for this lane: acc += sum_k w_k * V[corner_k]
template <typename VT, int CSB>
__device__ __forceinline__ void gather_fma(Chunk<VT> &acc, const SampleMeta mt, const float4 w,
                                           const char *__restrict__ p0, int runtime_csb)
{
    using C = Chunk<VT>;
    const int csb = cell_stride_bytes<CSB>(runtime_csb);
    const char *a0 = p0 + (ptrdiff_t)mt.off;
    const char *a2 = a0 + (mt.wm & 0x0fffffffu);
    if (mt.wm >= kAllCorners) {
        const C v0 = C::load(a0);
        const C v1 = C::load(a0 + csb);
        const C v2 = C::load(a2);
        const C v3 = C::load(a2 + csb);
        fma_chunk(acc, w.x, v0);
        fma_chunk(acc, w.y, v1);
        fma_chunk(acc, w.z, v2);
        fma_chunk(acc, w.w, v3);
    } else {
        const unsigned mask = mt.wm >> 28;
        if (mask & 1u) fma_chunk(acc, w.x, C::load(a0));
        if (mask & 2u) fma_chunk(acc, w.y, C::load(a0 + csb));
        if (mask & 4u) fma_chunk(acc, w.z, C::load(a2));
        if (mask & 8u) fma_chunk(acc, w.w, C::load(a2 + csb));
    }
}

// Same, over `nf` consecutive value frames (fused snippet kernel): the sample set-up is shared by all
// neighbour frames, so the fast/slow decision is taken once and the frame loop is branch-free,
// which lets the loads of two frames overlap.
template <typename VT, int CSB>
__device__ __forceinline__ void gather_fma_frames(Chunk<VT> &acc, const SampleMeta mt, const float4 w,
                                                  const char *__restrict__ pf, int64_t frame_bytes, int nf,
                                                  int runtime_csb)
{
    using C = Chunk<VT>;
    const int csb = cell_stride_bytes<CSB>(runtime_csb);
    const char *a0 = pf + (ptrdiff_t)mt.off;
    const ptrdiff_t row = (ptrdiff_t)(mt.wm & 0x0fffffffu);
    if (mt.wm >= kAllCorners) {
#pragma unroll 2
        for (int f = 0; f < nf; ++f, a0 += frame_bytes) {
            const C v0 = C::load(a0);
            const C v1 = C::load(a0 + csb);
            const C v2 = C::load(a0 + row);
            const C v3 = C::load(a0 + row + csb);
            fma_chunk(acc, w.x, v0);
            fma_chunk(acc, w.y, v1);
            fma_chunk(acc, w.z, v2);
            fma_chunk(acc, w.w, v3);
        }
    } else {
        const unsigned mask = mt.wm >> 28;
        if (mask == 0u) return;
        for (int f = 0; f < nf; ++f, a0 += frame_bytes) {
            if (mask & 1u) fma_chunk(acc, w.x, C::load(a0));
            if (mask & 2u) fma_chunk(acc, w.y, C::load(a0 + csb));
            if (mask & 4u) fma_chunk(acc, w.z, C::load(a0 + row));
            if (mask & 8u) fma_chunk(acc, w.w, C::load(a0 + row + csb));
        }
    }
}

// Per-sample scalars a backward lane needs, derived once per sample from {lx, ly, A}
// (outside the neighbour-frame loop of the fused kernel).
struct BwdWeights {
    float lx, ly, hx, hy;
    float w0, w1, w2, w3;      // bilinear corner weights
    float a0, a1, a2, a3;      // w_k * A  (what is scattered into grad_value, times G)
};

__device__ __forceinline__ BwdWeights make_bwd_weights(float lx, float ly, float at)
{
    BwdWeights b;
    b.lx = lx; b.ly = ly; b.hx = 1.f - lx; b.hy = 1.f - ly;
    b.w0 = b.hy * b.hx; b.w1 = b.hy * lx; b.w2 = ly * b.hx; b.w3 = ly * lx;
    b.a0 = b.w0 * at; b.a1 = b.w1 * at; b.a2 = b.w2 * at; b.a3 = b.w3 * at;
    return b;
}

// Backward work of one sample for this lane on one value frame: scatter w_k*A*G into grad_value
// (vector reductions) and accumulate the three per-sample partial dot products.
// "Dot first": d_k = <G, V_k> over this lane's channels, then
//     <G, val>      = sum_k w_k d_k
//     <G, dval/dx>  = hy (d1 - d0) + ly (d3 - d2)
//     <G, dval/dy>  = hx (d2 - d0) + lx (d3 - d1)
// -- 28 FP instructions (fp32) instead of the 60 of forming val / dval per channel and dotting after.
// gp0 addresses the fp32 grad_value buffer (head slice + RedView::lane_offset): its cell byte
// offsets are GS = 4 / sizeof(VT) times the value byte offsets held in the sample record.
template <typename VT, int CSB, bool SCATTER>
__device__ __forceinline__ void gather_scatter(const SampleMeta mt, const BwdWeights &b, const Chunk<VT> &g,
                                               const RedView<VT> &gr, const char *__restrict__ p0, char *gp0,
                                               int runtime_csb, float &pa, float &px, float &py)
{
    using C = Chunk<VT>;
    constexpr int GS = 4 / (int)sizeof(typename C::elem);
    const int csb = cell_stride_bytes<CSB>(runtime_csb);
    const ptrdiff_t o0 = (ptrdiff_t)mt.off;
    const ptrdiff_t o2 = o0 + (mt.wm & 0x0fffffffu);
    float d0, d1, d2, d3;
    if (mt.wm >= kAllCorners) {
        const C v0 = C::load(p0 + o0);
        const C v1 = C::load(p0 + o0 + csb);
        const C v2 = C::load(p0 + o2);
        const C v3 = C::load(p0 + o2 + csb);
        if (SCATTER) {
            gr.red(gp0 + GS * o0, b.a0);
            gr.red(gp0 + GS * (o0 + csb), b.a1);
            gr.red(gp0 + GS * o2, b.a2);
            gr.red(gp0 + GS * (o2 + csb), b.a3);
        }
        d0 = dot_chunk(g, v0); d1 = dot_chunk(g, v1); d2 = dot_chunk(g, v2); d3 = dot_chunk(g, v3);
    } else {
        const unsigned mask = mt.wm >> 28;
        if (mask == 0u) return;  // inactive sample contributes nothing anywhere
        d0 = 0.f; d1 = 0.f; d2 = 0.f; d3 = 0.f;
        if (mask & 1u) d0 = dot_chunk(g, C::load(p0 + o0));
        if (mask & 2u) d1 = dot_chunk(g, C::load(p0 + o0 + csb));
        if (mask & 4u) d2 = dot_chunk(g, C::load(p0 + o2));
        if (mask & 8u) d3 = dot_chunk(g, C::load(p0 + o2 + csb));
        if (SCATTER) {
            if (mask & 1u) gr.red(gp0 + GS * o0, b.a0);
            if (mask & 2u) gr.red(gp0 + GS * (o0 + csb), b.a1);
            if (mask & 4u) gr.red(gp0 + GS * o2, b.a2);
            if (mask & 8u) gr.red(gp0 + GS * (o2 + csb), b.a3);
        }
    }
    pa = fmaf(b.w0, d0, fmaf(b.w1, d1, fmaf(b.w2, d2, fmaf(b.w3, d3, pa))));
    px = fmaf(b.hy, d1 - d0, fmaf(b.ly, d3 - d2, px));
    py = fmaf(b.hx, d2 - d0, fmaf(b.lx, d3 - d1, py));
}

// Which 16-byte chunk of the head slice a lane owns.  For fp32 D = 48 a 192-byte slice starts at byte
// 0 or 64 of a 128-byte line and spans two lines; a query whose 12 lanes straddle a warp boundary
// (8|4 or 4|8) would make one of the two warps touch BOTH lines.  Rotating the chunk assignment of
// those queries puts whole lines on each side of the boundary: 2.0 instead of 2.12 L1 wavefronts
// per gathered slice (and per vector reduction).  Results do not depend on it.
template <typename VT, int LANES>
__device__ __forceinline__ int lane_chunk(int tid, int lane, int m)
{
    if (LANES == 12 && sizeof(typename Chunk<VT>::elem) == 4 && Chunk<VT>::BYTES == 16) {
        const int k = 32 - ((tid - lane) & 31);     // lanes of this query before the next warp boundary
        if (k < 12) {                                // k is 4 or 8
            const bool odd = ((m * LANES * 16) & 127) != 0;  // slice starts mid-line
            const int rot = odd ? (k == 8 ? 4 : 0) : (k == 8 ? 0 : 8);
            const int c = lane + rot;
            return c >= 12 ? c - 12 : c;
        }
    }
    return lane;
}

// Queries per CTA tile for D = 48.  The tuned default is 16; when that would leave the GPU with
// fewer than ~3 CTAs per SM (decoder: Lq = 60) halve the tile so twice as many CTAs are in flight
// -- those launches are latency-bound, not bandwidth-bound.
// benchmark knob: tile length from the environment (8, 16 or 32; anything else = the tuned 16)
inline int env_tile_pairs(const char *name)
{
    const char *e = getenv(name);
    if (e == nullptr) return 16;
    const int v = atoi(e);
    return (v == 8 || v == 16 || v == 32) ? v : 16;
}

inline int pick_pairs_d48(int configured, int Lq, int M, int nz)
{
    if (configured != 16) return configured;
    const long long ctas = (long long)((Lq + 15) / 16) * M * nz;
    return ctas < 148 * 3 ? 8 : 16;
}

// sum over the G (= 2 or 4) lanes of a shuffle sub-group (full-warp participation required)
template <int G>
__device__ __forceinline__ void subgroup_sum3(float &a, float &b, float &c)
{
    a += __shfl_xor_sync(0xffffffffu, a, 1);
    b += __shfl_xor_sync(0xffffffffu, b, 1);
    c += __shfl_xor_sync(0xffffffffu, c, 1);
    if (G == 4) {
        a += __shfl_xor_sync(0xffffffffu, a, 2);
        b += __shfl_xor_sync(0xffffffffu, b, 2);
        c += __shfl_xor_sync(0xffffffffu, c, 2);
    }
}

// lanes per shuffle sub-group for a pair of LANES lanes (pairs never straddle a sub-group)
__host__ __device__ constexpr int sub_group(int lanes) { return lanes % 4 == 0 ? 4 : 2; }

}  // namespace msda
