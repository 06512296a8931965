// Pieces shared by the fused snippet kernels (msda_snippet.cu: cell-major value / slots; msda_planar.cu: planar
// slots): launch arguments, the neighbour-frame range of a query frame, in-kernel encoder reference points and
// phase 1 (one thread per sample: biases, softmax, offset normalisation, bilinear set-up -> one 16-byte record).
#pragma once

#include "msda_fast.cuh"
#include "msda_internal.h"

namespace msda {

struct SnipArgs {
    SnippetDims d;
    int cell_bytes;            // M * D * sizeof(VT)
    unsigned magic_LP, magic_P;
    int n_local, n_slots;      // presummed: slot of query frame t1 = t1 < n_frame ? t1 : n_local
    int tile2d;                // planar kernels, Lq == S: CTA query slots walk 2-D pixel patches (msda_planar.cu tile_query)
};

__device__ __forceinline__ void frame_range(int t1, int n_frame, int T2, int &lo, int &hi)
{
    // reference ms_deform_attn.py:137-140 (observed frames) and :189,201 (future frames)
    if (t1 < n_frame) { lo = max(t1 - 1, 0); hi = min(t1 + 1, n_frame - 1); }
    else { lo = 0; hi = T2 - 1; }
}

// Encoder reference points as a function of the query index (reference get_reference_points,
// deformable_transformer.py:219-232): query q is pixel (y, x) of level lq; its reference point on level l is
//     ( (x + 0.5) / (vr[n,lq,0] * W_lq) * vr[n,l,0],  (y + 0.5) / (vr[n,lq,1] * H_lq) * vr[n,l,1] )
// -- same operations in the same order as the torch code (linspace(0.5, W - 0.5, W) is exactly x + 0.5), so the
// result is bit-identical to the tensor the reference materialises and re-reads in every layer.
__device__ __forceinline__ float2 analytic_reference_point(const LevelTable &lv, const float *__restrict__ vr, int L,
                                                           int q, int l)
{
    int lq = 0;
    while (lq + 1 < L && q >= lv.start[lq + 1]) ++lq;
    const int Wq = max(lv.W[lq], 1);
    const int r = q - lv.start[lq];
    const int y = r / Wq, x = r - y * Wq;
    const float rx = ((float)x + 0.5f) / (__ldg(vr + 2 * lq) * (float)lv.W[lq]);
    const float ry = ((float)y + 0.5f) / (__ldg(vr + 2 * lq + 1) * (float)lv.H[lq]);
    return make_float2(rx * __ldg(vr + 2 * l), ry * __ldg(vr + 2 * l + 1));
}

// Phase 1 of both kernels: one thread per sample.  Softmax over the L*P logits of each query (staged in
// shared memory), then loc = ref + offset / (W_l, H_l) in the reference's operation order
// (ms_deform_attn.py:164-165).
// Each sample is parked as ONE 16-byte record {lx, ly, A, off | mask}: A = softmax / k, `off` the
// byte offset of the (y0,x0) cell (a multiple of 16, so its low four bits carry the corner mask).
// One LDS.128 per sample and lane in phase 2 instead of an LDS.64 + an LDS.128 -- wide shared loads
// cost one L1 wavefront per quarter warp, and the L1 data pipe is what bounds these kernels
// (profiles/r01_run18_*); the row stride comes from the level table once per level, and the four
// corner weights are recomputed per lane (8 FP instructions, the issue slots are free).
template <int THREADS, int PAIRS>
__device__ __forceinline__ void snippet_phase1(float4 *rec, float *zs, LevelTable &lv, const int64_t *__restrict__ shapes,
                                               const int64_t *__restrict__ lsi, const SnipArgs &a, int n, int t1,
                                               int q0, int m, size_t qbase, const float *__restrict__ offsets,
                                               const float *__restrict__ logits,
                                               const float *__restrict__ ref, float inv_k)
{
    const SnippetDims &d = a.d;
    const int tid = threadIdx.x;
    const int LP = d.L * d.P;
    // pass 1: EVERY global load of the tile is issued here, back to back -- the level table, the logits, the
    // offsets and the reference points -- so the CTA waits for one memory round trip, not three in a row
    // (the projection rows stream from HBM, and with the neighbour-frame loop gone the set-up is ~40 % of a CTA's
    // life).  Raw {off.x, off.y, ref.u, ref.v} is parked in the record slot until pass 2.
    load_level_table(lv, shapes, lsi, d.L, d.S);
    for (int i = tid; i < PAIRS * LP; i += THREADS) {
        const int spl = fast_div(i, a.magic_LP);
        const int q = q0 + spl;
        const int lp = i - spl * LP;
        float z = 0.f;
        float4 raw = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q < d.Lq) {
            z = __ldg(logits + (qbase + q) * d.logit_row_stride + m * LP + lp);
            const float2 o = __ldg(reinterpret_cast<const float2 *>(offsets + (qbase + q) * d.off_row_stride) + m * LP + lp);
            raw = make_float4(o.x, o.y, 0.f, 0.f);
            if (d.valid_ratios == nullptr) {
                const int l = fast_div(lp, a.magic_P);
                const float *rp = ref + n * d.ref_stride_n + t1 * d.ref_stride_t + ((int64_t)q * d.L + l) * 2;
                raw.z = __ldg(rp);
                raw.w = __ldg(rp + 1);
            }
            if (d.logit_bias != nullptr) z += __ldg(d.logit_bias + m * LP + lp);
            if (d.off_bias != nullptr) {
                const float2 b = __ldg(reinterpret_cast<const float2 *>(d.off_bias) + m * LP + lp);
                raw.x += b.x; raw.y += b.y;
            }
        }
        zs[i] = z;
        rec[i + spl] = raw;  // records strided LP + 1 per query
    }
    __syncthreads();
    // pass 2: softmax over the query's L*P logits (every thread redoes the L*P exponentials of its query: a few
    // hundred MUFU ops per CTA, cheaper than a third barrier + a second staging array), then the sample set-up
    for (int i = tid; i < PAIRS * LP; i += THREADS) {
        const int spl = fast_div(i, a.magic_LP);
        const int lp = i - spl * LP;
        float4 r = empty_record();  // mask 0: inactive
        if (q0 + spl < d.Lq) {
            const float *z = zs + spl * LP;
            float mx = z[0];
            for (int j = 1; j < LP; ++j) mx = fmaxf(mx, z[j]);
            float sum = 0.f;
            for (int j = 0; j < LP; ++j) sum += expf(z[j] - mx);
            const float at = expf(z[lp] - mx) / sum * inv_k;
            const int l = fast_div(lp, a.magic_P);
            float4 raw = rec[i + spl];
            if (d.valid_ratios != nullptr) {
                const float2 rp = analytic_reference_point(lv, d.valid_ratios + (size_t)n * d.L * 2, d.L, q0 + spl, l);
                raw.z = rp.x;
                raw.w = rp.y;
            }
            const float u = raw.z + raw.x / (float)lv.W[l];
            const float v = raw.w + raw.y / (float)lv.H[l];
            const Sample<float> s = make_sample<float>(u, v, lv.H[l], lv.W[l], lv.start[l]);
            r = make_record(s, at, a.cell_bytes);
        }
        rec[i + spl] = r;
    }
    __syncthreads();
}

template <typename VT>
inline SnipArgs make_snip_args(const SnippetDims &d)
{
    SnipArgs a;
    a.d = d;
    a.cell_bytes = d.M * d.D * (int)sizeof(typename Chunk<VT>::elem);
    a.magic_LP = fast_magic(d.L * d.P);
    a.magic_P = fast_magic(d.P);
    a.n_local = d.T1 < d.n_frame ? d.T1 : d.n_frame;
    a.n_slots = snippet_num_slots(d.T1, d.n_frame);
    a.tile2d = 0;
    return a;
}

}  // namespace msda
