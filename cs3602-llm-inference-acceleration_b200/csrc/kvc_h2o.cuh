// kvc_h2o.cuh — H2O attention-score bookkeeping (kvc_h2o_accumulate, include/kvc.h).
//
// Replaces, per layer, the reference manager's attn.sum(dim=2), acc * decay, zeros + cat, acc + mass
// (h2o_attention.py:78-151) and the head sum of get_heavy_hitter_indices (:194-213) with one pass over the
// attention probabilities.  One CTA owns one (layer, batch entry, column tile of keys) and walks every head of
// that batch entry, so the head sum of the updated accumulators is complete when the walk ends: no second pass,
// no atomics, and a fixed summation order.
//
// Work split inside a CTA (16 warps): heads go in groups of G, each head of a group gets 16/G warps, and those
// warps split the queries into contiguous blocks (block s = queries [s*qb, (s+1)*qb), qb = ceil(n_query / (16/G))).
// G is chosen per layer from n_query: decode (n_query = 1) runs 16 heads side by side, prefill-sized n_query one
// head at a time with 16 query blocks in flight.  Summation order, fixed for a given n_query:
//   per column: each block sums its queries in ascending q (fp32), the blocks are added in ascending s (fp32),
//   the result is rounded once to the attention dtype (torch: one rounding of the fp32 sum);
//   the head sum adds the rounded accumulators in ascending h (fp32) and rounds once.
// A lane owns 16 consecutive bytes of a row (8 bf16/f16 or 4 fp32 columns), a warp 512 bytes: rows whose start is
// 16-byte aligned (strides and base pointer) are read with 16-byte streaming loads, others (HF eager attention rows
// of key_len * e bytes, rarely a multiple of 16) with element loads of the same columns.
#pragma once
#include "kvc_device.cuh"

namespace kvc {

constexpr int kH2oThreads = 512;
constexpr int kH2oWarps = kH2oThreads / 32;

struct H2oLayerDev {
    const char* attn;        // nullptr: re-score only
    int64_t asb, ash, asq;   // BYTE strides of attn (batch, head, query)
    char* acc;
    int64_t csb, csh;        // BYTE strides of acc (batch, head)
    char* score;             // [B, hi - lo] or nullptr
    int32_t Q, K, prev, lo, hi;
    int32_t vec;             // 1: every attn row starts on a 16-byte boundary
};

struct H2oBatchDev {
    int32_t B, H;
    float decay;
    int32_t pad;
    H2oLayerDev layers[KVC_MAX_LAYERS_PER_LAUNCH];
};

template <int DT>
__global__ void __launch_bounds__(kH2oThreads) kvc_h2o_accumulate_kernel(const __grid_constant__ H2oBatchDev bd) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    constexpr int E = Tr::kElemBytes;
    constexpr int VEC = 16 / E;      // columns per lane
    constexpr int TC = 32 * VEC;     // columns per CTA
    __shared__ float part[kH2oWarps][TC];  // per-warp query-block sums of the current head group
    __shared__ float upd[kH2oWarps][TC];   // updated accumulators of the current head group (rounded)

    const H2oLayerDev& L = bd.layers[blockIdx.z];
    const int b = blockIdx.y;
    const int j0 = blockIdx.x * TC;
    const int K = L.K;
    if (j0 >= K) return;  // block-uniform: layers of one launch may differ in key_len
    const int H = bd.H, Q = L.Q;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool update = L.attn != nullptr;
    const int prev = (L.prev < 0 || L.prev > K) ? 0 : L.prev;  // the reference's reset when the cache shrank

    // query blocks per head: the largest power of two <= n_query, at most 16 (block-uniform)
    int qs = 1;
    while (qs < kH2oWarps && qs * 2 <= Q) qs *= 2;
    if (!update) qs = kH2oWarps;
    const int G = kH2oWarps / qs;  // heads per group
    const int g_w = warp / qs, s_w = warp - g_w * qs;
    const int qb = (Q + qs - 1) / qs;
    const int qa = min(Q, s_w * qb), qe = min(Q, qa + qb);
    const int c0 = j0 + lane * VEC;  // first column of this lane
    const bool lane_vec = L.vec && c0 + VEC <= K;

    float hsum = 0.f;  // head sum of column j0 + tid (tid < TC)
    for (int h0 = 0; h0 < H; h0 += G) {
        if (update) {
            float v[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) v[i] = 0.f;
            const int h = h0 + g_w;
            if (h < H && qa < qe) {
                const char* row = L.attn + (int64_t)b * L.asb + (int64_t)h * L.ash + (int64_t)qa * L.asq;
                const int n = qe - qa;
                if (lane_vec) {
                    const char* p = row + (int64_t)c0 * E;
                    int q = 0;
                    for (; q + 4 <= n; q += 4) {  // four rows in flight per lane
                        int4 x[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) x[u] = ldg128_stream(p + (int64_t)(q + u) * L.asq);
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const uint32_t w[4] = {(uint32_t)x[u].x, (uint32_t)x[u].y, (uint32_t)x[u].z, (uint32_t)x[u].w};
#pragma unroll
                            for (int i = 0; i < VEC; ++i) {
                                const uint32_t raw = E == 4 ? w[i] : ((w[i / 2] >> (16 * (i & 1))) & 0xffffu);
                                v[i] += Tr::from_raw(raw);
                            }
                        }
                    }
                    for (; q < n; ++q) {
                        const int4 x = ldg128_stream(p + (int64_t)q * L.asq);
                        const uint32_t w[4] = {(uint32_t)x.x, (uint32_t)x.y, (uint32_t)x.z, (uint32_t)x.w};
#pragma unroll
                        for (int i = 0; i < VEC; ++i) {
                            const uint32_t raw = E == 4 ? w[i] : ((w[i / 2] >> (16 * (i & 1))) & 0xffffu);
                            v[i] += Tr::from_raw(raw);
                        }
                    }
                } else if (c0 < K) {
                    const Key* p = reinterpret_cast<const Key*>(row) + c0;
                    const int nc = min(VEC, K - c0);
                    for (int q = 0; q < n; ++q) {
                        const Key* r = reinterpret_cast<const Key*>(reinterpret_cast<const char*>(p) + (int64_t)q * L.asq);
                        Key x[VEC];
#pragma unroll
                        for (int i = 0; i < VEC; ++i) x[i] = i < nc ? __ldg(r + i) : (Key)0;
#pragma unroll
                        for (int i = 0; i < VEC; ++i) v[i] += Tr::from_raw((uint32_t)x[i]);
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < VEC; ++i) part[warp][lane * VEC + i] = v[i];
        }
        __syncthreads();
        // combine the query blocks, update the accumulators of the group's heads
        for (int t = tid; t < G * TC; t += kH2oThreads) {
            const int gi = t / TC, c = t - gi * TC;
            const int h = h0 + gi, j = j0 + c;
            float a = 0.f;
            if (h < H && j < K) {
                Key* ap = reinterpret_cast<Key*>(L.acc + (int64_t)b * L.csb + (int64_t)h * L.csh) + j;
                if (update) {
                    float m = part[gi * qs][c];
                    for (int s = 1; s < qs; ++s) m = __fadd_rn(m, part[gi * qs + s][c]);
                    m = round_dt<DT>(m);
                    // torch: (prev * decay) rounds, then (+ mass) rounds; __fmul_rn / __fadd_rn keep fp32 from
                    // contracting the two into one FMA
                    a = j < prev ? round_dt<DT>(__fadd_rn(round_dt<DT>(__fmul_rn(Tr::from_raw((uint32_t)*ap), bd.decay)), m))
                                 : m;
                    *ap = (Key)Tr::to_raw(a);
                } else {
                    a = Tr::from_raw((uint32_t)*ap);
                }
            }
            upd[gi][c] = a;
        }
        __syncthreads();
        if (tid < TC) {
            const int n = min(G, H - h0);
            for (int gi = 0; gi < n; ++gi) hsum = (h0 == 0 && gi == 0) ? upd[0][tid] : __fadd_rn(hsum, upd[gi][tid]);
        }
        // the next group writes part[] only after every thread has passed the barrier above, and upd[] only after
        // the first barrier of the next group: the reads of this group are complete by then
    }
    const int j = j0 + tid;
    if (L.score != nullptr && tid < TC && j >= L.lo && j < L.hi)
        reinterpret_cast<Key*>(L.score)[(int64_t)b * (L.hi - L.lo) + (j - L.lo)] = (Key)Tr::to_raw(hsum);
}

}  // namespace kvc
