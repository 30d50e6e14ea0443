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
#include "kvc_tma.cuh"

namespace kvc {

constexpr int kH2oThreads = 512;
constexpr int kH2oWarps = kH2oThreads / 32;

// ---------------------------------------------------------------- the accumulator update both entry points share
// One (head, column) of the update: mass is the fp32 query sum, rounded once here; torch rounds (acc * decay), then
// (+ mass).  __fmul_rn / __fadd_rn keep fp32 from contracting the two into one FMA.  Returns the updated value.
template <int DT>
__device__ __forceinline__ float h2o_update_acc(typename Traits<DT>::Key* ap, float mass, int j, int prev, float decay) {
    using Tr = Traits<DT>;
    const float m = round_dt<DT>(mass);
    const float a = j < prev ? round_dt<DT>(__fadd_rn(round_dt<DT>(__fmul_rn(Tr::from_raw((uint32_t)*ap), decay)), m)) : m;
    *ap = (typename Tr::Key)Tr::to_raw(a);
    return a;
}
// Head sum of the updated accumulators, ascending h (fp32).
__device__ __forceinline__ float h2o_head_sum(float hsum, float a, int h) { return h == 0 ? a : __fadd_rn(hsum, a); }
// score_out[b, j - lo] = round(head sum), lo <= j < hi.
template <int DT>
__device__ __forceinline__ void h2o_store_score(char* score, int b, int j, int lo, int hi, float hsum) {
    if (score != nullptr && j >= lo && j < hi)
        reinterpret_cast<typename Traits<DT>::Key*>(score)[(int64_t)b * (hi - lo) + (j - lo)] =
            (typename Traits<DT>::Key)Traits<DT>::to_raw(hsum);
}

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
                    a = h2o_update_acc<DT>(ap, m, j, prev, bd.decay);
                } else {
                    a = Tr::from_raw((uint32_t)*ap);
                }
            }
            upd[gi][c] = a;
        }
        __syncthreads();
        if (tid < TC) {
            const int n = min(G, H - h0);
            for (int gi = 0; gi < n; ++gi) hsum = h2o_head_sum(hsum, upd[gi][tid], h0 + gi);
        }
        // the next group writes part[] only after every thread has passed the barrier above, and upd[] only after
        // the first barrier of the next group: the reads of this group are complete by then
    }
    if (tid < TC) h2o_store_score<DT>(L.score, b, j0 + tid, L.lo, L.hi, hsum);
}

// ================================================================ kvc_h2o_accumulate_qk: the mass from q and K
// The probabilities are not read: they are rebuilt from the post-RoPE queries and the cached keys (include/kvc.h),
//   s[t,j] = scaling * sum_d fp32(q[t,d]) * fp32(k[j,d])       (one fmaf chain in ascending d, then one multiply)
//   p[t,j] = round(exp(s[t,j] - lse[t]))  where visible, 0 elsewhere,
// and handed to the update above.  Two launches:
//   pass 1, kvc_h2o_qk_stats_kernel: grid (key split x query tile, b * Hkv, layer).  A CTA streams the K rows of its
//     split through shared memory (bulk copies, two buffers) and keeps kQkQ1 queries of the KV head's G * T on chip;
//     thread r owns row r of every 128-row tile and a running (max, sum exp) per query, and the 128 partials of a query
//     are merged in a fixed tree.  Out: (max, sum exp) per (b, hk, query, split) in the workspace.
//   pass 2, kvc_h2o_qk_accumulate_kernel: grid (128-column tile, b, layer), as kvc_h2o_accumulate.  Per KV head the
//     CTA loads its K tile once; the G heads x T queries of the group reuse it.  A query chunk's lse is combined from
//     the split partials in ascending split order, thread r forms p for column j0 + r, sums it over t in ascending t,
//     and runs the shared tail (h2o_update_acc, h2o_head_sum, h2o_store_score).
// Both passes compute s with qk_logits from the same shared-memory copies, so they agree bit for bit.  Every split
// and tile decision depends on key_len, T, G, D and the dtype only: the bits do not depend on B, on the other layers
// of the launch or on the device.  Without a mask query t sees keys j <= key_len - T + t; tiles no query of the CTA
// sees are skipped.
constexpr int kQkThreads = 128;  // threads of both passes; one K row (pass 1) or one key column (pass 2) each
constexpr int kQkRows = 128;     // K rows per tile
constexpr int kQkQ1 = 16;        // queries per pass-1 CTA
constexpr int kQkQ2 = 32;        // queries per pass-2 chunk
constexpr int kQkMaxSplits = 32;  // key splits of pass 1
constexpr int kQkMaxRowBytes = 512;

struct H2oQkLayerDev {
    const char* q;
    int64_t qsb, qsh, qst;   // BYTE strides of q (batch, head, query)
    const char* k;
    int64_t ksb, ksh, kss;   // BYTE strides of K (batch, head, row)
    const uint8_t* mask;     // [B, T, key_len] bool or nullptr (causal)
    int64_t msb, mst;
    char* acc;
    int64_t csb, csh;        // BYTE strides of acc (batch, head)
    char* score;             // [B, hi - lo] or nullptr
    float2* ws;              // [B * Hkv, G * T, n_split] (max, sum exp) partials of pass 1
    float scaling;
    int32_t T, K, prev, lo, hi;
    int32_t n_split, split_tiles;  // pass-1 key splits, 128-row tiles per split
    int32_t n_qt;                  // pass-1 query tiles
    int32_t pad;
};

struct H2oQkBatchDev {
    int32_t B, Hkv, G, D;
    float decay;
    int32_t pitch;  // bytes between K rows in shared memory: an odd number of 16-byte units (no bank conflicts)
    H2oQkLayerDev layers[KVC_MAX_LAYERS_PER_LAUNCH];
};

template <int DT>
__device__ __forceinline__ void unpack16(int4 x, float* f) {
    const uint32_t w[4] = {(uint32_t)x.x, (uint32_t)x.y, (uint32_t)x.z, (uint32_t)x.w};
    if (DT == KVC_DTYPE_F32) {
#pragma unroll
        for (int i = 0; i < 4; ++i) f[i] = __uint_as_float(w[i]);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = Traits<DT>::from_raw((w[i / 2] >> (16 * (i & 1))) & 0xffffu);
    }
}

// s[u] = scaling * <q_u, k> for QT queries (fp32 rows of D in shared memory, D apart) and one K row in shared memory.
template <int DT, int QT>
__device__ __forceinline__ void qk_logits(const float* qs, int D, const char* krow, float scaling, float* s) {
    constexpr int VEC = 16 / Traits<DT>::kElemBytes;
    float acc[QT];
#pragma unroll
    for (int u = 0; u < QT; ++u) acc[u] = 0.f;
    for (int c = 0; c < D / VEC; ++c) {
        float kf[VEC];
        unpack16<DT>(*reinterpret_cast<const int4*>(krow + c * 16), kf);
#pragma unroll
        for (int u = 0; u < QT; ++u) {
            const float4* qp = reinterpret_cast<const float4*>(qs + u * D + c * VEC);
#pragma unroll
            for (int v = 0; v < VEC / 4; ++v) {
                const float4 qv = qp[v];
                acc[u] = fmaf(qv.x, kf[4 * v + 0], acc[u]);
                acc[u] = fmaf(qv.y, kf[4 * v + 1], acc[u]);
                acc[u] = fmaf(qv.z, kf[4 * v + 2], acc[u]);
                acc[u] = fmaf(qv.w, kf[4 * v + 3], acc[u]);
            }
        }
    }
#pragma unroll
    for (int u = 0; u < QT; ++u) s[u] = __fmul_rn(acc[u], scaling);
}

// (m, l) <- the (max, sum exp) of the union of two partials.
__device__ __forceinline__ void lse_merge(float& m, float& l, float m2, float l2) {
    const float M = fmaxf(m, m2);
    if (M == -INFINITY) return;
    l = __fadd_rn(__fmul_rn(l, expf(m - M)), __fmul_rn(l2, expf(m2 - M)));
    m = M;
}

__device__ __forceinline__ bool qk_visible(const H2oQkLayerDev& L, int b, int t, int j) {
    return L.mask ? L.mask[(int64_t)b * L.msb + (int64_t)t * L.mst + j] != 0 : j <= L.K - L.T + t;
}

// q[b, hk * G + g, t, :] of flattened queries -> fp32 rows in shared memory; rows [n, n_pad) are zeroed.
template <int DT>
__device__ __forceinline__ void qk_load_queries(const H2oQkLayerDev& L, int b, int hk, int G, int D, int n, int n_pad,
                                                int first, int t_lo, int nt, float* qs) {
    using Key = typename Traits<DT>::Key;
    for (int idx = threadIdx.x; idx < n_pad * D; idx += kQkThreads) {
        const int a = idx / D, d = idx - a * D;
        float v = 0.f;
        if (a < n) {
            const int f = first + a, g = f / nt, t = t_lo + (f - g * nt);
            const char* row = L.q + (int64_t)b * L.qsb + (int64_t)(hk * G + g) * L.qsh + (int64_t)t * L.qst;
            v = Traits<DT>::from_raw((uint32_t)__ldg(reinterpret_cast<const Key*>(row) + d));
        }
        qs[idx] = v;
    }
}

// Warp 0 issues the bulk copies of rows [r0, r0 + n) of K head hk into a tile buffer.
__device__ __forceinline__ void qk_issue_tile(const H2oQkLayerDev& L, int b, int hk, int r0, int n, int rb, int pitch,
                                              char* buf, uint32_t bar) {
    const int lane = threadIdx.x & 31;
    if (lane == 0) {
        fence_proxy_async_smem();  // the generic-proxy reads of this buffer's last use come first
        mbar_arrive_expect_tx(bar, (uint32_t)(n * rb));
    }
    __syncwarp();
    const char* src = L.k + (int64_t)b * L.ksb + (int64_t)hk * L.ksh;
    for (int r = lane; r < n; r += 32) bulk_g2s(smem_u32(buf + r * pitch), src + (int64_t)(r0 + r) * L.kss, rb, bar);
}

template <int DT, int QT>
__global__ void __launch_bounds__(kQkThreads) kvc_h2o_qk_stats_kernel(const __grid_constant__ H2oQkBatchDev bd) {
    const H2oQkLayerDev& L = bd.layers[blockIdx.z];
    const int qt = blockIdx.x / L.n_split, sp = blockIdx.x - qt * L.n_split;
    if (qt >= L.n_qt) return;  // block-uniform: layers of one launch differ in shape
    extern __shared__ __align__(128) unsigned char smem[];
    const int G = bd.G, D = bd.D, T = L.T, K = L.K, GT = G * T, pitch = bd.pitch;
    const int rb = D * Traits<DT>::kElemBytes;
    const int bh = blockIdx.y, b = bh / bd.Hkv, hk = bh - b * bd.Hkv;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int i0 = qt * kQkQ1, nq = min(kQkQ1, GT - i0), nq_pad = (nq + QT - 1) / QT * QT;
    const int k0 = sp * L.split_tiles * kQkRows;
    int k1 = min(K, k0 + L.split_tiles * kQkRows);
    if (!L.mask) {  // the last key the CTA's latest query sees
        int tmax = 0;
        for (int a = 0; a < nq; ++a) tmax = max(tmax, (i0 + a) % T);
        k1 = min(k1, K - T + tmax + 1);
    }
    const int n_tiles = k1 > k0 ? (k1 - k0 + kQkRows - 1) / kQkRows : 0;

    uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
    char* kbuf = reinterpret_cast<char*>(smem + 128);
    float* qs = reinterpret_cast<float*>(kbuf + 2 * kQkRows * pitch);
    float* st_m = qs + kQkQ1 * D;  // [kQkQ1][kQkThreads] running max per (query, thread)
    float* st_l = st_m + kQkQ1 * kQkThreads;
    if (tid == 0) {
        mbar_init(smem_u32(&bars[0]), 1);
        mbar_init(smem_u32(&bars[1]), 1);
        mbar_init_fence();
    }
    qk_load_queries<DT>(L, b, hk, G, D, nq, nq_pad, i0, 0, T, qs);
    for (int a = 0; a < nq; ++a) {
        st_m[a * kQkThreads + tid] = -INFINITY;
        st_l[a * kQkThreads + tid] = 0.f;
    }
    __syncthreads();
    if (warp == 0 && n_tiles > 0)
        qk_issue_tile(L, b, hk, k0, min(kQkRows, k1 - k0), rb, pitch, kbuf, smem_u32(&bars[0]));
    for (int it = 0; it < n_tiles; ++it) {
        const int kt = k0 + it * kQkRows;
        if (warp == 0 && it + 1 < n_tiles)
            qk_issue_tile(L, b, hk, kt + kQkRows, min(kQkRows, k1 - kt - kQkRows), rb, pitch,
                          kbuf + ((it + 1) & 1) * kQkRows * pitch, smem_u32(&bars[(it + 1) & 1]));
        mbar_wait(smem_u32(&bars[it & 1]), (it >> 1) & 1);
        const int j = kt + tid;
        if (j < k1) {
            const char* krow = kbuf + (it & 1) * kQkRows * pitch + tid * pitch;
            for (int a0 = 0; a0 < nq; a0 += QT) {
                float s[QT];
                qk_logits<DT, QT>(qs + a0 * D, D, krow, L.scaling, s);
#pragma unroll
                for (int u = 0; u < QT; ++u) {
                    const int a = a0 + u;
                    if (a < nq && qk_visible(L, b, (i0 + a) % T, j)) {
                        float m = st_m[a * kQkThreads + tid], l = st_l[a * kQkThreads + tid];
                        if (s[u] > m) {
                            l = __fadd_rn(__fmul_rn(l, expf(m - s[u])), 1.f);
                            m = s[u];
                        } else {
                            l = __fadd_rn(l, expf(s[u] - m));
                        }
                        st_m[a * kQkThreads + tid] = m;
                        st_l[a * kQkThreads + tid] = l;
                    }
                }
            }
        }
        __syncthreads();  // the buffer is free for the copy two tiles ahead
    }
    // merge the 128 partials of each query: 4 in ascending thread order per lane, then a butterfly over the lanes
    for (int a = warp; a < nq; a += kQkThreads / 32) {
        float m = -INFINITY, l = 0.f;
#pragma unroll
        for (int r = 0; r < kQkThreads / 32; ++r) lse_merge(m, l, st_m[a * kQkThreads + lane + 32 * r],
                                                           st_l[a * kQkThreads + lane + 32 * r]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float m2 = __shfl_xor_sync(0xffffffffu, m, o), l2 = __shfl_xor_sync(0xffffffffu, l, o);
            lse_merge(m, l, m2, l2);
        }
        if (lane == 0) L.ws[((int64_t)bh * GT + i0 + a) * L.n_split + sp] = make_float2(m, l);
    }
}

template <int DT, int QT>
__global__ void __launch_bounds__(kQkThreads) kvc_h2o_qk_accumulate_kernel(const __grid_constant__ H2oQkBatchDev bd) {
    using Key = typename Traits<DT>::Key;
    const H2oQkLayerDev& L = bd.layers[blockIdx.z];
    const int b = blockIdx.y;
    const int j0 = blockIdx.x * kQkRows;
    const int K = L.K;
    if (j0 >= K) return;  // block-uniform
    extern __shared__ __align__(128) unsigned char smem[];
    const int G = bd.G, D = bd.D, Hkv = bd.Hkv, T = L.T, GT = G * T, pitch = bd.pitch;
    constexpr int E = Traits<DT>::kElemBytes;
    const int rb = D * E;
    const int tid = threadIdx.x;
    const int prev = (L.prev < 0 || L.prev > K) ? 0 : L.prev;  // the reference's reset when the cache shrank
    const int t_lo = L.mask ? 0 : max(0, j0 - (K - T));         // earlier queries see no key of this tile
    const int nt = T - t_lo, n_act = G * nt;
    const int nrows = min(kQkRows, K - j0);
    const int j = j0 + tid;
    const bool col = j < K;

    uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
    char* kbuf = reinterpret_cast<char*>(smem + 128);
    float* qs = reinterpret_cast<float*>(kbuf + 2 * kQkRows * pitch);
    float* lse = qs + kQkQ2 * D;
    if (tid == 0) {
        mbar_init(smem_u32(&bars[0]), 1);
        mbar_init(smem_u32(&bars[1]), 1);
        mbar_init_fence();
    }
    __syncthreads();
    if (tid < 32) qk_issue_tile(L, b, 0, j0, nrows, rb, pitch, kbuf, smem_u32(&bars[0]));
    float hsum = 0.f;
    for (int hk = 0; hk < Hkv; ++hk) {
        if (tid < 32 && hk + 1 < Hkv)
            qk_issue_tile(L, b, hk + 1, j0, nrows, rb, pitch, kbuf + ((hk + 1) & 1) * kQkRows * pitch,
                          smem_u32(&bars[(hk + 1) & 1]));
        const char* krow = kbuf + (hk & 1) * kQkRows * pitch + tid * pitch;
        const float2* part = L.ws + (int64_t)(b * Hkv + hk) * GT * L.n_split;
        int g_cur = 0;
        float mass = 0.f;
        auto finish_head = [&](int g) {  // the tail of kvc_h2o_accumulate for head hk * G + g, column j
            const int h = hk * G + g;
            Key* ap = reinterpret_cast<Key*>(L.acc + (int64_t)b * L.csb + (int64_t)h * L.csh) + j;
            hsum = h2o_head_sum(hsum, h2o_update_acc<DT>(ap, mass, j, prev, bd.decay), h);
            mass = 0.f;
        };
        for (int c0 = 0; c0 < n_act; c0 += kQkQ2) {
            const int nc = min(kQkQ2, n_act - c0), nc_pad = (nc + QT - 1) / QT * QT;
            qk_load_queries<DT>(L, b, hk, G, D, nc, nc_pad, c0, t_lo, nt, qs);
            if (tid < nc) {  // lse of the chunk's queries: the split partials in ascending split order
                const int f = c0 + tid, g = f / nt, t = t_lo + (f - g * nt);
                const float2* pp = part + (int64_t)(g * T + t) * L.n_split;
                float2 x[kQkMaxSplits];  // every load in flight at once, then the merge in ascending split order
#pragma unroll
                for (int s = 0; s < kQkMaxSplits; ++s) x[s] = s < L.n_split ? __ldg(pp + s) : make_float2(-INFINITY, 0.f);
                float m = -INFINITY, l = 0.f;
#pragma unroll
                for (int s = 0; s < kQkMaxSplits; ++s) lse_merge(m, l, x[s].x, x[s].y);
                lse[tid] = l > 0.f ? m + logf(l) : INFINITY;  // no visible key: every p is 0
            }
            __syncthreads();
            if (c0 == 0) mbar_wait(smem_u32(&bars[hk & 1]), (hk >> 1) & 1);
            if (col) {
                for (int a0 = 0; a0 < nc; a0 += QT) {
                    float s[QT];
                    qk_logits<DT, QT>(qs + a0 * D, D, krow, L.scaling, s);
#pragma unroll
                    for (int u = 0; u < QT; ++u) {
                        const int a = a0 + u;
                        if (a < nc) {
                            const int f = c0 + a, g = f / nt, t = t_lo + (f - g * nt);
                            while (g_cur < g) finish_head(g_cur++);
                            if (qk_visible(L, b, t, j)) mass = __fadd_rn(mass, round_dt<DT>(expf(s[u] - lse[a])));
                        }
                    }
                }
            }
            __syncthreads();  // qs / lse are rewritten by the next chunk
        }
        if (n_act == 0) mbar_wait(smem_u32(&bars[hk & 1]), (hk >> 1) & 1);  // keep the barrier phases in step
        if (col)
            while (g_cur < G) finish_head(g_cur++);
        __syncthreads();  // this K buffer is free for the copy of head hk + 2
    }
    if (col) h2o_store_score<DT>(L.score, b, j, L.lo, L.hi, hsum);
}

}  // namespace kvc
