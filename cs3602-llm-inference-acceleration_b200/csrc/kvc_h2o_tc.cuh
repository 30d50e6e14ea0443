// kvc_h2o_tc.cuh — the H2O query update on the 5th-generation tensor cores (kvc_h2o_accumulate_qk_tc, include/kvc.h).
//
// The same update as kvc_h2o_accumulate_qk (kvc_h2o.cuh) with the logits from `tcgen05.mma ... kind::f16` and the
// exponentials in the exp2 domain.  Both passes run one kernel body, kvc_h2o_tc_kernel<DT, CPR, COLS>: a CTA holds
// one FIXED 128-row operand tile (the MMA's A) and streams 128-row tiles of the other operand through a TMA ring (the
// MMA's B), so TMEM lane = a row of the fixed tile, TMEM column = a row of the streamed tile.
//
//   pass 1 (COLS = false), grid (query tile, b * Hkv, layer): the fixed tile holds the G query heads of KV head hk for
//     tb = 128 / G consecutive positions t (row g * tb + u = head hk*G + g, position qt*tb + u: one 4-D tensor-map box
//     over q), the stream is the key tiles up to the last key the tile's latest query sees.  Thread r keeps the online
//     (max, sum exp2) of row r and writes lse2 = max + log2(sum) to the workspace, [b * Hkv + hk][qt][r].
//   pass 2 (COLS = true), grid (key tile, b * Hkv, layer): the fixed tile holds 128 keys, the stream is the query tiles
//     that see any of them, each with its 128 lse2 values (one 512-byte bulk copy on the same mbarrier).  Thread r owns
//     key j0 + r: for every head g it adds round(exp2(fma(s, c, -lse2))) over ascending t, one __fadd_rn chain per
//     (head, key) kept in shared memory between tiles, then runs h2o_update_acc.  The score row is a third launch
//     (kvc_h2o_accumulate_kernel with attn = NULL), which sums the updated accumulators over all heads in ascending h.
//
// Warp roles (192 threads, two CTAs per SM): warps 0-3 the math (TMEM lanes 0-127), warp 4 lane 0 the TMA producer,
// warp 5 allocates TMEM and its lane 0 issues the MMAs into two 128-column accumulators.  Tiles that every row of the
// fixed tile sees in full (causal rule) run a mask-free instantiation of the math.  Every tile and loop bound depends
// on (key_len, T, G, D, dtype) only: the bits do not depend on B, on the other layers of the launch or on the device.
#pragma once
#include <type_traits>

#include "kvc_device.cuh"
#include "kvc_h2o.cuh"
#include "kvc_tcgen05.cuh"
#include "kvc_tma.cuh"

namespace kvc {

constexpr int kTcRows = 128;     // rows of every operand tile: the MMA is M = 128 x N = 128
constexpr int kTcThreads = 192;  // warps 0-3 math, warp 4 TMA producer, warp 5 TMEM owner + MMA issuer
constexpr int kTcAcc = 2;        // TMEM accumulators of kTcRows fp32 columns
constexpr int kTcLayers = 32;    // layers per launch: four tensor maps each, kernel parameters are limited to 32 KB
constexpr int kTcHead = 4096;    // barriers | lse2 of the ring slots (pass 2)

// One operand tile: CPR / 8 boxes of 128 rows x 128 B (128-byte swizzle) + for D = 80 one box of 128 rows x 32 B
// (32-byte swizzle), i.e. the K-major SW128 / SW32 UMMA layouts.
__host__ __device__ constexpr int tc_tile_bytes(int cpr) { return (cpr / 8) * kTcRows * 128 + (cpr % 8) * kTcRows * 16; }
// Ring slots: the fixed tile, the ring and the per-head masses of pass 2 stay near 110 KB, so two CTAs share an SM.
__host__ __device__ constexpr int tc_ring(int cpr) {
    return (110 * 1024 - kTcHead - tc_tile_bytes(cpr)) / tc_tile_bytes(cpr) > 6
               ? 6
               : (110 * 1024 - kTcHead - tc_tile_bytes(cpr)) / tc_tile_bytes(cpr);
}
// Dynamic shared memory of both passes: head, per-head masses (G x 128 fp32, pass 2), fixed tile, ring.
__host__ __device__ constexpr int tc_mass_bytes(int group) { return ((group * kTcRows * 4) + 1023) & ~1023; }
__host__ __device__ constexpr int tc_smem_bytes(int cpr, int group) {
    return kTcHead + tc_mass_bytes(group) + (1 + tc_ring(cpr)) * tc_tile_bytes(cpr);
}

struct H2oTcLayerDev {
    alignas(64) CUtensorMap qmap;       // q [B, Hq, T, D] as (D, T, Hq, B), box (64, tb, G, 1), SWIZZLE_128B
    alignas(64) CUtensorMap qmap_tail;  // D = 80: box (16, tb, G, 1), SWIZZLE_32B
    alignas(64) CUtensorMap kmap;       // K [B, Hkv, key_len, D] as (D, key_len, Hkv, B), box (64, 128, 1, 1)
    alignas(64) CUtensorMap kmap_tail;  // D = 80: box (16, 128, 1, 1)
    const uint8_t* mask;                // [B, T, key_len] bool or nullptr (causal)
    int64_t msb, mst;
    char* acc;
    int64_t csb, csh;                   // BYTE strides of acc (batch, head)
    float* lse;                         // workspace: [B * Hkv][n_qt][128] lse2 per row of a query tile
    float c2;                           // scaling * log2(e), rounded once
    int32_t T, K, prev, n_qt, n_kt;
};

struct H2oTcBatchDev {
    int32_t B, Hkv, G, tb;  // tb = 128 / G positions per query tile
    float decay;
    int32_t pad[3];
    H2oTcLayerDev layers[kTcLayers];
};
static_assert(sizeof(H2oTcBatchDev) < 32 * 1024, "kernel parameters are limited to 32 KB");

__device__ __forceinline__ bool tc_visible(const H2oTcLayerDev& L, int b, int t, int j) {
    return L.mask ? L.mask[(int64_t)b * L.msb + (int64_t)t * L.mst + j] != 0 : j <= L.K - L.T + t;
}

// UMMA descriptor of K step ks (16 elements) of the tile at `base`.
template <int CPR>
__device__ __forceinline__ uint64_t tc_desc(uint32_t base, int ks) {
    constexpr int KH = CPR / 8;
    return (ks >> 2) < KH ? umma_smem_desc_sw128(base + (ks >> 2) * (kTcRows * 128) + (ks & 3) * 32)
                          : umma_smem_desc_sw32(base + KH * (kTcRows * 128));
}

template <int DT, int CPR, bool COLS>
__global__ void __launch_bounds__(kTcThreads, 2) kvc_h2o_tc_kernel(const __grid_constant__ H2oTcBatchDev bd) {
    static_assert(DT != KVC_DTYPE_F32, "kind::f16 takes 16-bit operands");
    static_assert(CPR == 8 || CPR == 10 || CPR == 16, "head_dim 64, 80 or 128");
    using Key = typename Traits<DT>::Key;
    constexpr int KH = CPR / 8, REM = CPR % 8;
    constexpr int BOX = kTcRows * 128;
    constexpr int TILE = tc_tile_bytes(CPR);
    constexpr int RING = tc_ring(CPR);
    constexpr uint32_t IDESC = umma_idesc_f16(DT == KVC_DTYPE_BF16 ? 1 : 0, kTcRows, kTcRows);

    const H2oTcLayerDev& L = bd.layers[blockIdx.z];
    const int tile = blockIdx.x;
    if (tile >= (COLS ? L.n_kt : L.n_qt)) return;  // block-uniform: layers of one launch differ in shape
    const int bh = blockIdx.y, b = bh / bd.Hkv, hk = bh - b * bd.Hkv;
    const int G = bd.G, tb = bd.tb, T = L.T, K = L.K;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool causal = L.mask == nullptr;

    // the streamed tiles [i_lo, i_lo + n_items)
    int i_lo = 0, n_items;
    if (!COLS) {  // key tiles up to the last key the tile's latest query sees
        const int t_last = min(T - 1, tile * tb + tb - 1);
        const int kend = causal ? min(K, K - T + t_last + 1) : K;
        n_items = (kend + kTcRows - 1) / kTcRows;
    } else {      // query tiles from the first position that sees key j0
        i_lo = causal ? max(0, tile * kTcRows - (K - T)) / tb : 0;
        n_items = L.n_qt - i_lo;
    }
    const int q_bytes = KH * G * tb * 128 + (REM ? G * tb * 32 : 0);  // out-of-range positions are zero-filled

    extern __shared__ __align__(1024) unsigned char smem_tc[];
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem_tc);
    const uint32_t bar_fixed = smem_u32(smem_tc + 8);        // count 1 (+ transaction bytes)
    const uint32_t bar_full = bar_fixed + 8;                  // [RING] count 1 (+ transaction bytes)
    const uint32_t bar_empty = bar_full + 8 * RING;           // [RING] tcgen05.commit (+ 128 math threads in pass 2)
    const uint32_t bar_tfull = bar_empty + 8 * RING;          // [kTcAcc] tcgen05.commit
    const uint32_t bar_tempty = bar_tfull + 8 * kTcAcc;       // [kTcAcc] 128 math threads
    float* s_lse = reinterpret_cast<float*>(smem_tc + 1024);  // [RING][128]
    float* s_mass = reinterpret_cast<float*>(smem_tc + kTcHead);  // [G][128]
    unsigned char* s_fixed = smem_tc + kTcHead + tc_mass_bytes(G);
    unsigned char* s_ring = s_fixed + TILE;

    if (tid == 0) {
        mbar_init(bar_fixed, 1);
        for (int i = 0; i < RING; ++i) {
            mbar_init(bar_full + 8 * i, 1);
            mbar_init(bar_empty + 8 * i, COLS ? 1 + kTcRows : 1);
        }
        for (int i = 0; i < kTcAcc; ++i) {
            mbar_init(bar_tfull + 8 * i, 1);
            mbar_init(bar_tempty + 8 * i, kTcRows);
        }
        mbar_init_fence();
    }
    if (COLS && tid < kTcRows)
        for (int g = 0; g < G; ++g) s_mass[g * kTcRows + tid] = 0.f;
    if (warp == 5) tmem_alloc(smem_u32(s_tmem), kTcAcc * kTcRows);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *s_tmem;

    if (warp == 4) {
        // ================================================================ TMA producer (one thread)
        if (lane == 0 && n_items > 0) {
            auto load_q = [&](uint32_t dst, int qt, uint32_t bar) {
#pragma unroll
                for (int kh = 0; kh < KH; ++kh) tma_load_4d(dst + kh * BOX, &L.qmap, kh * 64, qt * tb, hk * G, b, bar);
                if (REM) tma_load_4d(dst + KH * BOX, &L.qmap_tail, KH * 64, qt * tb, hk * G, b, bar);
            };
            auto load_k = [&](uint32_t dst, int kt, uint32_t bar) {
#pragma unroll
                for (int kh = 0; kh < KH; ++kh) tma_load_4d(dst + kh * BOX, &L.kmap, kh * 64, kt * kTcRows, hk, b, bar);
                if (REM) tma_load_4d(dst + KH * BOX, &L.kmap_tail, KH * 64, kt * kTcRows, hk, b, bar);
            };
            mbar_arrive_expect_tx(bar_fixed, COLS ? TILE : q_bytes);
            if (COLS) load_k(smem_u32(s_fixed), tile, bar_fixed);
            else load_q(smem_u32(s_fixed), tile, bar_fixed);
            for (int n = 0; n < n_items; ++n) {
                const int slot = n % RING;
                mbar_wait(bar_empty + 8 * slot, (uint32_t)(((n / RING) & 1) ^ 1));  // fresh barrier: passes
                const uint32_t dst = smem_u32(s_ring) + slot * TILE, bar = bar_full + 8 * slot;
                if (COLS) {
                    const int qt = i_lo + n;
                    mbar_arrive_expect_tx(bar, (uint32_t)(q_bytes + kTcRows * 4));
                    load_q(dst, qt, bar);
                    bulk_g2s(smem_u32(s_lse + slot * kTcRows), L.lse + ((int64_t)bh * L.n_qt + qt) * kTcRows, kTcRows * 4,
                             bar);
                } else {
                    mbar_arrive_expect_tx(bar, TILE);
                    load_k(dst, n, bar);
                }
            }
        }
    } else if (warp == 5) {
        // ================================================================ MMA issuer (one thread)
        if (lane == 0 && n_items > 0) {
            const uint32_t a_base = smem_u32(s_fixed), ring = smem_u32(s_ring);
            mbar_wait(bar_fixed, 0);
            for (int n = 0; n < n_items; ++n) {
                const int slot = n % RING, acc = n % kTcAcc;
                mbar_wait(bar_tempty + 8 * acc, (uint32_t)(((n / kTcAcc) & 1) ^ 1));  // accumulator drained
                mbar_wait(bar_full + 8 * slot, (uint32_t)((n / RING) & 1));           // tile landed
                tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < CPR / 2; ++ks)
                    umma_f16(tmem + acc * kTcRows, tc_desc<CPR>(a_base, ks), tc_desc<CPR>(ring + slot * TILE, ks), IDESC,
                             ks > 0 ? 1u : 0u);
                umma_commit(bar_tfull + 8 * acc);
                umma_commit(bar_empty + 8 * slot);
            }
        }
    } else {
        // ================================================================ math: thread tid = TMEM lane tid
        const uint32_t t_lane = tmem + ((uint32_t)(warp * 32) << 16);
        const float c2 = L.c2;
        if (!COLS) {
            // ---- pass 1: row tid = head hk*G + g, position t
            const int g = tid / tb, t = tile * tb + (tid - g * tb);
            const bool live = g < G && t < T;
            float m_run = -INFINITY, l_run = 0.f;
            // key tiles that every position of the tile sees in full (causal): the mask-free instantiation
            const int n_plain = causal ? min(n_items, max(0, (K - T + tile * tb + 1) / kTcRows)) : 0;
            auto row_tile = [&](int n, uint32_t tacc, auto masked_tag) {
                constexpr bool MASKED = decltype(masked_tag)::value;
                const int key0 = n * kTcRows;
#pragma unroll 1
                for (int ch = 0; ch < kTcRows / 32; ++ch) {
                    uint32_t v[32];
                    tmem_ld32(tacc + ch * 32, v);
                    bool vis[32];
                    float cmax = -INFINITY;
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        vis[c] = true;
                        if (MASKED) {
                            const int j = key0 + ch * 32 + c;
                            vis[c] = live && j < K && tc_visible(L, b, t, j);
                        }
                        if (vis[c]) cmax = fmaxf(cmax, __uint_as_float(v[c]) * c2);
                    }
                    const float m_new = fmaxf(m_run, cmax);
                    if (m_new > -INFINITY) {
                        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
                        for (int c = 0; c < 32; c += 4) {
                            a0 += vis[c] ? ex2(fmaf(__uint_as_float(v[c]), c2, -m_new)) : 0.f;
                            a1 += vis[c + 1] ? ex2(fmaf(__uint_as_float(v[c + 1]), c2, -m_new)) : 0.f;
                            a2 += vis[c + 2] ? ex2(fmaf(__uint_as_float(v[c + 2]), c2, -m_new)) : 0.f;
                            a3 += vis[c + 3] ? ex2(fmaf(__uint_as_float(v[c + 3]), c2, -m_new)) : 0.f;
                        }
                        if (m_new != m_run) l_run *= ex2(m_run - m_new);
                        l_run += (a0 + a1) + (a2 + a3);
                        m_run = m_new;
                    }
                }
            };
            for (int n = 0; n < n_items; ++n) {
                const int acc = n % kTcAcc;
                mbar_wait(bar_tfull + 8 * acc, (uint32_t)((n / kTcAcc) & 1));
                tc_fence_after();
                if (n < n_plain) row_tile(n, t_lane + acc * kTcRows, std::false_type{});
                else row_tile(n, t_lane + acc * kTcRows, std::true_type{});
                tc_fence_before();
                mbar_arrive(bar_tempty + 8 * acc);
            }
            // rows that see no key (and padding rows) get +inf: exp2(s - inf) = 0 in pass 2
            L.lse[((int64_t)bh * L.n_qt + tile) * kTcRows + tid] = live && l_run > 0.f ? m_run + log2f(l_run) : INFINITY;
        } else {
            // ---- pass 2: lane tid = key j; columns g * tb + u = head hk*G + g, position qt*tb + u
            const int j0 = tile * kTcRows, j = j0 + tid;
            const bool col_live = j < K;
            const int ncols = G * tb;
            auto col_tile = [&](int qt, uint32_t tacc, const float* lse, auto masked_tag) {
                constexpr bool MASKED = decltype(masked_tag)::value;
                const int t0 = qt * tb, u_end = min(tb, T - t0);
                int g = 0, u = 0;
                float cur = s_mass[tid];
#pragma unroll 1
                for (int ch = 0; ch * 32 < ncols; ++ch) {  // warp-uniform
                    uint32_t v[32];
                    tmem_ld32(tacc + ch * 32, v);
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        if (g < G) {
                            if (u < u_end && (!MASKED || (col_live && tc_visible(L, b, t0 + u, j))))
                                cur = __fadd_rn(cur, round_dt<DT>(ex2(fmaf(__uint_as_float(v[c]), c2, -lse[ch * 32 + c]))));
                            if (++u == tb) {
                                s_mass[g * kTcRows + tid] = cur;
                                u = 0;
                                if (++g < G) cur = s_mass[g * kTcRows + tid];
                            }
                        }
                    }
                }
            };
            for (int n = 0; n < n_items; ++n) {
                const int acc = n % kTcAcc, slot = n % RING, qt = i_lo + n;
                mbar_wait(bar_tfull + 8 * acc, (uint32_t)((n / kTcAcc) & 1));
                mbar_wait(bar_full + 8 * slot, (uint32_t)((n / RING) & 1));  // the lse2 of the slot (already landed)
                tc_fence_after();
                // every (position >= qt*tb, key < j0 + 128) pair visible: the mask-free instantiation
                const bool plain = causal && j0 + kTcRows - 1 <= K - T + qt * tb;
                if (plain) col_tile(qt, t_lane + acc * kTcRows, s_lse + slot * kTcRows, std::false_type{});
                else col_tile(qt, t_lane + acc * kTcRows, s_lse + slot * kTcRows, std::true_type{});
                tc_fence_before();
                mbar_arrive(bar_tempty + 8 * acc);
                mbar_arrive(bar_empty + 8 * slot);
            }
            if (col_live) {
                const int prev = (L.prev < 0 || L.prev > K) ? 0 : L.prev;  // the reference's reset when the cache shrank
                for (int g = 0; g < G; ++g) {
                    Key* ap = reinterpret_cast<Key*>(L.acc + (int64_t)b * L.csb + (int64_t)(hk * G + g) * L.csh) + j;
                    h2o_update_acc<DT>(ap, s_mass[g * kTcRows + tid], j, prev, bd.decay);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) tmem_dealloc(tmem, kTcAcc * kTcRows);
}

}  // namespace kvc
