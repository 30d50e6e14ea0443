// kvc_vote.cuh — SnapKV observation-window vote on the 5th-generation tensor cores (tcgen05 + TMEM).
//
// OPT-IN EXTENSION.  The reference's snapkv_lite has no queries and no q.K^T (snapkv_lite.py:93-100 ranks
// keys by inverted L2 norm); this kernel implements the vote the method is named after (reference
// docs/logsAndBugs/SnapKV_Feasibility_Analysis.md:29-62): the last W queries of every query head attend
// over the whole cache, and each prefix key's score is the attention mass it receives,
//
//     vote[b, hkv, j] = sum over the G query heads of the group and the W window queries i of
//                       softmax_j( q_i . k_j / sqrt(D)  [causal inside the window] )         for j < P = S - W
//
// One CTA (576 threads, one per SM) owns one (layer, batch, kv head).  Queries of the group are stacked into a
// 128-row operand (G*W <= 128; fewer rows are replicated, see below).  Keys stream in tiles of 128 rows, twice:
//
//   pass 1  S   = Q . Ktile^T  (M = query rows, N = keys): TMEM lane = query row, so each thread keeps the
//           online softmax statistics (running max m_i, sum l_i) of ITS row — no cross-thread traffic;
//   pass 2  S^T = Ktile . Q^T  (M = keys, N = query rows): TMEM lane = key, so each thread sums
//           exp2(s*c - m_i) / l_i over the columns of ITS key — the vote — and stores it.
//
// Pass 1 exists only to produce the softmax denominators.  An attention kernel that has just run those W
// queries already holds them (the log-sum-exp per query row every flash-attention forward returns): with
// kvc_vote_layer.lse the kernel runs pass 2 alone and K crosses HBM once instead of twice.
//
// Key tiles arrive through TMA tensor loads (128-byte-swizzled boxes = the K-major SW128 UMMA layout), the
// accumulators live in TMEM (4 x 128 columns), `tcgen05.mma` is issued by one thread, completion arrives on
// mbarriers through `tcgen05.commit`, and `tcgen05.ld` brings scores to registers.
//
// Fused tail (kvc_snapkv_vote_compress): once a unit's votes exist the SAME CTA pools them, radix-selects the
// kept rows and gathers K and V into the compacted output — snapkv_lite.py:104-150 behind the vote in ONE launch.
// The votes go through a [B,H,P] scratch array in the cache dtype (the rounding point of the two-launch form) that
// the CTA reads straight back out of L2; the key-tile ring, dead by then, becomes the select's key buffer and the
// gather's staging slots.
// Intensity is ~2*128 flop per key byte at most: the kernel stays HBM/MUFU-bound, not tensor-bound
// (SURVEY.md §7 "SnapKV vote spec gap") — the tensor pipe is reported, not chased.
#pragma once
#include <type_traits>

#include "kvc_device.cuh"
#include "kvc_fused_tma.cuh"
#include "kvc_tcgen05.cuh"
#include "kvc_tma.cuh"

namespace kvc {

constexpr int kVoteM = 128;     // rows of both MMA shapes
constexpr int kVoteTile = 128;  // keys per tile

// Lab build only.  KVC_VOTE_DEBUG=6: the exponentials of both passes replaced by the identity (everything but the MUFU
// work is timed); KVC_T0 / KVC_TACC: cycles a role spends inside its mbarrier waits, per CTA, into lab_timeline.
#ifdef KVC_LAB
#define KVC_EX2(x) (lab_noexp ? (x) : ex2(x))
#define KVC_T0() const long long _t0 = clock64()
#define KVC_TACC(var) var += clock64() - _t0
#else
#define KVC_EX2(x) ex2(x)
#define KVC_T0()
#define KVC_TACC(var)
#endif

// Chunk (row r, 16-byte chunk c) of a [rows][CPR chunks] operand tile in the canonical layout: dense
// 128-byte core matrices (8 rows x 16 B), K chunks kVoteLBO = 128 B apart, 8-row groups CPR*128 B apart.
constexpr int kVoteLBO = 128;
template <int CPR>
__device__ __forceinline__ uint32_t umma_off(int r, int c) {
    return (uint32_t)((r >> 3) * (CPR * kVoteLBO) + c * kVoteLBO + (r & 7) * 16);
}
// Work item q of a tile -> (row, chunk) such that 8 consecutive threads write the 8 rows of ONE core matrix
// (one 128-byte line of shared memory: conflict-free) while the 4 octets of a warp read 4 consecutive
// chunks of those rows (64 contiguous bytes per row: every 32-byte sector it touches is fully used).
template <int CPR>
__device__ __forceinline__ void tile_item(int q, int& r, int& c) {
    const int rg = q / (8 * CPR), rem = q - rg * (8 * CPR);
    c = rem >> 3;
    r = rg * 8 + (rem & 7);
}

// ---------------------------------------------------------------------------------------------
// Warp-specialised: ONE CTA per SM; warps 0-15 are four math groups (128 threads = the 128 TMEM lanes;
// group g owns accumulator g, 128 of the 512 TMEM columns, and reduces work items g, g+4, g+8, ...), one thread feeds
// a shared-memory ring of key tiles, one thread issues every tcgen05.mma (waits: slot full, accumulator drained) and
// commits to the accumulator-full and slot-empty mbarriers.  Work items are the tiles of pass 1 (all S keys, A = Q)
// followed by the tiles of pass 2 (P keys, A = keys); the copy and MMA threads run ahead across the pass boundary,
// only the math groups meet there to merge the row statistics.  (A cp.async-fed variant of this layout, four copy
// warps, was measured at 21.6 ms on c4_vote against 15.6 ms for the TMA-fed one and removed.)
// ---------------------------------------------------------------------------------------------
// TMA-fed warp-specialised form (head_dim * 2 bytes a multiple of 128: D = 64, 128).  Stage isolation of the
// cp.async-fed kernels showed the copy stage alone at 4.3 TB/s (16 of 22 ms at c4): 16-byte copies into the
// layout are the bottleneck, not the tensor core or the softmax math.  Here ONE thread feeds the ring with
// `cp.async.bulk.tensor.4d` loads through a per-layer tensor map (boxes of 128 rows x 64 elements, 128-byte
// swizzle = the K-major SW128 UMMA layout; rows beyond S are zero-filled by the TMA unit), warps 0-15 do the
// softmax math and one thread issues the MMAs (keys: SW128 descriptors, queries: no-swizzle).
struct VoteTmaLayerDev {
    alignas(64) CUtensorMap map;  // keys [B,H,S,D] as a 4-D tensor (D, S, H, B), box (64, 128, 1, 1), SWIZZLE_128B
    alignas(64) CUtensorMap map_tail;  // D % 64 == 16 (D = 80): box (16, 128, 1, 1), SWIZZLE_32B, for the last 16 elements
    const char* q;
    char* votes;
    const float* lse;  // optional [B, H*G, W] natural-log softmax denominators of the window queries: pass 2 only
    int64_t qsb, qsh, qss;
    int32_t S, pad;
    // fused tail (k_out != nullptr): pool the votes, keep the ksel highest of [0, S - W) + the last `tail` rows
    const char* k_in;
    const char* v_in;
    char* k_out;
    char* v_out;
    int32_t* idx_out;
    int64_t ksb, ksh, kss, vsb, vsh, vss;  // BYTE strides of K and V
    int32_t ksel, tail, pool, idx_cap;
};
struct VoteTmaBatchDev {
    int32_t B, H, G, W;
    float scale_log2e;
    int32_t pad[3];
    long long* lab_timeline;  // lab build: [CTAs][8] cycle counters, or nullptr
    VoteTmaLayerDev layers[32];
};

// Ring depth of the TMA-fed kernel.  A slot is held from the issue of its load until its MMAs have completed, ~3 us,
// so the ring depth bounds the tile rate: 5 slots of 20 KB (D = 80) left the MHA shape latency-bound (copies alone
// 6.0 ms, copies + MMAs 8.4 ms); narrower rows get as many slots as fit next to the Q operand.
__host__ __device__ constexpr int vote_tma_ring(int cpr) {
    const int tile = (cpr / 8) * kVoteTile * 128 + (cpr % 8) * kVoteTile * 16;
    const int q = (kVoteM / 8) * cpr * kVoteLBO;
    const int n = (225 * 1024 - 6144 - q) / tile;
    return n > 12 ? 12 : n;
}

template <int DT, int CPR>
__global__ void __launch_bounds__(576, 1) kvc_snapkv_vote_tma_kernel(const __grid_constant__ VoteTmaBatchDev bd) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    static_assert(DT != KVC_DTYPE_F32, "the vote runs on 16-bit caches (kind::f16)");
    static_assert(CPR % 8 == 0 || CPR % 8 == 2, "key rows = 128-byte boxes (+ one 32-byte box for D % 64 == 16)");
    constexpr int KH = CPR / 8;                       // 64-element (128-byte) boxes per key row
    constexpr int REM = CPR % 8;                      // 16-byte chunks left over: 0, or 2 (one 32-byte-swizzled box)
    constexpr int BOX_BYTES = kVoteTile * 128;        // one box: 128 rows x 128 B, 128B-swizzled
    constexpr int TAIL_BYTES = kVoteTile * 16 * REM;  // tail box: 128 rows x 32 B, 32B-swizzled
    constexpr int TILE_BYTES = KH * BOX_BYTES + TAIL_BYTES;
    constexpr int Q_BYTES = (kVoteM / 8) * CPR * kVoteLBO;
    constexpr int RING = vote_tma_ring(CPR);  // key-tile slots: as many as shared memory holds
    constexpr uint32_t IDESC = umma_idesc_f16(DT == KVC_DTYPE_BF16 ? 1 : 0, kVoteM, kVoteTile);

    const VoteTmaLayerDev& L = bd.layers[blockIdx.y];
    const int bh = blockIdx.x;
    const int b = bh / bd.H, h = bh - b * bd.H;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int S = L.S, W = bd.W, G = bd.G;
    const int P = S - W;
    const int rows_q = G * W;
    const bool no_tail = bd.pad[0] == 3;            // profiling: every stage on, tail box not loaded
    const bool one_k = bd.pad[0] == 4;              // profiling: no math, ONE K step per tile
#ifdef KVC_LAB
    const bool lab_noexp = bd.pad[0] == 6;          // profiling: every stage on, exp2 replaced by the identity
    const bool lab_l2_p2 = bd.pad[0] == 7;          // profiling: pass 2 re-reads 8 tiles that stay in L2 (no HBM traffic)
    const bool lab_l2_all = bd.pad[0] == 8;         // profiling: both passes read those 8 tiles
    const int dbg = (no_tail || lab_noexp || lab_l2_p2 || lab_l2_all) ? 0 : (one_k ? 1 : bd.pad[0]);  // 1 = no math, 2 = no math, no MMA
    long long lab_w1 = 0, lab_w2 = 0, lab_we = 0, lab_wt = 0, lab_wf = 0, lab_wb = 0, lab_tail = 0;
    const long long lab_start = clock64();
    unsigned long long lab_ns0;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(lab_ns0));
#else
    const int dbg = no_tail ? 0 : (one_k ? 1 : bd.pad[0]);  // profiling: 1 = no math, 2 = no math, no MMA
#endif
    const int RB = rows_q <= 32 ? 32 : (rows_q <= 64 ? 64 : 128);  // rows per replica block, F = 128 / RB replicas
    const bool have_lse = L.lse != nullptr;  // the caller holds the softmax denominators: no pass 1
    const int n1 = have_lse ? 0 : (S + kVoteTile - 1) / kVoteTile, n2 = (P + kVoteTile - 1) / kVoteTile;
    const int n_items = n1 + n2;

    extern __shared__ __align__(1024) unsigned char smem_tma[];  // swizzle atoms need 1024-byte alignment
    unsigned char* smem = smem_tma;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem);
    const uint32_t bar_full = smem_u32(smem + 64);        // [RING]  count = 1 (+ transaction bytes of the TMA loads)
    const uint32_t bar_empty = bar_full + 8 * RING;    // [RING]  count = 1 (tcgen05.commit)
    const uint32_t bar_tfull = bar_empty + 8 * RING;   // [4]        count = 1 (tcgen05.commit)
    const uint32_t bar_tempty = bar_tfull + 8 * 4;        // [4]        count = 128 (math threads)
    float* s_m = reinterpret_cast<float*>(smem + 512);
    float* s_part = reinterpret_cast<float*>(smem + 1536);  // [4 groups][2][128]
    const uint32_t bar_tail = smem_u32(smem + 5632);        // [18]  count = 1: the fused tail's staging slots
    unsigned char* s_q = smem + 6144;
    unsigned char* s_ring = s_q + Q_BYTES;  // 1024-byte aligned: swizzle atoms are 8 rows x 128 B

    if (tid == 0) {
        for (int i = 0; i < RING; ++i) {
            mbar_init(bar_full + 8 * i, 1);
            mbar_init(bar_empty + 8 * i, 1);
        }
        for (int i = 0; i < 4; ++i) {
            mbar_init(bar_tfull + 8 * i, 1);
            mbar_init(bar_tempty + 8 * i, 128);
        }
        for (int i = 0; i < 18; ++i) mbar_init(bar_tail + 8 * i, 1);
        mbar_init_fence();
    }
    if (warp == 17) tmem_alloc(smem_u32(s_tmem), 512);
    // Few query rows (MHA: G*W = 32): the rows are REPLICATED down the 128 MMA rows -- F copies of a block of RB =
    // 128 / F rows -- so that in pass 1 every lane quarter of an accumulator holds live rows and its warp takes 1/F of
    // the tile's key columns.  Without this only the warp of quarter 0 works in pass 1, and the four groups' quarter-0
    // warps all sit on the same SM sub-partition (a warp can only read the TMEM lanes of quarter warp_id % 4): a
    // quarter of the ex2 pipe carries the whole pass.
    for (int q = tid; q < kVoteM * CPR; q += 576) {
        int r, c;
        tile_item<CPR>(q, r, c);
        int4 v = make_int4(0, 0, 0, 0);
        const int qr = r & (RB - 1);  // MMA row r carries query row r mod RB
        if (qr < rows_q) {
            const int g = qr / W, w = qr - g * W;
            v = ldg128_stream(L.q + (int64_t)b * L.qsb + (int64_t)(h * G + g) * L.qsh + (int64_t)w * L.qss + c * 16);
        }
        *reinterpret_cast<int4*>(s_q + umma_off<CPR>(r, c)) = v;
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *s_tmem;
    const uint32_t q_addr = smem_u32(s_q), ring_addr = smem_u32(s_ring);
    const float c2 = bd.scale_log2e;

    if (warp < 16) {
        // ================================================================ math groups
        const int grp = warp >> 2, gt = tid & 127;
        const uint32_t t_lane = tmem + grp * kVoteTile + ((uint32_t)((warp & 3) * 32) << 16);
        float m_run = -INFINITY, l_run = 0.f;
        // the accumulator is read 16 columns at a time with the next 16 already in flight (two register sets); TMEM
        // itself is not a limit (tcgen05.ld measures ~460 B/clk/SM with 16 warps, scripts/lab/tmem_ld_bw.cu: ten
        // times what this kernel reads), the load's latency is what the second register set hides
        uint32_t va[16], vb[16];
        const int row = gt & (RB - 1);          // query row of this TMEM lane; replica gt / RB
        const int limit = P + ((row < rows_q) ? (row % W) : 0);
        const bool row_live = (((warp & 3) * 32) & (RB - 1)) < rows_q;
        const int c_lo = (gt / RB) * RB;        // this replica's share of a tile's key columns: [c_lo, c_lo + RB)
        const int nch = RB / 16;
        // One pass-1 tile: 16 columns at a time, running maximum and sum of exponentials of this thread's row.
        // MASKED is a template-like compile-time switch (two separate instantiations of the lambda body): only the
        // last one or two tiles of a pass meet the causal window or the end of the sequence, and when both cases
        // shared one loop the compiler if-converted the mask into two compares, an add and a select per score on
        // EVERY tile — 168 instructions per 16 columns instead of ~85 (profiles/r02_ncu_full_vote_fused_c4_b4.json).
        auto pass1_tile = [&](int i, auto masked_tag) {
            constexpr bool MASKED = decltype(masked_tag)::value;
            const int key0 = i * kVoteTile;
            tmem_ld16_async(t_lane + c_lo, va);
#pragma unroll
            for (int ch = 0; ch < kVoteTile / 16; ++ch) {
                if (ch >= nch) break;  // warp-uniform
                const int cb = c_lo + ch * 16;
                uint32_t(&v)[16] = (ch & 1) ? vb : va;
                tmem_ld_wait();
                if (ch + 1 < nch) tmem_ld16_async(t_lane + cb + 16, (ch & 1) ? va : vb);
                float cmax = -INFINITY;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    if (MASKED) {
                        const int key = key0 + cb + j;
                        if (key > limit || key >= S) v[j] = 0xff800000u;
                    }
                    cmax = fmaxf(cmax, __uint_as_float(v[j]));
                }
                const float m_new = fmaxf(m_run, cmax * c2);
                if (m_new > -INFINITY) {
                    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        acc0 += KVC_EX2(fmaf(__uint_as_float(v[j]), c2, -m_new));
                        acc1 += KVC_EX2(fmaf(__uint_as_float(v[j + 1]), c2, -m_new));
                        acc2 += KVC_EX2(fmaf(__uint_as_float(v[j + 2]), c2, -m_new));
                        acc3 += KVC_EX2(fmaf(__uint_as_float(v[j + 3]), c2, -m_new));
                    }
                    if (m_new != m_run) l_run *= ex2(m_run - m_new);  // the maximum settles after a few tiles
                    l_run += (acc0 + acc1) + (acc2 + acc3);
                    m_run = m_new;
                }
            }
        };
        const int n_plain = min(n1, P / kVoteTile);  // tiles that lie entirely inside the prefix: no mask
        int i = grp;
        for (; i < n_plain; i += 4) {
            {
                KVC_T0();
                mbar_wait(bar_tfull + 8 * grp, (uint32_t)((i >> 2) & 1));
                KVC_TACC(lab_w1);
            }
            tc_fence_after();
            if (row_live && dbg == 0) pass1_tile(i, std::false_type{});
            tc_fence_before();
            mbar_arrive(bar_tempty + 8 * grp);
        }
        for (; i < n1; i += 4) {
            {
                KVC_T0();
                mbar_wait(bar_tfull + 8 * grp, (uint32_t)((i >> 2) & 1));
                KVC_TACC(lab_w1);
            }
            tc_fence_after();
            if (row_live && dbg == 0) pass1_tile(i, std::true_type{});
            tc_fence_before();
            mbar_arrive(bar_tempty + 8 * grp);
        }
        // ---------------- pass boundary: merge the four groups' partial statistics
#ifdef KVC_LAB
        const long long lab_b0 = clock64();
#endif
        s_part[(grp * 2 + 0) * 128 + gt] = m_run;
        s_part[(grp * 2 + 1) * 128 + gt] = l_run;
        asm volatile("bar.sync 1, 512;" ::: "memory");
        if (have_lse) {
            // exp(s - lse) is the normalised probability: m = lse in the log2 domain, 1 / l = 1
            if (tid < 128) {
                const bool live = tid < rows_q;
                float lse = 0.f;
                if (live) lse = L.lse[((int64_t)b * bd.H * G + (int64_t)h * G + tid / W) * W + tid % W];
                s_m[tid] = live ? lse * 1.4426950408889634f : INFINITY;
            }
        } else if (tid < 128) {
            // query row `tid`: four groups x F replicas, always in the same order
            float m = -INFINITY;
            if (tid < RB) {
                for (int f = tid; f < 128; f += RB) {
#pragma unroll
                    for (int g4 = 0; g4 < 4; ++g4) m = fmaxf(m, s_part[(g4 * 2) * 128 + f]);
                }
            }
            float l = 0.f;
            if (m > -INFINITY) {
                for (int f = tid; f < 128; f += RB) {
#pragma unroll
                    for (int g4 = 0; g4 < 4; ++g4) {
                        const float mp = s_part[(g4 * 2) * 128 + f];
                        if (mp > -INFINITY) l += s_part[(g4 * 2 + 1) * 128 + f] * ex2(mp - m);
                    }
                }
            }
            // p / l = exp2(s*c - (m + log2 l)): the division folds into the exponent; rows that never vote (padding,
            // or an empty softmax row) get +inf, i.e. exp2(-inf) = 0
            const bool live = tid < rows_q && l > 0.f;
            s_m[tid] = live ? m + log2f(l) : INFINITY;
        }
        asm volatile("bar.sync 1, 512;" ::: "memory");
#ifdef KVC_LAB
        lab_wb = clock64() - lab_b0;
#endif
        // ---------------- pass 2: lane = key, columns = query rows
        for (; i < n_items; i += 4) {
            {
                KVC_T0();
                mbar_wait(bar_tfull + 8 * grp, (uint32_t)((i >> 2) & 1));
                KVC_TACC(lab_w2);
            }
            tc_fence_after();
            float vote0 = 0.f, vote1 = 0.f, vote2 = 0.f, vote3 = 0.f;
            if (dbg == 0) tmem_ld16_async(t_lane, va);
#pragma unroll
            for (int cb = 0; cb < kVoteM; cb += 16) {
                if (cb < rows_q && dbg == 0) {  // warp-uniform: padding query rows never vote
                    uint32_t(&v)[16] = ((cb >> 4) & 1) ? vb : va;
                    tmem_ld_wait();
                    if (cb + 16 < rows_q) tmem_ld16_async(t_lane + cb + 16, ((cb >> 4) & 1) ? va : vb);
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const float4 mm = *reinterpret_cast<const float4*>(s_m + cb + j);
                        vote0 += KVC_EX2(fmaf(__uint_as_float(v[j + 0]), c2, -mm.x));
                        vote1 += KVC_EX2(fmaf(__uint_as_float(v[j + 1]), c2, -mm.y));
                        vote2 += KVC_EX2(fmaf(__uint_as_float(v[j + 2]), c2, -mm.z));
                        vote3 += KVC_EX2(fmaf(__uint_as_float(v[j + 3]), c2, -mm.w));
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(bar_tempty + 8 * grp);
            const int key = (i - n1) * kVoteTile + gt;
            if (key < P) {
                Key* out = reinterpret_cast<Key*>(L.votes) + (int64_t)bh * P;
                out[key] = (Key)Tr::to_raw((vote0 + vote1) + (vote2 + vote3));
            }
        }
    } else if (warp == 16) {
        // ================================================================ TMA producer (one thread)
        if (lane == 0) {
            const bool tail = REM > 0 && !no_tail;  // KVC_VOTE_DEBUG=3: timing without the 32-byte tail box
            for (int i = 0; i < n_items; ++i) {
                const int slot = i % RING;
                {
                    KVC_T0();
                    mbar_wait(bar_empty + 8 * slot, (uint32_t)(((i / RING) & 1) ^ 1));  // fresh barrier: passes
                    KVC_TACC(lab_we);
                }
#ifdef KVC_LAB
                const int t = i < n1 ? (lab_l2_all ? (i & 7) : i) : ((lab_l2_p2 || lab_l2_all) ? ((i - n1) & 7) : i - n1);
#else
                const int t = i < n1 ? i : i - n1;
#endif
                mbar_arrive_expect_tx(bar_full + 8 * slot, tail || REM == 0 ? TILE_BYTES : KH * BOX_BYTES);
#pragma unroll
                for (int kh = 0; kh < KH; ++kh)  // rows beyond S are zero-filled by the TMA unit
                    tma_load_4d(ring_addr + slot * TILE_BYTES + kh * BOX_BYTES, &L.map, kh * 64, t * kVoteTile, h, b,
                                bar_full + 8 * slot);
                if (tail)
                    tma_load_4d(ring_addr + slot * TILE_BYTES + KH * BOX_BYTES, &L.map_tail, KH * 64, t * kVoteTile, h, b,
                                bar_full + 8 * slot);
            }
        }
    } else if (warp == 17 && lane == 0) {
        // ================================================================ MMA issuer
        // ONE thread issues everything, and a lone warp retires an instruction every ~5 clocks: stage isolation on the
        // MHA shape showed copies + MMAs (no math) at 8.9 ms of the 9.4 ms call and copies alone at 6.0 ms, i.e. the
        // ~180 instructions per tile spent building shared-memory descriptors were the bottleneck.  The descriptors
        // are affine in the shared address, so the Q descriptors and the slot-0 key descriptors are built once and
        // a tile costs one 32-bit add per K step.
        uint32_t qd_lo[CPR / 2], kd_lo0[CPR / 2];  // low words; the high words are per-layout constants
#pragma unroll
        for (int ks = 0; ks < CPR / 2; ++ks) {
            qd_lo[ks] = (uint32_t)umma_smem_desc(q_addr + ks * 2 * kVoteLBO, kVoteLBO, CPR * kVoteLBO);
            kd_lo0[ks] = (ks >> 2) < KH ? (uint32_t)umma_smem_desc_sw128(ring_addr + (ks >> 2) * BOX_BYTES + (ks & 3) * 32)
                                        : (uint32_t)umma_smem_desc_sw32(ring_addr + KH * BOX_BYTES);
        }
        const uint32_t qd_hi = (uint32_t)(umma_smem_desc(q_addr, kVoteLBO, CPR * kVoteLBO) >> 32);
        const uint32_t k128_hi = (uint32_t)(umma_smem_desc_sw128(ring_addr) >> 32);
        const uint32_t k32_hi = (uint32_t)(umma_smem_desc_sw32(ring_addr) >> 32);
        auto pack = [](uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; };
        // pass 2 only needs the live query rows as columns: N = G*W rounded up to 16 instead of 128 (MHA: 32) cuts the
        // tensor time and the shared-memory reads of the Q operand by the same factor
        const int n2cols = min(kVoteTile, (rows_q + 15) & ~15);
        const uint32_t idesc2 = umma_idesc_f16(DT == KVC_DTYPE_BF16 ? 1 : 0, kVoteM, n2cols);
        auto issue = [&](int i, auto keys_are_rows) {
            const int slot = i % RING, acc = i & 3;
            {
                KVC_T0();
                mbar_wait(bar_tempty + 8 * acc, (uint32_t)(((i >> 2) & 1) ^ 1));  // accumulator drained (fresh: passes)
                KVC_TACC(lab_wt);
            }
            {
                KVC_T0();
                mbar_wait(bar_full + 8 * slot, (uint32_t)((i / RING) & 1));    // tile landed
                KVC_TACC(lab_wf);
            }
            tc_fence_after();
            const uint32_t slot16 = (uint32_t)(slot * TILE_BYTES) >> 4;  // start-address field counts 16-byte units
            if (dbg < 2) {
#pragma unroll
                for (int ks = 0; ks < CPR / 2; ++ks) {
                    if (one_k && ks > 0) break;
                    // keys: 128B-swizzled K-major box (8-row groups 1024 B apart), 32 bytes per K step inside the
                    // box (D = 80: one 32B-swizzled tail box); queries: dense no-swizzle core matrices
                    const uint64_t kd = pack(kd_lo0[ks] + slot16, (ks >> 2) < KH ? k128_hi : k32_hi);
                    const uint64_t qd = pack(qd_lo[ks], qd_hi);
                    if (decltype(keys_are_rows)::value)
                        umma_f16(tmem + acc * kVoteTile, kd, qd, idesc2, ks > 0 ? 1u : 0u);
                    else
                        umma_f16(tmem + acc * kVoteTile, qd, kd, IDESC, ks > 0 ? 1u : 0u);
                }
            }
            umma_commit(bar_tfull + 8 * acc);
            umma_commit(bar_empty + 8 * slot);
        };
        for (int i = 0; i < n1; ++i) issue(i, std::false_type{});        // pass 1: A = Q, B = key tile
        for (int i = n1; i < n_items; ++i) issue(i, std::true_type{});   // pass 2: A = key tile, B = Q
    }
    tc_fence_before();
    __syncthreads();
#ifdef KVC_LAB
    const long long lab_vote_end = clock64();
    if (bd.lab_timeline != nullptr) {
        long long* t = bd.lab_timeline + ((long long)blockIdx.y * gridDim.x + blockIdx.x) * 16;
        if (tid == 0) {
            t[0] = lab_w1;                      // math group 0, lane 0: waiting for accumulators, pass 1
            t[1] = lab_w2;                      // ... pass 2
            t[2] = lab_vote_end - lab_start;    // the whole vote phase of this unit
            t[6] = lab_wb;                      // pass boundary (merge + two 512-thread barriers)
        }
        if (warp == 16 && lane == 0) t[3] = lab_we;                      // producer: waiting for a free ring slot
        if (warp == 17 && lane == 0) { t[4] = lab_wt; t[5] = lab_wf; }  // MMA issuer: waiting for accumulator / tile
    }
#endif
    if (warp == 17) tmem_dealloc(tmem, 512);
    if (L.k_out == nullptr) return;  // votes only (CTA-uniform)

    // ==================================================================== fused tail: pool -> select -> gather
    // Every MMA has completed (the math groups drained every accumulator), so the key-tile ring is dead: it becomes
    // histogram | kept indices | radix keys | staging slots.  The unit's votes were written by this CTA's own
    // threads before the barrier above: they are read back with plain loads (L2 hits), in the cache dtype — the
    // same rounding point as the two-launch form, so both keep the same rows.
    {
        constexpr int NT = 576;
        constexpr int RBYTES = CPR * 16;
        int32_t* misc = reinterpret_cast<int32_t*>(s_part);  // 512 B of scalars; the row statistics are dead
        uint32_t* hist = reinterpret_cast<uint32_t*>(s_ring);
        int32_t* sidx = reinterpret_cast<int32_t*>(s_ring + kHistBins * 4);
        Key* keys = reinterpret_cast<Key*>(s_ring + kHistBins * 4 + L.idx_cap * 4);
        const int keys_bytes = (P * (int)sizeof(Key) + 15) & ~15;
        const int off_stage = (kHistBins * 4 + L.idx_cap * 4 + keys_bytes + 127) & ~127;
        const int nstage = min(18, (RING * TILE_BYTES - off_stage) / (32 * RBYTES));  // >= 1: checked by the host
        const int ksel = L.ksel;
        fence_proxy_async_smem();
        for (int i = tid; i < kHistBins; i += NT) hist[i] = 0;
        const Key* src = reinterpret_cast<const Key*>(L.votes) + (int64_t)bh * P;
        load_keys_vectorised<DT, NT, /*NC=*/false>(src, P, keys, [&](int i, uint32_t raw) { keys[i] = (Key)raw; });
        __syncthreads();
        snapkv_transform<DT, NT>(keys, P, L.pool, hist, misc, /*invert=*/false);
        block_radix_select<Key, NT>(keys, P, ksel, hist, misc, sidx, 0);
        const int C = ksel + L.tail;
        const KeepMap src_row{sidx, 0, ksel, S - L.tail - ksel};
        if (L.idx_out != nullptr) {
            int32_t* io = L.idx_out + (int64_t)bh * C;
            for (int j = tid; j < C; j += NT) io[j] = src_row(j);
        }
        if (warp < nstage) {
            uint32_t parity = 0;
            gather_unit(src_row, C, L.k_in + (int64_t)b * L.ksb + (int64_t)h * L.ksh,
                        L.v_in + (int64_t)b * L.vsb + (int64_t)h * L.vsh, L.kss, L.vss,
                        L.k_out + (int64_t)bh * C * RBYTES, L.v_out + (int64_t)bh * C * RBYTES, RBYTES,
                        smem_u32(s_ring + off_stage) + (uint32_t)(warp * 32 * RBYTES), bar_tail + 8 * warp, parity, warp,
                        nstage, lane);
        }
#ifdef KVC_LAB
        __syncthreads();
        if (tid == 0 && bd.lab_timeline != nullptr) {
            long long* t = bd.lab_timeline + ((long long)blockIdx.y * gridDim.x + blockIdx.x) * 16;
            unsigned long long ns1;
            unsigned smid;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(ns1));
            asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
            t[7] = clock64() - lab_vote_end;
            t[8] = (long long)smid;
            t[9] = (long long)lab_ns0;
            t[10] = (long long)ns1;
            t[11] = clock64() - lab_start;
        }
#endif
    }
}

}  // namespace kvc
