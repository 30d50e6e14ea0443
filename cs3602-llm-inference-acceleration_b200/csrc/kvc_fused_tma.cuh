// kvc_fused_tma.cuh — the fused compress kernel for sm_100a: scan -> select -> gather, one CTA per
// (layer, batch, head) unit, every layer of a call in ONE launch.
//
// No key/value byte passes through registers on its way in or out:
//
//   scan   each staging warp owns one shared-memory slot of 32 rows and one mbarrier.  Lane 0
//          streams the unit's key rows into the slot with `cp.async.bulk` (one copy per 32 rows;
//          one per row when rows are not contiguous), the warp waits on the mbarrier, and every
//          lane reduces ONE whole row from shared memory: 128-bit LDS, fp32 FMA per 16-byte
//          chunk, chunk sums combined by a balanced tree.  Lanes read their chunks in an
//          XOR-swizzled order so that the 8 lanes of an LDS.128 phase hit 8 different bank
//          groups although the row pitch (D*e bytes) is a multiple of 32 B; the tree makes the
//          sum independent of that order (a+b == b+a), so a row's norm does not depend on the
//          lane that computed it.  (torch.norm, e.g. l2_compress.py:70)
//          When the caller holds the key norms already (kvc_layer_io.norms_in: a slab cache records
//          them at append time) the scan is skipped: the radix keys are built from 2-4 bytes per
//          row instead of D*e — on a host-resident cache that is the difference between pulling
//          the whole selection region over PCIe and pulling only the rows that are kept.
//   select radix select over the on-chip keys (kvc_device.cuh).
//   gather output rows are produced 32 at a time per staging warp: every run of consecutive
//          source rows becomes one bulk load into the slot, and the 32 rows leave with ONE bulk
//          store into the dense output (expand + gather x2 + cat x2, e.g. fix_size_l2.py:132-147).
//   carry  optional per-row state (kvc_carry_layer: H2O accumulators) compacted IN PLACE with the kept rows by
//          the whole CTA, between the select and the gather (carry_unit).
//
// Row widths: CPR (16-byte chunks per row) is a template parameter for the widths of real models
// (128/160/192/256/320/512-byte rows); CPR = 0 is the generic form for every other head_dim, same
// structure with run-time loops.  Bytes in flight per SM = (resident CTAs) x (staging warps) x 32 x D*e,
// chosen by the host.
#pragma once
#include "kvc_device.cuh"
#include "kvc_tma.cuh"

namespace kvc {

// log2 of the XOR-swizzle group: min(ctz(CPR), 3)
__host__ __device__ constexpr int swz_bits(int cpr) { return (cpr % 8 == 0) ? 3 : (cpr % 4 == 0) ? 2 : (cpr % 2 == 0) ? 1 : 0; }

// Sum of squares of one row held in a staging slot.  `row_addr` = shared address of the row.
// Compiled widths: chunk sums, balanced tree inside each aligned group of G chunks, groups in order.
// Generic width (CPR == 0): chunk sums added in chunk order (the G = 1 case of the same rule).
template <int DT, int CPR>
__device__ __forceinline__ float row_sumsq_smem(uint32_t row_addr, int lane, int cpr) {
    using Tr = Traits<DT>;
    if constexpr (CPR == 0) {
        float tot = 0.f;
        for (int c = 0; c < cpr; ++c) {
            const float a = Tr::sumsq(lds128(row_addr + c * 16), 0.f);
            tot = (c == 0) ? a : tot + a;
        }
        return tot;
    } else {
        constexpr int SB = swz_bits(CPR);
        constexpr int G = 1 << SB;
        const int x = (lane >> (3 - SB)) & (G - 1);
        uint32_t base[G];
#pragma unroll
        for (int m = 0; m < G; ++m) base[m] = row_addr + (uint32_t)(((m ^ x) - m) * 16);
        float acc[CPR];
#pragma unroll
        for (int c = 0; c < CPR; ++c) acc[c] = Tr::sumsq(lds128(base[c & (G - 1)] + c * 16), 0.f);
        float tot = 0.f;
#pragma unroll
        for (int g = 0; g < CPR / G; ++g) {
#pragma unroll
            for (int s = 1; s < G; s <<= 1) {
#pragma unroll
                for (int m = 0; m < G; m += 2 * s) acc[g * G + m] += acc[g * G + m + s];
            }
            tot = (g == 0) ? acc[0] : tot + acc[g * G];
        }
        return tot;
    }
}

// Load `rows` (1..32) rows of `rb` bytes into the warp's slot; lane l supplies the global address of row l.
// Consecutive rows (when `dense`: row stride == row bytes) are merged into one bulk copy per run.
// All 32 lanes must call; completion is observed with mbar_wait(bar, parity).
__device__ __forceinline__ void warp_load_rows(uint32_t slot, uint32_t bar, const char* src, int rows, bool dense,
                                               int lane, int rb) {
    const bool in = lane < rows;
    const unsigned long long a = (unsigned long long)src;
    const unsigned long long prev = __shfl_up_sync(0xffffffffu, a, 1);
    const bool head = in && (lane == 0 || !dense || a != prev + (unsigned)rb);
    const uint32_t heads = __ballot_sync(0xffffffffu, head);
    if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)(rows * rb));
    __syncwarp();
    if (head) {
        const uint32_t later = heads & ~((2u << lane) - 1u);  // heads above this lane
        const int next = later ? (__ffs(later) - 1) : rows;
        bulk_g2s(slot + (uint32_t)(lane * rb), src, (uint32_t)((next - lane) * rb), bar);
    }
}

// Source row of output row j of a unit: sink rows, then the selected rows, then the tail.
struct KeepMap {
    const int32_t* sidx;
    int sink, ksel, tail0;
    __device__ __forceinline__ int operator()(int j) const {
        return j < sink ? j : (j < sink + ksel ? sidx[j - sink] : j + tail0);
    }
};

// Per-row state of a unit follows its kept rows, in place (kvc_carry_layer): acc'[g][i] = acc[g][src(i)] when
// src(i) < prev, 0 otherwise, for the `group` acc rows of KV head h and i < C.  The group x C entries go in rounds of
// NT, g-major: every thread reads its entry, the CTA synchronises, every thread writes.  Kept rows ascend and never move
// up (src(i) >= i), so no later round reads an entry an earlier round wrote.  Entries that neither move nor become zero
// are not touched.  All NT threads call (CTA-uniform: c.acc != nullptr).
template <typename Key, int NT>
__device__ __forceinline__ void carry_unit(const CarryDev& c, const KeepMap& src_row, int C, int b, int h) {
    char* base = c.acc + (int64_t)b * c.asb + (int64_t)h * c.group * c.ash;
    const int n = c.group * C;
    for (int e0 = 0; e0 < n; e0 += NT) {
        const int e = e0 + (int)threadIdx.x;
        Key* row = nullptr;
        int i = 0;
        Key val = 0;
        bool write = false;
        if (e < n) {
            const int g = e / C;
            i = e - g * C;
            const int s = src_row(i);
            row = reinterpret_cast<Key*>(base + (int64_t)g * c.ash);
            write = s != i || s >= c.prev;
            if (write && s < c.prev) val = row[s];
        }
        __syncthreads();
        if (write) row[i] = val;
    }
}

// K3: rows [0, C) of the dense outputs from the kept source rows, K then V, 32 rows per staging warp per step.
// Called by the staging warps only (stage = this warp's index among the `nstage` of them).
__device__ __forceinline__ void gather_unit(const KeepMap& src_row, int C, const char* kbase, const char* vbase,
                                            int64_t kss, int64_t vss, char* ko, char* vo, int rb, uint32_t slot,
                                            uint32_t bar, uint32_t& parity, int stage, int nstage, int lane) {
    const bool kdense = kss == rb, vdense = vss == rb;
    const int nbc = (C + 31) >> 5;
    for (int t = stage; t < 2 * nbc; t += nstage) {
        const bool isv = t >= nbc;
        const int j0 = (isv ? t - nbc : t) << 5;
        const int rows = min(32, C - j0);
        const int row = lane < rows ? src_row(j0 + lane) : 0;
        const char* src = isv ? vbase + (int64_t)row * vss : kbase + (int64_t)row * kss;
        warp_load_rows(slot, bar, src, rows, isv ? vdense : kdense, lane, rb);
        mbar_wait(bar, parity);
        parity ^= 1;
        if (lane == 0) {
            bulk_s2g((isv ? vo : ko) + (int64_t)j0 * rb, slot, (uint32_t)(rows * rb));
            bulk_commit();
            bulk_wait_read<0>();  // the slot has been read out: it may be refilled
        }
        __syncwarp();
    }
}

// Radix keys of a selection region from per-row values held in global memory (stored key norms, or
// caller-supplied scores): level-0 histogram on the fly; snapkv keeps the raw values and their maximum for the
// pooling transform.  All NT threads call; hist must be zeroed and misc[kMiscMaxRaw] = 0 beforehand.
template <int DT, int NT>
__device__ __forceinline__ void keys_from_values(const typename Traits<DT>::Key* src, int R, int score,
                                                 typename Traits<DT>::Key* keys, uint32_t* hist, int32_t* misc) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    constexpr int kShift0 = Tr::kKeyBits - kHistBits;
    const bool snap = (score == KVC_SCORE_SNAPKV_POOL);
    const bool desc = (score == KVC_SCORE_L2_HIGH);
    uint32_t local_max = 0;
    load_keys_vectorised<DT, NT>(src, R, keys, [&](int i, uint32_t raw) {
        if (snap) {
            keys[i] = (Key)raw;
            local_max = max(local_max, raw);
        } else {
            const Key key = ordered_key<Key>(raw, desc);
            keys[i] = key;
            atomicAdd(&hist[(uint32_t)key >> kShift0], 1u);
        }
    });
    if (snap) {
        // norms are >= 0, so their raw bits order like unsigned integers
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) local_max = max(local_max, __shfl_xor_sync(0xffffffffu, local_max, o));
        if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<uint32_t*>(&misc[kMiscMaxRaw]), local_max);
    }
}

// Kept rows of a unit (layer descriptor L: LayerDev or SlabLayerDev, ksel > 0) from per-row values in memory:
//   GIVEN_INDEX                       caller-supplied rows (L.idx_in, [B,H,ksel]), clamped into the layer so that a bad
//                                     index can never become a wild bulk copy;
//   GIVEN_SCORE / GIVEN_SCORE_SHARED  caller-supplied scores of the region's rows (cache dtype, in the idx_in slot:
//                                     [B,H,R] per-head rows or [B,R] rows shared by the heads of a batch entry), pooled,
//                                     the highest kept;
//   otherwise                         stored key norms (norm_row: the unit's row of them), ranked like the scan would.
// All NT threads call.  hist and misc[kMiscMaxRaw] are reset here, behind a barrier before their first reader; sidx is
// complete after the caller's next __syncthreads().
template <int DT, int NT, typename Layer>
__device__ __forceinline__ void select_from_memory(const Layer& L, const typename Traits<DT>::Key* norm_row, int b, int bh,
                                                   typename Traits<DT>::Key* keys, uint32_t* hist, int32_t* misc,
                                                   int32_t* sidx) {
    using Key = typename Traits<DT>::Key;
    const int tid = threadIdx.x;
    const int R = L.hi - L.lo;
    if (L.score == KVC_SCORE_GIVEN_INDEX) {
        const int32_t* src = L.idx_in + (int64_t)bh * L.ksel;
        for (int i = tid; i < L.ksel; i += NT) sidx[i] = min(max(src[i], 0), L.S - 1);
        return;
    }
    for (int i = tid; i < kHistBins; i += NT) hist[i] = 0;
    if (tid == 0) misc[kMiscMaxRaw] = 0;
    __syncthreads();
    if (L.score == KVC_SCORE_GIVEN_SCORE || L.score == KVC_SCORE_GIVEN_SCORE_SHARED) {
        const Key* src = reinterpret_cast<const Key*>(L.idx_in) + (int64_t)(L.score == KVC_SCORE_GIVEN_SCORE ? bh : b) * R;
        load_keys_vectorised<DT, NT>(src, R, keys, [&](int i, uint32_t raw) { keys[i] = (Key)raw; });
        __syncthreads();
        snapkv_transform<DT, NT>(keys, R, L.pool, hist, misc, /*invert=*/false);
    } else {
        keys_from_values<DT, NT>(norm_row + L.lo, R, L.score, keys, hist, misc);
        __syncthreads();
        if (L.score == KVC_SCORE_SNAPKV_POOL) snapkv_transform<DT, NT>(keys, R, L.pool, hist, misc);
    }
    block_radix_select<Key, NT>(keys, R, L.ksel, hist, misc, sidx, L.lo);
}

template <int DT, int CPR, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) kvc_fused_tma_kernel(const __grid_constant__ BatchDev bd) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    constexpr int kShift0 = Tr::kKeyBits - kHistBits;
    const int cpr = CPR > 0 ? CPR : bd.cpr;
    const int RB = cpr * 16;  // row bytes

    const int bx = blockIdx.x, by = blockIdx.y;  // (batch, head) unit (or run of `upc` units) and layer of this CTA
    const LayerDev& L = bd.layers[by];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    extern __shared__ __align__(128) unsigned char smem[];
    int32_t* misc = reinterpret_cast<int32_t*>(smem);
    uint32_t* hist = reinterpret_cast<uint32_t*>(smem + bd.off_hist);
    int32_t* sidx = reinterpret_cast<int32_t*>(smem + bd.off_idx);
    Key* keys = reinterpret_cast<Key*>(smem + bd.off_keys);
    const int nsw = bd.nsw;
    const bool stager = warp < nsw;
    const uint32_t slot = smem_u32(smem + bd.off_stage) + (uint32_t)(warp * 32 * RB);
    const uint32_t bar = smem_u32(smem + kMiscInts * 4) + (uint32_t)warp * 8;
    uint32_t parity = 0;

    const int R = L.hi - L.lo;
    const int ksel = L.ksel;
    const int score = L.score;
    const bool kdense = L.kss == RB;
    const bool given_score = score == KVC_SCORE_GIVEN_SCORE || score == KVC_SCORE_GIVEN_SCORE_SHARED;
    const bool by_value = given_score || L.n_in != nullptr;  // per-row values come from memory
    const bool scan = ksel > 0 && score != KVC_SCORE_GIVEN_INDEX && !by_value;

    if (stager) {
        if (lane == 0) {
            mbar_init(bar, 1);
            mbar_init_fence();
        }
        __syncwarp();
    }
    // A CTA walks `upc` consecutive (batch, head) units (upc = 1 unless the lab build overrides it).
    const int n_units = bd.B * bd.H;
    const int bh_end = min(n_units, (bx + 1) * bd.upc);
    for (int bh = bx * bd.upc; bh < bh_end; ++bh) {
    const int b = bh / bd.H, h = bh - b * bd.H;
    if (bd.ws != nullptr) {  // selection too large for shared memory: keys / kept indices live in the workspace
        char* unit = bd.ws + ((int64_t)by * n_units + bh) * bd.ws_unit;
        keys = reinterpret_cast<Key*>(unit);
        sidx = reinterpret_cast<int32_t*>(unit + bd.ws_keys);
    }
    const char* kbase = L.k_in + (int64_t)b * L.ksb + (int64_t)h * L.ksh;
    const char* vbase = L.v_in + (int64_t)b * L.vsb + (int64_t)h * L.vsh;
    const char* kreg = kbase + (int64_t)L.lo * L.kss;
    const int nblk = (R + 31) >> 5;
    if (scan && stager && warp < nblk)  // first block is in flight while the histogram is cleared
        warp_load_rows(slot, bar, kreg + (int64_t)(warp * 32 + lane) * L.kss, min(32, R - warp * 32), kdense, lane, RB);

    if (ksel > 0 && (score == KVC_SCORE_GIVEN_INDEX || by_value)) {
        // ---------------------------------------------------------- kept rows, scores or stored key norms from memory
        const Key* norm_row = L.n_in ? reinterpret_cast<const Key*>(L.n_in + (int64_t)b * L.nsb + (int64_t)h * L.nsh)
                                     : nullptr;
        select_from_memory<DT, NT>(L, norm_row, b, bh, keys, hist, misc, sidx);
    } else if (ksel > 0) {
        // ---------------------------------------------------------- K1: scan
        for (int i = tid; i < kHistBins; i += NT) hist[i] = 0;
        if (tid == 0) misc[kMiscMaxRaw] = 0;
        __syncthreads();
        const bool snap = (score == KVC_SCORE_SNAPKV_POOL);
        const bool desc = (score == KVC_SCORE_L2_HIGH);
        uint32_t local_max = 0;
        if (stager) {
            for (int blk = warp; blk < nblk; blk += nsw) {
                const int r0 = blk << 5;
                const int rows = min(32, R - r0);
                mbar_wait(bar, parity);
                parity ^= 1;
                float ss = 0.f;
                if (lane < rows) ss = row_sumsq_smem<DT, CPR>(slot + (uint32_t)(lane * RB), lane, cpr);
                __syncwarp();  // every lane has consumed its row: the slot may be refilled
                const int nb = blk + nsw;
                if (nb < nblk)
                    warp_load_rows(slot, bar, kreg + (int64_t)(nb * 32 + lane) * L.kss, min(32, R - nb * 32), kdense,
                                   lane, RB);
                if (lane < rows) {
                    const uint32_t raw = Tr::to_raw(sqrtf(ss));
                    if (snap) {
                        keys[r0 + lane] = (Key)raw;
                        local_max = max(local_max, raw);
                    } else {
                        const Key key = ordered_key<Key>(raw, desc);
                        keys[r0 + lane] = key;
                        atomicAdd(&hist[(uint32_t)key >> kShift0], 1u);
                    }
                }
            }
        }
        if (snap) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) local_max = max(local_max, __shfl_xor_sync(0xffffffffu, local_max, o));
            if (lane == 0) atomicMax(reinterpret_cast<uint32_t*>(&misc[kMiscMaxRaw]), local_max);
        }
        __syncthreads();
        if (snap) snapkv_transform<DT, NT>(keys, R, L.pool, hist, misc);
        // ---------------------------------------------------------- K2: select
        block_radix_select<Key, NT>(keys, R, ksel, hist, misc, sidx, L.lo);
    }
    __syncthreads();  // sidx complete (GIVEN_INDEX path); no-op cost otherwise

    // -------------------------------------------------------------- K3: gather
    const int C = L.sink + ksel + L.tail;
    const KeepMap src_row{sidx, L.sink, ksel, L.S - L.tail - L.sink - ksel};
    if (L.idx_out != nullptr) {
        int32_t* io = L.idx_out + (int64_t)bh * C;
        for (int j = tid; j < C; j += NT) io[j] = src_row(j);
    }
    // accumulators follow their rows (sidx is complete: barrier above; it stays valid until the end-of-unit barrier)
    if (L.carry.acc != nullptr) carry_unit<Key, NT>(L.carry, src_row, C, b, h);
    if (stager)
        gather_unit(src_row, C, kbase, vbase, L.kss, L.vss, L.k_out + (int64_t)bh * C * RB,
                    L.v_out + (int64_t)bh * C * RB, RB, slot, bar, parity, warp, nsw, lane);
    __syncthreads();  // every warp is done with sidx / keys before the next unit reuses them
    }  // unit loop
}

}  // namespace kvc
