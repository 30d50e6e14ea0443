// kvc_slab.cuh — slab-cache kernels: in-place append (+ key norms) and in-place compaction.
//
// The container step on both sides of the compress call (SURVEY.md §8f rank 1): replaces the
// torch.cat of HF's cache.update (transformers cache_utils.py:119-120), the fresh-tensor gather of the
// compress functions and the rebuild in to_dynamic_cache (reference utils.py:12-27).
//
//   kvc_slab_append_kernel    one thread per appended row: copy K and V rows into the slab and
//                             record dtype(sqrt(sum k^2)) with the SAME chunk/tree summation as the
//                             fused scan (row_sumsq tree), so stored norms are bit-identical to what
//                             kvc_compress_layers would compute from the rows.
//   kvc_slab_compress_kernel  per (layer, batch, head): radix keys from the stored norms (2-4 B per
//                             token instead of D*e), select, then slide kept rows down in place.
//                             Rows move in rounds of (staging warps x 32) output rows: every warp
//                             bulk-loads its 32 source rows, the CTA synchronises, then every warp
//                             bulk-stores.  Kept rows are ascending and never move up (src >= dst),
//                             so sources of later rounds lie above every destination written so far.
//                             Optional per-row state (kvc_carry_layer: H2O accumulators, `group` rows per unit)
//                             slides the same way, before the early return of a unit whose rows all stay put.
#pragma once
#include "kvc_fused_tma.cuh"

namespace kvc {

struct SlabLayerDev {
    char* k;
    char* v;
    char* n;
    int32_t* idx_out;
    const int32_t* idx_in;
    int64_t ksb, ksh, vsb, vsh, nsb, nsh;  // BYTE strides (batch, head)
    int32_t S, sink, lo, hi, ksel, tail, score, pool;
    CarryDev carry;  // optional per-row state that slides with the kept rows
};
static_assert(sizeof(SlabLayerDev) == 152, "SlabLayerDev is passed by value in kernel params");

struct SlabBatchDev {
    int32_t B, H;
    int32_t idx_cap, nsw;
    int32_t cpr, pad0;  // cpr: 16-byte chunks per row (read by the generic-width kernel)
    int32_t off_hist, off_idx, off_keys, off_stage;
    char* ws;  // optional workspace (see BatchDev)
    int64_t ws_unit, ws_keys;
    SlabLayerDev layers[KVC_MAX_LAYERS_PER_LAUNCH];
};
static_assert(sizeof(SlabBatchDev) < 32 * 1024, "kernel parameters are limited to 32 KB");

struct AppendLayerDev {
    const char* k_new;
    const char* v_new;
    char* k;
    char* v;
    char* n;
    int64_t nksb, nksh, nkss, nvsb, nvsh, nvss;  // new rows: BYTE strides
    int64_t ksb, ksh, vsb, vsh, nsb, nsh;        // slab: BYTE strides
    int32_t cur_len, n_new;
};
static_assert(sizeof(AppendLayerDev) == 144, "AppendLayerDev is passed by value in kernel params");

struct AppendBatchDev {
    int32_t B, H;
    int32_t max_new, cpr;  // cpr: 16-byte chunks per row (read by the generic-width kernels)
    AppendLayerDev layers[KVC_MAX_LAYERS_PER_LAUNCH];
};

// One-layer form of the append parameters (the per-layer `update` of a decode loop): 160 bytes of kernel
// parameters instead of 9 KB, so the launch itself is as cheap as the torch.cat it replaces.
struct AppendOneDev {
    int32_t B, H;
    int32_t max_new, cpr;
    AppendLayerDev layers[1];
};

constexpr int kMiscFirst = 3;  // misc[] slot: first output row whose source row differs from it

// Same value as row_sumsq_smem (chunk sums + balanced tree; the tree is invariant under the
// scan's XOR read order), reading the row from global memory and optionally copying it.
template <int DT, int CPR>
__device__ __forceinline__ float row_sumsq_copy(const char* src, char* dst, int cpr) {
    using Tr = Traits<DT>;
    if constexpr (CPR == 0) {  // generic width: chunk sums in chunk order (row_sumsq_smem, CPR == 0)
        float tot = 0.f;
        for (int c = 0; c < cpr; ++c) {
            const int4 v = *reinterpret_cast<const int4*>(src + c * 16);
            const float a = Tr::sumsq(v, 0.f);
            tot = (c == 0) ? a : tot + a;
            *reinterpret_cast<int4*>(dst + c * 16) = v;
        }
        return tot;
    } else {
    constexpr int SB = swz_bits(CPR);
    constexpr int G = 1 << SB;
    float acc[CPR];
#pragma unroll
    for (int c = 0; c < CPR; ++c) {
        const int4 v = *reinterpret_cast<const int4*>(src + c * 16);
        acc[c] = Tr::sumsq(v, 0.f);
        *reinterpret_cast<int4*>(dst + c * 16) = v;
    }
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

template <int DT, int CPR, typename Params>
__global__ void __launch_bounds__(128) kvc_slab_append_kernel(const __grid_constant__ Params bd) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    const int cpr = CPR > 0 ? CPR : bd.cpr;
    const int RB = cpr * 16;
    const AppendLayerDev& L = bd.layers[blockIdx.y];
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // flat (bh, t)
    const int T = L.n_new;
    if (r >= (int64_t)bd.B * bd.H * T) return;
    const int bh = (int)(r / T), t = (int)(r - (int64_t)bh * T);
    const int b = bh / bd.H, h = bh - b * bd.H;
    const int row = L.cur_len + t;
    const char* ks = L.k_new + (int64_t)b * L.nksb + (int64_t)h * L.nksh + (int64_t)t * L.nkss;
    const char* vs = L.v_new + (int64_t)b * L.nvsb + (int64_t)h * L.nvsh + (int64_t)t * L.nvss;
    char* kd = L.k + (int64_t)b * L.ksb + (int64_t)h * L.ksh + (int64_t)row * RB;
    char* vd = L.v + (int64_t)b * L.vsb + (int64_t)h * L.vsh + (int64_t)row * RB;
    const float ss = row_sumsq_copy<DT, CPR>(ks, kd, cpr);
    if constexpr (CPR > 0) {
#pragma unroll
        for (int c = 0; c < CPR; ++c) *reinterpret_cast<int4*>(vd + c * 16) = *reinterpret_cast<const int4*>(vs + c * 16);
    } else {
        for (int c = 0; c < cpr; ++c) *reinterpret_cast<int4*>(vd + c * 16) = *reinterpret_cast<const int4*>(vs + c * 16);
    }
    Key* nd = reinterpret_cast<Key*>(L.n + (int64_t)b * L.nsb + (int64_t)h * L.nsh);
    nd[row] = (Key)Tr::to_raw(sqrtf(ss));
}

// Prefill-sized appends (T >= 32 rows per (b,h)): the thread-per-row kernel above reads and writes 16 B per
// lane at a row-sized stride (measured 2.2-2.8 TB/s).  Here every warp moves blocks of 32 rows through its own
// shared-memory slot with bulk copies — one load, one store per block when rows are contiguous — and each
// lane reduces one staged key row with the same chunk/tree summation (row_sumsq_smem) before the block leaves.
template <int DT, int CPR>
__global__ void __launch_bounds__(256, 3) kvc_slab_append_tma_kernel(const __grid_constant__ AppendBatchDev bd) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    const int cpr = CPR > 0 ? CPR : bd.cpr;
    const int RB = cpr * 16;
    const AppendLayerDev& L = bd.layers[blockIdx.y];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t bar = smem_u32(smem) + (uint32_t)warp * 8;
    const uint32_t slot = smem_u32(smem + 128) + (uint32_t)(warp * 32 * RB);
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_init_fence();
    }
    __syncwarp();
    const int T = L.n_new;
    const int nblk = (T + 31) >> 5;
    const int64_t n_items = (int64_t)bd.B * bd.H * nblk;
    const bool kdense = L.nkss == RB, vdense = L.nvss == RB;
    uint32_t parity = 0;
    for (int64_t item = (int64_t)blockIdx.x * 8 + warp; item < n_items; item += (int64_t)gridDim.x * 8) {
        const int bh = (int)(item / nblk), rb = (int)(item - (int64_t)bh * nblk);
        const int b = bh / bd.H, h = bh - b * bd.H;
        const int t0 = rb << 5;
        const int rows = min(32, T - t0);
        const int row0 = L.cur_len + t0;
        const char* ks = L.k_new + (int64_t)b * L.nksb + (int64_t)h * L.nksh + (int64_t)(t0 + lane) * L.nkss;
        const char* vs = L.v_new + (int64_t)b * L.nvsb + (int64_t)h * L.nvsh + (int64_t)(t0 + lane) * L.nvss;
        char* kd = L.k + (int64_t)b * L.ksb + (int64_t)h * L.ksh + (int64_t)row0 * RB;
        char* vd = L.v + (int64_t)b * L.vsb + (int64_t)h * L.vsh + (int64_t)row0 * RB;
        // keys: stage, reduce, store
        warp_load_rows(slot, bar, ks, rows, kdense, lane, RB);
        mbar_wait(bar, parity);
        parity ^= 1;
        if (lane < rows) {
            const float ss = row_sumsq_smem<DT, CPR>(slot + (uint32_t)(lane * RB), lane, cpr);
            Key* nd = reinterpret_cast<Key*>(L.n + (int64_t)b * L.nsb + (int64_t)h * L.nsh);
            nd[row0 + lane] = (Key)Tr::to_raw(sqrtf(ss));
        }
        __syncwarp();
        if (lane == 0) {
            bulk_s2g(kd, slot, (uint32_t)(rows * RB));
            bulk_commit();
            bulk_wait_read<0>();
        }
        __syncwarp();
        // values: stage, store
        warp_load_rows(slot, bar, vs, rows, vdense, lane, RB);
        mbar_wait(bar, parity);
        parity ^= 1;
        if (lane == 0) {
            bulk_s2g(vd, slot, (uint32_t)(rows * RB));
            bulk_commit();
            bulk_wait_read<0>();
        }
        __syncwarp();
    }
}

template <int DT, int CPR, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) kvc_slab_compress_kernel(const __grid_constant__ SlabBatchDev bd) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    const int RB = (CPR > 0 ? CPR : bd.cpr) * 16;

    const SlabLayerDev& L = bd.layers[blockIdx.y];
    const int bh = blockIdx.x;
    const int b = bh / bd.H, h = bh - b * bd.H;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    extern __shared__ __align__(128) unsigned char smem[];
    int32_t* misc = reinterpret_cast<int32_t*>(smem);
    uint32_t* hist = reinterpret_cast<uint32_t*>(smem + bd.off_hist);
    int32_t* sidx = reinterpret_cast<int32_t*>(smem + bd.off_idx);
    Key* keys = reinterpret_cast<Key*>(smem + bd.off_keys);
    if (bd.ws != nullptr) {
        char* unit = bd.ws + ((int64_t)blockIdx.y * gridDim.x + bh) * bd.ws_unit;
        keys = reinterpret_cast<Key*>(unit);
        sidx = reinterpret_cast<int32_t*>(unit + bd.ws_keys);
    }
    const int nsw = bd.nsw;
    const bool stager = warp < nsw;
    const uint32_t slot = smem_u32(smem + bd.off_stage) + (uint32_t)(warp * 32 * RB);
    const uint32_t bar = smem_u32(smem + kMiscInts * 4) + (uint32_t)warp * 8;
    uint32_t parity = 0;
    if (lane == 0) {  // every warp: the slide below stages rows in more slots than the launch plan has (see there)
        mbar_init(bar, 1);
        mbar_init_fence();
    }
    __syncwarp();

    const int ksel = L.ksel;
    char* kbase = L.k + (int64_t)b * L.ksb + (int64_t)h * L.ksh;
    char* vbase = L.v + (int64_t)b * L.vsb + (int64_t)h * L.vsh;
    Key* nbase = reinterpret_cast<Key*>(L.n + (int64_t)b * L.nsb + (int64_t)h * L.nsh);
    const int sink = L.sink;
    const int C = sink + ksel + L.tail;
    const int tail0 = L.S - L.tail - sink - ksel;  // src row = j + tail0 for tail rows

    if (tid == 0) misc[kMiscFirst] = C;
    // kept rows (strictly ascending absolute rows of the region, kvc.h), scores (the vote mode of snapkv_lite, H2O's
    // head-summed attention mass) or the stored norms
    if (ksel > 0) select_from_memory<DT, NT>(L, nbase, b, bh, keys, hist, misc, sidx);
    __syncthreads();

    const KeepMap src_row{sidx, sink, ksel, tail0};
    // ---------------------------------------------------------- first row that actually moves
    {
        int first = C;
        for (int j = tid; j < C; j += NT)
            if (src_row(j) != j) {
                first = j;
                break;  // rows are ascending: this thread's later rows move too
            }
        if (first < C) atomicMin(&misc[kMiscFirst], first);
    }
    if (L.idx_out != nullptr) {
        int32_t* io = L.idx_out + (int64_t)bh * C;
        for (int j = tid; j < C; j += NT) io[j] = src_row(j);
    }
    __syncthreads();
    const int jf = misc[kMiscFirst];
    // accumulators follow their rows, before the early return: entries past prev_len become 0 even when no row moves
    if (L.carry.acc != nullptr) carry_unit<Key, NT>(L.carry, src_row, C, b, h);
    if (jf >= C) return;  // nothing moves (CTA-uniform)

    // ---------------------------------------------------------- slide rows down, K then V, in rounds
    // The radix keys are dead once the kept indices exist: when they live on chip their shared memory joins the
    // staging area, so a round moves up to NT/32 blocks of 32 rows instead of `nsw` (at 32K rows the plan leaves 4
    // slots next to 64 KB of keys: 8 rounds of load -> barrier -> store per unit become 4).
    int g_nsw = nsw;
    uint32_t g_slot = slot;
    if (bd.ws == nullptr) {
        const int lo = (bd.off_keys + 127) & ~127;
        const int room = bd.off_stage + nsw * (32 * RB) - lo;
        g_nsw = min(NT / 32, room / (32 * RB));
        g_slot = smem_u32(smem + lo) + (uint32_t)(warp * 32 * RB);
    }
    const bool g_stager = warp < g_nsw;
    const int nb = (C - jf + 31) >> 5;
    for (int t0 = 0; t0 < 2 * nb; t0 += g_nsw) {
        const int t = t0 + warp;
        const bool active = g_stager && t < 2 * nb;
        const bool isv = t >= nb;
        const int j0 = jf + ((isv ? t - nb : t) << 5);
        const int rows = min(32, C - j0);
        if (active) {
            const int j = j0 + lane;
            const int row = lane < rows ? src_row(j) : 0;
            const char* src = (isv ? vbase : kbase) + (int64_t)row * RB;
            warp_load_rows(g_slot, bar, src, rows, true, lane, RB);
            mbar_wait(bar, parity);
            parity ^= 1;
        }
        __syncthreads();  // every source row of this round is on chip before any destination is written
        if (active) {
            if (lane == 0) {
                bulk_s2g((isv ? vbase : kbase) + (int64_t)j0 * RB, g_slot, (uint32_t)(rows * RB));
                bulk_commit();
                bulk_wait_read<0>();
            }
            __syncwarp();
        }
    }
    // ---------------------------------------------------------- norms slide with their rows
    for (int c0 = jf; c0 < C; c0 += NT) {
        const int j = c0 + tid;
        Key val = 0;
        if (j < C) val = nbase[src_row(j)];
        __syncthreads();
        if (j < C) nbase[j] = val;
    }
}

}  // namespace kvc
