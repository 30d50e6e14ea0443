// kvc_device.cuh — device-side building blocks of the sm_100a KV-compression path.
//
//   K1  Traits<DT>::sumsq         fp32 sum of squares of one 16-byte chunk of a key row (the rows themselves are
//                                 staged by the TMA unit, kvc_fused_tma.cuh)
//                                 (replaces torch.norm(K, p=2, dim=-1), e.g. l2_compress.py:70)
//   K2  block_radix_select        per-(b,h) radix select in shared memory: 11-bit histogram
//                                 fused into the scan, then refinement passes over the
//                                 on-chip keys; ties go to the lowest token index; indices
//                                 are emitted already ascending (replaces argsort + [:k] +
//                                 torch.sort, e.g. h2o_l2.py:128-132, and topk + sort,
//                                 snapkv_lite.py:134-137)
//
// Everything here is HBM-bound byte/compare work: no tensor cores on purpose.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "kvc.h"

namespace kvc {

constexpr int kHistBits = 11;
constexpr int kHistBins = 1 << kHistBits;  // 2048 bins * 4 B = 8 KB
constexpr int kMiscInts = 128;             // 512 B of per-CTA scalars / per-warp counters
constexpr int kMaxPoolHalo = 32;           // pooling_kernel <= 64

// misc[] slots
constexpr int kMiscBin = 0;     // find_bin result: bin
constexpr int kMiscBelow = 1;   // find_bin result: count strictly below bin
constexpr int kMiscMaxRaw = 2;  // snapkv: max norm (raw dtype bits, positive => integer order)
constexpr int kMiscWarpA = 32;  // 32 ints: per-warp counter A (scan totals / lt counts)
constexpr int kMiscWarpB = 64;  // 32 ints: per-warp counter B (eq counts)
constexpr int kMiscHalo = 96;   // 32 ints: snapkv pooling halo (raw norms of the previous tile's tail)

// ---------------------------------------------------------------- launch descriptors
// Per-row state that moves with the kept rows (kvc_carry_layer): `group` rows of acc per (batch, KV head) unit.
struct CarryDev {
    char* acc;             // nullptr: nothing to carry for this layer
    int64_t asb, ash;      // BYTE strides (batch, acc head)
    int32_t group, prev;   // prev: valid entries before the compaction, already clamped to S
};
static_assert(sizeof(CarryDev) == 32, "CarryDev is part of the kernel parameters");

struct LayerDev {
    const char* k_in;
    const char* v_in;
    char* k_out;
    char* v_out;
    int32_t* idx_out;
    const int32_t* idx_in;
    int64_t ksb, ksh, kss;  // BYTE strides of K (batch, head, row)
    int64_t vsb, vsh, vss;  // BYTE strides of V
    int32_t S, sink, lo, hi, ksel, tail, score, pool;
    const char* n_in;       // optional stored key norms [B,H,>=S] (cache dtype): scores without reading K
    int64_t nsb, nsh;       // BYTE strides of the norm array (batch, head)
    CarryDev carry;         // optional per-row state compacted in place with the kept rows
};
static_assert(sizeof(LayerDev) == 184, "LayerDev is passed by value in kernel params");

struct BatchDev {
    int32_t B, H;
    int32_t idx_cap;   // ints reserved for the kept-index list in shared memory
    int32_t cpr;       // 16-byte chunks per row (the generic-width kernels read it at run time)
    int32_t pad0, pad1;
    int32_t nsw;       // TMA form: warps that own a staging slot (<= warps per CTA)
    int32_t off_hist, off_idx, off_keys, off_stage;  // TMA form: shared-memory layout (bytes)
    int32_t upc;       // TMA form: consecutive (batch, head) units walked by one CTA
    // optional device workspace for selections that do not fit on chip: per unit, radix keys then kept indices
    char* ws;
    int64_t ws_unit;   // bytes per (layer, batch, head) unit
    int64_t ws_keys;   // bytes of the key part of a unit
    LayerDev layers[KVC_MAX_LAYERS_PER_LAUNCH];
};
static_assert(sizeof(BatchDev) < 32 * 1024, "kernel parameters are limited to 32 KB");

// ---------------------------------------------------------------- dtype traits
template <int DT>
struct Traits;
template <>
struct Traits<KVC_DTYPE_F32> {
    using Key = uint32_t;
    static constexpr int kElemBytes = 4;
    static constexpr int kKeyBits = 32;
    __device__ static __forceinline__ uint32_t to_raw(float x) { return __float_as_uint(x); }
    __device__ static __forceinline__ float from_raw(uint32_t r) { return __uint_as_float(r); }
    __device__ static __forceinline__ float sumsq(int4 v, float acc) {
        float a = __int_as_float(v.x), b = __int_as_float(v.y), c = __int_as_float(v.z), d = __int_as_float(v.w);
        acc = fmaf(a, a, acc);
        acc = fmaf(b, b, acc);
        acc = fmaf(c, c, acc);
        acc = fmaf(d, d, acc);
        return acc;
    }
};
template <>
struct Traits<KVC_DTYPE_BF16> {
    using Key = uint16_t;
    static constexpr int kElemBytes = 2;
    static constexpr int kKeyBits = 16;
    __device__ static __forceinline__ uint32_t to_raw(float x) {
        return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(x));
    }
    __device__ static __forceinline__ float from_raw(uint32_t r) { return __uint_as_float(r << 16); }
    __device__ static __forceinline__ float sumsq(int4 v, float acc) {
        const uint32_t w[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float lo = __uint_as_float(w[i] << 16);
            float hi = __uint_as_float(w[i] & 0xffff0000u);
            acc = fmaf(lo, lo, acc);
            acc = fmaf(hi, hi, acc);
        }
        return acc;
    }
};
template <>
struct Traits<KVC_DTYPE_F16> {
    using Key = uint16_t;
    static constexpr int kElemBytes = 2;
    static constexpr int kKeyBits = 16;
    __device__ static __forceinline__ uint32_t to_raw(float x) {
        return (uint32_t)__half_as_ushort(__float2half_rn(x));
    }
    __device__ static __forceinline__ float from_raw(uint32_t r) {
        return __half2float(__ushort_as_half((unsigned short)r));
    }
    __device__ static __forceinline__ float sumsq(int4 v, float acc) {
        const uint32_t w[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float lo = __half2float(__ushort_as_half((unsigned short)(w[i] & 0xffffu)));
            float hi = __half2float(__ushort_as_half((unsigned short)(w[i] >> 16)));
            acc = fmaf(lo, lo, acc);
            acc = fmaf(hi, hi, acc);
        }
        return acc;
    }
};

// Round an fp32 value to the storage dtype and back (what a torch op on that dtype returns).
template <int DT>
__device__ __forceinline__ float round_dt(float x) {
    return Traits<DT>::from_raw(Traits<DT>::to_raw(x));
}

// IEEE bits -> unsigned key whose integer order equals the float order (-x < +x, +NaN last).
template <typename Key>
__device__ __forceinline__ Key ordered_key(uint32_t raw, bool descending) {
    constexpr int kBits = sizeof(Key) * 8;
    const uint32_t sign = (raw >> (kBits - 1)) & 1u;
    uint32_t k = sign ? ~raw : (raw | (1u << (kBits - 1)));
    if (descending) k = ~k;
    return (Key)k;
}

// ---------------------------------------------------------------- memory helpers
__device__ __forceinline__ int4 ldg128_stream(const void* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg128_stream(void* p, int4 v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}

// ---------------------------------------------------------------- K1 (stand-alone kvc_key_norms): lane-group reduction
// Sum over groups of n consecutive lanes (n a power of two).
__device__ __forceinline__ float group_sum_pow2(float v, int n) {
    for (int o = n >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------- K2: block radix select
// Exclusive block scan over the histogram to find the bin holding the k-th smallest key
// (1-based k).  Writes misc[kMiscBin], misc[kMiscBelow]; ends with __syncthreads().
template <int NT>
__device__ __forceinline__ void find_bin(const uint32_t* hist, int nbins, uint32_t k, int32_t* misc) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (nbins + NT - 1) / NT;
    const int b0 = tid * per;
    uint32_t loc = 0;
    if ((per & 3) == 0) {
        for (int i = 0; i < per; i += 4) {
            if (b0 + i < nbins) {
                uint4 h = *reinterpret_cast<const uint4*>(hist + b0 + i);
                loc += h.x + h.y + h.z + h.w;
            }
        }
    } else {
        for (int i = 0; i < per; ++i)
            if (b0 + i < nbins) loc += hist[b0 + i];
    }
    uint32_t inc = loc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) misc[kMiscWarpA + warp] = (int32_t)inc;
    __syncthreads();
    uint32_t wbase = 0;
    for (int w = 0; w < warp; ++w) wbase += (uint32_t)misc[kMiscWarpA + w];
    const uint32_t excl = wbase + inc - loc;
    if (excl < k && k <= excl + loc) {  // exactly one thread
        uint32_t c = excl;
        for (int i = 0; i < per; ++i) {
            const uint32_t h = hist[b0 + i];
            if (c + h >= k) {
                misc[kMiscBin] = b0 + i;
                misc[kMiscBelow] = (int32_t)c;
                break;
            }
            c += h;
        }
    }
    __syncthreads();
}

// Select the k (1 <= k <= R) smallest keys of keys[0..R) (ties -> lowest index) and write
// their positions, ascending, as base + position into out_idx[0..k).
// Precondition: hist[] already holds the histogram of (key >> (KeyBits-12)) over all R keys
// (it is accumulated while the keys are produced), and a __syncthreads() has made keys/hist
// visible.  All NT threads must call.  Ends with __syncthreads().
template <typename Key, int NT>
__device__ __forceinline__ void block_radix_select(const Key* __restrict__ keys, int R, int k, uint32_t* hist,
                                                   int32_t* misc, int32_t* out_idx, int base) {
    constexpr int kBits = sizeof(Key) * 8;
    constexpr int kVec = 16 / sizeof(Key);  // keys per 128-bit shared load
    constexpr int NW = NT / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    uint32_t prefix = 0;  // the high `pbits` bits of the k-th key found so far
    int pbits = 0;
    uint32_t krem = (uint32_t)k;
    // level 0: the fused 11-bit histogram
    find_bin<NT>(hist, kHistBins, krem, misc);
    prefix = (uint32_t)misc[kMiscBin];
    krem -= (uint32_t)misc[kMiscBelow];
    pbits = kHistBits;
    // refinement levels over the remaining low bits
    while (pbits < kBits) {
        const int nb = (kBits - pbits) > kHistBits ? kHistBits : (kBits - pbits);
        const int shift = kBits - pbits - nb;
        const int nbins = 1 << nb;
        for (int i = tid; i < nbins; i += NT) hist[i] = 0;
        __syncthreads();
        const int nvec = (R + kVec - 1) / kVec;
        for (int v = tid; v < nvec; v += NT) {
            const int4 raw = *reinterpret_cast<const int4*>(keys + (size_t)v * kVec);
            const Key* kk = reinterpret_cast<const Key*>(&raw);
#pragma unroll
            for (int e = 0; e < kVec; ++e) {
                const uint32_t key = kk[e];
                if (v * kVec + e < R && (key >> (shift + nb)) == prefix)
                    atomicAdd(&hist[(key >> shift) & (uint32_t)(nbins - 1)], 1u);
            }
        }
        __syncthreads();
        find_bin<NT>(hist, nbins, krem, misc);
        prefix = (prefix << nb) | (uint32_t)misc[kMiscBin];
        krem -= (uint32_t)misc[kMiscBelow];
        pbits += nb;
    }
    // prefix == T, the k-th smallest key; take every key < T and the first `krem` keys == T.
    // Both passes read 16 bytes per lane (kVec consecutive keys), so a warp step covers 32 * kVec keys in index
    // order: lane-major, element-minor.  (One key per lane per step cost 0.9 warp instructions per key, a fifth of
    // the in-place kernel at 32K rows: profiles/r01_slab_ncu_full_c4.json.)
    const uint32_t T = prefix;
    const int r = (int)krem;
    constexpr int kStep = 32 * kVec;
    const int chunk = (((R + NW - 1) / NW) + kStep - 1) / kStep * kStep;  // keys per warp, multiple of a warp step
    const int w_lo = warp * chunk;
    const int w_hi = min(R, w_lo + chunk);
    int lt = 0, eq = 0;
    for (int i = w_lo + lane * kVec; i < w_hi; i += kStep) {
        const int4 raw = *reinterpret_cast<const int4*>(keys + i);  // the array is padded to 16 bytes
        const Key* kk = reinterpret_cast<const Key*>(&raw);
#pragma unroll
        for (int e = 0; e < kVec; ++e) {
            const uint32_t key = kk[e];
            const bool in = i + e < w_hi;
            lt += in && key < T;
            eq += in && key == T;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lt += __shfl_xor_sync(0xffffffffu, lt, o);
        eq += __shfl_xor_sync(0xffffffffu, eq, o);
    }
    __syncthreads();  // find_bin readers of misc[kMiscWarpA..] are done
    if (lane == 0) {
        misc[kMiscWarpA + warp] = lt;
        misc[kMiscWarpB + warp] = eq;
    }
    __syncthreads();
    int eq_before = 0, out_pos = 0;
    for (int w = 0; w < warp; ++w) {
        const int e = misc[kMiscWarpB + w];
        out_pos += misc[kMiscWarpA + w] + max(0, min(e, r - eq_before));
        eq_before += e;
    }
    auto warp_inclusive = [&](int v) {
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += t;
        }
        return v;
    };
    for (int i0 = w_lo; i0 < w_hi; i0 += kStep) {
        const int i = i0 + lane * kVec;
        uint32_t m_lt = 0, m_eq = 0;  // bit e: element e of this lane is < T / == T
        if (i < w_hi) {
            const int4 raw = *reinterpret_cast<const int4*>(keys + i);
            const Key* kk = reinterpret_cast<const Key*>(&raw);
#pragma unroll
            for (int e = 0; e < kVec; ++e) {
                const uint32_t key = kk[e];
                const bool in = i + e < w_hi;
                m_lt |= (uint32_t)(in && key < T) << e;
                m_eq |= (uint32_t)(in && key == T) << e;
            }
        }
        uint32_t m_take = m_lt;
        const bool any_eq = __any_sync(0xffffffffu, m_eq != 0);
        if (any_eq) {  // ties: the first r keys equal to T, in index order
            const int c_eq = __popc(m_eq);
            const int incl = warp_inclusive(c_eq);
            int seen = eq_before + incl - c_eq;
#pragma unroll
            for (int e = 0; e < kVec; ++e) {
                if ((m_eq >> e) & 1u) {
                    if (seen < r) m_take |= 1u << e;
                    ++seen;
                }
            }
            eq_before += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (__any_sync(0xffffffffu, m_take != 0)) {
            const int c_take = __popc(m_take);
            const int incl = warp_inclusive(c_take);
            int pos = out_pos + incl - c_take;
#pragma unroll
            for (int e = 0; e < kVec; ++e)
                if ((m_take >> e) & 1u) out_idx[pos++] = base + i + e;
            out_pos += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
    __syncthreads();
}


// ---------------------------------------------------------------- per-row scores from global memory
// Calls emit(i, raw) for every element of src[0..R) (dtype bits, 2 or 4 bytes): 16-byte loads, 4 in flight per
// thread (a one-element-per-thread loop is latency-bound: profiles/r01_slab_ncu_full_c5_before_vec.json — 48 % of
// stall samples on 2-byte loads).  Lines that straddle the ends are read element by element; short arrays keep
// one element per thread so that every thread is busy.
// NC = false: plain (coherent) loads, for values the SAME kernel wrote earlier (the fused vote's scores).
template <int DT, int NT, bool NC = true, typename Emit>
__device__ __forceinline__ void load_keys_vectorised(const typename Traits<DT>::Key* src, int R,
                                                     typename Traits<DT>::Key* /*keys*/, Emit emit) {
    using Key = typename Traits<DT>::Key;
    constexpr int KV = 16 / (int)sizeof(Key);
    constexpr int U = 4;
    const int tid = threadIdx.x;
    if (R < 8 * NT) {
        for (int i = tid; i < R; i += NT) emit(i, (uint32_t)src[i]);
        return;
    }
    const int a = (int)(((uintptr_t)src & 15) / sizeof(Key));  // elements of the first line before the array
    const int4* lines = reinterpret_cast<const int4*>((uintptr_t)src & ~(uintptr_t)15);
    const int nline = (a + R + KV - 1) / KV;
    for (int c0 = tid; c0 < nline; c0 += NT * U) {
        int4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + u * NT;
            const bool whole = c < nline && c * KV - a >= 0 && (c + 1) * KV - a <= R;
            v[u] = whole ? (NC ? __ldg(lines + c) : *(lines + c)) : make_int4(0, 0, 0, 0);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + u * NT;
            if (c >= nline) continue;
            const int i0 = c * KV - a;
            if (i0 >= 0 && i0 + KV <= R) {
                const Key* kk = reinterpret_cast<const Key*>(&v[u]);
#pragma unroll
                for (int e = 0; e < KV; ++e) emit(i0 + e, (uint32_t)kk[e]);
            } else {
                for (int e = 0; e < KV; ++e)
                    if (i0 + e >= 0 && i0 + e < R) emit(i0 + e, (uint32_t)src[i0 + e]);
            }
        }
    }
}

// ---------------------------------------------------------------- snapkv score transform
// keys[0..R) hold the RAW norms (dtype bits) and misc[kMiscMaxRaw] their maximum.  Rewrites them
// in place as descending-order radix keys of
//   score_i = dt(dt(max + 1e-6) - norm_i);  pooled_i = dt(fp32 left-to-right sum of the zero-padded
//   window / kernel)                        (snapkv_lite.py:96-121; avg_pool1d, count_include_pad)
// and accumulates the level-0 histogram.  Every warp owns a contiguous segment and walks it 32 rows
// at a time holding the previous / current / next 32 raw norms in registers (window taps are warp
// shuffles), so the rewrite is in place without per-tile barriers; only the two segment-boundary
// windows are read before a single __syncthreads().  All NT threads must call; ends synchronised.
// Pooling kernels 2..9 (the reference's default is 5), R >= PK.  Every lane owns FOUR consecutive rows of a 128-row
// block: each raw norm is turned into its score once, a window needs at most the four scores of the lane on either
// side (two shuffles up, two down for PK = 5; the block edges come from the previous block's lane 31 and the next
// block's lane 0, already in registers), and the taps are compile-time register indices.  ~0.9 warp instructions per
// row against 5.3 for the one-row-per-lane form below (profiles/r01_slab_ncu_full_c4.json: 57 % of the in-place
// kernel's samples sat in that loop).  Same left-to-right fp32 sums: a tap outside [0, R) adds +0.0f, which leaves a
// sum that started from +0.0f unchanged bit for bit.
template <int DT, int NT, int PK>
__device__ __forceinline__ void snapkv_transform_rows4(typename Traits<DT>::Key* keys, int R, uint32_t* hist,
                                                       float mxe, bool invert) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    constexpr int kShift0 = Tr::kKeyBits - kHistBits;
    constexpr int NW = NT / 32;
    constexpr int PAD = PK / 2;
    static_assert(PK >= 2 && PK <= 9, "window reaches at most four rows to either side");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float den = (float)PK;
    const int blocks = (R + 127) >> 7;
    const int bpw = (blocks + NW - 1) / NW;
    const int w_lo = warp * bpw * 128;
    const int w_hi = min(R, w_lo + bpw * 128);
    auto score = [&](uint32_t raw, int i) -> float {
        if (i < 0 || i >= R) return 0.f;
        return invert ? round_dt<DT>(mxe - Tr::from_raw(raw)) : Tr::from_raw(raw);
    };
    auto load4 = [&](int i0, float (&out)[4]) {  // scores of rows i0..i0+3 (i0 a multiple of 4)
        Key r[4] = {0, 0, 0, 0};
        if (i0 < R) {
            if (sizeof(Key) == 2)
                *reinterpret_cast<uint2*>(r) = *reinterpret_cast<const uint2*>(keys + i0);
            else
                *reinterpret_cast<uint4*>(r) = *reinterpret_cast<const uint4*>(keys + i0);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) out[k] = score((uint32_t)r[k], i0 + k);
    };
    // the same without the per-row range checks, for blocks that lie entirely inside [0, R)
    auto load4_inside = [&](int i0, float (&out)[4]) {
        Key r[4];
        if (sizeof(Key) == 2)
            *reinterpret_cast<uint2*>(r) = *reinterpret_cast<const uint2*>(keys + i0);
        else
            *reinterpret_cast<uint4*>(r) = *reinterpret_cast<const uint4*>(keys + i0);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            out[k] = invert ? round_dt<DT>(mxe - Tr::from_raw((uint32_t)r[k])) : Tr::from_raw((uint32_t)r[k]);
    };
    float left_edge[4], after[4], s[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int il = w_lo - 4 + k, ia = w_hi + k;
        left_edge[k] = score(il >= 0 && il < R ? (uint32_t)keys[il] : 0u, il);
        after[k] = score(ia >= 0 && ia < R ? (uint32_t)keys[ia] : 0u, ia);
    }
    load4(w_lo + 4 * lane, s);
    __syncthreads();  // every warp holds its boundary rows before any segment is rewritten
    // One 128-row block.  INSIDE (a compile-time switch, two instantiations of the body): the block AND the next one
    // lie entirely inside [0, R), so no load, store or histogram update needs a range check — all but the last one or
    // two blocks of a unit.  With the checks on every row the block cost 241 warp instructions, ~100 of them compares,
    // branches and index arithmetic (profiles/r02_slab_ncu_full_c4.json).
    auto block = [&](int b0, auto inside_tag) {
        constexpr bool INSIDE = decltype(inside_tag)::value;
        float n[4];
        if (b0 + 128 < w_hi) {
            if (INSIDE)
                load4_inside(b0 + 128 + 4 * lane, n);
            else
                load4(b0 + 128 + 4 * lane, n);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) n[k] = after[k];
        }
        float win[12];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float up = __shfl_up_sync(0xffffffffu, s[k], 1);
            const float dn = __shfl_down_sync(0xffffffffu, s[k], 1);
            const float nx = __shfl_sync(0xffffffffu, n[k], 0);
            win[k] = lane == 0 ? left_edge[k] : up;
            win[4 + k] = s[k];
            win[8 + k] = lane == 31 ? nx : dn;
        }
        const int i0 = b0 + 4 * lane;
        Key out[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            float acc = 0.f;
#pragma unroll
            for (int t = 0; t < PK; ++t) acc += win[4 + r + t - PAD];
            out[r] = ordered_key<Key>(Tr::to_raw(round_dt<DT>(acc / den)), /*descending=*/true);
        }
        if (INSIDE || i0 + 4 <= R) {
            if (sizeof(Key) == 2)
                *reinterpret_cast<uint2*>(keys + i0) = *reinterpret_cast<const uint2*>(out);
            else
                *reinterpret_cast<uint4*>(keys + i0) = *reinterpret_cast<const uint4*>(out);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            if (INSIDE || i0 + r < R) {
                if (!INSIDE && i0 + 4 > R) keys[i0 + r] = out[r];
                atomicAdd(&hist[(uint32_t)out[r] >> kShift0], 1u);
            }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            left_edge[k] = __shfl_sync(0xffffffffu, s[k], 31);
            s[k] = n[k];
        }
    };
    int b0 = w_lo;
    for (; b0 + 256 <= R && b0 < w_hi; b0 += 128) block(b0, std::true_type{});
    for (; b0 < w_hi; b0 += 128) block(b0, std::false_type{});
    __syncthreads();
}

template <int DT, int NT>
__device__ __forceinline__ void snapkv_transform(typename Traits<DT>::Key* keys, int R, int pk, uint32_t* hist,
                                                 int32_t* misc, bool invert = true) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    constexpr int kShift0 = Tr::kKeyBits - kHistBits;
    constexpr int NW = NT / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float mx = Tr::from_raw((uint32_t)misc[kMiscMaxRaw]);
    const float mxe = round_dt<DT>(mx + 1e-6f);
    if (R >= pk) {  // block-uniform
        switch (pk) {
            case 3: return snapkv_transform_rows4<DT, NT, 3>(keys, R, hist, mxe, invert);
            case 5: return snapkv_transform_rows4<DT, NT, 5>(keys, R, hist, mxe, invert);
            case 7: return snapkv_transform_rows4<DT, NT, 7>(keys, R, hist, mxe, invert);
            default: break;  // other kernel sizes (and no pooling) take the generic form
        }
    }
    const bool pooling = pk > 1 && R >= pk;
    const int pad = pooling ? pk / 2 : 0;
    const int taps = pooling ? pk : 1;
    const float den = (float)pk;
    const int steps = (R + 31) >> 5;
    const int spw = (steps + NW - 1) / NW;
    const int w_lo = warp * spw * 32;
    const int w_hi = min(R, w_lo + spw * 32);
    auto raw_at = [&](int i) -> uint32_t { return (i >= 0 && i < R) ? (uint32_t)keys[i] : 0u; };
    uint32_t prev = raw_at(w_lo - 32 + lane);
    const uint32_t after = raw_at(w_hi + lane);
    uint32_t cur = raw_at(w_lo + lane);
    __syncthreads();  // boundary windows are in registers before any segment is rewritten
    for (int i0 = w_lo; i0 < w_hi; i0 += 32) {
        const uint32_t next = (i0 + 32 >= w_hi) ? after : raw_at(i0 + 32 + lane);
        const int i = i0 + lane;
        float acc = 0.f;
        for (int t = 0; t < taps; ++t) {
            const int d = t - pad;
            const int sl = lane + d;
            const uint32_t vp = __shfl_sync(0xffffffffu, prev, sl & 31);
            const uint32_t vc = __shfl_sync(0xffffffffu, cur, sl & 31);
            const uint32_t vn = __shfl_sync(0xffffffffu, next, sl & 31);
            const uint32_t rj = sl < 0 ? vp : (sl >= 32 ? vn : vc);
            const int j = i + d;
            // invert: snapkv-lite's (max + 1e-6 - norm); otherwise the rows carry caller-supplied scores
            if (j >= 0 && j < R) acc += invert ? round_dt<DT>(mxe - Tr::from_raw(rj)) : Tr::from_raw(rj);
        }
        if (i < R) {
            const float outv = pooling ? round_dt<DT>(acc / den) : acc;
            const Key key = ordered_key<Key>(Tr::to_raw(outv), /*descending=*/true);
            keys[i] = key;
            atomicAdd(&hist[(uint32_t)key >> kShift0], 1u);
        }
        prev = cur;
        cur = next;
    }
    __syncthreads();
}

}  // namespace kvc
