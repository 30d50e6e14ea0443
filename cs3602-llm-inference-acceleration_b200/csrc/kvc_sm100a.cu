// kvc_sm100a.cu — kernels + C ABI (include/kvc.h) of the B200 KV-cache compression path.
//
// One launch compresses every layer of a call: grid = (B*H, n_layers); one CTA owns one
// (layer, batch, head) unit and runs
//   scan   (K1) stream the K rows of the selection region once, fp32 sum of squares, round the
//               norm to the cache dtype (torch.norm semantics), build the radix key in shared
//               memory and its 11-bit histogram on the fly;
//   select (K2) radix select over the on-chip keys, ties -> lowest index, ascending indices;
//   gather (K3) copy sink rows + selected rows + tail rows of K and V into the dense output.
// Several CTAs are resident per SM, so one unit's select overlaps its neighbours' HBM phases.
// Algorithmic HBM bytes per unit: e*D*(R + 4*C)  (SURVEY.md §8d).
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <type_traits>
#include <utility>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: a no-op call unless a profiler injected itself

#include "kvc_device.cuh"
#include "kvc_fused_tma.cuh"
#include "kvc_h2o.cuh"
#include "kvc_h2o_tc.cuh"
#include "kvc_slab.cuh"
#include "kvc_vote.cuh"

// The library is ONE source file, but its kernel instantiations compile serially: the build compiles it several
// times in parallel, each pass keeping one group of entry points (and only the kernels they launch), and links the
// objects.  KVC_PART is a bit mask: 1 = compress / select / norms entry points (+ the library-wide state) and the
// bf16 fused kernels, 2 = slab entry points and the bf16 in-place kernels, 4 = vote, 8 = slab append kernels,
// 16 = f16/f32 fused kernels, 32 = f16/f32 in-place kernels, 64 = H2O score accumulation (CUDA-core and tensor-core
// forms).
#ifndef KVC_PART
#define KVC_PART 127
#endif
#define KVC_HAS_CORE (KVC_PART & 1)
#define KVC_HAS_SLAB (KVC_PART & 2)
#define KVC_HAS_VOTE (KVC_PART & 4)
#define KVC_HAS_APPEND (KVC_PART & 8)
#define KVC_HAS_FUSED_OTHER (KVC_PART & 16)
#define KVC_HAS_SLAB_OTHER (KVC_PART & 32)
#define KVC_HAS_H2O (KVC_PART & 64)

#define KVC_STR2(x) #x
#define KVC_STR(x) KVC_STR2(x)

namespace kvc {

constexpr int kSmemFixed = kHistBins * 4 + kMiscInts * 4;

// ------------------------------------------------------------------ standalone K1
// One warp step = 32/lpr rows; grid-stride over row groups of one [B,H,R] problem.
template <int DT>
__global__ void __launch_bounds__(256) kvc_norm_kernel(const char* __restrict__ k_in, int64_t sb, int64_t sh,
                                                       int64_t ss, int H, int row_lo, int R, int64_t total_rows,
                                                       int lpr, int cpl, typename Traits<DT>::Key* __restrict__ out) {
    using Tr = Traits<DT>;
    const int lane = threadIdx.x & 31;
    const int rpw = 32 / lpr;
    const int sub = lane % lpr, rw = lane / lpr;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t g = warp_global * rpw; g < total_rows; g += n_warps * rpw) {
        const int64_t idx = g + rw;  // flat (bh, r)
        const bool ok = rw < rpw && idx < total_rows;
        float acc = 0.f;
        if (ok) {
            const int64_t bh = idx / R;
            const int r = (int)(idx - bh * R);
            const int64_t b = bh / H, h = bh - b * H;
            const char* p = k_in + b * sb + h * sh + (int64_t)(row_lo + r) * ss + (int64_t)sub * 16;
            for (int c = 0; c < cpl; ++c) acc = Tr::sumsq(ldg128_stream(p + (int64_t)c * lpr * 16), acc);
        }
        acc = group_sum_pow2(acc, lpr);
        if (ok && sub == 0) out[idx] = (typename Tr::Key)Tr::to_raw(sqrtf(acc));
    }
}

// ------------------------------------------------------------------ standalone K2
// One CTA per score row: load scores -> ordered keys + histogram in shared memory -> select.
template <int DT, int NT>
__global__ void __launch_bounds__(NT) kvc_select_kernel(const typename Traits<DT>::Key* __restrict__ scores, int n,
                                                        int k, int largest, int32_t* __restrict__ idx_out) {
    using Tr = Traits<DT>;
    using Key = typename Tr::Key;
    constexpr int kShift0 = Tr::kKeyBits - kHistBits;
    extern __shared__ __align__(128) unsigned char smem[];
    uint32_t* hist = reinterpret_cast<uint32_t*>(smem);
    int32_t* misc = reinterpret_cast<int32_t*>(smem + kHistBins * 4);
    int32_t* sidx = reinterpret_cast<int32_t*>(smem + kSmemFixed);
    Key* keys = reinterpret_cast<Key*>(smem + kSmemFixed + (size_t)((k + 3) & ~3) * 4);
    const int tid = threadIdx.x;
    const Key* src = scores + (int64_t)blockIdx.x * n;
    for (int i = tid; i < kHistBins; i += NT) hist[i] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += NT) {
        const Key key = ordered_key<Key>((uint32_t)src[i], largest != 0);
        keys[i] = key;
        atomicAdd(&hist[(uint32_t)key >> kShift0], 1u);
    }
    __syncthreads();
    block_radix_select<Key, NT>(keys, n, k, hist, misc, sidx, 0);
    int32_t* dst = idx_out + (int64_t)blockIdx.x * k;
    for (int i = tid; i < k; i += NT) dst[i] = sidx[i];
}

// ------------------------------------------------------------------ host side
#if KVC_HAS_CORE
thread_local char g_last_error[256] = "";
std::atomic<int64_t> g_launches{0};
#else
extern thread_local char g_last_error[256];
extern std::atomic<int64_t> g_launches;
#endif
constexpr int kMaxSmemOptin = 227 * 1024;

static int cuda_fail(cudaError_t e, const char* what) {
    snprintf(g_last_error, sizeof(g_last_error), "%s: %s", what, cudaGetErrorString(e));
    return KVC_ERR_CUDA;
}

// After a kernel launch: a launch error becomes KVC_ERR_CUDA with `what` in kvc_last_cuda_error, a launch is counted.
static int launched(const char* what) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, what);
    g_launches.fetch_add(1);
    return KVC_OK;
}

// Calls f(l0, nl) for the layers [l0, l0 + nl) of each launch (at most KVC_MAX_LAYERS_PER_LAUNCH layers); the first
// status other than KVC_OK ends the walk and is returned.
template <class F>
static int for_each_chunk(int n_layers, F&& f) {
    for (int l0 = 0; l0 < n_layers; l0 += KVC_MAX_LAYERS_PER_LAUNCH) {
        const int st = f(l0, std::min(n_layers - l0, KVC_MAX_LAYERS_PER_LAUNCH));
        if (st != KVC_OK) return st;
    }
    return KVC_OK;
}

// Kernel tables: f(std::integral_constant<int, X>{}) for the run-time value, so that f can name the instantiation.
// Rows of 16 B .. 2 KB: 128/160/192/256/320/512-byte rows (cpr 8/10/12/16/20/32) have kernels with compile-time widths,
// the rest run the generic-width (0) instantiation of the same kernels.
template <class F>
static auto by_cpr(int cpr, F&& f) {
    switch (cpr) {
        case 8: return f(std::integral_constant<int, 8>{});
        case 10: return f(std::integral_constant<int, 10>{});
        case 12: return f(std::integral_constant<int, 12>{});
        case 16: return f(std::integral_constant<int, 16>{});
        case 20: return f(std::integral_constant<int, 20>{});
        case 32: return f(std::integral_constant<int, 32>{});
        default: return f(std::integral_constant<int, 0>{});
    }
}
template <class F>
static auto by_dtype(int dtype, F&& f) {
    switch (dtype) {
        case KVC_DTYPE_F32: return f(std::integral_constant<int, KVC_DTYPE_F32>{});
        case KVC_DTYPE_F16: return f(std::integral_constant<int, KVC_DTYPE_F16>{});
        default: return f(std::integral_constant<int, KVC_DTYPE_BF16>{});
    }
}
static bool row_width_ok(int cpr) { return cpr >= 1 && cpr <= 128; }

static int elem_bytes(int dtype) { return dtype == KVC_DTYPE_F32 ? 4 : 2; }
static int key_bytes(int dtype) { return dtype == KVC_DTYPE_F32 ? 4 : 2; }

using FusedFn = void (*)(const BatchDev);
constexpr int kNT = 512;  // threads of the stand-alone select kernel

// Entry points run on shape->device and leave the calling thread's current device as they found it: torch keeps its
// own idea of the current device, and a library that moved it would send later allocations and stream queries of a
// multi-GPU process (device_map-style placement) to the wrong GPU.
struct DeviceGuard {
    int prev = -1;
    int status = KVC_OK;
    explicit DeviceGuard(int device) {
        cudaError_t e = cudaGetDevice(&prev);
        if (e != cudaSuccess) {
            prev = -1;
            status = cuda_fail(e, "cudaGetDevice");
            return;
        }
        if (prev == device) {
            prev = -1;  // nothing to restore
            return;
        }
        e = cudaSetDevice(device);
        if (e != cudaSuccess) {
            prev = -1;
            status = cuda_fail(e, "cudaSetDevice");
        }
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// One NVTX range per entry point (SURVEY.md §5: tracing): `ncu --nvtx --nvtx-include "kvc_compress_layers/"` or an
// nsys timeline then attribute every launch to the C-ABI call that made it.  Without a tool attached the push / pop
// are two calls through a null-checked function pointer.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

static int ensure_smem(const void* fn, size_t bytes) {
    // The attribute is sticky per function and context; raising it again is cheap.
    if (bytes > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmemOptin);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(max dynamic smem)");
    }
    return KVC_OK;
}

// Largest power of two dividing cpr, capped at 32 (generic-path lanes per row).
static int pow2_lanes(int cpr) {
    int l = 1;
    while (l < 32 && (cpr % (l * 2)) == 0) l *= 2;
    return l;
}

static size_t fused_smem_bytes(int dtype, int max_region, int idx_cap) {
    const size_t keys = ((size_t)max_region * key_bytes(dtype) + 15) & ~(size_t)15;
    return (size_t)kSmemFixed + (size_t)idx_cap * 4 + keys;
}


// ------------------------------------------------------------------ TMA form: variant + smem plan
constexpr int kSmemPerSM = 228 * 1024;  // per-SM shared memory; every resident CTA reserves 1 KB of it
constexpr int kSMs = 148;               // B200
constexpr int kTmaHead = kMiscInts * 4 + 32 * 8;  // misc scalars + one mbarrier per warp

struct TmaPlan {
    bool ok = false;
    int nt = 0, ctas = 0, nsw = 0, upc = 1;
    int slide_slots = 0;  // in-place plans: slots the slide can use (planned slots + the dead key array)
    int off_hist = 0, off_idx = 0, off_keys = 0, off_stage = 0;
    size_t smem = 0;
};

// Launch-shape overrides and stage isolation exist only in a lab build (-DKVC_LAB: scripts/build_lab.sh); the product
// library reads no environment variable, so nothing outside the call's arguments can change what it computes.
#ifdef KVC_LAB
static int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}
// KVC_VOTE_DEBUG switches stages of the vote kernel off for stage-isolation timing (1 = no math, 2 = no math, no
// MMA, 3 = no tail box, 4 = one K step): the votes it produces are NOT valid.
static int vote_debug_mode() { return env_int("KVC_VOTE_DEBUG", 0); }
#else
static inline int env_int(const char*, int dflt) { return dflt; }
static inline int vote_debug_mode() { return 0; }
#endif

// Choose threads per CTA, resident CTAs per SM and staging warps so that (a) the on-chip key
// buffer fits, (b) as close to 128 KB of rows as possible are in flight per SM, (c) as many CTAs as possible are
// resident so one unit's select phase hides under its neighbours' HBM phases.
// `units` / `unit_bytes` (optional): CTAs of the launch and the bytes one of them moves.  A launch of a few large
// units (c1: 960 units of 2.75 MB on 148 SMs) ends in a partial wave whose CTAs each run alone on their SM; with 3
// resident CTAs per SM that wave is a third of the whole launch, with one 512-thread CTA per SM a seventh
// (measured: 446 -> 402 us, 0.90 -> 1.00 of the copy peak, profiles/r02_plan_sweep_few_units.json).  Small units
// (decode steady state) and launches of many waves keep the residency-first choice.
// `in_place` (kvc_slab_compress with the keys on chip): the kept-index list is only written by the select's last pass,
// after the histogram's last reader, so it ALIASES the histogram (k_sel <= 2048); and the slide runs after the select,
// when the key array is dead and serves as staging, so the plan may hold NO slot of its own.  At 32K bf16 rows that is
// 72.7 KB instead of 84.6 KB per CTA: three resident CTAs per SM instead of two (one unit's select and slide rounds
// hide under its neighbours').
static TmaPlan plan_tma(int dtype, int cpr, int max_region, int idx_cap, bool any_select, bool light_traffic = false,
                        int64_t units = 0, int64_t unit_bytes = 0, bool in_place = false) {
    TmaPlan best;
    const int stage = 32 * cpr * 16;
    int end = kTmaHead;
    TmaPlan base;
    base.off_hist = base.off_idx = base.off_keys = kTmaHead;
    if (any_select) {
        base.off_hist = kTmaHead;
        base.off_idx = base.off_hist + kHistBins * 4;
        base.off_keys = base.off_idx + ((idx_cap * 4 + 15) & ~15);
        if (in_place && idx_cap <= kHistBins) {
            base.off_idx = base.off_hist;
            base.off_keys = base.off_hist + kHistBins * 4;
        }
        end = base.off_keys + (int)(((size_t)max_region * key_bytes(dtype) + 15) & ~(size_t)15);
    }
    base.off_stage = (end + 127) & ~127;
    const int dead_keys = in_place ? base.off_stage - ((base.off_keys + 127) & ~127) : 0;  // bytes the slide inherits
    const int force_nt = env_int("KVC_TMA_NT", 0), force_ctas = env_int("KVC_TMA_CTAS", 0),
              force_nsw = env_int("KVC_TMA_NSW", 0);
    static const int cand[][2] = {{256, 3}, {256, 2}, {512, 1}, {256, 1}};
    // a launch of a few large units: fewer than 8 waves at the highest residency that fits (then EVERY candidate is
    // ranked by estimated launch length, below)
    bool few_large_units = false;
    if (!light_traffic && units > 0 && unit_bytes >= (1 << 20) && !force_nt && !force_ctas) {
        for (const auto& c : cand) {
            int limit = kSmemPerSM / c[1] - 1024;
            if (limit > kMaxSmemOptin) limit = kMaxSmemOptin;
            if (limit - base.off_stage >= stage) {
                few_large_units = units / ((int64_t)c[1] * kSMs) < 8;
                break;  // candidates are listed by falling residency
            }
        }
    }
    long best_score = -1;
    for (const auto& c : cand) {
        const int nt = c[0], ctas = c[1];
        if (force_nt && nt != force_nt) continue;
        if (force_ctas && ctas != force_ctas) continue;
        int limit = kSmemPerSM / ctas - 1024;
        if (limit > kMaxSmemOptin) limit = kMaxSmemOptin;
        const int avail = limit - base.off_stage;
        if (avail < (in_place ? 0 : stage)) continue;
        int nsw = avail / stage;
        if (nsw > nt / 32) nsw = nt / 32;
        int slide = (dead_keys + nsw * stage) / stage;  // what the slab kernel computes for its rounds
        if (slide > nt / 32) slide = nt / 32;
        if (in_place && slide < 1) continue;
        if (force_nsw && force_nsw < nsw) nsw = force_nsw;
        const long inflight = (long)ctas * nsw * stage;
        // saturating score: bytes in flight up to 128 KB matter most (measured: c5 +8% from 64 -> 128 KB), then residency
        long score = (inflight < 131072 ? inflight : 131072) * 8 + ctas * 4096 + (inflight >> 6);
        // in-place compaction moves few bytes (scores come from stored norms): residency first, 2+ slots are enough
        if (light_traffic) score = ((in_place ? slide : nsw) >= 2 ? 1 : 0) * (1L << 30) + ctas * (1L << 20) + (in_place ? slide : nsw);
        if (few_large_units) {
            // rank by the estimated length of the launch: full waves plus a last partial wave that costs at least
            // ~0.35 of a full one (a lone CTA is latency-bound), over the rate this shape sustains — bytes in flight
            // (64 KB per SM measured 8 % behind 128 KB) and residency (3 CTAs hide a unit's select under its
            // neighbours' HBM phases: ~5 % on many-wave launches)
            const long slots = (long)ctas * kSMs;
            const long full = (long)(units / slots), rem = (long)(units - full * slots);
            const double est = (double)full * slots + (rem > 0 ? std::max((double)rem, 0.35 * slots) : 0.0);
            const double fill = (double)(inflight < 131072 ? inflight : 131072) / 131072.0;
            const double rate = (0.84 + 0.16 * fill) * (ctas >= 3 ? 1.05 : (ctas == 2 ? 1.03 : (nt == 512 ? 1.0 : 0.95)));
            score = (long)(1e12 / (est / rate + 1.0));
        }
        if (score > best_score) {
            best_score = score;
            best = base;
            best.ok = true;
            best.nt = nt;
            best.ctas = ctas;
            best.nsw = nsw;
            best.slide_slots = in_place ? slide : nsw;
            best.smem = (size_t)base.off_stage + (size_t)nsw * stage;
        }
    }
    best.upc = env_int("KVC_TMA_UPC", 1);
    if (best.upc < 1) best.upc = 1;
    return best;
}

// Keys + kept indices of one (layer, batch, head) unit when they live in the device workspace.
struct WsLayout {
    int64_t keys = 0, unit = 0;
};
static WsLayout ws_layout(int dtype, int max_region, int idx_cap) {
    WsLayout w;
    w.keys = ((int64_t)max_region * key_bytes(dtype) + 15) & ~(int64_t)15;
    w.unit = w.keys + (((int64_t)idx_cap * 4 + 15) & ~(int64_t)15);
    return w;
}
// The on-chip plan is good enough when it exists and keeps >= 48 KB of rows in flight per SM (scan kernels)
// or has at least two slots (in-place compaction, whose traffic is light).
static bool onchip_plan_ok(const TmaPlan& tp, int cpr, bool light_traffic) {
    if (!tp.ok) return false;
    if (light_traffic) return tp.slide_slots >= 2;
    return (long)tp.ctas * tp.nsw * 32 * cpr * 16 >= 48 * 1024;
}

#if KVC_HAS_CORE || KVC_HAS_FUSED_OTHER
template <int DT>
static FusedFn pick_tma_nt(int cpr, int nt) {
    return by_cpr(cpr, [&](auto c) {
        return nt == 512 ? FusedFn(kvc_fused_tma_kernel<DT, c, 512, 1>) : FusedFn(kvc_fused_tma_kernel<DT, c, 256, 3>);
    });
}
#endif
FusedFn pick_tma_bf16(int cpr, int nt);
FusedFn pick_tma_other(int dtype, int cpr, int nt);
#if KVC_HAS_CORE
FusedFn pick_tma_bf16(int cpr, int nt) { return pick_tma_nt<KVC_DTYPE_BF16>(cpr, nt); }
static FusedFn pick_tma(int dtype, int cpr, int nt) {
    return dtype == KVC_DTYPE_BF16 ? pick_tma_bf16(cpr, nt) : pick_tma_other(dtype, cpr, nt);
}
#endif
#if KVC_HAS_FUSED_OTHER
FusedFn pick_tma_other(int dtype, int cpr, int nt) {
    return dtype == KVC_DTYPE_F32 ? pick_tma_nt<KVC_DTYPE_F32>(cpr, nt) : pick_tma_nt<KVC_DTYPE_F16>(cpr, nt);
}
#endif

static int ensure_tma_attrs(const void* fn, int device) {
    // Function attributes are sticky per (function, device): set them once, not on every decode step.
    static std::mutex mu;
    static std::vector<std::pair<const void*, int>> done;
    {
        std::lock_guard<std::mutex> lock(mu);
        for (const auto& d : done)
            if (d.first == fn && d.second == device) return KVC_OK;
    }
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmemOptin);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(max dynamic smem)");
    e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(carveout)");
    std::lock_guard<std::mutex> lock(mu);
    done.emplace_back(fn, device);
    return KVC_OK;
}


// ------------------------------------------------------------------ slab kernels: variant tables
using SlabFn = void (*)(const SlabBatchDev);
using AppendFn = void (*)(const AppendBatchDev);
using AppendOneFn = void (*)(const AppendOneDev);
SlabFn pick_slab_bf16(int cpr, int nt);
SlabFn pick_slab_other(int dtype, int cpr, int nt);
AppendFn pick_append(int dtype, int cpr);          // thread-per-row form, all layers
AppendOneFn pick_append_one(int dtype, int cpr);   // thread-per-row form, one layer (small parameter block)
AppendFn pick_append_tma(int dtype, int cpr);      // bulk-copy form (prefill-sized appends)

#if KVC_HAS_SLAB || KVC_HAS_SLAB_OTHER
template <int DT>
static SlabFn pick_slab_nt(int cpr, int nt) {
    return by_cpr(cpr, [&](auto c) {
        return nt == 512 ? SlabFn(kvc_slab_compress_kernel<DT, c, 512, 1>) : SlabFn(kvc_slab_compress_kernel<DT, c, 256, 3>);
    });
}
#endif
#if KVC_HAS_SLAB
SlabFn pick_slab_bf16(int cpr, int nt) { return pick_slab_nt<KVC_DTYPE_BF16>(cpr, nt); }
static SlabFn pick_slab(int dtype, int cpr, int nt) {
    return dtype == KVC_DTYPE_BF16 ? pick_slab_bf16(cpr, nt) : pick_slab_other(dtype, cpr, nt);
}
#endif
#if KVC_HAS_SLAB_OTHER
SlabFn pick_slab_other(int dtype, int cpr, int nt) {
    return dtype == KVC_DTYPE_F32 ? pick_slab_nt<KVC_DTYPE_F32>(cpr, nt) : pick_slab_nt<KVC_DTYPE_F16>(cpr, nt);
}
#endif

#if KVC_HAS_APPEND
AppendOneFn pick_append_one(int dtype, int cpr) {
    return by_dtype(dtype, [&](auto dt) {
        return by_cpr(cpr, [&](auto c) { return AppendOneFn(kvc_slab_append_kernel<dt, c, AppendOneDev>); });
    });
}
AppendFn pick_append(int dtype, int cpr) {
    return by_dtype(dtype, [&](auto dt) {
        return by_cpr(cpr, [&](auto c) { return AppendFn(kvc_slab_append_kernel<dt, c, AppendBatchDev>); });
    });
}
AppendFn pick_append_tma(int dtype, int cpr) {
    return by_dtype(dtype, [&](auto dt) {
        return by_cpr(cpr, [&](auto c) { return AppendFn(kvc_slab_append_tma_kernel<dt, c>); });
    });
}
#endif  // KVC_HAS_APPEND

static int check_shape(const kvc_shape* shape, int* cpr_out) {
    if (!shape) return KVC_ERR_INVALID_ARG;
    const int B = shape->batch, H = shape->heads, D = shape->head_dim, dt = shape->dtype;
    if (B <= 0 || H <= 0 || D <= 0) return KVC_ERR_INVALID_ARG;
    if (dt != KVC_DTYPE_F32 && dt != KVC_DTYPE_F16 && dt != KVC_DTYPE_BF16) return KVC_ERR_UNSUPPORTED;
    const int e = elem_bytes(dt);
    if (((int64_t)D * e) % 16 != 0) return KVC_ERR_UNSUPPORTED;
    if ((int64_t)B * H > 0x7fffffffLL) return KVC_ERR_INVALID_ARG;
    *cpr_out = D * e / 16;
    return KVC_OK;
}

// A valid in-place compaction (the slab rule: C <= S, the selection region between the sinks and the tail), which makes
// every kept source row lie at or above its output row.
static inline bool in_place_ok(const kvc_layer_plan& p) {
    if ((int64_t)p.sink + p.k_sel + p.tail > p.seq_len) return false;
    return p.k_sel <= 0 || (p.sel_lo >= p.sink && p.sel_hi <= p.seq_len - p.tail);
}

// The plan checks of one layer, for both compaction forms, before anything is enqueued: KVC_OK or the status of the
// first failing check.  in_place: the kept rows are compacted within the layer's own rows.  has_idx / has_score: the
// caller supplied the rows a GIVEN_INDEX plan keeps / the scores a GIVEN_SCORE(_SHARED) plan ranks.  carry: the layer's
// kvc_carry_layer or nullptr; its copy runs in place, so a non-NULL acc needs a valid in-place compaction as well.
static int check_plan(const kvc_layer_plan& p, bool in_place, bool has_idx, bool has_score, const kvc_carry_layer* carry,
                      int e) {
    if (p.seq_len < 0 || p.sink < 0 || p.k_sel < 0 || p.tail < 0) return KVC_ERR_INVALID_ARG;
    if (p.sink > p.seq_len || p.tail > p.seq_len) return KVC_ERR_INVALID_ARG;
    if (in_place && !in_place_ok(p)) return KVC_ERR_INVALID_ARG;
    if (p.k_sel > 0) {
        if (p.sel_lo < 0 || p.sel_hi > p.seq_len || p.sel_lo > p.sel_hi) return KVC_ERR_INVALID_ARG;
        if (p.k_sel > p.sel_hi - p.sel_lo) return KVC_ERR_INVALID_ARG;
        if (p.score <= KVC_SCORE_NONE || p.score > KVC_SCORE_GIVEN_SCORE_SHARED) return KVC_ERR_INVALID_ARG;
        const bool given_score = p.score == KVC_SCORE_GIVEN_SCORE || p.score == KVC_SCORE_GIVEN_SCORE_SHARED;
        if (p.score == KVC_SCORE_GIVEN_INDEX && !has_idx) return KVC_ERR_INVALID_ARG;
        if (given_score && !has_score) return KVC_ERR_INVALID_ARG;
        if ((given_score || p.score == KVC_SCORE_SNAPKV_POOL) && p.pool_kernel > 2 * kMaxPoolHalo)
            return KVC_ERR_UNSUPPORTED;
    }
    if (carry && carry->acc) {
        if (carry->group < 1 || carry->prev_len < 0 || ((uintptr_t)carry->acc % (uintptr_t)e) != 0)
            return KVC_ERR_INVALID_ARG;
        if (!in_place_ok(p)) return KVC_ERR_INVALID_ARG;
    }
    return KVC_OK;
}

// The layer ranks its region by key norms (scanned from K, or stored ones the caller holds).
static inline bool ranked(const kvc_layer_plan& p) {
    return p.k_sel > 0 &&
           (p.score == KVC_SCORE_L2_LOW || p.score == KVC_SCORE_L2_HIGH || p.score == KVC_SCORE_SNAPKV_POOL);
}

// What one launch (layers [0, nl) of `plans`) has to plan for.  any_scan is only known with the io records: a ranked
// layer whose caller holds no key norms reads its region of K.
struct ChunkStats {
    int n_active = 0;      // layers with C > 0
    int max_region = 0;    // largest selection region whose radix keys are built (not GIVEN_INDEX)
    int idx_cap = 0;       // kept-index entries reserved per unit (largest k_sel, rounded up to 4)
    bool any_select = false, any_scan = false;
    int64_t rows_moved = 0;  // rows the units move if they scan K: the region once + kept rows of K and V read and written
};
static ChunkStats chunk_stats(const kvc_layer_plan* plans, const kvc_layer_io* io, int nl) {
    ChunkStats s;
    int max_ksel = 0;
    for (int l = 0; l < nl; ++l) {
        const kvc_layer_plan& p = plans[l];
        if (p.sink + p.k_sel + p.tail == 0) continue;
        ++s.n_active;
        s.rows_moved += (p.k_sel > 0 ? p.sel_hi - p.sel_lo : 0) + 4LL * (p.sink + p.k_sel + p.tail);
        if (p.k_sel > 0) {
            s.any_select = true;
            s.any_scan |= io != nullptr && ranked(p) && !io[l].norms_in;
            if (p.k_sel > max_ksel) max_ksel = p.k_sel;
            if (p.score != KVC_SCORE_GIVEN_INDEX && p.sel_hi - p.sel_lo > s.max_region) s.max_region = p.sel_hi - p.sel_lo;
        }
    }
    s.idx_cap = (max_ksel + 3) & ~3;
    return s;
}

// The launch plan of one launch.  When the on-chip plan is not good enough (onchip_plan_ok) and a workspace may be
// used, the radix keys and kept indices go to the workspace (layout w) and shared memory keeps the histogram and slots.
struct LaunchPlan {
    TmaPlan tp;
    bool ws = false;
    WsLayout w;
};
static LaunchPlan plan_launch(int dtype, int cpr, const ChunkStats& s, bool light_traffic, bool in_place, int64_t units,
                              int64_t unit_bytes, bool may_use_ws) {
    LaunchPlan lp;
    lp.tp = plan_tma(dtype, cpr, s.max_region, s.idx_cap, s.any_select, light_traffic, units, unit_bytes, in_place);
    lp.ws = s.any_select && may_use_ws && !onchip_plan_ok(lp.tp, cpr, light_traffic);
    if (lp.ws) {
        lp.w = ws_layout(dtype, s.max_region, s.idx_cap);
        lp.tp = plan_tma(dtype, cpr, 0, 0, true, light_traffic);
    }
    return lp;
}

// Zeroes the launch descriptor and fills the fields BatchDev and SlabBatchDev share from the launch plan: shape,
// kept-index capacity, workspace, shared-memory layout.  KVC_ERR_INVALID_ARG when the plan needs more workspace than the
// caller gave, KVC_ERR_TOO_LARGE when no plan fits.
template <class Batch>
static int fill_batch(Batch& bd, const kvc_shape* shape, int cpr, const ChunkStats& s, const LaunchPlan& lp,
                      void* workspace, int64_t workspace_bytes) {
    if (lp.ws && lp.w.unit * shape->batch * shape->heads * s.n_active > workspace_bytes) return KVC_ERR_INVALID_ARG;
    if (!lp.tp.ok) return KVC_ERR_TOO_LARGE;
    memset(&bd, 0, sizeof(bd));
    bd.B = shape->batch;
    bd.H = shape->heads;
    bd.cpr = cpr;
    bd.idx_cap = s.idx_cap;
    if (lp.ws) {
        bd.ws = (char*)workspace;
        bd.ws_unit = lp.w.unit;
        bd.ws_keys = lp.w.keys;
    }
    bd.nsw = lp.tp.nsw;
    bd.off_hist = lp.tp.off_hist;
    bd.off_idx = lp.tp.off_idx;
    bd.off_keys = lp.tp.off_keys;
    bd.off_stage = lp.tp.off_stage;
    return KVC_OK;
}

// The fields LayerDev and SlabLayerDev share: the plan and the carry (the descriptor was zeroed: no carry, acc == nullptr).
template <class Layer>
static void fill_layer_plan(Layer& d, const kvc_layer_plan& p, const kvc_carry_layer* carry, int e) {
    d.S = p.seq_len;
    d.sink = p.sink;
    d.lo = p.sel_lo;
    d.hi = p.sel_hi;
    d.ksel = p.k_sel;
    d.tail = p.tail;
    d.score = p.k_sel > 0 ? p.score : KVC_SCORE_NONE;
    d.pool = p.pool_kernel;
    if (!carry || !carry->acc) return;
    d.carry.acc = (char*)carry->acc;
    d.carry.asb = carry->acc_stride_b * e;
    d.carry.ash = carry->acc_stride_h * e;
    d.carry.group = carry->group;
    d.carry.prev = carry->prev_len < p.seq_len ? carry->prev_len : p.seq_len;
}

}  // namespace kvc

using namespace kvc;

extern "C" {

#if KVC_HAS_CORE
int kvc_abi_version(void) { return KVC_ABI_VERSION; }

const char* kvc_build_info(void) {
    return "libkvc_sm100a: sm_100a, nvcc " KVC_STR(__CUDACC_VER_MAJOR__) "." KVC_STR(__CUDACC_VER_MINOR__);
}

const char* kvc_status_string(int status) {
    switch (status) {
        case KVC_OK: return "ok";
        case KVC_ERR_INVALID_ARG: return "invalid argument";
        case KVC_ERR_UNSUPPORTED: return "unsupported dtype / head_dim / alignment";
        case KVC_ERR_TOO_LARGE: return "selection region too large for the on-chip score buffer";
        case KVC_ERR_CUDA: return "CUDA error";
        default: return "unknown status";
    }
}

const char* kvc_last_cuda_error(void) { return g_last_error; }

int64_t kvc_launch_count(void) { return g_launches.load(); }

int32_t kvc_max_region_rows(int32_t dtype, int32_t k_sel) {
    if (dtype < 0 || dtype > 2 || k_sel < 0) return 0;
    const int64_t idx = ((int64_t)k_sel + 3) & ~(int64_t)3;
    const int64_t left = (int64_t)kMaxSmemOptin - kSmemFixed - idx * 4;
    if (left <= 0) return 0;
    const int64_t rows = (left & ~(int64_t)15) / key_bytes(dtype);
    return (int32_t)(rows > 0x7fffffff ? 0x7fffffff : rows);
}

int kvc_compress_layers(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                        const kvc_layer_io* io, void* stream) {
    return kvc_compress_layers_ws(shape, n_layers, plans, io, nullptr, 0, stream);
}

// Both planning queries plan like a launch that scans K (light_traffic = false): KVSlabCache sizes the workspace of its
// in-place compaction with kvc_workspace_bytes as well.
int64_t kvc_workspace_bytes(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans) {
    int cpr = 0;
    if (check_shape(shape, &cpr) != KVC_OK || n_layers <= 0 || !plans || !row_width_ok(cpr)) return 0;
    const int64_t bh = (int64_t)shape->batch * shape->heads;
    int64_t need = 0;
    for_each_chunk(n_layers, [&](int l0, int nl) -> int {
        const ChunkStats s = chunk_stats(plans + l0, nullptr, nl);
        if (!s.any_select) return KVC_OK;
        const LaunchPlan lp = plan_launch(shape->dtype, cpr, s, false, false, bh * s.n_active,
                                          s.rows_moved / s.n_active * cpr * 16, true);
        if (lp.ws) need = std::max(need, lp.w.unit * bh * s.n_active);
        return KVC_OK;
    });
    return need;
}

int kvc_launch_shape(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans, int32_t out[4]) {
    int cpr = 0;
    int st = check_shape(shape, &cpr);
    if (st != KVC_OK) return st;
    if (n_layers <= 0 || !plans || !out) return KVC_ERR_INVALID_ARG;
    if (!row_width_ok(cpr)) return KVC_ERR_UNSUPPORTED;
    const ChunkStats s = chunk_stats(plans, nullptr, std::min(n_layers, KVC_MAX_LAYERS_PER_LAUNCH));
    if (s.n_active == 0) return KVC_ERR_INVALID_ARG;
    const int64_t units = (int64_t)shape->batch * shape->heads * s.n_active;
    const LaunchPlan lp = plan_launch(shape->dtype, cpr, s, false, false, units, s.rows_moved / s.n_active * cpr * 16, true);
    if (!lp.tp.ok) return KVC_ERR_TOO_LARGE;
    out[0] = lp.tp.nt;
    out[1] = lp.tp.ctas;
    out[2] = lp.tp.nsw;
    out[3] = lp.ws ? 1 : 0;
    return KVC_OK;
}

int kvc_compress_layers_ws(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                           const kvc_layer_io* io, void* workspace, int64_t workspace_bytes, void* stream) {
    return kvc_compress_layers_carry(shape, n_layers, plans, io, nullptr, workspace, workspace_bytes, stream);
}

int kvc_compress_layers_carry(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                              const kvc_layer_io* io, const kvc_carry_layer* carry, void* workspace,
                              int64_t workspace_bytes, void* stream) {
    if (!shape || n_layers < 0 || (n_layers > 0 && (!plans || !io))) return KVC_ERR_INVALID_ARG;
    if (n_layers == 0) return KVC_OK;
    int cpr = 0;
    int st = check_shape(shape, &cpr);
    if (st != KVC_OK) return st;
    if (!row_width_ok(cpr)) return KVC_ERR_UNSUPPORTED;
    const int B = shape->batch, H = shape->heads, dt = shape->dtype;
    const int e = elem_bytes(dt);

    // validate every layer before anything is enqueued
    for (int l = 0; l < n_layers; ++l) {
        const kvc_layer_plan& p = plans[l];
        const kvc_layer_io& x = io[l];
        st = check_plan(p, false, x.idx_in != nullptr, x.score_in != nullptr, carry ? carry + l : nullptr, e);
        if (st != KVC_OK) return st;
        const int64_t C = (int64_t)p.sink + p.k_sel + p.tail;
        if (C == 0) continue;
        if (!x.k_in || !x.v_in || !x.k_out || !x.v_out) return KVC_ERR_INVALID_ARG;
        if (C * cpr * 2 > 0x7fffffffLL) return KVC_ERR_TOO_LARGE;
        const uintptr_t a = (uintptr_t)x.k_in | (uintptr_t)x.v_in | (uintptr_t)x.k_out | (uintptr_t)x.v_out;
        if (a & 15) return KVC_ERR_UNSUPPORTED;
        const int64_t s = (x.k_stride_b | x.k_stride_h | x.k_stride_s | x.v_stride_b | x.v_stride_h | x.v_stride_s);
        if ((s * e) & 15) return KVC_ERR_UNSUPPORTED;
    }
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_compress_layers_ws");
    if (guard.status != KVC_OK) return guard.status;

    return for_each_chunk(n_layers, [&](int l0, int nl) -> int {
        const ChunkStats s = chunk_stats(plans + l0, io + l0, nl);
        if (s.n_active == 0) return KVC_OK;
        // no K scan in this launch (stored norms, caller-supplied scores or rows, pure slices with a select next to
        // them): only kept rows move -> residency over slot depth
        const bool light = s.any_select && !s.any_scan;
        const LaunchPlan lp = plan_launch(dt, cpr, s, light, false, (int64_t)B * H * s.n_active,
                                          s.rows_moved / s.n_active * cpr * 16, workspace != nullptr);
        BatchDev bd;
        int st = fill_batch(bd, shape, cpr, s, lp, workspace, workspace_bytes);
        if (st != KVC_OK) return st;
        bd.upc = lp.tp.upc;
        int m = 0;
        for (int l = l0; l < l0 + nl; ++l) {
            const kvc_layer_plan& p = plans[l];
            const kvc_layer_io& x = io[l];
            if (p.sink + p.k_sel + p.tail == 0) continue;
            LayerDev& d = bd.layers[m++];
            d.k_in = (const char*)x.k_in;
            d.v_in = (const char*)x.v_in;
            d.k_out = (char*)x.k_out;
            d.v_out = (char*)x.v_out;
            d.idx_out = x.idx_out;
            d.idx_in = (p.score == KVC_SCORE_GIVEN_SCORE || p.score == KVC_SCORE_GIVEN_SCORE_SHARED) ? (const int32_t*)x.score_in
                                                                                              : x.idx_in;
            d.ksb = x.k_stride_b * e;
            d.ksh = x.k_stride_h * e;
            d.kss = x.k_stride_s * e;
            d.vsb = x.v_stride_b * e;
            d.vsh = x.v_stride_h * e;
            d.vss = x.v_stride_s * e;
            if (ranked(p) && x.norms_in) {  // the caller holds the key norms: the scan is skipped
                d.n_in = (const char*)x.norms_in;
                d.nsb = x.n_stride_b * key_bytes(dt);
                d.nsh = x.n_stride_h * key_bytes(dt);
            }
            fill_layer_plan(d, p, carry ? carry + l : nullptr, e);
        }
        FusedFn fn = pick_tma(dt, cpr, lp.tp.nt);
        dim3 grid((unsigned)(((int64_t)B * H + lp.tp.upc - 1) / lp.tp.upc), (unsigned)s.n_active, 1);
        st = ensure_tma_attrs((const void*)fn, shape->device);
        if (st != KVC_OK) return st;
        fn<<<grid, lp.tp.nt, lp.tp.smem, (cudaStream_t)stream>>>(bd);
        return launched("kvc_fused_tma_kernel launch");
    });
}

int kvc_key_norms(const kvc_shape* shape, const void* k_in, int64_t stride_b, int64_t stride_h, int64_t stride_s,
                  int32_t row_lo, int32_t row_hi, void* norms_out, void* stream) {
    if (!shape || !k_in || !norms_out || row_lo < 0 || row_hi < row_lo) return KVC_ERR_INVALID_ARG;
    const int B = shape->batch, H = shape->heads, D = shape->head_dim, dt = shape->dtype;
    if (B <= 0 || H <= 0 || D <= 0) return KVC_ERR_INVALID_ARG;
    if (dt != KVC_DTYPE_F32 && dt != KVC_DTYPE_F16 && dt != KVC_DTYPE_BF16) return KVC_ERR_UNSUPPORTED;
    const int e = elem_bytes(dt);
    if (((int64_t)D * e) % 16 != 0 || ((uintptr_t)k_in & 15)) return KVC_ERR_UNSUPPORTED;
    if (((stride_b | stride_h | stride_s) * e) & 15) return KVC_ERR_UNSUPPORTED;
    const int R = row_hi - row_lo;
    const int64_t total = (int64_t)B * H * R;
    if (total == 0) return KVC_OK;
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_key_norms");
    if (guard.status != KVC_OK) return guard.status;
    const int cpr = D * e / 16;
    const int lpr = pow2_lanes(cpr), cpl = cpr / lpr;
    const int rpw = 32 / lpr;
    const int64_t warps_needed = (total + rpw - 1) / rpw;
    int64_t blocks = (warps_needed + 7) / 8;
    const int64_t cap = 148LL * 8 * 4;
    if (blocks > cap) blocks = cap;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t sb = stride_b * e, sh = stride_h * e, ss = stride_s * e;
    by_dtype(dt, [&](auto d) {
        kvc_norm_kernel<d><<<(unsigned)blocks, 256, 0, s>>>((const char*)k_in, sb, sh, ss, H, row_lo, R, total, lpr, cpl,
                                                            (typename Traits<d>::Key*)norms_out);
    });
    return launched("kvc_norm_kernel launch");
}

int kvc_select(int32_t dtype, int32_t device, const void* scores, int64_t n_rows, int32_t n, int32_t k,
               int32_t largest, int32_t* idx_out, void* stream) {
    if (!scores || !idx_out || n_rows < 0 || n < 0 || k < 0 || k > n) return KVC_ERR_INVALID_ARG;
    if (dtype != KVC_DTYPE_F32 && dtype != KVC_DTYPE_F16 && dtype != KVC_DTYPE_BF16) return KVC_ERR_UNSUPPORTED;
    if (n_rows == 0 || k == 0) return KVC_OK;
    if (n_rows > 0x7fffffffLL) return KVC_ERR_INVALID_ARG;
    const size_t smem = fused_smem_bytes(dtype, n, (k + 3) & ~3);
    if (smem > (size_t)kMaxSmemOptin) return KVC_ERR_TOO_LARGE;
    DeviceGuard guard(device);
    NvtxRange nvtx_range("kvc_select");
    if (guard.status != KVC_OK) return guard.status;
    return by_dtype(dtype, [&](auto d) -> int {
        const int st = ensure_smem((const void*)kvc_select_kernel<d, kNT>, smem);
        if (st != KVC_OK) return st;
        kvc_select_kernel<d, kNT><<<(unsigned)n_rows, kNT, smem, (cudaStream_t)stream>>>(
            (const typename Traits<d>::Key*)scores, n, k, largest, idx_out);
        return launched("kvc_select_kernel launch");
    });
}

#endif  // KVC_HAS_CORE

#if KVC_HAS_SLAB
int kvc_slab_append(const kvc_shape* shape, int32_t n_layers, const kvc_slab_layer* slabs,
                    const kvc_slab_new_rows* rows, void* stream) {
    int cpr = 0;
    int st = check_shape(shape, &cpr);
    if (st != KVC_OK) return st;
    if (n_layers < 0 || (n_layers > 0 && (!slabs || !rows))) return KVC_ERR_INVALID_ARG;
    if (n_layers == 0) return KVC_OK;
    if (!row_width_ok(cpr)) return KVC_ERR_UNSUPPORTED;
    const int B = shape->batch, H = shape->heads, dt = shape->dtype;
    const int e = elem_bytes(dt);
    for (int l = 0; l < n_layers; ++l) {
        const kvc_slab_layer& sl = slabs[l];
        const kvc_slab_new_rows& r = rows[l];
        if (r.n_new < 0 || r.cur_len < 0) return KVC_ERR_INVALID_ARG;
        if (r.n_new == 0) continue;
        if (!sl.k || !sl.v || !sl.norms || !r.k_new || !r.v_new) return KVC_ERR_INVALID_ARG;
        const uintptr_t a = (uintptr_t)sl.k | (uintptr_t)sl.v | (uintptr_t)r.k_new | (uintptr_t)r.v_new;
        if (a & 15) return KVC_ERR_UNSUPPORTED;
        const int64_t sb = sl.k_stride_b | sl.k_stride_h | sl.v_stride_b | sl.v_stride_h | r.k_stride_b | r.k_stride_h |
                           r.k_stride_s | r.v_stride_b | r.v_stride_h | r.v_stride_s;
        if ((sb * e) & 15) return KVC_ERR_UNSUPPORTED;
        if ((int64_t)B * H * r.n_new > 0x7fffffffLL) return KVC_ERR_TOO_LARGE;
    }
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_slab_append");
    if (guard.status != KVC_OK) return guard.status;
    auto fill = [&](AppendLayerDev& d, const kvc_slab_layer& sl, const kvc_slab_new_rows& r) {
        d.k_new = (const char*)r.k_new;
        d.v_new = (const char*)r.v_new;
        d.k = (char*)sl.k;
        d.v = (char*)sl.v;
        d.n = (char*)sl.norms;
        d.nksb = r.k_stride_b * e;
        d.nksh = r.k_stride_h * e;
        d.nkss = r.k_stride_s * e;
        d.nvsb = r.v_stride_b * e;
        d.nvsh = r.v_stride_h * e;
        d.nvss = r.v_stride_s * e;
        d.ksb = sl.k_stride_b * e;
        d.ksh = sl.k_stride_h * e;
        d.vsb = sl.v_stride_b * e;
        d.vsh = sl.v_stride_h * e;
        d.nsb = sl.n_stride_b * key_bytes(dt);
        d.nsh = sl.n_stride_h * key_bytes(dt);
        d.cur_len = r.cur_len;
        d.n_new = r.n_new;
    };
    if (n_layers == 1 && rows[0].n_new > 0 && rows[0].n_new < 32) {
        // the per-layer update of a decode loop: small parameter block, one small launch
        AppendOneDev one;
        one.B = B;
        one.H = H;
        one.max_new = rows[0].n_new;
        one.cpr = cpr;
        fill(one.layers[0], slabs[0], rows[0]);
        const int64_t threads = (int64_t)B * H * rows[0].n_new;
        pick_append_one(dt, cpr)<<<(unsigned)((threads + 127) / 128), 128, 0, (cudaStream_t)stream>>>(one);
        return launched("kvc_slab_append_kernel launch");
    }
    AppendFn fn = pick_append(dt, cpr);
    return for_each_chunk(n_layers, [&](int l0, int nl) -> int {
        AppendBatchDev bd;
        memset(&bd, 0, sizeof(bd));
        bd.B = B;
        bd.H = H;
        int n_active = 0, max_new = 0;
        for (int l = 0; l < nl; ++l) {
            const kvc_slab_layer& sl = slabs[l0 + l];
            const kvc_slab_new_rows& r = rows[l0 + l];
            if (r.n_new == 0) continue;
            fill(bd.layers[n_active++], sl, r);
            if (r.n_new > max_new) max_new = r.n_new;
        }
        if (n_active == 0) return KVC_OK;
        bd.max_new = max_new;
        bd.cpr = cpr;
        if (max_new >= 32) {
            // prefill / chunked prefill: rows move 32 at a time through shared memory with bulk copies
            AppendFn tfn = pick_append_tma(dt, cpr);
            const int st = ensure_tma_attrs((const void*)tfn, shape->device);
            if (st != KVC_OK) return st;
            const size_t smem = 128 + (size_t)8 * 32 * cpr * 16;
            const int64_t items = (int64_t)B * H * ((max_new + 31) / 32);
            int64_t blocks = (items + 7) / 8;
            const int64_t cap = 148LL * 3 * 8;  // a few waves; warps stride over the remaining blocks
            if (blocks > cap) blocks = cap;
            dim3 grid((unsigned)blocks, (unsigned)n_active, 1);
            tfn<<<grid, 256, smem, (cudaStream_t)stream>>>(bd);
        } else {
            const int64_t threads = (int64_t)B * H * max_new;
            dim3 grid((unsigned)((threads + 127) / 128), (unsigned)n_active, 1);
            fn<<<grid, 128, 0, (cudaStream_t)stream>>>(bd);
        }
        return launched("kvc_slab_append_kernel launch");
    });
}

int kvc_slab_compress(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                      const kvc_slab_layer* slabs, int32_t* const* idx_out, const int32_t* const* idx_in,
                      void* workspace, int64_t workspace_bytes, void* stream) {
    return kvc_slab_compress_carry(shape, n_layers, plans, slabs, idx_out, idx_in, nullptr, workspace, workspace_bytes,
                                   stream);
}

int kvc_slab_compress_carry(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                            const kvc_slab_layer* slabs, int32_t* const* idx_out, const int32_t* const* idx_in,
                            const kvc_carry_layer* carry, void* workspace, int64_t workspace_bytes, void* stream) {
    int cpr = 0;
    int st = check_shape(shape, &cpr);
    if (st != KVC_OK) return st;
    if (n_layers < 0 || (n_layers > 0 && (!slabs || !plans))) return KVC_ERR_INVALID_ARG;
    if (n_layers == 0) return KVC_OK;
    if (!row_width_ok(cpr)) return KVC_ERR_UNSUPPORTED;
    const int B = shape->batch, H = shape->heads, dt = shape->dtype;
    const int e = elem_bytes(dt);
    for (int l = 0; l < n_layers; ++l) {
        const kvc_layer_plan& p = plans[l];
        const kvc_slab_layer& sl = slabs[l];
        const bool given = idx_in && idx_in[l];  // kept rows or scores travel in the idx_in slot
        st = check_plan(p, true, given, given, carry ? carry + l : nullptr, e);
        if (st != KVC_OK) return st;
        if (p.sink + p.k_sel + p.tail == 0) continue;
        if (!sl.k || !sl.v || !sl.norms) return KVC_ERR_INVALID_ARG;
        if (((uintptr_t)sl.k | (uintptr_t)sl.v) & 15) return KVC_ERR_UNSUPPORTED;
        if (((sl.k_stride_b | sl.k_stride_h | sl.v_stride_b | sl.v_stride_h) * e) & 15) return KVC_ERR_UNSUPPORTED;
    }
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_slab_compress");
    if (guard.status != KVC_OK) return guard.status;
    return for_each_chunk(n_layers, [&](int l0, int nl) -> int {
        const ChunkStats s = chunk_stats(plans + l0, nullptr, nl);
        if (s.n_active == 0) return KVC_OK;
        const LaunchPlan lp = plan_launch(dt, cpr, s, /*light_traffic=*/true, /*in_place=*/true, 0, 0, workspace != nullptr);
        SlabBatchDev bd;
        int st = fill_batch(bd, shape, cpr, s, lp, workspace, workspace_bytes);
        if (st != KVC_OK) return st;
        int m = 0;
        for (int l = l0; l < l0 + nl; ++l) {
            const kvc_layer_plan& p = plans[l];
            const kvc_slab_layer& sl = slabs[l];
            if (p.sink + p.k_sel + p.tail == 0) continue;
            SlabLayerDev& d = bd.layers[m++];
            d.k = (char*)sl.k;
            d.v = (char*)sl.v;
            d.n = (char*)sl.norms;
            d.idx_out = idx_out ? idx_out[l] : nullptr;
            d.idx_in = idx_in ? idx_in[l] : nullptr;
            d.ksb = sl.k_stride_b * e;
            d.ksh = sl.k_stride_h * e;
            d.vsb = sl.v_stride_b * e;
            d.vsh = sl.v_stride_h * e;
            d.nsb = sl.n_stride_b * key_bytes(dt);
            d.nsh = sl.n_stride_h * key_bytes(dt);
            fill_layer_plan(d, p, carry ? carry + l : nullptr, e);
        }
        SlabFn fn = pick_slab(dt, cpr, lp.tp.nt);
        st = ensure_tma_attrs((const void*)fn, shape->device);
        if (st != KVC_OK) return st;
        dim3 grid((unsigned)((int64_t)B * H), (unsigned)s.n_active, 1);
        fn<<<grid, lp.tp.nt, lp.tp.smem, (cudaStream_t)stream>>>(bd);
        return launched("kvc_slab_compress_kernel launch");
    });
}

int kvc_batch_reorder(int32_t device, int32_t batch, const void* index, int32_t index_bits, int32_t n_regions,
                      const kvc_batch_region* regions, void* stream) {
    if (batch < 1 || batch > kReorderMaxBatch || !index || (index_bits != 32 && index_bits != 64) || n_regions < 0 ||
        (n_regions > 0 && !regions))
        return KVC_ERR_INVALID_ARG;
    int n_active = 0;
    for (int i = 0; i < n_regions; ++i) {
        const kvc_batch_region& r = regions[i];
        if (!r.base || r.stride_b < 0 || r.stride_u < 0 || r.unit_bytes < 0 || r.units < 0) return KVC_ERR_INVALID_ARG;
        if (r.units == 0 || r.unit_bytes == 0) continue;
        // every (entry, unit) of the region owns its bytes: entry-major ([B, U, ...]) or unit-major ([U, B, ...])
        const __int128 ub = r.unit_bytes, su = r.stride_u, sb = r.stride_b;
        const bool entry_major = (r.units == 1 || su >= ub) && (batch == 1 || sb >= su * (r.units - 1) + ub);
        const bool unit_major = (batch == 1 || sb >= ub) && (r.units == 1 || su >= sb * (batch - 1) + ub);
        if (!entry_major && !unit_major) return KVC_ERR_INVALID_ARG;
        if (r.elem_bytes != 2 && r.elem_bytes != 4) return KVC_ERR_UNSUPPORTED;
        if (((uintptr_t)r.base | (uint64_t)r.stride_b | (uint64_t)r.stride_u | (uint64_t)r.unit_bytes) % r.elem_bytes)
            return KVC_ERR_UNSUPPORTED;
        ++n_active;
    }
    if (n_active == 0) return KVC_OK;
    // staging: `batch` slots of `chunk` bytes plus four int16 tables; chunk is the largest power of two (16 B .. 16 KB)
    // that keeps them within 48 KB (no opt-in), so that several CTAs stay resident per SM at any batch
    int chunk = 16 * 1024;
    while (chunk > 16 && (int64_t)(chunk + 8) * batch > 48 * 1024) chunk >>= 1;
    const size_t smem = (size_t)batch * chunk + (size_t)batch * 8;
    const int per_sm = std::max(1, std::min(kReorderCtasPerSM, (int)(kSmemPerSM / (smem + 1024 + 16))));
    DeviceGuard guard(device);
    NvtxRange nvtx_range("kvc_batch_reorder");
    if (guard.status != KVC_OK) return guard.status;
    int st = KVC_OK;
    ReorderBatchDev bd;
    memset(&bd, 0, sizeof(bd));
    bd.index = index;
    bd.B = batch;
    bd.index_bits = index_bits;
    bd.chunk = chunk;
    auto launch = [&]() -> int {
        if (bd.n_regions == 0) return KVC_OK;
        const int64_t blocks = std::min<int64_t>(bd.n_items, (int64_t)kSMs * per_sm);  // CTAs stride over the rest
        kvc_batch_reorder_kernel<><<<(unsigned)blocks, kReorderThreads, smem, (cudaStream_t)stream>>>(bd);
        const int s = launched("kvc_batch_reorder_kernel launch");
        bd.n_regions = 0;
        bd.n_items = 0;
        return s;
    };
    for (int i = 0; i < n_regions; ++i) {
        const kvc_batch_region& r = regions[i];
        if (r.units == 0 || r.unit_bytes == 0) continue;
        if (bd.n_regions == kReorderMaxRegions && (st = launch()) != KVC_OK) return st;
        ReorderRegionDev& d = bd.r[bd.n_regions++];
        d.base = (char*)r.base;
        d.sb = r.stride_b;
        d.su = r.stride_u;
        d.unit_bytes = r.unit_bytes;
        d.item0 = bd.n_items;
        d.units = r.units;
        d.nchunk = (int32_t)((r.unit_bytes + chunk - 1) / chunk);
        const uint64_t a = (uintptr_t)r.base | (uint64_t)r.stride_b | (uint64_t)r.stride_u;
        d.g = (a % 16 == 0) ? 16 : (a % 8 == 0) ? 8 : (a % 4 == 0) ? 4 : 2;
        d.e = r.elem_bytes;
        bd.n_items += (int64_t)r.units * d.nchunk;
    }
    return launch();
}

#endif  // KVC_HAS_SLAB

#if KVC_HAS_VOTE
// Shared-memory bytes the fused tail needs inside the (dead) key-tile ring: histogram, kept indices, radix keys
// of the prefix, at least one staging slot of 32 rows.
static size_t vote_tail_bytes(int cpr, int prefix_rows, int idx_cap) {
    const size_t keys = ((size_t)prefix_rows * 2 + 15) & ~(size_t)15;
    return (((size_t)kHistBins * 4 + (size_t)idx_cap * 4 + keys + 127) & ~(size_t)127) + (size_t)32 * cpr * 16;
}

// TMA-fed vote kernel (kvc_vote.cuh): returns KVC_ERR_UNSUPPORTED when a tensor map cannot describe the keys.
// plans / io non-null: the fused form — pool, select and gather behind the vote in the same launch.
static int launch_vote_tma(const kvc_shape* shape, int32_t n_layers, const kvc_vote_layer* layers, int32_t group,
                           int32_t window, int cpr, const kvc_layer_plan* plans, const kvc_layer_io* io, void* stream) {
    EncodeTiledFn encode = tensor_map_encoder();
    if (!encode) return KVC_ERR_UNSUPPORTED;
    const int B = shape->batch, H = shape->heads, D = shape->head_dim, dt = shape->dtype;
    using Fn = void (*)(const VoteTmaBatchDev);
    Fn fn = nullptr;
    if (dt == KVC_DTYPE_BF16)
        fn = cpr == 8 ? kvc_snapkv_vote_tma_kernel<KVC_DTYPE_BF16, 8>
                      : cpr == 10 ? kvc_snapkv_vote_tma_kernel<KVC_DTYPE_BF16, 10> : kvc_snapkv_vote_tma_kernel<KVC_DTYPE_BF16, 16>;
    else
        fn = cpr == 8 ? kvc_snapkv_vote_tma_kernel<KVC_DTYPE_F16, 8>
                      : cpr == 10 ? kvc_snapkv_vote_tma_kernel<KVC_DTYPE_F16, 10> : kvc_snapkv_vote_tma_kernel<KVC_DTYPE_F16, 16>;
    const size_t tile = (size_t)(cpr / 8) * kVoteTile * 128 + (size_t)(cpr % 8) * kVoteTile * 16;
    const size_t smem = 6144 + (size_t)(kVoteM / 8) * cpr * kVoteLBO + (size_t)vote_tma_ring(cpr) * tile;
    int st = ensure_tma_attrs((const void*)fn, shape->device);
    if (st != KVC_OK) return st;
    for (int l0 = 0; l0 < n_layers; l0 += 32) {
        const int nl = (n_layers - l0) < 32 ? (n_layers - l0) : 32;
        static_assert(sizeof(VoteTmaBatchDev) < 32 * 1024, "kernel parameters are limited to 32 KB");
        VoteTmaBatchDev bd;
        memset(&bd, 0, sizeof(bd));
        bd.B = B;
        bd.H = H;
        bd.G = group;
        bd.W = window;
        bd.scale_log2e = 1.4426950408889634f / sqrtf((float)D);
        bd.pad[0] = vote_debug_mode();
#ifdef KVC_LAB
        {   // lab: KVC_VOTE_TIMELINE=<hex device pointer> of a [CTAs][8] int64 buffer
            const char* tl = getenv("KVC_VOTE_TIMELINE");
            bd.lab_timeline = (tl && *tl) ? (long long*)strtoull(tl, nullptr, 16) : nullptr;
        }
#endif
        for (int l = 0; l < nl; ++l) {
            const kvc_vote_layer& v = layers[l0 + l];
            VoteTmaLayerDev& d = bd.layers[l];
            const cuuint64_t dims[4] = {(cuuint64_t)D, (cuuint64_t)v.seq_len, (cuuint64_t)H, (cuuint64_t)B};
            const cuuint64_t strides[3] = {(cuuint64_t)v.k_stride_s * 2, (cuuint64_t)v.k_stride_h * 2,
                                           (cuuint64_t)v.k_stride_b * 2};
            // D = 80: the last 16 elements of every row through the 32-byte-swizzled tail map
            if (!encode_row_maps(encode, &d.map, &d.map_tail, dt == KVC_DTYPE_BF16, v.k_in, dims, strides, kVoteTile, 1))
                return KVC_ERR_UNSUPPORTED;
            d.q = (const char*)v.q_obs;
            d.votes = (char*)v.votes_out;
            d.lse = v.lse;
            d.qsb = v.q_stride_b * 2;
            d.qsh = v.q_stride_h * 2;
            d.qss = v.q_stride_s * 2;
            d.S = v.seq_len;
            if (plans != nullptr) {
                const kvc_layer_plan& p = plans[l0 + l];
                const kvc_layer_io& x = io[l0 + l];
                d.k_in = (const char*)x.k_in;
                d.v_in = (const char*)x.v_in;
                d.k_out = (char*)x.k_out;
                d.v_out = (char*)x.v_out;
                d.idx_out = x.idx_out;
                d.ksb = x.k_stride_b * 2;
                d.ksh = x.k_stride_h * 2;
                d.kss = x.k_stride_s * 2;
                d.vsb = x.v_stride_b * 2;
                d.vsh = x.v_stride_h * 2;
                d.vss = x.v_stride_s * 2;
                d.ksel = p.k_sel;
                d.tail = p.tail;
                d.pool = p.pool_kernel;
                d.idx_cap = (p.k_sel + 3) & ~3;
            }
        }
        dim3 grid((unsigned)((int64_t)B * H), (unsigned)nl, 1);
        fn<<<grid, 576, smem, (cudaStream_t)stream>>>(bd);
        st = launched("kvc_snapkv_vote_tma_kernel launch");
        if (st != KVC_OK) return st;
    }
    return KVC_OK;
}

// The call-wide checks both vote entry points make (the fused form's plans / io present: `more_ok`); KVC_OK with
// n_layers == 0 means there is nothing to do.
static int check_vote_call(const kvc_shape* shape, int32_t n_layers, const kvc_vote_layer* layers, bool more_ok,
                           int32_t group, int32_t window, int* cpr) {
    const int st = check_shape(shape, cpr);
    if (st != KVC_OK) return st;
    if (n_layers < 0 || (n_layers > 0 && (!layers || !more_ok)) || group <= 0 || window <= 0) return KVC_ERR_INVALID_ARG;
    if (n_layers == 0) return KVC_OK;
    if (shape->dtype == KVC_DTYPE_F32) return KVC_ERR_UNSUPPORTED;
    if (*cpr != 8 && *cpr != 10 && *cpr != 16) return KVC_ERR_UNSUPPORTED;
    if ((int64_t)group * window > kVoteM) return KVC_ERR_UNSUPPORTED;
    return KVC_OK;
}

// The checks of one kvc_vote_layer both vote entry points make.
static int check_vote_layer(const kvc_vote_layer& v, int32_t window) {
    if (!v.k_in || !v.q_obs || !v.votes_out || v.seq_len <= window) return KVC_ERR_INVALID_ARG;
    if (((uintptr_t)v.k_in | (uintptr_t)v.q_obs) & 15) return KVC_ERR_UNSUPPORTED;
    const int64_t sb = v.k_stride_b | v.k_stride_h | v.k_stride_s | v.q_stride_b | v.q_stride_h | v.q_stride_s;
    if ((sb * 2) & 15) return KVC_ERR_UNSUPPORTED;
    return KVC_OK;
}

int kvc_snapkv_vote(const kvc_shape* shape, int32_t n_layers, const kvc_vote_layer* layers, int32_t group,
                    int32_t window, void* stream) {
    int cpr = 0;
    int st = check_vote_call(shape, n_layers, layers, true, group, window, &cpr);
    if (st != KVC_OK || n_layers == 0) return st;
    for (int l = 0; l < n_layers; ++l) {
        st = check_vote_layer(layers[l], window);
        if (st != KVC_OK) return st;
    }
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_snapkv_vote");
    if (guard.status != KVC_OK) return guard.status;
    // key tiles arrive through TMA tensor loads: layouts a tensor map cannot describe are KVC_ERR_UNSUPPORTED (the
    // Python layer makes such keys contiguous first)
    return launch_vote_tma(shape, n_layers, layers, group, window, cpr, nullptr, nullptr, stream);
}

int kvc_snapkv_vote_compress(const kvc_shape* shape, int32_t n_layers, const kvc_vote_layer* layers,
                             const kvc_layer_plan* plans, const kvc_layer_io* io, int32_t group, int32_t window,
                             void* stream) {
    int cpr = 0;
    int st = check_vote_call(shape, n_layers, layers, plans && io, group, window, &cpr);
    if (st != KVC_OK || n_layers == 0) return st;
    const size_t ring_bytes = (size_t)vote_tma_ring(cpr) * ((size_t)(cpr / 8) * kVoteTile * 128 + (size_t)(cpr % 8) * kVoteTile * 16);
    for (int l = 0; l < n_layers; ++l) {
        const kvc_vote_layer& v = layers[l];
        const kvc_layer_plan& p = plans[l];
        const kvc_layer_io& x = io[l];
        st = check_vote_layer(v, window);
        if (st != KVC_OK) return st;
        // the plan of snapkv_lite in vote mode: no sinks, the prefix [0, S - W) ranked by pooled votes, the window kept
        if (p.seq_len != v.seq_len || p.sink != 0 || p.sel_lo != 0 || p.sel_hi != v.seq_len - window || p.k_sel <= 0 ||
            p.k_sel > p.sel_hi || p.tail < 0 || p.tail > window || p.score != KVC_SCORE_GIVEN_SCORE)
            return KVC_ERR_INVALID_ARG;
        if (p.pool_kernel > 2 * kMaxPoolHalo) return KVC_ERR_UNSUPPORTED;
        if (!x.k_in || !x.v_in || !x.k_out || !x.v_out || x.k_in != v.k_in) return KVC_ERR_INVALID_ARG;
        if (((uintptr_t)x.v_in | (uintptr_t)x.k_out | (uintptr_t)x.v_out) & 15) return KVC_ERR_UNSUPPORTED;
        if (((x.v_stride_b | x.v_stride_h | x.v_stride_s) * 2) & 15) return KVC_ERR_UNSUPPORTED;
        if (x.k_stride_b != v.k_stride_b || x.k_stride_h != v.k_stride_h || x.k_stride_s != v.k_stride_s)
            return KVC_ERR_INVALID_ARG;
        if (vote_tail_bytes(cpr, p.sel_hi, (p.k_sel + 3) & ~3) > ring_bytes) return KVC_ERR_TOO_LARGE;
    }
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_snapkv_vote_compress");
    if (guard.status != KVC_OK) return guard.status;
    return launch_vote_tma(shape, n_layers, layers, group, window, cpr, plans, io, stream);
}

int kvc_query_window_push(const kvc_shape* shape, int32_t window, int32_t n_layers, const kvc_qwin_layer* layers,
                          void* stream) {
    int cpr = 0;
    const int st = check_shape(shape, &cpr);
    if (st != KVC_OK) return st;
    if (window < 1 || window > kQwinMaxRows || n_layers < 0 || (n_layers > 0 && !layers)) return KVC_ERR_INVALID_ARG;
    if (shape->dtype == KVC_DTYPE_F32) return KVC_ERR_UNSUPPORTED;
    for (int l = 0; l < n_layers; ++l) {
        const kvc_qwin_layer& x = layers[l];
        if (!x.q_new || !x.window || x.filled < 0 || x.filled > window || x.n_new < 0) return KVC_ERR_INVALID_ARG;
        if (((uintptr_t)x.q_new | (uintptr_t)x.window) & 15) return KVC_ERR_UNSUPPORTED;
        if (((x.q_stride_b | x.q_stride_h | x.q_stride_s | x.w_stride_b | x.w_stride_h) * 2) & 15)
            return KVC_ERR_UNSUPPORTED;
    }
    if (n_layers == 0) return KVC_OK;
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_query_window_push");
    if (guard.status != KVC_OK) return guard.status;
    return for_each_chunk(n_layers, [&](int l0, int nl) -> int {
        QwinBatchDev bd;
        memset(&bd, 0, sizeof(bd));
        bd.Hq = shape->heads;
        bd.cpr = cpr;
        bd.window = window;
        int n_active = 0;
        for (int l = l0; l < l0 + nl; ++l) {
            const kvc_qwin_layer& x = layers[l];
            if (x.n_new == 0) continue;
            QwinLayerDev& d = bd.layers[n_active++];
            d.q = (const char*)x.q_new;
            d.qsb = x.q_stride_b * 2;
            d.qsh = x.q_stride_h * 2;
            d.qss = x.q_stride_s * 2;
            d.w = (char*)x.window;
            d.wsb = x.w_stride_b * 2;
            d.wsh = x.w_stride_h * 2;
            d.filled = x.filled;
            d.n_new = x.n_new;
        }
        if (n_active == 0) return KVC_OK;
        dim3 grid((unsigned)((int64_t)shape->batch * shape->heads), (unsigned)n_active, 1);
        kvc_query_window_push_kernel<kQwinChunks><<<grid, kQwinThreads, 0, (cudaStream_t)stream>>>(bd);
        return launched("kvc_query_window_push_kernel launch");
    });
}

#endif  // KVC_HAS_VOTE

#if KVC_HAS_H2O
// kvc_h2o_accumulate's launches, arguments already checked (also the score-row launch of kvc_h2o_accumulate_qk_tc).
static int launch_h2o_accumulate(int B, int H, int dt, int32_t n_layers, const kvc_h2o_layer* layers, float decay,
                                 void* stream) {
    const int e = elem_bytes(dt);
    const int tc = 32 * (16 / e);  // key columns per CTA
    return for_each_chunk(n_layers, [&](int l0, int nl) -> int {
        H2oBatchDev bd;
        memset(&bd, 0, sizeof(bd));
        bd.B = B;
        bd.H = H;
        bd.decay = decay;
        int n_active = 0, max_tiles = 0;
        for (int l = 0; l < nl; ++l) {
            const kvc_h2o_layer& x = layers[l0 + l];
            if (x.key_len == 0) continue;
            H2oLayerDev& d = bd.layers[n_active++];
            d.attn = (const char*)x.attn;
            d.asb = x.a_stride_b * e;
            d.ash = x.a_stride_h * e;
            d.asq = x.a_stride_q * e;
            d.acc = (char*)x.acc;
            d.csb = x.acc_stride_b * e;
            d.csh = x.acc_stride_h * e;
            d.score = x.score_hi > x.score_lo ? (char*)x.score_out : nullptr;
            d.Q = x.n_query;
            d.K = x.key_len;
            d.prev = x.prev_len;
            d.lo = x.score_lo;
            d.hi = x.score_hi;
            d.vec = x.attn && ((uintptr_t)x.attn % 16 == 0) && ((d.asb | d.ash | d.asq) % 16 == 0);
            const int tiles = (x.key_len + tc - 1) / tc;
            if (tiles > max_tiles) max_tiles = tiles;
        }
        if (n_active == 0) return KVC_OK;
        dim3 grid((unsigned)max_tiles, (unsigned)B, (unsigned)n_active);
        by_dtype(dt, [&](auto d) { kvc_h2o_accumulate_kernel<d><<<grid, kH2oThreads, 0, (cudaStream_t)stream>>>(bd); });
        return launched("kvc_h2o_accumulate_kernel launch");
    });
}

int kvc_h2o_accumulate(const kvc_shape* shape, int32_t n_layers, const kvc_h2o_layer* layers, float decay,
                       void* stream) {
    if (!shape || n_layers < 0 || (n_layers > 0 && !layers)) return KVC_ERR_INVALID_ARG;
    const int B = shape->batch, H = shape->heads, dt = shape->dtype;
    if (B <= 0 || H <= 0 || B > 65535) return KVC_ERR_INVALID_ARG;
    if (dt != KVC_DTYPE_F32 && dt != KVC_DTYPE_F16 && dt != KVC_DTYPE_BF16) return KVC_ERR_UNSUPPORTED;
    if (n_layers == 0) return KVC_OK;
    const int e = elem_bytes(dt);
    for (int l = 0; l < n_layers; ++l) {
        const kvc_h2o_layer& x = layers[l];
        if (x.key_len < 0 || !x.acc) return KVC_ERR_INVALID_ARG;
        if (x.attn && x.n_query <= 0) return KVC_ERR_INVALID_ARG;
        if (x.score_lo < 0 || x.score_hi < x.score_lo || x.score_hi > x.key_len) return KVC_ERR_INVALID_ARG;
        if (x.score_hi > x.score_lo && !x.score_out) return KVC_ERR_INVALID_ARG;
        if (((uintptr_t)x.attn | (uintptr_t)x.acc | (uintptr_t)x.score_out) % e) return KVC_ERR_UNSUPPORTED;
    }
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_h2o_accumulate");
    if (guard.status != KVC_OK) return guard.status;
    return launch_h2o_accumulate(B, H, dt, n_layers, layers, decay, stream);
}

// ------------------------------------------------------------------ kvc_h2o_accumulate_qk
// Pass-1 key splits: at most kQkMaxSplits, each a whole number of 128-row tiles (a function of key_len only).
static void qk_splits(int key_len, int* n_split, int* split_tiles) {
    const int tiles = (key_len + kQkRows - 1) / kQkRows;
    const int want = tiles < kQkMaxSplits ? tiles : kQkMaxSplits;
    *split_tiles = want > 0 ? (tiles + want - 1) / want : 1;
    *n_split = want > 0 ? (tiles + *split_tiles - 1) / *split_tiles : 0;
}

static int64_t qk_layer_ws(const kvc_shape* shape, int group, const kvc_h2o_qk_layer& x) {
    if (x.key_len <= 0) return 0;
    int n_split, split_tiles;
    qk_splits(x.key_len, &n_split, &split_tiles);
    const int64_t bytes = (int64_t)shape->batch * shape->heads * group * x.n_query * n_split * 8;
    return (bytes + 255) & ~(int64_t)255;
}

static int qk_validate(const kvc_shape* shape, int32_t group, int32_t n_layers, const kvc_h2o_qk_layer* layers) {
    if (!shape || n_layers < 0 || (n_layers > 0 && !layers) || group < 1) return KVC_ERR_INVALID_ARG;
    const int B = shape->batch, H = shape->heads, D = shape->head_dim, dt = shape->dtype;
    if (B <= 0 || H <= 0 || D <= 0 || (int64_t)B * H > 65535) return KVC_ERR_INVALID_ARG;
    if (dt != KVC_DTYPE_F32 && dt != KVC_DTYPE_F16 && dt != KVC_DTYPE_BF16) return KVC_ERR_UNSUPPORTED;
    const int e = elem_bytes(dt);
    if ((D * e) % 16 || D * e > kQkMaxRowBytes) return KVC_ERR_UNSUPPORTED;
    for (int l = 0; l < n_layers; ++l) {
        const kvc_h2o_qk_layer& x = layers[l];
        if (x.key_len < 0 || x.n_query <= 0 || !x.acc || !x.q || !x.k) return KVC_ERR_INVALID_ARG;
        if (!x.mask && x.n_query > x.key_len) return KVC_ERR_INVALID_ARG;
        if (x.score_lo < 0 || x.score_hi < x.score_lo || x.score_hi > x.key_len) return KVC_ERR_INVALID_ARG;
        if (x.score_hi > x.score_lo && !x.score_out) return KVC_ERR_INVALID_ARG;
        if (((uintptr_t)x.q | (uintptr_t)x.acc | (uintptr_t)x.score_out) % e) return KVC_ERR_UNSUPPORTED;
        if ((uintptr_t)x.k % 16 || (x.k_stride_b * e) % 16 || (x.k_stride_h * e) % 16 || (x.k_stride_s * e) % 16)
            return KVC_ERR_UNSUPPORTED;
    }
    return KVC_OK;
}

int64_t kvc_h2o_qk_workspace_bytes(const kvc_shape* shape, int32_t group, int32_t n_layers,
                                   const kvc_h2o_qk_layer* layers) {
    if (qk_validate(shape, group, n_layers, layers) != KVC_OK) return -1;
    int64_t total = 0;
    for (int l = 0; l < n_layers; ++l) total += qk_layer_ws(shape, group, layers[l]);
    return total;
}

using QkFn = void (*)(const H2oQkBatchDev);

extern "C++" {
template <int DT>
static QkFn pick_qk(bool stats, int qt) {
    if (stats) return qt == 8 ? kvc_h2o_qk_stats_kernel<DT, 8> : qt == 4 ? kvc_h2o_qk_stats_kernel<DT, 4>
                                                                          : kvc_h2o_qk_stats_kernel<DT, 1>;
    return qt == 8 ? kvc_h2o_qk_accumulate_kernel<DT, 8> : qt == 4 ? kvc_h2o_qk_accumulate_kernel<DT, 4>
                                                                   : kvc_h2o_qk_accumulate_kernel<DT, 1>;
}
}

int kvc_h2o_accumulate_qk(const kvc_shape* shape, int32_t group, int32_t n_layers, const kvc_h2o_qk_layer* layers,
                          float decay, void* workspace, int64_t workspace_bytes, void* stream) {
    const int v = qk_validate(shape, group, n_layers, layers);
    if (v != KVC_OK) return v;
    int64_t need = 0;
    for (int l = 0; l < n_layers; ++l) need += qk_layer_ws(shape, group, layers[l]);
    if (need > 0 && (!workspace || workspace_bytes < need || (uintptr_t)workspace % 16)) return KVC_ERR_INVALID_ARG;
    if (need == 0) return KVC_OK;  // every layer has key_len 0
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_h2o_accumulate_qk");
    if (guard.status != KVC_OK) return guard.status;
    const int B = shape->batch, Hkv = shape->heads, D = shape->head_dim, dt = shape->dtype;
    const int e = elem_bytes(dt);
    const int rb = D * e, pitch = ((rb / 16) | 1) * 16;
    char* ws = (char*)workspace;
    return for_each_chunk(n_layers, [&](int l0, int nl) -> int {
        H2oQkBatchDev bd;
        memset(&bd, 0, sizeof(bd));
        bd.B = B;
        bd.Hkv = Hkv;
        bd.G = group;
        bd.D = D;
        bd.decay = decay;
        bd.pitch = pitch;
        int n_active = 0, max_x1 = 0, max_tiles = 0, max_gt = 0;
        for (int l = 0; l < nl; ++l) {
            const kvc_h2o_qk_layer& x = layers[l0 + l];
            if (x.key_len == 0) continue;
            H2oQkLayerDev& d = bd.layers[n_active++];
            d.q = (const char*)x.q;
            d.qsb = x.q_stride_b * e;
            d.qsh = x.q_stride_h * e;
            d.qst = x.q_stride_t * e;
            d.k = (const char*)x.k;
            d.ksb = x.k_stride_b * e;
            d.ksh = x.k_stride_h * e;
            d.kss = x.k_stride_s * e;
            d.mask = x.mask;
            d.msb = x.m_stride_b;
            d.mst = x.m_stride_t;
            d.acc = (char*)x.acc;
            d.csb = x.acc_stride_b * e;
            d.csh = x.acc_stride_h * e;
            d.score = x.score_hi > x.score_lo ? (char*)x.score_out : nullptr;
            d.ws = (float2*)ws;
            ws += qk_layer_ws(shape, group, x);
            d.scaling = x.scaling;
            d.T = x.n_query;
            d.K = x.key_len;
            d.prev = x.prev_len;
            d.lo = x.score_lo;
            d.hi = x.score_hi;
            qk_splits(x.key_len, &d.n_split, &d.split_tiles);
            const int gt = group * x.n_query;
            d.n_qt = (gt + kQkQ1 - 1) / kQkQ1;
            if (d.n_split * d.n_qt > max_x1) max_x1 = d.n_split * d.n_qt;
            const int tiles = (x.key_len + kQkRows - 1) / kQkRows;
            if (tiles > max_tiles) max_tiles = tiles;
            if (gt > max_gt) max_gt = gt;
        }
        if (n_active == 0) return KVC_OK;
        // queries per register tile: the work of a (query, key) pair does not depend on it, only the speed does
        const int qt = max_gt >= 8 ? 8 : max_gt >= 4 ? 4 : 1;
        QkFn stats, accum;
        by_dtype(dt, [&](auto d) {
            stats = pick_qk<d>(true, qt);
            accum = pick_qk<d>(false, qt);
        });
        const size_t smem_k = 128 + 2 * (size_t)kQkRows * pitch;
        const size_t smem1 = smem_k + (size_t)kQkQ1 * D * 4 + 2 * (size_t)kQkQ1 * kQkThreads * 4;
        const size_t smem2 = smem_k + (size_t)kQkQ2 * D * 4 + (size_t)kQkQ2 * 4;
        int st = ensure_tma_attrs((const void*)stats, shape->device);
        if (st != KVC_OK) return st;
        st = ensure_tma_attrs((const void*)accum, shape->device);
        if (st != KVC_OK) return st;
        stats<<<dim3((unsigned)max_x1, (unsigned)(B * Hkv), (unsigned)n_active), kQkThreads, smem1,
                 (cudaStream_t)stream>>>(bd);
        st = launched("kvc_h2o_qk_stats_kernel launch");
        if (st != KVC_OK) return st;
        accum<<<dim3((unsigned)max_tiles, (unsigned)B, (unsigned)n_active), kQkThreads, smem2, (cudaStream_t)stream>>>(bd);
        return launched("kvc_h2o_qk_accumulate_kernel launch");
    });
}

// ------------------------------------------------------------------ kvc_h2o_accumulate_qk_tc
// Query tiles of a layer: tb = 128 / G positions each (G heads x tb positions = at most 128 MMA rows).
static int tc_query_tiles(int group, int n_query) { return (n_query + 128 / group - 1) / (128 / group); }

static int64_t tc_layer_ws(const kvc_shape* shape, int group, const kvc_h2o_qk_layer& x) {
    if (x.key_len <= 0) return 0;
    const int64_t bytes = (int64_t)shape->batch * shape->heads * tc_query_tiles(group, x.n_query) * kTcRows * 4;
    return (bytes + 255) & ~(int64_t)255;
}

// qk_validate's checks, then what the tensor-core form does not cover: fp32, head_dim outside {64, 80, 128}, more than
// 128 query heads per KV head, and q / K layouts a tensor map cannot describe (16-byte aligned base and strides).
static int tc_validate(const kvc_shape* shape, int32_t group, int32_t n_layers, const kvc_h2o_qk_layer* layers) {
    const int v = qk_validate(shape, group, n_layers, layers);
    if (v != KVC_OK) return v;
    const int D = shape->head_dim;
    if (shape->dtype == KVC_DTYPE_F32 || (D != 64 && D != 80 && D != 128) || group > kTcRows) return KVC_ERR_UNSUPPORTED;
    for (int l = 0; l < n_layers; ++l) {
        const kvc_h2o_qk_layer& x = layers[l];
        if ((uintptr_t)x.q % 16 || (x.q_stride_b * 2) % 16 || (x.q_stride_h * 2) % 16 || (x.q_stride_t * 2) % 16)
            return KVC_ERR_UNSUPPORTED;
    }
    return KVC_OK;
}

int64_t kvc_h2o_qk_tc_workspace_bytes(const kvc_shape* shape, int32_t group, int32_t n_layers,
                                      const kvc_h2o_qk_layer* layers) {
    if (tc_validate(shape, group, n_layers, layers) != KVC_OK) return -1;
    int64_t total = 0;
    for (int l = 0; l < n_layers; ++l) total += tc_layer_ws(shape, group, layers[l]);
    return total;
}

using TcFn = void (*)(const H2oTcBatchDev);

extern "C++" {
template <int DT>
static TcFn pick_tc(bool cols, int cpr) {
    if (cols) return cpr == 8 ? kvc_h2o_tc_kernel<DT, 8, true> : cpr == 10 ? kvc_h2o_tc_kernel<DT, 10, true>
                                                                           : kvc_h2o_tc_kernel<DT, 16, true>;
    return cpr == 8 ? kvc_h2o_tc_kernel<DT, 8, false> : cpr == 10 ? kvc_h2o_tc_kernel<DT, 10, false>
                                                                  : kvc_h2o_tc_kernel<DT, 16, false>;
}
}

int kvc_h2o_accumulate_qk_tc(const kvc_shape* shape, int32_t group, int32_t n_layers, const kvc_h2o_qk_layer* layers,
                             float decay, void* workspace, int64_t workspace_bytes, void* stream) {
    const int v = tc_validate(shape, group, n_layers, layers);
    if (v != KVC_OK) return v;
    int64_t need = 0;
    for (int l = 0; l < n_layers; ++l) need += tc_layer_ws(shape, group, layers[l]);
    if (need > 0 && (!workspace || workspace_bytes < need || (uintptr_t)workspace % 16)) return KVC_ERR_INVALID_ARG;
    if (need == 0) return KVC_OK;  // every layer has key_len 0
    DeviceGuard guard(shape->device);
    NvtxRange nvtx_range("kvc_h2o_accumulate_qk_tc");
    if (guard.status != KVC_OK) return guard.status;
    EncodeTiledFn encode = tensor_map_encoder();
    if (!encode) return KVC_ERR_UNSUPPORTED;
    const int B = shape->batch, Hkv = shape->heads, D = shape->head_dim, dt = shape->dtype;
    const int cpr = D * 2 / 16, tb = kTcRows / group;
    const bool bf16 = dt == KVC_DTYPE_BF16;
    const TcFn rows = bf16 ? pick_tc<KVC_DTYPE_BF16>(false, cpr) : pick_tc<KVC_DTYPE_F16>(false, cpr);
    const TcFn cols = bf16 ? pick_tc<KVC_DTYPE_BF16>(true, cpr) : pick_tc<KVC_DTYPE_F16>(true, cpr);
    const size_t smem = (size_t)tc_smem_bytes(cpr, group);
    int st = ensure_tma_attrs((const void*)rows, shape->device);
    if (st != KVC_OK) return st;
    st = ensure_tma_attrs((const void*)cols, shape->device);
    if (st != KVC_OK) return st;
    char* ws = (char*)workspace;
    for (int l0 = 0; l0 < n_layers; l0 += kTcLayers) {
        const int nl = std::min(n_layers - l0, kTcLayers);
        H2oTcBatchDev bd;
        memset(&bd, 0, sizeof(bd));
        bd.B = B;
        bd.Hkv = Hkv;
        bd.G = group;
        bd.tb = tb;
        bd.decay = decay;
        kvc_h2o_layer rescore[kTcLayers];
        int n_active = 0, n_scored = 0, max_qt = 0, max_kt = 0;
        for (int l = 0; l < nl; ++l) {
            const kvc_h2o_qk_layer& x = layers[l0 + l];
            if (x.key_len == 0) continue;
            H2oTcLayerDev& d = bd.layers[n_active++];
            const cuuint64_t qdims[4] = {(cuuint64_t)D, (cuuint64_t)x.n_query, (cuuint64_t)Hkv * group, (cuuint64_t)B};
            const cuuint64_t qstr[3] = {(cuuint64_t)x.q_stride_t * 2, (cuuint64_t)x.q_stride_h * 2,
                                        (cuuint64_t)x.q_stride_b * 2};
            const cuuint64_t kdims[4] = {(cuuint64_t)D, (cuuint64_t)x.key_len, (cuuint64_t)Hkv, (cuuint64_t)B};
            const cuuint64_t kstr[3] = {(cuuint64_t)x.k_stride_s * 2, (cuuint64_t)x.k_stride_h * 2,
                                        (cuuint64_t)x.k_stride_b * 2};
            if (!encode_row_maps(encode, &d.qmap, &d.qmap_tail, bf16, x.q, qdims, qstr, tb, group) ||
                !encode_row_maps(encode, &d.kmap, &d.kmap_tail, bf16, x.k, kdims, kstr, kTcRows, 1))
                return KVC_ERR_UNSUPPORTED;
            d.mask = x.mask;
            d.msb = x.m_stride_b;
            d.mst = x.m_stride_t;
            d.acc = (char*)x.acc;
            d.csb = x.acc_stride_b * 2;
            d.csh = x.acc_stride_h * 2;
            d.lse = (float*)ws;
            ws += tc_layer_ws(shape, group, x);
            d.c2 = x.scaling * 1.4426950408889634f;
            d.T = x.n_query;
            d.K = x.key_len;
            d.prev = x.prev_len;
            d.n_qt = tc_query_tiles(group, x.n_query);
            d.n_kt = (x.key_len + kTcRows - 1) / kTcRows;
            max_qt = std::max(max_qt, d.n_qt);
            max_kt = std::max(max_kt, d.n_kt);
            if (x.score_hi > x.score_lo) {  // the score row: kvc_h2o_accumulate's re-score of the updated accumulators
                kvc_h2o_layer& r = rescore[n_scored++];
                memset(&r, 0, sizeof(r));
                r.acc = x.acc;
                r.acc_stride_b = x.acc_stride_b;
                r.acc_stride_h = x.acc_stride_h;
                r.score_out = x.score_out;
                r.key_len = x.key_len;
                r.prev_len = x.key_len;
                r.score_lo = x.score_lo;
                r.score_hi = x.score_hi;
            }
        }
        if (n_active == 0) continue;
        rows<<<dim3((unsigned)max_qt, (unsigned)(B * Hkv), (unsigned)n_active), kTcThreads, smem, (cudaStream_t)stream>>>(bd);
        st = launched("kvc_h2o_tc_kernel (rows) launch");
        if (st != KVC_OK) return st;
        cols<<<dim3((unsigned)max_kt, (unsigned)(B * Hkv), (unsigned)n_active), kTcThreads, smem, (cudaStream_t)stream>>>(bd);
        st = launched("kvc_h2o_tc_kernel (columns) launch");
        if (st != KVC_OK) return st;
        if (n_scored > 0) {
            st = launch_h2o_accumulate(B, Hkv * group, dt, n_scored, rescore, decay, stream);
            if (st != KVC_OK) return st;
        }
    }
    return KVC_OK;
}
#endif  // KVC_HAS_H2O

}  // extern "C"
