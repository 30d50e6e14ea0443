/*
 * kvc.h — C ABI of libkvc_sm100a.so: the B200 (sm_100a) per-step KV-cache
 * compression hot path of `kvcompress`.
 *
 * The reference has no FFI layer: its plugin boundary is the Python callable
 *   fn(past_key_values, <method kwargs>, skip_layers=..., **kwargs)
 *       -> List[Tuple[Tensor, Tensor]]
 * (reference kvcompress/methods/base.py:12-33, registry methods/__init__.py:21-78).
 * Every one of the eight hot-path methods reduces, per layer, to one descriptor
 *   keep [0,sink)  U  (k_sel rows of [sel_lo,sel_hi) chosen by a key)  U  [S-tail,S)
 * emitted in ascending token order for K and V (SURVEY.md §8a).  The Python
 * planner computes the integers exactly as the reference does; this library does
 * all device work.  Entry points and the reference code they replace:
 *
 *   kvc_compress_layers  per-layer  torch.norm -> argsort/topk -> sort -> expand ->
 *                        gather x2 -> cat x2, for every layer of the call in ONE launch
 *                        (l2_compress.py:70-88, fix_size_l2.py:104-147,
 *                         streaming_llm.py:99-107, h2o_l2.py:116-149,
 *                         snapkv_lite.py:93-150, pyramid_kv.py:150-181,
 *                         adaptive_l2.py:116-143,176-197)
 *   kvc_key_norms        torch.norm(K, p=2, dim=-1)            (e.g. l2_compress.py:70)
 *   kvc_select           argsort()[..., :k] + torch.sort / torch.topk + torch.sort
 *                        over caller-supplied scores           (e.g. h2o_l2.py:128-132,
 *                         snapkv_lite.py:134-137)
 *
 * Conventions: plain pointers and sizes only; the library allocates nothing and
 * never synchronises; all work is enqueued on `stream` (a cudaStream_t passed as
 * void*); every function returns a kvc_status (0 = ok).  Tensors are device
 * pointers to [B, H, S, D] arrays whose last dimension is dense (stride 1) and
 * whose rows are 16-byte aligned; B/H/S strides are given in ELEMENTS.  Outputs are
 * dense [B, H, C, D] with C = sink + k_sel + tail.  There is no CPU path.
 * "Device pointer" includes page-locked host memory mapped into the device's address
 * space (cudaHostAlloc / cudaHostRegister under UVA): an offloaded cache is then read
 * and written in place over PCIe, each needed row crossing the link once per read.
 * Every entry point runs on shape->device and restores the calling thread's current CUDA
 * device before it returns.  The library reads no environment variable.  Each entry point that
 * launches opens an NVTX range named after itself (kvc_compress_layers_ws, kvc_slab_append, ...),
 * so profilers attribute every kernel to the C-ABI call that enqueued it.
 */
#ifndef KVC_H_
#define KVC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Additions that leave every existing struct layout, enum value and entry point as it was (a new score kind, the
 * kvc_h2o_layer / kvc_h2o_qk_layer / kvc_carry_layer structs and their entry points) keep the version: a caller built against an older header sees the
 * same ABI, and a caller that uses the additions fails to link or gets KVC_ERR_INVALID_ARG from an older library. */
#define KVC_ABI_VERSION 5

typedef enum kvc_status {
    KVC_OK = 0,
    KVC_ERR_INVALID_ARG = 1, /* null pointer, negative size, inconsistent plan */
    KVC_ERR_UNSUPPORTED = 2, /* dtype / head_dim / alignment the kernels do not cover */
    KVC_ERR_TOO_LARGE = 3,   /* selection region does not fit the on-chip score buffer */
    KVC_ERR_CUDA = 4         /* launch or runtime failure; see kvc_last_cuda_error() */
} kvc_status;

typedef enum kvc_dtype {
    KVC_DTYPE_F32 = 0,
    KVC_DTYPE_F16 = 1,
    KVC_DTYPE_BF16 = 2
} kvc_dtype;

/* How rows of [sel_lo, sel_hi) are ranked. Ties always go to the lowest token index. */
typedef enum kvc_score_kind {
    KVC_SCORE_NONE = 0,        /* k_sel must be 0: pure sink + tail slice (streaming_llm.py:99-107) */
    KVC_SCORE_L2_LOW = 1,      /* keep the k_sel lowest  ||K||_2  (norm().argsort()[:k])            */
    KVC_SCORE_L2_HIGH = 2,     /* keep the k_sel highest ||K||_2  (argsort(descending=True)[:k])    */
    KVC_SCORE_SNAPKV_POOL = 3, /* (max norm + 1e-6 - norm) -> avg_pool1d -> topk (snapkv_lite.py:96-134) */
    KVC_SCORE_GIVEN_INDEX = 4, /* caller supplies ascending absolute row indices (fix_size_l2 "random") */
    KVC_SCORE_GIVEN_SCORE = 5, /* caller supplies per-row scores (score_in): avg_pool1d(pool_kernel) -> keep the
                                  k_sel HIGHEST (snapkv vote mode: kvc_snapkv_vote output; h2o_attention.py:194-213) */
    KVC_SCORE_GIVEN_SCORE_SHARED = 6 /* as GIVEN_SCORE, but score_in is [B, sel_hi-sel_lo] (cache dtype, dense): ONE
                                        row per batch entry, used by every head (H2O's head-summed attention mass,
                                        h2o_attention.py:194-213; kvc_h2o_accumulate's score_out) */
} kvc_score_kind;

/* One layer's keep-plan: integers computed by the host planner (reference arithmetic). */
typedef struct kvc_layer_plan {
    int32_t seq_len;     /* S of this layer's input                           */
    int32_t sink;        /* rows [0, sink) are kept                            */
    int32_t sel_lo;      /* selection region [sel_lo, sel_hi)                  */
    int32_t sel_hi;
    int32_t k_sel;       /* rows to keep from the region, 0 <= k_sel <= sel_hi - sel_lo */
    int32_t tail;        /* rows [S - tail, S) are kept                        */
    int32_t score;       /* kvc_score_kind                                     */
    int32_t pool_kernel; /* SNAPKV_POOL: avg_pool1d kernel size (<=1: no pooling) */
} kvc_layer_plan;

/* One layer's device buffers. */
typedef struct kvc_layer_io {
    const void* k_in;  /* [B,H,S,D] keys                         */
    const void* v_in;  /* [B,H,S,D] values                       */
    void* k_out;       /* [B,H,C,D] dense                        */
    void* v_out;       /* [B,H,C,D] dense                        */
    int64_t k_stride_b, k_stride_h, k_stride_s; /* elements      */
    int64_t v_stride_b, v_stride_h, v_stride_s; /* elements      */
    int32_t* idx_out;      /* optional [B,H,C] kept absolute row indices, ascending; may be NULL */
    const int32_t* idx_in; /* GIVEN_INDEX only: [B,H,k_sel] ascending absolute rows inside the region (rows outside
                              [0, seq_len) are clamped into the layer, never dereferenced) */
    const void* score_in;  /* GIVEN_SCORE only: [B,H,sel_hi-sel_lo] scores of the region's rows, cache dtype, dense */
    /* Optional stored key norms (L2_LOW / L2_HIGH / SNAPKV_POOL): norms_in[b,h,s] = what torch.norm(K, p=2, dim=-1)
     * returns for row s, cache dtype, rows [0, seq_len) valid.  When given, the K rows of the selection region are NOT
     * read for scoring (2-4 bytes per row instead of head_dim*e): a slab cache records the norms at append time
     * (kvc_slab_append).  The kept set is the one the scan would have produced from the same norms.  NULL: scan K. */
    const void* norms_in;
    int64_t n_stride_b, n_stride_h; /* elements */
} kvc_layer_io;

typedef struct kvc_shape {
    int32_t batch;    /* B */
    int32_t heads;    /* H (KV heads) */
    int32_t head_dim; /* D; D * sizeof(dtype) must be a multiple of 16 */
    int32_t dtype;    /* kvc_dtype */
    int32_t device;   /* CUDA device ordinal all pointers live on */
} kvc_shape;

/* ABI / build information. */
int kvc_abi_version(void);
const char* kvc_build_info(void);      /* e.g. "sm_100a nvcc 12.9" */
const char* kvc_status_string(int status);
const char* kvc_last_cuda_error(void); /* text of the last CUDA failure seen by this thread */
/* Number of kernels this library has launched in this process (monotonic). */
int64_t kvc_launch_count(void);
/* Largest selection region (rows) kvc_compress_layers can score on chip for this dtype / k_sel. */
int32_t kvc_max_region_rows(int32_t dtype, int32_t k_sel);

/* Compress n_layers layers in one launch (chunks of KVC_MAX_LAYERS_PER_LAUNCH). */
#define KVC_MAX_LAYERS_PER_LAUNCH 64
int kvc_compress_layers(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                        const kvc_layer_io* io, void* stream);

/* Selections too large for shared memory (radix keys of the region + kept indices: e.g. l2_compress with
 * keep_ratio 0.8 at 32K fp32 rows, or any region beyond kvc_max_region_rows) keep those two arrays in a
 * caller-provided device workspace instead (they stay L2-resident: 2-4 B per row against D*e for the scan).
 * kvc_workspace_bytes: bytes kvc_compress_layers_ws / kvc_slab_compress need for these plans, 0 if everything
 * fits on chip.  kvc_compress_layers(...) == kvc_compress_layers_ws(..., NULL, 0, ...), which reports
 * KVC_ERR_TOO_LARGE when a workspace would have been needed. */
int64_t kvc_workspace_bytes(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans);
/* Pure host arithmetic, for tests and profiling notes: the launch shape kvc_compress_layers would use for the first
 * launch of these plans when it scans K — out = {threads per CTA, resident CTAs per SM, staging slots of 32 rows per
 * CTA, 1 if keys / kept indices go to the workspace}. */
int kvc_launch_shape(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans, int32_t out[4]);
int kvc_compress_layers_ws(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                           const kvc_layer_io* io, void* workspace, int64_t workspace_bytes, void* stream);

/* norms[b,h,r] = dtype( sqrt( sum_d fp32(K[b,h,row_lo+r,d])^2 ) ), r in [0,row_hi-row_lo);
 * fp32 accumulation, result rounded once to the input dtype (torch.norm semantics). */
int kvc_key_norms(const kvc_shape* shape, const void* k_in, int64_t stride_b, int64_t stride_h,
                  int64_t stride_s, int32_t row_lo, int32_t row_hi, void* norms_out, void* stream);

/* Per (b,h) row of `scores` ([n_rows, n] of `dtype`, dense): the k smallest (largest if
 * `largest`) entries, ties to the lowest index, written as ascending int32 indices [n_rows, k]. */
int kvc_select(int32_t dtype, int32_t device, const void* scores, int64_t n_rows, int32_t n,
               int32_t k, int32_t largest, int32_t* idx_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SnapKV observation-window vote on the tensor cores (tcgen05 + TMEM) — OPT-IN EXTENSION.
 * The reference's snapkv_lite ranks keys by inverted L2 norm (snapkv_lite.py:93-100: no queries, no
 * q.K^T); this entry computes the vote the method is named after (reference
 * docs/logsAndBugs/SnapKV_Feasibility_Analysis.md:29-62):
 *   votes[b,h,j] = sum_{g<G} sum_{i<W} softmax_j( Q[b,h*G+g,i,:] . K[b,h,j,:] / sqrt(D) ),  j < S - W,
 * the softmax running over all S keys with the causal mask inside the window.  16-bit caches only;
 * head_dim*2/16 in {8,10,16}; G*W <= 128.  Feed votes to kvc_compress_layers as KVC_SCORE_GIVEN_SCORE. */
typedef struct kvc_vote_layer {
    const void* k_in;   /* [B,H,S,D] keys */
    const void* q_obs;  /* [B,H*G,W,D] queries of the last W positions, last dim dense */
    void* votes_out;    /* [B,H,S-W] votes, cache dtype, dense */
    int64_t k_stride_b, k_stride_h, k_stride_s; /* elements */
    int64_t q_stride_b, q_stride_h, q_stride_s; /* elements */
    int32_t seq_len;    /* S */
    int32_t reserved;
    /* Optional [B, H*G, W] fp32, dense: lse[b,hq,i] = log(sum_j exp(q_i . k_j / sqrt(D))) over the keys query i sees
     * (all S keys, causal inside the window) — the log-sum-exp an attention forward over these queries returns.  With
     * it the kernel skips its first pass (the softmax denominators) and reads K once instead of twice.  NULL: two passes. */
    const float* lse;
} kvc_vote_layer;
int kvc_snapkv_vote(const kvc_shape* shape, int32_t n_layers, const kvc_vote_layer* layers, int32_t group,
                    int32_t window, void* stream);
/* The vote, then snapkv_lite.py:104-150 in the SAME launch: the CTA that produced a (b,h)'s votes pools them
 * (avg_pool1d(plans[l].pool_kernel)), keeps the plans[l].k_sel highest of the prefix [0, S - W) plus the last
 * plans[l].tail rows, and gathers K and V into io[l].k_out / v_out.  plans[l]: sink 0, sel [0, S - W), score
 * KVC_SCORE_GIVEN_SCORE; io[l].k_in / strides must be layers[l]'s keys; layers[l].votes_out is still written (the votes
 * pass through it in the cache dtype).  KVC_ERR_TOO_LARGE when the prefix keys + kept indices exceed the shared
 * memory of the key ring (~70-90K rows, by head_dim): run kvc_snapkv_vote + kvc_compress_layers_ws instead. */
int kvc_snapkv_vote_compress(const kvc_shape* shape, int32_t n_layers, const kvc_vote_layer* layers,
                             const kvc_layer_plan* plans, const kvc_layer_io* io, int32_t group, int32_t window,
                             void* stream);

/* ---------------------------------------------------------------------------------------------
 * Slab cache: the container step on both sides of the compress call (SURVEY.md §8f rank 1).
 *
 * The reference's decode loop re-allocates and copies the whole cache twice per step: HF
 * DynamicLayer.update appends with torch.cat (transformers cache_utils.py:119-120), the compress
 * function gathers into fresh tensors, and to_dynamic_cache (reference utils.py:12-27) rebuilds
 * the container.  Here one layer's K and V live in pre-allocated [B, H, capacity, D] slabs with
 * dense rows, next to a [B, H, capacity] array of key norms in the cache dtype (exactly what
 * torch.norm(K, p=2, dim=-1) returns for those rows: fp32 sum of squares, one rounding).
 *
 *   kvc_slab_append    copies n_new rows per (b,h) to rows [cur_len, cur_len + n_new) of the slabs
 *                      and records their key norms — replaces the torch.cat of cache.update.
 *   kvc_slab_compress  applies a keep-plan IN PLACE: scores come from the stored norms (K is not
 *                      re-read), kept rows slide down to rows [0, C) of the same slabs (rows whose
 *                      position does not change are not touched), norms slide with them.  Same kept
 *                      set and same bytes as kvc_compress_layers on the same cache.
 */
typedef struct kvc_slab_layer {
    void* k;      /* [B,H,capacity,D] keys,   rows dense */
    void* v;      /* [B,H,capacity,D] values, rows dense */
    void* norms;  /* [B,H,capacity] key norms, cache dtype */
    int64_t k_stride_b, k_stride_h; /* elements */
    int64_t v_stride_b, v_stride_h; /* elements */
    int64_t n_stride_b, n_stride_h; /* elements */
} kvc_slab_layer;

typedef struct kvc_slab_new_rows {
    const void* k_new; /* [B,H,n_new,D] rows to append, last dim dense */
    const void* v_new;
    int64_t k_stride_b, k_stride_h, k_stride_s; /* elements */
    int64_t v_stride_b, v_stride_h, v_stride_s; /* elements */
    int32_t cur_len;   /* rows already valid in this layer's slab */
    int32_t n_new;     /* rows to append */
} kvc_slab_new_rows;

/* Append rows to n_layers slabs in one launch (any row width that is a multiple of 16 bytes, up to 2 KB). */
int kvc_slab_append(const kvc_shape* shape, int32_t n_layers, const kvc_slab_layer* slabs,
                    const kvc_slab_new_rows* rows, void* stream);

/* Compact n_layers slabs in place in one launch.  plans[l].seq_len = rows currently valid.
 * idx_out[l] (optional, may be NULL / hold NULLs): [B,H,C] kept absolute rows; idx_in[l]: GIVEN_INDEX rows, which
 * must be STRICTLY ASCENDING inside [sel_lo, sel_hi) per (b,h): kept rows only ever move towards row 0, which is what
 * makes the compaction safe in place (values outside [0, seq_len) are clamped, never dereferenced).
 * KVC_SCORE_GIVEN_SCORE: idx_in[l] carries, instead, the [B,H,sel_hi-sel_lo] scores of the region's rows (cache dtype,
 * dense; e.g. kvc_snapkv_vote's output) — pooled with plans[l].pool_kernel, the k_sel highest kept. */
int kvc_slab_compress(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                      const kvc_slab_layer* slabs, int32_t* const* idx_out, const int32_t* const* idx_in,
                      void* workspace, int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * H2O attention-score bookkeeping (reference h2o_attention.py:78-213) on the device.
 *
 * Per layer, per batch entry b, query head h and key j < key_len, with fp32 arithmetic and a rounding to the
 * attention dtype at exactly the points where the reference's torch expressions round:
 *   mass             = round( sum_q fp32(attn[b,h,q,j]) )               (attn.sum(dim=2))
 *   acc[b,h,j]       = round( fp32(round(fp32(acc[b,h,j]) * decay)) + fp32(mass) )   j <  prev_len
 *   acc[b,h,j]       = mass                                                          j >= prev_len
 *   score_out[b, j - score_lo] = round( sum_h fp32(acc[b,h,j]) ),  score_lo <= j < score_hi
 * prev_len < 0 or prev_len > key_len: every acc entry starts from zero (the reference's reset when the cache
 * shrank).  The query sum runs over fixed, contiguous query blocks in ascending order, the blocks then added in
 * ascending order; with n_query = 1 mass is attn itself.  The head sum runs in ascending h.  attn == NULL: acc is
 * neither read for an update nor written, only score_out is produced from it.  score_out may be NULL (or
 * score_lo == score_hi) when no score row is wanted.  One launch covers every layer (KVC_MAX_LAYERS_PER_LAUNCH
 * chunks); feed score_out to kvc_compress_layers / kvc_slab_compress as KVC_SCORE_GIVEN_SCORE_SHARED. */
typedef struct kvc_h2o_layer {
    const void* attn;        /* [B, Hq, n_query, key_len] attention probabilities, last dim dense; NULL: re-score only */
    int64_t a_stride_b, a_stride_h, a_stride_q; /* elements */
    void* acc;               /* [B, Hq, >= key_len] accumulators, attention dtype, last dim dense */
    int64_t acc_stride_b, acc_stride_h;         /* elements */
    void* score_out;         /* optional [B, score_hi - score_lo], dense: sum over heads of the updated acc */
    int32_t n_query, key_len;
    int32_t prev_len;        /* valid acc entries before the update; < 0 or > key_len: start from zero */
    int32_t score_lo, score_hi;
    int32_t reserved;
} kvc_h2o_layer;
/* shape: batch = B, heads = Hq (query heads), dtype = the attention dtype, device; head_dim is not used. */
int kvc_h2o_accumulate(const kvc_shape* shape, int32_t n_layers, const kvc_h2o_layer* layers, float decay,
                       void* stream);

/* The same update with the attention probabilities rebuilt from the post-RoPE queries and the cached keys, so that the
 * model can run any attention backend (SDPA, flash) and never materialise [B, Hq, n_query, key_len] probabilities.
 * Per layer, batch entry b, query head h (KV head h / G, G = group), query t < T = n_query and key j < key_len:
 *   s[t,j]   = scaling * sum_d fp32(q[b,h,t,d]) * fp32(k[b,h/G,j,d])    fp32, one fmaf chain in ascending d
 *   vis(t,j) = mask[b,t,j] (nonzero = visible) if mask != NULL, else j <= key_len - T + t (causal: the queries are the
 *              last T positions)
 *   lse[t]   = log sum_{vis} exp(s[t,j])                                  fp32, max-shifted
 *   attn     = round(exp(s[t,j] - lse[t])) where visible, 0 elsewhere (a query with no visible key adds 0)
 * then exactly kvc_h2o_accumulate's update with that attn (the query sum in ascending t).  This is HF eager attention's
 * softmax(..., dtype=float32).to(query.dtype) of fp32 logits; eager attention in a 16-bit model rounds the logits to
 * the model dtype before its softmax, SDPA and flash do not.  Two launches per KVC_MAX_LAYERS_PER_LAUNCH layers: the
 * per-split (max, sum exp) partials go to the workspace, the update combines them in a fixed order.  Every split and
 * tile depends only on (key_len, n_query, group, head_dim, dtype): a layer's bits do not depend on B, the other layers
 * of the call or the device.  KVC_ERR_INVALID_ARG: n_query > key_len without a mask, group < 1, a score region outside
 * [0, key_len], NULL acc / q / k, a workspace smaller than kvc_h2o_qk_workspace_bytes.  KVC_ERR_UNSUPPORTED: a dtype
 * other than f32 / f16 / bf16, head_dim * e not a multiple of 16 or above 512 bytes (D <= 256 in 16-bit, D <= 128 in
 * fp32), K rows not 16-byte aligned. */
typedef struct kvc_h2o_qk_layer {
    const void* q;          /* [B, Hq, n_query, D] queries, last dim dense */
    int64_t q_stride_b, q_stride_h, q_stride_t; /* elements */
    const void* k;          /* [B, Hkv, key_len, D] keys, rows 16-byte aligned (a slab view qualifies) */
    int64_t k_stride_b, k_stride_h, k_stride_s; /* elements */
    const uint8_t* mask;    /* optional [B, n_query, key_len] bool, last dim dense; NULL: the causal rule */
    int64_t m_stride_b, m_stride_t;             /* elements (bytes) */
    void* acc;              /* [B, Hq, >= key_len] accumulators, as kvc_h2o_layer */
    int64_t acc_stride_b, acc_stride_h;         /* elements */
    void* score_out;        /* optional [B, score_hi - score_lo], dense */
    float scaling;
    int32_t n_query, key_len, prev_len, score_lo, score_hi;
} kvc_h2o_qk_layer;
/* shape: batch = B, heads = Hkv (KV heads), head_dim = D, dtype of q, K and acc, device; group = G = Hq / Hkv.
 * Bytes of device workspace kvc_h2o_accumulate_qk needs for these layers (the sum over the layers; 0 when there is
 * nothing to do); -1 when the arguments are invalid. */
int64_t kvc_h2o_qk_workspace_bytes(const kvc_shape* shape, int32_t group, int32_t n_layers,
                                   const kvc_h2o_qk_layer* layers);
int kvc_h2o_accumulate_qk(const kvc_shape* shape, int32_t group, int32_t n_layers, const kvc_h2o_qk_layer* layers,
                          float decay, void* workspace, int64_t workspace_bytes, void* stream);

/* The same update with the logits on the 5th-generation tensor cores, for prompt-sized n_query (opt-in: its bits differ
 * from kvc_h2o_accumulate_qk's).  The same records and the same visibility, prev_len and score rules; per layer:
 *   a[t,j]   = sum_d q[b,h,t,d] * k[b,h/G,j,d]    tcgen05.mma kind::f16: 16-bit operands, fp32 accumulation in the
 *              tensor core's order
 *   c        = fp32(scaling * log2(e))
 *   lse2[t]  = m + log2(sum_{vis} exp2(fma(a[t,j], c, -m))),  m = max_{vis} a[t,j] * c   (online over 128-key tiles in
 *              ascending order; +inf for a query that sees no key)
 *   attn     = round(exp2(fma(a[t,j], c, -lse2[t]))) where visible, 0 elsewhere   (exp2: ex2.approx.ftz.f32)
 * then exactly kvc_h2o_accumulate_qk's tail: one __fadd_rn chain over ascending t per (head, key), h2o_update_acc, and
 * the score row as the sum of the updated accumulators in ascending h (a kvc_h2o_accumulate launch with attn = NULL).
 * Only the logits and the exponential differ from the CUDA-core form; against fp64 logits -> softmax -> round the
 * accumulators agree within 2 ulps of the attention dtype.  Launches per 32 layers: a statistics pass, a column-sum
 * pass, and the score-row launch when a layer asks for a score row.  Every tile depends only on (key_len, n_query,
 * group, head_dim, dtype): a layer's bits do not depend on B, the other layers of the call or the device.  The entry
 * point allocates nothing and never synchronises.  Refusals, before any CUDA call: everything kvc_h2o_accumulate_qk
 * refuses; KVC_ERR_UNSUPPORTED for fp32, head_dim outside {64, 80, 128}, group > 128, and q or K whose base or
 * b / h / t strides are not 16-byte multiples (a tensor map cannot describe them). */
int64_t kvc_h2o_qk_tc_workspace_bytes(const kvc_shape* shape, int32_t group, int32_t n_layers,
                                      const kvc_h2o_qk_layer* layers);
int kvc_h2o_accumulate_qk_tc(const kvc_shape* shape, int32_t group, int32_t n_layers, const kvc_h2o_qk_layer* layers,
                             float decay, void* workspace, int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Per-row state that moves with the kept rows (cumulative H2O: the accumulators of kvc_h2o_accumulate keep describing
 * the token they were accumulated for across a compaction).  Per layer, batch entry b, KV head h, g < group and output
 * row i < C = sink + k_sel + tail, with src(i) the source row of output row i for KV head h:
 *   acc'[b, h*group+g, i] = acc[b, h*group+g, src(i)]   if src(i) < min(prev_len, seq_len)
 *                         = 0                           otherwise
 * The copy is bit-exact, in place, and runs in the same launch as the compaction / gather of K and V (the CTA that
 * moves a (layer, b, h)'s rows moves its `group` accumulator rows).  Entries at and past C are unspecified afterwards.
 * carry == NULL, or acc == NULL on every layer, is exactly kvc_slab_compress / kvc_compress_layers_ws.
 * KVC_ERR_INVALID_ARG, before any CUDA call, on a layer with a non-NULL acc: group < 1, prev_len < 0, or acc rows not
 * aligned to the element size (4 bytes for fp32, 2 for 16-bit). */
typedef struct kvc_carry_layer {
    void* acc;                          /* [B, H*group, >= seq_len] per-row state, dtype = shape->dtype, last dim dense;
                                           NULL: nothing to carry for this layer */
    int64_t acc_stride_b, acc_stride_h; /* elements */
    int32_t group;                      /* rows of acc per KV head (Hq / Hkv); KV head h owns acc heads [h*group, (h+1)*group) */
    int32_t prev_len;                   /* valid entries before the compaction (clamped to seq_len) */
} kvc_carry_layer;
/* kvc_slab_compress with carry[l] for layer l (carry may be NULL). */
int kvc_slab_compress_carry(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                            const kvc_slab_layer* slabs, int32_t* const* idx_out, const int32_t* const* idx_in,
                            const kvc_carry_layer* carry, void* workspace, int64_t workspace_bytes, void* stream);
/* kvc_compress_layers_ws with carry[l] for layer l (carry may be NULL); K and V are still written out of place, only
 * acc is compacted in place. */
int kvc_compress_layers_carry(const kvc_shape* shape, int32_t n_layers, const kvc_layer_plan* plans,
                              const kvc_layer_io* io, const kvc_carry_layer* carry, void* workspace,
                              int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KVC_H_ */
