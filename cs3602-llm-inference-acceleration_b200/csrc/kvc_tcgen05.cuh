// kvc_tcgen05.cuh — 5th-generation tensor-core primitives (tcgen05 + TMEM), UMMA shared-memory descriptors, TMA
// tensor-map loads and the host-side tensor-map encoder, shared by every kernel that runs on the tensor cores (the
// SnapKV vote, kvc_vote.cuh; the tensor-core H2O query update, kvc_h2o_tc.cuh).
#pragma once
#include <cuda.h>  // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)
#include <cuda_runtime.h>
#include <stdint.h>

namespace kvc {

// ---------------------------------------------------------------- tcgen05 wrappers
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem] . B[smem]^T, bf16/fp16 inputs, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrive once every previously issued tcgen05.mma of this thread has completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (lane = TMEM lane base + laneid).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 32 lanes x 16 consecutive fp32 columns, asynchronous: tmem_ld_wait() before the registers are read.
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, no swizzle: 8x16-byte core matrices; LBO = step between the two 16-byte K chunks of one
// K=16 instruction, SBO = step between 8-row groups (cute/arch/mma_sm100_desc.hpp, SmemDescriptor).
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
    return d;                // base_offset 0, lbo_mode 0, layout_type 0 = SWIZZLE_NONE
}
// Instruction descriptor (cute/arch/mma_sm100_desc.hpp, InstrDescriptor): fp32 accumulate, K-major A and B.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int fmt /*0 f16, 1 bf16*/, int m, int n) {
    return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// K-major, 32-byte swizzle: rows 32 B apart inside an 8-row atom, atoms 256 B apart (SBO), LBO = 16 B.
__device__ __forceinline__ uint64_t umma_smem_desc_sw32(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(256 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)6 << 61;  // layout type SWIZZLE_32B
    return d;
}
// K-major, 128-byte swizzle: rows 128 B apart inside an 8-row atom, atoms 1024 B apart (SBO), LBO = 16 B.
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)1 << 16;           // leading byte offset 16 B (unused by swizzled K-major layouts)
    d |= (uint64_t)(1024 >> 4) << 32;  // stride byte offset: 8 rows x 128 B
    d |= (uint64_t)1 << 46;           // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;           // layout type SWIZZLE_128B
    return d;
}

__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tma_load_4d(uint32_t dst_smem, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                            uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(dst_smem), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
        : "memory");
}

// ---------------------------------------------------------------- host: tensor maps
// cuTensorMapEncodeTiled through the runtime (the library links cudart statically and never links libcuda).
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static inline EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}

// The maps of a 16-bit [d3, d2, d1, D] tensor (dims / byte strides innermost first) read as K-major UMMA row tiles:
// `main` covers the first 64 elements of a row (box (64, box1, box2, 1), 128-byte swizzle), `tail` the last 16 when
// D % 64 == 16 (box (16, box1, box2, 1), 32-byte swizzle).  Elements outside the tensor are zero-filled.  False when
// a tensor map cannot describe the tensor (alignment, strides).
static inline bool encode_row_maps(EncodeTiledFn encode, CUtensorMap* main, CUtensorMap* tail, bool bf16, const void* base,
                                   const cuuint64_t (&dims)[4], const cuuint64_t (&strides)[3], int box1, int box2) {
    const CUtensorMapDataType t = bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    const cuuint32_t box[4] = {64, (cuuint32_t)box1, (cuuint32_t)box2, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    if (encode(main, t, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return false;
    if (dims[0] % 64 == 0) return true;
    const cuuint32_t box_tail[4] = {16, (cuuint32_t)box1, (cuuint32_t)box2, 1};
    return encode(tail, t, 4, const_cast<void*>(base), dims, strides, box_tail, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) ==
           CUDA_SUCCESS;
}

}  // namespace kvc
