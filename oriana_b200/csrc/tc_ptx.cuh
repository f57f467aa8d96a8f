// tc_ptx.cuh -- inline-PTX wrappers for the sm_100a tensor path: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (TMEM alloc / ld / st / mma / commit) and the shared-memory / instruction descriptors of
// kind::tf32 MMAs.  Everything here is hand-written for this repo; the descriptor bit layouts follow the
// PTX ISA tables for tcgen05 (matrix descriptor: start address [0,14), LBO [16,30), SBO [32,46),
// version [46,48) = 1, swizzle mode [61,64); instruction descriptor: D format [4,6), A/B format [7,10) /
// [10,13), A/B major [15]/[16], N>>3 [17,23), M>>4 [24,29)).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a launch failure, never as a hung GPU.
#ifndef ORI_MBAR_TIMEOUT_CYCLES
#define ORI_MBAR_TIMEOUT_CYCLES 6000000000ll
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int tag = 0) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > ORI_MBAR_TIMEOUT_CYCLES) {
            printf("oriana_b200: mbarrier timeout tag=%d block=%d thread=%d parity=%u\n", tag, blockIdx.x, threadIdx.x, parity);
            __trap();
        }
    }
}

// one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// Wait on two barriers whose completion latencies should overlap (both try_waits are in flight together).
__device__ __forceinline__ void mbar_wait2(uint64_t* bar_a, uint32_t par_a, uint64_t* bar_b, uint32_t par_b, int tag = 0) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q, [%3], %4;\n\t"
        "and.pred p, p, q;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar_a)), "r"(par_a), "r"(smem_u32(bar_b)), "r"(par_b)
        : "memory");
    if (ok) return;
    mbar_wait(bar_a, par_a, tag);
    mbar_wait(bar_b, par_b, tag + 1);
}

// ---- TMA ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

// L2 eviction-priority policies (createpolicy.fractional.L2::evict_*, fraction 1.0), as precomputed descriptors
constexpr uint64_t L2_EVICT_FIRST = 0x12F0000000000000ull;   // streamed once: the count matrix
constexpr uint64_t L2_EVICT_LAST = 0x14F0000000000000ull;    // re-read by every CTA: the factor operands
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                                 uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
// CTA-pair form: executed by both CTAs of a pair, each filling its own shared memory; the transaction bytes are
// credited to the mbarrier of the pair's leader (even rank): peer bit of the barrier address cleared
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                                 uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}

// ---- clusters ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the mbarrier at the same shared-memory offset in CTA `rank` of the cluster (default .release.cta: a
// cluster-scope release costs a full memory barrier per arrive; what the leader reads afterwards is TMEM, ordered by
// tcgen05.wait::st + tcgen05.fence::before_thread_sync on this side and tcgen05.fence::after_thread_sync on the other)
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(smem_u32(bar)), "r"(rank) : "memory");
}

// ---- TMEM ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // the same warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {   // the same warp of both CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {                          // one thread
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// CTA pair: arrive on the barrier at this offset in both CTAs when every MMA issued so far has completed
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {                     // one thread of the leader
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

// 32 lanes x 32 bit, 16 consecutive columns per thread (thread l of warp w <-> TMEM lane 32*(w%4)+l)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {     // 8 consecutive columns per thread
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
        : "memory");
}

// ---- descriptors ----------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, 128-byte swizzle.  K-major operand: rows of 128 B (32 tf32), 8-row groups
// `sbo` bytes apart (LBO unused).  MN-major operand: 128 B (32 elements) contiguous along M/N, 8 K-rows per
// swizzle atom, atoms `sbo` bytes apart along K and `lbo` bytes apart along M/N.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
    d |= 1ull << 46;   // descriptor version (Blackwell)
    d |= 2ull << 61;   // SWIZZLE_128B
    return d;
}
// kind::tf32, fp32 accumulate
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N, bool a_mn_major, bool b_mn_major) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// kind::f16 with bf16 operands, fp32 accumulate (A / B format 1 = BF16; K = 16 elements = 32 bytes per instruction)
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void mma_tf32_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}

// CTA pair, M = 256: rows 0-127 are CTA 0's TMEM lanes, rows 128-255 CTA 1's; each CTA's shared memory holds
// half of the N rows of B at the descriptor's offset
__device__ __forceinline__ void mma_tf32_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}

// bf16 operands, CTA pair: A from TMEM (two consecutive K elements per 32-bit cell, lower index in the low half), B from smem
__device__ __forceinline__ void mma_bf16_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}
// {lo, hi} -> one 32-bit word of two bf16 (round to nearest even), `lo` in the low half
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

__device__ __forceinline__ float to_tf32_rna(float x) {   // round to nearest (ties away), low 13 bits cleared
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// ---- host side: tensor maps -------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// float32 row-major [rows x cols] with row stride ld (elements); box = box_cols x box_rows, 128-byte swizzle
// (box_cols * 4 must be 128).  Out-of-bounds elements are filled with zeros.
inline bool make_tmap_f32(CUtensorMap* map, const float* base, uint64_t rows, uint64_t cols, uint64_t ld,
                          uint32_t box_cols, uint32_t box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * sizeof(float)};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace tc
