// tc.cuh -- sm_100a tensor-core plumbing written as inline PTX: TMA tensor loads (cp.async.bulk.tensor),
// tcgen05 (alloc / mma / commit / ld / st) and the shared-memory / instruction descriptors of
// tcgen05.mma.kind::f16; the mbarriers they complete on are in ptx.cuh.  Used by gemm.cu (MLP tower) and
// topk.cu (predict).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "ptx.cuh"

namespace trs {
namespace tc {

// ---- TMA ----------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
// 2-D tile load: coordinates are (innermost, outer) element indices; completion on `bar`.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

// ---- tcgen05 --------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_out, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_out)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrive when every tcgen05.mma issued so far by this thread has completed
// D[tmem] (+)= A[tmem] * B[smem]^T: the A tile sits in tensor memory (row m in lane m, K elements packed two
// bf16 per 32-bit column: element k in column k / 2, low half first), so the MMA reads only B from shared memory.
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// registers -> TMEM: this warp's 32 lanes x 8 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// One lane of a converged warp.  Issuing tcgen05.mma / commit under this predicate (instead of `lane == 0`)
// keeps the surrounding control flow warp-uniform, so descriptors and loop counters stay in uniform registers
// and the compiler does not wrap every UTCHMMA in a per-lane election loop.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// TMEM -> registers: this warp's 32 lanes (rows) x 32 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- descriptors --------------------------------------------------------------------------------
// Shared-memory matrix descriptor of a K-major bf16 tile stored as rows of 64 elements (128 bytes)
// with the 128-byte swizzle TMA applies (tile base 1024-byte aligned): 8-row groups are 1024 bytes
// apart (stride byte offset), the leading byte offset is unused for a single swizzle atom along K.
// Bits: [0,14) address>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version = 1, [61,64) layout = 2
// (SWIZZLE_128B).  Advancing by k elements along K inside the atom adds k*2 bytes to the address.
__device__ __forceinline__ uint64_t smem_desc_sw128(const void* tile, int k_elem_offset) {
    const uint32_t addr = smem_u32(tile) + (uint32_t)k_elem_offset * 2u;
    uint64_t d = 0;
    d |= (uint64_t)((addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// MN-major bf16 tile: rows of 64 mn-elements (128 bytes, swizzled by TMA), one row per k.  `tile` points at
// the first k row of the slice; lbo_bytes = distance between consecutive 64-mn blocks.
__device__ __forceinline__ uint64_t smem_desc_sw128_mn(const void* tile, uint32_t lbo_bytes) {
    const uint32_t addr = smem_u32(tile);
    uint64_t d = 0;
    d |= (uint64_t)((addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// Instruction descriptor of kind::f16: D fp32 (bits 4-5 = 1), A and B bf16 (bits 7-9, 10-12 = 1), both
// K-major (bits 15, 16 = 0), N>>3 at bits 17-22, M>>4 at bits 24-28.
__host__ __device__ constexpr uint32_t idesc_bf16_f32(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

}  // namespace tc

// host side: a 2-D bf16 row-major [rows, cols] tensor map with box [box_rows, 64 cols], 128B swizzle
int make_tmap_bf16(CUtensorMap* out, const void* base, int64_t rows, int64_t cols, int64_t ld_elems, int box_rows);

}  // namespace trs
