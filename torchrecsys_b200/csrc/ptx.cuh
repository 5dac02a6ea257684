// ptx.cuh -- the inline-PTX primitives the kernels share, each defined once: shared-memory addresses, the global
// timer, L2 prefetch and cache policies, cp.async, scoped relaxed / acquire memory operations and fences, mbarriers
// and the non-tensor bulk copy.  tc.cuh adds what is specific to the tensor cores.
#pragma once
#include <stdint.h>

namespace trs {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)::"memory");
    return t;
}

__device__ __forceinline__ void prefetch_l2(const void* p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// ---- L2 cache policies ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void st_v4_hint(float* p, const float4& v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w), "l"(pol)
                 : "memory");
}

// ---- cp.async: 16-byte copies global -> shared, visible to the issuing thread after its wait_group ---------------
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async16_hint(void* smem, const void* gmem, uint64_t pol) {
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(smem_u32(smem)), "l"(gmem),
                 "l"(pol)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// at most n copy groups still pending (n must be a compile-time constant after inlining and unrolling)
__device__ __forceinline__ void cp_async_wait(int n) {
    switch (n) {
        case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
        case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
        case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
        case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
        case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
        case 5: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
        case 6: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
        default: asm volatile("cp.async.wait_group 7;" ::: "memory"); break;
    }
}

// ---- scoped memory operations on a 32-bit counter in global memory -----------------------------------------------
__device__ __forceinline__ unsigned ld_relaxed_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_relaxed_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// *p += 1
__device__ __forceinline__ void red_relaxed_gpu(unsigned* p) {
    asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(p) : "memory");
}
__device__ __forceinline__ void red_relaxed_sys(unsigned* p) {
    asm volatile("red.relaxed.sys.global.add.u32 [%0], 1;" ::"l"(p) : "memory");
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void fence_acq_rel_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }

// ---- mbarrier (shared::cta) ------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// Non-suspending poll: try_wait may park the warp for a hardware time slice when the phase is not complete at
// the first look; on a hand-off that completes within a few hundred cycles that slice is the critical path.
__device__ __forceinline__ void mbar_wait_spin(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}

// ---- bulk async copy (TMA engine, no tensor map): `bytes` (a multiple of 16) global -> shared, completing on bar --
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

}  // namespace trs
