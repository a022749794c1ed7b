// Thin inline-PTX wrappers for the sm_100a features the conv/GEMM kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and
// the proxy / thread-sync fences that order them.  Nothing here is portable to
// other architectures on purpose.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace b200 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- mbarrier --
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// try_wait blocks in hardware until the phase completes or the suspend-time hint (ns) runs out, then reports the
// phase.  A generous hint costs no latency (completion wakes the thread at once) and keeps the waiting producer /
// MMA / epilogue warps from spending issue slots on poll loops: with the default (short) limit 18 % of the
// instructions the block-tail kernels issued were SYNCS / BRA / YIELD polls (profiles/r2_tail_opmix.txt).
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trapped launch (an error the host sees), never as
// a kernel that spins forever on the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > 8000000u) __trap();  // each failed try sleeps up to 20 us: seconds to minutes of waiting - a protocol bug, not a slow tile
    }
}

// --------------------------------------------------------------------- TMA --
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const void* tmap, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
        "[%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// TMA store of a shared-memory box (bulk-group completion) and the fences around it.
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_4d(const void* tmap, const void* src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// Wait until at most N bulk groups of this thread still READ their shared-memory source.
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// Make generic-proxy shared-memory writes visible to the async proxy (TMA) before a bulk store.
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ----------------------------------------------------------------- tcgen05 --
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {  // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t addr) {  // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "n"(kCols) : "memory");
}

// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate, single CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on an mbarrier once every previously issued tcgen05.mma has retired.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
// 32 registers per thread -> 32 lanes x 32 consecutive fp32 columns (the inverse of tmem_ld_32x32).  Asynchronous:
// tmem_st_wait() before a tcgen05.mma (after the usual fence / barrier) may read or accumulate onto them.
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]),
        "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]),
        "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 32 lanes x 16 consecutive fp32 columns -> 16 registers per thread.
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// Same wait, but tied to the destination registers of an earlier tcgen05.ld so that the compiler cannot
// move their first use above it (the load is asynchronous until this instruction).
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&r)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :
                 : "memory");
}

__device__ __forceinline__ void tmem_ld_wait32(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]),
                   "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]),
                   "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}

// Shared-memory matrix descriptor for a K-major bf16 operand tile stored as
// rows of 128 bytes under the 128-byte swizzle (what a TMA box with a 64-element
// inner dimension and CU_TENSOR_MAP_SWIZZLE_128B writes): 8-row groups are
// 1024 B apart (SBO), LBO is unused for swizzled K-major layouts, version = 1
// for sm_100, layout type 2 = SWIZZLE_128B.  Field positions follow the
// tcgen05 shared-memory descriptor format.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // start address, bits [0,14)
    d |= static_cast<uint64_t>(1) << 16;                      // leading byte offset (ignored), bits [16,30)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;              // stride byte offset, bits [32,46)
    d |= static_cast<uint64_t>(1) << 46;                      // descriptor version, bits [46,48)
    d |= static_cast<uint64_t>(2) << 61;                      // SWIZZLE_128B, bits [61,64)
    return d;
}

// Instruction descriptor for kind::f16 with bf16 A/B (both K-major), fp32 D.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t m, uint32_t n) {
    return (1u << 4)            // D format: f32
           | (1u << 7)          // A format: bf16
           | (1u << 10)         // B format: bf16
           | ((n >> 3) << 17)   // N / 8
           | ((m >> 4) << 24);  // M / 16
}

// 2^x on the SFU (MUFU.EX2), denormals flushed: the softmax numerator needs no more than bf16 accuracy
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ void prefetch_l2(const void* ptr) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr));
}

}  // namespace b200
