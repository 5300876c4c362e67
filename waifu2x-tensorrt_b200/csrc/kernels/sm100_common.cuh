// PTX wrappers for the sm_100a programming model used by the convolution kernels: mbarrier, TMA (cp.async.bulk.tensor)
// loads/stores, tcgen05 (MMA issue, commit, TMEM alloc/ld, fences), UMMA shared-memory descriptors.
// Instruction strings and descriptor bit layouts follow the CUTLASS/CuTe sm100 headers (cute/arch/mma_sm100_desc.hpp,
// copy_sm90_tma.hpp, tmem_allocator_sm100.hpp, cutlass/arch/barrier.h) vendored in the image.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace w2x {
namespace sm100 {

__device__ __forceinline__ uint32_t smemU32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ----
__device__ __forceinline__ void mbarInit(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbarInitFence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbarExpectTx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbarArrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbarWait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}

// non-blocking probe of a phase (mbarrier.test_wait never suspends): lets the MMA issuer look at the NEXT tile's barriers while
// the current tile's MMAs are still being queued, so that the blocking wait at the top of the next tile normally falls through
__device__ __forceinline__ uint32_t mbarTest(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done;
}

// spin on test_wait: for short hand-offs between two roles that are nearly in step (try_wait may park the thread and its wake-up
// latency then dominates the hand-off)
__device__ __forceinline__ void mbarSpin(uint32_t bar, uint32_t parity) {
    while (!mbarTest(bar, parity)) {}
}

// ---- TMA ----
__device__ __forceinline__ void tmaPrefetchDesc(const CUtensorMap* tm) { asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory"); }
__device__ __forceinline__ void tmaLoad5d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(dst),
        "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void tmaLoad3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
                 "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tmaLoad2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
                 "l"(tm), "r"(bar), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tmaStore5d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2, int c3, int c4) {
    asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(tm), "r"(src), "r"(c0),
                 "r"(c1), "r"(c2), "r"(c3), "r"(c4)
                 : "memory");
}
__device__ __forceinline__ void bulkCommit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most n of this thread's bulk groups still READ their shared-memory source
__device__ __forceinline__ void bulkWaitRead(int n) {
    if (n <= 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    else if (n == 1) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
    else asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory");
}
__device__ __forceinline__ void bulkWaitAll() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy smem writes -> visible to the async proxy (TMA store)
__device__ __forceinline__ void fenceProxyAsync() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void namedBarSync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

// ---- tcgen05 ----
__device__ __forceinline__ void tcFenceBefore() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcFenceAfter() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcCommit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmemAlloc(uint32_t slotSmemAddr, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slotSmemAddr), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmemDealloc(uint32_t tmemBase, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmemBase), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (fp16/bf16 inputs, fp32 accumulate), issued by ONE thread
__device__ __forceinline__ void umma(uint32_t tmemD, uint64_t descA, uint64_t descB, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmemD),
        "l"(descA), "l"(descB), "r"(idesc), "r"(accumulate)
        : "memory");
}
// same, with the descriptors given as (lo, hi) 32-bit halves so the issue loop only does 32-bit adds on `lo`
__device__ __forceinline__ void ummaLoHi(uint32_t tmemD, uint32_t aLo, uint32_t aHi, uint32_t bLo, uint32_t bHi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
        "}" ::"r"(tmemD),
        "r"(aLo), "r"(aHi), "r"(bLo), "r"(bHi), "r"(idesc), "r"(accumulate)
        : "memory");
}
// the same with kind::tf32 (fp32 operands in shared memory, TF32 multiply, fp32 accumulate): one K step is 8 elements = 32 bytes,
// like the 16 fp16 elements of kind::f16, so the descriptors advance exactly as for fp16
__device__ __forceinline__ void ummaTf32LoHi(uint32_t tmemD, uint32_t aLo, uint32_t aHi, uint32_t bLo, uint32_t bHi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t"
        "}" ::"r"(tmemD),
        "r"(aLo), "r"(aHi), "r"(bLo), "r"(bHi), "r"(idesc), "r"(accumulate)
        : "memory");
}
// one elected lane of a fully converged warp
__device__ __forceinline__ bool electOne() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint32_t descLo(uint32_t smemAddr) { return ((smemAddr >> 4) & 0x3FFFu) | (1u << 16); }
__device__ __forceinline__ void tmemLd32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmemLd16(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmemLdWait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major swizzled operand descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30) (unused for swizzled
// K-major), SBO>>4 [32,46), version=1 [46,48), base_offset [49,52) = 0, layout type [61,64) (2 = 128B swizzle, 4 = 64B).
// Measured on B200 (w2x_probe_umma, profiles/r01_umma_probe.txt): the swizzle XOR is taken from the ABSOLUTE shared-memory
// address bits, so a descriptor may start at any 128-byte row of a TMA-written swizzled tile and use any SBO with
// base_offset = 0 -- which is what lets one loaded input patch serve all nine 3x3 taps.
__device__ __forceinline__ uint32_t descHi(uint32_t sboBytes, uint32_t layoutType) {
    return (sboBytes >> 4) | (1u << 14) | (layoutType << 29);
}
__device__ __forceinline__ uint64_t makeDesc(uint32_t smemAddr, uint32_t hi) {
    return (uint64_t)((smemAddr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)hi << 32);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D=F32 [4,6), A=B=F16 (0), K-major both, N>>3 [17,23), M>>4 [24,29)
__host__ __device__ __forceinline__ uint32_t instrDescF16(int m, int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// the same with A=B=TF32 (format 2 in bits [7,10) and [10,13))
__host__ __device__ __forceinline__ uint32_t instrDescTf32(int m, int n) {
    return instrDescF16(m, n) | (2u << 7) | (2u << 10);
}

__device__ __forceinline__ uint4 ldsV4(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void stsV4(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

}  // namespace sm100
}  // namespace w2x
