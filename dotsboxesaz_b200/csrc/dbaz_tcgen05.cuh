// dbaz_tcgen05.cuh -- PTX wrappers shared by the tcgen05 kernels (dbaz_tower.cu, dbaz_trunk.cu): mbarriers with bounded
// waits, TMA / bulk copies, shared-memory matrix descriptors, tcgen05.mma / commit / ld, and the driver's tensor-map encoder.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace dbaz {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ uint64_t global_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// Every wait is bounded: a protocol bug must end in a trap (a failed launch), never in a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err, int code) {
    if (mbar_try_wait(bar, parity)) return;
    const uint64_t t0 = global_ns();
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 255u) == 0 && global_ns() - t0 > 2000000000ull) {
            if (err) atomicExch(err, code);
            __threadfence_system();
            __trap();
        }
    }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 2-D tiled TMA load: box at {c0, c1}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}
// 3-D tiled TMA load: box at {c0, c1, c2}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
                 "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
                 : "memory");
}
// plain bulk copy global -> shared (16-byte aligned, size a multiple of 16)
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                 "r"(bar)
                 : "memory");
}

// Shared-memory matrix descriptor, K-major, no swizzle ("interleave"): 8-row x 16-byte core matrices; row groups SBO
// bytes apart, the two 16-byte K halves of one K = 16 step LBO bytes apart.  With SBO = 128 rows are 16 bytes apart
// linearly, so the start may point at any row.  Bits: start >> 4 [0,14), LBO >> 4 [16,30), SBO >> 4 [32,46), descriptor
// version 1 [46,48), base offset 0, layout type 0 (no swizzle) [61,64).
// desc64(): the descriptor from a precomputed low word (start >> 4 | LBO >> 4 << 16): adding to it moves the start in 16-byte units
__device__ __forceinline__ uint64_t desc64(uint32_t lo) { return ((uint64_t)((128u >> 4) | (1u << 14)) << 32) | (uint64_t)lo; }
// The same for a K-major operand in the 128-byte swizzle TMA writes: rows of 64 bf16 (128 bytes), 8-row groups SBO = 1024
// bytes apart, layout type 2 (SWIZZLE_128B); the tile starts 1024-byte aligned, and the k-th K = 16 step of a row starts
// 32 k bytes further (the hardware applies the swizzle to the computed addresses).
__device__ __forceinline__ uint64_t desc64_sw128(uint32_t lo) {
    return ((uint64_t)((1024u >> 4) | (1u << 14) | (2u << 29)) << 32) | (uint64_t)lo;
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// Instruction descriptor of tcgen05.mma.kind::f16: D fp32, A/B bf16, both K-major, M = 128, N
__device__ __forceinline__ uint32_t umma_idesc(uint32_t n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on `bar` when every MMA issued so far by this thread has completed (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// {bf16(max(hi, 0)), bf16(max(lo, 0))}: the ReLU rides in the conversion
__device__ __forceinline__ uint32_t pack_relu_bf16(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled from the driver the runtime loaded (nullptr if unavailable)
inline EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

}  // namespace dbaz
