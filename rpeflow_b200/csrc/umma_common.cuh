// umma_common.cuh — tcgen05 (5th-generation tensor core) PTX wrappers shared by corr3d_tc.cu and the PointConv kernels:
// shared-memory matrix descriptors (K-major, 128-byte swizzle), the kind::tf32 instruction descriptor, MMA issue,
// commit -> mbarrier, mbarrier wait, TMEM load.
#pragma once
#include "common.cuh"

namespace b200 {

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor: K-major operand, rows of 128 bytes, 128-byte swizzle, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3fffu)          // start address
           | ((uint64_t)(1024u >> 4) << 32)           // stride byte offset (between 8-row groups); leading offset unused
           | ((uint64_t)1 << 46)                      // descriptor version 1 (sm_100)
           | ((uint64_t)2 << 61);                     // SWIZZLE_128B
}
// instruction descriptor: D = F32, A = B = TF32, both K-major, dense
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void tc_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "TC_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra TC_DONE_%=;\n\t"
        "bra TC_WAIT_%=;\n\t"
        "TC_DONE_%=:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- SW64 operand layout, mbarrier ring and TMEM load of the second-generation PointConv (pointconv_v2.cu, pointconv_bwd.cu)
// K-major operand, rows of 64 bytes, 64-byte swizzle (16-byte chunk index ^= address bits 7-8), 8-row groups 512 bytes apart
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)(512u >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)4 << 61);
}
__device__ __forceinline__ uint32_t p2_sw64(uint32_t r, uint32_t q) { return r * 64u + ((q ^ ((r >> 1) & 3u)) << 4); }

__device__ __forceinline__ void p2_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t p2_mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    return done;
}
// bounded wait: a protocol bug traps (launch error) instead of hanging the device; the fast path is one try_wait
static __device__ __noinline__ void p2_mbar_wait_slow(uint32_t bar, uint32_t parity) {
    for (uint32_t spin = 0; !p2_mbar_try(bar, parity); ++spin)
        if (spin > (1u << 26)) __trap();
}
__device__ __forceinline__ void p2_mbar_wait(uint32_t bar, uint32_t parity) {
    if (!p2_mbar_try(bar, parity)) p2_mbar_wait_slow(bar, parity);
}
__device__ __forceinline__ void p2_tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr));
}

__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xffffe000u); }

}  // namespace b200
