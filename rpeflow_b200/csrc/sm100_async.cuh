// sm100_async.cuh — the sm_100a asynchronous-unit PTX used by the TMA and tensor-core kernels, one definition each:
// mbarriers, proxy fences and named barriers, TMA and bulk copies, tcgen05 (TMEM allocation, fences, kind::tf32 MMA,
// commit, TMEM loads), and the shared-memory operand layouts the MMAs read.
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>

#include "common.cuh"

namespace b200 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// makes the initialised barriers visible to the other threads and to the async proxy (TMA, tcgen05.commit)
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a protocol bug traps (launch error) instead of hanging the device
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    bool done = false;
    for (uint32_t spin = 0; !done; ++spin) {
        done = mbar_try(bar, parity);
        if (spin > (1u << 26)) __trap();
    }
}

// generic-proxy writes to shared memory -> visible to the async proxy (TMA, tcgen05.mma)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// named barrier ID over the first N threads that reach it (N a multiple of 32)
template <int ID, int N>
__device__ __forceinline__ void named_bar_sync() { asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(N) : "memory"); }

// ---- TMA and bulk copies -------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar) : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
// contiguous global -> shared copy of `bytes` (a multiple of 16), completing as transaction bytes on `bar`
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
static inline PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = []() -> PFN_cuTensorMapEncodeTiled_v12000 {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }();
    return fn;
}

// ---- tcgen05: tensor memory, fences, MMA -----------------------------------------------------------------------------
// one whole warp: allocates `cols` TMEM columns, writes their address to shared `slot`, and gives up the allocation permit
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(cols) : "memory");
}
// order tcgen05 operations before / after a thread synchronisation (barrier or mbarrier wait)
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor: K-major operand, rows of 128 bytes, 128-byte swizzle, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3fffu)          // start address
           | ((uint64_t)(1024u >> 4) << 32)           // stride byte offset (between 8-row groups); leading offset unused
           | ((uint64_t)1 << 46)                      // descriptor version 1 (sm_100)
           | ((uint64_t)2 << 61);                     // SWIZZLE_128B
}
// byte offset of 16-byte chunk q of row r in that layout
__host__ __device__ __forceinline__ uint32_t sw128(uint32_t r, uint32_t q) { return r * 128u + ((q ^ (r & 7u)) << 4); }
// K-major operand, rows of 64 bytes, 64-byte swizzle (16-byte chunk index ^= address bits 7-8), 8-row groups 512 bytes apart
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)(512u >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)4 << 61);
}
__host__ __device__ __forceinline__ uint32_t sw64(uint32_t r, uint32_t q) { return r * 64u + ((q ^ ((r >> 1) & 3u)) << 4); }
// instruction descriptor: D = F32, A = B = TF32, both K-major, dense
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// the TF32 part of v (3xTF32 splits v into tf32_hi(v) + the rest)
__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xffffe000u); }

__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on `bar` once every MMA this thread issued before it has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// ---- tcgen05: TMEM -> registers, 32 lanes x 32 bits, 8 / 16 / 32 columns; the registers are valid after tmem_ld_wait()
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

}  // namespace b200
