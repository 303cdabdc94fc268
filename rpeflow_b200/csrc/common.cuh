// common.cuh — shared host/device helpers for libb200flow.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "b200flow.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libb200flow is written for sm_100a (B200) only"
#endif

namespace b200 {

// ---- host-side error plumbing (thread-local message, reference: TORCH_CHECK -> RuntimeError) ----
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define B200_REQUIRE(cond, ...)                                  \
    do {                                                         \
        if (!(cond)) {                                           \
            ::b200::set_error(__VA_ARGS__);                      \
            return B200_EINVAL;                                  \
        }                                                        \
    } while (0)

#define B200_CUDA(call)                                          \
    do {                                                         \
        cudaError_t e_ = (call);                                 \
        if (e_ != cudaSuccess) return ::b200::cuda_fail(e_, #call); \
    } while (0)

#define B200_LAUNCH_CHECK(name)                                  \
    do {                                                         \
        cudaError_t e_ = cudaGetLastError();                     \
        if (e_ != cudaSuccess) return ::b200::cuda_fail(e_, name); \
    } while (0)

static inline cudaStream_t as_stream(b200_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
int sm_count();   // SMs of the current device (cached per device)

// ---- device helpers ----
#ifdef __CUDACC__
constexpr unsigned FULL = 0xffffffffu;

// The stated distance rule (SURVEY §8a): every product and sum rounded separately, left to right.
// __f*_rn intrinsics are never contracted into FFMA by nvcc.
__device__ __forceinline__ float sqdist3_rule(float ax, float ay, float az, float bx, float by, float bz) {
    float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}
__device__ __forceinline__ float sqdist2_rule(float ax, float ay, float bx, float by) {
    float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by);
    return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}

// ---- packed fp32x2 arithmetic (Blackwell FADD2 / FFMA2): two independent fp32 lanes per instruction ----
typedef unsigned long long u64;
__device__ __forceinline__ u64 pack2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(u64 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
// d = a*b + d on both halves (FFMA2)
__device__ __forceinline__ void fma2(u64& d, u64 a, u64 b) {
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b));
}
__device__ __forceinline__ void ffma2(float2& d, const float2& a, const float2& b) {
    u64 dd = pack2(d.x, d.y);
    fma2(dd, pack2(a.x, a.y), pack2(b.x, b.y));
    unpack2(dd, d.x, d.y);
}
__device__ __forceinline__ u64 sub2(u64 a, u64 b) {
    u64 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
    u64 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// a*a rounded ONCE.  ptxas (CUDA 12.9) contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even under --fmad=false,
// which would break the non-fused distance rule; fma(a, a, -0.0) with the -0.0 coming from a kernel argument is a
// correctly rounded product that leaves nothing to contract.
__device__ __forceinline__ u64 sqr2(u64 a, u64 negzero2) {
    u64 r;
    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(r) : "l"(a), "l"(negzero2));
    return r;
}
// The distance rule on two (a,b) pairs at once: ((dx*dx + dy*dy) + dz*dz), each step rounded separately.
template <int D>
__device__ __forceinline__ u64 sqdist_pair(u64 ax, u64 ay, u64 az, u64 bx, u64 by, u64 bz, u64 nz) {
    const u64 xx = sqr2(sub2(ax, bx), nz), yy = sqr2(sub2(ay, by), nz);
    u64 s = add2(xx, yy);
    if (D == 3) s = add2(s, sqr2(sub2(az, bz), nz));
    return s;
}

// ---- shared-memory accesses by 32-bit shared address (ptxas folds "+ constant" into the LDS / STS immediate) ----
__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ float2 lds_v2(uint32_t addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ u64 lds_b64(uint32_t addr) {      // two fp32 as one packed FFMA2 operand
    u64 v;
    asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ float4 lds_v4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, float a, float b, float c, float d) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, bool valid) {
    unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    int bytes = valid ? 16 : 0;   // src-size 0 -> the 16 destination bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(gmem_src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src, bool valid) {
    unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    int bytes = valid ? 4 : 0;    // src-size 0 -> the destination word is zero-filled
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(gmem_src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// LeakyReLU(0.1): max(v, 0.1 v) selects the same value as (v > 0 ? v : 0.1 v) in two instructions instead of three
__device__ __forceinline__ float leaky01(float v) { return fmaxf(v, 0.1f * v); }
#endif

}  // namespace b200
