// event_voxel.cu — a9/a10: event stream -> voxel grid by atomic scatter.
//
// Replaces:
//   a9  event_utils.py:109-128 -> :23-39, :264-303, :211-261, :162-208   (20 full passes over all events, each an
//       index_put_(accumulate=True) that mostly adds zeros)
//   a10 dsec.py:570-604 -> :536-568                                     (8 masked put_ passes)
// with ONE pass: a thread per event, 128-bit coalesced event loads, at most 2 (a9) / 8 (a10) fire-and-forget
// RED.ADD.F32 into the L2-resident grid.  HBM traffic = 16 B/event + one zero-fill + the final write-back.
//
// Arithmetic follows the reference operation by operation in fp32 (each step rounded separately); only the
// ORDER in which contributions reach a voxel differs (atomics), hence the stated tolerance 1e-5*max(1,count).
#include <limits.h>

#include <algorithm>

#include "common.cuh"

namespace b200 {

__global__ void __launch_bounds__(256)
event_voxel_int_kernel(const float4* __restrict__ ev, int64_t n, float* __restrict__ vox, int bins, int H, int W,
                       int polarity, int* __restrict__ status) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const float t_first = __ldg(&ev[0]).z, t_last = __ldg(&ev[n - 1]).z;          // event_utils.py:30-31 ([-1] and [0])
    const float den = __fadd_rn(__fsub_rn(t_last, t_first), 1e-6f);                 // :33-34 (NumPy>=2 keeps fp32)
    const float ts0 = __fdiv_rn(__fsub_rn(t_first, t_first), den);
    const float tsl = __fdiv_rn(__fsub_rn(t_last, t_first), den);
    const float dt = __fsub_rn(tsl, ts0);                                           // :240

    const float4 e = __ldg(&ev[i]);
    int x = (int)e.x, y = (int)e.y;                                                 // astype(int32): truncation (:24-25)
    const int p = (int)e.w;
    if (x < -W || x >= W || y < -H || y >= H) {                                     // IndexError in the reference
        atomicAdd(status, 1);
        return;
    }
    if (x < 0) x += W;                                                              // torch negative-index wrap
    if (y < 0) y += H;
    const float ts = __fdiv_rn(__fsub_rn(e.z, t_first), den);
    const float tn = __fmul_rn(__fdiv_rn(__fsub_rn(ts, ts0), dt), (float)(bins - 1));   // :242
    float wgt;
    size_t base;
    const size_t HW = (size_t)H * W;
    if (polarity) { wgt = 1.0f; base = p > 0 ? 0 : (size_t)bins * HW; }             // :293-296: both polarities weigh +1
    else          { wgt = (float)p; base = 0; }
    float* cell = vox + base + (size_t)y * W + x;
    if (tn != tn) {
        // Zero-length window (t_last == t_first): tn = 0/0.  torch.clamp keeps the NaN, so every bin of the event's pixel
        // gets a NaN weight, in the other polarity's grid too (its weight-0 pass adds 0 * NaN).
        const float qnan = __int_as_float(0x7fffffff);
        float* pix = vox + (size_t)y * W + x;
        for (int b = 0; b < bins * (polarity ? 2 : 1); ++b) atomicAdd(pix + (size_t)b * HW, qnan);
        return;
    }
    const float fl = floorf(tn);
    if (!(fabsf(fl) < 1e9f)) return;                                                // +-inf or huge tn: every clamped bin weight is 0
    const int b0 = (int)fl;
#pragma unroll
    for (int k = 0; k < 2; ++k) {                                                   // only bins floor(tn), floor(tn)+1 can be > 0
        const int b = b0 + k;
        if (b < 0 || b >= bins) continue;
        const float bw = __fsub_rn(1.0f, fabsf(__fsub_rn(tn, (float)b)));           // max(0, 1-|tn-b|) (:246)
        if (bw > 0.0f) atomicAdd(cell + (size_t)b * HW, __fmul_rn(wgt, bw));
    }
}

// ---- a10 -------------------------------------------------------------------------------------------------------
// scratch[0..3] = {first index with p>0, last index with p>0, first with p<=0, last with p<=0}
__global__ void trilinear_init_kernel(int* scratch) {
    if (threadIdx.x == 0) { scratch[0] = INT_MAX; scratch[1] = -1; scratch[2] = INT_MAX; scratch[3] = -1; }
}

// Grid-stride pass, one set of four atomics per CTA (r1 issued them per warp: 187 k same-address atomics per scalar at
// 1.5 M events serialised to 131 us — twice the cost of the splat itself; ncu r2).
__global__ void __launch_bounds__(256)
trilinear_bounds_kernel(const float* __restrict__ p, int64_t n, int* __restrict__ scratch) {
    __shared__ unsigned s_red[4][8];
    unsigned fpos = 0x7fffffffu, lpos = 0u, fneg = 0x7fffffffu, lneg = 0u;     // l*: last index + 1 (0 = none)
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const bool pos = __ldg(p + i) > 0.0f;
        const unsigned ii = (unsigned)i;
        if (pos) { fpos = min(fpos, ii); lpos = max(lpos, ii + 1); }
        else     { fneg = min(fneg, ii); lneg = max(lneg, ii + 1); }
    }
    fpos = __reduce_min_sync(FULL, fpos); lpos = __reduce_max_sync(FULL, lpos);
    fneg = __reduce_min_sync(FULL, fneg); lneg = __reduce_max_sync(FULL, lneg);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_red[0][warp] = fpos; s_red[1][warp] = lpos; s_red[2][warp] = fneg; s_red[3][warp] = lneg; }
    __syncthreads();
    if (warp == 0) {
        fpos = __reduce_min_sync(FULL, lane < 8 ? s_red[0][lane] : 0x7fffffffu);
        lpos = __reduce_max_sync(FULL, lane < 8 ? s_red[1][lane] : 0u);
        fneg = __reduce_min_sync(FULL, lane < 8 ? s_red[2][lane] : 0x7fffffffu);
        lneg = __reduce_max_sync(FULL, lane < 8 ? s_red[3][lane] : 0u);
        if (lane == 0) {
            if (lpos) { atomicMin(scratch + 0, (int)fpos); atomicMax(scratch + 1, (int)lpos - 1); }
            if (lneg) { atomicMin(scratch + 2, (int)fneg); atomicMax(scratch + 3, (int)lneg - 1); }
        }
    }
}

__global__ void __launch_bounds__(256)
event_voxel_trilinear_kernel(const float* __restrict__ xs, const float* __restrict__ ys, const int64_t* __restrict__ t,
                             const float* __restrict__ ps, int64_t n, float* __restrict__ vox, int bins, int H, int W,
                             int polarity, const int* __restrict__ scratch) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int64_t t0 = __ldg(t);
    const float last = (float)(__ldg(t + n - 1) - t0);                               // dsec.py:577-578
    const float p = __ldg(ps + i);
    const bool is_pos = p > 0.0f;
    int ia = 0, ib = (int)(n - 1);
    float value;
    size_t base = 0;
    if (polarity) {
        ia = scratch[is_pos ? 0 : 2];
        ib = scratch[is_pos ? 1 : 3];
        value = is_pos ? __fsub_rn(__fmul_rn(2.0f, p), 1.0f) : 1.0f;                 // :549 and :597-598 (neg_weights = 1)
        base = is_pos ? 0 : (size_t)bins * H * W;
    } else {
        value = __fsub_rn(__fmul_rn(2.0f, p), 1.0f);
    }
    const float ts = __fdiv_rn((float)(__ldg(t + i) - t0), last);
    const float ta = __fdiv_rn((float)(__ldg(t + ia) - t0), last);
    const float tb = __fdiv_rn((float)(__ldg(t + ib) - t0), last);
    const float tn = __fdiv_rn(__fmul_rn((float)(bins - 1), __fsub_rn(ts, ta)), __fsub_rn(tb, ta));   // :543
    const float x = __ldg(xs + i), y = __ldg(ys + i);
    if (!(fabsf(x) < 1e9f) || !(fabsf(y) < 1e9f) || !(fabsf(tn) < 1e9f)) return;    // .int() of such values is masked out
    const int x0 = (int)x, y0 = (int)y, tq = (int)tn;                                // .int(): truncation (:545-547)
    float* g = vox + base;
    const float* vox_end = vox + (size_t)bins * (polarity ? 2 : 1) * H * W;
    // The two x taps of a (row, bin) pair are neighbours in memory: when the left one sits on an 8-byte boundary they go
    // out as ONE red.global.add.v2.f32 (the kernel is bound by the SMs' RED issue rate — 1.5 M events x 8 taps at ~1.3
    // cycles per lane — so every merged pair is a tap less; ncu r2).
    const float wx0 = __fmul_rn(value, __fsub_rn(1.0f, fabsf(__fsub_rn((float)x0, x))));            // :557, left to right
    const float wx1 = __fmul_rn(value, __fsub_rn(1.0f, fabsf(__fsub_rn((float)(x0 + 1), x))));
    const bool vx0 = x0 >= 0 && x0 < W, vx1 = x0 + 1 >= 0 && x0 + 1 < W;
#pragma unroll
    for (int cy = 0; cy < 2; ++cy)
#pragma unroll
        for (int ct = 0; ct < 2; ++ct) {
            const int yl = y0 + cy, tl = tq + ct;
            if (yl < 0 || yl >= H || tl < 0 || tl >= bins) continue;                                  // :555-556
            const float wy = __fsub_rn(1.0f, fabsf(__fsub_rn((float)yl, y)));
            const float wt = __fsub_rn(1.0f, fabsf(__fsub_rn((float)tl, tn)));
            const float a = __fmul_rn(__fmul_rn(wx0, wy), wt), b = __fmul_rn(__fmul_rn(wx1, wy), wt);   // :558-559
            float* cell = g + ((size_t)tl * H + yl) * W + x0;
            const uintptr_t ca = reinterpret_cast<uintptr_t>(cell);
            if (vx0 && vx1 && (ca & 7) == 0) {
                asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(cell), "f"(a), "f"(b) : "memory");
            } else if (vx0 && vx1 && (ca & 15) == 4 && cell > vox && cell + 2 < vox_end) {
                // the pair sits in the middle of a 16-byte group: one v4 with zeros on the outer lanes (x + 0 = x) instead of two
                // scalar REDs; the outer lanes are this row's neighbours or, at a row end, the next row's first cell
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(cell - 1), "f"(0.0f), "f"(a), "f"(b), "f"(0.0f) : "memory");
            } else {
                if (vx0) atomicAdd(cell, a);
                if (vx1) atomicAdd(cell + 1, b);
            }
        }
}

}  // namespace b200

extern "C" int b200_event_voxel_int(const float* events, int64_t n, float* vox, int bins, int H, int W, int polarity,
                                    int* status, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE(events && vox && status, "b200_event_voxel_int: null pointer");
    B200_REQUIRE(n >= 1, "b200_event_voxel_int: need at least one event (the reference indexes events[-1])");
    B200_REQUIRE(bins >= 1 && H >= 1 && W >= 1, "b200_event_voxel_int: bad sizes bins=%d H=%d W=%d", bins, H, W);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(events) & 15) == 0, "b200_event_voxel_int: events must be 16-byte aligned");
    B200_REQUIRE(n < (1ll << 31) * 256, "b200_event_voxel_int: too many events");
    cudaStream_t st = as_stream(stream);
    const size_t cells = (size_t)bins * (polarity ? 2 : 1) * H * W;
    B200_CUDA(cudaMemsetAsync(vox, 0, cells * sizeof(float), st));
    B200_CUDA(cudaMemsetAsync(status, 0, sizeof(int), st));
    event_voxel_int_kernel<<<ceil_div(n, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(events), n, vox, bins, H, W,
                                                            polarity, status);
    B200_LAUNCH_CHECK("b200_event_voxel_int");
    return B200_OK;
}

extern "C" int b200_event_voxel_trilinear(const float* x, const float* y, const int64_t* t, const float* p, int64_t n,
                                          float* vox, int bins, int H, int W, int polarity, int* scratch,
                                          b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE(x && y && t && p && vox && scratch, "b200_event_voxel_trilinear: null pointer");
    B200_REQUIRE(n >= 1 && n < INT_MAX, "b200_event_voxel_trilinear: need 1 <= n < 2^31 events");
    B200_REQUIRE(bins >= 1 && H >= 1 && W >= 1, "b200_event_voxel_trilinear: bad sizes bins=%d H=%d W=%d", bins, H, W);
    cudaStream_t st = as_stream(stream);
    const size_t cells = (size_t)bins * (polarity ? 2 : 1) * H * W;
    B200_CUDA(cudaMemsetAsync(vox, 0, cells * sizeof(float), st));
    if (polarity) {
        trilinear_init_kernel<<<1, 32, 0, st>>>(scratch);
        trilinear_bounds_kernel<<<std::min(ceil_div(n, 256), sm_count() * 8), 256, 0, st>>>(p, n, scratch);
    }
    event_voxel_trilinear_kernel<<<ceil_div(n, 256), 256, 0, st>>>(x, y, t, p, n, vox, bins, H, W, polarity, scratch);
    B200_LAUNCH_CHECK("b200_event_voxel_trilinear");
    return B200_OK;
}
