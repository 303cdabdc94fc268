// fps_common.cuh — what the two pruned FPS scans share (fps.cu: one CTA per cloud, N <= 8192; fps_large.cu: one
// thread-block cluster per cloud, any N): the monotone float <-> uint map the warp collectives reduce on, and the box test
// that proves a group of points unchanged by a new centre.
#pragma once
#include "common.cuh"

namespace b200 {

__device__ __forceinline__ unsigned fps_orderable(float v) {          // monotone float -> uint map (for redux min/max)
    const unsigned b = __float_as_uint(v);
    return b ^ ((b >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float fps_unorder(unsigned u) {
    return __uint_as_float(u ^ ((u >> 31) ? 0x80000000u : 0xFFFFFFFFu));
}

// The distance rule (sqdist3_rule) evaluated on the gap vector from the centre c to the box [lo, hi]:
//     g = max(fl(lo - c), fl(c - hi), 0) per axis,   d_box = ((gx*gx + gy*gy) + gz*gz)   (same non-fused fp32 ops).
// fp32 subtraction, multiplication and addition are monotone, so d_box <= the rule's distance from c to EVERY point in the
// box.  A box whose d_box is >= the cached maximum running distance of its points cannot lower any of them (running
// distances only ever take min(dist, d)), so the points and their cached (max, index) stay as they are.  NaN coordinates
// never enter a box (fminf/fmaxf drop them); a NaN centre gives g = 0 on that axis, i.e. the box is visited.
__device__ __forceinline__ float fps_box_dist(float lox, float loy, float loz, float hix, float hiy, float hiz,
                                              float cx, float cy, float cz) {
    const float gx = fmaxf(fmaxf(__fsub_rn(lox, cx), __fsub_rn(cx, hix)), 0.0f);
    const float gy = fmaxf(fmaxf(__fsub_rn(loy, cy), __fsub_rn(cy, hiy)), 0.0f);
    const float gz = fmaxf(fmaxf(__fsub_rn(loz, cz), __fsub_rn(cz, hiz)), 0.0f);
    return __fadd_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)), __fmul_rn(gz, gz));
}

// Box test: true when the box may hold a point whose running distance the centre lowers (NaN d_box -> visit).
__device__ __forceinline__ bool fps_box_may_change(float dbox, float cached_max) { return !(dbox >= cached_max); }

}  // namespace b200
