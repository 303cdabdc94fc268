// decoder_common.cuh — the per-sample arithmetic that the forward kernels of the decoder and projection ops (gather.cu)
// and their backwards (decoder_bwd.cu) share: the backwards recompute taps, weights, distances and gather indices
// instead of saving them, so both sides must run exactly the same fp32 operations.
#pragma once
#include "common.cuh"

namespace b200 {

// ---- a6: a gather index as the gathers treat it ----
__device__ __forceinline__ int64_t wrap_index(int64_t j, int N, int* bad) {
    if (j < 0) j += N;                                   // python-style wrap of negative indices (torch.gather itself raises on them)
    if (j < 0 || j >= N) {                               // torch would raise; we clamp and count (deliberate: see projection.py)
        if (bad) atomicAdd(bad, 1);
        j = j < 0 ? 0 : N - 1;
    }
    return j;
}

// ---- bilinear taps, exactly the arithmetic of models/utils.py:290-291 followed by grid_sample(align_corners=True) ----
struct Taps {
    int o00, o01, o10, o11;      // offsets inside one H*W plane, -1 when the tap is outside the image (zero padding)
    float w00, w01, w10, w11;
};
__device__ __forceinline__ float renorm_coord(float x, int size) {
    const float sm1 = (float)(size - 1);
    const float g = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, x), sm1), 1.0f);        // 2*x/(size-1) - 1
    return __fmul_rn(__fdiv_rn(__fadd_rn(g, 1.0f), 2.0f), sm1);                  // ((g+1)/2)*(size-1)
}

// a7 (grid_sample_wrapper, zero padding): the top-left tap of one sample and its 1-D weights.  Huge or non-finite
// coordinates get x0 = y0 = -2 (guards the float->int conversion), which leaves every tap outside the image.
struct ZeroSample {
    int x0, y0;
    float wx0, wx1, wy0, wy1;
};
__device__ __forceinline__ ZeroSample zero_sample(float x, float y, int H, int W) {
    const float ix = renorm_coord(x, W), iy = renorm_coord(y, H);
    const float fx = floorf(ix), fy = floorf(iy);
    ZeroSample s;
    s.wx1 = ix - fx; s.wy1 = iy - fy; s.wx0 = (fx + 1.0f) - ix; s.wy0 = (fy + 1.0f) - iy;
    const bool finite = fabsf(ix) < 1e9f && fabsf(iy) < 1e9f;
    s.x0 = finite ? (int)fx : -2; s.y0 = finite ? (int)fy : -2;
    return s;
}
__device__ __forceinline__ Taps zero_taps(const ZeroSample& s, int H, int W) {
    const int x0 = s.x0, y0 = s.y0, x1 = x0 + 1, y1 = y0 + 1;
    const bool vx0 = x0 >= 0 && x0 < W, vx1 = x1 >= 0 && x1 < W, vy0 = y0 >= 0 && y0 < H, vy1 = y1 >= 0 && y1 < H;
    Taps t;
    t.o00 = (vy0 && vx0) ? y0 * W + x0 : -1; t.w00 = s.wx0 * s.wy0;
    t.o01 = (vy0 && vx1) ? y0 * W + x1 : -1; t.w01 = s.wx1 * s.wy0;
    t.o10 = (vy1 && vx0) ? y1 * W + x0 : -1; t.w10 = s.wx0 * s.wy1;
    t.o11 = (vy1 && vx1) ? y1 * W + x1 : -1; t.w11 = s.wx1 * s.wy1;
    return t;
}
__device__ __forceinline__ Taps make_taps(float x, float y, int H, int W) {
    return zero_taps(zero_sample(x, y, H, W), H, W);
}

// f3: backwarp_2d (models/utils.py:186-198) with padding_mode='border': out[b,c,p] = bilinear(x[b,c], pixel p + flow[b,:,p]).
// The grid takes the reference's round trip (mesh + flow, 2*g/(W-1)-1, then grid_sample's ((g+1)/2)*(W-1)), is then
// clamped to [0, size-1] (ATen clip_coordinates) and sampled like a7; a clamped x0 = W-1 leaves the right tap outside
// the image with weight 0, exactly as ATen's within_bounds test does.
// The sample position of one pixel: un-clamped coordinates (the backward's clip test reads them), the top-left tap of
// the clamped position and its 1-D weights.
struct BorderSample {
    float rx, ry;                  // after the round trip, before the clamp
    int x0, y0;                    // inside the image; x0 + 1 == W / y0 + 1 == H is outside (weight 0 there)
    float wx0, wx1, wy0, wy1;
};
__device__ __forceinline__ BorderSample border_sample(float gx, float gy, int H, int W) {
    BorderSample s;
    s.rx = renorm_coord(gx, W);
    s.ry = renorm_coord(gy, H);
    const float ix = fminf((float)(W - 1), fmaxf(s.rx, 0.0f));
    const float iy = fminf((float)(H - 1), fmaxf(s.ry, 0.0f));
    const float fx = floorf(ix), fy = floorf(iy);
    s.wx1 = ix - fx; s.wy1 = iy - fy; s.wx0 = (fx + 1.0f) - ix; s.wy0 = (fy + 1.0f) - iy;
    s.x0 = (int)fx; s.y0 = (int)fy;                                          // clamped: always finite and in range
    return s;
}
__device__ __forceinline__ Taps border_taps(const BorderSample& s, int H, int W) {
    const int x0 = s.x0, y0 = s.y0, x1 = x0 + 1, y1 = y0 + 1;
    const bool vx1 = x1 < W, vy1 = y1 < H;
    Taps t;
    t.o00 = y0 * W + x0;                 t.w00 = s.wx0 * s.wy0;
    t.o01 = vx1 ? y0 * W + x1 : -1;      t.w01 = s.wx1 * s.wy0;
    t.o10 = vy1 ? y1 * W + x0 : -1;      t.w10 = s.wx0 * s.wy1;
    t.o11 = (vy1 && vx1) ? y1 * W + x1 : -1; t.w11 = s.wx1 * s.wy1;
    return t;
}
__device__ __forceinline__ Taps make_taps_border(float gx, float gy, int H, int W) {
    return border_taps(border_sample(gx, gy, H, W), H, W);
}

// ---- f2: knn_interpolation's inverse-distance weights (models/utils.py:140-156) ----
constexpr int KI_KMAX = 8;       // largest k the kernels take (the model uses 3)

// A neighbour index as the gathers treat it: negative indices wrap once, anything still out of range is clamped.
__device__ __forceinline__ int knn_point(int64_t t, int M) {
    if (t < 0) t += M;
    return (int)(t < 0 ? 0 : (t >= M ? M - 1 : t));
}
// Un-normalised weight 1 / max(|xyz[j] - q|, 1e-8) of point j (xyz: one batch item, [3,M]); u = xyz[j] - q and r = |u|
// are returned for the backward.  Every operation is rounded separately in the reference's order.
__device__ __forceinline__ float idw_weight(const float* __restrict__ xyz, int M, int j, float qx, float qy, float qz,
                                            float u[3], float& r) {
    u[0] = __fsub_rn(__ldg(xyz + j), qx);
    u[1] = __fsub_rn(__ldg(xyz + (size_t)M + j), qy);
    u[2] = __fsub_rn(__ldg(xyz + (size_t)2 * M + j), qz);
    r = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(u[0], u[0]), __fmul_rn(u[1], u[1])), __fmul_rn(u[2], u[2])));
    const float d = r < 1e-8f ? 1e-8f : r;                                        // .clamp(1e-8)
    return __fdiv_rn(1.0f, d);
}

}  // namespace b200
