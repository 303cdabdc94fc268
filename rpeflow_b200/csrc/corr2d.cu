// corr2d.cu — a1/a2: PWC-style 2-D local correlation cost volume (max displacement md, (2md+1)^2 channels).
//
// Replaces models/csrc/correlation/correlation_forward_kernel.cu:11-55 (one warp per output pixel, 81 serial
// shuffle reductions, 4-byte stores H*W apart) and correlation_backward_kernel.cu:4-89.
//
// Forward design (HBM-bound at level 1, at the fp32 ridge — SURVEY §7):
//   * CTA = output tile of 8 rows x 24 columns for ALL (2md+1)^2 displacements; one warp per row-shift dy.
//   * feature tiles (in1: 8x24 pixels, in2: (8+2md)x(24+2md) halo) are staged in shared memory in 16-channel
//     chunks with 16-byte cp.async (zero-fill outside the image = the reference's zero padding), double buffered.
//   * lane -> (row = lane%8, strip = lane/8); a thread owns a 6-pixel strip and all 2md+1 column shifts:
//     54 outputs, each accumulated as an (even-channel, odd-channel) pair so the inner loop is pure packed
//     FFMA2 (fma.rn.f32x2) fed by 128-bit shared loads; rows are padded by 16 B so the 8 lanes of a quarter
//     warp hit 8 different 16-byte bank groups (conflict-free LDS.128).
//   * every in2 value loaded is used by up to 6 pixels x 2 packed lanes; every in1 value by 9 shifts.
//   * stores: each thread writes 6 consecutive floats per displacement channel, the 4 strips of a row are contiguous.
#include <algorithm>

#include "common.cuh"

namespace b200 {

// corr2d_tma.cu: the persistent TMA-fed kernel (md = 4, C % 4 == 0, 16-byte aligned inputs)
bool corr2d_tma_eligible(const float* in1, const float* in2, int B, int C, int H, int W, int md);
cudaError_t corr2d_fwd_tma(const float* in1, const float* in2, float* out, int B, int C, int H, int W, cudaStream_t st);

constexpr int C2_TH = 8, C2_PX = 6, C2_TW = 4 * C2_PX, C2_CC = 16;   // 9 warps/CTA cap a thread at 168 registers: 6-pixel strips fit

template <int MD>
struct Corr2dCfg {
    static constexpr int ND = 2 * MD + 1;
    static constexpr int HR = C2_TH + 2 * MD;            // halo rows
    static constexpr int HC = C2_TW + 2 * MD;            // halo columns
    static constexpr int WIN = C2_PX + 2 * MD;           // in2 pixels one strip touches
    static constexpr int RS2 = HC * C2_CC + 4;           // floats per in2 row (+16 B: bank rotation across rows)
    static constexpr int RS1 = C2_TW * C2_CC + 4;
    static constexpr int STAGE = HR * RS2 + C2_TH * RS1; // floats per pipeline stage
    static constexpr int THREADS = ND * 32;
    static constexpr size_t SMEM = 2 * STAGE * sizeof(float);
};

template <int MD, bool VEC>
__device__ __forceinline__ void corr2d_load_stage(float* stage, const float* __restrict__ in1, const float* __restrict__ in2,
                                                  int b, int y0, int x0, int c0, int C, int H, int W) {
    using K = Corr2dCfg<MD>;
    float* s2 = stage;
    float* s1 = stage + K::HR * K::RS2;
    constexpr int Q = C2_CC / 4;
    // in2 halo
    for (int e = threadIdx.x; e < K::HR * K::HC * Q; e += K::THREADS) {
        const int q = e % Q, px = (e / Q) % K::HC, r = e / (Q * K::HC);
        const int gy = y0 + r - MD, gx = x0 + px - MD, c = c0 + q * 4;
        const bool in = gy >= 0 && gy < H && gx >= 0 && gx < W;
        float* dst = s2 + r * K::RS2 + px * C2_CC + q * 4;
        const float* src = in2 + (((size_t)b * H + (in ? gy : 0)) * W + (in ? gx : 0)) * C + c;
        if (VEC) {
            cp_async16(dst, in && c < C ? src : in2, in && c < C);
        } else {
#pragma unroll
            for (int t = 0; t < 4; ++t) dst[t] = (in && c + t < C) ? __ldg(src + t) : 0.0f;
        }
    }
    // in1 tile
    for (int e = threadIdx.x; e < C2_TH * C2_TW * Q; e += K::THREADS) {
        const int q = e % Q, px = (e / Q) % C2_TW, r = e / (Q * C2_TW);
        const int gy = y0 + r, gx = x0 + px, c = c0 + q * 4;
        const bool in = gy < H && gx < W;
        float* dst = s1 + r * K::RS1 + px * C2_CC + q * 4;
        const float* src = in1 + (((size_t)b * H + (in ? gy : 0)) * W + (in ? gx : 0)) * C + c;
        if (VEC) {
            cp_async16(dst, in && c < C ? src : in1, in && c < C);
        } else {
#pragma unroll
            for (int t = 0; t < 4; ++t) dst[t] = (in && c + t < C) ? __ldg(src + t) : 0.0f;
        }
    }
}

template <int MD, bool VEC>
__global__ void __launch_bounds__(Corr2dCfg<MD>::THREADS, 1)
corr2d_fwd_kernel(const float* __restrict__ in1, const float* __restrict__ in2, float* __restrict__ out,
                  int C, int H, int W, int tiles_x, int tiles_y) {
    using K = Corr2dCfg<MD>;
    extern __shared__ float4 smem_f4[];
    float* smem = reinterpret_cast<float*>(smem_f4);

    const int tile = blockIdx.x;
    const int b = tile / (tiles_x * tiles_y);
    const int ty = (tile / tiles_x) % tiles_y, tx = tile % tiles_x;
    const int y0 = ty * C2_TH, x0 = tx * C2_TW;
    const int dyw = threadIdx.x >> 5;                    // warp = row shift index, dy = dyw - MD
    const int lane = threadIdx.x & 31, ly = lane & 7, lx = lane >> 3;

    float2 acc[C2_PX][K::ND];
#pragma unroll
    for (int i = 0; i < C2_PX; ++i)
#pragma unroll
        for (int d = 0; d < K::ND; ++d) acc[i][d] = make_float2(0.0f, 0.0f);

    const int nchunks = (C + C2_CC - 1) / C2_CC;
    corr2d_load_stage<MD, VEC>(smem, in1, in2, b, y0, x0, 0, C, H, W);
    cp_async_commit();

    for (int ch = 0; ch < nchunks; ++ch) {
        float* cur = smem + (ch & 1) * K::STAGE;
        if (ch + 1 < nchunks) {
            corr2d_load_stage<MD, VEC>(smem + ((ch + 1) & 1) * K::STAGE, in1, in2, b, y0, x0, (ch + 1) * C2_CC, C, H, W);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();

        const float* r2 = cur + (ly + dyw) * K::RS2 + (lx * C2_PX) * C2_CC;
        const float* r1 = cur + K::HR * K::RS2 + ly * K::RS1 + (lx * C2_PX) * C2_CC;
#pragma unroll
        for (int q = 0; q < C2_CC / 4; ++q) {
            float4 a[C2_PX];
#pragma unroll
            for (int i = 0; i < C2_PX; ++i) a[i] = *reinterpret_cast<const float4*>(r1 + i * C2_CC + q * 4);
#pragma unroll
            for (int j = 0; j < K::WIN; ++j) {
                const float4 v = *reinterpret_cast<const float4*>(r2 + j * C2_CC + q * 4);
                const float2 vlo = make_float2(v.x, v.y), vhi = make_float2(v.z, v.w);
#pragma unroll
                for (int i = 0; i < C2_PX; ++i) {
                    const int d = j - i;                 // column shift index, dx = d - MD
                    if (d >= 0 && d < K::ND) {
                        ffma2(acc[i][d], make_float2(a[i].x, a[i].y), vlo);
                        ffma2(acc[i][d], make_float2(a[i].z, a[i].w), vhi);
                    }
                }
            }
        }
        __syncthreads();                                 // everyone done with `cur` before it is refilled
    }

    // epilogue: out[b, dyw*ND + d, y, x0 + lx*6 .. +5]
    const int y = y0 + ly, xs = x0 + lx * C2_PX;
    if (y >= H || xs >= W) return;
    const float fc = (float)C;
    const size_t plane = (size_t)H * W;
    float* obase = out + ((size_t)b * K::ND * K::ND + (size_t)dyw * K::ND) * plane + (size_t)y * W + xs;
    const bool vec = (W % 2 == 0) && (xs + C2_PX <= W) && ((reinterpret_cast<uintptr_t>(out) & 7) == 0);
#pragma unroll
    for (int d = 0; d < K::ND; ++d) {
        float r[C2_PX];
#pragma unroll
        for (int i = 0; i < C2_PX; ++i) r[i] = __fdiv_rn(acc[i][d].x + acc[i][d].y, fc);   // sum / C (correlation_forward_kernel.cu:46)
        float* o = obase + (size_t)d * plane;
        if (vec) {
#pragma unroll
            for (int i = 0; i < C2_PX; i += 2)                                                   // streaming: never re-read here
                __stcs(reinterpret_cast<float2*>(o + i), make_float2(r[i], r[i + 1]));
        } else {
#pragma unroll
            for (int i = 0; i < C2_PX; ++i)
                if (xs + i < W) o[i] = r[i];
        }
    }
}

template <int MD>
static cudaError_t launch_corr2d_fwd(const float* in1, const float* in2, float* out, int B, int C, int H, int W, cudaStream_t st) {
    using K = Corr2dCfg<MD>;
    const int tiles_x = ceil_div(W, C2_TW), tiles_y = ceil_div(H, C2_TH);
    const int64_t tiles = (int64_t)B * tiles_x * tiles_y;
    if (tiles > 0x7fffffff) return cudaErrorInvalidValue;
    const bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(in1) & 15) == 0) && ((reinterpret_cast<uintptr_t>(in2) & 15) == 0);
    cudaError_t e;
    if (vec) {
        auto kern = corr2d_fwd_kernel<MD, true>;
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K::SMEM);
        if (e != cudaSuccess) return e;
        kern<<<(unsigned)tiles, K::THREADS, K::SMEM, st>>>(in1, in2, out, C, H, W, tiles_x, tiles_y);
    } else {
        auto kern = corr2d_fwd_kernel<MD, false>;
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K::SMEM);
        if (e != cudaSuccess) return e;
        kern<<<(unsigned)tiles, K::THREADS, K::SMEM, st>>>(in1, in2, out, C, H, W, tiles_x, tiles_y);
    }
    return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------------------
// Backward (a2).  Correct-first kernel (training only; SURVEY §8f ranks its tuning last):
//   gin1[b,c,y,x] = (1/C) sum_{dy,dx} gout[b,t,y,x]       * in2[b,y+dy,x+dx,c]
//   gin2[b,c,y,x] = (1/C) sum_{dy,dx} gout[b,t,y-dy,x-dx] * in1[b,y-dy,x-dx,c]        t = (dy+md)*(2md+1)+(dx+md)
// CTA = one image row segment of 32 pixels; the partner feature halo ((2md+1) rows x (32+2md) px x 32 channels)
// and the needed grad_out values ((2md+1)^2 x (32+2md)) are staged in shared memory; thread = (pixel, 2 channels).
// Outputs are NCHW like the reference (wrapper.py:34-35 permutes them).
constexpr int BW_TW = 32, BW_CC = 16, BW_CPT = BW_CC / 8;   // 8 channel groups per CTA

template <int MD, int WHICH>   // WHICH = 1: grad wrt in1 (partner = in2); 2: grad wrt in2 (partner = in1)
__global__ void __launch_bounds__(256)
corr2d_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ partner, float* __restrict__ gin,
                  int C, int H, int W, int tiles_x) {
    constexpr int ND = 2 * MD + 1, HC = BW_TW + 2 * MD, PS = BW_CC + 1;   // odd pixel stride: conflict-free across pixels
    __shared__ float s_f[ND * HC * PS];
    __shared__ float s_g[ND * ND * HC];
    const int b = blockIdx.z, y = blockIdx.y, x0 = blockIdx.x * BW_TW;
    const int tx = threadIdx.x & 31, cg = threadIdx.x >> 5;              // 8 channel groups of BW_CPT
    const size_t plane = (size_t)H * W;

    // grad_out values: for WHICH=1 row y of every plane; for WHICH=2 plane t=(dy,dx) at row y-dy.
    for (int e = threadIdx.x; e < ND * ND * HC; e += 256) {
        const int px = e % HC, t = e / HC, dyi = t / ND;
        const int gy = WHICH == 1 ? y : y - (dyi - MD);
        const int gx = x0 + px - MD;
        float v = 0.0f;
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) v = __ldg(gout + ((size_t)b * ND * ND + t) * plane + (size_t)gy * W + gx);
        s_g[e] = v;
    }

    for (int c0 = 0; c0 < C; c0 += BW_CC) {
        __syncthreads();
        // partner rows: WHICH=1 -> in2 rows y+dy ; WHICH=2 -> in1 rows y-dy   (row slot = dyi)
        for (int e = threadIdx.x; e < ND * HC * BW_CC; e += 256) {
            const int c = e % BW_CC, px = (e / BW_CC) % HC, dyi = e / (BW_CC * HC);
            const int gy = WHICH == 1 ? y + (dyi - MD) : y - (dyi - MD);
            const int gx = x0 + px - MD;
            float v = 0.0f;
            if (gy >= 0 && gy < H && gx >= 0 && gx < W && c0 + c < C)
                v = __ldg(partner + (((size_t)b * H + gy) * W + gx) * C + c0 + c);
            s_f[(dyi * HC + px) * PS + c] = v;
        }
        __syncthreads();

        float acc[BW_CPT];
#pragma unroll
        for (int u = 0; u < BW_CPT; ++u) acc[u] = 0.0f;
#pragma unroll
        for (int dyi = 0; dyi < ND; ++dyi)
#pragma unroll
            for (int dxi = 0; dxi < ND; ++dxi) {
                const int t = dyi * ND + dxi;
                // WHICH=1: gout at own pixel (halo col tx+MD), partner at x+dx (halo col tx+dxi)
                // WHICH=2: gout and partner both at x-dx (halo col tx+2MD-dxi)
                const int pcol = WHICH == 1 ? tx + dxi : tx + 2 * MD - dxi;
                const int gcol = WHICH == 1 ? tx + MD : pcol;
                const float g = s_g[t * HC + gcol];
                const float* f = s_f + (dyi * HC + pcol) * PS + cg * BW_CPT;
#pragma unroll
                for (int u = 0; u < BW_CPT; ++u) acc[u] += g * f[u];
            }
        const int x = x0 + tx;
        if (x < W) {
#pragma unroll
            for (int u = 0; u < BW_CPT; ++u) {
                const int c = c0 + cg * BW_CPT + u;
                if (c < C) gin[((size_t)b * C + c) * plane + (size_t)y * W + x] = __fdiv_rn(acc[u], (float)C);
            }
        }
    }
}

bool corr2d_bwd_tiled_eligible(const float* gout, const float* in1, const float* in2, const float* g1, const float* g2,
                               int B, int C, int H, int W, int md);                       // corr2d_bwd_tiled.cu
cudaError_t corr2d_bwd_tiled(const float* gout, const float* in1, const float* in2, float* g1, float* g2, int B, int C, int H,
                             int W, cudaStream_t st);

template <int MD>
static cudaError_t launch_corr2d_bwd(const float* gout, const float* in1, const float* in2, float* g1, float* g2,
                                     int B, int C, int H, int W, cudaStream_t st) {
    const int tiles_x = ceil_div(W, BW_TW);
    dim3 grid(tiles_x, H, B);
    corr2d_bwd_kernel<MD, 1><<<grid, 256, 0, st>>>(gout, in2, g1, C, H, W, tiles_x);
    corr2d_bwd_kernel<MD, 2><<<grid, 256, 0, st>>>(gout, in1, g2, C, H, W, tiles_x);
    return cudaGetLastError();
}

// ---- any max_displacement (md > 4): plain kernels, correctness first ---------------------------------------------------
// The reference kernels take any md (correlation_forward_kernel.cu:11-55); RPEFlow only ever passes 4, so these are not
// tuned: a warp per (pixel, displacement) with lanes over channels for the forward (coalesced NHWC rows), a thread per
// (pixel, channel) for the backward.
__global__ void __launch_bounds__(256)
corr2d_fwd_any_kernel(const float* __restrict__ in1, const float* __restrict__ in2, float* __restrict__ out, int C, int H, int W,
                      int md, int64_t items) {
    const int D = 2 * md + 1;
    const int lane = threadIdx.x & 31;
    for (int64_t it = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); it < items; it += (int64_t)gridDim.x * 8) {
        const int x = (int)(it % W);
        int64_t r = it / W;
        const int y = (int)(r % H); r /= H;
        const int tc = (int)(r % (D * D));
        const int b = (int)(r / (D * D));
        const int dy = tc / D - md, dx = tc % D - md;
        const int y2 = y + dy, x2 = x + dx;
        float s = 0.0f;
        if (y2 >= 0 && y2 < H && x2 >= 0 && x2 < W) {
            const float* a = in1 + (((size_t)b * H + y) * W + x) * C;
            const float* c2 = in2 + (((size_t)b * H + y2) * W + x2) * C;
            for (int c = lane; c < C; c += 32) s += __ldg(a + c) * __ldg(c2 + c);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
        }
        if (lane == 0) out[(((size_t)b * D * D + tc) * H + y) * W + x] = s / (float)C;
    }
}

__global__ void __launch_bounds__(256)
corr2d_bwd_any_kernel(const float* __restrict__ gout, const float* __restrict__ in1, const float* __restrict__ in2,
                      float* __restrict__ gin1, float* __restrict__ gin2, int C, int H, int W, int md, int64_t items) {
    const int D = 2 * md + 1;
    for (int64_t it = (int64_t)blockIdx.x * 256 + threadIdx.x; it < items; it += (int64_t)gridDim.x * 256) {
        const int c = (int)(it % C);                          // channel fastest: NHWC partner reads coalesce
        int64_t r = it / C;
        const int x = (int)(r % W); r /= W;
        const int y = (int)(r % H);
        const int b = (int)(r / H);
        float s1 = 0.0f, s2 = 0.0f;
        for (int dy = -md; dy <= md; ++dy)
            for (int dx = -md; dx <= md; ++dx) {
                const int tc = (dy + md) * D + (dx + md);
                const int y2 = y + dy, x2 = x + dx;            // grad wrt in1[y,x]: partner in2[y+dy,x+dx]
                if (y2 >= 0 && y2 < H && x2 >= 0 && x2 < W)
                    s1 += __ldg(gout + (((size_t)b * D * D + tc) * H + y) * W + x) * __ldg(in2 + (((size_t)b * H + y2) * W + x2) * C + c);
                const int y1 = y - dy, x1 = x - dx;            // grad wrt in2[y,x]: partner in1[y-dy,x-dx]
                if (y1 >= 0 && y1 < H && x1 >= 0 && x1 < W)
                    s2 += __ldg(gout + (((size_t)b * D * D + tc) * H + y1) * W + x1) * __ldg(in1 + (((size_t)b * H + y1) * W + x1) * C + c);
            }
        gin1[(((size_t)b * C + c) * H + y) * W + x] = s1 / (float)C;
        gin2[(((size_t)b * C + c) * H + y) * W + x] = s2 / (float)C;
    }
}

}  // namespace b200

extern "C" int b200_corr2d_fwd(const float* in1, const float* in2, float* out, int B, int C, int H, int W, int md,
                               b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0) || (in1 && in2 && out), "b200_corr2d_fwd: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 1 && H >= 1 && W >= 1, "b200_corr2d_fwd: bad sizes B=%d C=%d H=%d W=%d", B, C, H, W);
    B200_REQUIRE(md >= 1 && md <= 64, "b200_corr2d_fwd: max_displacement must be in [1,64] (got %d)", md);
    if (B == 0) return B200_OK;
    cudaError_t e;
    if (md > 4) {                                             // not a shape RPEFlow uses: plain kernel
        const int64_t items = (int64_t)B * (2 * md + 1) * (2 * md + 1) * H * W;
        const int grid = (int)std::min<int64_t>((items + 7) / 8, (int64_t)sm_count() * 32);
        corr2d_fwd_any_kernel<<<grid, 256, 0, as_stream(stream)>>>(in1, in2, out, C, H, W, md, items);
        B200_LAUNCH_CHECK("b200_corr2d_fwd(any md)");
        return B200_OK;
    }
    if (corr2d_tma_eligible(in1, in2, B, C, H, W, md)) {
        e = corr2d_fwd_tma(in1, in2, out, B, C, H, W, as_stream(stream));
        if (e != cudaSuccess) return cuda_fail(e, "b200_corr2d_fwd(tma)");
        return B200_OK;
    }
    switch (md) {
        case 1: e = launch_corr2d_fwd<1>(in1, in2, out, B, C, H, W, as_stream(stream)); break;
        case 2: e = launch_corr2d_fwd<2>(in1, in2, out, B, C, H, W, as_stream(stream)); break;
        case 3: e = launch_corr2d_fwd<3>(in1, in2, out, B, C, H, W, as_stream(stream)); break;
        default: e = launch_corr2d_fwd<4>(in1, in2, out, B, C, H, W, as_stream(stream)); break;
    }
    if (e != cudaSuccess) return cuda_fail(e, "b200_corr2d_fwd");
    return B200_OK;
}

extern "C" int b200_corr2d_bwd(const float* gout, const float* in1, const float* in2, float* gin1, float* gin2,
                               int B, int C, int H, int W, int md, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0) || (gout && in1 && in2 && gin1 && gin2), "b200_corr2d_bwd: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 1 && H >= 1 && W >= 1, "b200_corr2d_bwd: bad sizes B=%d C=%d H=%d W=%d", B, C, H, W);
    B200_REQUIRE(md >= 1 && md <= 64, "b200_corr2d_bwd: max_displacement must be in [1,64] (got %d)", md);
    B200_REQUIRE(H <= 65535 && B <= 65535, "b200_corr2d_bwd: H or B exceeds the grid limit");
    if (B == 0) return B200_OK;
    cudaError_t e;
    if (md > 4) {
        const int64_t items = (int64_t)B * H * W * C;
        const int grid = (int)std::min<int64_t>((items + 255) / 256, (int64_t)sm_count() * 32);
        corr2d_bwd_any_kernel<<<grid, 256, 0, as_stream(stream)>>>(gout, in1, in2, gin1, gin2, C, H, W, md, items);
        B200_LAUNCH_CHECK("b200_corr2d_bwd(any md)");
        return B200_OK;
    }
    if (corr2d_bwd_tiled_eligible(gout, in1, in2, gin1, gin2, B, C, H, W, md)) {
        e = corr2d_bwd_tiled(gout, in1, in2, gin1, gin2, B, C, H, W, as_stream(stream));
        if (e != cudaSuccess) return cuda_fail(e, "b200_corr2d_bwd(tiled)");
        return B200_OK;
    }
    switch (md) {
        case 1: e = launch_corr2d_bwd<1>(gout, in1, in2, gin1, gin2, B, C, H, W, as_stream(stream)); break;
        case 2: e = launch_corr2d_bwd<2>(gout, in1, in2, gin1, gin2, B, C, H, W, as_stream(stream)); break;
        case 3: e = launch_corr2d_bwd<3>(gout, in1, in2, gin1, gin2, B, C, H, W, as_stream(stream)); break;
        default: e = launch_corr2d_bwd<4>(gout, in1, in2, gin1, gin2, B, C, H, W, as_stream(stream)); break;
    }
    if (e != cudaSuccess) return cuda_fail(e, "b200_corr2d_bwd");
    return B200_OK;
}
