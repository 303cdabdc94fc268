// corr2d_bwd_tiled.cu — a2 (SURVEY §8f rank 4): backward of the 81-channel correlation, md = 4, register-tiled.
//
// Replaces correlation_backward_kernel.cu:4-89 (one thread per input element, 81 uncoalesced taps each) and the first,
// correct-only kernel of corr2d.cu (0.67 FMA per shared-memory load).  Both gradients are one contraction
//     gin[c, y, x] = (1/C) * sum_{dy,dx} G[(dy,dx)](y, x) * partner[y + sy*dy, x + sx*dx, c]
// with  gin1: G = grad_out at the output pixel itself,             partner = in2, (sy, sx) = (+1, +1)
//       gin2: G = grad_out read at (y - dy, x - dx) (pre-shifted),  partner = in1, (sy, sx) = (-1, -1),
// so ONE kernel serves both: the grad_out tile is staged in shared memory already shifted for gin2, and gin2 walks the
// partner halo with mirrored offsets.
//
//   tile   8 rows x 32 px of the gradient, 32 channels per chunk; 128 threads: lane = (channel group of 8, 8-px strip,
//          row parity), warp = row pair.  A thread owns 8 px x 8 channels = 64 accumulators.
//   smem   partner halo [16][40][32 ch] (82 KB per chunk) + the grad_out planes of ONE row offset [9][8][32], double-buffered
//          (2 x 9 KB): the next row offset's planes stream in by cp.async under the current one's FMAs, and at 100 KB two
//          CTAs share an SM, so one CTA's staging overlaps the other's arithmetic; a pixel's
//          32 channels are one 128-byte line, its 16-byte chunks XOR-swizzled with bit 3 of the column so the eight
//          lanes of an LDS.128 phase (4 channel groups x 2 neighbouring strips) hit eight different bank groups.
//   loop   per row offset: the 72 grad_out values (9 column offsets x 8 px) go to registers; then 16 halo columns, each
//          2 x LDS.128 (8 channels) feeding every (pixel, column offset) pair that lands on it: 576 FMAs per 50 LDS.128
//          — the operand ratio of the forward kernels' first TMA generation.
//   out    NCHW like the reference (wrapper.py:34-35 permutes): 8 contiguous pixels per channel = two 16-byte stores.
#include "common.cuh"

namespace b200 {

constexpr int BT_TH = 8, BT_TW = 32, BT_P = 8, BT_CC = 32, BT_CB = 8, BT_MD = 4, BT_ND = 9;
constexpr int BT_HR = BT_TH + 2 * BT_MD, BT_HC = BT_TW + 2 * BT_MD;          // 16 x 40 halo
constexpr int BT_THREADS = 128;
constexpr int BT_G_FLOATS = BT_ND * BT_TH * BT_TW;                           // grad_out planes of one row offset: 2304
constexpr int BT_H_FLOATS = BT_HR * BT_HC * BT_CC;                           // 20480
constexpr size_t BT_SMEM = (size_t)(2 * BT_G_FLOATS + BT_H_FLOATS) * sizeof(float);   // 100 KB: two CTAs per SM

template <int WHICH>   // 1: grad wrt in1 (partner = in2), 2: grad wrt in2 (partner = in1)
__global__ void __launch_bounds__(BT_THREADS, 2)
corr2d_bwd_tiled_kernel(const float* __restrict__ gout, const float* __restrict__ partner, float* __restrict__ gin,
                        int C, int H, int W, int tiles_x, int tiles_y) {
    extern __shared__ __align__(16) float bt_smem[];
    float* s_g = bt_smem;                                // 2 x [9][8][32]: double-buffered per row offset, pre-shifted for WHICH = 2
    float* s_h = bt_smem + 2 * BT_G_FLOATS;                  // [16][40] pixels x 32 channels, 16-byte chunks swizzled
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cg = lane & 3, strip = (lane >> 2) & 3, r = warp * 2 + (lane >> 4);
    int tile = blockIdx.x;
    const int tx = tile % tiles_x; tile /= tiles_x;
    const int ty = tile % tiles_y, b = tile / tiles_y;
    const int y0 = ty * BT_TH, x0 = tx * BT_TW;
    const size_t plane = (size_t)H * W;

    // grad_out planes of ONE partner row offset (9 planes x 8 rows x 32 px) into buffer `buf`; slot pdx holds plane
    // t(pdy, pdx), for WHICH = 2 read at (y - dy, x - dx).  cp.async with zero fill outside the image.
    auto stage_g = [&](int pdy, int buf) {
        float* dst = s_g + buf * BT_G_FLOATS;
        if (WHICH == 1) {                                // 16-byte pieces: x0 and W are multiples of 4
            for (int e = tid; e < BT_G_FLOATS / 4; e += BT_THREADS) {
                const int i = (e % (BT_TW / 4)) * 4, rr = (e / (BT_TW / 4)) % BT_TH, pdx = e / ((BT_TW / 4) * BT_TH);
                const int t = pdy * BT_ND + pdx, gy = y0 + rr, gx = x0 + i;
                const bool in = gy < H && gx < W;
                cp_async16(dst + e * 4, gout + ((size_t)b * BT_ND * BT_ND + t) * plane + (in ? (size_t)gy * W + gx : 0), in);
            }
        } else {                                         // shifted by the plane's own displacement: 4-byte pieces
            for (int e = tid; e < BT_G_FLOATS; e += BT_THREADS) {
                const int i = e % BT_TW, rr = (e / BT_TW) % BT_TH, pdx = e / (BT_TW * BT_TH);
                const int dyi = BT_ND - 1 - pdy, dxi = BT_ND - 1 - pdx, t = dyi * BT_ND + dxi;
                const int gy = y0 + rr - (dyi - BT_MD), gx = x0 + i - (dxi - BT_MD);
                const bool in = gy >= 0 && gy < H && gx >= 0 && gx < W;
                cp_async4(dst + e, gout + ((size_t)b * BT_ND * BT_ND + t) * plane + (in ? (size_t)gy * W + gx : 0), in);
            }
        }
    };

    const float inv_scale = (float)C;
    for (int c0 = 0; c0 < C; c0 += BT_CC) {
        __syncthreads();                                 // the previous chunk's readers are done with both buffers
        // partner halo, NHWC: 16-byte chunks (4 channels) by cp.async, zero fill outside the image / beyond C
        constexpr int HCHUNKS = BT_HR * BT_HC * (BT_CC / 4);
        for (int e = tid; e < HCHUNKS; e += BT_THREADS) {
            const int ch = e % (BT_CC / 4), col = (e / (BT_CC / 4)) % BT_HC, row = e / ((BT_CC / 4) * BT_HC);
            const int gy = y0 + row - BT_MD, gx = x0 + col - BT_MD, c = c0 + 4 * ch;
            const bool in = gy >= 0 && gy < H && gx >= 0 && gx < W && c < C;          // C % 4 == 0: a chunk is in or out whole
            cp_async16(s_h + ((row * BT_HC + col) * BT_CC) + ((ch ^ ((col >> 3) & 1)) << 2),
                       partner + (in ? (((size_t)b * H + gy) * W + gx) * C + c : 0), in);
        }
        stage_g(0, 0);
        cp_async_commit();

        float acc[BT_P][BT_CB];
#pragma unroll
        for (int j = 0; j < BT_P; ++j)
#pragma unroll
            for (int c = 0; c < BT_CB; ++c) acc[j][c] = 0.0f;

#pragma unroll 1
        for (int pdy = 0; pdy < BT_ND; ++pdy) {          // partner row offset inside the halo
            const int buf = pdy & 1;
            if (pdy + 1 < BT_ND) {                       // next row offset's planes stream in under this one's FMAs
                stage_g(pdy + 1, buf ^ 1);
                cp_async_commit();
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncthreads();
            // the 72 grad_out values of this row offset (9 column offsets x 8 px) go to registers
            float g[BT_ND][BT_P];
            const float* gb = s_g + buf * BT_G_FLOATS;
#pragma unroll
            for (int pdx = 0; pdx < BT_ND; ++pdx) {
                const float4* gp = reinterpret_cast<const float4*>(gb + (pdx * BT_TH + r) * BT_TW + strip * BT_P);
                const float4 a = gp[0], c = gp[1];
                g[pdx][0] = a.x; g[pdx][1] = a.y; g[pdx][2] = a.z; g[pdx][3] = a.w;
                g[pdx][4] = c.x; g[pdx][5] = c.y; g[pdx][6] = c.z; g[pdx][7] = c.w;
            }
            const float* hrow = s_h + (size_t)((r + pdy) * BT_HC + strip * BT_P) * BT_CC;
#pragma unroll
            for (int cc = 0; cc < BT_P + 2 * BT_MD; ++cc) {      // halo column strip*8 + cc
                const int sw = ((strip * BT_P + cc) >> 3) & 1;
                const float4 f0 = *reinterpret_cast<const float4*>(hrow + cc * BT_CC + (((2 * cg) ^ sw) << 2));
                const float4 f1 = *reinterpret_cast<const float4*>(hrow + cc * BT_CC + (((2 * cg + 1) ^ sw) << 2));
                const float f[BT_CB] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
#pragma unroll
                for (int j = 0; j < BT_P; ++j) {
                    const int pdx = cc - j;                       // compile time after unrolling
                    if (pdx < 0 || pdx >= BT_ND) continue;
#pragma unroll
                    for (int c = 0; c < BT_CB; ++c) acc[j][c] = fmaf(g[pdx][j], f[c], acc[j][c]);
                }
            }
            __syncthreads();                             // buffer `buf` is free for the row offset after next
        }

        const int y = y0 + r, x = x0 + strip * BT_P;
        if (y < H) {
#pragma unroll
            for (int c = 0; c < BT_CB; ++c) {
                const int ch = c0 + cg * BT_CB + c;
                if (ch >= C) continue;
                float* o = gin + ((size_t)b * C + ch) * plane + (size_t)y * W + x;
#pragma unroll
                for (int m = 0; m < BT_P / 4; ++m)
                    if (x + 4 * m < W)                            // W % 4 == 0: a float4 is inside or outside as a whole
                        *reinterpret_cast<float4*>(o + 4 * m) =
                            make_float4(__fdiv_rn(acc[4 * m][c], inv_scale), __fdiv_rn(acc[4 * m + 1][c], inv_scale),
                                        __fdiv_rn(acc[4 * m + 2][c], inv_scale), __fdiv_rn(acc[4 * m + 3][c], inv_scale));
            }
        }
    }
}

bool corr2d_bwd_tiled_eligible(const float* gout, const float* in1, const float* in2, const float* g1, const float* g2,
                               int B, int C, int H, int W, int md) {
    if (md != BT_MD || (C & 3) || (W & 3)) return false;
    const uintptr_t bits = reinterpret_cast<uintptr_t>(gout) | reinterpret_cast<uintptr_t>(in1) | reinterpret_cast<uintptr_t>(in2) |
                           reinterpret_cast<uintptr_t>(g1) | reinterpret_cast<uintptr_t>(g2);
    if (bits & 15) return false;
    const int64_t tiles = (int64_t)B * ceil_div(W, BT_TW) * ceil_div(H, BT_TH);
    return tiles > 0 && tiles < 0x7fffffff;
}

cudaError_t corr2d_bwd_tiled(const float* gout, const float* in1, const float* in2, float* g1, float* g2, int B, int C, int H,
                             int W, cudaStream_t st) {
    const int tiles_x = ceil_div(W, BT_TW), tiles_y = ceil_div(H, BT_TH);
    const int grid = B * tiles_x * tiles_y;
    cudaError_t e = cudaFuncSetAttribute(corr2d_bwd_tiled_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BT_SMEM);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(corr2d_bwd_tiled_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BT_SMEM);
    if (e != cudaSuccess) return e;
    corr2d_bwd_tiled_kernel<1><<<grid, BT_THREADS, BT_SMEM, st>>>(gout, in2, g1, C, H, W, tiles_x, tiles_y);
    corr2d_bwd_tiled_kernel<2><<<grid, BT_THREADS, BT_SMEM, st>>>(gout, in1, g2, C, H, W, tiles_x, tiles_y);
    return cudaGetLastError();
}

}  // namespace b200
