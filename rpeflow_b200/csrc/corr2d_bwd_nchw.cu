// corr2d_bwd_nchw.cu — a2 on NCHW feature maps: the backward of correlation2d(input1, input2, 4) without the
// wrapper's permutes (models/csrc/wrapper.py:68-69 in the forward, :34-35 and autograd's permute backward after it).
//
// The contraction is the one corr2d_bwd_tiled.cu computes,
//     gin[c, y, x] = (1/C) * sum_{dy,dx} G[(dy,dx)](y, x) * partner[c, y + sy*dy, x + sx*dx],
// with grad_out pre-shifted for gin2, and so is the skeleton: 8 x 32 px x 32 channels per tile, 128 threads owning
// 8 px x 8 channels each, 72 grad_out values in registers per row offset, that row offset's planes double-buffered by
// cp.async, two CTAs per SM.  Only the partner halo changes: [32 ch][16 rows][44] planes read straight from NCHW.
//   lanes  lane = (row, 8-px strip), warp = channel group (as corr2d_nchw.cu).  A thread's 16 halo columns of one
//          channel are contiguous: 4 x LDS.128 per (channel, row offset) feed 72 FMAs.  Row pitches of 44 (halo) and 36
//          (grad_out) floats are odd in 16-byte units, so the 8 rows of an LDS.128 phase hit 8 bank groups.
//   order  row offset outer, column offset ascending inner, one fmaf chain from 0, then __fdiv_rn(acc, C): the order of
//          corr2d_bwd_tiled.cu, so wherever b200_corr2d_bwd takes that kernel this one returns the same bits.
//   ALIGNED (W % 4 == 0, all pointers 16-byte aligned): 16-byte cp.async pieces and float4 stores; otherwise 4-byte
//          pieces and scalar stores.  Channels are planes, so C needs no rounding: channels >= C are zero-filled.
// Every address comes from corr2d_bwd_nchw_index.cuh, which tests/corr2d_bwd_nchw_audit.cpp checks on the CPU.
#include "common.cuh"
#include "corr2d_bwd_nchw_index.cuh"

namespace b200 {

template <int WHICH, bool ALIGNED>   // WHICH 1: grad wrt in1 (partner = in2), 2: grad wrt in2 (partner = in1)
__global__ void __launch_bounds__(bn::THREADS, 2)
corr2d_bwd_nchw_kernel(const float* __restrict__ gout, const float* __restrict__ partner, float* __restrict__ gin,
                       int C, int H, int W, int tiles_x, int tiles_y) {
    using namespace bn;
    extern __shared__ __align__(16) float bn_smem[];
    float* s_g = bn_smem;                        // 2 x [9][8][36]: double-buffered per row offset
    float* s_h = bn_smem + 2 * G_FLOATS;         // [32][16][44]
    const int tid = threadIdx.x;
    const Tile t = tile_of(blockIdx.x, tiles_x, tiles_y);

    auto stage_g = [&](int pdy, int buf) {
        float* dst = s_g + buf * G_FLOATS;
#pragma unroll 1
        for (int e = tid; e < grad_pieces<WHICH, ALIGNED>(); e += THREADS) {
            const Piece p = grad_piece<WHICH, ALIGNED>(e, pdy, t, H, W);
            if (grad_width<WHICH, ALIGNED>() == 4) cp_async16(dst + p.dst, gout + p.src, p.in);
            else                                   cp_async4(dst + p.dst, gout + p.src, p.in);
        }
    };

    const float inv_scale = (float)C;
    for (int c0 = 0; c0 < C; c0 += CC) {
        __syncthreads();                         // the previous chunk's readers are done with both buffers
#pragma unroll 1
        for (int e = tid; e < halo_pieces<ALIGNED>(); e += THREADS) {
            const Piece p = halo_piece<ALIGNED>(e, t, c0, C, H, W);
            if (ALIGNED) cp_async16(s_h + p.dst, partner + p.src, p.in);
            else         cp_async4(s_h + p.dst, partner + p.src, p.in);
        }
        stage_g(0, 0);
        cp_async_commit();

        float acc[P][CB];
#pragma unroll
        for (int j = 0; j < P; ++j)
#pragma unroll
            for (int c = 0; c < CB; ++c) acc[j][c] = 0.0f;

#pragma unroll 1
        for (int pdy = 0; pdy < ND; ++pdy) {
            const int buf = pdy & 1;
            if (pdy + 1 < ND) {                  // next row offset's planes stream in under this one's FMAs
                stage_g(pdy + 1, buf ^ 1);
                cp_async_commit();
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncthreads();
            float g[ND][P];
            const float* gb = s_g + buf * G_FLOATS;
#pragma unroll
            for (int pdx = 0; pdx < ND; ++pdx) {
                const float4* gp = reinterpret_cast<const float4*>(gb + grad_read(tid, pdx));
                const float4 a = gp[0], c = gp[1];
                g[pdx][0] = a.x; g[pdx][1] = a.y; g[pdx][2] = a.z; g[pdx][3] = a.w;
                g[pdx][4] = c.x; g[pdx][5] = c.y; g[pdx][6] = c.z; g[pdx][7] = c.w;
            }
#pragma unroll
            for (int c = 0; c < CB; ++c) {
                const float4* hp = reinterpret_cast<const float4*>(s_h + halo_read(tid, c, pdy));
                // two halves of 8 columns keep 8 halo values live; per accumulator the column offsets still ascend
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const float4 f0 = hp[2 * half], f1 = hp[2 * half + 1];
                    const float f[P] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
#pragma unroll
                    for (int k = 0; k < P; ++k) {
                        const int cc = half * P + k;              // halo column strip*8 + cc
#pragma unroll
                        for (int j = 0; j < P; ++j) {
                            const int pdx = cc - j;               // compile time after unrolling
                            if (pdx < 0 || pdx >= ND) continue;
                            acc[j][c] = fmaf(g[pdx][j], f[k], acc[j][c]);
                        }
                    }
                }
            }
            __syncthreads();                     // buffer `buf` is free for the row offset after next
        }

        const int y = t.y0 + thread_row(tid), x = t.x0 + thread_strip(tid) * P;
        if (y < H) {
#pragma unroll
            for (int c = 0; c < CB; ++c) {
                const int ch = c0 + thread_cg(tid) * CB + c;
                if (ch >= C) continue;
                float* o = gin + out_offset(t.b, ch, y, x, C, H, W);
                if (ALIGNED) {
#pragma unroll
                    for (int m = 0; m < P / 4; ++m)
                        if (x + 4 * m < W)       // W % 4 == 0: a float4 is inside or outside as a whole
                            *reinterpret_cast<float4*>(o + 4 * m) =
                                make_float4(__fdiv_rn(acc[4 * m][c], inv_scale), __fdiv_rn(acc[4 * m + 1][c], inv_scale),
                                            __fdiv_rn(acc[4 * m + 2][c], inv_scale), __fdiv_rn(acc[4 * m + 3][c], inv_scale));
                } else {
#pragma unroll
                    for (int j = 0; j < P; ++j)
                        if (x + j < W) o[j] = __fdiv_rn(acc[j][c], inv_scale);
                }
            }
        }
    }
}

template <bool ALIGNED>
static cudaError_t corr2d_bwd_nchw(const float* gout, const float* in1, const float* in2, float* g1, float* g2, int C,
                                   int H, int W, int grid, int tiles_x, int tiles_y, cudaStream_t st) {
    cudaError_t e;
    if (g1) {
        e = cudaFuncSetAttribute(corr2d_bwd_nchw_kernel<1, ALIGNED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bn::SMEM);
        if (e != cudaSuccess) return e;
        corr2d_bwd_nchw_kernel<1, ALIGNED><<<grid, bn::THREADS, bn::SMEM, st>>>(gout, in2, g1, C, H, W, tiles_x, tiles_y);
    }
    if (g2) {
        e = cudaFuncSetAttribute(corr2d_bwd_nchw_kernel<2, ALIGNED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bn::SMEM);
        if (e != cudaSuccess) return e;
        corr2d_bwd_nchw_kernel<2, ALIGNED><<<grid, bn::THREADS, bn::SMEM, st>>>(gout, in1, g2, C, H, W, tiles_x, tiles_y);
    }
    return cudaGetLastError();
}

}  // namespace b200

extern "C" int b200_corr2d_bwd_nchw(const float* gout, const float* in1, const float* in2, float* gin1, float* gin2,
                                    int B, int C, int H, int W, int md, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE(B >= 0 && C >= 1 && H >= 1 && W >= 1, "b200_corr2d_bwd_nchw: bad sizes B=%d C=%d H=%d W=%d", B, C, H, W);
    B200_REQUIRE(md >= 1 && md <= 64, "b200_corr2d_bwd_nchw: max_displacement must be in [1,64] (got %d)", md);
    const bool empty = B == 0 || !(gin1 || gin2);
    B200_REQUIRE(empty || (gout && in1 && in2), "b200_corr2d_bwd_nchw: null pointer");   // empty calls carry null pointers
    const int64_t tiles_x = ceil_div(W, bn::TW), tiles_y = ceil_div(H, bn::TH);       // one CTA per tile on grid.x
    B200_REQUIRE(tiles_x * tiles_y <= 0x7fffffff / (B > 0 ? B : 1), "b200_corr2d_bwd_nchw: B*H*W exceeds the grid limit");
    if (md != bn::MD) {
        set_error("b200_corr2d_bwd_nchw: needs md=4 (got %d; permute to NHWC and call b200_corr2d_bwd)", md);
        return B200_ENOSUP;
    }
    if (empty) return B200_OK;
    const uintptr_t bits = reinterpret_cast<uintptr_t>(gout) | reinterpret_cast<uintptr_t>(in1) | reinterpret_cast<uintptr_t>(in2) |
                           reinterpret_cast<uintptr_t>(gin1) | reinterpret_cast<uintptr_t>(gin2);
    const bool aligned = W % 4 == 0 && (bits & 15) == 0;
    const int grid = (int)(B * tiles_x * tiles_y);
    const cudaError_t e = aligned
        ? corr2d_bwd_nchw<true>(gout, in1, in2, gin1, gin2, C, H, W, grid, (int)tiles_x, (int)tiles_y, as_stream(stream))
        : corr2d_bwd_nchw<false>(gout, in1, in2, gin1, gin2, C, H, W, grid, (int)tiles_x, (int)tiles_y, as_stream(stream));
    if (e != cudaSuccess) return cuda_fail(e, "b200_corr2d_bwd_nchw");
    return B200_OK;
}
