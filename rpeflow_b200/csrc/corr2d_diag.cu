// corr2d_diag.cu — a1, wrapper-level call on NCHW maps (md = 4), second generation of corr2d_nchw.cu.
//
// corr2d_nchw.cu is bound by the shared-memory data pipe (ncu: l1tex data-pipe wavefronts 72-76 % of peak, FMA pipe
// 22-25 %): a thread that owns (row y, row shift dy, 8 pixels x 9 column shifts) loads 24 operand floats for 72 FMAs.
// This kernel raises the FMAs per loaded float from 3.0 to 4.15 with a DIAGONAL register tile: the outputs
// (y, dy) and (y+1, dy-1) read the same in2 row y+dy, so one thread owns both — 2 rows x 6 pixels x 9 column shifts =
// 108 accumulators from 12 in1 + 14 in2 floats.  Same operands, same fp32 FMA order over channels as before.
//
//   * tile = 8 rows x 48 px (240 = 5 x 48: no ragged column at level 1); lane = (strip of 6 px, row pair), row pair
//     fastest.  Rows are staged with a pitch of 60 floats for BOTH boxes: a lane's LDS.64 addresses are
//     (2*rp + const)*60 + 6*strip + 2*j floats, i.e. banks 24*rp + 6*strip (+const) mod 32 — the 16 lanes of a
//     half-warp (4 strips x 4 row pairs) cover all 32 banks exactly once: conflict-free without swizzle.
//   * warp o = 1..8 owns in2 halo row offset o: outputs (row 2rp, dy index o) and (row 2rp+1, dy index o-1).  The two
//     ends of the diagonal have one output only: warp 8 -> (row 2rp, dy index 0), warp 9 -> (row 2rp+1, dy index 8);
//     they are half-work warps placed on different schedulers (warp % 4), the producer sits on a third.
//   * FFMA2 pairs two column shifts of one pixel exactly as in corr2d_nchw.cu (every in2 pair is an LDS.64 result).
//   * 4-stage mbarrier ring of 8-channel TMA boxes (60 x 8 and 60 x 16 px, zero fill outside the image = the
//     reference's padding, correlation_forward_kernel.cu:36-41).
//   * epilogue: 6 px = 24 bytes per (row, column shift): one 16-byte and one 8-byte streaming store, order chosen by
//     the strip's parity so both are naturally aligned; the 8 strips of a row fill 192 contiguous bytes.
#include "sm100_async.cuh"

namespace b200 {

constexpr int D_P = 6, D_NS = 8, D_TW = D_P * D_NS, D_TH = 8, D_MD = 4, D_ND = 2 * D_MD + 1;
constexpr int D_PITCH = 60;                      // floats; 2*pitch = 24 (mod 32) banks between row pairs
constexpr int D_HR = D_TH + 2 * D_MD;            // 16 halo rows
constexpr int D_CC = 8;                          // channels per stage
constexpr int D_B_CH = D_HR * D_PITCH * 4;       // 3840 bytes per channel of the in2 halo
constexpr int D_A_CH = D_TH * D_PITCH * 4;       // 1920 bytes per channel of the in1 tile
constexpr int D_B_BYTES = D_CC * D_B_CH, D_A_BYTES = D_CC * D_A_CH;
constexpr int D_STAGE = D_B_BYTES + D_A_BYTES;   // 46080
constexpr int D_NSTAGE = 4;
constexpr int D_CONSUMERS = D_ND + 1;            // 8 diagonal warps + 2 end-of-diagonal warps
constexpr int D_THREADS = (D_CONSUMERS + 1) * 32;
constexpr size_t D_SMEM = (size_t)D_NSTAGE * D_STAGE + 1024 + 64;
static_assert(D_B_BYTES % 128 == 0 && D_STAGE % 128 == 0, "TMA destinations stay 128-byte aligned");
static_assert(D_TW + 2 * D_MD <= D_PITCH, "the halo row fits the pitch");

struct DAcc {                                    // the 9 column shifts of one pixel: 4 packed pairs + 1 scalar
    u64 p[4];
    float s;
};

// One stage (8 channels) for one consumer thread.  pa: shared address of the thread's first in1 pixel (row 0 of its
// rows) in channel 0 of the stage, pb: of its first in2 pixel.  ROWS = 2: the diagonal pair, ROWS = 1: a diagonal end.
template <int ROWS>
__device__ __forceinline__ void corr2d_diag_consume(DAcc (&acc)[ROWS][D_P], uint32_t pa, uint32_t pb) {
#pragma unroll
    for (int c = 0; c < D_CC; ++c) {
        float a[ROWS][D_P], b[D_P + 2 * D_MD];
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
#pragma unroll
            for (int m = 0; m < D_P / 2; ++m) {
                const float2 v = lds_v2(pa + (D_B_BYTES + c * D_A_CH + r * D_PITCH * 4 + m * 8));
                a[r][2 * m] = v.x; a[r][2 * m + 1] = v.y;
            }
#pragma unroll
        for (int m = 0; m < (D_P + 2 * D_MD) / 2; ++m) {
            const float2 v = lds_v2(pb + (c * D_B_CH + m * 8));
            b[2 * m] = v.x; b[2 * m + 1] = v.y;
        }
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
#pragma unroll
            for (int i = 0; i < D_P; ++i) {
                const u64 aa = pack2(a[r][i], a[r][i]);
                const int odd = i & 1;               // strips start at even pixels
#pragma unroll
                for (int q = 0; q < 4; ++q) fma2(acc[r][i].p[q], aa, pack2(b[i + odd + 2 * q], b[i + odd + 2 * q + 1]));
                acc[r][i].s = fmaf(a[r][i], odd ? b[i] : b[i + 8], acc[r][i].s);
            }
    }
}

// Stores one output row of a thread (6 px x 9 column shifts) and clears the accumulators.
__device__ __forceinline__ void corr2d_diag_store(DAcc (&acc)[D_P], float* __restrict__ o, size_t plane, float inv_c,
                                                  float slope, bool even, bool ok4, bool ok2) {
    float lo[D_P][4], hi[D_P][4];
#pragma unroll
    for (int i = 0; i < D_P; ++i)
#pragma unroll
        for (int q = 0; q < 4; ++q) unpack2(acc[i].p[q], lo[i][q], hi[i][q]);
    float* p4 = o + (even ? 0 : 2);
    float* p2 = o + (even ? 4 : 0);
#pragma unroll
    for (int d = 0; d < D_ND; ++d) {
        float v[D_P];
#pragma unroll
        for (int i = 0; i < D_P; ++i) {
            float t;
            if ((i & 1) == 0) t = d == 8 ? acc[i].s : ((d & 1) ? hi[i][d >> 1] : lo[i][d >> 1]);
            else              t = d == 0 ? acc[i].s : ((d & 1) ? lo[i][(d - 1) >> 1] : hi[i][(d - 1) >> 1]);
            t *= inv_c;
            v[i] = fmaxf(t, t * slope);              // leaky_relu epilogue (slope 1 = none): RPEFlow_core.py:362
        }
        const float4 f4 = even ? make_float4(v[0], v[1], v[2], v[3]) : make_float4(v[2], v[3], v[4], v[5]);
        const float2 f2 = even ? make_float2(v[4], v[5]) : make_float2(v[0], v[1]);
        if (ok4) __stcs(reinterpret_cast<float4*>(p4), f4);
        if (ok2) __stcs(reinterpret_cast<float2*>(p2), f2);
        p4 += plane;
        p2 += plane;
    }
#pragma unroll
    for (int i = 0; i < D_P; ++i) {
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[i].p[q] = 0ull;
        acc[i].s = 0.0f;
    }
}

template <int ROWS>
__device__ __forceinline__ void corr2d_diag_consumer(uint32_t base, uint32_t bar_full, uint32_t bar_empty, float* __restrict__ out,
                                                     int H, int W, int tiles_x, int per_img, int num_tiles, int nchunks,
                                                     float inv_c, float slope, int warp, int lane) {
    const int rp = lane & 3, strip = lane >> 2;
    // in2 halo row offset o of this warp; first in1 row of the thread inside its row pair; dy index of acc[0]
    const int o = warp < 8 ? warp + 1 : (warp == 8 ? 0 : 9);
    const int arow = 2 * rp + (warp == 9 ? 1 : 0);
    const int dy0 = warp == 9 ? 8 : o;            // full warps: acc[0] -> dy index o, acc[1] -> dy index o - 1
    const uint32_t pa = base + (uint32_t)((arow * D_PITCH + strip * D_P) * 4);
    const uint32_t pb = base + (uint32_t)(((2 * rp + o) * D_PITCH + strip * D_P) * 4);
    const bool even = (strip & 1) == 0;

    DAcc acc[ROWS][D_P];
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
        for (int i = 0; i < D_P; ++i) {
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[r][i].p[q] = 0ull;
            acc[r][i].s = 0.0f;
        }

    const size_t plane = (size_t)H * W;
    int s = 0;
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (int ch = 0; ch < nchunks; ++ch) {
            mbar_wait(bar_full + 8 * s, ph);                      // TMA bytes have landed
            corr2d_diag_consume<ROWS>(acc, pa + s * D_STAGE, pb + s * D_STAGE);
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty + 8 * s);        // this warp is done with the slot
            if (++s == D_NSTAGE) { s = 0; ph ^= 1u; }
        }
        const int b = tile / per_img, r = tile - b * per_img;
        const int ty = r / tiles_x, tx = r - ty * tiles_x;
        const int x = tx * D_TW + strip * D_P;
        const bool ok4 = even ? x < W : x + 2 < W, ok2 = even ? x + 4 < W : x < W;   // W % 4 == 0: pieces are in or out whole
#pragma unroll
        for (int rr = 0; rr < ROWS; ++rr) {
            const int y = ty * D_TH + arow + rr;
            float* op = out + ((size_t)b * (D_ND * D_ND) + (size_t)(dy0 - rr) * D_ND) * plane + (size_t)y * W + x;
            const bool yok = y < H;
            corr2d_diag_store(acc[rr], op, plane, inv_c, slope, even, yok && ok4, yok && ok2);
        }
    }
}

__global__ void __launch_bounds__(D_THREADS, 1)
corr2d_fwd_diag_kernel(const __grid_constant__ CUtensorMap map1, const __grid_constant__ CUtensorMap map2,
                       float* __restrict__ out, int C, int H, int W, int tiles_x, int tiles_y, int num_tiles, float inv_c, float slope) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_full = base + D_NSTAGE * D_STAGE;
    const uint32_t bar_empty = bar_full + 8 * D_NSTAGE;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < D_NSTAGE; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, D_CONSUMERS);
        }
        mbar_init_fence();
    }
    __syncthreads();

    const int nchunks = (C + D_CC - 1) / D_CC;
    const int per_img = tiles_x * tiles_y;

    if (warp == D_CONSUMERS) {                                    // ---------------- producer
        if (lane == 0) {
            prefetch_tensormap(&map1);
            prefetch_tensormap(&map2);
            int s = 0;
            uint32_t ph = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int b = tile / per_img, r = tile - b * per_img;
                const int ty = r / tiles_x, tx = r - ty * tiles_x;
                const int y0 = ty * D_TH, x0 = tx * D_TW;
                for (int ch = 0; ch < nchunks; ++ch) {
                    while (!mbar_try(bar_empty + 8 * s, ph ^ 1u)) __nanosleep(64);    // consumers have drained this slot
                    mbar_arrive_expect_tx(bar_full + 8 * s, D_STAGE);
                    // boxes are (x, y, channel, batch); out-of-image pixels and channels >= C arrive as zeros
                    tma_load_4d(base + s * D_STAGE, &map2, x0 - D_MD, y0 - D_MD, ch * D_CC, b, bar_full + 8 * s);
                    tma_load_4d(base + s * D_STAGE + D_B_BYTES, &map1, x0, y0, ch * D_CC, b, bar_full + 8 * s);
                    if (++s == D_NSTAGE) { s = 0; ph ^= 1u; }
                }
            }
        }
        return;
    }
    if (warp < 8)
        corr2d_diag_consumer<2>(base, bar_full, bar_empty, out, H, W, tiles_x, per_img, num_tiles, nchunks, inv_c, slope, warp, lane);
    else
        corr2d_diag_consumer<1>(base, bar_full, bar_empty, out, H, W, tiles_x, per_img, num_tiles, nchunks, inv_c, slope, warp, lane);
}

// ---- host side -------------------------------------------------------------------------------------------------
static bool make_diag_map(CUtensorMap* m, const float* ptr, int B, int C, int H, int W, int box_h) {
    auto enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)C, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4, (cuuint64_t)C * H * W * 4};
    const cuuint32_t box[4] = {(cuuint32_t)D_PITCH, (cuuint32_t)box_h, (cuuint32_t)D_CC, 1u};
    const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(ptr), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Columns computed per useful column for the two tilings; the diagonal kernel is taken unless its 48-px tiles waste
// clearly more of a narrow map than the 32-px tiles of corr2d_nchw.cu do.
bool corr2d_diag_preferred(int W) {
    const double w48 = (double)ceil_div(W, D_TW) * D_TW / W, w32 = (double)ceil_div(W, 32) * 32 / W;
    return w48 <= 1.2 * w32;
}

cudaError_t corr2d_fwd_diag(const float* in1, const float* in2, float* out, int B, int C, int H, int W, float slope,
                            cudaStream_t st) {
    CUtensorMap m1, m2;
    if (!make_diag_map(&m1, in1, B, C, H, W, D_TH) || !make_diag_map(&m2, in2, B, C, H, W, D_HR)) return cudaErrorInvalidValue;
    const int tiles_x = ceil_div(W, D_TW), tiles_y = ceil_div(H, D_TH);
    const int num_tiles = B * tiles_x * tiles_y;
    cudaError_t e = cudaFuncSetAttribute(corr2d_fwd_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)D_SMEM);
    if (e != cudaSuccess) return e;
    const int grid = num_tiles < sm_count() ? num_tiles : sm_count();
    corr2d_fwd_diag_kernel<<<grid, D_THREADS, D_SMEM, st>>>(m1, m2, out, C, H, W, tiles_x, tiles_y, num_tiles, 1.0f / (float)C, slope);
    return cudaGetLastError();
}

}  // namespace b200
