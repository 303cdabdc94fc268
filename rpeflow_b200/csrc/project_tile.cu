// project_tile.cu — a8 (+ a7 by-product), second generation: project_feat_with_nn_corr with ONE pass over feat_2d.
//
// models/utils.py:297-317 needs every feature map twice: grid_sample at the projected points (S = bilinear(feat_2d, xy))
// and the per-pixel correlation mean_c(S[c, nn[p]] * feat_2d[c, p]).  The first generation (gather.cu) did that in two
// kernels — a per-point sampler whose 4-byte taps touch nearly every 32-byte sector of the map (8-ish pixels per point),
// then a per-pixel pass that streams the map again — so the map crossed HBM twice (2.9 GB of traffic for 1.9 GB of
// algorithmic bytes on the level-1 decoder call) and both kernels sat at 36-57 % of DRAM peak, latency-bound.
//
// Here a persistent CTA owns a 60 x 32 pixel tile of one sample, and a producer warp streams the tile plus a 4-pixel
// halo, 4 channels at a time, through a TMA/mbarrier ring (4-D boxes over the NCHW map; out-of-image pixels and
// channels arrive as zeros = grid_sample's zero padding).  While a chunk is resident the consumers do both jobs:
//   * pixel job: the nearest point of a pixel lies within a few pixels of it, so its four bilinear taps are almost always
//     inside the resident window: S is re-blended from shared memory (same operation order as the point job, so the value
//     is bit-identical to the sampled tensor) and multiplied into the pixel's own feature: 5 LDS + 6 FP ops per
//     (pixel, channel), no global traffic; cheaper still when the point is one of the tile's own (next item): its S is
//     then read from the chunk's table, one LDS.128 per pixel.  A pixel whose taps leave the window (sparse clouds, far
//     outliers) is left to project_far_pixels_kernel, which reads everything from global memory afterwards (correct for
//     any input, slow only where it happens; nothing with DRAM latency sits inside the chunk loop);
//   * point job: the points whose top-left tap lies in this tile (binned per sample by project_bin_kernel) are sampled
//     from the same window into the chunk's shared-memory table and into point-major rows S[b,n,:] (one 16-byte store per
//     point and chunk: whole sectors, where
//     4-byte stores into the channel-first tensor left partially written sectors that L2 evicted and re-fetched);
//     project_rows_to_cf_kernel then transposes the rows into the [B,C2,N] tensor grid_sample_wrapper(feat_2d, xy) returns.
// 60 x 32 tiles: halo rows are re-read from HBM, not from L2 — a streaming kernel turns the L2 over faster than the
// neighbouring tile comes by (ncu: 1.9 GB read for a 0.98 GB map with 64 x 16 tiles, 1.2-1.3 GB with these).
// The feat_3d copy to pixels (output channels 3..) stays the gather kernel of gather.cu, fed by point-major rows T.
#include "project_common.cuh"
#include "sm100_async.cuh"

namespace b200 {

// 15 consumer warps + the producer warp = 16 warps: 128 registers per thread (a 17th warp would cap them at 96: registers
// are handed out to four warps at a time).  480 threads = 15 pixel quads x 32 rows: a thread owns four consecutive pixels
// of one row, so its own features are one LDS.128 per channel and its outputs 16-byte stores; 60 divides the map widths
// of the 960- and 1920-wide pyramids (240, 120, 60; 480).
constexpr int PT_TW = 60, PT_TH = 32, PT_HALO = 4;
constexpr int PT_WW = PT_TW + 2 * PT_HALO, PT_WH = PT_TH + 2 * PT_HALO;        // resident window: 68 x 40 pixels (272-byte rows)
constexpr int PT_CC = 4;                                                       // channels per stage
constexpr int PT_CH_BYTES = PT_WW * PT_WH * 4;                                 // 10880
constexpr int PT_STAGE = PT_CC * PT_CH_BYTES;                                  // 43520
constexpr int PT_NSTAGE = 4;
constexpr int PT_CONSUMERS = 480, PT_THREADS = PT_CONSUMERS + 32;
constexpr int PT_QX = PT_TW / 4;                                               // 15 quads per tile row
constexpr int PT_PPT = 2, PT_TABLE = PT_PPT * PT_CONSUMERS;                    // points a tile's table holds (two per thread)
constexpr int PT_SBUF = PT_TABLE * PT_CC * 4;                                  // one chunk's table: S[point][4 channels]
constexpr size_t PT_SMEM = (size_t)PT_NSTAGE * PT_STAGE + 2 * PT_SBUF + 1024 + 64;
constexpr int PT_MAX_TILES = 4095;                                             // per sample: the binning histogram lives in shared memory
static_assert(PT_STAGE % 128 == 0, "TMA destinations stay 128-byte aligned");
static_assert(PT_QX * PT_TH == PT_CONSUMERS, "one quad per consumer thread");

// ---- bilinear taps as (x0, y0) + weights: the arithmetic of decoder_common.cuh::make_taps-------------------------------
struct TapXY {
    int x0, y0;                  // top-left tap; -2^30 when the coordinate is not finite (all taps invalid)
    float w00, w01, w10, w11;
};
__device__ __forceinline__ float pt_renorm(float x, int size) {
    const float sm1 = (float)(size - 1);
    const float g = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, x), sm1), 1.0f);        // 2*x/(size-1) - 1        (models/utils.py:290)
    return __fmul_rn(__fdiv_rn(__fadd_rn(g, 1.0f), 2.0f), sm1);                  // ((g+1)/2)*(size-1)      (grid_sample, align_corners)
}
__device__ __forceinline__ TapXY pt_taps(float x, float y, int H, int W) {
    const float ix = pt_renorm(x, W), iy = pt_renorm(y, H);
    const float fx = floorf(ix), fy = floorf(iy);
    const float wx1 = ix - fx, wy1 = iy - fy, wx0 = (fx + 1.0f) - ix, wy0 = (fy + 1.0f) - iy;
    const bool finite = fabsf(ix) < 1e9f && fabsf(iy) < 1e9f;
    TapXY t;
    t.x0 = finite ? (int)fx : -(1 << 30);
    t.y0 = finite ? (int)fy : -(1 << 30);
    t.w00 = wx0 * wy0; t.w01 = wx1 * wy0; t.w10 = wx0 * wy1; t.w11 = wx1 * wy1;
    return t;
}
// left column first, then right column, summed: the order of gather.cu's two-lane sampler (half_blend + shuffle add)
__device__ __forceinline__ float pt_blend(float f00, float f01, float f10, float f11, float w00, float w01, float w10, float w11) {
    const float l = __fmaf_rn(f10, w10, __fmaf_rn(f00, w00, 0.0f));           // "v = 0; v += f*w" twice, as the sampler compiles
    const float r = __fmaf_rn(f11, w11, __fmaf_rn(f01, w01, 0.0f));
    return __fadd_rn(l, r);
}
__device__ __forceinline__ int pt_tile_of(const TapXY& t, int H, int W, int tiles_x) {
    const int cx = min(max(t.x0, 0), W - 1), cy = min(max(t.y0, 0), H - 1);
    return (cy / PT_TH) * tiles_x + cx / PT_TW;
}

// ---- binning: per sample, the points of every tile (by their top-left tap, clamped into the image) --------------------
// One block per sample.  tile_start[b, 0..tiles] = exclusive prefix of the per-tile counts, list[b, :] = point ids by tile,
// pos[b, n] = rank of point n inside its tile's list.
constexpr int PB_THREADS = 256;
__device__ __forceinline__ void project_bin_block(int b, const float* __restrict__ xy, int* __restrict__ list, int* __restrict__ pos,
                                                  int* __restrict__ tile_start, int N, int H, int W, int tiles_x, int tiles) {
    extern __shared__ int pb_smem[];
    int* count = pb_smem;                 // [tiles + 1]
    int* cursor = pb_smem + tiles + 1;    // [tiles]
    __shared__ int chunk_sum[PB_THREADS];
    const int t = threadIdx.x;
    for (int i = t; i <= tiles; i += PB_THREADS) count[i] = 0;
    __syncthreads();
    const float* X = xy + (size_t)b * 2 * N;
    for (int n = t; n < N; n += PB_THREADS) {
        const TapXY tp = pt_taps(__ldg(X + n), __ldg(X + N + n), H, W);
        atomicAdd(&count[pt_tile_of(tp, H, W, tiles_x)], 1);
    }
    __syncthreads();
    // exclusive scan: each thread owns a run of consecutive tiles
    const int per = (tiles + PB_THREADS - 1) / PB_THREADS;
    const int lo = min(t * per, tiles), hi = min(lo + per, tiles);
    int s = 0;
    for (int i = lo; i < hi; ++i) s += count[i];
    chunk_sum[t] = s;
    __syncthreads();
    if (t == 0) {
        int run = 0;
        for (int i = 0; i < PB_THREADS; ++i) { const int v = chunk_sum[i]; chunk_sum[i] = run; run += v; }
    }
    __syncthreads();
    int run = chunk_sum[t];
    for (int i = lo; i < hi; ++i) { const int v = count[i]; count[i] = run; cursor[i] = run; run += v; }
    __syncthreads();
    if (t == 0) count[tiles] = N;
    __syncthreads();
    int* ts = tile_start + (size_t)b * (tiles + 1);
    for (int i = t; i <= tiles; i += PB_THREADS) ts[i] = count[i];
    int* L = list + (size_t)b * N;
    for (int n = t; n < N; n += PB_THREADS) {
        const TapXY tp = pt_taps(__ldg(X + n), __ldg(X + N + n), H, W);
        const int tile = pt_tile_of(tp, H, W, tiles_x);
        const int p = atomicAdd(&cursor[tile], 1);
        L[p] = n;
        pos[(size_t)b * N + n] = p - count[tile];            // rank of the point inside its tile's list
    }
}

// ---- layout changes between channel-first tensors and point-major rows (32 x 32 tiles through shared memory) -----------
// cf [B,C,N] -> rows [B,N,stride] at column offset col0 (T rows for the feat3d gather)
__device__ __forceinline__ void project_cf_to_rows_block(int bx, int by, int b, const float* __restrict__ cf, float* __restrict__ rows,
                                                         int C, int N, int stride, int col0) {
    __shared__ float tile[32][33];
    const int n0 = bx * 32, c0 = by * 32;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int c = c0 + w * 4 + u, n = n0 + lane;
        tile[w * 4 + u][lane] = (c < C && n < N) ? __ldg(cf + ((size_t)b * C + c) * N + n) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int n = n0 + w * 4 + u, c = c0 + lane;
        if (n < N && c < C) rows[((size_t)b * N + n) * stride + col0 + c] = tile[lane][w * 4 + u];
    }
}
// rows [B,N,stride] -> cf [B,C,N] (the sampled tensor grid_sample_wrapper returns)
__device__ __forceinline__ void project_rows_to_cf_block(int bx, int by, int b, const float* __restrict__ rows, float* __restrict__ cf,
                                                         int C, int N, int stride) {
    __shared__ float tile[32][33];
    const int n0 = bx * 32, c0 = by * 32;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int n = n0 + w * 4 + u, c = c0 + lane;
        tile[w * 4 + u][lane] = (n < N && c < C) ? __ldg(rows + ((size_t)b * N + n) * stride + c) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int c = c0 + w * 4 + u, n = n0 + lane;
        if (c < C && n < N) cf[((size_t)b * C + c) * N + n] = tile[lane][w * 4 + u];
    }
}

// prep launch: the first B blocks bin the points of one sample each (the long pole: started first), the rest transpose
// feat3d into the point-major rows T
__global__ void __launch_bounds__(256)
project_prep_kernel(const float* __restrict__ xy, const float* __restrict__ feat3d, float* __restrict__ trows, int* __restrict__ list,
                    int* __restrict__ pos, int* __restrict__ tile_start, int B, int C3, int N, int H, int W, int tiles_x, int tiles) {
    int blk = blockIdx.x;
    if (blk < B) {
        project_bin_block(blk, xy, list, pos, tile_start, N, H, W, tiles_x, tiles);
        return;
    }
    blk -= B;
    const int nx = (N + 31) / 32, ny = (C3 + 31) / 32;
    const int bx = blk % nx, by = (blk / nx) % ny, b = blk / (nx * ny);
    project_cf_to_rows_block(bx, by, b, feat3d, trows, C3, N, round4(C3), 0);
}

// ---- the tile kernel ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PT_THREADS, 1)
project_tile_kernel(const __grid_constant__ CUtensorMap map, const float* __restrict__ feat2d, const float* __restrict__ xy,
                    const int64_t* __restrict__ nn, const int* __restrict__ list, const int* __restrict__ pos,
                    const int* __restrict__ tile_start, float* __restrict__ out, float* __restrict__ srows, int C2, int C3,
                    int H, int W, int N, int tiles_x, int tiles_y, int num_tiles) {
    constexpr int CH = PT_CH_BYTES, ROW = PT_WW * 4;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sbuf0 = base + PT_NSTAGE * PT_STAGE;           // S of the tile's points for the resident chunk, double-buffered
    const uint32_t bar_full = sbuf0 + 2 * PT_SBUF;
    const uint32_t bar_empty = bar_full + 8 * PT_NSTAGE;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int CW = PT_CONSUMERS / 32;                         // consumer warps

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < PT_NSTAGE; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, CW);
        }
        mbar_init_fence();
    }
    __syncthreads();

    const int nchunks = (C2 + PT_CC - 1) / PT_CC;
    const int per_img = tiles_x * tiles_y;

    if (warp == CW) {                                             // ---------------- producer
        if (lane == 0) {
            prefetch_tensormap(&map);
            int s = 0;
            uint32_t ph = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int b = tile / per_img, r = tile - b * per_img;
                const int ty = r / tiles_x, tx = r - ty * tiles_x;
                for (int ch = 0; ch < nchunks; ++ch) {
                    while (!mbar_try(bar_empty + 8 * s, ph ^ 1u)) __nanosleep(32);
                    mbar_arrive_expect_tx(bar_full + 8 * s, PT_STAGE);
                    tma_load_4d(base + s * PT_STAGE, &map, tx * PT_TW - PT_HALO, ty * PT_TH - PT_HALO, ch * PT_CC, b,
                                bar_full + 8 * s);
                    if (++s == PT_NSTAGE) { s = 0; ph ^= 1u; }
                }
            }
        }
        return;
    }

    // ---------------- consumers: thread = pixel quad q of tile row `row`
    const int t = threadIdx.x;
    const int q = t % PT_QX, row = t / PT_QX;
    const uint32_t ctr = (uint32_t)((row + PT_HALO) * ROW + (4 * q + PT_HALO) * 4);     // own quad inside a channel of the window
    const int HW = H * W;
    const int C2p = (C2 + 3) & ~3;
    int s = 0;
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int b = tile / per_img, r = tile - b * per_img;
        const int ty = r / tiles_x, tx = r - ty * tiles_x;
        const int wx0 = tx * PT_TW - PT_HALO, wy0 = ty * PT_TH - PT_HALO;               // window origin in the image
        const float* Xb = xy + (size_t)b * 2 * N;
        const int x = tx * PT_TW + 4 * q, y = ty * PT_TH + row;
        const bool active = x < W && y < H;                       // W % 4 == 0: a quad is inside or outside as a whole

        // -- pixel set-up: nearest point -> how the pixel gets S[c, nn] while a chunk is resident:
        //    table : the point is among the first 960 of this tile's list: off = byte offset of its S in the chunk's table
        //    taps  : its taps lie inside the window: off = byte offset of the top-left tap in a channel of the window
        //    slow  : neither (sparse clouds, far outliers): skipped here, project_far_pixels_kernel computes the pixel from
        //            global memory afterwards — no global load, hence no DRAM latency, sits inside the chunk loop
        uint32_t off[4];
        float w00[4], w01[4], w10[4], w11[4], acc[4];
        uint32_t taps = 0, slow = 0;
        {
            int j[4] = {0, 0, 0, 0};
            if (active) {
                const longlong2* p2 = reinterpret_cast<const longlong2*>(nn + (size_t)b * HW + (size_t)y * W + x);
                const longlong2 a = __ldg(p2), c = __ldg(p2 + 1);
                const int64_t jj[4] = {a.x, a.y, c.x, c.y};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    int64_t v = jj[i];
                    if (v < 0) v += N;
                    j[i] = (int)(v < 0 ? 0 : (v >= N ? N - 1 : v));
                }
            }
            float X[4], Y[4];
            int pj[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                X[i] = __ldg(Xb + j[i]); Y[i] = __ldg(Xb + N + j[i]);
                pj[i] = __ldg(pos + (size_t)b * N + j[i]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const TapXY tp = pt_taps(X[i], Y[i], H, W);
                const int ox = tp.x0 - wx0, oy = tp.y0 - wy0;
                const bool in_window = ox >= 0 && ox + 1 < PT_WW && oy >= 0 && oy + 1 < PT_WH;
                const bool in_table = pt_tile_of(tp, H, W, tiles_x) == r && pj[i] < PT_TABLE;
                if (active && !in_table) {
                    if (in_window) taps |= 1u << i; else slow |= 1u << i;
                }
                off[i] = (!active || in_table) ? (uint32_t)((active ? pj[i] : 0) * 16)
                                               : (in_window ? (uint32_t)(oy * ROW + ox * 4) : (uint32_t)j[i]);
                w00[i] = tp.w00; w01[i] = tp.w01; w10[i] = tp.w10; w11[i] = tp.w11;
                acc[i] = 0.0f;
            }
        }
        // -- point set-up: thread t owns the tile's points t and t + 480 (points beyond 960 are walked by everybody, see below)
        const int* ts = tile_start + (size_t)b * (per_img + 1) + r;
        const int p_begin = __ldg(ts), npts = __ldg(ts + 1) - p_begin;
        int pn[PT_PPT];
        float pw00[PT_PPT], pw01[PT_PPT], pw10[PT_PPT], pw11[PT_PPT];
        uint32_t poff[PT_PPT];
        uint32_t pfast = 0;
#pragma unroll
        for (int k = 0; k < PT_PPT; ++k) {
            pn[k] = 0; poff[k] = 0; pw00[k] = pw01[k] = pw10[k] = pw11[k] = 0.0f;
            if (t + k * PT_CONSUMERS < npts) {
                pn[k] = __ldg(list + (size_t)b * N + p_begin + t + k * PT_CONSUMERS);
                const TapXY tp = pt_taps(__ldg(Xb + pn[k]), __ldg(Xb + N + pn[k]), H, W);
                const int ox = tp.x0 - wx0, oy = tp.y0 - wy0;
                if (ox >= 0 && ox + 1 < PT_WW && oy >= 0 && oy + 1 < PT_WH) {
                    pfast |= 1u << k;
                    poff[k] = (uint32_t)(oy * ROW + ox * 4);
                }
                pw00[k] = tp.w00; pw01[k] = tp.w01; pw10[k] = tp.w10; pw11[k] = tp.w11;
            }
        }
        float* const srow_b = srows != nullptr ? srows + (size_t)b * N * C2p : nullptr;

        for (int ch = 0; ch < nchunks; ++ch) {
            mbar_wait(bar_full + 8 * s, ph);
            const uint32_t sb = base + s * PT_STAGE;
            const uint32_t sbuf = sbuf0 + (uint32_t)(ch & 1) * PT_SBUF;
            const int c0 = ch * PT_CC, cend = min(PT_CC, C2 - c0);
            // point job: S of the tile's points for these 4 channels -> the chunk's table (+ one 16-byte row segment in HBM)
#pragma unroll
            for (int k = 0; k < PT_PPT; ++k) {
                if (t + k * PT_CONSUMERS < npts) {
                    float v[PT_CC];
                    if ((pfast >> k) & 1u) {
                        const uint32_t pa = sb + poff[k];
                        float f[PT_CC][4];
#pragma unroll
                        for (int c = 0; c < PT_CC; ++c) {
                            f[c][0] = lds_f32(pa + c * CH);       f[c][1] = lds_f32(pa + c * CH + 4);
                            f[c][2] = lds_f32(pa + c * CH + ROW); f[c][3] = lds_f32(pa + c * CH + ROW + 4);
                        }
#pragma unroll
                        for (int c = 0; c < PT_CC; ++c) v[c] = pt_blend(f[c][0], f[c][1], f[c][2], f[c][3], pw00[k], pw01[k], pw10[k], pw11[k]);
                    } else {                      // taps outside the window of the point's own tile = outside the image: S = 0
#pragma unroll
                        for (int c = 0; c < PT_CC; ++c) v[c] = 0.0f;
                    }
                    sts_v4(sbuf + (t + k * PT_CONSUMERS) * 16, v[0], v[1], v[2], v[3]);
                    if (srow_b != nullptr)
                        *reinterpret_cast<float4*>(srow_b + (size_t)pn[k] * C2p + c0) = make_float4(v[0], v[1], v[2], v[3]);
                }
            }
            if (srow_b != nullptr && npts > PT_TABLE) {
                // crowded tile (more points than table slots): the rest of the list, taps recomputed per chunk
                for (int u = PT_TABLE + t; u < npts; u += PT_CONSUMERS) {
                    const int n = __ldg(list + (size_t)b * N + p_begin + u);
                    const float X = __ldg(Xb + n), Y = __ldg(Xb + N + n);
                    const TapXY tq = pt_taps(X, Y, H, W);
                    const int ox = tq.x0 - wx0, oy = tq.y0 - wy0;
                    const bool fq = ox >= 0 && ox + 1 < PT_WW && oy >= 0 && oy + 1 < PT_WH;
                    const uint32_t pa = sb + (fq ? (uint32_t)(oy * ROW + ox * 4) : 0u);
                    float v[PT_CC];
#pragma unroll
                    for (int c = 0; c < PT_CC; ++c)
                        v[c] = fq ? pt_blend(lds_f32(pa + c * CH), lds_f32(pa + c * CH + 4), lds_f32(pa + c * CH + ROW),
                                             lds_f32(pa + c * CH + ROW + 4), tq.w00, tq.w01, tq.w10, tq.w11) : 0.0f;
                    *reinterpret_cast<float4*>(srow_b + (size_t)n * C2p + c0) = make_float4(v[0], v[1], v[2], v[3]);
                }
            }
            named_bar_sync<1, PT_CONSUMERS>();       // the chunk's table is complete
            // pixel job, table pixels: branch-free — 4 LDS.128 of own features (one per channel), 4 LDS.128 of S (one per
            // pixel), 16 FMAs.  Pixels on the other two paths load slot 0 and discard the product.
            float own[PT_CC][4];
            {
                float4 cv[PT_CC], sv[4];
#pragma unroll
                for (int c = 0; c < PT_CC; ++c) cv[c] = lds_v4(sb + ctr + c * CH);
#pragma unroll
                for (int i = 0; i < 4; ++i) sv[i] = lds_v4(sbuf + ((((taps | slow) >> i) & 1u) ? 0u : off[i]));
#pragma unroll
                for (int c = 0; c < PT_CC; ++c) { own[c][0] = cv[c].x; own[c][1] = cv[c].y; own[c][2] = cv[c].z; own[c][3] = cv[c].w; }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float a = acc[i];
                    a = __fmaf_rn(sv[i].x, own[0][i], a);
                    a = __fmaf_rn(sv[i].y, own[1][i], a);
                    a = __fmaf_rn(sv[i].z, own[2][i], a);
                    a = __fmaf_rn(sv[i].w, own[3][i], a);
                    acc[i] = (((taps | slow) >> i) & 1u) ? acc[i] : a;
                }
            }
            // the other two paths (pixels whose nearest point belongs to another tile's list)
            if (taps) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if ((taps >> i) & 1u) {
                        const uint32_t pa = sb + off[i];
                        float f[PT_CC][4];
#pragma unroll
                        for (int c = 0; c < PT_CC; ++c) {
                            f[c][0] = lds_f32(pa + c * CH);       f[c][1] = lds_f32(pa + c * CH + 4);
                            f[c][2] = lds_f32(pa + c * CH + ROW); f[c][3] = lds_f32(pa + c * CH + ROW + 4);
                        }
#pragma unroll
                        for (int c = 0; c < PT_CC; ++c)
                            if (c < cend)
                                acc[i] = __fmaf_rn(pt_blend(f[c][0], f[c][1], f[c][2], f[c][3], w00[i], w01[i], w10[i], w11[i]), own[c][i], acc[i]);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty + 8 * s);
            if (++s == PT_NSTAGE) { s = 0; ph ^= 1u; }
        }

        // -- epilogue: pixel offsets to the nearest point + channel-mean correlation (output channels 0..2)
        if (active) {
            const longlong2* p2 = reinterpret_cast<const longlong2*>(nn + (size_t)b * HW + (size_t)y * W + x);
            const longlong2 a = __ldg(p2), c = __ldg(p2 + 1);
            const int64_t jj[4] = {a.x, a.y, c.x, c.y};
            float ox[4], oy[4], oc[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                int64_t v = jj[i];
                if (v < 0) v += N;
                v = v < 0 ? 0 : (v >= N ? N - 1 : v);
                ox[i] = __ldg(Xb + v) - (float)(x + i);                       // mesh_grid: x in channel 0 (models/utils.py:177-179)
                oy[i] = __ldg(Xb + N + v) - (float)y;
                oc[i] = __fdiv_rn(acc[i], (float)C2);                          // torch.mean over channels
            }
            float* o = out + (size_t)b * (C3 + 3) * HW + (size_t)y * W + x;
            __stcs(reinterpret_cast<float4*>(o), make_float4(ox[0], ox[1], ox[2], ox[3]));
            __stcs(reinterpret_cast<float4*>(o + (size_t)HW), make_float4(oy[0], oy[1], oy[2], oy[3]));
            if (slow == 0) {
                __stcs(reinterpret_cast<float4*>(o + (size_t)2 * HW), make_float4(oc[0], oc[1], oc[2], oc[3]));
            } else {                                      // far pixels get their correlation from project_far_pixels_kernel
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (!((slow >> i) & 1u)) o[(size_t)2 * HW + i] = oc[i];
            }
        }
    }
}

// ---- far pixels: the nearest point's taps lie outside the tile's window (and the point is not in the tile's table) -----
// One thread per pixel re-derives the tile kernel's classification; the few far ones (0.25 % of the pixels of a uniform
// 8-pixels-per-point cloud, all of them under a sparse cloud) are queued in shared memory and then taken by whole warps:
// lane = channel, so all 5 * C2 loads of a pixel are in flight at once (one DRAM round trip instead of C2 / 4), and lane 0
// accumulates the products in channel order through shuffles — the tile kernel's operation order, bit for bit.
__device__ __forceinline__ void project_far_pixels_block(int bx, int b, const float* __restrict__ feat2d, const float* __restrict__ xy,
                                                         const int64_t* __restrict__ nn, const int* __restrict__ pos,
                                                         float* __restrict__ out, int C2, int C3, int H, int W, int N, int tiles_x) {
    __shared__ int queue[256];
    __shared__ int n_far;
    const int HW = H * W;
    const int p = bx * 256 + threadIdx.x;
    const float* Xb = xy + (size_t)b * 2 * N;
    if (threadIdx.x == 0) n_far = 0;
    __syncthreads();
    if (p < HW) {
        const int y = p / W, x = p - y * W;
        int64_t jj = __ldg(nn + (size_t)b * HW + p);
        if (jj < 0) jj += N;
        const int j = (int)(jj < 0 ? 0 : (jj >= N ? N - 1 : jj));
        const TapXY tp = pt_taps(__ldg(Xb + j), __ldg(Xb + N + j), H, W);
        const int tx = x / PT_TW, ty = y / PT_TH, r = ty * tiles_x + tx;
        const int ox = tp.x0 - (tx * PT_TW - PT_HALO), oy = tp.y0 - (ty * PT_TH - PT_HALO);
        const bool in_window = ox >= 0 && ox + 1 < PT_WW && oy >= 0 && oy + 1 < PT_WH;
        if (!in_window && !(pt_tile_of(tp, H, W, tiles_x) == r && __ldg(pos + (size_t)b * N + j) < PT_TABLE))
            queue[atomicAdd(&n_far, 1)] = p;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* f = feat2d + (size_t)b * C2 * HW;
    for (int e = warp; e < n_far; e += 8) {
        const int pp = queue[e];
        int64_t jj = __ldg(nn + (size_t)b * HW + pp);
        if (jj < 0) jj += N;
        const int j = (int)(jj < 0 ? 0 : (jj >= N ? N - 1 : jj));
        const TapXY tp = pt_taps(__ldg(Xb + j), __ldg(Xb + N + j), H, W);
        const int x0 = tp.x0, y0 = tp.y0, x1 = x0 + 1, y1 = y0 + 1;
        const bool vx0 = x0 >= 0 && x0 < W, vx1 = x1 >= 0 && x1 < W, vy0 = y0 >= 0 && y0 < H, vy1 = y1 >= 0 && y1 < H;
        const bool v00 = vy0 && vx0, v01 = vy0 && vx1, v10 = vy1 && vx0, v11 = vy1 && vx1;
        // invalid taps are skipped, not multiplied by zero: non-finite coordinates carry NaN weights
        const size_t o00 = v00 ? (size_t)y0 * W + x0 : 0, o01 = v01 ? (size_t)y0 * W + x1 : 0;
        const size_t o10 = v10 ? (size_t)y1 * W + x0 : 0, o11 = v11 ? (size_t)y1 * W + x1 : 0;
        float acc = 0.0f;
        for (int c0 = 0; c0 < C2; c0 += 128) {                   // four channels per lane and round
            float S[4], own[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int c = c0 + u * 32 + lane;
                S[u] = 0.0f; own[u] = 0.0f;
                if (c < C2) {
                    const float* pl = f + (size_t)c * HW;
                    const float t00 = v00 ? __ldg(pl + o00) : 0.0f, t01 = v01 ? __ldg(pl + o01) : 0.0f;
                    const float t10 = v10 ? __ldg(pl + o10) : 0.0f, t11 = v11 ? __ldg(pl + o11) : 0.0f;
                    own[u] = __ldg(pl + pp);
                    float l = 0.0f, rr = 0.0f;
                    if (v00) l = __fmaf_rn(t00, tp.w00, l);
                    if (v10) l = __fmaf_rn(t10, tp.w10, l);
                    if (v01) rr = __fmaf_rn(t01, tp.w01, rr);
                    if (v11) rr = __fmaf_rn(t11, tp.w11, rr);
                    S[u] = __fadd_rn(l, rr);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int left = min(32, C2 - (c0 + u * 32));     // warp-uniform
                for (int k = 0; k < left; ++k)
                    acc = __fmaf_rn(__shfl_sync(FULL, S[u], k), __shfl_sync(FULL, own[u], k), acc);
            }
        }
        if (lane == 0) out[((size_t)b * (C3 + 3) + 2) * HW + pp] = __fdiv_rn(acc, (float)C2);
    }
}

// post launch, three kinds of 256-thread blocks, independent of each other: far pixels (latency tails: first), the
// sampled rows S -> channel-first tensor, and the feat3d slabs of output channels 3.. (batch visited last-to-first: the
// tile kernel has just streamed the tail of the batch through L2)
__global__ void __launch_bounds__(256)
project_post_kernel(const float* __restrict__ feat2d, const float* __restrict__ xy, const int64_t* __restrict__ nn,
                    const int* __restrict__ pos, const float* __restrict__ srows, const float* __restrict__ trows,
                    float* __restrict__ out, float* __restrict__ sampled_cf, int B, int C2, int C3, int H, int W, int N, int tiles_x) {
    const int HW = H * W;
    const int px_blocks = (HW + 255) / 256;
    int blk = blockIdx.x;
    const int n_far_blocks = px_blocks * B;
    if (blk < n_far_blocks) {
        project_far_pixels_block(blk % px_blocks, blk / px_blocks, feat2d, xy, nn, pos, out, C2, C3, H, W, N, tiles_x);
        return;
    }
    blk -= n_far_blocks;
    if (sampled_cf != nullptr) {
        const int nx = (N + 31) / 32, ny = (C2 + 31) / 32;
        if (blk < nx * ny * B) {
            project_rows_to_cf_block(blk % nx, (blk / nx) % ny, blk / (nx * ny), srows, sampled_cf, C2, N, round4(C2));
            return;
        }
        blk -= nx * ny * B;
    }
    const int slab = blk / (px_blocks * B), rest = blk - slab * (px_blocks * B);
    const int b = B - 1 - rest / px_blocks;
    const int p = (rest % px_blocks) * 256 + threadIdx.x;
    if (p >= HW) return;
    int64_t j = __ldg(nn + (size_t)b * HW + p);
    if (j < 0) j += N;
    j = j < 0 ? 0 : (j >= N ? N - 1 : j);
    const int C3p = round4(C3);
    project_slab_copy(trows + ((size_t)b * N + j) * C3p, out + (size_t)b * (C3 + 3) * HW + p, HW, slab * PN_SLAB,
                      min(slab * PN_SLAB + PN_SLAB, C3));
}

// ---- host side -------------------------------------------------------------------------------------------------
static bool make_window_map(CUtensorMap* m, const float* ptr, int B, int C, int H, int W) {
    auto enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)C, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4, (cuuint64_t)C * H * W * 4};
    const cuuint32_t box[4] = {(cuuint32_t)PT_WW, (cuuint32_t)PT_WH, (cuuint32_t)PT_CC, 1u};
    const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(ptr), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Scratch layout of the tiled route, in floats, inside b200_project_nn_corr_scratch_floats(B, C2, C3, N):
//   [ S rows: B*N*round4(C2) | T rows: B*N*round4(C3) | list: B*N ints | pos: B*N ints | tile_start: B*(tiles+1) ints, tiles <= 4095 ]
int64_t project_tile_extra_scratch_floats(int B, int N) { return (int64_t)2 * B * N + (int64_t)B * (PT_MAX_TILES + 1); }

bool project_tile_eligible(const float* feat2d, const int64_t* nn, const float* out, int B, int C2, int C3, int H, int W, int N) {
    if (W % 4 != 0) return false;                                                    // TMA row pitch; pixel quads
    if ((reinterpret_cast<uintptr_t>(feat2d) & 15) || (reinterpret_cast<uintptr_t>(nn) & 15) ||
        (reinterpret_cast<uintptr_t>(out) & 15)) return false;                       // 16-byte loads / stores of a quad
    if ((int64_t)C2 * H * W * 4 >= (int64_t(1) << 40)) return false;
    const int64_t tiles = (int64_t)ceil_div(W, PT_TW) * ceil_div(H, PT_TH);
    if (tiles > PT_MAX_TILES || tiles * B >= 0x7fffffff) return false;
    return tensor_map_encoder() != nullptr;
}

// Channels 0..2 of the output, the sampled tensor (sampled_cf, may be null) and the T rows for the feat3d gather.
cudaError_t project_tile_launch(const float* xy, const float* feat2d, const float* feat3d, const int64_t* nn, float* out,
                                float* scratch, float* sampled_cf, int B, int C2, int C3, int H, int W, int N, cudaStream_t st) {
    const int C2p = (C2 + 3) & ~3, C3p = (C3 + 3) & ~3;
    const int tiles_x = ceil_div(W, PT_TW), tiles_y = ceil_div(H, PT_TH), tiles = tiles_x * tiles_y;
    float* srows = scratch;
    float* trows = srows + (size_t)B * N * C2p;
    int* list = reinterpret_cast<int*>(trows + (size_t)B * N * C3p);
    int* pos = list + (size_t)B * N;
    int* tile_start = pos + (size_t)B * N;
    CUtensorMap map;
    if (!make_window_map(&map, feat2d, B, C2, H, W)) return cudaErrorInvalidValue;
    cudaError_t e;
    const size_t bin_smem = (size_t)(2 * tiles + 1) * sizeof(int);
    const int64_t prep_blocks = (int64_t)B + (int64_t)ceil_div(N, 32) * ceil_div(C3, 32) * B;
    const int64_t px_blocks = ceil_div((int64_t)H * W, 256);
    const int64_t post_blocks = px_blocks * B + (sampled_cf ? (int64_t)ceil_div(N, 32) * ceil_div(C2, 32) * B : 0) +
                                px_blocks * B * ceil_div(C3, PN_SLAB);
    if (prep_blocks >= 0x7fffffff || post_blocks >= 0x7fffffff) return cudaErrorInvalidValue;
    project_prep_kernel<<<(unsigned)prep_blocks, 256, bin_smem, st>>>(xy, feat3d, trows, list, pos, tile_start, B, C3, N, H, W, tiles_x, tiles);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    e = cudaFuncSetAttribute(project_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PT_SMEM);
    if (e != cudaSuccess) return e;
    const int num_tiles = B * tiles;
    const int grid = num_tiles < sm_count() ? num_tiles : sm_count();
    project_tile_kernel<<<grid, PT_THREADS, PT_SMEM, st>>>(map, feat2d, xy, nn, list, pos, tile_start, out,
                                                          sampled_cf ? srows : nullptr, C2, C3, H, W, N, tiles_x, tiles_y, num_tiles);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    project_post_kernel<<<(unsigned)post_blocks, 256, 0, st>>>(feat2d, xy, nn, pos, srows, trows, out, sampled_cf, B, C2, C3, H, W, N, tiles_x);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    return cudaSuccess;
}

}  // namespace b200
