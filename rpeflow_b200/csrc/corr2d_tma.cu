// corr2d_tma.cu — a1, the production forward kernel for max_displacement 4: persistent, warp-specialised, TMA-fed.
//
// Replaces models/csrc/correlation/correlation_forward_kernel.cu:11-55 (one warp per output pixel, 81 serial
// shuffle reductions, 4-byte stores H*W apart).
//
//   * grid = one CTA per SM, each walks tiles t = blockIdx.x, +gridDim.x, ... of 8 rows x 24 columns of output
//     pixels (all 81 displacements); neighbouring tiles run at the same time, so halo re-reads hit L2.
//   * warp 9 = producer: one elected lane issues two 4-D TMA loads per stage — the in1 tile and the in2 halo
//     (16 x 32 pixels) for 32 channels — into a 2-stage ring (88 KB per stage) guarded by full/empty mbarriers.
//     Out-of-image pixels (and channels >= C) are zero-filled by the TMA unit: that IS the reference's zero
//     padding, and no thread spends an instruction on load addresses or bounds.
//   * the tensor maps list the dimensions as (C, H, W, B) — rows before columns — so a box lands in shared memory
//     COLUMN-major: pixel line index = x*rows + y, 128 bytes (32 channels) per line, written with the 128-byte
//     swizzle (16-byte chunk index ^= line index & 7).  A thread walks along x in one row, so all of its lines
//     share one swizzle phase (its row & 7): one XOR per 4-channel step and every LDS.128 address is
//     register + immediate.  The 8 lanes of a quarter-warp sit in 8 different rows -> 8 different bank groups:
//     conflict-free without padding (LDS.128 costs 4 clk/warp/SM unless all lanes agree, see
//     profiles/microbench/lds_patterns.cu — shared-memory bandwidth is the co-limiter of this kernel).
//   * warps 0..8 = consumers, warp w owns row shift dy = w-4.  lane -> (row = lane%8, strip = lane/8); a thread
//     owns 6 consecutive pixels x 9 column shifts = 54 outputs, each accumulated as an (even, odd) channel pair
//     so the inner loop is packed FFMA2 (fma.rn.f32x2) fed straight from 64-bit halves of LDS.128:
//     108 FFMA2 per 20 LDS.128 per 4 channels (10 warps are allocated registers as 12 -> 168 per thread, which a
//     7-pixel strip would exceed).
//   * epilogue: pair-sum, scale by 1/C; neighbouring strips trade two values by shuffle so that every store is an
//     aligned 16-byte st.global.cs (scalar stores when W % 4 != 0).
#include "sm100_async.cuh"

namespace b200 {

constexpr int T_P = 6, T_S = 4, T_TW = T_P * T_S, T_TH = 8, T_MD = 4, T_ND = 2 * T_MD + 1;
constexpr int T_HC = T_TW + 2 * T_MD;          // in2 halo columns (32)
constexpr int T_HR = T_TH + 2 * T_MD;          // in2 halo rows (16)
constexpr int T_CC = 32;                       // channels per stage = one 128-byte swizzle line per pixel
constexpr int T_B_BYTES = T_HC * T_HR * 128;   // 65536
constexpr int T_A_BYTES = T_TW * T_TH * 128;   // 24576
constexpr int T_STAGE = T_B_BYTES + T_A_BYTES; // 90112 (both parts multiples of 1024: swizzle atoms stay aligned)
static_assert(T_B_BYTES % 1024 == 0 && T_A_BYTES % 1024 == 0, "stage parts must keep the 1024-byte swizzle alignment");
constexpr int T_NSTAGE = 2;
constexpr int T_UNROLL = 1;
constexpr int T_CONSUMERS = T_ND;              // warps
constexpr int T_THREADS = (T_CONSUMERS + 1) * 32;
constexpr size_t T_SMEM = (size_t)T_NSTAGE * T_STAGE + 1024 + 64;

// One stage (32 channels) of one tile for one consumer thread, two channels (one FFMA2 operand pair) per step.
// SOFF = byte offset of the stage (compile time: rides in the LDS immediates).  pa0 / pb0 = shared address of the
// thread's first in1 / in2 line with the thread's swizzle phase folded in; XOR with step<<3 selects the channel
// pair (bits 4..6 = 16-byte chunk through the swizzle, bit 3 = half of the chunk).
template <int SOFF>
__device__ __forceinline__ void corr2d_consume(u64 (&acc)[T_P][T_ND], uint32_t pa0, uint32_t pb0) {
#pragma unroll T_UNROLL
    for (int step = 0; step < T_CC / 2; ++step) {
        const uint32_t aq = pa0 ^ (uint32_t)(step << 3), bq = pb0 ^ (uint32_t)(step << 3);
        u64 a[T_P];
#pragma unroll
        for (int i = 0; i < T_P; ++i) a[i] = lds_b64(aq + (SOFF + T_B_BYTES + i * T_TH * 128));
#pragma unroll
        for (int j = 0; j < T_P + 2 * T_MD; ++j) {
            const u64 v = lds_b64(bq + (SOFF + j * T_HR * 128));
#pragma unroll
            for (int i = 0; i < T_P; ++i) {
                const int d = j - i;                     // column shift index, dx = d - 4
                if (d >= 0 && d < T_ND) fma2(acc[i][d], a[i], v);
            }
        }
    }
}

__global__ void __launch_bounds__(T_THREADS, 1)   // 10 warps are allocated as 12: 168 registers per thread
corr2d_fwd_tma_kernel(const __grid_constant__ CUtensorMap map1, const __grid_constant__ CUtensorMap map2,
                      float* __restrict__ out, int C, int H, int W, int tiles_x, int tiles_y, int num_tiles, float inv_c,
                      int vec_store) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_full = base + T_NSTAGE * T_STAGE;          // 2 x 8 B
    const uint32_t bar_empty = bar_full + 8 * T_NSTAGE;           // 2 x 8 B
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < T_NSTAGE; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, T_CONSUMERS);
        }
        mbar_init_fence();
    }
    __syncthreads();

    const int nchunks = (C + T_CC - 1) / T_CC;
    const int per_img = tiles_x * tiles_y;

    if (warp == T_CONSUMERS) {                                    // ---------------- producer
        if (lane == 0) {
            prefetch_tensormap(&map1);
            prefetch_tensormap(&map2);
            int it = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int b = tile / per_img, r = tile - b * per_img;
                const int ty = r / tiles_x, tx = r - ty * tiles_x;
                const int y0 = ty * T_TH, x0 = tx * T_TW;
                for (int ch = 0; ch < nchunks; ++ch, ++it) {
                    const int s = it & 1;
                    const uint32_t ph = (uint32_t)(it >> 1) & 1u;
                    while (!mbar_try(bar_empty + 8 * s, ph ^ 1u)) __nanosleep(128);   // consumers have drained this slot
                    mbar_arrive_expect_tx(bar_full + 8 * s, T_STAGE);
                    tma_load_4d(base + s * T_STAGE, &map2, ch * T_CC, y0 - T_MD, x0 - T_MD, b, bar_full + 8 * s);
                    tma_load_4d(base + s * T_STAGE + T_B_BYTES, &map1, ch * T_CC, y0, x0, b, bar_full + 8 * s);
                }
            }
        }
        return;
    }

    // ---------------- consumers: warp = row shift dy, lane = (row, strip)
    const int row = lane & 7, strip = lane >> 3;
    // line index = x * rows + y; every line of this thread has swizzle phase (y & 7)
    // (LDS.64 is served per half-warp = 8 rows x 2 strips: odd strips visit the two halves of every 16-byte chunk in
    // swapped order, so the 16 lanes cover all 16 eight-byte bank pairs)
    const uint32_t half = (uint32_t)(strip & 1) << 3;
    const uint32_t pa0 = base + (uint32_t)((strip * T_P * T_TH + row) * 128) + (((uint32_t)row << 4) | half);
    const uint32_t pb0 = base + (uint32_t)((strip * T_P * T_HR + row + warp) * 128) + (((uint32_t)((row + warp) & 7) << 4) | half);

    u64 acc[T_P][T_ND];
#pragma unroll
    for (int i = 0; i < T_P; ++i)
#pragma unroll
        for (int d = 0; d < T_ND; ++d) acc[i][d] = 0ull;

    const size_t plane = (size_t)H * W;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (int ch = 0; ch < nchunks; ++ch, ++it) {
            const int s = it & 1;
            const uint32_t ph = (uint32_t)(it >> 1) & 1u;
            mbar_wait(bar_full + 8 * s, ph);                      // TMA bytes have landed
            if (s == 0) corr2d_consume<0>(acc, pa0, pb0);
            else        corr2d_consume<T_STAGE>(acc, pa0, pb0);
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty + 8 * s);        // this warp is done with the slot
        }
        const int b = tile / per_img, r = tile - b * per_img;
        const int ty = r / tiles_x, tx = r - ty * tiles_x;
        const int y = ty * T_TH + row, xt = tx * T_TW;
        float* orow = out + ((size_t)b * (T_ND * T_ND) + (size_t)warp * T_ND) * plane + (size_t)y * W + xt;
        const bool yok = y < H;
        if (vec_store) {
            // strips 1 and 3 take pixels 4,5 of their left neighbour: they then hold 8 pixels = two aligned float4,
            // strips 0 and 2 keep their first four.
            const bool odd = strip & 1;
            const int px = strip * T_P - (odd ? 2 : 0);           // first pixel this lane stores: 0, 4, 12, 16
            float* o = orow + px;
            const bool ok0 = yok && xt + px < W, ok1 = odd && yok && xt + px + 4 < W;
#pragma unroll
            for (int d = 0; d < T_ND; ++d) {
                float v[T_P];
#pragma unroll
                for (int i = 0; i < T_P; ++i) {
                    float lo, hi;
                    unpack2(acc[i][d], lo, hi);
                    acc[i][d] = 0ull;
                    v[i] = (lo + hi) * inv_c;
                }
                const float n4 = __shfl_up_sync(FULL, v[4], 8), n5 = __shfl_up_sync(FULL, v[5], 8);
                const float4 first = odd ? make_float4(n4, n5, v[0], v[1]) : make_float4(v[0], v[1], v[2], v[3]);
                if (ok0) __stcs(reinterpret_cast<float4*>(o), first);                       // streaming: never re-read here
                if (ok1) __stcs(reinterpret_cast<float4*>(o + 4), make_float4(v[2], v[3], v[4], v[5]));
                o += plane;
            }
        } else {
            float* o = orow + strip * T_P;
#pragma unroll
            for (int d = 0; d < T_ND; ++d) {
#pragma unroll
                for (int i = 0; i < T_P; ++i) {
                    float lo, hi;
                    unpack2(acc[i][d], lo, hi);
                    acc[i][d] = 0ull;
                    if (yok && xt + strip * T_P + i < W) __stcs(o + i, (lo + hi) * inv_c);
                }
                o += plane;
            }
        }
    }
}

// ---- host side -------------------------------------------------------------------------------------------------
static bool make_map(CUtensorMap* m, const float* ptr, int B, int C, int H, int W, int box_w, int box_h) {
    auto enc = tensor_map_encoder();
    if (!enc) return false;
    // dimensions listed as (C, H, W, B): rows BEFORE columns, so a box is laid out column-major in shared memory
    const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)H, (cuuint64_t)W, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)W * C * 4, (cuuint64_t)C * 4, (cuuint64_t)H * W * C * 4};
    const cuuint32_t box[4] = {(cuuint32_t)T_CC, (cuuint32_t)box_h, (cuuint32_t)box_w, 1u};
    const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(ptr), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// true when the TMA kernel can take this call (else the caller uses the generic cp.async kernel of corr2d.cu)
bool corr2d_tma_eligible(const float* in1, const float* in2, int B, int C, int H, int W, int md) {
    if (md != T_MD || C % 4 != 0) return false;                               // global strides must be 16-byte multiples
    if ((reinterpret_cast<uintptr_t>(in1) & 15) || (reinterpret_cast<uintptr_t>(in2) & 15)) return false;
    if ((int64_t)H * W * C * 4 >= (int64_t(1) << 40)) return false;           // tensor-map stride limit
    const int64_t tiles = (int64_t)B * ceil_div(W, T_TW) * ceil_div(H, T_TH);
    return tiles > 0 && tiles < 0x7fffffff && tensor_map_encoder() != nullptr;
}

cudaError_t corr2d_fwd_tma(const float* in1, const float* in2, float* out, int B, int C, int H, int W, cudaStream_t st) {
    CUtensorMap m1, m2;
    if (!make_map(&m1, in1, B, C, H, W, T_TW, T_TH) || !make_map(&m2, in2, B, C, H, W, T_HC, T_HR))
        return cudaErrorInvalidValue;
    const int tiles_x = ceil_div(W, T_TW), tiles_y = ceil_div(H, T_TH);
    const int num_tiles = B * tiles_x * tiles_y;
    cudaError_t e = cudaFuncSetAttribute(corr2d_fwd_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T_SMEM);
    if (e != cudaSuccess) return e;
    const int grid = num_tiles < sm_count() ? num_tiles : sm_count();
    const int vec_store = (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    corr2d_fwd_tma_kernel<<<grid, T_THREADS, T_SMEM, st>>>(m1, m2, out, C, H, W, tiles_x, tiles_y, num_tiles, 1.0f / (float)C,
                                                           vec_store);
    return cudaGetLastError();
}

}  // namespace b200
