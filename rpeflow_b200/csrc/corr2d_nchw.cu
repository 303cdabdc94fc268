// corr2d_nchw.cu — a1 for the wrapper-level call: correlation2d(input1, input2) on NCHW feature maps, md = 4.
//
// models/csrc/wrapper.py:68-70 permutes both feature maps to NHWC (two full read+write passes in torch) before the
// extension runs; this kernel takes the NCHW maps as the model holds them (SURVEY §8f rank 3: "the wrapper's
// NCHW->NHWC permutes"), so correlation2d() is a single pass: 4*H*W*(2C+81) bytes per sample.
//
// Same skeleton as corr2d_tma.cu — persistent CTAs, one producer warp issuing 4-D TMA boxes into an mbarrier
// ring (3 stages here), consumer warps per row shift dy (roles below) — but the channel-major layout changes the inner loop:
//   * a stage holds 16 channels of the in1 tile (8 x 32 px, row pitch 36 floats) and the in2 halo (16 x 40 px, row
//     pitch 44 floats); the pitches are 9 and 11 sixteen-byte units, odd, so the 8 lanes of a quarter-warp (8 rows,
//     same strip) read 8 different bank groups: conflict-free LDS.128 with no swizzle.  3-stage ring.
//   * lane = (row, strip), a thread owns 8 consecutive pixels x 9 column shifts.  With pixels contiguous in shared
//     memory, FFMA2 pairs two column shifts of one pixel: acc(dx, dx+1) += a[x] (broadcast) * (b[x+dx], b[x+dx+1]).
//     Even pixels pair (0,1)(2,3)(4,5)(6,7) and keep dx=8 scalar, odd pixels keep dx=0 scalar and pair
//     (1,2)(3,4)(5,6)(7,8): every b pair then starts at an even pixel = an aligned 64-bit half of an LDS.128, and one
//     register per output suffices (the channel-pair scheme of the NHWC kernel needs two).  Per channel and thread:
//     6 LDS.128, 32 FFMA2 + 8 FFMA.  An FFMA2 occupies its scheduler for two issue cycles (measured:
//     profiles/microbench), so the kernel is bound by issue slots on the busiest scheduler (3 of the 9 consumer
//     warps share one); the short strip keeps registers at ~120 so the loop body carries no spill or fix-up moves.
//   * epilogue: a thread's 8 pixels are 2 aligned float4 per displacement: plain 16-byte streaming stores.
#include "sm100_async.cuh"

namespace b200 {

constexpr int N_P = 8, N_S = 4, N_TW = N_P * N_S, N_TH = 8, N_MD = 4, N_ND = 2 * N_MD + 1;
constexpr int N_AP = 36;                         // in1 row pitch (floats): 32 + 4 ->  9 sixteen-byte units
constexpr int N_BP = 44;                         // in2 row pitch (floats): 40 + 4 -> 11 sixteen-byte units
constexpr int N_HR = N_TH + 2 * N_MD;            // 16 halo rows
constexpr int N_CC = 16;                         // channels per stage
constexpr int N_B_CH = N_HR * N_BP * 4;          // bytes per channel of the in2 halo (2816)
constexpr int N_A_CH = N_TH * N_AP * 4;          // bytes per channel of the in1 tile (1152)
constexpr int N_B_BYTES = N_CC * N_B_CH, N_A_BYTES = N_CC * N_A_CH;
constexpr int N_STAGE = N_B_BYTES + N_A_BYTES;   // 63488
constexpr int N_NSTAGE = 3;
// Warp roles.  Nine row shifts over four schedulers would leave one scheduler with three full warps (and the kernel is
// bound by issue slots on the busiest scheduler), so the ninth row shift is split by CHANNELS over two warps:
//   warps 0..7 : row shift dy = warp - 4, all 16 channels of a stage          (2 per scheduler)
//   warp  8    : row shift +4, channels 0..7 ; adds warp 9's partial sums and stores the plane   (scheduler 0: 2.5)
//   warp  9    : row shift +4, channels 8..15; hands its accumulators over through shared memory (scheduler 1: 2.5)
//   warp 10    : TMA producer                                                                     (scheduler 2)
constexpr int N_CONSUMERS = N_ND + 1;
constexpr int N_THREADS = (N_CONSUMERS + 1) * 32;
constexpr int N_COMB_BYTES = 2 * N_P * N_ND * 32 * 4;   // two hand-over buffers [72 accumulators][32 lanes]
constexpr size_t N_SMEM = (size_t)N_NSTAGE * N_STAGE + N_COMB_BYTES + 1024 + 64;
static_assert(N_B_BYTES % 128 == 0 && N_STAGE % 128 == 0, "TMA destinations stay 128-byte aligned");
static_assert(N_NSTAGE == 3, "the consumer dispatches on three compile-time stage offsets");

struct NAcc {                                    // the 9 column shifts of one pixel: 4 packed pairs + 1 scalar
    u64 p[4];
    float s;
};

// One stage (16 channels) for one consumer thread.  pa / pb: shared addresses of the thread's first in1 / in2 pixel
// in channel 0 of stage 0; SOFF: byte offset of the stage (compile time -> LDS immediates).
template <int SOFF>
__device__ __forceinline__ void corr2d_nchw_consume(NAcc (&acc)[N_P], uint32_t pa, uint32_t pb, int c_begin, int c_end) {
    pa += c_begin * N_A_CH;
    pb += c_begin * N_B_CH;
#pragma unroll 2                     // the second channel's loads are issued under the first one's FMAs
    for (int c = c_begin; c < c_end; ++c) {
        float a[N_P], b[N_P + 2 * N_MD];
#pragma unroll
        for (int m = 0; m < N_P / 4; ++m) {
            const float4 v = lds_v4(pa + (SOFF + N_B_BYTES + m * 16));
            a[4 * m] = v.x; a[4 * m + 1] = v.y; a[4 * m + 2] = v.z; a[4 * m + 3] = v.w;
        }
#pragma unroll
        for (int m = 0; m < (N_P + 2 * N_MD) / 4; ++m) {
            const float4 v = lds_v4(pb + (SOFF + m * 16));
            b[4 * m] = v.x; b[4 * m + 1] = v.y; b[4 * m + 2] = v.z; b[4 * m + 3] = v.w;
        }
#pragma unroll
        for (int i = 0; i < N_P; ++i) {
            const u64 aa = pack2(a[i], a[i]);    // ptxas turns the duplicated operand into FFMA2's scalar-broadcast form
            const int odd = i & 1;               // pixel parity = parity of i (strips start at even pixels)
#pragma unroll
            for (int q = 0; q < 4; ++q) fma2(acc[i].p[q], aa, pack2(b[i + odd + 2 * q], b[i + odd + 2 * q + 1]));
            acc[i].s = fmaf(a[i], odd ? b[i] : b[i + 8], acc[i].s);
        }
        pa += N_A_CH;
        pb += N_B_CH;
    }
}

__global__ void __launch_bounds__(N_THREADS, 1)   // 11 warps are allocated as 12: 168 registers per thread
corr2d_fwd_nchw_kernel(const __grid_constant__ CUtensorMap map1, const __grid_constant__ CUtensorMap map2,
                       float* __restrict__ out, int C, int H, int W, int tiles_x, int tiles_y, int num_tiles, float inv_c, float slope) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_full = base + N_NSTAGE * N_STAGE + N_COMB_BYTES;
    const uint32_t bar_empty = bar_full + 8 * N_NSTAGE;
    float* comb = reinterpret_cast<float*>(smem_raw + (base - smem_u32(smem_raw)) + N_NSTAGE * N_STAGE);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < N_NSTAGE; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, N_CONSUMERS);
        }
        mbar_init_fence();
    }
    __syncthreads();

    const int nchunks = (C + N_CC - 1) / N_CC;
    const int per_img = tiles_x * tiles_y;

    if (warp == N_CONSUMERS) {                                    // ---------------- producer
        if (lane == 0) {
            prefetch_tensormap(&map1);
            prefetch_tensormap(&map2);
            int s = 0;
            uint32_t ph = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int b = tile / per_img, r = tile - b * per_img;
                const int ty = r / tiles_x, tx = r - ty * tiles_x;
                const int y0 = ty * N_TH, x0 = tx * N_TW;
                for (int ch = 0; ch < nchunks; ++ch) {
                    while (!mbar_try(bar_empty + 8 * s, ph ^ 1u)) __nanosleep(128);   // consumers have drained this slot
                    mbar_arrive_expect_tx(bar_full + 8 * s, N_STAGE);
                    // boxes are (x, y, channel, batch); out-of-image pixels and channels >= C arrive as zeros
                    tma_load_4d(base + s * N_STAGE, &map2, x0 - N_MD, y0 - N_MD, ch * N_CC, b, bar_full + 8 * s);
                    tma_load_4d(base + s * N_STAGE + N_B_BYTES, &map1, x0, y0, ch * N_CC, b, bar_full + 8 * s);
                    if (++s == N_NSTAGE) { s = 0; ph ^= 1u; }
                }
            }
        }
        return;
    }

    // ---------------- consumers: warp -> (row shift, channel range), lane = (row, strip)
    const int row = lane & 7, strip = lane >> 3;
    const int dyw = warp < N_ND ? warp : N_ND - 1;                // row-shift index of this warp (warps 8 and 9 share +4)
    const int c_begin = warp == N_ND ? N_CC / 2 : 0, c_end = warp == N_ND - 1 ? N_CC / 2 : N_CC;
    const uint32_t pa = base + (uint32_t)((row * N_AP + strip * N_P) * 4);
    const uint32_t pb = base + (uint32_t)(((row + dyw) * N_BP + strip * N_P) * 4);

    NAcc acc[N_P];
#pragma unroll
    for (int i = 0; i < N_P; ++i) {
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[i].p[q] = 0ull;
        acc[i].s = 0.0f;
    }

    const size_t plane = (size_t)H * W;
    int s = 0, tcount = 0;
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++tcount) {
        for (int ch = 0; ch < nchunks; ++ch) {
            mbar_wait(bar_full + 8 * s, ph);                      // TMA bytes have landed
            if (s == 0)      corr2d_nchw_consume<0>(acc, pa, pb, c_begin, c_end);
            else if (s == 1) corr2d_nchw_consume<N_STAGE>(acc, pa, pb, c_begin, c_end);
            else             corr2d_nchw_consume<2 * N_STAGE>(acc, pa, pb, c_begin, c_end);
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty + 8 * s);        // this warp is done with the slot
            if (++s == N_NSTAGE) { s = 0; ph ^= 1u; }
        }
        if (warp >= N_ND - 1) {
            // hand-over of the split row shift: warp 9 parks its 72 partial sums per lane in buffer (tile parity); the
            // pair meets at named barrier 1.  Warp 9 rewrites a buffer two tiles later, after a meeting that warp 8 only
            // reaches once it has consumed that buffer, so one barrier per tile is enough.
            float* cb = comb + (size_t)(tcount & 1) * (N_P * N_ND * 32) + lane;
            if (warp == N_ND) {
#pragma unroll
                for (int i = 0; i < N_P; ++i) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float l, h;
                        unpack2(acc[i].p[q], l, h);
                        cb[(i * N_ND + 2 * q) * 32] = l;
                        cb[(i * N_ND + 2 * q + 1) * 32] = h;
                        acc[i].p[q] = 0ull;
                    }
                    cb[(i * N_ND + 8) * 32] = acc[i].s;
                    acc[i].s = 0.0f;
                }
                named_bar_sync<1, 64>();
                continue;                                         // warp 8 stores the plane
            }
            named_bar_sync<1, 64>();
#pragma unroll
            for (int i = 0; i < N_P; ++i) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float l, h;
                    unpack2(acc[i].p[q], l, h);
                    acc[i].p[q] = pack2(l + cb[(i * N_ND + 2 * q) * 32], h + cb[(i * N_ND + 2 * q + 1) * 32]);
                }
                acc[i].s += cb[(i * N_ND + 8) * 32];
            }
        }
        const int b = tile / per_img, r = tile - b * per_img;
        const int ty = r / tiles_x, tx = r - ty * tiles_x;
        const int y = ty * N_TH + row, x = tx * N_TW + strip * N_P;
        float* o = out + ((size_t)b * (N_ND * N_ND) + (size_t)dyw * N_ND) * plane + (size_t)y * W + x;
        const bool yok = y < H;
        // out(i, d): even pixel -> pair d/2 (lo: even d, hi: odd d), d = 8 scalar; odd pixel -> d = 0 scalar, pair (d-1)/2
        float lo[N_P][4], hi[N_P][4];
#pragma unroll
        for (int i = 0; i < N_P; ++i)
#pragma unroll
            for (int q = 0; q < 4; ++q) unpack2(acc[i].p[q], lo[i][q], hi[i][q]);
#pragma unroll
        for (int d = 0; d < N_ND; ++d) {
            float v[N_P];
#pragma unroll
            for (int i = 0; i < N_P; ++i) {
                float t;
                if ((i & 1) == 0) t = d == 8 ? acc[i].s : ((d & 1) ? hi[i][d >> 1] : lo[i][d >> 1]);
                else              t = d == 0 ? acc[i].s : ((d & 1) ? lo[i][(d - 1) >> 1] : hi[i][(d - 1) >> 1]);
                t *= inv_c;
                v[i] = fmaxf(t, t * slope);              // leaky_relu epilogue (slope 1 = none): RPEFlow_core.py:362
            }
#pragma unroll
            for (int m = 0; m < N_P / 4; ++m)
                if (yok && x + 4 * m < W)                          // W % 4 == 0: a float4 is inside or outside as a whole
                    __stcs(reinterpret_cast<float4*>(o + 4 * m), make_float4(v[4 * m], v[4 * m + 1], v[4 * m + 2], v[4 * m + 3]));
            o += plane;
        }
#pragma unroll
        for (int i = 0; i < N_P; ++i) {
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[i].p[q] = 0ull;
            acc[i].s = 0.0f;
        }
    }
}

// ---- host side -------------------------------------------------------------------------------------------------
static bool make_nchw_map(CUtensorMap* m, const float* ptr, int B, int C, int H, int W, int box_w, int box_h) {
    auto enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)C, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4, (cuuint64_t)C * H * W * 4};
    const cuuint32_t box[4] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)N_CC, 1u};
    const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(ptr), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool corr2d_nchw_eligible(const float* in1, const float* in2, const float* out, int B, int C, int H, int W, int md) {
    if (md != N_MD || W % 4 != 0) return false;                               // row stride must be a 16-byte multiple
    if ((reinterpret_cast<uintptr_t>(in1) & 15) || (reinterpret_cast<uintptr_t>(in2) & 15) ||
        (reinterpret_cast<uintptr_t>(out) & 15)) return false;
    if ((int64_t)C * H * W * 4 >= (int64_t(1) << 40)) return false;
    const int64_t tiles = (int64_t)B * ceil_div(W, N_TW) * ceil_div(H, N_TH);
    return tiles > 0 && tiles < 0x7fffffff && tensor_map_encoder() != nullptr;
}

bool corr2d_diag_preferred(int W);                                              // corr2d_diag.cu
cudaError_t corr2d_fwd_diag(const float* in1, const float* in2, float* out, int B, int C, int H, int W, float slope,
                            cudaStream_t st);

cudaError_t corr2d_fwd_nchw(const float* in1, const float* in2, float* out, int B, int C, int H, int W, float slope,
                            cudaStream_t st) {
    if (corr2d_diag_preferred(W)) return corr2d_fwd_diag(in1, in2, out, B, C, H, W, slope, st);
    CUtensorMap m1, m2;
    if (!make_nchw_map(&m1, in1, B, C, H, W, N_AP, N_TH) || !make_nchw_map(&m2, in2, B, C, H, W, N_BP, N_HR))
        return cudaErrorInvalidValue;
    const int tiles_x = ceil_div(W, N_TW), tiles_y = ceil_div(H, N_TH);
    const int num_tiles = B * tiles_x * tiles_y;
    cudaError_t e = cudaFuncSetAttribute(corr2d_fwd_nchw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)N_SMEM);
    if (e != cudaSuccess) return e;
    const int grid = num_tiles < sm_count() ? num_tiles : sm_count();
    corr2d_fwd_nchw_kernel<<<grid, N_THREADS, N_SMEM, st>>>(m1, m2, out, C, H, W, tiles_x, tiles_y, num_tiles, 1.0f / (float)C, slope);
    return cudaGetLastError();
}

}  // namespace b200

static int corr2d_fwd_nchw_entry(const char* who, const float* in1, const float* in2, float* out, int B, int C, int H, int W,
                                 int md, float slope, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0) || (in1 && in2 && out), "%s: null pointer", who);   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 1 && H >= 1 && W >= 1, "%s: bad sizes B=%d C=%d H=%d W=%d", who, B, C, H, W);
    B200_REQUIRE(md >= 1 && md <= 4, "%s: max_displacement must be in [1,4] (got %d)", who, md);
    B200_REQUIRE(slope >= 0.0f && slope <= 1.0f, "%s: negative_slope must be in [0,1] (got %g)", who, (double)slope);
    if (B == 0) return B200_OK;
    if (!corr2d_nchw_eligible(in1, in2, out, B, C, H, W, md)) {
        set_error("%s: needs md=4, W %% 4 == 0 and 16-byte aligned pointers (permute to NHWC and call b200_corr2d_fwd otherwise)",
                  who);
        return B200_ENOSUP;
    }
    const cudaError_t e = corr2d_fwd_nchw(in1, in2, out, B, C, H, W, slope, as_stream(stream));
    if (e != cudaSuccess) return cuda_fail(e, who);
    return B200_OK;
}

extern "C" int b200_corr2d_fwd_nchw(const float* in1, const float* in2, float* out, int B, int C, int H, int W, int md,
                                    b200_stream_t stream) {
    return corr2d_fwd_nchw_entry("b200_corr2d_fwd_nchw", in1, in2, out, B, C, H, W, md, 1.0f, stream);
}

extern "C" int b200_corr2d_fwd_nchw_leaky(const float* in1, const float* in2, float* out, int B, int C, int H, int W, int md,
                                          float negative_slope, b200_stream_t stream) {
    return corr2d_fwd_nchw_entry("b200_corr2d_fwd_nchw_leaky", in1, in2, out, B, C, H, W, md, negative_slope, stream);
}
