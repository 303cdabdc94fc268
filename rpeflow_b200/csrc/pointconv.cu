// pointconv.cu — f1 (SURVEY §8f rank 1): PointConvDownSampling / PointConvNoSampling forward, fused.
//
// Replaces models/pointconv.py:33-61 and :90-122 after their k_nearest_neighbor call: the two batch_indexing gathers,
// the weight net (MLP2d 3 -> 8 -> 16), torch.matmul(weights, knn_features), the view, nn.Linear(16*(C+3), out) and the
// LeakyReLU — five materialised [B,S,k,*] / [B,S,16*(C+3)] tensors in the reference, none here.
//
//   pass 0  pointconv_prep_kernel   features [xyz ; feat] transposed to point-major rows of Cp = roundup32(C+3) floats
//                                   (a neighbour's channels become one contiguous row) and the Linear weight re-laid
//                                   as Lp[o][w*Cp + c] with zero padding, so every K block below is 32 aligned floats.
//   pass 1  pointconv_tc_kernel     CTA = 64 sampled points.  meta: neighbour index + the 16 weight-net outputs of
//                                   every (point, neighbour) -> shared memory.  K loop over (c-block of 32 channels, w):
//                                   4 threads per point hold the gathered 16 x 8 feature slab of the c-block in
//                                   registers (read once per c-block, coalesced 128-byte rows) and form
//                                   A[p][32] = sum_k w_k[w] * F[k][c-block]  (the [16 x k].[k x (C+3)] product, one row of
//                                   it per w) straight into the K-major, 128B-swizzled A tile; the matching block of Lp
//                                   is the B tile; one thread issues tcgen05.mma kind::tf32 (M128 — rows 64..127 idle —
//                                   x N=out x K8) into a TMEM accumulator that lives across the whole K loop.
//                                   epilogue: tcgen05.ld, + bias, LeakyReLU(0.1), channel-first coalesced stores.
// precision 1 = TF32 operands, 2 = 3xTF32 (hi/lo split of both operands, three MMAs: fp32-level accuracy).
#include "sm100_async.cuh"

namespace b200 {

constexpr int PC_PTS = 64, PC_THREADS = 256, PC_K = 16, PC_NW = 16, PC_KB = 32;
constexpr int PC_WT_STRIDE = PC_NW * PC_K + 4;            // floats per point in s_wt (+4: rotates the bank group per point)

__device__ __forceinline__ float lrelu01(float v) { return v > 0.0f ? v : 0.1f * v; }

// ---- pass 0 ---------------------------------------------------------------------------------------------------
// grid (ceil(N/32), B): Fpm[b][n][c] ; plus, on blockIdx.y == 0 only, a grid-stride copy of the Linear weight into Lp.
__global__ void __launch_bounds__(256)
pointconv_prep_kernel(const float* __restrict__ xyz, const float* __restrict__ feat, const float* __restrict__ L,
                      float* __restrict__ Fpm, float* __restrict__ Lp, int C, int Cp, int N, int Cout, int Npad) {
    __shared__ float tile[32][33];
    const int b = blockIdx.y, n0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;       // 8 rows of 32
    const int Cf = C + 3;
    for (int c0 = 0; c0 < Cp; c0 += 32) {
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {                             // read: lane = point (contiguous in the source rows)
            const int c = c0 + ty * 4 + u, n = n0 + tx;
            float v = 0.0f;
            if (n < N && c < Cf) v = c < 3 ? __ldg(xyz + ((size_t)b * 3 + c) * N + n) : __ldg(feat + ((size_t)b * C + (c - 3)) * N + n);
            tile[ty * 4 + u][tx] = v;
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {                             // write: lane = channel (contiguous in Fpm)
            const int n = n0 + ty * 4 + u;
            if (n < N) Fpm[((size_t)b * N + n) * Cp + c0 + tx] = tile[tx][ty * 4 + u];
        }
    }
    if (b == 0) {
        const int64_t total = (int64_t)Npad * PC_NW * Cp;
        for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (int64_t)gridDim.x * 256) {
            const int c = (int)(e % Cp), w = (int)((e / Cp) % PC_NW), o = (int)(e / ((int64_t)Cp * PC_NW));
            Lp[e] = (o < Cout && c < Cf) ? __ldg(L + (size_t)o * PC_NW * Cf + (size_t)w * Cf + c) : 0.0f;
        }
    }
}

// ---- pass 1 ---------------------------------------------------------------------------------------------------
struct PcSmem {
    int a_hi, a_lo, w_hi, w_lo, wt, jj, small, bars, total;
};
__host__ __device__ inline PcSmem pc_layout(int Npad, int split) {
    PcSmem S;
    const int a = 128 * 128, w = ((Npad * 128 + 1023) / 1024) * 1024;
    int off = 0;
    S.a_hi = off; off += a;
    S.a_lo = off; if (split) off += a;
    S.w_hi = off; off += w;
    S.w_lo = off; if (split) off += w;
    S.wt = off;   off += PC_PTS * PC_WT_STRIDE * 4;
    S.jj = off;   off += PC_PTS * PC_K * 4;
    S.small = off; off += (24 + 8 + 128 + 16) * 4 + Npad * 4;     // Wa, ba, Wb, bb, bias
    off = (off + 15) & ~15;
    S.bars = off; off += 64;                                      // free, done, tmem slot
    S.total = off;
    return S;
}

template <int SPLIT>
__global__ void __launch_bounds__(PC_THREADS, 1)
pointconv_tc_kernel(const float* __restrict__ xyz, const float* __restrict__ sampled, const int64_t* __restrict__ knn,
                    const float* __restrict__ Fpm, const float* __restrict__ Lp, const float* __restrict__ Wa,
                    const float* __restrict__ ba, const float* __restrict__ Wb, const float* __restrict__ bb,
                    const float* __restrict__ bias, float* __restrict__ out, int Cp, int N, int S, int Cout, int Npad,
                    uint32_t tmem_cols) {
    extern __shared__ uint8_t pc_smem_raw[];
    const uint32_t sbase = (smem_u32(pc_smem_raw) + 1023u) & ~1023u;
    uint8_t* g = pc_smem_raw + (sbase - smem_u32(pc_smem_raw));
    const PcSmem Ls = pc_layout(Npad, SPLIT);
    float* s_wt = reinterpret_cast<float*>(g + Ls.wt);
    int* s_j = reinterpret_cast<int*>(g + Ls.jj);
    float* s_small = reinterpret_cast<float*>(g + Ls.small);      // Wa[24] ba[8] Wb[128] bb[16] bias[Npad]
    const uint32_t bar_free = sbase + Ls.bars, bar_done = bar_free + 16, tmem_slot = bar_free + 24;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(g + Ls.bars + 24);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y, s0 = blockIdx.x * PC_PTS;

    if (tid == 0) {
        mbar_init(bar_free, 1);
        mbar_init(bar_done, 1);
        mbar_init_fence();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, tmem_cols);
    }
    for (int e = tid; e < 176 + Npad; e += PC_THREADS) {
        float v;
        if (e < 24) v = __ldg(Wa + e);
        else if (e < 32) v = __ldg(ba + e - 24);
        else if (e < 160) v = __ldg(Wb + e - 32);
        else if (e < 176) v = __ldg(bb + e - 160);
        else v = e - 176 < Cout ? __ldg(bias + e - 176) : 0.0f;
        s_small[e] = v;
    }
    __syncthreads();

    // ---- meta: weight net of every (point, neighbour) pair of the tile
    for (int r = tid; r < PC_PTS * PC_K; r += PC_THREADS) {
        const int p = r >> 4, kk = r & 15;
        const int i = min(s0 + p, S - 1);
        int64_t j = __ldg(knn + ((size_t)b * S + i) * PC_K + kk);
        if (j < 0) j += N;
        j = j < 0 ? 0 : (j >= N ? N - 1 : j);
        s_j[r] = (int)j;
        float d[3], h1[8];
#pragma unroll
        for (int a = 0; a < 3; ++a) d[a] = __ldg(xyz + ((size_t)b * 3 + a) * N + j) - __ldg(sampled + ((size_t)b * 3 + a) * S + i);
#pragma unroll
        for (int o = 0; o < 8; ++o) {
            float v = s_small[24 + o];
#pragma unroll
            for (int a = 0; a < 3; ++a) v = fmaf(s_small[o * 3 + a], d[a], v);
            h1[o] = lrelu01(v);
        }
#pragma unroll
        for (int o = 0; o < PC_NW; ++o) {
            float v = s_small[160 + o];
#pragma unroll
            for (int m = 0; m < 8; ++m) v = fmaf(s_small[32 + o * 8 + m], h1[m], v);
            s_wt[p * PC_WT_STRIDE + o * PC_K + kk] = lrelu01(v);
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot_ptr;

    // ---- K loop
    const int p = tid >> 2, q8 = tid & 3;                  // 4 threads per point, 8 channels of the c-block each
    const uint32_t idesc = umma_idesc_tf32(128, Npad);
    const int ncb = Cp / PC_KB;
    const size_t lp_row = (size_t)PC_NW * Cp;              // floats per output channel in Lp
    int kbi = 0;                                           // K-block counter (barrier phase)
    for (int cb = 0; cb < ncb; ++cb) {
        float f[PC_K][8];
#pragma unroll
        for (int kk = 0; kk < PC_K; ++kk) {
            const float* row = Fpm + ((size_t)b * N + s_j[p * PC_K + kk]) * Cp + cb * PC_KB + q8 * 8;
            const float4 v0 = __ldg(reinterpret_cast<const float4*>(row)), v1 = __ldg(reinterpret_cast<const float4*>(row) + 1);
            f[kk][0] = v0.x; f[kk][1] = v0.y; f[kk][2] = v0.z; f[kk][3] = v0.w;
            f[kk][4] = v1.x; f[kk][5] = v1.y; f[kk][6] = v1.z; f[kk][7] = v1.w;
        }
        for (int w = 0; w < PC_NW; ++w, ++kbi) {
            // the B tile's global loads (Lp[o][w*Cp + cb*32 .. +32), L2-resident) go out first: their latency hides under
            // the 128 FMAs of the A rows and the wait for the previous block's MMAs
            constexpr int NBV = 256 * 8 / PC_THREADS;          // float4 per thread at out_channels = 256
            float4 bv[NBV];
#pragma unroll
            for (int n = 0; n < NBV; ++n) {
                const int e = tid + n * PC_THREADS;
                if (e < Npad * 8)
                    bv[n] = __ldg(reinterpret_cast<const float4*>(Lp + (size_t)(e >> 3) * lp_row + (size_t)w * Cp + cb * PC_KB + 4 * (e & 7)));
            }
            float acc[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[c] = 0.0f;
            const float4* wt4 = reinterpret_cast<const float4*>(s_wt + p * PC_WT_STRIDE + w * PC_K);
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
                const float4 wv = wt4[k4];
                const float ws[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
                for (int u = 0; u < 4; ++u)
#pragma unroll
                    for (int c = 0; c < 8; ++c) acc[c] = fmaf(ws[u], f[k4 * 4 + u][c], acc[c]);
            }
            if (kbi >= 1) mbar_wait(bar_free, (uint32_t)((kbi - 1) & 1));     // the MMAs reading the tiles are done
#pragma unroll
            for (int h = 0; h < 2; ++h) {                  // two 16-byte chunks of row p
                const float4 v = make_float4(acc[4 * h], acc[4 * h + 1], acc[4 * h + 2], acc[4 * h + 3]);
                const uint32_t off = (uint32_t)p * 128u + (uint32_t)(((2 * q8 + h) ^ (p & 7)) << 4);
                if (SPLIT) {
                    const float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
                    *reinterpret_cast<float4*>(g + Ls.a_hi + off) = hi;
                    *reinterpret_cast<float4*>(g + Ls.a_lo + off) = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
                } else {
                    *reinterpret_cast<float4*>(g + Ls.a_hi + off) = v;
                }
            }
#pragma unroll
            for (int n = 0; n < NBV; ++n) {                        // B tile into its swizzled rows
                const int e = tid + n * PC_THREADS;
                if (e >= Npad * 8) break;
                const int o = e >> 3, qq = e & 7;
                const float4 v = bv[n];
                const uint32_t off = (uint32_t)o * 128u + (uint32_t)((qq ^ (o & 7)) << 4);
                if (SPLIT) {
                    const float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
                    *reinterpret_cast<float4*>(g + Ls.w_hi + off) = hi;
                    *reinterpret_cast<float4*>(g + Ls.w_lo + off) = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
                } else {
                    *reinterpret_cast<float4*>(g + Ls.w_hi + off) = v;
                }
            }
            fence_proxy_async();
            __syncthreads();
            if (tid == 0) {
                tcgen05_fence_after();
#pragma unroll
                for (int ks = 0; ks < PC_KB / 8; ++ks) {
                    const uint64_t ah = umma_desc_sw128(sbase + Ls.a_hi + ks * 32), wh = umma_desc_sw128(sbase + Ls.w_hi + ks * 32);
                    umma_tf32(tmem, ah, wh, idesc, (kbi | ks) != 0);
                    if (SPLIT) {
                        const uint64_t al = umma_desc_sw128(sbase + Ls.a_lo + ks * 32), wl = umma_desc_sw128(sbase + Ls.w_lo + ks * 32);
                        umma_tf32(tmem, ah, wl, idesc, 1u);
                        umma_tf32(tmem, al, wh, idesc, 1u);
                    }
                }
                umma_commit(bar_free);
                if (cb == ncb - 1 && w == PC_NW - 1) umma_commit(bar_done);
            }
        }
    }
    mbar_wait(bar_done, 0u);
    tcgen05_fence_after();

    // ---- epilogue: warps 0 and 1 own TMEM lanes 0..63 = the tile's points
    if (warp < 2) {
        const int sp = s0 + warp * 32 + lane;
        for (int cb = 0; cb < Npad; cb += 32) {
            uint32_t raw[32];
            tmem_ld(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)cb, raw);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 32; ++c) {
                const int o = cb + c;
                if (o < Cout && sp < S) out[((size_t)b * Cout + o) * S + sp] = lrelu01(__uint_as_float(raw[c]) + s_small[176 + o]);
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, tmem_cols);
}

// second generation (pointconv_v2.cu): 128 points per CTA, warp-specialised; this file's kernel stays as the route for
// clouds of more than 65536 points
int pointconv_v2_run(const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                     const b200_pointconv_weights* w, float* out, float* scratch, int B, int C, int Cout, int N, int S,
                     int precision, int act, cudaStream_t st);
int64_t pointconv_v2_scratch_floats(int B, int C, int Cout, int N);

static inline int pc_cp(int C) { return (C + 3 + 31) / 32 * 32; }
static inline int pc_npad(int Cout) { return (Cout + 31) / 32 * 32; }      // 32: the epilogue reads 32 TMEM columns at a time

}  // namespace b200

extern "C" int64_t b200_pointconv_scratch_floats(int B, int C, int Cout, int N) {
    if (B < 0 || C < 0 || Cout < 1 || N < 1) return 0;
    const int64_t cp = b200::pc_cp(C);
    const int64_t v1 = (((int64_t)B * N * cp + 63) & ~int64_t(63)) + (int64_t)b200::pc_npad(Cout) * b200::PC_NW * cp;
    const int64_t v2 = b200::pointconv_v2_scratch_floats(B, C, Cout, N);
    return v1 > v2 ? v1 : v2;
}

extern "C" int b200_pointconv_fwd_linear(const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                                         const b200_pointconv_weights* w, float* out, float* scratch, int B, int C, int Cout,
                                         int N, int S, int k, int precision, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0 || S == 0) || (xyz && sampled_xyz && knn && w && out && scratch && (feat || C == 0)), "b200_pointconv_fwd_linear: null pointer");
    B200_REQUIRE(w != nullptr || B == 0 || S == 0, "b200_pointconv_fwd_linear: null weight struct");
    B200_REQUIRE(w == nullptr || (w->Wa && w->ba && w->Wb && w->bb && w->L && w->bias), "b200_pointconv_fwd_linear: null weight pointer");
    B200_REQUIRE(B >= 0 && C >= 0 && Cout >= 1 && N >= 1 && S >= 0, "b200_pointconv_fwd_linear: bad sizes");
    B200_REQUIRE(B <= 65535, "b200_pointconv_fwd_linear: B exceeds the grid limit");
    B200_REQUIRE(precision >= 0 && precision <= 2, "b200_pointconv_fwd_linear: precision must be 0, 1 (TF32) or 2 (3xTF32), got %d", precision);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "b200_pointconv_fwd_linear: scratch must be 16-byte aligned");
    if (k != PC_K || Cout > 256 || N > 65536) {
        set_error("b200_pointconv_fwd_linear: built for k = 16 neighbours, out_channels <= 256 and N <= 65536 (got k=%d, out=%d, N=%d)",
                  k, Cout, N);
        return B200_ENOSUP;
    }
    if (B == 0 || S == 0) return B200_OK;
    return pointconv_v2_run(xyz, feat, sampled_xyz, knn, w, out, scratch, B, C, Cout, N, S, precision, 0, as_stream(stream));
}

extern "C" int b200_pointconv_fwd(const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                                  const b200_pointconv_weights* w, float* out, float* scratch, int B, int C, int Cout,
                                  int N, int S, int k, int precision, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0 || S == 0) || (xyz && sampled_xyz && knn && w && out && scratch && (feat || C == 0)), "b200_pointconv_fwd: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(w != nullptr || B == 0 || S == 0, "b200_pointconv_fwd: null weight struct");
    B200_REQUIRE(w == nullptr || (w->Wa && w->ba && w->Wb && w->bb && w->L && w->bias), "b200_pointconv_fwd: null weight pointer");
    B200_REQUIRE(B >= 0 && C >= 0 && Cout >= 1 && N >= 1 && S >= 0, "b200_pointconv_fwd: bad sizes");
    B200_REQUIRE(B <= 65535, "b200_pointconv_fwd: B exceeds the grid limit");
    B200_REQUIRE(precision >= 0 && precision <= 2, "b200_pointconv_fwd: precision must be 0, 1 (TF32) or 2 (3xTF32), got %d", precision);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "b200_pointconv_fwd: scratch must be 16-byte aligned");
    if (k != PC_K || Cout > 256) {
        set_error("b200_pointconv_fwd: built for k = 16 neighbours and out_channels <= 256 (got k=%d, out=%d)", k, Cout);
        return B200_ENOSUP;
    }
    if (B == 0 || S == 0) return B200_OK;
    cudaStream_t st = as_stream(stream);
    if (N <= 65536)
        return pointconv_v2_run(xyz, feat, sampled_xyz, knn, w, out, scratch, B, C, Cout, N, S, precision, 1, st);
    const int Cp = pc_cp(C), Npad = pc_npad(Cout);
    float* Fpm = scratch;
    float* Lp = scratch + (((int64_t)B * N * Cp + 63) & ~int64_t(63));
    pointconv_prep_kernel<<<dim3(ceil_div(N, 32), B), 256, 0, st>>>(xyz, feat, w->L, Fpm, Lp, C, Cp, N, Cout, Npad);
    B200_LAUNCH_CHECK("pointconv_prep_kernel");
    const int split = precision != 1;                      // precision 0 (fp32 request) is served by 3xTF32
    const size_t smem = (size_t)pc_layout(Npad, split).total + 1024;
    uint32_t cols = 32;
    while ((int)cols < Npad) cols <<= 1;
    dim3 grid(ceil_div(S, PC_PTS), B);
    cudaError_t e;
    if (split) {
        e = cudaFuncSetAttribute(pointconv_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e, "pointconv_tc_kernel(attr)");
        pointconv_tc_kernel<1><<<grid, PC_THREADS, smem, st>>>(xyz, sampled_xyz, knn, Fpm, Lp, w->Wa, w->ba, w->Wb, w->bb, w->bias,
                                                              out, Cp, N, S, Cout, Npad, cols);
    } else {
        e = cudaFuncSetAttribute(pointconv_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e, "pointconv_tc_kernel(attr)");
        pointconv_tc_kernel<0><<<grid, PC_THREADS, smem, st>>>(xyz, sampled_xyz, knn, Fpm, Lp, w->Wa, w->ba, w->Wb, w->bb, w->bias,
                                                              out, Cp, N, S, Cout, Npad, cols);
    }
    B200_LAUNCH_CHECK("pointconv_tc_kernel");
    return B200_OK;
}
