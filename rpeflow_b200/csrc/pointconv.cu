// pointconv.cu — f1 (SURVEY §8f rank 1): PointConvDownSampling / PointConvNoSampling forward, fused.
//
// Replaces models/pointconv.py:33-61 and :90-122 after their k_nearest_neighbor call: the two batch_indexing gathers, the
// weight net (3 -> 8 -> 16), torch.matmul(weights, knn_features) (the [16 x k].[k x (C+3)] product per point), the view,
// nn.Linear(16*(C+3), out) and LeakyReLU(0.1) in one pass — five materialised [B,S,k,*] / [B,S,16*(C+3)] tensors in the
// reference, none here.  Design and measurements: DESIGN §4, profiles/r2_notes.md.
//   * CTA = 120 sampled points on the M = 128 rows of a cta_group::1 tcgen05.mma: 15 worker warps + the MMA warp = 512
//     threads, the largest block that still gets 128 registers per thread.
//   * warp-specialised: 15 worker warps (4 threads per point; a thread keeps the gathered 16 neighbours x 4 channels slab
//     of a 16-channel block in 64 registers and forms one 16-byte chunk of an A row per weight-net output w) and ONE
//     MMA warp that only waits on "full" mbarriers, issues tcgen05.mma and commits to "empty" mbarriers: a ring of 1-4
//     stages, as deep as shared memory allows.
//   * K block = 16 floats (one w, 16 channels): rows of 64 bytes, SWIZZLE_64B operand tiles, which is what lets the
//     128-point weight table (133 KB), the rings and the neighbour index table share 227 KB.  The index table is uint16
//     (3.75 KB) for clouds of up to 65536 points and uint32 (7.5 KB, one ring stage fewer at some widths) above.
//   * 3xTF32 with the two halves of the B operand stacked along N: D[:, 0:N) += Ah.Bh + Al.Bh, D[:, N:2N) += Ah.Bl is two
//     MMAs per k-step instead of three (out_channels <= 128; above that three MMAs); the halves are summed in the epilogue.
//   * the Linear weight is re-laid once per call as one contiguous [hi | lo] image per K block, already in the swizzled
//     operand layout; one thread of warp 0 brings it into the stage with cp.async.bulk (expect_tx on the stage's "full"
//     barrier) as soon as the stage is free; the weight-net outputs of the next K block are fetched under this block's FMAs.
// precision 1 = TF32 operands, 2 (and 0) = 3xTF32.
#include <type_traits>

#include "sm100_async.cuh"

namespace b200 {

constexpr int P2_PTS = 120, P2_ROWS = 128, P2_WORKERS = 4 * P2_PTS, P2_THREADS = P2_WORKERS + 32, P2_K = 16, P2_NW = 16, P2_CB = 16;
static_assert(P2_THREADS == 512, "512 threads: 128 registers each (the register file is allocated per 4 warps)");
constexpr int P2_WT_STRIDE = P2_NW * P2_K + 4;           // floats per point in the weight table (+4 rotates the bank group per point)
constexpr int P2_A_TILE = P2_ROWS * 64;                  // one 128-row x 16-float operand tile: 8 KB (rows 120..127 idle)
constexpr int P2_SMEM_MAX = 232448;

__device__ __forceinline__ float p2_lrelu(float v) { return v > 0.0f ? v : 0.1f * v; }

// ---- pass 0 ---------------------------------------------------------------------------------------------------
// grid (ceil(N/32), B): Fpm[b][n][0..Cp) = [xyz ; feat ; 0] point-major (Cp = roundup16(C+3)); on blockIdx.y == 0 also the
// Linear weight as Limg[kb = cb*16 + w][hi|lo][o][c'] = L[o][w*(C+3) + cb*16 + c'] (zero beyond C+3 / out_channels),
// split into TF32 hi / lo parts (3xTF32) and stored in the swizzled layout of the B operand tile: one bulk copy per K block.
__global__ void __launch_bounds__(256)
pointconv_v2_prep_kernel(const float* __restrict__ xyz, const float* __restrict__ feat, const float* __restrict__ L,
                         float* __restrict__ Fpm, float* __restrict__ Limg, int C, int Cp, int N, int Cout, int Npad, int split) {
    __shared__ float tile[32][33];
    const int b = blockIdx.y, n0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int Cf = C + 3;
    for (int c0 = 0; c0 < Cp; c0 += 32) {
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = c0 + ty * 4 + u, n = n0 + tx;
            float v = 0.0f;
            if (n < N && c < Cf) v = c < 3 ? __ldg(xyz + ((size_t)b * 3 + c) * N + n) : __ldg(feat + ((size_t)b * C + (c - 3)) * N + n);
            tile[ty * 4 + u][tx] = v;
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int n = n0 + ty * 4 + u;
            if (n < N && c0 + tx < Cp) Fpm[((size_t)b * N + n) * Cp + c0 + tx] = tile[tx][ty * 4 + u];
        }
    }
    if (b == 0 && Limg != nullptr) {
        // K block kb = cb*16 + w: [hi | lo] tiles of Npad rows x 64 bytes, already in the swizzled operand layout
        const int total = P2_NW * Cp * Npad;                                  // (Cp/16 * 16 K blocks) * Npad * 16
        for (int e = blockIdx.x * 256 + threadIdx.x; e < total; e += gridDim.x * 256) {
            const int cc = e & 15, o = (e >> 4) % Npad, kb = (e >> 4) / Npad;
            const int c = (kb >> 4) * P2_CB + cc, w = kb & 15;
            const float v = (o < Cout && c < Cf) ? __ldg(L + (size_t)o * P2_NW * Cf + (size_t)w * Cf + c) : 0.0f;
            const uint32_t off = (sw64((uint32_t)o, (uint32_t)(cc >> 2)) >> 2) + (uint32_t)(cc & 3);
            float* tile = Limg + (size_t)kb * (split ? 2 : 1) * Npad * 16;
            if (split) {
                const float hi = tf32_hi(v);
                tile[off] = hi;
                tile[Npad * 16 + off] = v - hi;
            } else {
                tile[off] = v;
            }
        }
    }
}

// ---- pass 1 ---------------------------------------------------------------------------------------------------
struct P2Smem {
    int ring, a_bytes, b_bytes, stage, wt, jj, small, bars, total;
};
__host__ __device__ inline P2Smem p2_layout(int Npad, int split, int depth, int index_bytes) {
    P2Smem S;
    S.a_bytes = (split ? 2 : 1) * P2_A_TILE;
    S.b_bytes = (split ? 2 : 1) * Npad * 64;
    S.stage = S.a_bytes + S.b_bytes;
    int off = 0;                                                               // fixed-offset tables first, the ring after them
    S.wt = off;    off += P2_PTS * P2_WT_STRIDE * 4;
    S.jj = off;    off += P2_PTS * P2_K * index_bytes;                         // neighbour indices
    off = (off + 1023) & ~1023;
    S.ring = off;  off += depth * S.stage;
    S.small = off; off += (24 + 8 + 128 + 16 + Npad) * 4;                      // Wa, ba, Wb, bb, bias
    off = (off + 15) & ~15;
    S.bars = off;  off += 128;                                                 // full[4], empty[4], accf, tmem slot
    S.total = off;
    return S;
}

// MODE 0: TF32 (one MMA per k-step); 1: 3xTF32, B halves stacked along N (two MMAs, Npad <= 128); 2: 3xTF32, three MMAs.
// WIDE: uint32 neighbour indices, for clouds of more than 65536 points.
template <int MODE, bool WIDE>
__global__ void __launch_bounds__(P2_THREADS, 1)
pointconv_v2_kernel(const float* __restrict__ xyz, const float* __restrict__ sampled, const int64_t* __restrict__ knn,
                    const float* __restrict__ Fpm, const float* __restrict__ Limg, const float* __restrict__ Wa,
                    const float* __restrict__ ba, const float* __restrict__ Wb, const float* __restrict__ bb,
                    const float* __restrict__ bias, float* __restrict__ out, int Cp, int N, int S, int Cout, int Npad,
                    uint32_t tmem_cols, int depth, int act) {
    constexpr int SPLIT = MODE != 0;
    using Index = std::conditional_t<WIDE, uint32_t, uint16_t>;
    extern __shared__ uint8_t p2_smem_raw[];
    const uint32_t sbase = (smem_u32(p2_smem_raw) + 1023u) & ~1023u;
    uint8_t* g = p2_smem_raw + (sbase - smem_u32(p2_smem_raw));
    const P2Smem Ls = p2_layout(Npad, SPLIT, depth, sizeof(Index));
    float* s_wt = reinterpret_cast<float*>(g + Ls.wt);
    Index* s_j = reinterpret_cast<Index*>(g + Ls.jj);
    float* s_small = reinterpret_cast<float*>(g + Ls.small);      // Wa[24] ba[8] Wb[128] bb[16] bias[Npad]
    const uint32_t bars = sbase + Ls.bars;                        // full[s] = bars + 8s, empty[s] = bars + 32 + 8s
    const uint32_t bar_accf = bars + 64u, tmem_slot = bars + 72u;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(g + Ls.bars + 72);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y, s0 = blockIdx.x * P2_PTS;
    const int ncb = Cp / P2_CB, nkb = ncb * P2_NW;
    const uint32_t stage_bytes = (uint32_t)Ls.stage, b_bytes = (uint32_t)Ls.b_bytes;

    if (tid == 0) {
        for (uint32_t s = 0; s < 4; ++s) {
            mbar_init(bars + 8u * s, P2_WORKERS / 32 + 1);      // one arrival per worker warp + the bulk copy's expect_tx arrival
            mbar_init(bars + 32u + 8u * s, 1);                  // stage free: tcgen05.commit
        }
        mbar_init(bar_accf, 1);
        mbar_init_fence();
    }
    if (warp == P2_WORKERS / 32) {
        tmem_alloc(tmem_slot, tmem_cols);
    }
    for (int e = tid; e < 176 + Npad; e += P2_THREADS) {
        float v;
        if (e < 24) v = __ldg(Wa + e);
        else if (e < 32) v = __ldg(ba + e - 24);
        else if (e < 160) v = __ldg(Wb + e - 32);
        else if (e < 176) v = __ldg(bb + e - 160);
        else v = e - 176 < Cout ? __ldg(bias + e - 176) : 0.0f;
        s_small[e] = v;
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot_ptr;

    if (warp == P2_WORKERS / 32) {
        // ================================================ MMA warp ================================================
        if (lane == 0) {
            const uint32_t idesc1 = umma_idesc_tf32(128, Npad), idesc2 = umma_idesc_tf32(128, 2 * Npad);
            const uint32_t a_bytes = (uint32_t)Ls.a_bytes, blo = (uint32_t)Npad * 64u;
            uint32_t s = 0, ph = 0;
            for (int kbi = 0; kbi < nkb; ++kbi) {
                mbar_wait(bars + 8u * s, ph & 1u);
                tcgen05_fence_after();
                const uint32_t a_hi = sbase + Ls.ring + s * stage_bytes, a_lo = a_hi + P2_A_TILE;
                const uint32_t b_hi = a_hi + a_bytes, b_lo = b_hi + blo;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const uint64_t ah = umma_desc_sw64(a_hi + ks * 32), bh = umma_desc_sw64(b_hi + ks * 32);
                    const uint32_t first = (kbi | ks) != 0;
                    if (MODE == 0) {
                        umma_tf32(tmem, ah, bh, idesc1, first);
                    } else if (MODE == 1) {
                        umma_tf32(tmem, ah, bh, idesc2, first);                                   // [Ah.Bh | Ah.Bl]
                        umma_tf32(tmem, umma_desc_sw64(a_lo + ks * 32), bh, idesc1, 1u);         // + Al.Bh
                    } else {
                        umma_tf32(tmem, ah, bh, idesc1, first);
                        umma_tf32(tmem, ah, umma_desc_sw64(b_lo + ks * 32), idesc1, 1u);
                        umma_tf32(tmem, umma_desc_sw64(a_lo + ks * 32), bh, idesc1, 1u);
                    }
                }
                umma_commit(bars + 32u + 8u * s);
                if (++s == (uint32_t)depth) { s = 0; ++ph; }
            }
            umma_commit(bar_accf);
        }
        __syncwarp();
    } else {
        // ================================================ workers =================================================
        const int p = tid >> 2, q = tid & 3;                    // 4 threads per point; q = neighbours 4q..4q+3 (meta) / channels 4q..4q+3
        {   // ---- meta: neighbour indices + the weight net of the point's 16 neighbours -> shared memory
            const int i = min(s0 + p, S - 1);
            float sx[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) sx[a] = __ldg(sampled + ((size_t)b * 3 + a) * S + i);
            const longlong2* kp = reinterpret_cast<const longlong2*>(knn + ((size_t)b * S + i) * P2_K + 4 * q);
            const longlong2 k01 = __ldg(kp), k23 = __ldg(kp + 1);
            const int64_t jraw[4] = {k01.x, k01.y, k23.x, k23.y};
            float wv[P2_NW][4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                int64_t j = jraw[u];
                if (j < 0) j += N;
                j = j < 0 ? 0 : (j >= N ? N - 1 : j);
                s_j[p * P2_K + 4 * q + u] = (Index)j;
                float d[3], h1[8];
#pragma unroll
                for (int a = 0; a < 3; ++a) d[a] = __ldg(xyz + ((size_t)b * 3 + a) * N + j) - sx[a];
#pragma unroll
                for (int o = 0; o < 8; ++o) {
                    float v = s_small[24 + o];
#pragma unroll
                    for (int a = 0; a < 3; ++a) v = fmaf(s_small[o * 3 + a], d[a], v);
                    h1[o] = p2_lrelu(v);
                }
#pragma unroll
                for (int o = 0; o < P2_NW; ++o) {
                    float v = s_small[160 + o];
#pragma unroll
                    for (int m = 0; m < 8; ++m) v = fmaf(s_small[32 + o * 8 + m], h1[m], v);
                    wv[o][u] = p2_lrelu(v);
                }
            }
#pragma unroll
            for (int o = 0; o < P2_NW; ++o)
                *reinterpret_cast<float4*>(s_wt + p * P2_WT_STRIDE + o * P2_K + 4 * q) = make_float4(wv[o][0], wv[o][1], wv[o][2], wv[o][3]);
        }
        named_bar_sync<1, P2_WORKERS>();

        // ---- K loop: K block kbi = (cb, w).  Per block: wait for the stage, 64 FMAs with the weights fetched one block ahead, one
        // 16-byte chunk of the A row (hi, lo) into the stage, one arrival per warp.
        const float* frow = Fpm + (size_t)b * N * Cp + 4 * q;
        const float4* wt4 = reinterpret_cast<const float4*>(s_wt + p * P2_WT_STRIDE);
        uint8_t* const st0 = g + Ls.ring + sw64((uint32_t)p, (uint32_t)q);
        const uint8_t* bsrc = reinterpret_cast<const uint8_t*>(Limg);      // this K block's B tile in global memory
        const uint32_t bdst0 = sbase + Ls.ring + (uint32_t)Ls.a_bytes;
        uint8_t* st = st0;                                      // this thread's chunk of the A row in the current stage
        uint32_t bdst = bdst0, bar_f = bars, s = 0, par_e = 1;  // parity 1 on a fresh mbarrier passes at once (first round)
        float4 wc[4];
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) wc[k4] = wt4[k4];
        for (int cb = 0; cb < ncb; ++cb) {
            float f[P2_K][4];
            {
                uint32_t jv[P2_K];
                if constexpr (WIDE) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint4 v = reinterpret_cast<const uint4*>(s_j + p * P2_K)[i];
                        jv[4 * i] = v.x; jv[4 * i + 1] = v.y; jv[4 * i + 2] = v.z; jv[4 * i + 3] = v.w;
                    }
                } else {
                    const uint4 j0 = *reinterpret_cast<const uint4*>(s_j + p * P2_K), j1 = *reinterpret_cast<const uint4*>(s_j + p * P2_K + 8);
                    const uint32_t jw[8] = {j0.x, j0.y, j0.z, j0.w, j1.x, j1.y, j1.z, j1.w};
#pragma unroll
                    for (int kk = 0; kk < P2_K; ++kk) jv[kk] = (jw[kk >> 1] >> ((kk & 1) * 16)) & 0xffffu;
                }
#pragma unroll
                for (int kk = 0; kk < P2_K; ++kk) {
                    const float4 v = __ldg(reinterpret_cast<const float4*>(frow + (size_t)jv[kk] * Cp + cb * P2_CB));
                    f[kk][0] = v.x; f[kk][1] = v.y; f[kk][2] = v.z; f[kk][3] = v.w;
                }
            }
#pragma unroll 1
            for (int w = 1; w <= P2_NW; ++w) {
                if (warp == 0) {                                // warp 0 takes the stage first: one thread starts the bulk copy of the B tile
                    mbar_wait(bar_f + 32u, par_e);           // the MMAs that read this stage are done
                    if (lane == 0) {
                        mbar_arrive_expect_tx(bar_f, b_bytes);
                        bulk_g2s(bdst, bsrc, b_bytes, bar_f);
                    }
                    bsrc += b_bytes;
                }
                const float4* wnx = wt4 + (w & 15) * 4;         // next block's weights: each quarter re-loaded right after its use
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int k4 = 0; k4 < 4; ++k4) {
                    const float ws[4] = {wc[k4].x, wc[k4].y, wc[k4].z, wc[k4].w};
#pragma unroll
                    for (int u = 0; u < 4; ++u)
#pragma unroll
                        for (int c = 0; c < 4; ++c) acc[c] = fmaf(ws[u], f[k4 * 4 + u][c], acc[c]);
                    wc[k4] = wnx[k4];
                }
                if (warp != 0) mbar_wait(bar_f + 32u, par_e);    // the other warps need the stage only now, after their FMAs
                if (SPLIT) {
                    const float4 hi = make_float4(tf32_hi(acc[0]), tf32_hi(acc[1]), tf32_hi(acc[2]), tf32_hi(acc[3]));
                    *reinterpret_cast<float4*>(st) = hi;
                    *reinterpret_cast<float4*>(st + P2_A_TILE) = make_float4(acc[0] - hi.x, acc[1] - hi.y, acc[2] - hi.z, acc[3] - hi.w);
                } else {
                    *reinterpret_cast<float4*>(st) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_f);
                if (++s == (uint32_t)depth) { s = 0; par_e ^= 1u; st = st0; bdst = bdst0; bar_f = bars; }
                else { st += stage_bytes; bdst += stage_bytes; bar_f += 8u; }
            }
        }

    }

    // ---- epilogue, all 16 warps: warp -> TMEM lane quarter (warp & 3) = 32 points, column group (warp >> 2) = Npad/4 channels
    {
        mbar_wait(bar_accf, 0u);
        tcgen05_fence_after();
        const int qd = warp & 3, cg = warp >> 2, ncol = Npad >> 2;
        const int row = qd * 32 + lane, sp = s0 + row;
        const bool live = row < P2_PTS && sp < S;
        const uint32_t tbase = tmem + ((uint32_t)(qd * 32) << 16);
        for (int c0 = cg * ncol; c0 < (cg + 1) * ncol; c0 += 8) {
            uint32_t r0[8], r1[8];
            tmem_ld(tbase + (uint32_t)c0, r0);
            if (MODE == 1) tmem_ld(tbase + (uint32_t)(Npad + c0), r1);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int o = c0 + c;
                float v = __uint_as_float(r0[c]);
                if (MODE == 1) v += __uint_as_float(r1[c]);
                if (o < Cout && live) {
                    const float y = v + s_small[176 + o];
                    out[((size_t)b * Cout + o) * S + sp] = act ? p2_lrelu(y) : y;      // act = 0: the Linear output (training)
                }
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == P2_WORKERS / 32) tmem_dealloc(tmem, tmem_cols);
}

int p2_cp(int C) { return (C + 3 + 15) / 16 * 16; }
int p2_npad(int Cout) { return (Cout + 31) / 32 * 32; }

template <int MODE, bool WIDE>
static int p2_launch(const float* xyz, const float* sampled, const int64_t* knn, const float* Fpm, const float* Limg,
                     const b200_pointconv_weights* w, float* out, int B, int Cp, int N, int S, int Cout, int Npad, int act,
                     cudaStream_t st) {
    const int split = MODE != 0, index_bytes = WIDE ? 4 : 2;
    int depth = 4;
    while (depth > 1 && p2_layout(Npad, split, depth, index_bytes).total + 1024 > P2_SMEM_MAX) --depth;
    const size_t smem = (size_t)p2_layout(Npad, split, depth, index_bytes).total + 1024;
    if (smem > (size_t)P2_SMEM_MAX) {
        set_error("b200_pointconv_fwd: out_channels = %d does not fit the shared-memory budget", Cout);
        return B200_ENOSUP;
    }
    const int ncols = MODE == 1 ? 2 * Npad : Npad;
    uint32_t cols = 32;
    while ((int)cols < ncols) cols <<= 1;
    cudaError_t e = cudaFuncSetAttribute(pointconv_v2_kernel<MODE, WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "pointconv_v2_kernel(attr)");
    pointconv_v2_kernel<MODE, WIDE><<<dim3(ceil_div(S, P2_PTS), B), P2_THREADS, smem, st>>>(
        xyz, sampled, knn, Fpm, Limg, w->Wa, w->ba, w->Wb, w->bb, w->bias, out, Cp, N, S, Cout, Npad, cols, depth, act);
    B200_LAUNCH_CHECK("pointconv_v2_kernel");
    return B200_OK;
}

// called by b200_pointconv_fwd / _fwd_linear after their argument checks; scratch sized by b200_pointconv_scratch_floats.
// act = 1: LeakyReLU(0.1) epilogue; 0: the Linear output y.
static int pointconv_v2_run(const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                            const b200_pointconv_weights* w, float* out, float* scratch, int B, int C, int Cout, int N, int S,
                            int precision, int act, cudaStream_t st) {
    const int Cp = p2_cp(C), Npad = p2_npad(Cout);
    float* Fpm = scratch;
    float* Limg = scratch + (((int64_t)B * N * Cp + 63) & ~int64_t(63));
    pointconv_v2_prep_kernel<<<dim3(ceil_div(N, 32), B), 256, 0, st>>>(xyz, feat, w->L, Fpm, Limg, C, Cp, N, Cout, Npad, precision != 1);
    B200_LAUNCH_CHECK("pointconv_v2_prep_kernel");
    auto launch = [&](auto wide) {
        constexpr bool WIDE = decltype(wide)::value;
        if (precision == 1) return p2_launch<0, WIDE>(xyz, sampled_xyz, knn, Fpm, Limg, w, out, B, Cp, N, S, Cout, Npad, act, st);
        return Npad <= 128 ? p2_launch<1, WIDE>(xyz, sampled_xyz, knn, Fpm, Limg, w, out, B, Cp, N, S, Cout, Npad, act, st)
                           : p2_launch<2, WIDE>(xyz, sampled_xyz, knn, Fpm, Limg, w, out, B, Cp, N, S, Cout, Npad, act, st);
    };
    return N > 65536 ? launch(std::true_type{}) : launch(std::false_type{});          // uint16 indices reach 65535
}

// the point-major rows alone (Fpm [B][N][p2_cp(C)] = [xyz ; feat ; 0]), for the backward (pointconv_bwd.cu)
int pointconv_v2_rows(const float* xyz, const float* feat, float* Fpm, int B, int C, int N, cudaStream_t st) {
    pointconv_v2_prep_kernel<<<dim3(ceil_div(N, 32), B), 256, 0, st>>>(xyz, feat, nullptr, Fpm, nullptr, C, p2_cp(C), N, 1, 32, 0);
    B200_LAUNCH_CHECK("pointconv_v2_prep_kernel");
    return B200_OK;
}

// the argument checks of both forward entries; who names the entry in the messages
static int pointconv_fwd_args(const char* who, const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                              const b200_pointconv_weights* w, const float* out, const float* scratch, int B, int C, int Cout,
                              int N, int S, int precision) {
    B200_REQUIRE((B == 0 || S == 0) || (xyz && sampled_xyz && knn && w && out && scratch && (feat || C == 0)), "%s: null pointer", who);   // empty calls carry null pointers
    B200_REQUIRE(w != nullptr || B == 0 || S == 0, "%s: null weight struct", who);
    B200_REQUIRE(w == nullptr || (w->Wa && w->ba && w->Wb && w->bb && w->L && w->bias), "%s: null weight pointer", who);
    B200_REQUIRE(B >= 0 && C >= 0 && Cout >= 1 && N >= 1 && S >= 0, "%s: bad sizes", who);
    B200_REQUIRE(B <= 65535, "%s: B exceeds the grid limit", who);
    B200_REQUIRE(precision >= 0 && precision <= 2, "%s: precision must be 0, 1 (TF32) or 2 (3xTF32), got %d", who, precision);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "%s: scratch must be 16-byte aligned", who);
    return B200_OK;
}

}  // namespace b200

extern "C" int64_t b200_pointconv_scratch_floats(int B, int C, int Cout, int N) {
    if (B < 0 || C < 0 || Cout < 1 || N < 1) return 0;
    const int64_t cp = b200::p2_cp(C);
    return (((int64_t)B * N * cp + 63) & ~int64_t(63)) + 2 * (int64_t)b200::p2_npad(Cout) * b200::P2_NW * cp;
}

extern "C" int b200_pointconv_fwd_linear(const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                                         const b200_pointconv_weights* w, float* out, float* scratch, int B, int C, int Cout,
                                         int N, int S, int k, int precision, b200_stream_t stream) {
    using namespace b200;
    if (const int e = pointconv_fwd_args("b200_pointconv_fwd_linear", xyz, feat, sampled_xyz, knn, w, out, scratch, B, C, Cout, N, S, precision))
        return e;
    if (k != P2_K || Cout > 256 || N > 65536) {
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
    if (const int e = pointconv_fwd_args("b200_pointconv_fwd", xyz, feat, sampled_xyz, knn, w, out, scratch, B, C, Cout, N, S, precision))
        return e;
    if (k != P2_K || Cout > 256) {
        set_error("b200_pointconv_fwd: built for k = 16 neighbours and out_channels <= 256 (got k=%d, out=%d)", k, Cout);
        return B200_ENOSUP;
    }
    if (B == 0 || S == 0) return B200_OK;
    return pointconv_v2_run(xyz, feat, sampled_xyz, knn, w, out, scratch, B, C, Cout, N, S, precision, 1, as_stream(stream));
}
