// corr3d_tc.cu — a5 pass 2 on the 5th-generation tensor cores: the Cout x Cout layer of cost_mlp as tcgen05.mma
// (kind::tf32, fp32 accumulate in tensor memory), fused with the neighbour gather that produces its input and with
// the PointConv-style weighting + sum over the k neighbours that consumes its output.
//
// Replaces the second 1x1 Conv2d of cost_mlp, weight_net2 and the mul+sum of models/pwc3d_core.py:91-101.
// north_star allows tensor cores exactly here ("the dense per-neighbour MLP contraction"); precision 1 = TF32
// operands (what cuDNN does for the reference's convs under torch's default allow_tf32), precision 2 = 3xTF32
// (hi/lo operand split, three MMAs per slice: ~fp32 accuracy, meets the fp32 tolerance of the parity tests).
//
// One CTA = one tile of 128 rows = 8 points x 16 neighbours (MMA M = 128), N = Cout, K = Cout in blocks of 32
// channels.  4 warps; thread r owns row r (and TMEM lane r in the epilogue):
//   meta      thread r: neighbour index j, offset d = xyz2[j] - xyz1[i], weight-net hidden vector (8 registers).
//   produce   per K block: h1 = lrelu(A1[i] + G2[j] + W1c.d) for 128 rows x 32 channels (8 lanes per row -> every
//             gathered G2 row segment is one coalesced 128-byte read) and the matching W2 block, both written to
//             shared memory K-major with the 128-byte swizzle the MMA descriptors name; one stage, reuse gated by
//             tcgen05.commit -> mbarrier (several CTAs per SM overlap each other's gather / MMA / epilogue phases).
//   mma       one thread issues 4 (x3 for 3xTF32) tcgen05.mma per K block: D[128 x Cout] += A[128 x 8] . B[Cout x 8]^T.
//   epilogue  tcgen05.ld 32 columns at a time: v = lrelu(D + b2) * relu(bc + Wc.hid); the 16 rows of a point are
//             summed by recursive halving (30 shuffles per 32 columns), lane m ends with columns 2m, 2m+1 -> one
//             coalesced 128-byte store of P per point and column chunk.
#include "corr3d_common.cuh"
#include "sm100_async.cuh"

namespace b200 {

constexpr int TC_ROWS = 128, TC_KB = 32, TC_THREADS = 128, TC_K = 16;   // TC_K: neighbours per point this kernel is built for

struct TcSmem {                      // byte offsets from the 1024-aligned base
    int a_hi, a_lo, w_hi, w_lo, stage_bytes, epi, w1c, wn, meta_j, meta_d, bars, total;
};
__host__ __device__ inline TcSmem tc_layout(int Cout, int split) {
    TcSmem L;
    const int a = TC_ROWS * 128, w = ((Cout * 128 + 1023) / 1024) * 1024;
    L.a_hi = 0;
    L.a_lo = split ? a : 0;
    L.w_hi = (split ? 2 : 1) * a;
    L.w_lo = split ? L.w_hi + w : L.w_hi;
    L.stage_bytes = (split ? 2 : 1) * (a + w);
    int off = L.stage_bytes;                           // one stage: co-resident CTAs (not a ring) hide the gather latency
    L.epi = off;     off += Cout * 48;                 // per output channel: b2, bc, -, -, Wc[0..7]
    L.w1c = off;     off += 3 * Cout * 4;
    L.wn = off;      off += WN_FLOATS * 4;              // weight net parameters (16-byte aligned: Cout % 32 == 0)
    L.meta_j = off;  off += TC_ROWS * 4;
    L.meta_d = off;  off += TC_ROWS * 16;
    off = (off + 15) & ~15;
    L.bars = off;    off += 64;                        // free, done, tmem base slot
    L.total = off;
    return L;
}

template <int SPLIT>   // 0: TF32, 1: 3xTF32
__global__ void __launch_bounds__(TC_THREADS)
corr3d_stage1_tc_kernel(const float* __restrict__ xyz1, const float* __restrict__ xyz2, const int64_t* __restrict__ knn12,
                        const float* __restrict__ A1, const float* __restrict__ G2, const float* __restrict__ W2,
                        const float* __restrict__ W1cT, const float* __restrict__ b2, const float* __restrict__ Wa,
                        const float* __restrict__ ba, const float* __restrict__ Wb, const float* __restrict__ bb,
                        const float* __restrict__ WcT, const float* __restrict__ bc, float* __restrict__ P,
                        int Cout, int N1, int N2, uint32_t tmem_cols, int tiles_per_cta) {
    extern __shared__ uint8_t tc_smem_raw[];
    const uint32_t sbase = (smem_u32(tc_smem_raw) + 1023u) & ~1023u;
    uint8_t* gbase = tc_smem_raw + (sbase - smem_u32(tc_smem_raw));
    const TcSmem L = tc_layout(Cout, SPLIT);
    float* s_epi = reinterpret_cast<float*>(gbase + L.epi);
    float* s_w1c = reinterpret_cast<float*>(gbase + L.w1c);
    float* s_wn = reinterpret_cast<float*>(gbase + L.wn);
    int* s_j = reinterpret_cast<int*>(gbase + L.meta_j);
    float4* s_d = reinterpret_cast<float4*>(gbase + L.meta_d);
    const uint32_t bar_free = sbase + L.bars, bar_done = bar_free + 16, tmem_slot = bar_free + 24;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + L.bars + 24);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y;

    if (tid == 0) {
        mbar_init(bar_free, 1);
        mbar_init(bar_done, 1);
        mbar_init_fence();
    }
    if (warp == 0) {                                   // tensor-memory columns for the 128 x Cout fp32 accumulator
        tmem_alloc(tmem_slot, tmem_cols);
    }

    // per-CTA constants: epilogue table, W1c; then the tensor-memory base address
    for (int o = tid; o < Cout; o += TC_THREADS) {
        float* e = s_epi + o * 12;
        e[0] = __ldg(b2 + o); e[1] = __ldg(bc + o); e[2] = 0.0f; e[3] = 0.0f;
#pragma unroll
        for (int m = 0; m < 8; ++m) e[4 + m] = __ldg(WcT + (size_t)m * Cout + o);
    }
    for (int e = tid; e < 3 * Cout; e += TC_THREADS) s_w1c[e] = __ldg(W1cT + e);
    weight_net_stage(s_wn, Wa, ba, Wb, bb, tid, TC_THREADS);
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot_ptr;

    const int nkb = Cout / TC_KB;
    const uint32_t idesc = umma_idesc_tf32(TC_ROWS, Cout);
    const int q = lane & 7;                            // 16-byte chunk (4 channels) of the 128-byte row this lane handles
    uint32_t it = 0;                                   // MMA batches committed to bar_free so far (its phase counter)

    // A CTA walks `tiles_per_cta` consecutive tiles: the tensor-memory allocation, the barriers, the constants above and
    // (when Cout = 32, a single K block) the W2 tile are set up once, not once per 8 points.
    for (int tt = 0; tt < tiles_per_cta; ++tt) {
    const int i0 = (blockIdx.x * tiles_per_cta + tt) * (TC_ROWS / TC_K);
    if (i0 >= N1) break;

    // ---- meta: thread r owns row r = (point r/16, neighbour r%16)
    float hid[8];
    {
        const int i = min(i0 + (tid >> 4), N1 - 1);
        int64_t j = __ldg(knn12 + ((size_t)b * N1 + i) * TC_K + (tid & 15));
        j = j < 0 ? 0 : (j >= N2 ? N2 - 1 : j);
        const float dx = __ldg(xyz2 + ((size_t)b * 3 + 0) * N2 + j) - __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + i);
        const float dy = __ldg(xyz2 + ((size_t)b * 3 + 1) * N2 + j) - __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + i);
        const float dz = __ldg(xyz2 + ((size_t)b * 3 + 2) * N2 + j) - __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + i);
        s_j[tid] = (int)j;
        s_d[tid] = make_float4(dx, dy, dz, 0.0f);
        weight_net_hidden_s(s_wn, dx, dy, dz, hid);
    }
    __syncthreads();                                   // s_j / s_d of this tile are visible to the gathering lanes

    // ---- K loop: produce a stage, one thread issues its MMAs
    for (int kb = 0; kb < nkb; ++kb, ++it) {
        constexpr int st = 0;
        if (it >= 1) mbar_wait(bar_free, (it - 1) & 1u);               // the MMAs that read the stage are done
        const uint32_t stage = sbase;
        const int c0 = kb * TC_KB + 4 * q;
        const float4 wx = *reinterpret_cast<const float4*>(s_w1c + c0);
        const float4 wy = *reinterpret_cast<const float4*>(s_w1c + Cout + c0);
        const float4 wz = *reinterpret_cast<const float4*>(s_w1c + 2 * Cout + c0);
#pragma unroll 4
        for (int step = 0; step < 8; ++step) {         // 4 rows per warp-step, 8 lanes per row
            const int row = warp * 32 + step * 4 + (lane >> 3);
            const int i = min(i0 + (row >> 4), N1 - 1);
            const float4 d = s_d[row];
            const float4 a = __ldg(reinterpret_cast<const float4*>(A1 + ((size_t)b * N1 + i) * Cout + c0));
            const float4 g = __ldg(reinterpret_cast<const float4*>(G2 + ((size_t)b * N2 + s_j[row]) * Cout + c0));
            float4 v;
            v.x = leaky01(a.x + g.x + fmaf(wz.x, d.z, fmaf(wy.x, d.y, wx.x * d.x)));
            v.y = leaky01(a.y + g.y + fmaf(wz.y, d.z, fmaf(wy.y, d.y, wx.y * d.x)));
            v.z = leaky01(a.z + g.z + fmaf(wz.z, d.z, fmaf(wy.z, d.y, wx.z * d.x)));
            v.w = leaky01(a.w + g.w + fmaf(wz.w, d.z, fmaf(wy.w, d.y, wx.w * d.x)));
            const uint32_t off = (uint32_t)row * 128u + (uint32_t)((q ^ (row & 7)) << 4);
            if (SPLIT) {
                const float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
                *reinterpret_cast<float4*>(gbase + st * L.stage_bytes + L.a_hi + off) = hi;
                *reinterpret_cast<float4*>(gbase + st * L.stage_bytes + L.a_lo + off) =
                    make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
            } else {
                *reinterpret_cast<float4*>(gbase + st * L.stage_bytes + L.a_hi + off) = v;
            }
        }
        if (nkb > 1 || tt == 0)                                // a single K block: the W2 tile of the first tile stays valid
        for (int e = tid; e < Cout * 8; e += TC_THREADS) {     // W2[o][kb*32 .. +32): the B operand, K-major
            const int o = e >> 3, qq = e & 7;
            const float4 v = __ldg(reinterpret_cast<const float4*>(W2 + (size_t)o * Cout + kb * TC_KB + 4 * qq));
            const uint32_t off = (uint32_t)o * 128u + (uint32_t)((qq ^ (o & 7)) << 4);
            if (SPLIT) {
                const float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
                *reinterpret_cast<float4*>(gbase + st * L.stage_bytes + L.w_hi + off) = hi;
                *reinterpret_cast<float4*>(gbase + st * L.stage_bytes + L.w_lo + off) =
                    make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
            } else {
                *reinterpret_cast<float4*>(gbase + st * L.stage_bytes + L.w_hi + off) = v;
            }
        }
        fence_proxy_async();   // generic-proxy writes -> visible to the MMA's async proxy
        __syncthreads();
        if (tid == 0) {
            tcgen05_fence_after();
#pragma unroll
            for (int ks = 0; ks < TC_KB / 8; ++ks) {   // one MMA consumes K = 8 tf32 = 32 bytes of every row
                const uint64_t ah = umma_desc_sw128(stage + L.a_hi + ks * 32), wh = umma_desc_sw128(stage + L.w_hi + ks * 32);
                umma_tf32(tmem, ah, wh, idesc, (kb | ks) != 0);
                if (SPLIT) {
                    const uint64_t al = umma_desc_sw128(stage + L.a_lo + ks * 32), wl = umma_desc_sw128(stage + L.w_lo + ks * 32);
                    umma_tf32(tmem, ah, wl, idesc, 1u);
                    umma_tf32(tmem, al, wh, idesc, 1u);
                }
            }
            umma_commit(bar_free);                     // arrives when the MMAs issued so far have finished reading smem
            if (kb == nkb - 1) umma_commit(bar_done);
        }
    }
    mbar_wait(bar_done, (uint32_t)(tt & 1));        // accumulator complete (one commit per tile)
    tcgen05_fence_after();

    // ---- epilogue: thread = row (TMEM lane), 32 columns at a time
    const int m = lane & 15;                           // position in the 16-row group of one point
    const int pt = i0 + warp * 2 + (lane >> 4);
    float* prow = P + ((size_t)b * N1 + min(pt, N1 - 1)) * Cout;
    for (int cb = 0; cb < Cout; cb += 32) {
        uint32_t raw[32];
        tmem_ld(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)cb, raw);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) {
            const float4 e0 = *reinterpret_cast<const float4*>(s_epi + (cb + c) * 12);        // b2, bc (broadcast reads)
            const float4 e1 = *reinterpret_cast<const float4*>(s_epi + (cb + c) * 12 + 4);
            const float4 e2 = *reinterpret_cast<const float4*>(s_epi + (cb + c) * 12 + 8);
            float w = e0.y;
            w = fmaf(e1.x, hid[0], w); w = fmaf(e1.y, hid[1], w); w = fmaf(e1.z, hid[2], w); w = fmaf(e1.w, hid[3], w);
            w = fmaf(e2.x, hid[4], w); w = fmaf(e2.y, hid[5], w); w = fmaf(e2.z, hid[6], w); w = fmaf(e2.w, hid[7], w);
            v[c] = fmaxf(w, 0.0f) * leaky01(__uint_as_float(raw[c]) + e0.x);
        }
        // sum over the 16 rows of the point by recursive halving: after the step with mask h a lane keeps the half of
        // its columns selected by its bit h, so lane m ends with the totals of columns 2m and 2m+1.
#pragma unroll
        for (int h = 8, n = 16; h >= 1; h >>= 1, n >>= 1) {
            const bool up = (m & h) != 0;
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                if (t < n) {
                    const float keep = up ? v[n + t] : v[t];
                    const float send = up ? v[t] : v[n + t];
                    v[t] = keep + __shfl_xor_sync(FULL, send, h);
                }
            }
        }
        if (pt < N1) *reinterpret_cast<float2*>(prow + cb + 2 * m) = make_float2(v[0], v[1]);
    }
    // every warp has read its accumulator rows before the next tile's first MMA overwrites them (and before s_j / s_d change)
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    }   // tiles of this CTA

    if (warp == 0) tmem_dealloc(tmem, tmem_cols);
}

bool corr3d_stage1_tc_eligible(int Cout, int k, int precision) {
    if (precision != 1 && precision != 2) return false;
    if (k != TC_K) return false;                       // 16 neighbours = one half-warp of rows per point
    if (Cout % 32 != 0 || Cout < 32 || Cout > 256) return false;
    return tc_layout(Cout, precision == 2).total + 1024 <= 227 * 1024;
}

cudaError_t corr3d_stage1_tc(const float* xyz1, const float* xyz2, const int64_t* knn12, const Corr3dScratch& s,
                             const b200_corr3d_weights* w, int B, int Cout, int N1, int N2, int k, int precision,
                             cudaStream_t st) {
    (void)k;
    const int split = precision == 2;
    const size_t smem = (size_t)tc_layout(Cout, split).total + 1024;
    uint32_t cols = 32;
    while ((int)cols < Cout) cols <<= 1;
    const int tiles = ceil_div(N1, TC_ROWS / TC_K);
    const int tpc = tiles >= 128 ? 4 : (tiles >= 32 ? 2 : 1);      // tiles per CTA: amortise the per-CTA set-up, keep >= 16 CTAs per sample
    dim3 grid(ceil_div(tiles, tpc), B);
    cudaError_t e;
    if (split) {
        e = cudaFuncSetAttribute(corr3d_stage1_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        corr3d_stage1_tc_kernel<1><<<grid, TC_THREADS, smem, st>>>(xyz1, xyz2, knn12, s.A1, s.G2, w->W2, s.W1cT, w->b2, w->n2_Wa,
                                                                   w->n2_ba, w->n2_Wb, w->n2_bb, s.n2WcT, w->n2_bc, s.P, Cout, N1,
                                                                   N2, cols, tpc);
    } else {
        e = cudaFuncSetAttribute(corr3d_stage1_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        corr3d_stage1_tc_kernel<0><<<grid, TC_THREADS, smem, st>>>(xyz1, xyz2, knn12, s.A1, s.G2, w->W2, s.W1cT, w->b2, w->n2_Wa,
                                                                   w->n2_ba, w->n2_Wb, w->n2_bb, s.n2WcT, w->n2_bc, s.P, Cout, N1,
                                                                   N2, cols, tpc);
    }
    return cudaGetLastError();
}

}  // namespace b200
