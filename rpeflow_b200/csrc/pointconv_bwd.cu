// pointconv_bwd.cu — f1 backward: gradients of the PointConv body (b200_pointconv_fwd_linear, the Linear output y) with
// respect to both clouds, the features and the six parameters.
//
// Replaces the autograd graph of models/pointconv.py:33-61 / :90-122 (gathers, weight net, the [16 x k].[k x (C+3)]
// matmul and nn.Linear, whose [B,S,16,C+3] gathered rows, weight-net activations and [B,S,16(C+3)] mixed tensor the
// reference keeps for its backward).  Notation as the forward: F = [xyz ; feat] (C+3 channels), j_t = knn[s,t],
// rel_t = xyz_j - sampled_s, W[w,t] = lrelu(Wb.lrelu(Wa.rel_t + ba) + bb), M[s,w,c] = sum_t W[w,t] F[c,j_t],
// y[o,s] = sum_{w,c} L[o, w(C+3)+c] M[s,w,c] + bias[o].  Nothing but the inputs, the indices and the weights is read:
// M and W are recomputed.
//
// The B*S sampled points are walked in chunks of P points whose M and dM images (P x 16*Cp floats each) are at most
// 32 MB, so both stay in the 126 MB L2 between the kernels that produce and consume them and the scratch does not grow
// with the batch.  Per chunk:
//   pass 1  pcb_gemm_kernel<0>  dM = dy . L on tcgen05 (3xTF32): M = 128 points, N = 128 columns (w, c), K = Cout
//   pass 2  pcb_point_kernel    per point (one warp): W recomputed; per channel block M (-> chunk image), dF rows
//                               (scattered with float atomics), dW = dM . F^T; then the weight-net backward per
//                               (point, neighbour) row: dxyz / dsampled (atomics), weight-net parameter gradients
//                               summed by thread-owned entries into per-CTA partials (persistent grid, fixed order)
//   pass 3  pcb_gemm_kernel<1>  dL | dbias = dy^T . [M | 1] on tcgen05 (3xTF32), split-K over the chunk's points into
//                               per-split partials (each owned by one CTA; chunks add in launch order)
// After the last chunk: pcb_reduce_kernel sums the partials in a fixed order (dL, dbias, dWa, dba, dWb, dbb are bit-
// reproducible); pcb_finish_kernel turns the point-major dF rows into dfeat [B,C,N] and adds dF[0:3] into dxyz.
#include "sm100_async.cuh"

namespace b200 {

int pointconv_v2_rows(const float* xyz, const float* feat, float* Fpm, int B, int C, int N, cudaStream_t st);
int p2_cp(int C);

constexpr int PB_K = 16, PB_NW = 16;
constexpr int G_THREADS = 256, G_DEPTH = 3, G_TILE = 128 * 64;      // one operand tile: 128 rows x 16 floats (SW64)
constexpr int G_STAGE = 4 * G_TILE;                                  // Ah | Al | Bh | Bl (Bl right after Bh: one N = 256 MMA)
constexpr int G_SMEM = G_DEPTH * G_STAGE + 64 + 1024;
constexpr int PT_WARPS = 4, PT_THREADS = 32 * PT_WARPS;              // point kernel: one point per warp
constexpr int WN_N = 176;                                            // Wb 128 | bb 16 | Wa 24 | ba 8 (partial entry order)
constexpr int PT_PARTS = 4 * 148;
constexpr int64_t CHUNK_BYTES = 32ll << 20;

__device__ __forceinline__ float pb_lrelu(float v) { return v > 0.0f ? v : 0.1f * v; }
__device__ __forceinline__ float pb_slope(float act) { return act > 0.0f ? 1.0f : 0.1f; }   // lrelu(x) > 0 iff x > 0

// ---- chunking and scratch ---------------------------------------------------------------------------------------
struct PbPlan {
    int Cp, C3, NL, P, nsplit, mt, nt;
    int64_t Fpm, dFpm, Mc, dMc, dLp, wp, total;      // float offsets into the scratch
};
static inline int64_t pb_al(int64_t n) { return (n + 63) & ~int64_t(63); }
static PbPlan pb_plan(int B, int C, int Cout, int N, int S) {
    PbPlan p;
    p.Cp = p2_cp(C);
    p.C3 = C + 3;
    p.NL = 16 * p.Cp + 1;                                              // dL columns (w, c) and the bias column
    const int64_t BS = (int64_t)B * S;
    int64_t P = CHUNK_BYTES / (16 * (int64_t)p.Cp * 4) / 128 * 128;
    P = P < 128 ? 128 : P;
    const int64_t need = (BS + 127) / 128 * 128;
    p.P = (int)(P < need ? P : (need > 0 ? need : 128));
    p.mt = (Cout + 127) / 128;
    p.nt = (p.NL + 127) / 128;
    const int kbc = (p.P + 15) / 16, by_grid = 2 * 148 / (p.mt * p.nt);
    p.nsplit = by_grid < 1 ? 1 : (by_grid > kbc ? kbc : by_grid);
    int64_t o = 0;
    p.Fpm = o;  o += pb_al((int64_t)B * N * p.Cp);
    p.dFpm = o; o += pb_al((int64_t)B * N * p.Cp);
    p.Mc = o;   o += pb_al((int64_t)p.P * 16 * p.Cp);
    p.dMc = o;  o += pb_al((int64_t)p.P * 16 * p.Cp);
    p.dLp = o;  o += pb_al((int64_t)p.nsplit * Cout * p.NL);
    p.wp = o;   o += pb_al((int64_t)PT_PARTS * WN_N);
    p.total = o;
    return p;
}

// ---- passes 1 and 3: tcgen05 GEMM, 3xTF32 ---------------------------------------------------------------------
// D[m, n] = sum_k A(m, k) B(n, k) over one 128 x 128 tile; K blocks of 16 floats staged by all threads (global ->
// hi/lo split -> the forward's SW64 operand layout), one thread issues Ah.[Bh|Bl] (N = 256) and Al.Bh per 8-wide k-step
// and commits to the stage's mbarrier; a 3-deep ring lets the loads of the next blocks run under the MMAs.
//   OP 0 (dM):  A(m = point, k = o) = dy[b,o,s];  B(n = w*Cp + c, k = o) = L[o, w(C+3) + c];  out dMc[m][n]
//   OP 1 (dL):  A(m = o, k = point) = dy[b,o,s];  B(n, k = point) = Mc[k][n], column 16*Cp = 1 (-> dbias);
//               out part[split][o][n] (= on the first chunk, += after)
struct GemmArgs {
    const float* dy;
    const float* L;
    const float* Mc;
    float* out;
    int S, Cout, C3, Cp, NL, Pc, kb_per_split, first;
    int64_t p0;
};

template <int OP>
__device__ __forceinline__ float pb_load_a(const GemmArgs& a, int m, int k) {
    const int pt = OP == 0 ? m : k, o = OP == 0 ? k : m;
    if (pt >= a.Pc || o >= a.Cout) return 0.0f;
    const int64_t q = a.p0 + pt, b = q / a.S, s = q - b * a.S;
    return __ldg(a.dy + ((size_t)b * a.Cout + o) * a.S + s);
}
template <int OP>
__device__ __forceinline__ float pb_load_b(const GemmArgs& a, int n, int k) {
    if (OP == 0) {
        const int w = n / a.Cp, c = n - w * a.Cp;
        if (w >= PB_NW || c >= a.C3 || k >= a.Cout) return 0.0f;
        return __ldg(a.L + (size_t)k * PB_NW * a.C3 + (size_t)w * a.C3 + c);
    }
    if (k >= a.Pc) return 0.0f;
    const int nm = 16 * a.Cp;
    return n < nm ? __ldg(a.Mc + (size_t)k * nm + n) : (n == nm ? 1.0f : 0.0f);
}
__device__ __forceinline__ void pb_put(uint8_t* tile, int r, int kk, float v) {
    float* t = reinterpret_cast<float*>(tile);
    const uint32_t off = (sw64((uint32_t)r, (uint32_t)(kk >> 2)) >> 2) + (uint32_t)(kk & 3);
    const float hi = tf32_hi(v);
    t[off] = hi;
    t[G_TILE / 4 + off] = v - hi;
}

template <int OP>
__global__ void __launch_bounds__(G_THREADS, 1) pcb_gemm_kernel(GemmArgs a) {
    extern __shared__ uint8_t pb_smem_raw[];
    const uint32_t sbase = (smem_u32(pb_smem_raw) + 1023u) & ~1023u;
    uint8_t* g = pb_smem_raw + (sbase - smem_u32(pb_smem_raw));
    const uint32_t bars = sbase + G_DEPTH * G_STAGE;                 // empty[s] = bars + 8s, accf = bars + 32, slot = bars + 40
    const uint32_t bar_accf = bars + 32u, tmem_slot = bars + 40u;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(g + G_DEPTH * G_STAGE + 40);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.x * 128, n0 = blockIdx.y * 128;
    const int Mreal = OP == 0 ? a.Pc : a.Cout, Nreal = OP == 0 ? 16 * a.Cp : a.NL;
    int kb0 = 0, nkb;
    if (OP == 0) {
        nkb = (a.Cout + 15) / 16;
    } else {
        const int kbc = (a.Pc + 15) / 16;
        kb0 = blockIdx.z * a.kb_per_split;
        nkb = kb0 >= kbc ? 0 : min(a.kb_per_split, kbc - kb0);
    }
    auto out_at = [&](int m, int n) -> float* {
        return OP == 0 ? a.out + (size_t)m * (16 * a.Cp) + n : a.out + ((size_t)blockIdx.z * a.Cout + m) * a.NL + n;
    };
    if (nkb == 0) {                                                  // an empty split: its partial is zero
        if (a.first)
            for (int e = tid; e < 128 * 128; e += G_THREADS) {
                const int m = m0 + (e >> 7), n = n0 + (e & 127);
                if (m < Mreal && n < Nreal) *out_at(m, n) = 0.0f;
            }
        return;
    }
    if (tid == 0) {
        for (uint32_t s = 0; s < G_DEPTH; ++s) mbar_init(bars + 8u * s, 1);
        mbar_init(bar_accf, 1);
        mbar_init_fence();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, 256);
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot_ptr;
    const uint32_t idesc1 = umma_idesc_tf32(128, 128), idesc2 = umma_idesc_tf32(128, 256);

    for (int i = 0; i < nkb; ++i) {
        const int s = i % G_DEPTH, kbase = (kb0 + i) * 16;
        if (i >= G_DEPTH) mbar_wait(bars + 8u * s, (uint32_t)((i / G_DEPTH - 1) & 1));   // the MMAs that read it are done
        uint8_t* st = g + s * G_STAGE;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = tid + u * G_THREADS;
            // coalesced order: along m for OP 0 (points), along k for OP 1 (points again)
            const int r = OP == 0 ? (e & 127) : (e >> 4), kk = OP == 0 ? (e >> 7) : (e & 15);
            pb_put(st, r, kk, pb_load_a<OP>(a, m0 + r, kbase + kk));
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = tid + u * G_THREADS, r = e & 127, kk = e >> 7;
            pb_put(st + 2 * G_TILE, r, kk, pb_load_b<OP>(a, n0 + r, kbase + kk));
        }
        fence_proxy_async();
        __syncthreads();
        if (tid == 0) {
            tcgen05_fence_after();
            const uint32_t a_hi = sbase + s * G_STAGE, a_lo = a_hi + G_TILE, b_hi = a_hi + 2 * G_TILE;
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                const uint64_t ah = umma_desc_sw64(a_hi + ks * 32), bh = umma_desc_sw64(b_hi + ks * 32);
                umma_tf32(tmem, ah, bh, idesc2, (uint32_t)((i | ks) != 0));               // [Ah.Bh | Ah.Bl]
                umma_tf32(tmem, umma_desc_sw64(a_lo + ks * 32), bh, idesc1, 1u);         // + Al.Bh
            }
            umma_commit(bars + 8u * s);
        }
    }
    if (tid == 0) umma_commit(bar_accf);
    mbar_wait(bar_accf, 0u);
    tcgen05_fence_after();
    {   // epilogue: warp -> TMEM lane quarter (warp & 3), column half (warp >> 2)
        const int qd = warp & 3, row = qd * 32 + lane, m = m0 + row;
        const uint32_t tbase = tmem + ((uint32_t)(qd * 32) << 16);
        for (int c0 = (warp >> 2) * 64; c0 < (warp >> 2) * 64 + 64; c0 += 8) {
            uint32_t r0[8], r1[8];
            tmem_ld(tbase + (uint32_t)c0, r0);
            tmem_ld(tbase + (uint32_t)(128 + c0), r1);
            tmem_ld_wait();
            if (m >= Mreal) continue;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int n = n0 + c0 + c;
                if (n >= Nreal) continue;
                const float v = __uint_as_float(r0[c]) + __uint_as_float(r1[c]);
                float* p = out_at(m, n);
                *p = (OP == 1 && !a.first) ? *p + v : v;
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

// ---- pass 2: per point ------------------------------------------------------------------------------------------
struct PointArgs {
    const float* xyz;
    const float* sampled;
    const int64_t* knn;
    const float* Fpm;
    const float* dMc;       // NULL: no dM (only M is wanted)
    float* Mc;              // NULL: M not wanted (no dL / dbias)
    float* dFpm;            // NULL: no dF
    float* dxyz;
    float* dsampled;
    float* part;            // NULL: no weight-net parameter gradients
    const float *Wa, *ba, *Wb, *bb;
    int N, S, C3, Cp, Pc, wnet;
    int64_t p0;
};

__global__ void __launch_bounds__(PT_THREADS) pcb_point_kernel(PointArgs a) {
    __shared__ float s_wn[WN_N];                                     // Wa 24 | ba 8 | Wb 128 | bb 16 (forward order)
    __shared__ __align__(16) float s_wt[PT_WARPS][PB_K][20];         // W[w][t] stored [t][w]
    __shared__ __align__(16) float s_dm[PT_WARPS][PB_NW][36];        // dM[w][c] of the current 32-channel block
    __shared__ __align__(16) float s_f[PT_WARPS][PB_K][36];          // F[c][j_t] of the current block
    __shared__ float s_dw[PT_WARPS][PB_NW][17];                      // dW[w][t]
    __shared__ int s_j[PT_WARPS][PB_K];
    __shared__ float s_row[PT_WARPS * PB_K][36];                     // rel[4] | h1[8] | dz2[16] | dz1[8] per (point, t) row
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int e = tid; e < WN_N; e += PT_THREADS)
        s_wn[e] = e < 24 ? __ldg(a.Wa + e) : e < 32 ? __ldg(a.ba + e - 24) : e < 160 ? __ldg(a.Wb + e - 32) : __ldg(a.bb + e - 160);
    float acc0 = 0.0f, acc1 = 0.0f;                                  // this thread's partial entries tid and tid + 128
    const int ntiles = (a.Pc + PT_WARPS - 1) / PT_WARPS;
    const int myw = lane >> 1, t0 = (lane & 1) * 8;
    __syncthreads();
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int pl = tile * PT_WARPS + warp;
        const bool live = pl < a.Pc;
        const int64_t q = a.p0 + (live ? pl : 0);
        const int b = (int)(q / a.S), s = (int)(q - (int64_t)b * a.S);
        float* row = s_row[warp * PB_K + (lane & 15)];
        if (lane < 16) {                                             // neighbour t = lane: rel, h1, W (the forward's order)
            const int t = lane;
            int64_t j = live ? __ldg(a.knn + ((size_t)b * a.S + s) * PB_K + t) : 0;
            if (j < 0) j += a.N;
            j = j < 0 ? 0 : (j >= a.N ? a.N - 1 : j);
            s_j[warp][t] = (int)j;
            float d[3], h1[8];
#pragma unroll
            for (int x = 0; x < 3; ++x) d[x] = __ldg(a.xyz + ((size_t)b * 3 + x) * a.N + j) - __ldg(a.sampled + ((size_t)b * 3 + x) * a.S + s);
#pragma unroll
            for (int o = 0; o < 8; ++o) {
                float v = s_wn[24 + o];
#pragma unroll
                for (int x = 0; x < 3; ++x) v = fmaf(s_wn[o * 3 + x], d[x], v);
                h1[o] = pb_lrelu(v);
            }
#pragma unroll
            for (int o = 0; o < PB_NW; ++o) {
                float v = s_wn[160 + o];
#pragma unroll
                for (int m = 0; m < 8; ++m) v = fmaf(s_wn[32 + o * 8 + m], h1[m], v);
                s_wt[warp][t][o] = pb_lrelu(v);
            }
#pragma unroll
            for (int x = 0; x < 3; ++x) row[x] = d[x];
#pragma unroll
            for (int m = 0; m < 8; ++m) row[4 + m] = h1[m];
        }
        __syncwarp();
        float dw[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) dw[i] = 0.0f;
        if (live) {
            const float* frow = a.Fpm + (size_t)b * a.N * a.Cp;
            const float* dmrow = a.dMc ? a.dMc + (size_t)pl * 16 * a.Cp : nullptr;
            for (int c0 = 0; c0 < a.Cp; c0 += 32) {
                const int c = c0 + lane;
                const bool ok = c < a.Cp;
                float f[PB_K], dm[PB_NW];
#pragma unroll
                for (int t = 0; t < PB_K; ++t) f[t] = ok ? __ldg(frow + (size_t)s_j[warp][t] * a.Cp + c) : 0.0f;
                if (a.Mc != nullptr && ok) {                         // M[w][c] = sum_t W[w][t] F[c][j_t]
                    float m[PB_NW];
#pragma unroll
                    for (int w = 0; w < PB_NW; ++w) m[w] = 0.0f;
#pragma unroll
                    for (int t = 0; t < PB_K; ++t) {
                        const float4* wt = reinterpret_cast<const float4*>(s_wt[warp][t]);
#pragma unroll
                        for (int w4 = 0; w4 < 4; ++w4) {
                            const float4 v = wt[w4];
                            m[w4 * 4 + 0] = fmaf(v.x, f[t], m[w4 * 4 + 0]);
                            m[w4 * 4 + 1] = fmaf(v.y, f[t], m[w4 * 4 + 1]);
                            m[w4 * 4 + 2] = fmaf(v.z, f[t], m[w4 * 4 + 2]);
                            m[w4 * 4 + 3] = fmaf(v.w, f[t], m[w4 * 4 + 3]);
                        }
                    }
                    float* mrow = a.Mc + (size_t)pl * 16 * a.Cp + c;
#pragma unroll
                    for (int w = 0; w < PB_NW; ++w) mrow[(size_t)w * a.Cp] = m[w];
                }
                if (dmrow == nullptr) continue;
#pragma unroll
                for (int w = 0; w < PB_NW; ++w) dm[w] = ok ? __ldg(dmrow + (size_t)w * a.Cp + c) : 0.0f;
                if (a.dFpm != nullptr && c < a.C3) {                 // dF[c][j_t] += sum_w W[w][t] dM[w][c]
                    float* drow = a.dFpm + (size_t)b * a.N * a.Cp + c;
#pragma unroll
                    for (int t = 0; t < PB_K; ++t) {
                        const float4* wt = reinterpret_cast<const float4*>(s_wt[warp][t]);
                        float gsum = 0.0f;
#pragma unroll
                        for (int w4 = 0; w4 < 4; ++w4) {
                            const float4 v = wt[w4];
                            gsum = fmaf(v.x, dm[w4 * 4 + 0], gsum);
                            gsum = fmaf(v.y, dm[w4 * 4 + 1], gsum);
                            gsum = fmaf(v.z, dm[w4 * 4 + 2], gsum);
                            gsum = fmaf(v.w, dm[w4 * 4 + 3], gsum);
                        }
                        atomicAdd(drow + (size_t)s_j[warp][t] * a.Cp, gsum);
                    }
                }
                if (!a.wnet) continue;
#pragma unroll
                for (int w = 0; w < PB_NW; ++w) s_dm[warp][w][lane] = dm[w];
#pragma unroll
                for (int t = 0; t < PB_K; ++t) s_f[warp][t][lane] = f[t];
                __syncwarp();
#pragma unroll 2
                for (int cc = 0; cc < 32; cc += 4) {                 // dW[w][t] += sum_c dM[w][c] F[c][j_t]: lane -> (w, 8 t)
                    const float4 x = *reinterpret_cast<const float4*>(&s_dm[warp][myw][cc]);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 y = *reinterpret_cast<const float4*>(&s_f[warp][t0 + i][cc]);
                        dw[i] = fmaf(x.x, y.x, fmaf(x.y, y.y, fmaf(x.z, y.z, fmaf(x.w, y.w, dw[i]))));
                    }
                }
                __syncwarp();
            }
        }
        if (a.wnet) {
#pragma unroll
            for (int i = 0; i < 8; ++i) s_dw[warp][myw][t0 + i] = dw[i];
            __syncwarp();
            if (lane < 16) {                                         // weight-net backward of row (point, t = lane)
                const int t = lane;
                float dz2[PB_NW], dz1[8], dr[3];
#pragma unroll
                for (int w = 0; w < PB_NW; ++w) dz2[w] = live ? s_dw[warp][w][t] * pb_slope(s_wt[warp][t][w]) : 0.0f;
#pragma unroll
                for (int m = 0; m < 8; ++m) {
                    float v = 0.0f;
#pragma unroll
                    for (int w = 0; w < PB_NW; ++w) v = fmaf(s_wn[32 + w * 8 + m], dz2[w], v);
                    dz1[m] = v * pb_slope(row[4 + m]);
                }
#pragma unroll
                for (int x = 0; x < 3; ++x) {
                    float v = 0.0f;
#pragma unroll
                    for (int m = 0; m < 8; ++m) v = fmaf(s_wn[m * 3 + x], dz1[m], v);
                    dr[x] = v;
                }
#pragma unroll
                for (int w = 0; w < PB_NW; ++w) row[12 + w] = dz2[w];
#pragma unroll
                for (int m = 0; m < 8; ++m) row[28 + m] = dz1[m];
                if (live) {
                    const int j = s_j[warp][t];
#pragma unroll
                    for (int x = 0; x < 3; ++x) {
                        if (a.dxyz) atomicAdd(a.dxyz + ((size_t)b * 3 + x) * a.N + j, dr[x]);
                        if (a.dsampled) atomicAdd(a.dsampled + ((size_t)b * 3 + x) * a.S + s, -dr[x]);
                    }
                }
            }
        }
        __syncthreads();
        if (a.part != nullptr) {                                     // thread-owned entries, rows in a fixed order
            for (int r = 0; r < PT_WARPS * PB_K; ++r) {
                const float* R = s_row[r];
                {
                    const int e = tid;                               // < 128: dWb[w][m] = dz2[w] h1[m]
                    acc0 = fmaf(R[12 + (e >> 3)], R[4 + (e & 7)], acc0);
                }
                const int e = tid + 128;
                if (e < 144) acc1 += R[12 + e - 128];                                      // dbb
                else if (e < 168) acc1 = fmaf(R[28 + (e - 144) / 3], R[(e - 144) % 3], acc1);   // dWa[m][x] = dz1[m] rel[x]
                else if (e < WN_N) acc1 += R[28 + e - 168];                                // dba
            }
        }
        __syncthreads();
    }
    if (a.part != nullptr) {
        float* mp = a.part + (size_t)blockIdx.x * WN_N;
        mp[tid] += acc0;
        if (tid + 128 < WN_N) mp[tid + 128] += acc1;
    }
}

// ---- after the chunks ----------------------------------------------------------------------------------------
struct ReduceArgs {
    const float* dLp;
    const float* wp;
    float *L, *bias, *Wa, *ba, *Wb, *bb;
    int Cout, C3, Cp, NL, nsplit, nparts;
};
__global__ void __launch_bounds__(256) pcb_reduce_kernel(ReduceArgs a) {
    const int64_t nl = (int64_t)a.Cout * PB_NW * a.C3, total = nl + a.Cout + WN_N;
    for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < total; l += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.0f;
        if (l < nl + a.Cout) {
            float* dst;
            int64_t src;
            if (l < nl) {
                const int o = (int)(l / (PB_NW * a.C3)), r = (int)(l - (int64_t)o * PB_NW * a.C3), w = r / a.C3, c = r - w * a.C3;
                dst = a.L ? a.L + l : nullptr;
                src = (int64_t)o * a.NL + w * a.Cp + c;
            } else {
                const int o = (int)(l - nl);
                dst = a.bias ? a.bias + o : nullptr;
                src = (int64_t)o * a.NL + 16 * a.Cp;
            }
            if (dst == nullptr) continue;
            for (int g = 0; g < a.nsplit; ++g) s += __ldg(a.dLp + (int64_t)g * a.Cout * a.NL + src);
            *dst = s;
        } else {
            const int e = (int)(l - nl - a.Cout);
            float* dst = e < 128 ? (a.Wb ? a.Wb + e : nullptr) : e < 144 ? (a.bb ? a.bb + e - 128 : nullptr)
                       : e < 168 ? (a.Wa ? a.Wa + e - 144 : nullptr) : (a.ba ? a.ba + e - 168 : nullptr);
            if (dst == nullptr) continue;
            for (int p = 0; p < a.nparts; ++p) s += __ldg(a.wp + (size_t)p * WN_N + e);
            *dst = s;
        }
    }
}

// dFpm [B][N][Cp] point-major -> dfeat [B][C][N]; dxyz [B][3][N] += dFpm[..][0:3]
__global__ void __launch_bounds__(256) pcb_finish_kernel(const float* __restrict__ dFpm, float* __restrict__ dxyz,
                                                         float* __restrict__ dfeat, int C, int Cp, int N) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, n0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int n = n0 + ty * 4 + u, c = c0 + tx;
        tile[ty * 4 + u][tx] = (n < N && c < C + 3) ? dFpm[((size_t)b * N + n) * Cp + c] : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int c = c0 + ty * 4 + u, n = n0 + tx;
        if (n >= N || c >= C + 3) continue;
        const float v = tile[tx][ty * 4 + u];
        if (c < 3) { if (dxyz) dxyz[((size_t)b * 3 + c) * N + n] += v; }
        else if (dfeat) dfeat[((size_t)b * C + (c - 3)) * N + n] = v;
    }
}

}  // namespace b200

extern "C" int64_t b200_pointconv_bwd_scratch_floats(int B, int C, int Cout, int N, int S) {
    if (B < 0 || C < 0 || Cout < 1 || N < 1 || S < 0) return 0;
    return b200::pb_plan(B, C, Cout, N, S).total;
}

extern "C" int b200_pointconv_bwd(const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                                  const b200_pointconv_weights* w, const float* grad_y, const b200_pointconv_grads* grads,
                                  float* scratch, int B, int C, int Cout, int N, int S, int k, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0 || S == 0) || (xyz && sampled_xyz && knn && grad_y && scratch && (feat || C == 0)),
                 "b200_pointconv_bwd: null pointer");
    B200_REQUIRE(w != nullptr && grads != nullptr, "b200_pointconv_bwd: null weight or gradient struct");
    B200_REQUIRE(w->Wa && w->ba && w->Wb && w->bb && w->L && w->bias, "b200_pointconv_bwd: null weight pointer");
    B200_REQUIRE(B >= 0 && C >= 0 && Cout >= 1 && N >= 1 && S >= 0, "b200_pointconv_bwd: bad sizes");
    B200_REQUIRE(B <= 65535, "b200_pointconv_bwd: B exceeds the grid limit");
    B200_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "b200_pointconv_bwd: scratch must be 16-byte aligned");
    if (k != PB_K || Cout > 256 || N > 65536) {
        set_error("b200_pointconv_bwd: built for k = 16 neighbours, out_channels <= 256 and N <= 65536 (got k=%d, out=%d, N=%d)",
                  k, Cout, N);
        return B200_ENOSUP;
    }
    if (B == 0 || S == 0) return B200_OK;
    cudaStream_t st = as_stream(stream);
    const b200_pointconv_grads& g = *grads;
    const PbPlan pl = pb_plan(B, C, Cout, N, S);
    const bool need_params = g.Wa || g.ba || g.Wb || g.bb;
    const bool need_wnet = need_params || g.xyz || g.sampled_xyz;
    const bool need_dF = g.xyz || (g.feat && C > 0);
    const bool need_dL = g.L || g.bias;
    const bool need_dM = need_wnet || need_dF;
    if (!need_dM && !need_dL) return B200_OK;

    float* Fpm = scratch + pl.Fpm;
    float* dFpm = need_dF ? scratch + pl.dFpm : nullptr;
    if (g.xyz) B200_CUDA(cudaMemsetAsync(g.xyz, 0, sizeof(float) * 3 * (size_t)B * N, st));
    if (g.sampled_xyz) B200_CUDA(cudaMemsetAsync(g.sampled_xyz, 0, sizeof(float) * 3 * (size_t)B * S, st));
    if (dFpm) B200_CUDA(cudaMemsetAsync(dFpm, 0, sizeof(float) * (size_t)B * N * pl.Cp, st));
    if (need_params) B200_CUDA(cudaMemsetAsync(scratch + pl.wp, 0, sizeof(float) * (size_t)PT_PARTS * WN_N, st));
    const int er = pointconv_v2_rows(xyz, feat, Fpm, B, C, N, st);
    if (er != B200_OK) return er;
    B200_CUDA(cudaFuncSetAttribute(pcb_gemm_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, G_SMEM));
    B200_CUDA(cudaFuncSetAttribute(pcb_gemm_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, G_SMEM));

    const int64_t BS = (int64_t)B * S;
    for (int64_t p0 = 0; p0 < BS; p0 += pl.P) {
        const int Pc = (int)(BS - p0 < pl.P ? BS - p0 : pl.P);
        GemmArgs ga{grad_y, w->L, scratch + pl.Mc, nullptr, S, Cout, pl.C3, pl.Cp, pl.NL, Pc, 0, p0 == 0, p0};
        if (need_dM) {
            ga.out = scratch + pl.dMc;
            pcb_gemm_kernel<0><<<dim3(ceil_div(Pc, 128), ceil_div(16 * pl.Cp, 128)), G_THREADS, G_SMEM, st>>>(ga);
            B200_LAUNCH_CHECK("pcb_gemm_kernel<dM>");
        }
        PointArgs pa{xyz, sampled_xyz, knn, Fpm, need_dM ? scratch + pl.dMc : nullptr, need_dL ? scratch + pl.Mc : nullptr,
                     dFpm, g.xyz, g.sampled_xyz, need_params ? scratch + pl.wp : nullptr, w->Wa, w->ba, w->Wb, w->bb,
                     N, S, pl.C3, pl.Cp, Pc, need_wnet ? 1 : 0, p0};
        const int tiles = ceil_div(Pc, PT_WARPS);
        pcb_point_kernel<<<tiles < PT_PARTS ? tiles : PT_PARTS, PT_THREADS, 0, st>>>(pa);
        B200_LAUNCH_CHECK("pcb_point_kernel");
        if (need_dL) {
            ga.out = scratch + pl.dLp;
            ga.kb_per_split = ceil_div(ceil_div(Pc, 16), pl.nsplit);
            pcb_gemm_kernel<1><<<dim3(pl.mt, pl.nt, pl.nsplit), G_THREADS, G_SMEM, st>>>(ga);
            B200_LAUNCH_CHECK("pcb_gemm_kernel<dL>");
        }
    }
    if (need_dL || need_params) {
        ReduceArgs ra{scratch + pl.dLp, scratch + pl.wp, g.L, g.bias, g.Wa, g.ba, g.Wb, g.bb, Cout, pl.C3, pl.Cp, pl.NL,
                      pl.nsplit, PT_PARTS};
        if (!need_dL) ra.L = ra.bias = nullptr;
        if (!need_params) ra.Wa = ra.ba = ra.Wb = ra.bb = nullptr;
        const int64_t total = (int64_t)Cout * PB_NW * pl.C3 + Cout + WN_N;
        pcb_reduce_kernel<<<ceil_div(total, 256), 256, 0, st>>>(ra);
        B200_LAUNCH_CHECK("pcb_reduce_kernel");
    }
    if (need_dF) {
        pcb_finish_kernel<<<dim3(ceil_div(N, 32), ceil_div(C + 3, 32), B), 256, 0, st>>>(dFpm, g.xyz, C > 0 ? g.feat : nullptr,
                                                                                       C, pl.Cp, N);
        B200_LAUNCH_CHECK("pcb_finish_kernel");
    }
    return B200_OK;
}
