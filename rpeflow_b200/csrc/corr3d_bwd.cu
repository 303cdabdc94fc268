// corr3d_bwd.cu — a5 backward: gradients of the pwc3d_core point cost volume (Correlation3D.forward) with respect to
// both clouds, both feature maps and all 16 parameters, fp32 FFMA arithmetic.
//
// Replaces the autograd graph of models/pwc3d_core.py:69-117 (the [B,2C+3,N,k] concat, 8 1x1 convs, 4 gathers and 2
// mul+sum reductions, with their [B,C,N,k] activations kept for backward).  Same algebra as the forward (corr3d.cu):
// layer 1 factorises into per-point terms, so its backward is per-row work plus two per-point GEMMs.  Per row (i,s),
// j = knn12[i,s], m = knn11[i,s], d = xyz2_j - xyz1_i, e = xyz1_m - xyz1_i:
//
//   pass 0  corr3d_prep_weights + pointwise_linear x2 (corr3d.cu): W2^T, W1c^T, Wc^T, and A1 / G2 recomputed
//   pass 1  corr3d_bwd_stage2   : dv = G_i*P_m, dP_m += v*G_i (scatter), weight_net1 backward, dxyz1[m] += de, [i] -= de
//   pass 2  corr3d_bwd_stage1   : z1,h1,z2,h2,w2 recomputed per tile; dz2 = dP_i*w2*lrelu'(z2); dW2 += dz2 (x) h1;
//                                 dz1 = (W2^T dz2)*lrelu'(z1); dA1_i = sum_s dz1; dG2_j += dz1 (scatter); dW1c += dz1 (x) d;
//                                 weight_net2 backward of dP_i*h2; dxyz2[j] += dd, dxyz1[i] -= dd
//   pass 3  corr3d_bwd_reduce   : the per-CTA weight-gradient partials of passes 1-2 summed into the outputs
//   pass 4  linear_bwd_x / linear_bwd_w : dfeat = W1{a,b}^T dA1/dG2 (channel-first); dW1{a,b}, db1 split-K over B*N
//
// Passes 1 and 2 are persistent: each CTA walks tiles and keeps its weight gradients in shared memory / registers,
// except dW2 (Cout^2 floats, larger than what is left of shared memory next to the two row tiles), which each CTA
// accumulates in its own slice of the scratch (L2-resident read-modify-write, no atomics).  Every weight gradient is
// then one fixed-order sum over the CTAs' partials.  The partials themselves are not reproducible: dP, dG2, dxyz and the
// split-K dW1a/dW1b/db1 use global float atomics, and the Wc/bc, W1c and b2 partials shared-memory float atomics; every
// stage-1 gradient reads dP.  Only the weight_net1 3->8->8 gradients (thread-owned sums) are bit-reproducible.
//
// b200_corr3d_bwd_det runs the same passes with DET = true and no float atomics anywhere:
//   - knn11 and knn12 are inverted first: rows r = (b*N1 + i)*k + s sorted by key b*N + clamp(idx) (cub radix sort,
//     stable, so ascending r inside a destination) and segment offsets per destination (CSR);
//   - pass 1 writes the dP rows relu(vpre)*g_i and the de rows to row buffers; its Wc / bc partials go to per-warp slices
//     (CTA-owned scratch, read-modify-write) summed in warp order;
//   - corr3d_det_pull_kernel sums, per destination, its rows in ascending r: dP and dxyz1 (minus the point's own de rows
//     in ascending s) over knn11, then after pass 2 dG2 and dxyz2 over knn12;
//   - pass 2 writes dz1 rows (into the buffer that held the dP rows) and t = dd + de rows; du2, the Wc / bc / b2 and W1c
//     partials are per-tile reductions in ascending row order; the point's own -t, summed in ascending s, is subtracted
//     from dxyz1 by the one CTA that owns the point;
//   - pass 4 writes its split-K partials to scratch and linear_bwd_w_reduce_kernel sums them in ascending split order.
#include <algorithm>
#include <climits>

#include <cub/device/device_radix_sort.cuh>

#include "corr3d_common.cuh"

namespace b200 {

constexpr int BWD_THREADS = 256;
constexpr int WN_SMALL = 104;                           // Wb 64 | bb 8 | Wa 24 | ba 8 (the 3->8->8 part of a weight net)

static inline int bwd_parts(int Cout) { return Cout <= 256 ? 296 : 148; }     // persistent CTAs (2 or 1 per B200 SM)
__host__ __device__ inline int c4of(int C) { return (C + 3) & ~3; }

// Per-CTA partial layout: stage-1 section then stage-2 section.
struct PartLayout {
    int64_t W2, b2, W1c, n2Wc, n2bc, n2s, n1Wc, n1bc, n1s, total;
};
__host__ __device__ inline PartLayout part_layout(int C) {
    PartLayout L;
    const int64_t C4 = (C + 3) & ~3;
    int64_t o = 0;
    L.W2 = o;   o += C4 * C4;                           // [C4][C4]
    L.b2 = o;   o += C4;
    L.W1c = o;  o += 3 * C4;                            // [C][3]
    L.n2Wc = o; o += 8 * C4;                            // [C][8]
    L.n2bc = o; o += C4;
    L.n2s = o;  o += WN_SMALL;
    L.n1Wc = o; o += 8 * C4;
    L.n1bc = o; o += C4;
    L.n1s = o;  o += WN_SMALL;
    L.total = o;
    return L;
}

struct BwdScratch {
    Corr3dScratch f;            // A1, G2 (recomputed here), W2T, W1cT, n1WcT, n2WcT; its P is not used (read from the forward's)
    float *dP, *dA1, *dG2, *part;
    int64_t total;
};
static inline BwdScratch carve_bwd(float* base, int B, int Cout, int N1, int N2) {
    BwdScratch s;
    s.f = carve(base, B, Cout, N1, N2);
    int64_t off = s.f.total;
    auto take = [&](int64_t n) { float* p = base ? base + off : nullptr; off += align4(n); return p; };
    s.dP = take((int64_t)B * N1 * Cout);
    s.dA1 = take((int64_t)B * N1 * Cout);
    s.dG2 = take((int64_t)B * N2 * Cout);
    s.part = take((int64_t)bwd_parts(Cout) * part_layout(Cout).total);
    s.total = off;
    return s;
}

// Row buffers of the deterministic path (passed last, so the DET = false kernels keep their parameter layout).
struct DetRows {
    float* rows;        // [B*N1*k][c4of(C)]: pass 1 dP rows, pass 2 dz1 rows; NULL = not needed
    float4* xrows;      // [B*N1*k]: pass 1 de, pass 2 t = dd + de (w = 0); NULL = not needed
    float* wslice;      // pass 1: [CTA][warp][9][C] Wc (8 rows) and bc partials
};

// ---- device helpers -------------------------------------------------------------------------------------------
__device__ __forceinline__ float lrelu_d(float pre) { return pre > 0.0f ? 1.0f : 0.1f; }     // torch: slope where x <= 0

// u1 = relu(Wa.e + ba), u2 = relu(Wb.u1 + bb) in weight_net_hidden's operation order
__device__ __forceinline__ void wn_hidden2(const float* __restrict__ Wa, const float* __restrict__ ba, const float* __restrict__ Wb,
                                           const float* __restrict__ bb, float ex, float ey, float ez, float* u1, float* u2) {
#pragma unroll
    for (int o = 0; o < 8; ++o) {
        float s = __ldg(ba + o);
        s = fmaf(__ldg(Wa + o * 3 + 0), ex, s);
        s = fmaf(__ldg(Wa + o * 3 + 1), ey, s);
        s = fmaf(__ldg(Wa + o * 3 + 2), ez, s);
        u1[o] = fmaxf(s, 0.0f);
    }
#pragma unroll
    for (int o = 0; o < 8; ++o) {
        float s = __ldg(bb + o);
#pragma unroll
        for (int i = 0; i < 8; ++i) s = fmaf(__ldg(Wb + o * 8 + i), u1[i], s);
        u2[o] = fmaxf(s, 0.0f);
    }
}

// Backward of the 3->8->8 part of a weight net for one row: du2 in, du2pre/du1pre (pre-activation gradients) and de out.
__device__ __forceinline__ void wn_small_bwd(const float* __restrict__ Wa, const float* __restrict__ Wb, const float* u1,
                                             const float* u2, float* du2, float* du1, float* de) {
#pragma unroll
    for (int q = 0; q < 8; ++q) du2[q] = u2[q] > 0.0f ? du2[q] : 0.0f;
#pragma unroll
    for (int p = 0; p < 8; ++p) {
        float s = 0.0f;
#pragma unroll
        for (int q = 0; q < 8; ++q) s = fmaf(__ldg(Wb + q * 8 + p), du2[q], s);
        du1[p] = u1[p] > 0.0f ? s : 0.0f;
    }
#pragma unroll
    for (int x = 0; x < 3; ++x) {
        float s = 0.0f;
#pragma unroll
        for (int p = 0; p < 8; ++p) s = fmaf(__ldg(Wa + p * 3 + x), du1[p], s);
        de[x] = s;
    }
}

// Warp reduce-scatter of 8 per-lane values: afterwards lane L holds the warp sum of v[L / 4] (9 shuffles, not 40).
__device__ __forceinline__ float warp_reduce8(const float* v, int lane) {
    float a[4], b2[2];
    const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float keep = h16 ? v[i + 4] : v[i], send = h16 ? v[i] : v[i + 4];
        a[i] = keep + __shfl_xor_sync(FULL, send, 16);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const float keep = h8 ? a[i + 2] : a[i], send = h8 ? a[i] : a[i + 2];
        b2[i] = keep + __shfl_xor_sync(FULL, send, 8);
    }
    float x = (h4 ? b2[1] : b2[0]) + __shfl_xor_sync(FULL, h4 ? b2[0] : b2[1], 4);
    x += __shfl_xor_sync(FULL, x, 2);
    x += __shfl_xor_sync(FULL, x, 1);
    return x;
}

// Per-row small-net gradients, summed over the rows of a tile by thread-owned entries (two row halves per entry).
//   entry t: [0,64) Wb[q][p] | [64,72) bb[q] | [72,96) Wa[p][x] | [96,104) ba[p]
__device__ __forceinline__ float wn_small_entry(int t, int r, const float* du2s, const float* du1s, const float* u1s,
                                                const float* es) {
    if (t < 64) return du2s[r * 8 + (t >> 3)] * u1s[r * 8 + (t & 7)];
    if (t < 72) return du2s[r * 8 + t - 64];
    if (t < 96) { const int q = t - 72; return du1s[r * 8 + q / 3] * es[r * 4 + q % 3]; }
    return du1s[r * 8 + t - 96];
}
__device__ __forceinline__ void wn_small_flush(float* part_small, float acc, float* s_tmp, int tid) {
    // threads [0,104) and [128,232) hold the two halves of the same entries
    __syncthreads();
    if (tid >= 128 && tid < 128 + WN_SMALL) s_tmp[tid - 128] = acc;
    __syncthreads();
    if (tid < WN_SMALL) part_small[tid] = acc + s_tmp[tid];
}

// ---- pass 1: stage-2 backward --------------------------------------------------------------------------------
// Tile = 16 points x k rows.  Warp w owns points w and w+8; its lanes walk the channels.
// Dynamic smem: Gs[C][17] | u1[rows][8] | u2[rows][8] | e[rows][4] | du2[rows][8] | du1[rows][8] | jj[rows] | sWc[C][9]
// DET: dP rows and de rows go to det.rows / det.xrows (dP, dxyz1 only flag what is needed), sWc is replaced by det.wslice.
constexpr int S2_TP = 16;
template <bool DET>
__global__ void __launch_bounds__(BWD_THREADS)
corr3d_bwd_stage2_kernel(const float* __restrict__ xyz1, const int64_t* __restrict__ knn11, const float* __restrict__ P,
                         const float* __restrict__ G, const float* __restrict__ Wa, const float* __restrict__ ba,
                         const float* __restrict__ Wb, const float* __restrict__ bb, const float* __restrict__ Wc,
                         const float* __restrict__ bc, float* __restrict__ dP, float* __restrict__ dxyz1,
                         float* __restrict__ part, int64_t part_stride, int B, int C, int N1, int k, int small, DetRows det) {
    extern __shared__ float4 smem_f4[];
    float* Gs = reinterpret_cast<float*>(smem_f4);
    const int rows = S2_TP * k;
    float* u1s = Gs + (size_t)C * 17;
    float* u2s = u1s + rows * 8;
    float* es = u2s + rows * 8;
    float* du2s = es + rows * 4;
    float* du1s = du2s + rows * 8;
    int* jj = reinterpret_cast<int*>(du1s + rows * 8);
    float* sWc = reinterpret_cast<float*>(jj + rows);            // [C][9]: Wc row gradient then bc
    __shared__ float s_tmp[WN_SMALL];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const PartLayout L = part_layout(C);
    float* mypart = part + (size_t)blockIdx.x * part_stride;

    float* wslice = nullptr;                                          // DET: this warp's [9][C] Wc / bc slice
    if constexpr (DET) {
        wslice = det.wslice + ((size_t)blockIdx.x * (BWD_THREADS / 32) + warp) * 9 * C;
        for (int e = lane; e < C * 9; e += 32) wslice[e] = 0.0f;
    } else {
        for (int e = tid; e < C * 9; e += BWD_THREADS) sWc[e] = 0.0f;
    }
    float small_acc = 0.0f;
    const int tiles_per_b = (N1 + S2_TP - 1) / S2_TP;
    for (int tile = blockIdx.x; tile < B * tiles_per_b; tile += gridDim.x) {
        const int b = tile / tiles_per_b, i0 = (tile - b * tiles_per_b) * S2_TP;
        const size_t row0 = ((size_t)b * N1 + i0) * k;                // global row of the tile's row 0
        __syncthreads();
        for (int e = tid; e < C * S2_TP; e += BWD_THREADS) {          // grad_out tile, coalesced over points
            const int o = e / S2_TP, pt = e - o * S2_TP;
            Gs[o * 17 + pt] = i0 + pt < N1 ? __ldg(G + ((size_t)b * C + o) * N1 + i0 + pt) : 0.0f;
        }
        for (int r = tid; r < rows; r += BWD_THREADS) {
            const int pt = r / k, i = min(i0 + pt, N1 - 1);
            int64_t m = __ldg(knn11 + ((size_t)b * N1 + i) * k + (r - pt * k));
            m = m < 0 ? 0 : (m >= N1 ? N1 - 1 : m);
            const float ex = __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + m) - __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + i);
            const float ey = __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + m) - __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + i);
            const float ez = __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + m) - __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + i);
            jj[r] = (int)m;
            es[r * 4 + 0] = ex; es[r * 4 + 1] = ey; es[r * 4 + 2] = ez; es[r * 4 + 3] = 0.0f;
            wn_hidden2(Wa, ba, Wb, bb, ex, ey, ez, u1s + r * 8, u2s + r * 8);
#pragma unroll
            for (int q = 0; q < 8; ++q) du2s[r * 8 + q] = 0.0f;
        }
        __syncthreads();

        for (int pt = warp; pt < S2_TP; pt += BWD_THREADS / 32) {
            if (i0 + pt >= N1) continue;                              // warp-uniform
            for (int o0 = 0; o0 < C; o0 += 32) {
                const int o = o0 + lane;
                const bool ok = o < C;
                float wc[8], gw[8], gb = 0.0f;
#pragma unroll
                for (int q = 0; q < 8; ++q) { wc[q] = ok ? __ldg(Wc + (size_t)o * 8 + q) : 0.0f; gw[q] = 0.0f; }
                const float bco = ok ? __ldg(bc + o) : 0.0f;
                const float g = ok ? Gs[o * 17 + pt] : 0.0f;
                for (int s = 0; s < k; ++s) {
                    const int r = pt * k + s, m = jj[r];
                    const float* u2 = u2s + r * 8;
                    float vpre = bco;
#pragma unroll
                    for (int q = 0; q < 8; ++q) vpre = fmaf(wc[q], u2[q], vpre);
                    const float pm = ok ? __ldg(P + ((size_t)b * N1 + m) * C + o) : 0.0f;
                    if constexpr (DET) {
                        if (dP != nullptr && ok) det.rows[(row0 + r) * c4of(C) + o] = fmaxf(vpre, 0.0f) * g;
                    } else {
                        if (dP != nullptr && ok) atomicAdd(dP + ((size_t)b * N1 + m) * C + o, fmaxf(vpre, 0.0f) * g);
                    }
                    const float dvpre = vpre > 0.0f ? g * pm : 0.0f;
                    float du2[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) { gw[q] = fmaf(dvpre, u2[q], gw[q]); du2[q] = wc[q] * dvpre; }
                    gb += dvpre;
                    if (small) {
                        const float red = warp_reduce8(du2, lane);
                        if ((lane & 3) == 0) du2s[r * 8 + (lane >> 2)] += red;     // the warp owns row r
                    }
                }
                if (ok) {
                    if constexpr (DET) {
#pragma unroll
                        for (int q = 0; q < 8; ++q) wslice[q * C + o] += gw[q];
                        wslice[8 * C + o] += gb;
                    } else {
#pragma unroll
                        for (int q = 0; q < 8; ++q) atomicAdd(sWc + o * 9 + q, gw[q]);
                        atomicAdd(sWc + o * 9 + 8, gb);
                    }
                }
            }
        }
        if (!small) continue;
        __syncthreads();
        for (int r = tid; r < rows; r += BWD_THREADS) {
            const int pt = r / k, i = i0 + pt;
            float du2[8], du1[8], de[3];
#pragma unroll
            for (int q = 0; q < 8; ++q) du2[q] = du2s[r * 8 + q];
            wn_small_bwd(Wa, Wb, u1s + r * 8, u2s + r * 8, du2, du1, de);
#pragma unroll
            for (int q = 0; q < 8; ++q) { du2s[r * 8 + q] = du2[q]; du1s[r * 8 + q] = du1[q]; }
            if (dxyz1 != nullptr && i < N1) {
                if constexpr (DET) {
                    det.xrows[row0 + r] = make_float4(de[0], de[1], de[2], 0.0f);
                } else {
                    const int m = jj[r];
#pragma unroll
                    for (int x = 0; x < 3; ++x) {
                        atomicAdd(dxyz1 + ((size_t)b * 3 + x) * N1 + m, de[x]);
                        atomicAdd(dxyz1 + ((size_t)b * 3 + x) * N1 + i, -de[x]);
                    }
                }
            }
        }
        __syncthreads();
        {
            const int t = tid & 127, half = tid >> 7;
            if (t < WN_SMALL)
                for (int r = half; r < rows; r += 2) small_acc += wn_small_entry(t, r, du2s, du1s, u1s, es);
        }
    }
    wn_small_flush(mypart + L.n1s, small_acc, s_tmp, tid);
    if constexpr (DET) {
        const float* cta = det.wslice + (size_t)blockIdx.x * (BWD_THREADS / 32) * 9 * C;
        for (int e = tid; e < C * 9; e += BWD_THREADS) {
            const int q = e / C, o = e - q * C;
            float s = 0.0f;
            for (int w = 0; w < BWD_THREADS / 32; ++w) s += cta[(size_t)w * 9 * C + e];
            if (q < 8) mypart[L.n1Wc + o * 8 + q] = s;
            else mypart[L.n1bc + o] = s;
        }
    } else {
        for (int e = tid; e < C * 9; e += BWD_THREADS) {
            const int o = e / 9, q = e - o * 9;
            if (q < 8) mypart[L.n1Wc + o * 8 + q] = sWc[e];
            else mypart[L.n1bc + o] = sWc[e];
        }
    }
}

// ---- pass 2: stage-1 backward --------------------------------------------------------------------------------
// Tile = TP points x k rows (TP*k <= 128).  Dynamic smem:
//   h1[rows][LD] (later dz1) | dz2[rows][LD] | u1[rows][8] | u2[rows][8] | d[rows][4] | du2[rows][8] | du1[rows][8] |
//   dd[rows][4] | jj[rows] | sWc[C][9] | sW1c[C][3] | sb2[C] | DET: dw[rows][LD] (dwpre, the weight_net2 output gradient)
static inline size_t s1_smem(int tp, int k, int C, bool det) {
    const size_t r = (size_t)tp * k, LD = c4of(C) + 4;
    return ((det ? 3 : 2) * r * LD + r * (8 + 8 + 4 + 8 + 8 + 4 + 1) + (size_t)C * 13) * sizeof(float);
}

// DET: dz1 rows and t rows go to det.rows / det.xrows (dG2, dxyz2 only flag what is needed); du2 and the Wc / bc / b2 /
// W1c partials are reduced per tile in ascending row order; dxyz1[i] -= (own t summed in ascending s), read-modify-write.
template <int KMAX, bool DET>
__global__ void __launch_bounds__(BWD_THREADS, 1)
corr3d_bwd_stage1_kernel(const float* __restrict__ xyz1, const float* __restrict__ xyz2, const int64_t* __restrict__ knn12,
                         const float* __restrict__ A1, const float* __restrict__ G2, const float* __restrict__ W2,
                         const float* __restrict__ W2T, const float* __restrict__ W1cT, const float* __restrict__ b2,
                         const float* __restrict__ Wa, const float* __restrict__ ba, const float* __restrict__ Wb,
                         const float* __restrict__ bb, const float* __restrict__ WcT, const float* __restrict__ bc,
                         const float* __restrict__ dP, float* __restrict__ dA1, float* __restrict__ dG2,
                         float* __restrict__ dxyz1, float* __restrict__ dxyz2, float* __restrict__ part, int64_t part_stride,
                         int B, int C, int N1, int N2, int k, int TP, DetRows det) {
    extern __shared__ float4 smem_f4[];
    float* smem = reinterpret_cast<float*>(smem_f4);
    const int rows = TP * k, C4 = c4of(C), LD = C4 + 4;
    float* h1 = smem;
    float* dz2 = h1 + (size_t)rows * LD;
    float* u1s = dz2 + (size_t)rows * LD;
    float* u2s = u1s + rows * 8;
    float* ds = u2s + rows * 8;
    float* du2s = ds + rows * 4;
    float* du1s = du2s + rows * 8;
    float* dds = du1s + rows * 8;
    int* jj = reinterpret_cast<int*>(dds + rows * 4);
    float* sWc = reinterpret_cast<float*>(jj + rows);       // [C][9]
    float* sW1c = sWc + C * 9;                              // [C][3]
    float* sb2 = sW1c + C * 3;                              // [C]
    float* dws = sb2 + C;                                   // DET only: [rows][LD]
    __shared__ float s_tmp[WN_SMALL];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const PartLayout L = part_layout(C);
    float* mypart = part + (size_t)blockIdx.x * part_stride;
    const bool warp_rows = (C & 31) == 0;                   // a warp's (point, channel) items share one point

    for (int e = tid; e < C * 13; e += BWD_THREADS) sWc[e] = 0.0f;
    const int nblk = (C4 / 4) * (C4 / 4);
    for (int bi = tid; bi < nblk; bi += BWD_THREADS) {      // this thread's dW2 blocks start at zero
        const int ob = bi / (C4 / 4), cb = bi - ob * (C4 / 4);
#pragma unroll
        for (int a = 0; a < 4; ++a)
            *reinterpret_cast<float4*>(mypart + L.W2 + (size_t)(ob * 4 + a) * C4 + cb * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float small_acc = 0.0f;
    const int tiles_per_b = (N1 + TP - 1) / TP;
    for (int tile = blockIdx.x; tile < B * tiles_per_b; tile += gridDim.x) {
        const int b = tile / tiles_per_b, i0 = (tile - b * tiles_per_b) * TP;
        const size_t row0 = ((size_t)b * N1 + i0) * k;      // global row of the tile's row 0
        __syncthreads();
        // (a) neighbour, offset, weight_net2 hidden layers per row
        for (int r = tid; r < rows; r += BWD_THREADS) {
            const int pt = r / k, i = min(i0 + pt, N1 - 1);
            int64_t j = __ldg(knn12 + ((size_t)b * N1 + i) * k + (r - pt * k));
            j = j < 0 ? 0 : (j >= N2 ? N2 - 1 : j);
            const float dx = __ldg(xyz2 + ((size_t)b * 3 + 0) * N2 + j) - __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + i);
            const float dy = __ldg(xyz2 + ((size_t)b * 3 + 1) * N2 + j) - __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + i);
            const float dz = __ldg(xyz2 + ((size_t)b * 3 + 2) * N2 + j) - __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + i);
            jj[r] = (int)j;
            ds[r * 4 + 0] = dx; ds[r * 4 + 1] = dy; ds[r * 4 + 2] = dz; ds[r * 4 + 3] = 0.0f;
            wn_hidden2(Wa, ba, Wb, bb, dx, dy, dz, u1s + r * 8, u2s + r * 8);
#pragma unroll
            for (int q = 0; q < 8; ++q) du2s[r * 8 + q] = 0.0f;
        }
        __syncthreads();
        // (b) h1 = lrelu(A1_i + G2_j + W1c.d); padding columns zero
        for (int e = tid; e < rows * C4; e += BWD_THREADS) {
            const int r = e / C4, c = e - r * C4;
            float v = 0.0f;
            if (c < C) {
                const int i = min(i0 + r / k, N1 - 1);
                v = __ldg(A1 + ((size_t)b * N1 + i) * C + c) + __ldg(G2 + ((size_t)b * N2 + jj[r]) * C + c) +
                    fmaf(__ldg(W1cT + 2 * C + c), ds[r * 4 + 2], fmaf(__ldg(W1cT + C + c), ds[r * 4 + 1], __ldg(W1cT + c) * ds[r * 4 + 0]));
                v = leaky01(v);
            }
            h1[(size_t)r * LD + c] = v;
            dz2[(size_t)r * LD + c] = 0.0f;
        }
        __syncthreads();
        // (c) per (point, out-channel): z2 for the k rows, h2, w2; dz2 -> smem; weight_net2 gradients
        for (int e = tid; e < TP * C; e += BWD_THREADS) {
            const int pt = e / C, o = e - pt * C, i = i0 + pt;
            float acc[KMAX];
            const float bias2 = __ldg(b2 + o);
#pragma unroll
            for (int s = 0; s < KMAX; ++s) acc[s] = bias2;
            const float* hrow = h1 + (size_t)pt * k * LD;
            for (int c = 0; c < C4; c += 4) {
                const float w0 = __ldg(W2T + (size_t)(c + 0) * C + o);
                const float w1 = c + 1 < C ? __ldg(W2T + (size_t)(c + 1) * C + o) : 0.0f;
                const float w2 = c + 2 < C ? __ldg(W2T + (size_t)(c + 2) * C + o) : 0.0f;
                const float w3 = c + 3 < C ? __ldg(W2T + (size_t)(c + 3) * C + o) : 0.0f;
#pragma unroll
                for (int s = 0; s < KMAX; ++s) {
                    if (s < k) {
                        const float4 h = *reinterpret_cast<const float4*>(hrow + (size_t)s * LD + c);
                        acc[s] = fmaf(w3, h.w, fmaf(w2, h.z, fmaf(w1, h.y, fmaf(w0, h.x, acc[s]))));
                    }
                }
            }
            float wc[8], gw[8], gb = 0.0f, gb2 = 0.0f;
#pragma unroll
            for (int q = 0; q < 8; ++q) { wc[q] = __ldg(WcT + (size_t)q * C + o); gw[q] = 0.0f; }
            const float bco = __ldg(bc + o);
            const float dp = i < N1 ? __ldg(dP + ((size_t)b * N1 + i) * C + o) : 0.0f;
#pragma unroll
            for (int s = 0; s < KMAX; ++s) {
                if (s < k) {
                    const int r = pt * k + s;
                    const float* u2 = u2s + r * 8;
                    float wpre = bco;
#pragma unroll
                    for (int q = 0; q < 8; ++q) wpre = fmaf(wc[q], u2[q], wpre);
                    const float z2 = acc[s];
                    const float d2 = dp * fmaxf(wpre, 0.0f) * lrelu_d(z2);
                    dz2[(size_t)r * LD + o] = d2;
                    if constexpr (DET) {
                        dws[(size_t)r * LD + o] = wpre > 0.0f ? dp * leaky01(z2) : 0.0f;
                        continue;
                    }
                    gb2 += d2;
                    const float dwpre = wpre > 0.0f ? dp * leaky01(z2) : 0.0f;
                    float du2[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) { gw[q] = fmaf(dwpre, u2[q], gw[q]); du2[q] = wc[q] * dwpre; }
                    gb += dwpre;
                    if (warp_rows) {
                        const float red = warp_reduce8(du2, lane);
                        if ((lane & 3) == 0) atomicAdd(du2s + r * 8 + (lane >> 2), red);
                    } else {
#pragma unroll
                        for (int q = 0; q < 8; ++q) atomicAdd(du2s + r * 8 + q, du2[q]);
                    }
                }
            }
            if constexpr (!DET) {
#pragma unroll
                for (int q = 0; q < 8; ++q) atomicAdd(sWc + o * 9 + q, gw[q]);
                atomicAdd(sWc + o * 9 + 8, gb);
                atomicAdd(sb2 + o, gb2);
            }
        }
        __syncthreads();
        if constexpr (DET) {
            // (c') du2 = Wc^T dw per row (ascending o); Wc / bc / b2 partials += sums over the tile's rows (ascending r)
            for (int e = tid; e < rows * 8; e += BWD_THREADS) {
                const int r = e >> 3, q = e & 7;
                float s = 0.0f;
                for (int o = 0; o < C; ++o) s = fmaf(__ldg(WcT + (size_t)q * C + o), dws[(size_t)r * LD + o], s);
                du2s[e] = s;
            }
            for (int e = tid; e < C * 10; e += BWD_THREADS) {
                const int o = e / 10, q = e - o * 10;
                float s = 0.0f;
                if (q < 8)
                    for (int r = 0; r < rows; ++r) s = fmaf(dws[(size_t)r * LD + o], u2s[r * 8 + q], s);
                else
                    for (int r = 0; r < rows; ++r) s += (q == 8 ? dws : dz2)[(size_t)r * LD + o];
                if (q < 9) sWc[o * 9 + q] += s;
                else sb2[o] += s;
            }
        }
        // (d) dW2 += dz2^T h1 over the tile's rows: 4x4 register blocks, read-modify-write of this CTA's partial
        for (int bi = tid; bi < nblk; bi += BWD_THREADS) {
            const int ob = bi / (C4 / 4), cb = bi - ob * (C4 / 4);
            float a16[4][4];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) a16[a][c] = 0.0f;
            for (int r = 0; r < rows; ++r) {
                const float4 g = *reinterpret_cast<const float4*>(dz2 + (size_t)r * LD + ob * 4);
                const float4 h = *reinterpret_cast<const float4*>(h1 + (size_t)r * LD + cb * 4);
                const float gv[4] = {g.x, g.y, g.z, g.w}, hv[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int c = 0; c < 4; ++c) a16[a][c] = fmaf(gv[a], hv[c], a16[a][c]);
            }
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                float4* p = reinterpret_cast<float4*>(mypart + L.W2 + (size_t)(ob * 4 + a) * C4 + cb * 4);
                float4 v = *p;
                v.x += a16[a][0]; v.y += a16[a][1]; v.z += a16[a][2]; v.w += a16[a][3];
                *p = v;
            }
        }
        __syncthreads();
        // (e) per (point, in-channel): dh1 = W2^T dz2 for the k rows; dz1 -> h1 (in place); dA1, dG2, dW1c
        for (int e = tid; e < TP * C; e += BWD_THREADS) {
            const int pt = e / C, c = e - pt * C, i = i0 + pt;
            float acc[KMAX];
#pragma unroll
            for (int s = 0; s < KMAX; ++s) acc[s] = 0.0f;
            const float* grow = dz2 + (size_t)pt * k * LD;
            for (int o = 0; o < C4; o += 4) {
                const float w0 = __ldg(W2 + (size_t)(o + 0) * C + c);
                const float w1 = o + 1 < C ? __ldg(W2 + (size_t)(o + 1) * C + c) : 0.0f;
                const float w2 = o + 2 < C ? __ldg(W2 + (size_t)(o + 2) * C + c) : 0.0f;
                const float w3 = o + 3 < C ? __ldg(W2 + (size_t)(o + 3) * C + c) : 0.0f;
#pragma unroll
                for (int s = 0; s < KMAX; ++s) {
                    if (s < k) {
                        const float4 g = *reinterpret_cast<const float4*>(grow + (size_t)s * LD + o);
                        acc[s] = fmaf(w3, g.w, fmaf(w2, g.z, fmaf(w1, g.y, fmaf(w0, g.x, acc[s]))));
                    }
                }
            }
            float da = 0.0f, gx = 0.0f, gy = 0.0f, gz = 0.0f;
#pragma unroll
            for (int s = 0; s < KMAX; ++s) {
                if (s < k) {
                    const int r = pt * k + s;
                    float* hp = h1 + (size_t)r * LD + c;
                    const float dz1 = acc[s] * lrelu_d(*hp);         // h1 > 0 exactly when z1 > 0
                    *hp = dz1;
                    da += dz1;
                    if constexpr (DET) {
                        if (dG2 != nullptr && i < N1) det.rows[(row0 + r) * C4 + c] = dz1;
                        continue;
                    }
                    if (dG2 != nullptr && i < N1) atomicAdd(dG2 + ((size_t)b * N2 + jj[r]) * C + c, dz1);
                    gx = fmaf(dz1, ds[r * 4 + 0], gx); gy = fmaf(dz1, ds[r * 4 + 1], gy); gz = fmaf(dz1, ds[r * 4 + 2], gz);
                }
            }
            if (dA1 != nullptr && i < N1) dA1[((size_t)b * N1 + i) * C + c] = da;
            if constexpr (!DET) {
                atomicAdd(sW1c + c * 3 + 0, gx); atomicAdd(sW1c + c * 3 + 1, gy); atomicAdd(sW1c + c * 3 + 2, gz);
            }
        }
        __syncthreads();
        if constexpr (DET) {
            // (e') W1c partials += sum over the tile's rows of dz1 (x) d, ascending r
            for (int e = tid; e < C * 3; e += BWD_THREADS) {
                const int c = e / 3, x = e - c * 3;
                float s = 0.0f;
                for (int r = 0; r < rows; ++r) s = fmaf(h1[(size_t)r * LD + c], ds[r * 4 + x], s);
                sW1c[e] += s;
            }
        }
        // (f) dd = W1c^T dz1: one warp per row
        for (int r = warp; r < rows; r += BWD_THREADS / 32) {
            float sx = 0.0f, sy = 0.0f, sz = 0.0f;
            for (int c = lane; c < C; c += 32) {
                const float g = h1[(size_t)r * LD + c];
                sx = fmaf(__ldg(W1cT + c), g, sx); sy = fmaf(__ldg(W1cT + C + c), g, sy); sz = fmaf(__ldg(W1cT + 2 * C + c), g, sz);
            }
#pragma unroll
            for (int off = 16; off; off >>= 1) {
                sx += __shfl_xor_sync(FULL, sx, off); sy += __shfl_xor_sync(FULL, sy, off); sz += __shfl_xor_sync(FULL, sz, off);
            }
            if (lane == 0) { dds[r * 4 + 0] = sx; dds[r * 4 + 1] = sy; dds[r * 4 + 2] = sz; }
        }
        __syncthreads();
        // (g) weight_net2 3->8->8 backward per row; d-gradient to both clouds
        for (int r = tid; r < rows; r += BWD_THREADS) {
            const int pt = r / k, i = i0 + pt;
            float du2[8], du1[8], de[3];
#pragma unroll
            for (int q = 0; q < 8; ++q) du2[q] = du2s[r * 8 + q];
            wn_small_bwd(Wa, Wb, u1s + r * 8, u2s + r * 8, du2, du1, de);
#pragma unroll
            for (int q = 0; q < 8; ++q) { du2s[r * 8 + q] = du2[q]; du1s[r * 8 + q] = du1[q]; }
            if (i < N1) {
                if constexpr (DET) {
                    float t[3];
#pragma unroll
                    for (int x = 0; x < 3; ++x) { t[x] = dds[r * 4 + x] + de[x]; dds[r * 4 + x] = t[x]; }
                    if (dxyz2 != nullptr) det.xrows[row0 + r] = make_float4(t[0], t[1], t[2], 0.0f);
                } else {
                    const int j = jj[r];
#pragma unroll
                    for (int x = 0; x < 3; ++x) {
                        const float t = dds[r * 4 + x] + de[x];
                        if (dxyz2 != nullptr) atomicAdd(dxyz2 + ((size_t)b * 3 + x) * N2 + j, t);
                        if (dxyz1 != nullptr) atomicAdd(dxyz1 + ((size_t)b * 3 + x) * N1 + i, -t);
                    }
                }
            }
        }
        __syncthreads();
        if constexpr (DET) {
            // (g') the point's own t rows, summed in ascending s, leave dxyz1[i] (this CTA owns point i)
            if (dxyz1 != nullptr)
                for (int pt = tid; pt < TP && i0 + pt < N1; pt += BWD_THREADS)
#pragma unroll
                    for (int x = 0; x < 3; ++x) {
                        float s = 0.0f;
                        for (int q = 0; q < k; ++q) s += dds[(pt * k + q) * 4 + x];
                        float* p = dxyz1 + ((size_t)b * 3 + x) * N1 + i0 + pt;
                        *p = *p - s;
                    }
        }
        {
            const int t = tid & 127, half = tid >> 7;
            if (t < WN_SMALL)
                for (int r = half; r < rows; r += 2) small_acc += wn_small_entry(t, r, du2s, du1s, u1s, ds);
        }
    }
    wn_small_flush(mypart + L.n2s, small_acc, s_tmp, tid);
    for (int e = tid; e < C * 13; e += BWD_THREADS) {
        if (e < C * 9) {
            const int o = e / 9, q = e - o * 9;
            if (q < 8) mypart[L.n2Wc + o * 8 + q] = sWc[e];
            else mypart[L.n2bc + o] = sWc[e];
        } else if (e < C * 12) {
            mypart[L.W1c + (e - C * 9)] = sW1c[e - C * 9];
        } else {
            mypart[L.b2 + (e - C * 12)] = sb2[e - C * 12];
        }
    }
}

// ---- pass 3: sum of the per-CTA partials into the weight-gradient outputs ---------------------------------------
__device__ __forceinline__ void small_target(const b200_corr3d_grads& g, int net, int t, float** dst) {
    float* Wa = net ? g.n2_Wa : g.n1_Wa; float* ba = net ? g.n2_ba : g.n1_ba;
    float* Wb = net ? g.n2_Wb : g.n1_Wb; float* bb = net ? g.n2_bb : g.n1_bb;
    if (t < 64) *dst = Wb ? Wb + t : nullptr;
    else if (t < 72) *dst = bb ? bb + t - 64 : nullptr;
    else if (t < 96) *dst = Wa ? Wa + t - 72 : nullptr;
    else *dst = ba ? ba + t - 96 : nullptr;
}

__global__ void corr3d_bwd_reduce_kernel(const float* __restrict__ part, int64_t stride, int nparts, b200_corr3d_grads g,
                                         int C, int Cin, int do_s1, int do_s2) {
    const PartLayout L = part_layout(C);
    const int C4 = c4of(C), Kin = 2 * Cin + 3;
    for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < L.total; l += (int64_t)gridDim.x * blockDim.x) {
        float* dst = nullptr;
        const bool s2 = l >= L.n1Wc;
        if (s2 ? !do_s2 : !do_s1) continue;
        if (l < L.b2) {
            const int o = (int)(l / C4), c = (int)(l % C4);
            if (g.W2 && o < C && c < C) dst = g.W2 + (size_t)o * C + c;
        } else if (l < L.W1c) {
            const int o = (int)(l - L.b2);
            if (g.b2 && o < C) dst = g.b2 + o;
        } else if (l < L.n2Wc) {
            const int q = (int)(l - L.W1c), o = q / 3, x = q % 3;
            if (g.W1 && o < C) dst = g.W1 + (size_t)o * Kin + 2 * Cin + x;
        } else if (l < L.n2bc) {
            const int q = (int)(l - L.n2Wc);
            if (g.n2_Wc && q < 8 * C) dst = g.n2_Wc + q;
        } else if (l < L.n2s) {
            const int o = (int)(l - L.n2bc);
            if (g.n2_bc && o < C) dst = g.n2_bc + o;
        } else if (l < L.n1Wc) {
            small_target(g, 1, (int)(l - L.n2s), &dst);
        } else if (l < L.n1bc) {
            const int q = (int)(l - L.n1Wc);
            if (g.n1_Wc && q < 8 * C) dst = g.n1_Wc + q;
        } else if (l < L.n1s) {
            const int o = (int)(l - L.n1bc);
            if (g.n1_bc && o < C) dst = g.n1_bc + o;
        } else {
            small_target(g, 0, (int)(l - L.n1s), &dst);
        }
        if (dst == nullptr) continue;
        float s = 0.0f;
        for (int p = 0; p < nparts; ++p) s += __ldg(part + (size_t)p * stride + l);
        *dst = s;
    }
}

// ---- pass 4: linear backward ------------------------------------------------------------------------------------
// out[b,c,n] = sum_o W[o, coff + c] * D[b,n,o]      D point-major [B,N,Cout], out channel-first [B,Cin,N]
constexpr int LB_T = 64, LB_K = 16;
__global__ void __launch_bounds__(256)
linear_bwd_x_kernel(const float* __restrict__ D, const float* __restrict__ Wm, float* __restrict__ out, int Cout, int ldw,
                    int coff, int Cin, int N) {
    __shared__ __align__(16) float Ds[LB_K][LB_T];       // [o][n]
    __shared__ __align__(16) float Ws[LB_K][LB_T];       // [o][c]
    const int b = blockIdx.z, n0 = blockIdx.x * LB_T, c0 = blockIdx.y * LB_T;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;      // tx -> 4 points, ty -> 4 channels
    float acc[4][4] = {};
    for (int k0 = 0; k0 < Cout; k0 += LB_K) {
        __syncthreads();
        for (int e = threadIdx.x; e < LB_K * LB_T; e += 256) {
            const int kk = e % LB_K, nn = e / LB_K, o = k0 + kk, n = n0 + nn;
            Ds[kk][nn] = (o < Cout && n < N) ? __ldg(D + ((size_t)b * N + n) * Cout + o) : 0.0f;
        }
        for (int e = threadIdx.x; e < LB_K * LB_T; e += 256) {
            const int cc = e % LB_T, kk = e / LB_T, o = k0 + kk, c = c0 + cc;
            Ws[kk][cc] = (o < Cout && c < Cin) ? __ldg(Wm + (size_t)o * ldw + coff + c) : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < LB_K; ++kk) {
            const float4 d = *reinterpret_cast<const float4*>(&Ds[kk][tx * 4]);
            const float4 w = *reinterpret_cast<const float4*>(&Ws[kk][ty * 4]);
            const float dv[4] = {d.x, d.y, d.z, d.w}, wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[a][j] = fmaf(wv[a], dv[j], acc[a][j]);
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int c = c0 + ty * 4 + a;
        if (c >= Cin) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n < N) out[((size_t)b * Cin + c) * N + n] = acc[a][j];
        }
    }
}

// dW[o, coff + c] += sum_{b,n} D[b,n,o] * X[b,c,n]; column c == Cin is the constant 1 (-> dbias[o]).  Split-K over B*N.
// DET: split z writes its partials to part[z][o][c] (c < Cx) instead; linear_bwd_w_reduce_kernel sums them.  There the
// bias column is present when bias_col is set, whether or not dbias is wanted, so the split plan (and with it every sum
// order) does not depend on which gradients the caller asks for.
template <bool DET>
__global__ void __launch_bounds__(256)
linear_bwd_w_kernel(const float* __restrict__ D, const float* __restrict__ X, float* __restrict__ dW, float* __restrict__ dbias,
                    int Cout, int ldw, int coff, int Cin, int N, int64_t BN, int64_t chunk, float* __restrict__ part,
                    int bias_col) {
    __shared__ __align__(16) float Ds[LB_K][LB_T];       // [p][o]
    __shared__ __align__(16) float Xs[LB_K][LB_T];       // [p][c]
    const int o0 = blockIdx.x * LB_T, c0 = blockIdx.y * LB_T;
    const int64_t p_begin = blockIdx.z * chunk, p_end = min(BN, p_begin + chunk);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;      // tx -> 4 in-channels, ty -> 4 out-channels
    const int Cx = (DET ? bias_col : dbias != nullptr) ? Cin + 1 : Cin;
    float acc[4][4] = {};
    for (int64_t p0 = p_begin; p0 < p_end; p0 += LB_K) {
        __syncthreads();
        for (int e = threadIdx.x; e < LB_K * LB_T; e += 256) {
            const int oo = e % LB_T, kk = e / LB_T, o = o0 + oo;
            const int64_t p = p0 + kk;
            Ds[kk][oo] = (o < Cout && p < p_end) ? __ldg(D + p * Cout + o) : 0.0f;
        }
        for (int e = threadIdx.x; e < LB_K * LB_T; e += 256) {
            const int kk = e % LB_K, cc = e / LB_K, c = c0 + cc;
            const int64_t p = p0 + kk;
            float v = 0.0f;
            if (p < p_end && c < Cx) {
                const int64_t b = p / N, n = p - b * N;
                v = c < Cin ? __ldg(X + ((size_t)b * Cin + c) * N + n) : 1.0f;
            }
            Xs[kk][cc] = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < LB_K; ++kk) {
            const float4 d = *reinterpret_cast<const float4*>(&Ds[kk][ty * 4]);
            const float4 x = *reinterpret_cast<const float4*>(&Xs[kk][tx * 4]);
            const float dv[4] = {d.x, d.y, d.z, d.w}, xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[a][j] = fmaf(dv[a], xv[j], acc[a][j]);
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int o = o0 + ty * 4 + a;
        if (o >= Cout) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = c0 + tx * 4 + j;
            if constexpr (DET) {
                if (c < Cx) part[((size_t)blockIdx.z * Cout + o) * Cx + c] = acc[a][j];
            } else {
                if (c < Cin) { if (dW) atomicAdd(dW + (size_t)o * ldw + coff + c, acc[a][j]); }
                else if (c == Cin && dbias) atomicAdd(dbias + o, acc[a][j]);
            }
        }
    }
}

// dW[o, coff + c] (c < Cin) and dbias[o] (c == Cin < Cx) = the splits' partials of linear_bwd_w_kernel<true>, ascending z
__global__ void __launch_bounds__(256)
linear_bwd_w_reduce_kernel(const float* __restrict__ part, int splits, float* __restrict__ dW, float* __restrict__ dbias,
                           int Cout, int ldw, int coff, int Cin, int Cx) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < (int64_t)Cout * Cx; e += (int64_t)gridDim.x * blockDim.x) {
        const int o = (int)(e / Cx), c = (int)(e - (int64_t)o * Cx);
        float s = 0.0f;
        for (int z = 0; z < splits; ++z) s += __ldg(part + (size_t)z * Cout * Cx + e);
        if (c < Cin) { if (dW) dW[(size_t)o * ldw + coff + c] = s; }
        else if (dbias) dbias[o] = s;
    }
}

// split-K plan of linear_bwd_w_kernel: number of splits, and the rows of B*N each takes
static int64_t linear_bwd_w_splits(int Cout, int Cx, int64_t BN, int64_t* chunk_out) {
    const int tiles = ceil_div(Cout, LB_T) * ceil_div(Cx, LB_T);
    int64_t splits = std::max<int64_t>(1, std::min<int64_t>((BN + 255) / 256, (2 * 148 + tiles - 1) / tiles));
    int64_t chunk = (BN + splits - 1) / splits;
    chunk = (chunk + LB_K - 1) / LB_K * LB_K;
    *chunk_out = chunk;
    return (BN + chunk - 1) / chunk;
}

// bias_col: X gets the constant-1 column (always when dbias is wanted; on the DET path also when it is not).
// DET: part holds linear_bwd_w_splits(Cout, Cx, B*N) * Cout * Cx floats (det_lpart_floats covers both calls).
template <bool DET>
static cudaError_t launch_linear_bwd_w(const float* D, const float* X, float* dW, float* dbias, bool bias_col, int Cout,
                                       int ldw, int coff, int Cin, int B, int N, cudaStream_t st, float* part = nullptr) {
    const int64_t BN = (int64_t)B * N;
    const int Cx = bias_col ? Cin + 1 : Cin;
    int64_t chunk;
    const int64_t splits = linear_bwd_w_splits(Cout, Cx, BN, &chunk);
    linear_bwd_w_kernel<DET><<<dim3(ceil_div(Cout, LB_T), ceil_div(Cx, LB_T), (unsigned)splits), 256, 0, st>>>(
        D, X, dW, dbias, Cout, ldw, coff, Cin, N, BN, chunk, part, bias_col ? 1 : 0);
    if (DET) {
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        linear_bwd_w_reduce_kernel<<<ceil_div((int64_t)Cout * Cx, 256), 256, 0, st>>>(part, (int)splits, dW, dbias, Cout, ldw,
                                                                                      coff, Cin, Cx);
    }
    return cudaGetLastError();
}

template <int KMAX, bool DET>
static cudaError_t launch_bwd_stage1(const float* xyz1, const float* xyz2, const int64_t* knn12, const BwdScratch& s,
                                     const b200_corr3d_weights* w, float* dA1, float* dG2, float* dxyz1, float* dxyz2,
                                     int64_t part_stride, int nparts, int B, int C, int N1, int N2, int k, cudaStream_t st,
                                     DetRows det = DetRows{}) {
    int TP = 128 / k > 0 ? 128 / k : 1;
    while (TP > 1 && s1_smem(TP, k, C, DET) > 200 * 1024) TP /= 2;
    if (s1_smem(TP, k, C, DET) > 227 * 1024) return cudaErrorInvalidConfiguration;
    const size_t smem = s1_smem(TP, k, C, DET);
    auto kern = corr3d_bwd_stage1_kernel<KMAX, DET>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<nparts, BWD_THREADS, smem, st>>>(xyz1, xyz2, knn12, s.f.A1, s.f.G2, w->W2, s.f.W2T, s.f.W1cT, w->b2, w->n2_Wa, w->n2_ba,
                                           w->n2_Wb, w->n2_bb, s.f.n2WcT, w->n2_bc, s.dP, dA1, dG2, dxyz1, dxyz2, s.part,
                                           part_stride, B, C, N1, N2, k, TP, det);
    return cudaGetLastError();
}

// ---- deterministic path: inverse knn index (CSR) and the pull ------------------------------------------------------
// key of row r = b*N + clamp(knn[r]) with the kernels' clamp rule; value = r
__global__ void corr3d_det_keys_kernel(const int64_t* __restrict__ knn, int64_t R, int64_t rows_per_b, int N,
                                       unsigned* __restrict__ keys, int* __restrict__ vals) {
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        int64_t m = __ldg(knn + r);
        m = m < 0 ? 0 : (m >= N ? N - 1 : m);
        keys[r] = (unsigned)((r / rows_per_b) * N + m);
        vals[r] = (int)r;
    }
}

// offs[d] = the first sorted position whose key is >= d, d in [0, D]: destination d's rows are [offs[d], offs[d+1])
__global__ void corr3d_det_offsets_kernel(const unsigned* __restrict__ keys, int64_t R, int64_t D, int* __restrict__ offs) {
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p <= R; p += (int64_t)gridDim.x * blockDim.x) {
        const int64_t lo = p > 0 ? (int64_t)keys[p - 1] + 1 : 0, hi = p < R ? (int64_t)keys[p] : D;
        for (int64_t d = lo; d <= hi; ++d) offs[d] = (int)p;
    }
}

// Destination d = b*N + n sums its rows (order[offs[d] .. offs[d+1])) in ascending row order from +0.0: dst[d][0..C)
// from rows[r][0..C) (row stride c4of(C), 128-bit loads) and dxyz[b][0..3)[n] from xrows[r].  self_k > 0 (knn11):
// the point's own rows d*self_k + s, summed in ascending s, are then subtracted from the dxyz sum.  NULL dst / dxyz: skipped.
__global__ void __launch_bounds__(256)
corr3d_det_pull_kernel(const int* __restrict__ order, const int* __restrict__ offs, const float* __restrict__ rows,
                       float* __restrict__ dst, const float4* __restrict__ xrows, float* __restrict__ dxyz, int self_k, int C,
                       int N, int64_t D) {
    const int nq = dst ? c4of(C) / 4 : 0, items = nq + (dxyz ? 1 : 0);
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < D * items; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t d = e / items;
        const int q = (int)(e - d * items), p0 = __ldg(offs + d), p1 = __ldg(offs + d + 1);
        float4 s = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (q < nq) {
            for (int p = p0; p < p1; ++p) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(rows + (size_t)__ldg(order + p) * (nq * 4)) + q);
                s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            }
            float* out = dst + d * C + q * 4;
            out[0] = s.x;
            if (q * 4 + 1 < C) out[1] = s.y;
            if (q * 4 + 2 < C) out[2] = s.z;
            if (q * 4 + 3 < C) out[3] = s.w;
        } else {
            for (int p = p0; p < p1; ++p) {
                const float4 v = __ldg(xrows + __ldg(order + p));
                s.x += v.x; s.y += v.y; s.z += v.z;
            }
            float4 own = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            for (int t = 0; t < self_k; ++t) {
                const float4 v = __ldg(xrows + d * self_k + t);
                own.x += v.x; own.y += v.y; own.z += v.z;
            }
            const int64_t b = d / N, n = d - b * N;
            dxyz[(b * 3 + 0) * N + n] = s.x - own.x;
            dxyz[(b * 3 + 1) * N + n] = s.y - own.y;
            dxyz[(b * 3 + 2) * N + n] = s.z - own.z;
        }
    }
}

// Scratch of b200_corr3d_bwd_det: the float scratch of b200_corr3d_bwd, then the row buffers, the CSR lists of both
// index sets, the sort's key / value buffers and its temporary storage.  Every region starts 256-byte aligned.
struct DetScratch {
    BwdScratch s;
    DetRows rows;
    float* lpart;                               // pass-4 split-K partials
    unsigned *keys_in, *keys_out;
    int *vals_in, *order11, *order12, *offs11, *offs12;
    void* sort_tmp;
    size_t sort_bytes, total;
};

static int key_bits(int64_t D) {                // bits of the largest key D - 1 (at least 1)
    int b = 1;
    while (b < 32 && (int64_t(1) << b) < D) ++b;
    return b;
}

static cudaError_t sort_bytes(int64_t R, int64_t D, size_t* bytes) {
    *bytes = 0;
    return cub::DeviceRadixSort::SortPairs(nullptr, *bytes, (const unsigned*)nullptr, (unsigned*)nullptr, (const int*)nullptr,
                                           (int*)nullptr, (int)R, 0, key_bits(D));
}

// pass-4 partials of the DET path: the call over feat1 always carries the bias column (Cx = Cin + 1, B*N1 rows), the
// call over feat2 never does (Cx = Cin, B*N2 rows); the two run one after the other on one buffer
static int64_t det_lpart_floats(int B, int Cin, int Cout, int N1, int N2) {
    int64_t c1, c2;
    return std::max(linear_bwd_w_splits(Cout, Cin + 1, (int64_t)B * N1, &c1) * Cout * (Cin + 1),
                    linear_bwd_w_splits(Cout, Cin, (int64_t)B * N2, &c2) * Cout * Cin);
}

static cudaError_t carve_det(char* base, int B, int Cin, int Cout, int N1, int N2, int k, DetScratch* out) {
    DetScratch& d = *out;
    const int64_t R = (int64_t)B * N1 * k, D11 = (int64_t)B * N1, D12 = (int64_t)B * N2;
    size_t sb11 = 0, sb12 = 0;
    cudaError_t e = sort_bytes(R, D11, &sb11);
    if (e == cudaSuccess) e = sort_bytes(R, D12, &sb12);
    if (e != cudaSuccess) return e;
    d.sort_bytes = std::max(sb11, sb12);
    size_t off = 0;
    auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off += (bytes + 255) & ~size_t(255); return p; };
    const int64_t nf = carve_bwd(nullptr, B, Cout, N1, N2).total;
    d.s = carve_bwd(reinterpret_cast<float*>(take(sizeof(float) * nf)), B, Cout, N1, N2);
    d.rows.rows = reinterpret_cast<float*>(take(sizeof(float) * R * c4of(Cout)));
    d.rows.xrows = reinterpret_cast<float4*>(take(sizeof(float4) * R));
    d.rows.wslice = reinterpret_cast<float*>(take(sizeof(float) * (size_t)bwd_parts(Cout) * (BWD_THREADS / 32) * 9 * Cout));
    d.lpart = reinterpret_cast<float*>(take(sizeof(float) * det_lpart_floats(B, Cin, Cout, N1, N2)));
    d.keys_in = reinterpret_cast<unsigned*>(take(sizeof(unsigned) * R));
    d.keys_out = reinterpret_cast<unsigned*>(take(sizeof(unsigned) * R));
    d.vals_in = reinterpret_cast<int*>(take(sizeof(int) * R));
    d.order11 = reinterpret_cast<int*>(take(sizeof(int) * R));
    d.order12 = reinterpret_cast<int*>(take(sizeof(int) * R));
    d.offs11 = reinterpret_cast<int*>(take(sizeof(int) * (D11 + 1)));
    d.offs12 = reinterpret_cast<int*>(take(sizeof(int) * (D12 + 1)));
    d.sort_tmp = take(d.sort_bytes);
    d.total = off;
    return cudaSuccess;
}

// knn -> order (rows grouped by destination, ascending inside a group) and offs (D + 1 segment offsets)
static cudaError_t build_csr(const int64_t* knn, int B, int N1, int N, int k, const DetScratch& d, int* order, int* offs,
                             cudaStream_t st) {
    const int64_t R = (int64_t)B * N1 * k, D = (int64_t)B * N;
    const int grid = (int)std::min<int64_t>(ceil_div(R + 1, 256), 148 * 8);
    corr3d_det_keys_kernel<<<grid, 256, 0, st>>>(knn, R, (int64_t)N1 * k, N, d.keys_in, d.vals_in);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    size_t bytes = d.sort_bytes;
    e = cub::DeviceRadixSort::SortPairs(d.sort_tmp, bytes, d.keys_in, d.keys_out, d.vals_in, order, (int)R, 0, key_bits(D), st);
    if (e != cudaSuccess) return e;
    corr3d_det_offsets_kernel<<<grid, 256, 0, st>>>(d.keys_out, R, D, offs);
    return cudaGetLastError();
}

static cudaError_t launch_pull(const int* order, const int* offs, const float* rows, float* dst, const float4* xrows, float* dxyz,
                               int self_k, int C, int N, int64_t D, cudaStream_t st) {
    const int64_t items = D * ((dst ? c4of(C) / 4 : 0) + (dxyz ? 1 : 0));
    if (items == 0) return cudaSuccess;
    corr3d_det_pull_kernel<<<(int)std::min<int64_t>(ceil_div(items, 256), 148 * 16), 256, 0, st>>>(order, offs, rows, dst, xrows,
                                                                                                  dxyz, self_k, C, N, D);
    return cudaGetLastError();
}

// the argument checks of both entries (fn names the entry in the messages)
static int bwd_check(const char* fn, const float* xyz1, const float* feat1, const float* xyz2, const float* feat2,
                     const int64_t* knn12, const int64_t* knn11, const b200_corr3d_weights* w, const float* grad_out,
                     const float* fwd_scratch, const b200_corr3d_grads* grads, const void* scratch, int B, int Cin, int Cout,
                     int N1, int N2, int k) {
    B200_REQUIRE((B == 0) || (xyz1 && feat1 && xyz2 && feat2 && knn12 && knn11 && w && grad_out && fwd_scratch && grads && scratch),
                 "%s: null pointer", fn);
    B200_REQUIRE(B >= 0 && Cin >= 1 && Cout >= 1 && N1 >= 1 && N2 >= 1, "%s: bad sizes", fn);
    B200_REQUIRE(k >= 1 && k <= 32, "%s: k must be in [1,32] (got %d)", fn, k);
    B200_REQUIRE(Cout <= 512, "%s: Cout=%d exceeds 512", fn, Cout);
    B200_REQUIRE(B <= 65535, "%s: B exceeds the grid limit", fn);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0 && (reinterpret_cast<uintptr_t>(fwd_scratch) & 15) == 0,
                 "%s: scratch and fwd_scratch must be 16-byte aligned", fn);
    B200_REQUIRE(w != nullptr && grads != nullptr, "%s: null weight or gradient struct", fn);
    B200_REQUIRE(w->W1 && w->b1 && w->W2 && w->b2 && w->n1_Wa && w->n1_ba && w->n1_Wb && w->n1_bb && w->n1_Wc && w->n1_bc &&
                 w->n2_Wa && w->n2_ba && w->n2_Wb && w->n2_bb && w->n2_Wc && w->n2_bc, "%s: null weight pointer", fn);
    return B200_OK;
}

}  // namespace b200

extern "C" int64_t b200_corr3d_bwd_scratch_floats(int B, int Cin, int Cout, int N1, int N2, int k) {
    (void)Cin; (void)k;
    return b200::carve_bwd(nullptr, B, Cout, N1, N2).total;
}


extern "C" int64_t b200_corr3d_bwd_det_scratch_bytes(int B, int Cin, int Cout, int N1, int N2, int k) {
    if (B < 1 || Cin < 1 || Cout < 1 || N1 < 1 || N2 < 1 || k < 1) return 0;
    b200::DetScratch d;
    const cudaError_t e = b200::carve_det(nullptr, B, Cin, Cout, N1, N2, k, &d);
    if (e != cudaSuccess) return b200::cuda_fail(e, "b200_corr3d_bwd_det_scratch_bytes (cub::DeviceRadixSort temporary size)");
    return (int64_t)d.total;
}

namespace b200 {

// The body of both entries: DET = false is b200_corr3d_bwd (float atomics), DET = true b200_corr3d_bwd_det.
template <bool DET>
static int corr3d_bwd_run(const char* fn, const float* xyz1, const float* feat1, const float* xyz2, const float* feat2,
                          const int64_t* knn12, const int64_t* knn11, const b200_corr3d_weights* w, const float* grad_out,
                          const float* fwd_scratch, const b200_corr3d_grads* grads, float* scratch, int B, int Cin, int Cout,
                          int N1, int N2, int k, b200_stream_t stream) {
    const int rc = bwd_check(fn, xyz1, feat1, xyz2, feat2, knn12, knn11, w, grad_out, fwd_scratch, grads, scratch, B, Cin, Cout,
                             N1, N2, k);
    if (rc != B200_OK) return rc;
    if (B == 0) return B200_OK;
    if (DET)
        B200_REQUIRE((int64_t)B * N1 * k <= INT_MAX && (int64_t)B * N2 <= INT_MAX, "%s: B*N1*k and B*N2 must be below 2^31", fn);
    cudaStream_t st = as_stream(stream);
    const b200_corr3d_grads& g = *grads;
    DetScratch d{};
    if (DET) {
        const cudaError_t e = carve_det(reinterpret_cast<char*>(scratch), B, Cin, Cout, N1, N2, k, &d);
        if (e != cudaSuccess) return cuda_fail(e, "cub::DeviceRadixSort (temporary size)");
    }
    const BwdScratch s = DET ? d.s : carve_bwd(scratch, B, Cout, N1, N2);
    const float* P = carve(const_cast<float*>(fwd_scratch), B, Cout, N1, N2).P;
    const int Kin = 2 * Cin + 3;
    const PartLayout L = part_layout(Cout);
    const int nparts = bwd_parts(Cout);

    const bool need_n1 = g.n1_Wa || g.n1_ba || g.n1_Wb || g.n1_bb || g.n1_Wc || g.n1_bc;
    const bool need_n2 = g.n2_Wa || g.n2_ba || g.n2_Wb || g.n2_bb || g.n2_Wc || g.n2_bc;
    const bool need_s1 = need_n2 || g.W1 || g.b1 || g.W2 || g.b2 || g.feat1 || g.feat2 || g.xyz1 || g.xyz2;
    const bool need_dA1 = g.feat1 || g.W1 || g.b1, need_dG2 = g.feat2 || g.W1;
    if (!need_s1 && !need_n1 && !g.xyz1) return B200_OK;

    if (DET) {
        // every output is written whole, nothing accumulates: no zero-fill.  need_s1 covers g.xyz1, g.xyz2 and need_dG2.
        if (need_s1) B200_CUDA(build_csr(knn11, B, N1, N1, k, d, d.order11, d.offs11, st));
        if (need_dG2 || g.xyz2) B200_CUDA(build_csr(knn12, B, N1, N2, k, d, d.order12, d.offs12, st));
    } else {
        if (g.xyz1) B200_CUDA(cudaMemsetAsync(g.xyz1, 0, sizeof(float) * 3 * B * (size_t)N1, st));
        if (g.xyz2) B200_CUDA(cudaMemsetAsync(g.xyz2, 0, sizeof(float) * 3 * B * (size_t)N2, st));
        if (g.W1) B200_CUDA(cudaMemsetAsync(g.W1, 0, sizeof(float) * (size_t)Cout * Kin, st));
        if (g.b1) B200_CUDA(cudaMemsetAsync(g.b1, 0, sizeof(float) * Cout, st));
        if (need_s1) B200_CUDA(cudaMemsetAsync(s.dP, 0, sizeof(float) * (size_t)B * N1 * Cout, st));
        if (need_s1 && need_dG2) B200_CUDA(cudaMemsetAsync(s.dG2, 0, sizeof(float) * (size_t)B * N2 * Cout, st));
    }

    // pass 1: stage-2 backward (dP, weight_net1, dxyz1 via e)
    {
        const int rows = S2_TP * k;
        const size_t smem = ((size_t)Cout * 17 + (size_t)rows * (8 + 8 + 4 + 8 + 8 + 1) + (size_t)Cout * 9) * sizeof(float);
        auto kern = corr3d_bwd_stage2_kernel<DET>;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e, "corr3d_bwd_stage2_kernel(attr)");
        kern<<<nparts, BWD_THREADS, smem, st>>>(
            xyz1, knn11, P, grad_out, w->n1_Wa, w->n1_ba, w->n1_Wb, w->n1_bb, w->n1_Wc, w->n1_bc, need_s1 ? s.dP : nullptr,
            g.xyz1, s.part, L.total, B, Cout, N1, k, (need_n1 || g.xyz1) ? 1 : 0, d.rows);
        B200_LAUNCH_CHECK("corr3d_bwd_stage2_kernel");
    }
    if (DET && need_s1)        // dP and dxyz1 = pulled de - own de; pass 2 reads dP
        B200_CUDA(launch_pull(d.order11, d.offs11, d.rows.rows, s.dP, d.rows.xrows, g.xyz1, k, Cout, N1, (int64_t)B * N1, st));
    if (need_s1) {
        const cudaError_t ep = corr3d_prep_and_linears(feat1, feat2, w, s.f, B, Cin, Cout, N1, N2, st);
        if (ep != cudaSuccess) return cuda_fail(ep, "corr3d_prep_weights / pointwise_linear_kernel");
        float* dA1 = need_dA1 ? s.dA1 : nullptr;
        float* dG2 = need_dG2 ? s.dG2 : nullptr;
        cudaError_t e;
        if (k <= 4) e = launch_bwd_stage1<4, DET>(xyz1, xyz2, knn12, s, w, dA1, dG2, g.xyz1, g.xyz2, L.total, nparts, B, Cout, N1, N2, k, st, d.rows);
        else if (k <= 8) e = launch_bwd_stage1<8, DET>(xyz1, xyz2, knn12, s, w, dA1, dG2, g.xyz1, g.xyz2, L.total, nparts, B, Cout, N1, N2, k, st, d.rows);
        else if (k <= 16) e = launch_bwd_stage1<16, DET>(xyz1, xyz2, knn12, s, w, dA1, dG2, g.xyz1, g.xyz2, L.total, nparts, B, Cout, N1, N2, k, st, d.rows);
        else e = launch_bwd_stage1<32, DET>(xyz1, xyz2, knn12, s, w, dA1, dG2, g.xyz1, g.xyz2, L.total, nparts, B, Cout, N1, N2, k, st, d.rows);
        if (e != cudaSuccess) return cuda_fail(e, "corr3d_bwd_stage1_kernel");
        if (DET && (dG2 || g.xyz2))
            B200_CUDA(launch_pull(d.order12, d.offs12, d.rows.rows, dG2, d.rows.xrows, g.xyz2, 0, Cout, N2, (int64_t)B * N2, st));
    }
    corr3d_bwd_reduce_kernel<<<ceil_div(L.total, 256), 256, 0, st>>>(s.part, L.total, nparts, g, Cout, Cin, need_s1 ? 1 : 0,
                                                                      need_n1 ? 1 : 0);
    B200_LAUNCH_CHECK("corr3d_bwd_reduce_kernel");
    if (!need_s1) return B200_OK;

    // pass 4: linear backward
    if (g.feat1)
        linear_bwd_x_kernel<<<dim3(ceil_div(N1, LB_T), ceil_div(Cin, LB_T), B), 256, 0, st>>>(s.dA1, w->W1, g.feat1, Cout, Kin, 0,
                                                                                             Cin, N1);
    if (g.feat2)
        linear_bwd_x_kernel<<<dim3(ceil_div(N2, LB_T), ceil_div(Cin, LB_T), B), 256, 0, st>>>(s.dG2, w->W1, g.feat2, Cout, Kin, Cin,
                                                                                             Cin, N2);
    B200_LAUNCH_CHECK("linear_bwd_x_kernel");
    cudaError_t e = cudaSuccess;
    if (g.W1 || g.b1)
        e = launch_linear_bwd_w<DET>(s.dA1, feat1, g.W1, g.b1, DET || g.b1, Cout, Kin, 0, Cin, B, N1, st, d.lpart);
    if (e == cudaSuccess && g.W1)
        e = launch_linear_bwd_w<DET>(s.dG2, feat2, g.W1, nullptr, false, Cout, Kin, Cin, Cin, B, N2, st, d.lpart);
    if (e != cudaSuccess) return cuda_fail(e, "linear_bwd_w_kernel");
    return B200_OK;
}

}  // namespace b200

extern "C" int b200_corr3d_bwd(const float* xyz1, const float* feat1, const float* xyz2, const float* feat2,
                               const int64_t* knn12, const int64_t* knn11, const b200_corr3d_weights* w, const float* grad_out,
                               const float* fwd_scratch, const b200_corr3d_grads* grads, float* scratch, int B, int Cin,
                               int Cout, int N1, int N2, int k, b200_stream_t stream) {
    return b200::corr3d_bwd_run<false>("b200_corr3d_bwd", xyz1, feat1, xyz2, feat2, knn12, knn11, w, grad_out, fwd_scratch,
                                       grads, scratch, B, Cin, Cout, N1, N2, k, stream);
}

extern "C" int b200_corr3d_bwd_det(const float* xyz1, const float* feat1, const float* xyz2, const float* feat2,
                                   const int64_t* knn12, const int64_t* knn11, const b200_corr3d_weights* w,
                                   const float* grad_out, const float* fwd_scratch, const b200_corr3d_grads* grads,
                                   float* scratch, int B, int Cin, int Cout, int N1, int N2, int k, b200_stream_t stream) {
    return b200::corr3d_bwd_run<true>("b200_corr3d_bwd_det", xyz1, feat1, xyz2, feat2, knn12, knn11, w, grad_out, fwd_scratch,
                                      grads, scratch, B, Cin, Cout, N1, N2, k, stream);
}
