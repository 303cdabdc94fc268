// corr3d.cu — a5: the pwc3d_core point cost volume (Correlation3D.forward), forward only.
//
// Replaces models/pwc3d_core.py:69-117, which materialises a [B,2C+3,N,k] concat and runs 2 + 3 + 3 1x1 convs,
// 4 strided torch.gathers and 2 mul+sum kernels over [B,C,N,k] tensors.
//
// Algebra used (SURVEY §8 a5): the first cost_mlp layer is linear before its LeakyReLU, so
//     W1 . [feat1_i ; feat2_j ; d_ij] + b1  =  (W1a.feat1_i + b1)  +  (W1b.feat2_j)  +  W1c.d_ij
// and the two big terms are per-POINT, not per-(point,neighbour): they are computed once (pass 1, a small dense
// GEMM each) into POINT-MAJOR scratch so that the per-neighbour gather of W1b.feat2_j is one contiguous row read
// with 128-bit loads.  That removes 16x of the layer-1 flops and all of the concat traffic.
//
//   pass 0  corr3d_prep_weights : W2^T, W1c^T, Wc^T(weight_net1/2) -> scratch (coalesced reads in the hot loops)
//   pass 1  pointwise_linear    : A1[b,i,:] = W1a.feat1[b,:,i] + b1 ; G2[b,j,:] = W1b.feat2[b,:,j]
//   pass 2  corr3d_stage1       : per point i, neighbours j in knn12: h1 = lrelu(A1_i + G2_j + W1c.d) (shared mem),
//                                 h2 = lrelu(W2.h1 + b2), w = weight_net2(d), P[b,i,:] = sum_j w*h2
//   pass 3  corr3d_stage2       : out[b,:,i] = sum_{j in knn11(i)} weight_net1(xyz1_j - xyz1_i) * P[b,j,:]
//
// precision 0 = fp32 FFMA throughout (this file).  Tensor-core variants of pass 2 live in corr3d_tc.cu.
#include "corr3d_common.cuh"

namespace b200 {

// ---- pass 0 --------------------------------------------------------------------------------------------------
__global__ void corr3d_prep_weights(const float* __restrict__ W1, const float* __restrict__ W2,
                                    const float* __restrict__ n1Wc, const float* __restrict__ n2Wc,
                                    float* __restrict__ W2T, float* __restrict__ W1cT, float* __restrict__ n1WcT,
                                    float* __restrict__ n2WcT, int Cin, int Cout) {
    const int Kin = 2 * Cin + 3;
    const int total = Cout * Cout + 3 * Cout + 16 * Cout;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        if (e < Cout * Cout) {
            const int c = e / Cout, o = e % Cout;                 // W2T[c][o] = W2[o][c]
            W2T[e] = __ldg(W2 + (size_t)o * Cout + c);
        } else if (e < Cout * Cout + 3 * Cout) {
            const int r = e - Cout * Cout, a = r / Cout, o = r % Cout;
            W1cT[r] = __ldg(W1 + (size_t)o * Kin + 2 * Cin + a);  // columns of the concatenated xyz offset
        } else {
            const int r = e - Cout * Cout - 3 * Cout;
            const int which = r / (8 * Cout), q = r % (8 * Cout), m = q / Cout, o = q % Cout;
            (which ? n2WcT : n1WcT)[q] = __ldg((which ? n2Wc : n1Wc) + (size_t)o * 8 + m);
        }
    }
}

// ---- pass 1: out[b,n,o] = bias[o] + sum_c W[o, coff + c] * X[b,c,n]      X channel-first, out point-major --------
constexpr int PL_TN = 64, PL_TO = 64, PL_TK = 16;

__global__ void __launch_bounds__(256)
pointwise_linear_kernel(const float* __restrict__ X, const float* __restrict__ Wm, const float* __restrict__ bias,
                        float* __restrict__ out, int Cin, int ldw, int coff, int Cout, int N) {
    __shared__ __align__(16) float Xs[PL_TK][PL_TN];
    __shared__ __align__(16) float Ws[PL_TK][PL_TO];
    const int b = blockIdx.z, n0 = blockIdx.x * PL_TN, o0 = blockIdx.y * PL_TO;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

    for (int k0 = 0; k0 < Cin; k0 += PL_TK) {
        __syncthreads();
        for (int e = threadIdx.x; e < PL_TK * PL_TN; e += 256) {
            const int kk = e / PL_TN, nn = e % PL_TN;
            const int c = k0 + kk, n = n0 + nn;
            Xs[kk][nn] = (c < Cin && n < N) ? __ldg(X + ((size_t)b * Cin + c) * N + n) : 0.0f;
        }
        for (int e = threadIdx.x; e < PL_TK * PL_TO; e += 256) {
            const int kk = e % PL_TK, oo = e / PL_TK;
            const int c = k0 + kk, o = o0 + oo;
            Ws[kk][oo] = (c < Cin && o < Cout) ? __ldg(Wm + (size_t)o * ldw + coff + c) : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < PL_TK; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&Xs[kk][ty * 4]);
            const float4 w = *reinterpret_cast<const float4*>(&Ws[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
        }
    }
    const int ob = o0 + tx * 4;
    float bv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) bv[j] = (bias && ob + j < Cout) ? __ldg(bias + ob + j) : 0.0f;
    const bool vec = (Cout & 3) == 0 && ob + 3 < Cout;               // rows of out are 16-byte aligned when Cout % 4 == 0
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty * 4 + i;
        if (n >= N) continue;
        float* o = out + ((size_t)b * N + n) * Cout + ob;
        if (vec) {
            *reinterpret_cast<float4*>(o) = make_float4(acc[i][0] + bv[0], acc[i][1] + bv[1], acc[i][2] + bv[2], acc[i][3] + bv[3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (ob + j < Cout) o[j] = acc[i][j] + bv[j];
        }
    }
}

// ---- pass 2 --------------------------------------------------------------------------------------------------
// CTA = TP points x k neighbours (TP*k <= 128 rows).  Dynamic smem: h1[rows][Cout+4] | hid[rows][8] | d[rows][4] | j[rows]
template <int KMAX>
__global__ void __launch_bounds__(256)
corr3d_stage1_kernel(const float* __restrict__ xyz1, const float* __restrict__ xyz2, const int64_t* __restrict__ knn12,
                     const float* __restrict__ A1, const float* __restrict__ G2, const float* __restrict__ W2T,
                     const float* __restrict__ W1cT, const float* __restrict__ b2, const float* __restrict__ Wa,
                     const float* __restrict__ ba, const float* __restrict__ Wb, const float* __restrict__ bb,
                     const float* __restrict__ WcT, const float* __restrict__ bc, float* __restrict__ P,
                     int Cout, int N1, int N2, int k, int TP) {
    extern __shared__ float4 smem_f4[];
    float* smem = reinterpret_cast<float*>(smem_f4);
    const int rows = TP * k, LD = ((Cout + 3) & ~3) + 4;
    float* h1 = smem;                               // [rows][LD]
    float* hid = h1 + (size_t)rows * LD;            // [rows][8]
    float* dl = hid + (size_t)rows * 8;             // [rows][4]
    int* jj = reinterpret_cast<int*>(dl + (size_t)rows * 4);

    const int b = blockIdx.y, i0 = blockIdx.x * TP;
    const int tid = threadIdx.x;

    // (a)+(b): neighbour index, offset, weight-net hidden vector per row
    for (int r = tid; r < rows; r += 256) {
        const int pt = r / k, i = min(i0 + pt, N1 - 1);
        int64_t j = __ldg(knn12 + ((size_t)b * N1 + i) * k + (r - pt * k));
        j = j < 0 ? 0 : (j >= N2 ? N2 - 1 : j);
        const float dx = __ldg(xyz2 + ((size_t)b * 3 + 0) * N2 + j) - __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + i);
        const float dy = __ldg(xyz2 + ((size_t)b * 3 + 1) * N2 + j) - __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + i);
        const float dz = __ldg(xyz2 + ((size_t)b * 3 + 2) * N2 + j) - __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + i);
        jj[r] = (int)j;
        dl[r * 4 + 0] = dx; dl[r * 4 + 1] = dy; dl[r * 4 + 2] = dz; dl[r * 4 + 3] = 0.0f;
        weight_net_hidden(Wa, ba, Wb, bb, dx, dy, dz, hid + r * 8);
    }
    __syncthreads();

    // (c): h1[r][c] = lrelu(A1[i][c] + G2[j][c] + W1c[c].d)
    if ((Cout & 3) == 0) {
        const int q4 = Cout >> 2;
        for (int e = tid; e < rows * q4; e += 256) {
            const int r = e / q4, c = (e - r * q4) * 4;
            const int i = min(i0 + r / k, N1 - 1);
            const float4 a = __ldg(reinterpret_cast<const float4*>(A1 + ((size_t)b * N1 + i) * Cout + c));
            const float4 g = __ldg(reinterpret_cast<const float4*>(G2 + ((size_t)b * N2 + jj[r]) * Cout + c));   // contiguous row gather
            const float4 wx = __ldg(reinterpret_cast<const float4*>(W1cT + c));
            const float4 wy = __ldg(reinterpret_cast<const float4*>(W1cT + Cout + c));
            const float4 wz = __ldg(reinterpret_cast<const float4*>(W1cT + 2 * Cout + c));
            const float dx = dl[r * 4 + 0], dy = dl[r * 4 + 1], dz = dl[r * 4 + 2];
            float4 v;
            v.x = leaky01(a.x + g.x + fmaf(wz.x, dz, fmaf(wy.x, dy, wx.x * dx)));
            v.y = leaky01(a.y + g.y + fmaf(wz.y, dz, fmaf(wy.y, dy, wx.y * dx)));
            v.z = leaky01(a.z + g.z + fmaf(wz.z, dz, fmaf(wy.z, dy, wx.z * dx)));
            v.w = leaky01(a.w + g.w + fmaf(wz.w, dz, fmaf(wy.w, dy, wx.w * dx)));
            *reinterpret_cast<float4*>(h1 + (size_t)r * LD + c) = v;
        }
    } else {
        for (int e = tid; e < rows * Cout; e += 256) {
            const int r = e / Cout, c = e - r * Cout;
            const int i = min(i0 + r / k, N1 - 1);
            const float v = __ldg(A1 + ((size_t)b * N1 + i) * Cout + c) + __ldg(G2 + ((size_t)b * N2 + jj[r]) * Cout + c) +
                            fmaf(__ldg(W1cT + 2 * Cout + c), dl[r * 4 + 2],
                                 fmaf(__ldg(W1cT + Cout + c), dl[r * 4 + 1], __ldg(W1cT + c) * dl[r * 4 + 0]));
            h1[(size_t)r * LD + c] = leaky01(v);
        }
    }
    __syncthreads();

    // (d): one (point, out-channel) per thread item: k accumulators, W2T read coalesced, h1 rows broadcast from smem
    for (int e = tid; e < TP * Cout; e += 256) {
        const int pt = e / Cout, o = e - pt * Cout;
        const int i = i0 + pt;
        float acc[KMAX];
        const float bias2 = __ldg(b2 + o);
#pragma unroll
        for (int s = 0; s < KMAX; ++s) acc[s] = bias2;
        const float* hrow = h1 + (size_t)pt * k * LD;
        int c = 0;
        for (; c + 3 < Cout; c += 4) {
            const float w0 = __ldg(W2T + (size_t)(c + 0) * Cout + o), w1 = __ldg(W2T + (size_t)(c + 1) * Cout + o);
            const float w2 = __ldg(W2T + (size_t)(c + 2) * Cout + o), w3 = __ldg(W2T + (size_t)(c + 3) * Cout + o);
#pragma unroll
            for (int s = 0; s < KMAX; ++s) {
                if (s < k) {
                    const float4 h = *reinterpret_cast<const float4*>(hrow + (size_t)s * LD + c);
                    acc[s] = fmaf(w3, h.w, fmaf(w2, h.z, fmaf(w1, h.y, fmaf(w0, h.x, acc[s]))));
                }
            }
        }
        for (; c < Cout; ++c) {
            const float w0 = __ldg(W2T + (size_t)c * Cout + o);
#pragma unroll
            for (int s = 0; s < KMAX; ++s)
                if (s < k) acc[s] = fmaf(w0, hrow[(size_t)s * LD + c], acc[s]);
        }
        float wc[8];
#pragma unroll
        for (int m = 0; m < 8; ++m) wc[m] = __ldg(WcT + (size_t)m * Cout + o);
        const float bco = __ldg(bc + o);
        float sum = 0.0f;
#pragma unroll
        for (int s = 0; s < KMAX; ++s) {
            if (s < k) {
                const float* hd = hid + (size_t)(pt * k + s) * 8;
                float w = bco;
#pragma unroll
                for (int m = 0; m < 8; ++m) w = fmaf(wc[m], hd[m], w);
                sum = fmaf(fmaxf(w, 0.0f), leaky01(acc[s]), sum);
            }
        }
        if (i < N1) P[((size_t)b * N1 + i) * Cout + o] = sum;
    }
}

// ---- pass 3 --------------------------------------------------------------------------------------------------
// CTA = 32 points.  Dynamic smem: hid[32*k][8] | j[32*k] | tile[Cout][33]
__global__ void __launch_bounds__(256)
corr3d_stage2_kernel(const float* __restrict__ xyz1, const int64_t* __restrict__ knn11, const float* __restrict__ P,
                     const float* __restrict__ Wa, const float* __restrict__ ba, const float* __restrict__ Wb,
                     const float* __restrict__ bb, const float* __restrict__ WcT, const float* __restrict__ bc,
                     float* __restrict__ out, int Cout, int N1, int k) {
    extern __shared__ float4 smem_f4[];
    float* smem = reinterpret_cast<float*>(smem_f4);
    const int rows = 32 * k;
    float* hid = smem;                                   // [rows][8]
    int* jj = reinterpret_cast<int*>(hid + (size_t)rows * 8);
    float* tile = reinterpret_cast<float*>(jj + rows);   // [Cout][33]
    __shared__ __align__(16) float s_wn[WN_FLOATS];
    const int b = blockIdx.y, i0 = blockIdx.x * 32, tid = threadIdx.x;
    weight_net_stage(s_wn, Wa, ba, Wb, bb, tid, 256);
    __syncthreads();

    for (int r = tid; r < rows; r += 256) {
        const int pt = r / k, i = min(i0 + pt, N1 - 1);
        int64_t j = __ldg(knn11 + ((size_t)b * N1 + i) * k + (r - pt * k));
        j = j < 0 ? 0 : (j >= N1 ? N1 - 1 : j);
        const float dx = __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + j) - __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + i);
        const float dy = __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + j) - __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + i);
        const float dz = __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + j) - __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + i);
        jj[r] = (int)j;
        weight_net_hidden_s(s_wn, dx, dy, dz, hid + r * 8);
    }
    __syncthreads();

    for (int e = tid; e < 32 * Cout; e += 256) {
        const int pt = e / Cout, o = e - pt * Cout;
        float wc[8];
#pragma unroll
        for (int m = 0; m < 8; ++m) wc[m] = __ldg(WcT + (size_t)m * Cout + o);
        const float bco = __ldg(bc + o);
        float sum = 0.0f;
#pragma unroll 4
        for (int s = 0; s < k; ++s) {
            const int r = pt * k + s;
            const float4 h0 = *reinterpret_cast<const float4*>(hid + (size_t)r * 8);          // warp-wide broadcast reads
            const float4 h1 = *reinterpret_cast<const float4*>(hid + (size_t)r * 8 + 4);
            float w = bco;
            w = fmaf(wc[0], h0.x, w); w = fmaf(wc[1], h0.y, w); w = fmaf(wc[2], h0.z, w); w = fmaf(wc[3], h0.w, w);
            w = fmaf(wc[4], h1.x, w); w = fmaf(wc[5], h1.y, w); w = fmaf(wc[6], h1.z, w); w = fmaf(wc[7], h1.w, w);
            sum = fmaf(fmaxf(w, 0.0f), __ldg(P + ((size_t)b * N1 + jj[r]) * Cout + o), sum);   // row gather, coalesced over o
        }
        tile[o * 33 + pt] = sum;
    }
    __syncthreads();
    for (int e = tid; e < 32 * Cout; e += 256) {         // channel-first output, 32 consecutive points per row
        const int o = e >> 5, pt = e & 31;
        if (i0 + pt < N1) out[((size_t)b * Cout + o) * N1 + i0 + pt] = tile[o * 33 + pt];
    }
}

template <int KMAX>
static cudaError_t launch_stage1(const float* xyz1, const float* xyz2, const int64_t* knn12, const Corr3dScratch& s,
                                 const b200_corr3d_weights* w, int B, int Cout, int N1, int N2, int k, cudaStream_t st) {
    int TP = 128 / k > 0 ? 128 / k : 1;
    auto smem_for = [&](int tp) {
        const size_t r = (size_t)tp * k;
        return (r * (((Cout + 3) & ~3) + 4) + r * 8 + r * 4 + r) * sizeof(float);
    };
    while (TP > 1 && smem_for(TP) > 200 * 1024) TP /= 2;      // wide layers (Cout > ~400): fewer points per CTA, not a launch error
    if (smem_for(TP) > 227 * 1024) return cudaErrorInvalidConfiguration;
    const size_t smem = smem_for(TP);
    auto kern = corr3d_stage1_kernel<KMAX>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<dim3(ceil_div(N1, TP), B), 256, smem, st>>>(xyz1, xyz2, knn12, s.A1, s.G2, s.W2T, s.W1cT, w->b2, w->n2_Wa, w->n2_ba,
                                                      w->n2_Wb, w->n2_bb, s.n2WcT, w->n2_bc, s.P, Cout, N1, N2, k, TP);
    return cudaGetLastError();
}

// passes 0 and 1 for the backward (corr3d_bwd.cu), which recomputes A1 / G2 into its own copy of the scratch layout
cudaError_t corr3d_prep_and_linears(const float* feat1, const float* feat2, const b200_corr3d_weights* w, const Corr3dScratch& s,
                                    int B, int Cin, int Cout, int N1, int N2, cudaStream_t st) {
    const int Kin = 2 * Cin + 3;
    corr3d_prep_weights<<<ceil_div(Cout * (Cout + 19), 256), 256, 0, st>>>(w->W1, w->W2, w->n1_Wc, w->n2_Wc, s.W2T, s.W1cT,
                                                                         s.n1WcT, s.n2WcT, Cin, Cout);
    pointwise_linear_kernel<<<dim3(ceil_div(N1, PL_TN), ceil_div(Cout, PL_TO), B), 256, 0, st>>>(feat1, w->W1, w->b1, s.A1, Cin,
                                                                                               Kin, 0, Cout, N1);
    pointwise_linear_kernel<<<dim3(ceil_div(N2, PL_TN), ceil_div(Cout, PL_TO), B), 256, 0, st>>>(feat2, w->W1, nullptr, s.G2, Cin,
                                                                                               Kin, Cin, Cout, N2);
    return cudaGetLastError();
}

}  // namespace b200

extern "C" int64_t b200_corr3d_scratch_floats(int B, int Cin, int Cout, int N1, int N2, int k) {
    (void)Cin; (void)k;
    return b200::carve(nullptr, B, Cout, N1, N2).total;
}

extern "C" int b200_corr3d_fwd(const float* xyz1, const float* feat1, const float* xyz2, const float* feat2,
                               const int64_t* knn12, const int64_t* knn11, const b200_corr3d_weights* w, float* out,
                               float* scratch, int B, int Cin, int Cout, int N1, int N2, int k, int precision,
                               b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0) || (xyz1 && feat1 && xyz2 && feat2 && knn12 && knn11 && w && out && scratch), "b200_corr3d_fwd: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && Cin >= 1 && Cout >= 1 && N1 >= 1 && N2 >= 1, "b200_corr3d_fwd: bad sizes");
    B200_REQUIRE(k >= 1 && k <= 32, "b200_corr3d_fwd: k must be in [1,32] (got %d)", k);
    B200_REQUIRE(Cout <= 512, "b200_corr3d_fwd: Cout=%d exceeds 512", Cout);
    B200_REQUIRE(B <= 65535, "b200_corr3d_fwd: B exceeds the grid limit");
    B200_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "b200_corr3d_fwd: scratch must be 16-byte aligned");
    B200_REQUIRE(w != nullptr, "b200_corr3d_fwd: null weight struct");
    B200_REQUIRE(w->W1 && w->b1 && w->W2 && w->b2 && w->n1_Wa && w->n1_ba && w->n1_Wb && w->n1_bb && w->n1_Wc && w->n1_bc &&
                 w->n2_Wa && w->n2_ba && w->n2_Wb && w->n2_bb && w->n2_Wc && w->n2_bc, "b200_corr3d_fwd: null weight pointer");
    B200_REQUIRE(precision >= 0 && precision <= 2, "b200_corr3d_fwd: precision must be 0 (fp32), 1 (TF32) or 2 (3xTF32), got %d",
                 precision);
    if (B == 0) return B200_OK;
    cudaStream_t st = as_stream(stream);
    const Corr3dScratch s = carve(scratch, B, Cout, N1, N2);
    const int Kin = 2 * Cin + 3;

    if (Cin == Cout && corr3d_v2_eligible(Cout, k, precision)) {
        // second generation (corr3d_v2.cu): all three passes on tcgen05; needs W1cT from the common prep kernel
        corr3d_prep_weights<<<ceil_div(Cout * (Cout + 19), 256), 256, 0, st>>>(w->W1, w->W2, w->n1_Wc, w->n2_Wc, s.W2T, s.W1cT,
                                                                             s.n1WcT, s.n2WcT, Cin, Cout);
        B200_LAUNCH_CHECK("corr3d_prep_weights");
        const cudaError_t e2 = corr3d_v2_run(xyz1, feat1, xyz2, feat2, knn12, knn11, s, w, out, B, Cout, N1, N2, st);
        if (e2 != cudaSuccess) return cuda_fail(e2, "corr3d_v2");
        return B200_OK;
    }

    corr3d_prep_weights<<<ceil_div(Cout * (Cout + 19), 256), 256, 0, st>>>(w->W1, w->W2, w->n1_Wc, w->n2_Wc, s.W2T, s.W1cT,
                                                                         s.n1WcT, s.n2WcT, Cin, Cout);
    B200_LAUNCH_CHECK("corr3d_prep_weights");
    pointwise_linear_kernel<<<dim3(ceil_div(N1, PL_TN), ceil_div(Cout, PL_TO), B), 256, 0, st>>>(feat1, w->W1, w->b1, s.A1, Cin,
                                                                                               Kin, 0, Cout, N1);
    pointwise_linear_kernel<<<dim3(ceil_div(N2, PL_TN), ceil_div(Cout, PL_TO), B), 256, 0, st>>>(feat2, w->W1, nullptr, s.G2, Cin,
                                                                                               Kin, Cin, Cout, N2);
    B200_LAUNCH_CHECK("pointwise_linear_kernel");

    cudaError_t e;
    if (precision != 0 && corr3d_stage1_tc_eligible(Cout, k, precision))
        e = corr3d_stage1_tc(xyz1, xyz2, knn12, s, w, B, Cout, N1, N2, k, precision, st);
    else if (k <= 4) e = launch_stage1<4>(xyz1, xyz2, knn12, s, w, B, Cout, N1, N2, k, st);
    else if (k <= 8) e = launch_stage1<8>(xyz1, xyz2, knn12, s, w, B, Cout, N1, N2, k, st);
    else if (k <= 16) e = launch_stage1<16>(xyz1, xyz2, knn12, s, w, B, Cout, N1, N2, k, st);
    else e = launch_stage1<32>(xyz1, xyz2, knn12, s, w, B, Cout, N1, N2, k, st);
    if (e != cudaSuccess) return cuda_fail(e, "corr3d_stage1_kernel");

    const size_t smem2 = ((size_t)32 * k * 8 + (size_t)32 * k + (size_t)Cout * 33) * sizeof(float);
    e = cudaFuncSetAttribute(corr3d_stage2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
    if (e != cudaSuccess) return cuda_fail(e, "corr3d_stage2_kernel(attr)");
    corr3d_stage2_kernel<<<dim3(ceil_div(N1, 32), B), 256, smem2, st>>>(xyz1, knn11, s.P, w->n1_Wa, w->n1_ba, w->n1_Wb, w->n1_bb,
                                                                      s.n1WcT, w->n1_bc, out, Cout, N1, k);
    B200_LAUNCH_CHECK("corr3d_stage2_kernel");
    return B200_OK;
}
