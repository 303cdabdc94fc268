// corr3d_common.cuh — pieces shared by the fp32 (corr3d.cu) and tensor-core (corr3d_tc.cu) paths of a5.
#pragma once
#include "common.cuh"

namespace b200 {

static inline int64_t align4(int64_t v) { return (v + 3) & ~int64_t(3); }

struct Corr3dScratch {
    float *A1, *G2, *P, *W2T, *W1cT, *n1WcT, *n2WcT;
    float *v2_W2img, *v2_wcimg;     // corr3d_v2.cu: W2 pre-split into its swizzled tile image; Wc / bias images of both weight nets
    float *v2_W1img;                // ... and the two C x C halves of W1
    int64_t total;
};
static inline Corr3dScratch carve(float* base, int B, int Cout, int N1, int N2) {
    Corr3dScratch s;
    int64_t off = 0;
    auto take = [&](int64_t n) { float* p = base ? base + off : nullptr; off += align4(n); return p; };
    s.A1 = take((int64_t)B * N1 * Cout);
    s.G2 = take((int64_t)B * N2 * Cout);
    s.P = take((int64_t)B * N1 * Cout);
    s.W2T = take((int64_t)Cout * Cout);
    s.W1cT = take(3ll * Cout);
    s.n1WcT = take(8ll * Cout);
    s.n2WcT = take(8ll * Cout);
    s.v2_W2img = take(2ll * Cout * Cout);
    s.v2_wcimg = take(2ll * Cout * 32);
    s.v2_W1img = take(4ll * Cout * Cout);
    s.total = off;
    return s;
}

// ---- the PointConv-style weight net: hidden 8-vector of relu(Wb.relu(Wa.d+ba)+bb) -------------------------------
__device__ __forceinline__ void weight_net_hidden(const float* __restrict__ Wa, const float* __restrict__ ba,
                                                  const float* __restrict__ Wb, const float* __restrict__ bb,
                                                  float dx, float dy, float dz, float* hid) {
    float h1[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) {
        float s = __ldg(ba + o);
        s = fmaf(__ldg(Wa + o * 3 + 0), dx, s);
        s = fmaf(__ldg(Wa + o * 3 + 1), dy, s);
        s = fmaf(__ldg(Wa + o * 3 + 2), dz, s);
        h1[o] = fmaxf(s, 0.0f);
    }
#pragma unroll
    for (int o = 0; o < 8; ++o) {
        float s = __ldg(bb + o);
#pragma unroll
        for (int i = 0; i < 8; ++i) s = fmaf(__ldg(Wb + o * 8 + i), h1[i], s);
        hid[o] = fmaxf(s, 0.0f);
    }
}

// The same net with its 104 parameters staged once per CTA in shared memory as [Wa 24 | ba 8 | Wb 64 | bb 8] (16-byte
// aligned): 26 broadcast LDS.128 per call instead of 104 uniform global loads.
constexpr int WN_FLOATS = 104;
__device__ __forceinline__ void weight_net_stage(float* s_wn, const float* __restrict__ Wa, const float* __restrict__ ba,
                                                 const float* __restrict__ Wb, const float* __restrict__ bb, int tid, int nthreads) {
    for (int e = tid; e < WN_FLOATS; e += nthreads)
        s_wn[e] = e < 24 ? __ldg(Wa + e) : e < 32 ? __ldg(ba + e - 24) : e < 96 ? __ldg(Wb + e - 32) : __ldg(bb + e - 96);
}
__device__ __forceinline__ void weight_net_hidden_s(const float* s_wn, float dx, float dy, float dz, float* hid) {
    const float4* w4 = reinterpret_cast<const float4*>(s_wn);
    float wa[24], h1[8];
#pragma unroll
    for (int i = 0; i < 6; ++i) { const float4 v = w4[i]; wa[4 * i] = v.x; wa[4 * i + 1] = v.y; wa[4 * i + 2] = v.z; wa[4 * i + 3] = v.w; }
    const float4 ba0 = w4[6], ba1 = w4[7];
    const float bav[8] = {ba0.x, ba0.y, ba0.z, ba0.w, ba1.x, ba1.y, ba1.z, ba1.w};
#pragma unroll
    for (int o = 0; o < 8; ++o) {                      // same operation order as weight_net_hidden
        float s = bav[o];
        s = fmaf(wa[o * 3 + 0], dx, s);
        s = fmaf(wa[o * 3 + 1], dy, s);
        s = fmaf(wa[o * 3 + 2], dz, s);
        h1[o] = fmaxf(s, 0.0f);
    }
    const float4 bb0 = w4[24], bb1 = w4[25];
    const float bbv[8] = {bb0.x, bb0.y, bb0.z, bb0.w, bb1.x, bb1.y, bb1.z, bb1.w};
#pragma unroll
    for (int o = 0; o < 8; ++o) {
        const float4 r0 = w4[8 + 2 * o], r1 = w4[9 + 2 * o];
        float s = bbv[o];
        s = fmaf(r0.x, h1[0], s); s = fmaf(r0.y, h1[1], s); s = fmaf(r0.z, h1[2], s); s = fmaf(r0.w, h1[3], s);
        s = fmaf(r1.x, h1[4], s); s = fmaf(r1.y, h1[5], s); s = fmaf(r1.z, h1[6], s); s = fmaf(r1.w, h1[7], s);
        hid[o] = fmaxf(s, 0.0f);
    }
}


// corr3d.cu: the weight transposes and the two pointwise linears (A1 with b1, G2) into s, fp32
cudaError_t corr3d_prep_and_linears(const float* feat1, const float* feat2, const b200_corr3d_weights* w, const Corr3dScratch& s,
                                    int B, int Cin, int Cout, int N1, int N2, cudaStream_t st);

// corr3d_tc.cu: pass 2 on tcgen05 tensor cores (precision 1 = TF32, 2 = 3xTF32); false -> caller uses the fp32 kernel
bool corr3d_stage1_tc_eligible(int Cout, int k, int precision);
cudaError_t corr3d_stage1_tc(const float* xyz1, const float* xyz2, const int64_t* knn12, const Corr3dScratch& s,
                             const b200_corr3d_weights* w, int B, int Cout, int N1, int N2, int k, int precision,
                             cudaStream_t st);

// corr3d_v2.cu: second-generation passes 2 + 3 (warp-specialised, every contraction on tcgen05); 3xTF32 only
bool corr3d_v2_eligible(int C, int k, int precision);
cudaError_t corr3d_v2_run(const float* xyz1, const float* feat1, const float* xyz2, const float* feat2, const int64_t* knn12,
                          const int64_t* knn11, const Corr3dScratch& s, const b200_corr3d_weights* w, float* out, int B, int C, int N1,
                          int N2, cudaStream_t st);

}  // namespace b200
