/*
 * oracle/spec.c — CPU restatement of the RPEFlow correlation / cost-volume hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under rpeflow_b200/ may import, link or call this file; it exists so
 * that tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs can check and
 * time the CUDA path against an independent scalar implementation.
 *
 * Parity status: PINNED — tests/test_oracle_golden.py checks every function here against fixtures under
 * tests/golden/ that were produced by importing the unmodified reference (torch CPU path) from
 * /root/reference with tests/golden/make_golden.py.
 *
 * Plain C99, fp32 arithmetic written so that the compiler cannot contract a*b+c into an FMA
 * (build with -ffp-contract=off).  OpenMP only parallelises loops whose iterations are independent, so
 * results do not depend on the thread count.
 *
 * Citations are file:line in the reference repo (danqu130/RPEFlow).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_API __attribute__((visibility("default")))

/* The squared distance of the stated exactness rule (SURVEY §8a): ((dx*dx + dy*dy) + dz*dz), every
 * operation rounded to fp32 separately.  Equals torch.sum((xyz - c) ** 2, -1) on CPU, i.e. the FPS fallback
 * models/csrc/wrapper.py:92, bit for bit. */
static inline float sqdist3(const float* a, const float* b) {
    volatile float dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
    volatile float xx = dx * dx, yy = dy * dy, zz = dz * dz;
    volatile float s = xx + yy;
    return s + zz;
}
static inline float sqdist2(const float* a, const float* b) {
    volatile float dx = a[0] - b[0], dy = a[1] - b[1];
    volatile float xx = dx * dx, yy = dy * dy;
    return xx + yy;
}
/* The arithmetic nvcc generates for the reference CUDA kernels (FMUL; FFMA; FFMA — SURVEY §2a),
 * k_nearest_neighbor_kernel.cu:33,77 and furthest_point_sampling_kernel.cu:63. Only used to study how
 * far the reference's own GPU rounding is from the stated rule. */
static inline float sqdist_fused(const float* a, const float* b, int D) {
    float dx = a[0] - b[0], dy = a[1] - b[1];
    float s = fmaf(dy, dy, dx * dx);
    if (D == 3) { float dz = a[2] - b[2]; s = fmaf(dz, dz, s); }
    return s;
}

/* ---------------------------------------------------------------------------------------------------
 * a3 furthest point sampling — models/csrc/wrapper.py:83-96 (semantics, init 1e10, start index 0,
 * torch.max -> first maximum) and furthest_point_sampling_kernel.cu:48-77 (same loop on the GPU).
 * xyz [B,N,3] -> idx [B,S] int64. */
ORC_API void orc_fps(const float* xyz, int64_t* idx, int B, int N, int S) {
#pragma omp parallel for schedule(dynamic, 1)
    for (int b = 0; b < B; ++b) {
        const float* p = xyz + (size_t)b * N * 3;
        float* dist = (float*)malloc(sizeof(float) * (size_t)N);
        for (int i = 0; i < N; ++i) dist[i] = 1e10f;
        int64_t cur = 0;
        for (int s = 0; s < S; ++s) {
            idx[(size_t)b * S + s] = cur;
            const float* c = p + cur * 3;
            float best = -1.0f; int64_t besti = 0;
            for (int i = 0; i < N; ++i) {
                float d = sqdist3(p + (size_t)i * 3, c);
                if (d < dist[i]) dist[i] = d;            /* wrapper.py:93-94 */
                if (dist[i] > best) { best = dist[i]; besti = i; }   /* strict > : lowest index wins */
            }
            cur = besti;
        }
        free(dist);
    }
}

/* ---------------------------------------------------------------------------------------------------
 * a4 k nearest neighbours — k_nearest_neighbor_kernel.cu:63-93 (direct distance, ascending insertion)
 * with the stated tie rule: order by (distance, index), both ascending.  fused!=0 switches to the
 * FMA-contracted distance of the reference's compiled kernel.
 * input [B,M,D], query [B,Q,D] -> idx [B,Q,k] int64 (zeros where M < k, k_nearest_neighbor.cpp:16). */
ORC_API void orc_knn(const float* input, const float* query, int64_t* idx,
                     int B, int M, int Q, int D, int k, int fused) {
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int q = 0; q < Q; ++q) {
            float nd[32]; int ni[32]; int cnt = 0;
            const float* qp = query + ((size_t)b * Q + q) * D;
            const float* ip = input + (size_t)b * M * D;
            for (int j = 0; j < M; ++j) {
                float d = fused ? sqdist_fused(qp, ip + (size_t)j * D, D)
                                : (D == 3 ? sqdist3(qp, ip + (size_t)j * 3) : sqdist2(qp, ip + (size_t)j * 2));
                if (cnt == k && !(d < nd[k - 1])) continue;   /* equal distance, later index: loses */
                if (d != d) continue;                          /* NaN never enters */
                int pos = cnt < k ? cnt : k - 1;
                while (pos > 0 && nd[pos - 1] > d) { nd[pos] = nd[pos - 1]; ni[pos] = ni[pos - 1]; --pos; }
                nd[pos] = d; ni[pos] = j;
                if (cnt < k) ++cnt;
            }
            int64_t* o = idx + ((size_t)b * Q + q) * k;
            for (int s = 0; s < k; ++s) o[s] = s < cnt ? ni[s] : 0;
        }
}

/* ---------------------------------------------------------------------------------------------------
 * a1 2-D correlation forward — correlation_forward_kernel.cu:11-49 (NHWC in, NCHW out, dy slow index,
 * out-of-image taps are 0 because correlation.cpp:17 allocates zeros). */
ORC_API void orc_corr2d_fwd(const float* in1, const float* in2, float* out,
                            int B, int C, int H, int W, int md) {
    const int D = 2 * md + 1;
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int y = 0; y < H; ++y)
            for (int x = 0; x < W; ++x) {
                const float* a = in1 + (((size_t)b * H + y) * W + x) * C;
                for (int dy = -md; dy <= md; ++dy)
                    for (int dx = -md; dx <= md; ++dx) {
                        int y2 = y + dy, x2 = x + dx;
                        float v = 0.0f;
                        if (y2 >= 0 && y2 < H && x2 >= 0 && x2 < W) {
                            const float* c2 = in2 + (((size_t)b * H + y2) * W + x2) * C;
                            float s = 0.0f;
                            for (int c = 0; c < C; ++c) s += a[c] * c2[c];
                            v = s / (float)C;                      /* correlation_forward_kernel.cu:46 */
                        }
                        int tc = (dy + md) * D + (dx + md);
                        out[(((size_t)b * D * D + tc) * H + y) * W + x] = v;
                    }
            }
}

/* a2 2-D correlation backward — correlation_backward_kernel.cu:4-74.  grads are NCHW. */
ORC_API void orc_corr2d_bwd(const float* gout, const float* in1, const float* in2,
                            float* gin1, float* gin2, int B, int C, int H, int W, int md) {
    const int D = 2 * md + 1;
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int y = 0; y < H; ++y)
            for (int x = 0; x < W; ++x)
                for (int c = 0; c < C; ++c) {
                    float s1 = 0.0f, s2 = 0.0f;
                    for (int dy = -md; dy <= md; ++dy)
                        for (int dx = -md; dx <= md; ++dx) {
                            int tc = (dy + md) * D + (dx + md);
                            int y2 = y + dy, x2 = x + dx;           /* grad wrt in1[y,x]: partner in2[y+dy,x+dx] */
                            if (y2 >= 0 && y2 < H && x2 >= 0 && x2 < W)
                                s1 += gout[(((size_t)b * D * D + tc) * H + y) * W + x] *
                                      in2[(((size_t)b * H + y2) * W + x2) * C + c];
                            int y1 = y - dy, x1 = x - dx;           /* grad wrt in2[y,x]: partner in1[y-dy,x-dx] */
                            if (y1 >= 0 && y1 < H && x1 >= 0 && x1 < W)
                                s2 += gout[(((size_t)b * D * D + tc) * H + y1) * W + x1] *
                                      in1[(((size_t)b * H + y1) * W + x1) * C + c];
                        }
                    gin1[(((size_t)b * C + c) * H + y) * W + x] = s1 / (float)C;
                    gin2[(((size_t)b * C + c) * H + y) * W + x] = s2 / (float)C;
                }
}

/* ---------------------------------------------------------------------------------------------------
 * a6 gathers — models/utils.py:119-137 and :101-116.  4-byte elements. */
ORC_API void orc_gather_cf(const uint32_t* data, const int64_t* idx, uint32_t* out,
                           int B, int C, int N, int64_t I) {
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int c = 0; c < C; ++c)
            for (int64_t i = 0; i < I; ++i) {
                int64_t j = idx[(size_t)b * I + i]; if (j < 0) j += N;
                out[((size_t)b * C + c) * I + i] = data[((size_t)b * C + c) * N + j];
            }
}
ORC_API void orc_gather_cl(const uint32_t* data, const int64_t* idx, uint32_t* out,
                           int B, int C, int N, int64_t I) {
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int64_t i = 0; i < I; ++i) {
            int64_t j = idx[(size_t)b * I + i]; if (j < 0) j += N;
            memcpy(out + ((size_t)b * I + i) * C, data + ((size_t)b * N + j) * C, sizeof(uint32_t) * (size_t)C);
        }
}

/* ---------------------------------------------------------------------------------------------------
 * f1 PointConv — models/pointconv.py:33-61 (PointConvDownSampling.forward) and :90-122 (PointConvNoSampling.forward,
 * which is the same computation with sampled_xyz = xyz): per sampled point p with neighbours j_k = knn[p][k]
 *   d_k  = xyz[:,j_k] - sampled[:,p]
 *   w_k  = lrelu(Wb . lrelu(Wa . d_k + ba) + bb)            weight_net = MLP2d(3,[8,16]), LeakyReLU(0.1) after both
 *   M    = sum_k w_k (16) x [xyz_jk ; feat_jk] (C+3)        flattened index = w*(C+3) + c   (pointconv.py:55-57)
 *   out  = lrelu(L . M + bias)                              nn.Linear(16*(C+3), out), norm = None, LeakyReLU(0.1) */
ORC_API void orc_pointconv_fwd(const float* xyz, const float* feat, const float* sampled, const int64_t* knn,
                               const float* Wa, const float* ba, const float* Wb, const float* bb,
                               const float* L, const float* bias, float* out,
                               int B, int C, int N, int S, int k, int Cout) {
    const int Cf = C + 3;
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int p = 0; p < S; ++p) {
            float* M = (float*)calloc((size_t)16 * Cf, sizeof(float));
            for (int s = 0; s < k; ++s) {
                const int64_t j = knn[((size_t)b * S + p) * k + s];
                float d[3], h1[8], w[16];
                for (int a = 0; a < 3; ++a) d[a] = xyz[((size_t)b * 3 + a) * N + j] - sampled[((size_t)b * 3 + a) * S + p];
                for (int o = 0; o < 8; ++o) {
                    float v = ba[o];
                    for (int a = 0; a < 3; ++a) v += Wa[o * 3 + a] * d[a];
                    h1[o] = v > 0.0f ? v : 0.1f * v;
                }
                for (int o = 0; o < 16; ++o) {
                    float v = bb[o];
                    for (int i = 0; i < 8; ++i) v += Wb[o * 8 + i] * h1[i];
                    w[o] = v > 0.0f ? v : 0.1f * v;
                }
                for (int o = 0; o < 16; ++o)
                    for (int c = 0; c < Cf; ++c) {
                        const float f = c < 3 ? xyz[((size_t)b * 3 + c) * N + j] : feat[((size_t)b * C + (c - 3)) * N + j];
                        M[o * Cf + c] += w[o] * f;
                    }
            }
            for (int o = 0; o < Cout; ++o) {
                float v = bias[o];
                for (int i = 0; i < 16 * Cf; ++i) v += L[(size_t)o * 16 * Cf + i] * M[i];
                out[((size_t)b * Cout + o) * S + p] = v > 0.0f ? v : 0.1f * v;
            }
            free(M);
        }
}

/* ---------------------------------------------------------------------------------------------------
 * f2 knn_interpolation — models/utils.py:140-156 (backwarp_3d :159-169 is this with xyz1+flow, -flow):
 * inverse-distance weights over the k nearest inputs, distance = ||x_j - q|| clamped at 1e-8, weights
 * normalised to sum 1, out[b,c,q] = sum_k w_k * feat[b,c,idx_k].  Indices are supplied by the caller. */
ORC_API void orc_knn_interpolate(const float* in_xyz, const float* feat, const float* q_xyz, const int64_t* idx,
                                 float* out, int B, int C, int M, int Q, int k) {
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int q = 0; q < Q; ++q) {
            float w[32], wsum = 0.0f;
            for (int s = 0; s < k; ++s) {
                const int64_t j = idx[((size_t)b * Q + q) * k + s];
                float d2 = 0.0f;
                for (int a = 0; a < 3; ++a) {
                    const float d = in_xyz[((size_t)b * 3 + a) * M + j] - q_xyz[((size_t)b * 3 + a) * Q + q];
                    d2 += d * d;
                }
                float d = sqrtf(d2);
                if (d < 1e-8f) d = 1e-8f;
                w[s] = 1.0f / d;
                wsum += w[s];
            }
            for (int c = 0; c < C; ++c) {
                float acc = 0.0f;
                for (int s = 0; s < k; ++s) {
                    const int64_t j = idx[((size_t)b * Q + q) * k + s];
                    acc += feat[((size_t)b * C + c) * M + j] * (w[s] / wsum);
                }
                out[((size_t)b * C + c) * Q + q] = acc;
            }
        }
}

/* ---------------------------------------------------------------------------------------------------
 * a7 grid_sample_wrapper — models/utils.py:288-294: normalise (2*x/(W-1) - 1), then F.grid_sample
 * bilinear, align_corners=True, zero padding, which un-normalises ((g+1)/2)*(W-1) and blends the four
 * in-bounds taps. */
static inline float bilinear_zero(const float* plane, int H, int W, float ix, float iy) {
    float fx = floorf(ix), fy = floorf(iy);
    int x0 = (int)fx, y0 = (int)fy, x1 = x0 + 1, y1 = y0 + 1;
    float wx1 = ix - fx, wy1 = iy - fy, wx0 = (fx + 1.0f) - ix, wy0 = (fy + 1.0f) - iy;
    float v = 0.0f;
    if (y0 >= 0 && y0 < H && x0 >= 0 && x0 < W) v += plane[(size_t)y0 * W + x0] * (wx0 * wy0);
    if (y0 >= 0 && y0 < H && x1 >= 0 && x1 < W) v += plane[(size_t)y0 * W + x1] * (wx1 * wy0);
    if (y1 >= 0 && y1 < H && x0 >= 0 && x0 < W) v += plane[(size_t)y1 * W + x0] * (wx0 * wy1);
    if (y1 >= 0 && y1 < H && x1 >= 0 && x1 < W) v += plane[(size_t)y1 * W + x1] * (wx1 * wy1);
    return v;
}
static inline float renorm_coord(float x, int size) {
    float g = 2.0f * x / (float)(size - 1) - 1.0f;          /* models/utils.py:290-291 */
    return ((g + 1.0f) / 2.0f) * (float)(size - 1);           /* grid_sample, align_corners=True */
}
ORC_API void orc_grid_sample_pts(const float* feat, const float* xy, float* out,
                                 int B, int C, int H, int W, int N) {
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int c = 0; c < C; ++c)
            for (int n = 0; n < N; ++n) {
                float ix = renorm_coord(xy[((size_t)b * 2 + 0) * N + n], W);
                float iy = renorm_coord(xy[((size_t)b * 2 + 1) * N + n], H);
                out[((size_t)b * C + c) * N + n] =
                    bilinear_zero(feat + ((size_t)b * C + c) * H * W, H, W, ix, iy);
            }
}

/* f3 backwarp_2d, padding_mode='border' — models/utils.py:186-198: grid = mesh_grid + flow, normalised as above,
 * then F.grid_sample(align_corners=True, padding_mode='border'): un-normalise, clamp to [0, size-1], blend the
 * in-bounds taps (a clamped x0 = W-1 leaves x1 = W out of bounds, weight 0). */
ORC_API void orc_backwarp2d_border(const float* x, const float* flow, float* out, int B, int C, int H, int W) {
    const size_t HW = (size_t)H * W;
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int c = 0; c < C; ++c)
            for (int py = 0; py < H; ++py)
                for (int px = 0; px < W; ++px) {
                    const size_t p = (size_t)py * W + px;
                    float gx = (float)px + flow[((size_t)b * 2 + 0) * HW + p];
                    float gy = (float)py + flow[((size_t)b * 2 + 1) * HW + p];
                    float ix = renorm_coord(gx, W), iy = renorm_coord(gy, H);
                    ix = fminf((float)(W - 1), fmaxf(ix, 0.0f));
                    iy = fminf((float)(H - 1), fmaxf(iy, 0.0f));
                    out[((size_t)b * C + c) * HW + p] = bilinear_zero(x + ((size_t)b * C + c) * HW, H, W, ix, iy);
                }
}

/* f4 convex_upsample — models/utils.py:201-214: softmax over the 9 taps, F.unfold(flow*s, 3x3, padding=1), weighted sum,
 * permute to [B,2,H*s,W*s].  mask channel = (k*s + i)*s + j. */
ORC_API void orc_convex_upsample(const float* flow, const float* mask, float* out, int B, int H, int W, int s) {
    const size_t HW = (size_t)H * W;
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int y = 0; y < H; ++y)
            for (int x = 0; x < W; ++x)
                for (int i = 0; i < s; ++i)
                    for (int j = 0; j < s; ++j) {
                        float v[9], mx = -INFINITY, sum = 0.0f;
                        for (int k = 0; k < 9; ++k) {
                            v[k] = mask[((size_t)b * 9 * s * s + (size_t)(k * s + i) * s + j) * HW + (size_t)y * W + x];
                            if (v[k] > mx) mx = v[k];
                        }
                        for (int k = 0; k < 9; ++k) { v[k] = expf(v[k] - mx); sum += v[k]; }
                        for (int c = 0; c < 2; ++c) {
                            float acc = 0.0f;
                            for (int k = 0; k < 9; ++k) {
                                int yy = y + k / 3 - 1, xx = x + k % 3 - 1;
                                float f = (yy >= 0 && yy < H && xx >= 0 && xx < W)
                                              ? flow[((size_t)b * 2 + c) * HW + (size_t)yy * W + xx] * (float)s : 0.0f;
                                acc += (v[k] / sum) * f;
                            }
                            out[(((size_t)b * 2 + c) * H * s + (size_t)y * s + i) * W * s + (size_t)x * s + j] = acc;
                        }
                    }
}

/* a8 project_feat_with_nn_corr — models/utils.py:297-317 with nn_indices given. */
ORC_API void orc_project_nn_corr(const float* xy, const float* feat2d, const float* feat3d,
                                 const int64_t* nn, float* out,
                                 int B, int C2, int C3, int H, int W, int N) {
    const size_t HW = (size_t)H * W;
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (size_t p = 0; p < HW; ++p) {
            int64_t j = nn[(size_t)b * HW + p];
            float px = (float)(p % W), py = (float)(p / W);     /* mesh_grid, models/utils.py:177-179 */
            float x = xy[((size_t)b * 2 + 0) * N + j], y = xy[((size_t)b * 2 + 1) * N + j];
            float* o = out + (size_t)b * (C3 + 3) * HW;
            o[0 * HW + p] = x - px;
            o[1 * HW + p] = y - py;
            float ix = renorm_coord(x, W), iy = renorm_coord(y, H);
            float s = 0.0f;
            for (int c = 0; c < C2; ++c) {
                const float* plane = feat2d + ((size_t)b * C2 + c) * HW;
                s += bilinear_zero(plane, H, W, ix, iy) * plane[p];
            }
            o[2 * HW + p] = s / (float)C2;
            for (int c = 0; c < C3; ++c) o[(3 + c) * HW + p] = feat3d[((size_t)b * C3 + c) * N + j];
        }
}

/* ---------------------------------------------------------------------------------------------------
 * a5 Correlation3D.forward — models/pwc3d_core.py:69-117, un-factorised, exactly in the reference's
 * order: concat [feat1, feat2[knn], dxyz] -> cost_mlp (2 x (1x1 conv + LeakyReLU 0.1)) ->
 * * weight_net2(dxyz) -> sum_k -> gather at self neighbours -> * weight_net1 -> sum_k. */
typedef struct {
    const float *W1, *b1, *W2, *b2;
    const float *n1_Wa, *n1_ba, *n1_Wb, *n1_bb, *n1_Wc, *n1_bc;
    const float *n2_Wa, *n2_ba, *n2_Wb, *n2_bb, *n2_Wc, *n2_bc;
} orc_corr3d_weights;

static void weight_net(const float* Wa, const float* ba, const float* Wb, const float* bb,
                       const float* Wc, const float* bc, const float* d, int Cout, float* w) {
    float h1[8], h2[8];
    for (int o = 0; o < 8; ++o) {
        float s = ba[o]; for (int i = 0; i < 3; ++i) s += Wa[o * 3 + i] * d[i];
        h1[o] = s > 0.0f ? s : 0.0f;
    }
    for (int o = 0; o < 8; ++o) {
        float s = bb[o]; for (int i = 0; i < 8; ++i) s += Wb[o * 8 + i] * h1[i];
        h2[o] = s > 0.0f ? s : 0.0f;
    }
    for (int o = 0; o < Cout; ++o) {
        float s = bc[o]; for (int i = 0; i < 8; ++i) s += Wc[o * 8 + i] * h2[i];
        w[o] = s > 0.0f ? s : 0.0f;                               /* ReLU after the last layer too */
    }
}

ORC_API void orc_corr3d_fwd(const float* xyz1, const float* feat1, const float* xyz2, const float* feat2,
                            const int64_t* knn12, const int64_t* knn11, const orc_corr3d_weights* wt,
                            float* out, int B, int Cin, int Cout, int N1, int N2, int k) {
    const int Kin = 2 * Cin + 3;
    float* p2n = (float*)malloc(sizeof(float) * (size_t)B * N1 * Cout);     /* [B,N1,Cout] */
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int i = 0; i < N1; ++i) {
            float* in = (float*)malloc(sizeof(float) * (size_t)(Kin + 3 * Cout));
            float *h1 = in + Kin, *h2 = h1 + Cout, *w = h2 + Cout;
            float* acc = p2n + ((size_t)b * N1 + i) * Cout;
            for (int o = 0; o < Cout; ++o) acc[o] = 0.0f;
            for (int c = 0; c < Cin; ++c) in[c] = feat1[((size_t)b * Cin + c) * N1 + i];
            for (int s = 0; s < k; ++s) {
                int64_t j = knn12[((size_t)b * N1 + i) * k + s];
                for (int c = 0; c < Cin; ++c) in[Cin + c] = feat2[((size_t)b * Cin + c) * N2 + j];
                float d[3];
                for (int a = 0; a < 3; ++a)
                    d[a] = xyz2[((size_t)b * 3 + a) * N2 + j] - xyz1[((size_t)b * 3 + a) * N1 + i];
                in[2 * Cin + 0] = d[0]; in[2 * Cin + 1] = d[1]; in[2 * Cin + 2] = d[2];
                for (int o = 0; o < Cout; ++o) {
                    float t = wt->b1[o]; const float* r = wt->W1 + (size_t)o * Kin;
                    for (int c = 0; c < Kin; ++c) t += r[c] * in[c];
                    h1[o] = t > 0.0f ? t : 0.1f * t;
                }
                for (int o = 0; o < Cout; ++o) {
                    float t = wt->b2[o]; const float* r = wt->W2 + (size_t)o * Cout;
                    for (int c = 0; c < Cout; ++c) t += r[c] * h1[c];
                    h2[o] = t > 0.0f ? t : 0.1f * t;
                }
                weight_net(wt->n2_Wa, wt->n2_ba, wt->n2_Wb, wt->n2_bb, wt->n2_Wc, wt->n2_bc, d, Cout, w);
                for (int o = 0; o < Cout; ++o) acc[o] += w[o] * h2[o];
            }
            free(in);
        }
#pragma omp parallel for collapse(2) schedule(static)
    for (int b = 0; b < B; ++b)
        for (int i = 0; i < N1; ++i) {
            float* w = (float*)malloc(sizeof(float) * (size_t)Cout * 2);
            float* acc = w + Cout;
            for (int o = 0; o < Cout; ++o) acc[o] = 0.0f;
            for (int s = 0; s < k; ++s) {
                int64_t j = knn11[((size_t)b * N1 + i) * k + s];
                float d[3];
                for (int a = 0; a < 3; ++a)
                    d[a] = xyz1[((size_t)b * 3 + a) * N1 + j] - xyz1[((size_t)b * 3 + a) * N1 + i];
                weight_net(wt->n1_Wa, wt->n1_ba, wt->n1_Wb, wt->n1_bb, wt->n1_Wc, wt->n1_bc, d, Cout, w);
                const float* src = p2n + ((size_t)b * N1 + j) * Cout;
                for (int o = 0; o < Cout; ++o) acc[o] += w[o] * src[o];
            }
            for (int o = 0; o < Cout; ++o) out[((size_t)b * Cout + o) * N1 + i] = acc[o];
            free(w);
        }
    free(p2n);
}

/* ---------------------------------------------------------------------------------------------------
 * a9 eventsToVoxel (integer pixels, temporal bilinear) — event_utils.py:23-39 (truncate x,y; normalise t by
 * (t_last - t_first + 1e-6) in fp32), :241-246 (t_norm, bin weight max(0, 1-|t_norm-b|)), :293-301
 * (polarity split, both weights +1), :207 (index_put_ accumulate in event order).  Serial on purpose: the
 * accumulation order per pixel is the event order, as in the reference on CPU.
 * Returns the number of events whose pixel falls outside [-W,W) x [-H,H) (IndexError in the reference). */
ORC_API int64_t orc_event_voxel_int(const float* ev, int64_t n, float* vox, int bins, int H, int W, int polarity) {
    const size_t HW = (size_t)H * W;
    memset(vox, 0, sizeof(float) * HW * (size_t)bins * (polarity ? 2 : 1));
    if (n <= 0) return 0;
    const float t_first = ev[2], t_last = ev[(size_t)(n - 1) * 4 + 2];
    volatile float dT = t_last - t_first;
    volatile float den = dT + 1e-6f;                                 /* NumPy>=2: python float is weak -> fp32 */
    volatile float ts0 = (t_first - t_first) / den;
    volatile float tsl = (t_last - t_first) / den;
    volatile float dt = tsl - ts0;                                    /* event_utils.py:241 */
    int64_t bad = 0;
    for (int64_t i = 0; i < n; ++i) {
        const float* e = ev + (size_t)i * 4;
        int x = (int)e[0], y = (int)e[1], p = (int)e[3];
        if (x < -W || x >= W || y < -H || y >= H) { ++bad; continue; }
        if (x < 0) x += W;
        if (y < 0) y += H;
        volatile float ts = (e[2] - t_first) / den;
        volatile float tn = (ts - ts0) / dt * (float)(bins - 1);      /* event_utils.py:242 */
        if (tn != tn) {                   /* zero-length window: tn = 0/0, clamp keeps NaN, NaN in every bin of every grid */
            for (int b = 0; b < bins * (polarity ? 2 : 1); ++b) vox[(size_t)b * HW + (size_t)y * W + x] += NAN;
            continue;
        }
        float wgt; size_t base;
        if (polarity) { wgt = 1.0f; base = p > 0 ? 0 : (size_t)bins * HW; }
        else          { wgt = (float)p; base = 0; }
        for (int b = 0; b < bins; ++b) {
            float bw = 1.0f - fabsf(tn - (float)b);
            if (bw > 0.0f) vox[base + (size_t)b * HW + (size_t)y * W + x] += wgt * bw;
        }
    }
    return bad;
}

/* a10 eventsToVoxelInter (float pixels, tri-linear) — dsec.py:570-604 and :536-568.  The eight corner
 * passes run in the reference's loop order so that per-voxel accumulation order matches it on CPU. */
static void trilinear_subset(const float* xs, const float* ys, const float* ts, const float* ps,
                             const int64_t* sel, int64_t m, int use_p, float* grid, int C, int H, int W) {
    if (m <= 0) return;
    const float t_a = ts[sel[0]], t_b = ts[sel[m - 1]];
    volatile float span = t_b - t_a;
    for (int cx = 0; cx < 2; ++cx)
        for (int cy = 0; cy < 2; ++cy)
            for (int ct = 0; ct < 2; ++ct)
                for (int64_t s = 0; s < m; ++s) {
                    int64_t i = sel[s];
                    volatile float num = (float)(C - 1) * (ts[i] - t_a);
                    volatile float tn = num / span;                          /* dsec.py:543 */
                    int xl = (int)xs[i] + cx, yl = (int)ys[i] + cy, tl = (int)tn + ct;
                    if (xl < 0 || xl >= W || yl < 0 || yl >= H || tl < 0 || tl >= C) continue;
                    float value = use_p ? 2.0f * ps[i] - 1.0f : 1.0f;        /* dsec.py:549, :597-598 */
                    volatile float w = value * (1.0f - fabsf((float)xl - xs[i]));
                    w = w * (1.0f - fabsf((float)yl - ys[i]));
                    w = w * (1.0f - fabsf((float)tl - tn));
                    grid[((size_t)tl * H + yl) * W + xl] += w;
                }
}
ORC_API int orc_event_voxel_trilinear(const float* x, const float* y, const int64_t* t, const float* p,
                                      int64_t n, float* vox, int bins, int H, int W, int polarity) {
    const size_t HW = (size_t)H * W;
    memset(vox, 0, sizeof(float) * HW * (size_t)bins * (polarity ? 2 : 1));
    if (n <= 0) return -1;
    float* ts = (float*)malloc(sizeof(float) * (size_t)n);
    int64_t* sel = (int64_t*)malloc(sizeof(int64_t) * (size_t)n);
    for (int64_t i = 0; i < n; ++i) ts[i] = (float)(t[i] - t[0]);              /* dsec.py:577 */
    const float last = ts[n - 1];
    for (int64_t i = 0; i < n; ++i) ts[i] = ts[i] / last;                      /* dsec.py:578 */
    if (!polarity) {
        for (int64_t i = 0; i < n; ++i) sel[i] = i;
        trilinear_subset(x, y, ts, p, sel, n, 1, vox, bins, H, W);
    } else {
        int64_t m = 0;
        for (int64_t i = 0; i < n; ++i) if (p[i] > 0.0f) sel[m++] = i;
        trilinear_subset(x, y, ts, p, sel, m, 1, vox, bins, H, W);
        m = 0;
        for (int64_t i = 0; i < n; ++i) if (!(p[i] > 0.0f)) sel[m++] = i;
        trilinear_subset(x, y, ts, p, sel, m, 0, vox + (size_t)bins * HW, bins, H, W);
    }
    free(ts); free(sel);
    return 0;
}
