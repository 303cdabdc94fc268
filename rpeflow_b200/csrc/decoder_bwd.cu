// decoder_bwd.cu — backwards of the decoder's f2 / f3 / f4 and the projection gathers' a6 / a7 forwards in gather.cu:
//   f2 knn_interpolation (models/utils.py:140-156; backwarp_3d :159-169 is the same op on (xyz1+flow, -flow)),
//   f3 backwarp_2d with padding_mode='border' (:186-198),
//   f4 convex_upsample (:201-214),
//   a6 batch_indexing_channel_first / _last (:119-137 torch.gather, :101-116 advanced indexing),
//   a7 grid_sample_wrapper (:288-294, F.grid_sample bilinear, align_corners=True, zero padding).
//
// Nothing of the forward is saved beyond its inputs and indices: every kernel recomputes the taps, weights, softmax and
// gather indices with the forward's own fp32 operations (decoder_common.cuh), so the gradient belongs to exactly the
// output the forward produced.  All of them are HBM / L2-atomic bound; there is no tensor-core work here.
//
// f2, f3, a6 and a7 scatter into the gradient of the gathered tensor with float atomics (not bit-reproducible); their
// other gradients are reduced in a fixed order and written once.  f4 uses no atomics at all: a per-pixel pass writes the
// mask gradient and 18 per-tap partials, a second pass gathers the flow gradient from them in tap order.
#include "common.cuh"
#include "decoder_common.cuh"

namespace b200 {

constexpr int DB_PTS = 32;       // f2 / f3 / a6 cf / a7: queries (pixels, points, columns) per CTA on threadIdx.x
constexpr int DB_LANES = 8;      // f2 / f3 / a6 cf / a7: at most this many channel lanes per query on threadIdx.y

static int channel_lanes(int C) { return C < DB_LANES ? (C < 1 ? 1 : C) : DB_LANES; }

// f2 backward.  CTA = 32 queries x blockDim.y channel lanes; each lane recomputes its query's weights and walks the
// channels c = lane, lane + blockDim.y, ...:
//   d_feat[b,c,j_s] += wn_s g_c                                      (atomics)
//   a_s = sum_c g_c feat[b,c,j_s]                                    (lane partials, summed in lane order)
// then lane 0 of each query:  dw_s = (a_s - sum_t wn_t a_t) / W,  dr_s = -dw_s w_s^2 where r_s >= 1e-8 (clamp_min's
// backward; 0 below),  du_s = dr_s u_s / r_s,  d_xyz[:,j_s] += du_s (atomics),  d_q[:,q] = -sum_s du_s (one write).
__global__ void __launch_bounds__(DB_PTS * DB_LANES)
knn_interpolate_bwd_kernel(const float* __restrict__ in_xyz, const float* __restrict__ feat, const float* __restrict__ q_xyz,
                           const int64_t* __restrict__ idx, const float* __restrict__ grad_out, float* __restrict__ d_xyz,
                           float* __restrict__ d_feat, float* __restrict__ d_q, int C, int M, int Q, int k) {
    __shared__ float part[DB_LANES][KI_KMAX][DB_PTS];
    const int b = blockIdx.y;
    const int tx = threadIdx.x, lane = threadIdx.y, lanes = blockDim.y;
    const int q = blockIdx.x * DB_PTS + tx;
    const bool ok = q < Q;
    const bool want_xyz = d_xyz != nullptr || d_q != nullptr;          // uniform over the grid
    int j[KI_KMAX];
    float u[KI_KMAX][3], r[KI_KMAX], w[KI_KMAX], wn[KI_KMAX], a[KI_KMAX];
    float wsum = 0.0f;
    const float* xyz = in_xyz + (size_t)b * 3 * M;
#pragma unroll
    for (int s = 0; s < KI_KMAX; ++s) {
        a[s] = 0.0f;
        j[s] = 0;
        w[s] = wn[s] = r[s] = u[s][0] = u[s][1] = u[s][2] = 0.0f;
    }
    if (ok) {
        const float qx = __ldg(q_xyz + ((size_t)b * 3 + 0) * Q + q), qy = __ldg(q_xyz + ((size_t)b * 3 + 1) * Q + q),
                    qz = __ldg(q_xyz + ((size_t)b * 3 + 2) * Q + q);
#pragma unroll
        for (int s = 0; s < KI_KMAX; ++s) {
            if (s < k) {
                j[s] = knn_point(__ldg(idx + ((size_t)b * Q + q) * k + s), M);
                w[s] = idw_weight(xyz, M, j[s], qx, qy, qz, u[s], r[s]);
                wsum = __fadd_rn(wsum, w[s]);
            }
        }
#pragma unroll
        for (int s = 0; s < KI_KMAX; ++s)
            if (s < k) wn[s] = __fdiv_rn(w[s], wsum);
        const float* f = feat + (size_t)b * C * M;
        const float* g = grad_out + (size_t)b * C * Q + q;
        float* df = d_feat != nullptr ? d_feat + (size_t)b * C * M : nullptr;
        for (int c = lane; c < C; c += lanes) {
            const float gc = __ldg(g + (size_t)c * Q);
            if (df != nullptr) {
#pragma unroll
                for (int s = 0; s < KI_KMAX; ++s)
                    if (s < k) atomicAdd(df + (size_t)c * M + j[s], wn[s] * gc);
            }
            if (want_xyz) {
                const float* fc = f + (size_t)c * M;
#pragma unroll
                for (int s = 0; s < KI_KMAX; ++s)
                    if (s < k) a[s] += gc * __ldg(fc + j[s]);
            }
        }
    }
    if (!want_xyz) return;
#pragma unroll
    for (int s = 0; s < KI_KMAX; ++s) part[lane][s][tx] = a[s];
    __syncthreads();
    if (lane != 0 || !ok) return;
    float abar = 0.0f;
#pragma unroll
    for (int s = 0; s < KI_KMAX; ++s) {
        if (s < k) {
            float t = 0.0f;
            for (int l = 0; l < lanes; ++l) t += part[l][s][tx];
            a[s] = t;
            abar += wn[s] * t;
        }
    }
    float dq[3] = {0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int s = 0; s < KI_KMAX; ++s) {
        if (s < k && r[s] >= 1e-8f) {
            const float dw = (a[s] - abar) / wsum;
            const float scale = -dw * w[s] * w[s] / r[s];                  // dr / r
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                const float du = scale * u[s][d];
                if (d_xyz != nullptr) atomicAdd(d_xyz + ((size_t)b * 3 + d) * M + j[s], du);
                dq[d] -= du;
            }
        }
    }
    if (d_q != nullptr) {
#pragma unroll
        for (int d = 0; d < 3; ++d) d_q[((size_t)b * 3 + d) * Q + q] = dq[d];
    }
}

// f3 backward.  CTA = 32 pixels x blockDim.y channel lanes, the forward's taps (make_taps_border) per pixel:
//   dx[b,c,tap] += w_tap g_c for every in-image tap                  (atomics)
//   dflow[b,0,p] = mx sum_c g_c ((v01 - v00) wy0 + (v11 - v10) wy1),  dflow[b,1,p] = my sum_c g_c ((v10 - v00) wx0 +
//   (v11 - v01) wx1), out-of-image taps reading 0; lane partials summed in lane order and written once.  mx / my is
// ATen's clip_coordinates_set_grad: 0 where the un-clamped coordinate is <= 0 or >= size - 1 (a sample exactly on the
// border counts as clipped), 1 otherwise.  The normalise / un-normalise factors 2/(W-1) and (W-1)/2 cancel.
__global__ void __launch_bounds__(DB_PTS * DB_LANES)
backwarp2d_border_bwd_kernel(const float* __restrict__ x, const float* __restrict__ flow, const float* __restrict__ grad_out,
                             float* __restrict__ dx, float* __restrict__ dflow, int C, int H, int W) {
    __shared__ float part[2][DB_LANES][DB_PTS];
    const int b = blockIdx.y;
    const int tx = threadIdx.x, lane = threadIdx.y, lanes = blockDim.y;
    const int HW = H * W;
    const int p = blockIdx.x * DB_PTS + tx;
    const bool ok = p < HW;
    float sx = 0.0f, sy = 0.0f;
    bool mx = false, my = false;
    if (ok) {
        const float gx = __fadd_rn((float)(p % W), __ldg(flow + ((size_t)b * 2 + 0) * HW + p));    // mesh_grid + flow12
        const float gy = __fadd_rn((float)(p / W), __ldg(flow + ((size_t)b * 2 + 1) * HW + p));
        const BorderSample bs = border_sample(gx, gy, H, W);
        const Taps t = border_taps(bs, H, W);
        mx = bs.rx > 0.0f && bs.rx < (float)(W - 1);
        my = bs.ry > 0.0f && bs.ry < (float)(H - 1);
        const float* xb = x + (size_t)b * C * HW;
        const float* g = grad_out + (size_t)b * C * HW + p;
        float* dxb = dx != nullptr ? dx + (size_t)b * C * HW : nullptr;
        for (int c = lane; c < C; c += lanes) {
            const float gc = __ldg(g + (size_t)c * HW);
            if (dxb != nullptr) {
                float* d = dxb + (size_t)c * HW;
                atomicAdd(d + t.o00, t.w00 * gc);
                if (t.o01 >= 0) atomicAdd(d + t.o01, t.w01 * gc);
                if (t.o10 >= 0) atomicAdd(d + t.o10, t.w10 * gc);
                if (t.o11 >= 0) atomicAdd(d + t.o11, t.w11 * gc);
            }
            if (dflow != nullptr) {
                const float* plane = xb + (size_t)c * HW;
                const float v00 = __ldg(plane + t.o00);
                const float v01 = t.o01 >= 0 ? __ldg(plane + t.o01) : 0.0f;
                const float v10 = t.o10 >= 0 ? __ldg(plane + t.o10) : 0.0f;
                const float v11 = t.o11 >= 0 ? __ldg(plane + t.o11) : 0.0f;
                sx += gc * ((v01 - v00) * bs.wy0 + (v11 - v10) * bs.wy1);
                sy += gc * ((v10 - v00) * bs.wx0 + (v11 - v01) * bs.wx1);
            }
        }
    }
    if (dflow == nullptr) return;                                         // uniform over the grid
    part[0][lane][tx] = sx;
    part[1][lane][tx] = sy;
    __syncthreads();
    if (lane != 0 || !ok) return;
    float tx_sum = 0.0f, ty_sum = 0.0f;
    for (int l = 0; l < lanes; ++l) {
        tx_sum += part[0][l][tx];
        ty_sum += part[1][l][tx];
    }
    dflow[((size_t)b * 2 + 0) * HW + p] = mx ? tx_sum : 0.0f;
    dflow[((size_t)b * 2 + 1) * HW + p] = my ? ty_sum : 0.0f;
}

// a7 backward.  CTA = 32 points x blockDim.y channel lanes, the forward's taps (zero_sample / zero_taps) per point:
//   dfeat[b,c,tap] += w_tap g_c for every in-image tap                (atomics)
//   dxy[b,0,n] = sum_c g_c ((v01 - v00) wy0 + (v11 - v10) wy1),  dxy[b,1,n] = sum_c g_c ((v10 - v00) wx0 + (v11 - v01) wx1)
// with out-of-image taps reading 0 and nothing clipped (ATen's grid_sampler_2d backward with zero padding); lane
// partials summed in lane order and written once.  The normalise / un-normalise factors 2/(W-1) and (W-1)/2 cancel.
// A point with no tap inside the image (far outside it, or a huge / non-finite coordinate) skips the channel loop and
// gets dxy = 0.
__global__ void __launch_bounds__(DB_PTS * DB_LANES)
grid_sample_pts_bwd_kernel(const float* __restrict__ feat, const float* __restrict__ xy, const float* __restrict__ grad_out,
                           float* __restrict__ dfeat, float* __restrict__ dxy, int C, int H, int W, int N) {
    __shared__ float part[2][DB_LANES][DB_PTS];
    const int b = blockIdx.y;
    const int tx = threadIdx.x, lane = threadIdx.y, lanes = blockDim.y;
    const int n = blockIdx.x * DB_PTS + tx;
    const size_t plane = (size_t)H * W;
    float sx = 0.0f, sy = 0.0f;
    if (n < N) {
        const ZeroSample s = zero_sample(__ldg(xy + ((size_t)b * 2 + 0) * N + n), __ldg(xy + ((size_t)b * 2 + 1) * N + n), H, W);
        const Taps t = zero_taps(s, H, W);
        if (t.o00 >= 0 || t.o01 >= 0 || t.o10 >= 0 || t.o11 >= 0) {
            const float* fb = feat + (size_t)b * C * plane;
            const float* g = grad_out + (size_t)b * C * N + n;
            float* dfb = dfeat != nullptr ? dfeat + (size_t)b * C * plane : nullptr;
            for (int c = lane; c < C; c += lanes) {
                const float gc = __ldg(g + (size_t)c * N);
                if (dfb != nullptr) {
                    float* d = dfb + (size_t)c * plane;
                    if (t.o00 >= 0) atomicAdd(d + t.o00, t.w00 * gc);
                    if (t.o01 >= 0) atomicAdd(d + t.o01, t.w01 * gc);
                    if (t.o10 >= 0) atomicAdd(d + t.o10, t.w10 * gc);
                    if (t.o11 >= 0) atomicAdd(d + t.o11, t.w11 * gc);
                }
                if (dxy != nullptr) {
                    const float* f = fb + (size_t)c * plane;
                    const float v00 = t.o00 >= 0 ? __ldg(f + t.o00) : 0.0f;
                    const float v01 = t.o01 >= 0 ? __ldg(f + t.o01) : 0.0f;
                    const float v10 = t.o10 >= 0 ? __ldg(f + t.o10) : 0.0f;
                    const float v11 = t.o11 >= 0 ? __ldg(f + t.o11) : 0.0f;
                    sx += gc * ((v01 - v00) * s.wy0 + (v11 - v10) * s.wy1);
                    sy += gc * ((v10 - v00) * s.wx0 + (v11 - v01) * s.wx1);
                }
            }
        }
    }
    if (dxy == nullptr) return;                                           // uniform over the grid
    part[0][lane][tx] = sx;
    part[1][lane][tx] = sy;
    __syncthreads();
    if (lane != 0 || n >= N) return;
    float tx_sum = 0.0f, ty_sum = 0.0f;
    for (int l = 0; l < lanes; ++l) {
        tx_sum += part[0][l][tx];
        ty_sum += part[1][l][tx];
    }
    dxy[((size_t)b * 2 + 0) * N + n] = tx_sum;
    dxy[((size_t)b * 2 + 1) * N + n] = ty_sum;
}

// a6 channel-first backward: ddata[b,c,j(i)] += grad_out[b,c,i], j = the forward's wrap_index of idx[b,i].  CTA = 32
// output columns x blockDim.y channel lanes: the index is read once per column, grad_out rows are read coalesced.
__global__ void __launch_bounds__(DB_PTS * DB_LANES)
gather_cf_bwd_kernel(const float* __restrict__ grad_out, const int64_t* __restrict__ idx, float* __restrict__ ddata,
                     int C, int N, int64_t I) {
    const int b = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * DB_PTS + threadIdx.x;
    if (i >= I) return;
    const int64_t j = wrap_index(__ldg(idx + (size_t)b * I + i), N, nullptr);
    const float* g = grad_out + (size_t)b * C * I + i;
    float* d = ddata + (size_t)b * C * N + j;
    for (int c = threadIdx.y; c < C; c += blockDim.y) atomicAdd(d + (size_t)c * N, __ldg(g + (size_t)c * I));
}

// a6 channel-last backward: ddata[b,j(i),:] += grad_out[b,i,:].  One thread per 16-byte (VEC: one red.global.add.v4.f32)
// or 4-byte element of a grad_out row, as in the forward.
template <bool VEC>
__global__ void __launch_bounds__(256)
gather_cl_bwd_kernel(const float* __restrict__ grad_out, const int64_t* __restrict__ idx, float* __restrict__ ddata,
                     int C, int N, int64_t I) {
    const int b = blockIdx.y;
    const int per_row = VEC ? C / 4 : C;
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= I * per_row) return;
    const int64_t i = e / per_row;
    const int c = (int)(e - i * per_row);
    const int64_t j = wrap_index(__ldg(idx + (size_t)b * I + i), N, nullptr);
    if (VEC) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(grad_out + ((size_t)b * I + i) * C) + c);
        float* dst = ddata + ((size_t)b * N + j) * C + 4 * c;
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
    } else {
        atomicAdd(ddata + ((size_t)b * N + j) * C + c, __ldg(grad_out + ((size_t)b * I + i) * C + c));
    }
}

// f4 backward, pass 1: thread = low-res pixel (y, x), all s*s sub-pixels (i, j) in order.  With p_k the forward's softmax
// over the 9 taps, F_{k,c} = s * flow[c, y+ky-1, x+kx-1] (0 outside) and G_c = grad_out[c, ys+i, xs+j]:
//   dmask[(k*s+i)*s+j] = p_k (a_k - sum_t p_t a_t),  a_k = sum_c G_c F_{k,c}
//   P[(k*2+c)] = s * sum_{i,j} p_k G_c       (scratch [B,18,H*W]: per-tap partials of the flow gradient; NULL: skipped)
template <int S>
__global__ void __launch_bounds__(256)
convex_upsample_bwd_pass1_kernel(const float* __restrict__ flow, const float* __restrict__ mask,
                                 const float* __restrict__ grad_out, float* __restrict__ dmask, float* __restrict__ P,
                                 int H, int W) {
    const int b = blockIdx.y;
    const int HW = H * W;
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p >= HW) return;
    const int y = p / W, x = p - y * W;
    float f[2][9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const int yy = y + k / 3 - 1, xx = x + k % 3 - 1;
        const bool in = yy >= 0 && yy < H && xx >= 0 && xx < W;                    // F.unfold(padding=1): zeros outside
#pragma unroll
        for (int c = 0; c < 2; ++c)
            f[c][k] = in ? __fmul_rn(__ldg(flow + ((size_t)b * 2 + c) * HW + yy * W + xx), (float)S) : 0.0f;
    }
    const float* m = mask + (size_t)b * 9 * S * S * HW + p;
    float* dm = dmask != nullptr ? dmask + (size_t)b * 9 * S * S * HW + p : nullptr;
    const size_t OW = (size_t)W * S, OHW = (size_t)H * S * OW;
    float acc[2][9];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[0][k] = acc[1][k] = 0.0f;
#pragma unroll 1
    for (int i = 0; i < S; ++i) {
        float G[2][S];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const float* src = grad_out + ((size_t)b * 2 + c) * OHW + (size_t)(y * S + i) * OW + (size_t)x * S;
            if (S == 2) {
                const float2 v = __ldg(reinterpret_cast<const float2*>(src));     // 8-byte aligned: 16-byte base, even offset
                G[c][0] = v.x; G[c][1] = v.y;
            } else {
#pragma unroll
                for (int j = 0; j < S; j += 4) {
                    const float4 v = __ldg(reinterpret_cast<const float4*>(src + j));
                    G[c][j] = v.x; G[c][j + 1] = v.y; G[c][j + 2] = v.z; G[c][j + 3] = v.w;
                }
            }
        }
#pragma unroll
        for (int j = 0; j < S; ++j) {
            float v[9], mx = -3.402823466e38f;
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                v[k] = __ldg(m + (size_t)((k * S + i) * S + j) * HW);
                mx = fmaxf(mx, v[k]);
            }
            float sum = 0.0f;
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                v[k] = expf(v[k] - mx);                                              // the forward's softmax, op for op
                sum += v[k];
            }
            float a[9], abar = 0.0f;
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                v[k] = __fdiv_rn(v[k], sum);
                a[k] = G[0][j] * f[0][k] + G[1][j] * f[1][k];
                abar += v[k] * a[k];
                acc[0][k] += v[k] * G[0][j];
                acc[1][k] += v[k] * G[1][j];
            }
            if (dm != nullptr) {
#pragma unroll
                for (int k = 0; k < 9; ++k) dm[(size_t)((k * S + i) * S + j) * HW] = v[k] * (a[k] - abar);
            }
        }
    }
    if (P != nullptr) {
        float* pp = P + (size_t)b * 18 * HW + p;
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            pp[(size_t)(2 * k) * HW] = acc[0][k] * (float)S;
            pp[(size_t)(2 * k + 1) * HW] = acc[1][k] * (float)S;
        }
    }
}

// f4 backward, pass 2: dflow[c, y', x'] = sum_k P[(k*2+c), y'-ky+1, x'-kx+1] over the in-image neighbours, in k order.
__global__ void __launch_bounds__(256)
convex_upsample_bwd_pass2_kernel(const float* __restrict__ P, float* __restrict__ dflow, int H, int W) {
    const int b = blockIdx.y;
    const int HW = H * W;
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p >= HW) return;
    const int y = p / W, x = p - y * W;
    const float* pp = P + (size_t)b * 18 * HW;
    float d0 = 0.0f, d1 = 0.0f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const int yy = y - k / 3 + 1, xx = x - k % 3 + 1;
        if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
            d0 += __ldg(pp + (size_t)(2 * k) * HW + yy * W + xx);
            d1 += __ldg(pp + (size_t)(2 * k + 1) * HW + yy * W + xx);
        }
    }
    dflow[((size_t)b * 2 + 0) * HW + p] = d0;
    dflow[((size_t)b * 2 + 1) * HW + p] = d1;
}

static int zero_fill(float* p, size_t n, cudaStream_t st) {
    if (p != nullptr && n > 0) B200_CUDA(cudaMemsetAsync(p, 0, n * sizeof(float), st));
    return B200_OK;
}

}  // namespace b200

extern "C" int b200_knn_interpolate_bwd(const float* input_xyz, const float* input_feat, const float* query_xyz,
                                        const int64_t* knn_idx, const float* grad_out, float* d_input_xyz,
                                        float* d_input_feat, float* d_query_xyz, int B, int C, int M, int Q, int k,
                                        b200_stream_t stream) {
    using namespace b200;
    const bool empty = B == 0 || C == 0 || Q == 0;
    B200_REQUIRE(empty || (input_xyz && input_feat && query_xyz && knn_idx && grad_out),
                 "b200_knn_interpolate_bwd: null pointer");                // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 0 && M >= 1 && Q >= 0, "b200_knn_interpolate_bwd: bad sizes");
    B200_REQUIRE(k >= 1 && k <= KI_KMAX, "b200_knn_interpolate_bwd: k must be in [1,%d] (got %d)", KI_KMAX, k);
    B200_REQUIRE(B <= 65535, "b200_knn_interpolate_bwd: B exceeds the grid limit");
    cudaStream_t st = as_stream(stream);
    int rc;
    if ((rc = zero_fill(d_input_feat, (size_t)B * C * M, st)) != B200_OK) return rc;
    if ((rc = zero_fill(d_input_xyz, (size_t)B * 3 * M, st)) != B200_OK) return rc;
    if (empty || !(d_input_xyz || d_input_feat || d_query_xyz)) {
        // no channel (C = 0) or no query: the query gradient is zero, everything else was zero-filled above
        return zero_fill(d_query_xyz, (size_t)B * 3 * Q, st);
    }
    const dim3 grid(ceil_div(Q, DB_PTS), B), block(DB_PTS, channel_lanes(C));
    knn_interpolate_bwd_kernel<<<grid, block, 0, st>>>(input_xyz, input_feat, query_xyz, knn_idx, grad_out, d_input_xyz,
                                                       d_input_feat, d_query_xyz, C, M, Q, k);
    B200_LAUNCH_CHECK("b200_knn_interpolate_bwd");
    return B200_OK;
}

extern "C" int b200_backwarp2d_bwd(const float* x, const float* flow, const float* grad_out, float* dx, float* dflow,
                                   int B, int C, int H, int W, b200_stream_t stream) {
    using namespace b200;
    const bool empty = B == 0 || C == 0;
    B200_REQUIRE(empty || (x && flow && grad_out), "b200_backwarp2d_bwd: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 0 && H >= 1 && W >= 1, "b200_backwarp2d_bwd: bad sizes");
    B200_REQUIRE((int64_t)H * W < (1ll << 31) && B <= 65535, "b200_backwarp2d_bwd: plane or batch too large");
    cudaStream_t st = as_stream(stream);
    const int64_t HW = (int64_t)H * W;
    int rc;
    if ((rc = zero_fill(dx, (size_t)B * C * HW, st)) != B200_OK) return rc;
    if (empty || !(dx || dflow)) return zero_fill(dflow, (size_t)B * 2 * HW, st);     // C = 0: the flow gradient is zero
    const dim3 grid(ceil_div(HW, DB_PTS), B), block(DB_PTS, channel_lanes(C));
    backwarp2d_border_bwd_kernel<<<grid, block, 0, st>>>(x, flow, grad_out, dx, dflow, C, H, W);
    B200_LAUNCH_CHECK("b200_backwarp2d_bwd");
    return B200_OK;
}

extern "C" int64_t b200_convex_upsample_bwd_scratch_floats(int B, int H, int W, int scale) {
    if (B < 0 || H < 0 || W < 0 || scale < 0) return 0;
    return (int64_t)18 * B * H * W;                 // per low-res pixel: the 9 taps' partial flow gradients, 2 channels
}

extern "C" int b200_convex_upsample_bwd(const float* flow, const float* mask, const float* grad_out, float* dflow,
                                        float* dmask, float* scratch, int B, int H, int W, int scale, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0) || (flow && mask && grad_out), "b200_convex_upsample_bwd: null pointer");   // empty calls carry null pointers
    B200_REQUIRE((B == 0) || !dflow || scratch, "b200_convex_upsample_bwd: null pointer (scratch is needed for dflow)");
    B200_REQUIRE(B >= 0 && H >= 1 && W >= 1, "b200_convex_upsample_bwd: bad sizes");
    B200_REQUIRE(scale == 2 || scale == 4 || scale == 8, "b200_convex_upsample_bwd: scale_factor must be 2, 4 or 8 (got %d)", scale);
    B200_REQUIRE((int64_t)H * W * scale * scale < (1ll << 31) && B <= 65535, "b200_convex_upsample_bwd: plane or batch too large");
    B200_REQUIRE((reinterpret_cast<uintptr_t>(grad_out) & 15) == 0, "b200_convex_upsample_bwd: grad_out must be 16-byte aligned");
    if (B == 0 || !(dflow || dmask)) return B200_OK;
    const dim3 grid(ceil_div((int64_t)H * W, 256), B);
    float* P = dflow != nullptr ? scratch : nullptr;
    cudaStream_t st = as_stream(stream);
    if (scale == 2) convex_upsample_bwd_pass1_kernel<2><<<grid, 256, 0, st>>>(flow, mask, grad_out, dmask, P, H, W);
    else if (scale == 4) convex_upsample_bwd_pass1_kernel<4><<<grid, 256, 0, st>>>(flow, mask, grad_out, dmask, P, H, W);
    else convex_upsample_bwd_pass1_kernel<8><<<grid, 256, 0, st>>>(flow, mask, grad_out, dmask, P, H, W);
    B200_LAUNCH_CHECK("b200_convex_upsample_bwd(pass 1)");
    if (dflow != nullptr) {
        convex_upsample_bwd_pass2_kernel<<<grid, 256, 0, st>>>(P, dflow, H, W);
        B200_LAUNCH_CHECK("b200_convex_upsample_bwd(pass 2)");
    }
    return B200_OK;
}

extern "C" int b200_grid_sample_pts_bwd(const float* feat, const float* xy, const float* grad_out, float* dfeat, float* dxy,
                                        int B, int C, int H, int W, int N, b200_stream_t stream) {
    using namespace b200;
    const bool empty = B == 0 || C == 0 || N == 0;
    B200_REQUIRE(empty || (feat && xy && grad_out), "b200_grid_sample_pts_bwd: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 0 && H >= 1 && W >= 1 && N >= 0, "b200_grid_sample_pts_bwd: bad sizes");
    B200_REQUIRE((int64_t)H * W < (1ll << 31) && B <= 65535, "b200_grid_sample_pts_bwd: plane or batch too large");
    cudaStream_t st = as_stream(stream);
    int rc;
    if ((rc = zero_fill(dfeat, (size_t)B * C * H * W, st)) != B200_OK) return rc;
    if (empty || !(dfeat || dxy)) return zero_fill(dxy, (size_t)B * 2 * N, st);      // C = 0: the point gradient is zero
    const dim3 grid(ceil_div(N, DB_PTS), B), block(DB_PTS, channel_lanes(C));
    grid_sample_pts_bwd_kernel<<<grid, block, 0, st>>>(feat, xy, grad_out, dfeat, dxy, C, H, W, N);
    B200_LAUNCH_CHECK("b200_grid_sample_pts_bwd");
    return B200_OK;
}

extern "C" int b200_gather_cf_bwd(const float* grad_out, const int64_t* idx, float* ddata, int B, int C, int N, int64_t I,
                                  b200_stream_t stream) {
    using namespace b200;
    const bool empty = B == 0 || C == 0 || I == 0;
    B200_REQUIRE(B == 0 || C == 0 || (ddata && (I == 0 || (grad_out && idx))), "b200_gather_cf_bwd: null pointer");
    B200_REQUIRE(B >= 0 && C >= 0 && N >= 1 && I >= 0, "b200_gather_cf_bwd: bad sizes");
    B200_REQUIRE(B <= 65535 && I <= ((1ll << 31) - 1) * DB_PTS, "b200_gather_cf_bwd: batch or index count exceeds the grid limit");
    cudaStream_t st = as_stream(stream);
    int rc;
    if ((rc = zero_fill(ddata, (size_t)B * C * N, st)) != B200_OK) return rc;
    if (empty) return B200_OK;
    const dim3 grid(ceil_div(I, DB_PTS), B), block(DB_PTS, channel_lanes(C));
    gather_cf_bwd_kernel<<<grid, block, 0, st>>>(grad_out, idx, ddata, C, N, I);
    B200_LAUNCH_CHECK("b200_gather_cf_bwd");
    return B200_OK;
}

extern "C" int b200_gather_cl_bwd(const float* grad_out, const int64_t* idx, float* ddata, int B, int C, int N, int64_t I,
                                  b200_stream_t stream) {
    using namespace b200;
    const bool empty = B == 0 || C == 0 || I == 0;
    B200_REQUIRE(B == 0 || C == 0 || (ddata && (I == 0 || (grad_out && idx))), "b200_gather_cl_bwd: null pointer");
    B200_REQUIRE(B >= 0 && C >= 0 && N >= 1 && I >= 0, "b200_gather_cl_bwd: bad sizes");
    B200_REQUIRE(B <= 65535 && (C == 0 || I <= ((1ll << 31) - 1) * 256 / C),
                 "b200_gather_cl_bwd: batch or index count exceeds the grid limit");
    cudaStream_t st = as_stream(stream);
    int rc;
    if ((rc = zero_fill(ddata, (size_t)B * N * C, st)) != B200_OK) return rc;
    if (empty) return B200_OK;
    const bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(grad_out) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(ddata) & 15) == 0);
    const dim3 grid(ceil_div(I * (vec ? C / 4 : C), 256), B);
    if (vec) gather_cl_bwd_kernel<true><<<grid, 256, 0, st>>>(grad_out, idx, ddata, C, N, I);
    else     gather_cl_bwd_kernel<false><<<grid, 256, 0, st>>>(grad_out, idx, ddata, C, N, I);
    B200_LAUNCH_CHECK("b200_gather_cl_bwd");
    return B200_OK;
}
