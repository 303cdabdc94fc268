// gather.cu — a6/a7/a8: batched index gathers and the image<->point bilinear projection gathers.
//
// Replaces (all torch-op chains in the reference):
//   a6 models/utils.py:119-137 batch_indexing_channel_first  (torch.gather with an expanded [B,C,I] int64 index:
//      8 B of index traffic per 4 B moved) and :101-116 batch_indexing_channel_last;
//   a7 models/utils.py:288-294 grid_sample_wrapper           (normalise + F.grid_sample on NCHW);
//   a8 models/utils.py:297-317 project_feat_with_nn_corr     (grid_sample + 3 gathers + mul + mean + cat).
//
// All are HBM/L2-bandwidth bound.  Rules followed: index read ONCE per output column (not once per channel),
// consecutive threads on the contiguous output axis (full 128-B store lines), point-major scratch for rows that
// are later gathered so that gather reads are contiguous 128-bit loads, enough CTAs to fill 148 SMs by
// splitting the channel loop over blockIdx.y when the point axis alone is too short.
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "decoder_common.cuh"
#include "project_common.cuh"

namespace b200 {

// wrap_index: decoder_common.cuh
// out[b,c,i] = data[b,c,idx[b,i]]     grid: (ceil(I/256), csplit, B)
__global__ void __launch_bounds__(256)
gather_cf_kernel(const uint32_t* __restrict__ data, const int64_t* __restrict__ idx, uint32_t* __restrict__ out,
                 int C, int N, int64_t I, int* bad) {
    const int b = blockIdx.z;
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= I) return;
    const int64_t j = wrap_index(__ldg(idx + (size_t)b * I + i), N, blockIdx.y == 0 ? bad : nullptr);
    const uint32_t* src = data + (size_t)b * C * N + j;
    uint32_t* dst = out + (size_t)b * C * I + i;
    const int cstep = gridDim.y;
    int c = blockIdx.y;
    for (; c + 3 * cstep < C; c += 4 * cstep) {          // 4 independent loads in flight
        const uint32_t v0 = __ldg(src + (size_t)c * N), v1 = __ldg(src + (size_t)(c + cstep) * N);
        const uint32_t v2 = __ldg(src + (size_t)(c + 2 * cstep) * N), v3 = __ldg(src + (size_t)(c + 3 * cstep) * N);
        dst[(size_t)c * I] = v0; dst[(size_t)(c + cstep) * I] = v1;
        dst[(size_t)(c + 2 * cstep) * I] = v2; dst[(size_t)(c + 3 * cstep) * I] = v3;
    }
    for (; c < C; c += cstep) dst[(size_t)c * I] = __ldg(src + (size_t)c * N);
}

// out[b,i,:] = data[b,idx[b,i],:]     one thread per 16-byte (VEC) or 4-byte element of the output row
template <bool VEC>
__global__ void __launch_bounds__(256)
gather_cl_kernel(const uint32_t* __restrict__ data, const int64_t* __restrict__ idx, uint32_t* __restrict__ out,
                 int C, int N, int64_t I, int* bad) {
    const int b = blockIdx.y;
    const int per_row = VEC ? C / 4 : C;
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= I * per_row) return;
    const int64_t i = e / per_row;
    const int c = (int)(e - i * per_row);
    const int64_t j = wrap_index(__ldg(idx + (size_t)b * I + i), N, c == 0 ? bad : nullptr);
    if (VEC) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(data + ((size_t)b * N + j) * C) + c);
        reinterpret_cast<uint4*>(out + ((size_t)b * I + i) * C)[c] = v;
    } else {
        out[((size_t)b * I + i) * C + c] = __ldg(data + ((size_t)b * N + j) * C + c);
    }
}

// zero-padding taps: make_taps (decoder_common.cuh)
__device__ __forceinline__ float blend(const float* __restrict__ plane, const Taps& t) {
    // same accumulation order as ATen's grid_sampler_2d (nw, ne, sw, se), out-of-image taps skipped
    float v = 0.0f;
    if (t.o00 >= 0) v += __ldg(plane + t.o00) * t.w00;
    if (t.o01 >= 0) v += __ldg(plane + t.o01) * t.w01;
    if (t.o10 >= 0) v += __ldg(plane + t.o10) * t.w10;
    if (t.o11 >= 0) v += __ldg(plane + t.o11) * t.w11;
    return v;
}

// Two lanes per point: lane `side` owns the left (side 0) or right (side 1) tap of both rows, so the two horizontally
// adjacent taps of a row are requested by neighbouring lanes of ONE load instruction and share a 32-byte sector
// request (7 times out of 8) — with a thread per point every 4-byte tap pulls its own sector and these gathers are
// bound by L2 sector bandwidth (8x over-fetch), not by HBM.
struct HalfTaps {
    int o0, o1;          // this side's offsets in row y0 / y1 (-1: outside the image)
    float w0, w1;
};
__device__ __forceinline__ HalfTaps half_taps(const Taps& t, int side) {
    HalfTaps h;
    h.o0 = side ? t.o01 : t.o00; h.w0 = side ? t.w01 : t.w00;
    h.o1 = side ? t.o11 : t.o10; h.w1 = side ? t.w11 : t.w10;
    return h;
}
__device__ __forceinline__ float half_blend(const float* __restrict__ plane, const HalfTaps& h) {
    float v = 0.0f;
    if (h.o0 >= 0) v += __ldg(plane + h.o0) * h.w0;
    if (h.o1 >= 0) v += __ldg(plane + h.o1) * h.w1;
    return v;
}

// a7: out[b,c,n] = bilinear(feat[b,c], xy[b,:,n])       grid: (ceil(N/128), csplit, B); a warp covers 16 points
__global__ void __launch_bounds__(256)
grid_sample_pts_kernel(const float* __restrict__ feat, const float* __restrict__ xy, float* __restrict__ out,
                       int C, int H, int W, int N) {
    const int b = blockIdx.z;
    const int side = threadIdx.x & 1;
    const int n = blockIdx.x * 128 + (threadIdx.x >> 1);
    const bool ok = n < N;
    Taps t = {-1, -1, -1, -1, 0.0f, 0.0f, 0.0f, 0.0f};
    if (ok) t = make_taps(__ldg(xy + ((size_t)b * 2 + 0) * N + n), __ldg(xy + ((size_t)b * 2 + 1) * N + n), H, W);
    const HalfTaps h = half_taps(t, side);
    const size_t plane = (size_t)H * W;
    const float* f = feat + (size_t)b * C * plane;
    float* o = out + (size_t)b * C * N + n;
    // two channels per step: both lanes of a point accumulate both channels, lane `side` stores channel c + side
    int c = blockIdx.y * 2;
    for (; c + 1 < C; c += gridDim.y * 2) {
        float v0 = half_blend(f + (size_t)c * plane, h), v1 = half_blend(f + (size_t)(c + 1) * plane, h);
        v0 += __shfl_xor_sync(FULL, v0, 1);
        v1 += __shfl_xor_sync(FULL, v1, 1);
        if (ok) o[(size_t)(c + side) * N] = side ? v1 : v0;
    }
    if (c < C) {                                         // odd channel count: the last channel of this CTA's slice
        float v0 = half_blend(f + (size_t)c * plane, h);
        v0 += __shfl_xor_sync(FULL, v0, 1);
        if (ok && side == 0) o[(size_t)c * N] = v0;
    }
}

// f3: backwarp_2d with padding_mode='border' (taps: make_taps_border in decoder_common.cuh).
// grid: (ceil(HW/128), csplit, B); two lanes per pixel as in grid_sample_pts_kernel
__global__ void __launch_bounds__(256)
backwarp2d_border_kernel(const float* __restrict__ x, const float* __restrict__ flow, float* __restrict__ out,
                         int C, int H, int W) {
    const int b = blockIdx.z;
    const int side = threadIdx.x & 1;
    const int HW = H * W;
    const int p = blockIdx.x * 128 + (threadIdx.x >> 1);
    const bool ok = p < HW;
    Taps t = {-1, -1, -1, -1, 0.0f, 0.0f, 0.0f, 0.0f};
    if (ok) {
        const float gx = __fadd_rn((float)(p % W), __ldg(flow + ((size_t)b * 2 + 0) * HW + p));    // mesh_grid + flow12
        const float gy = __fadd_rn((float)(p / W), __ldg(flow + ((size_t)b * 2 + 1) * HW + p));
        t = make_taps_border(gx, gy, H, W);
    }
    const HalfTaps h = half_taps(t, side);
    const float* f = x + (size_t)b * C * HW;
    float* o = out + (size_t)b * C * HW + p;
    int c = blockIdx.y * 2;
    for (; c + 1 < C; c += gridDim.y * 2) {
        float v0 = half_blend(f + (size_t)c * HW, h), v1 = half_blend(f + (size_t)(c + 1) * HW, h);
        v0 += __shfl_xor_sync(FULL, v0, 1);
        v1 += __shfl_xor_sync(FULL, v1, 1);
        if (ok) o[(size_t)(c + side) * HW] = side ? v1 : v0;
    }
    if (c < C) {
        float v0 = half_blend(f + (size_t)c * HW, h);
        v0 += __shfl_xor_sync(FULL, v0, 1);
        if (ok && side == 0) o[(size_t)c * HW] = v0;
    }
}

// f4: convex_upsample (models/utils.py:201-214; caller RPEFlow_core.py:424, scale 4): RAFT's learned upsampling.
//   out[b,c,y*s+i,x*s+j] = sum_k softmax_k(mask[b,(k*s+i)*s+j,y,x]) * (s * flow[b,c,y+ky-1,x+kx-1]),  k = ky*3+kx, zero padding.
// Thread = (low-res pixel, sub-row i): reads its 9*s mask values plane by plane (coalesced over x), the 3x3 flow
// patch once, and writes the s output pixels of its sub-row for both flow channels as contiguous runs
// (16 bytes per thread for s = 4, adjacent threads adjacent in memory).  HBM-bound: the mask is 9*s*s planes.
template <int S>
__global__ void __launch_bounds__(256)
convex_upsample_kernel(const float* __restrict__ flow, const float* __restrict__ mask, float* __restrict__ out, int H, int W) {
    const int b = blockIdx.z, i = blockIdx.y;
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
    float o[2][S];
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
            v[k] = expf(v[k] - mx);                                                  // torch.softmax: exp(x - max) / sum
            sum += v[k];
        }
        float a0 = 0.0f, a1 = 0.0f;
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            const float w = __fdiv_rn(v[k], sum);
            a0 += w * f[0][k];
            a1 += w * f[1][k];
        }
        o[0][j] = a0; o[1][j] = a1;
    }
    const size_t OW = (size_t)W * S, OHW = (size_t)H * S * OW;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        float* dst = out + ((size_t)b * 2 + c) * OHW + (size_t)(y * S + i) * OW + (size_t)x * S;
        if (S % 4 == 0) {
#pragma unroll
            for (int j = 0; j < S; j += 4) __stcs(reinterpret_cast<float4*>(dst + j), make_float4(o[c][j], o[c][j + 1], o[c][j + 2], o[c][j + 3]));
        } else {
#pragma unroll
            for (int j = 0; j < S; ++j) dst[j] = o[c][j];
        }
    }
}

// a8, pass 1: one point-major row per point, R[b,n,:] = [ S (C2p floats) | T (C3p floats) ] with
//   S[c] = bilinear(feat2d[b,c], xy[b,:,n])   and   T[k] = feat3d[b,k,n]   (C2p, C3p = C2, C3 rounded up to 4),
// so that pass 2 gathers both with 128-bit loads from ONE contiguous row per pixel (channel-first feat3d costs a
// 32-byte sector per 4-byte element there: ncu showed that gather to be the largest consumer of L1 sector slots).
// Block = 16 points; compute: a warp owns 4 of every 32 channels, lanes = 16 points x 2 tap sides (see half_taps);
// write: lane = channel (contiguous in R).
// cf (optional): the same samples channel-first [B,C2,N] — exactly what grid_sample_wrapper(feat2d, xy) returns
// (same taps, same arithmetic as grid_sample_pts_kernel), written as 64-byte runs from the compute lanes.  The model asks
// for that tensor right after this call in four of its five fuser pairs per level (RPEFlow_core.py:31+53, :80+107,
// :134+157), so sampling once here saves a second pass over the whole feature map.

__global__ void __launch_bounds__(256)
sample_point_major_kernel(const float* __restrict__ feat, const float* __restrict__ xy, const float* __restrict__ feat3d,
                          float* __restrict__ R, float* __restrict__ cf, int C, int C3, int H, int W, int N) {
    __shared__ float tile[32][17];
    const int b = blockIdx.y;
    const int n0 = blockIdx.x * 16;
    const int lane = threadIdx.x & 31, tc = threadIdx.x >> 5;
    const int side = lane & 1, tp = lane >> 1;
    const int n = n0 + tp;
    const bool ok = n < N;
    const int stride = round4(C) + round4(C3);
    Taps t = {-1, -1, -1, -1, 0.0f, 0.0f, 0.0f, 0.0f};
    if (ok) t = make_taps(__ldg(xy + ((size_t)b * 2 + 0) * N + n), __ldg(xy + ((size_t)b * 2 + 1) * N + n), H, W);
    const HalfTaps h = half_taps(t, side);
    const size_t plane = (size_t)H * W;
    const float* f = feat + (size_t)b * C * plane;
    for (int c0 = 0; c0 < C; c0 += 32) {
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = c0 + tc * 4 + u;
            float v = c < C ? half_blend(f + (size_t)c * plane, h) : 0.0f;
            v += __shfl_xor_sync(FULL, v, 1);
            if (side == 0) {
                tile[tc * 4 + u][tp] = v;
                if (cf != nullptr && ok && c < C) cf[((size_t)b * C + c) * N + n] = v;
            }
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int p = tc * 2 + u, c = c0 + lane;
            if (n0 + p < N && c < C) R[((size_t)b * N + n0 + p) * stride + c] = tile[lane][p];
        }
    }
    // T: feat3d[b, k, n0..n0+15] -> R[b, n, C2p + k].  Read: a half-warp = 16 consecutive points of one channel (64 bytes).
    const int pt = lane & 15, ksub = lane >> 4;
    const float* g = feat3d + (size_t)b * C3 * N;
    float* Rt = R + round4(C);
    for (int k0 = 0; k0 < C3; k0 += 32) {
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int kk = tc * 4 + u * 2 + ksub, k = k0 + kk;
            tile[kk][pt] = (k < C3 && n0 + pt < N) ? __ldg(g + (size_t)k * N + n0 + pt) : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int p = tc * 2 + u, k = k0 + lane;
            if (n0 + p < N && k < C3) Rt[((size_t)b * N + n0 + p) * stride + k] = tile[lane][p];
        }
    }
}

// a8, pass 2: one thread per pixel.  blockIdx.z = 0: pixel offsets + channel-mean correlation; blockIdx.z >= 1: copies
// a slab of 32 feat3d channels of the nearest point (128-bit loads from the point's row of R, coalesced streaming stores).
// Batch items are visited last-to-first: pass 1 has just streamed feat2d through L2 in ascending order, so the tail of
// the batch is still resident when this kernel starts.

__global__ void __launch_bounds__(256)
project_nn_corr_kernel(const float* __restrict__ xy, const float* __restrict__ feat2d, const int64_t* __restrict__ nn,
                       const float* __restrict__ R, float* __restrict__ out, int C2, int C3, int H, int W, int N) {
    const int role = blockIdx.z;
    const int b = gridDim.y - 1 - blockIdx.y;
    const int HW = H * W;
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p >= HW) return;
    int64_t j = __ldg(nn + (size_t)b * HW + p);
    if (j < 0) j += N;
    j = j < 0 ? 0 : (j >= N ? N - 1 : j);
    float* o = out + (size_t)b * (C3 + 3) * HW + p;
    const int C2p = round4(C2), stride = C2p + round4(C3);
    const float* row = R + ((size_t)b * N + j) * stride;                // 16-byte aligned: stride % 4 == 0

    if (role == 0) {
        const float px = (float)(p % W), py = (float)(p / W);          // mesh_grid: x in channel 0 (models/utils.py:177-179)
        o[0] = __ldg(xy + ((size_t)b * 2 + 0) * N + j) - px;
        o[(size_t)HW] = __ldg(xy + ((size_t)b * 2 + 1) * N + j) - py;
        const float* f = feat2d + (size_t)b * C2 * HW + p;
        float acc = 0.0f;
        int c = 0;
        for (; c + 8 <= C2; c += 8) {                                   // 8 plane reads in flight per thread
            const float4 s0 = __ldg(reinterpret_cast<const float4*>(row + c));
            const float4 s1 = __ldg(reinterpret_cast<const float4*>(row + c + 4));
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = __ldg(f + (size_t)(c + u) * HW);
            acc += s0.x * v[0]; acc += s0.y * v[1]; acc += s0.z * v[2]; acc += s0.w * v[3];
            acc += s1.x * v[4]; acc += s1.y * v[5]; acc += s1.z * v[6]; acc += s1.w * v[7];
        }
        for (; c < C2; ++c) acc += __ldg(row + c) * __ldg(f + (size_t)c * HW);
        o[(size_t)2 * HW] = __fdiv_rn(acc, (float)C2);                  // torch.mean over channels
        return;
    }
    const int k0 = (role - 1) * PN_SLAB, k1 = min(k0 + PN_SLAB, C3);
    project_slab_copy(row + C2p, o, HW, k0, k1);
}

// f2: knn_interpolation (models/utils.py:140-156): out[b,c,q] = sum_s wn_s * feat[b,c,idx[b,q,s]], wn = normalised inverse
// distances (clamped at 1e-8).  Thread per query (weights computed once), channels split over blockIdx.y.  Every
// operation is rounded separately in the reference's order, so the result equals the oracle bit for bit.
__global__ void __launch_bounds__(256)
knn_interpolate_kernel(const float* __restrict__ in_xyz, const float* __restrict__ feat, const float* __restrict__ q_xyz,
                       const int64_t* __restrict__ idx, float* __restrict__ out, int C, int M, int Q, int k) {
    const int b = blockIdx.z;
    const int q = blockIdx.x * 256 + threadIdx.x;
    if (q >= Q) return;
    int j[KI_KMAX];
    float w[KI_KMAX];
    float wsum = 0.0f;
    const float qx = __ldg(q_xyz + ((size_t)b * 3 + 0) * Q + q), qy = __ldg(q_xyz + ((size_t)b * 3 + 1) * Q + q),
                qz = __ldg(q_xyz + ((size_t)b * 3 + 2) * Q + q);
    const float* xyz = in_xyz + (size_t)b * 3 * M;
#pragma unroll
    for (int s = 0; s < KI_KMAX; ++s) {
        if (s < k) {
            j[s] = knn_point(__ldg(idx + ((size_t)b * Q + q) * k + s), M);
            float u[3], r;
            w[s] = idw_weight(xyz, M, j[s], qx, qy, qz, u, r);
            wsum = __fadd_rn(wsum, w[s]);
        }
    }
#pragma unroll
    for (int s = 0; s < KI_KMAX; ++s)
        if (s < k) w[s] = __fdiv_rn(w[s], wsum);
    const float* f = feat + (size_t)b * C * M;
    float* o = out + (size_t)b * C * Q + q;
    for (int c = blockIdx.y; c < C; c += gridDim.y) {
        const float* fc = f + (size_t)c * M;
        float acc = 0.0f;
#pragma unroll
        for (int s = 0; s < KI_KMAX; ++s)
            if (s < k) acc = __fadd_rn(acc, __fmul_rn(__ldg(fc + j[s]), w[s]));
        o[(size_t)c * Q] = acc;
    }
}

// project_tile.cu
bool project_tile_eligible(const float* feat2d, const int64_t* nn, const float* out, int B, int C2, int C3, int H, int W, int N);
cudaError_t project_tile_launch(const float* xy, const float* feat2d, const float* feat3d, const int64_t* nn, float* out,
                                float* scratch, float* sampled_cf, int B, int C2, int C3, int H, int W, int N, cudaStream_t st);
int64_t project_tile_extra_scratch_floats(int B, int N);

// Which route a call takes.  B200_PROJECT_ROUTE = "two_pass" | "tiled" | unset (automatic), read per call: for ablations and tests.
// Automatic: the tiled route where TMA can address the map and the cloud is dense enough that a pixel's nearest point
// normally lies inside the 4-pixel halo (<= 16 pixels per point); small maps (pyramid levels 3-5 of a 960-wide image:
// a few 60 x 32 tiles per sample cannot fill 148 persistent CTAs) stay on the two-pass kernels.
static bool project_route_tiled(const float* feat2d, const int64_t* nn, const float* out, int B, int C2, int C3, int H, int W, int N) {
    const char* v = getenv("B200_PROJECT_ROUTE");
    const int forced = !v ? 0 : (strcmp(v, "two_pass") == 0 ? 1 : (strcmp(v, "tiled") == 0 ? 2 : 0));
    if (forced == 1 || !project_tile_eligible(feat2d, nn, out, B, C2, C3, H, W, N)) return false;
    if (forced == 2) return true;
    return (int64_t)H * W >= 4096 && (int64_t)H * W <= (int64_t)16 * N;
}

static int pick_csplit(int64_t cols, int B, int C) {
    const int64_t ctas = (int64_t)ceil_div(cols, 256) * B;
    const int64_t want = (int64_t)sm_count() * 4;
    int64_t s = (want + ctas - 1) / ctas;
    if (s < 1) s = 1;
    if (s > C) s = C;
    if (s > 65535) s = 65535;
    return (int)s;
}

}  // namespace b200

extern "C" int b200_gather_cf(const void* data, const int64_t* idx, void* out, int B, int C, int N, int64_t I,
                              int* bad_count, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0 || C == 0 || I == 0) || (data && idx && out), "b200_gather_cf: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 0 && N >= 1 && I >= 0, "b200_gather_cf: bad sizes");
    B200_REQUIRE(B <= 65535, "b200_gather_cf: B exceeds the grid limit");
    if (B == 0 || C == 0 || I == 0) return B200_OK;
    dim3 grid(ceil_div(I, 256), pick_csplit(I, B, C), B);
    gather_cf_kernel<<<grid, 256, 0, as_stream(stream)>>>((const uint32_t*)data, idx, (uint32_t*)out, C, N, I, bad_count);
    B200_LAUNCH_CHECK("b200_gather_cf");
    return B200_OK;
}

extern "C" int b200_gather_cl(const void* data, const int64_t* idx, void* out, int B, int C, int N, int64_t I,
                              int* bad_count, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0 || C == 0 || I == 0) || (data && idx && out), "b200_gather_cl: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 0 && N >= 1 && I >= 0, "b200_gather_cl: bad sizes");
    B200_REQUIRE(B <= 65535, "b200_gather_cl: B exceeds the grid limit");
    if (B == 0 || C == 0 || I == 0) return B200_OK;
    const bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(data) & 15) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    const int64_t elems = I * (vec ? C / 4 : C);
    dim3 grid(ceil_div(elems, 256), B);
    if (vec) gather_cl_kernel<true><<<grid, 256, 0, as_stream(stream)>>>((const uint32_t*)data, idx, (uint32_t*)out, C, N, I, bad_count);
    else     gather_cl_kernel<false><<<grid, 256, 0, as_stream(stream)>>>((const uint32_t*)data, idx, (uint32_t*)out, C, N, I, bad_count);
    B200_LAUNCH_CHECK("b200_gather_cl");
    return B200_OK;
}

extern "C" int b200_grid_sample_pts(const float* feat, const float* xy, float* out, int B, int C, int H, int W, int N,
                                    b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0 || C == 0 || N == 0) || (feat && xy && out), "b200_grid_sample_pts: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 0 && H >= 1 && W >= 1 && N >= 0, "b200_grid_sample_pts: bad sizes");
    B200_REQUIRE((int64_t)H * W < (1ll << 31) && B <= 65535, "b200_grid_sample_pts: plane or batch too large");
    if (B == 0 || C == 0 || N == 0) return B200_OK;
    int csplit = pick_csplit((int64_t)N * 2, B, (C + 1) / 2);
    dim3 grid(ceil_div(N, 128), csplit, B);
    grid_sample_pts_kernel<<<grid, 256, 0, as_stream(stream)>>>(feat, xy, out, C, H, W, N);
    B200_LAUNCH_CHECK("b200_grid_sample_pts");
    return B200_OK;
}

extern "C" int b200_backwarp2d(const float* x, const float* flow, float* out, int B, int C, int H, int W, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0 || C == 0) || (x && flow && out), "b200_backwarp2d: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 0 && H >= 1 && W >= 1, "b200_backwarp2d: bad sizes");
    B200_REQUIRE((int64_t)H * W < (1ll << 31) && B <= 65535, "b200_backwarp2d: plane or batch too large");
    if (B == 0 || C == 0) return B200_OK;
    const int64_t HW = (int64_t)H * W;
    int csplit = pick_csplit(HW * 2, B, (C + 1) / 2);
    dim3 grid(ceil_div(HW, 128), csplit, B);
    backwarp2d_border_kernel<<<grid, 256, 0, as_stream(stream)>>>(x, flow, out, C, H, W);
    B200_LAUNCH_CHECK("b200_backwarp2d");
    return B200_OK;
}

extern "C" int b200_convex_upsample(const float* flow, const float* mask, float* out, int B, int H, int W, int scale,
                                    b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0) || (flow && mask && out), "b200_convex_upsample: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && H >= 1 && W >= 1, "b200_convex_upsample: bad sizes");
    B200_REQUIRE(scale == 2 || scale == 4 || scale == 8, "b200_convex_upsample: scale_factor must be 2, 4 or 8 (got %d)", scale);
    B200_REQUIRE((int64_t)H * W * scale * scale < (1ll << 31) && B <= 65535, "b200_convex_upsample: plane or batch too large");
    B200_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "b200_convex_upsample: out must be 16-byte aligned");
    if (B == 0) return B200_OK;
    dim3 grid(ceil_div((int64_t)H * W, 256), scale, B);
    cudaStream_t st = as_stream(stream);
    if (scale == 2) convex_upsample_kernel<2><<<grid, 256, 0, st>>>(flow, mask, out, H, W);
    else if (scale == 4) convex_upsample_kernel<4><<<grid, 256, 0, st>>>(flow, mask, out, H, W);
    else convex_upsample_kernel<8><<<grid, 256, 0, st>>>(flow, mask, out, H, W);
    B200_LAUNCH_CHECK("b200_convex_upsample");
    return B200_OK;
}

extern "C" int64_t b200_project_nn_corr_scratch_floats(int B, int C2, int C3, int N) {
    if (B < 0 || C2 < 0 || C3 < 0 || N < 0) return 0;
    // point-major rows [S | T] (both routes) + the tiled route's per-tile point lists
    return (int64_t)B * N * (b200::round4(C2) + b200::round4(C3)) + b200::project_tile_extra_scratch_floats(B, N);
}

extern "C" int b200_project_nn_corr(const float* xy, const float* feat2d, const float* feat3d, const int64_t* nn,
                                    float* out, float* scratch, int B, int C2, int C3, int H, int W, int N,
                                    b200_stream_t stream) {
    return b200_project_nn_corr_sampled(xy, feat2d, feat3d, nn, out, scratch, nullptr, B, C2, C3, H, W, N, stream);
}

extern "C" int b200_project_nn_corr_sampled(const float* xy, const float* feat2d, const float* feat3d, const int64_t* nn,
                                            float* out, float* scratch, float* sampled_cf, int B, int C2, int C3, int H,
                                            int W, int N, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0) || (xy && feat2d && feat3d && nn && out && scratch), "b200_project_nn_corr: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C2 >= 1 && C3 >= 0 && H >= 1 && W >= 1 && N >= 1, "b200_project_nn_corr: bad sizes");
    B200_REQUIRE((int64_t)H * W < (1ll << 31) && B <= 65535, "b200_project_nn_corr: plane or batch too large");
    B200_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "b200_project_nn_corr: scratch must be 16-byte aligned");
    if (B == 0) return B200_OK;
    cudaStream_t st = as_stream(stream);
    if (project_route_tiled(feat2d, nn, out, B, C2, C3, H, W, N)) {
        // one pass over feat2d (project_tile.cu): prep (T rows + per-tile point lists) -> tile kernel -> post (far pixels,
        // sampled tensor to channel-first, feat3d slabs)
        const cudaError_t e = project_tile_launch(xy, feat2d, feat3d, nn, out, scratch, sampled_cf, B, C2, C3, H, W, N, st);
        if (e != cudaSuccess) return cuda_fail(e, "b200_project_nn_corr(tile)");
        return B200_OK;
    }
    sample_point_major_kernel<<<dim3(ceil_div(N, 16), B), 256, 0, st>>>(feat2d, xy, feat3d, scratch, sampled_cf, C2, C3, H, W, N);
    B200_LAUNCH_CHECK("b200_project_nn_corr(sample)");
    project_nn_corr_kernel<<<dim3(ceil_div((int64_t)H * W, 256), B, 1 + ceil_div(C3, PN_SLAB)), 256, 0, st>>>(
        xy, feat2d, nn, scratch, out, C2, C3, H, W, N);
    B200_LAUNCH_CHECK("b200_project_nn_corr");
    return B200_OK;
}

extern "C" int b200_knn_interpolate(const float* input_xyz, const float* input_feat, const float* query_xyz,
                                    const int64_t* knn_idx, float* out, int B, int C, int M, int Q, int k,
                                    b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0 || C == 0 || Q == 0) || (input_xyz && input_feat && query_xyz && knn_idx && out), "b200_knn_interpolate: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && C >= 0 && M >= 1 && Q >= 0, "b200_knn_interpolate: bad sizes");
    B200_REQUIRE(k >= 1 && k <= KI_KMAX, "b200_knn_interpolate: k must be in [1,%d] (got %d)", KI_KMAX, k);
    B200_REQUIRE(B <= 65535, "b200_knn_interpolate: B exceeds the grid limit");
    if (B == 0 || C == 0 || Q == 0) return B200_OK;
    dim3 grid(ceil_div(Q, 256), pick_csplit(Q, B, C), B);
    knn_interpolate_kernel<<<grid, 256, 0, as_stream(stream)>>>(input_xyz, input_feat, query_xyz, knn_idx, out, C, M, Q, k);
    B200_LAUNCH_CHECK("b200_knn_interpolate");
    return B200_OK;
}
