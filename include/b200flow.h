/*
 * b200flow.h — C-ABI of libb200flow.so: the RPEFlow correlation / cost-volume hot path on B200 (sm_100a).
 *
 * Every entry point takes plain DEVICE pointers + sizes + a CUDA stream (as void*), owns no memory, keeps no
 * global state, and launches on the stream it is given (so it is CUDA-graph capturable and usable from
 * one-process-per-GPU shards).  Outputs and any scratch are allocated by the caller (the reference does the
 * same: its C++ wrappers allocate with torch and hand raw pointers to the kernels).
 *
 * Return value: 0 on success, a negative B200_E* code otherwise; b200_last_error() gives the message of the
 * last failure on the calling thread.  The reference's TORCH_CHECKs map to B200_EINVAL; the reference never
 * checks CUDA errors after launch, this library does (B200_ECUDA).
 *
 * Reference citations are relative to the reference repo root (danqu130/RPEFlow).
 */
#ifndef B200FLOW_H_
#define B200FLOW_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK       0
#define B200_EINVAL  (-1)   /* bad argument (shape, k>32, N<=n_samples, null pointer, ...)            */
#define B200_ECUDA   (-2)   /* CUDA runtime/driver error at or after launch                          */
#define B200_ENOSUP  (-3)   /* valid in the reference but outside what this build supports            */

typedef void* b200_stream_t;            /* a cudaStream_t; NULL = legacy default stream                */

#if defined(__GNUC__)
#define B200_API __attribute__((visibility("default")))
#else
#define B200_API
#endif

/* Library identification. b200_abi_version() changes whenever a signature below changes. */
B200_API int         b200_abi_version(void);
B200_API const char* b200_build_info(void);      /* "sm_100a; <nvcc version>; <date>"                            */
B200_API const char* b200_last_error(void);      /* thread-local; "" if none                                    */

/* ------------------------------------------------------------------------------------------------------
 * a1  2-D local correlation cost volume, forward.
 * Replaces: models/csrc/correlation/correlation.cpp:11-22 (correlation_forward_cuda) +
 *           correlation_forward_kernel.cu:11-55; Python binding `_correlation_forward_cuda`
 *           (correlation.cpp:39), called from models/csrc/wrapper.py:24.
 *   in1, in2 : [B,H,W,C] fp32, NHWC contiguous            out : [B,(2md+1)^2,H,W] fp32, NCHW
 *   out[b,(dy+md)*(2md+1)+(dx+md),y,x] = (1/C) * sum_c in1[b,y,x,c]*in2[b,y+dy,x+dx,c]; 0 outside the image.
 * Every output element is written (the caller does not need to zero `out`).
 * Limits: 1 <= md <= 64, C >= 1.  md <= 4 takes the tuned kernels (the model uses 4); larger displacements a plain one.
 */
B200_API int b200_corr2d_fwd(const float* in1_nhwc, const float* in2_nhwc, float* out_nchw,
                    int B, int C, int H, int W, int md, b200_stream_t stream);

/* a1 as the wrapper calls it (models/csrc/wrapper.py:55-72): the same cost volume straight from NCHW feature maps, so
 * the wrapper's two NCHW->NHWC permutes (wrapper.py:68-69) disappear.  Same result as b200_corr2d_fwd on the permuted
 * inputs up to fp32 summation order.
 *   in1, in2 : [B,C,H,W] fp32, NCHW contiguous, 16-byte aligned        out : [B,81,H,W] fp32, 16-byte aligned
 * Limits: md == 4 and W % 4 == 0 (TMA cannot address rows that are not 16-byte multiples); anything else returns
 * B200_ENOSUP (permute and call b200_corr2d_fwd, as the reference's wrapper does).
 */
B200_API int b200_corr2d_fwd_nchw(const float* in1_nchw, const float* in2_nchw, float* out_nchw,
                         int B, int C, int H, int W, int md, b200_stream_t stream);

/* f3  a1 with the caller's activation fused (SURVEY §8f rank 3): leaky_relu(correlation2d(f1, f2_warp, md), slope),
 * models/RPEFlow_core.py:362 — the activation is the epilogue of the same kernels, no extra pass over the 81 planes.
 * negative_slope in [0,1]; 1 is the identity (== b200_corr2d_fwd_nchw).  Same limits as b200_corr2d_fwd_nchw.
 */
B200_API int b200_corr2d_fwd_nchw_leaky(const float* in1_nchw, const float* in2_nchw, float* out_nchw,
                               int B, int C, int H, int W, int md, float negative_slope, b200_stream_t stream);

/* f3  backwarp_2d with padding_mode='border' (models/utils.py:186-198; caller RPEFlow_core.py:351): the producer of
 * in2 for the call above at every level but the coarsest.
 *   x : [B,C,H,W] NCHW fp32;  flow : [B,2,H,W] (x then y displacement, pixels)  ->  out : [B,C,H,W]
 *   out[b,c,y,x] = bilinear(x[b,c], (x + flow[b,0,y,x], y + flow[b,1,y,x])), align_corners=True, coordinates clamped to
 *   the image (border).  Coordinates take the reference's normalise / un-normalise round trip in fp32.
 */
B200_API int b200_backwarp2d(const float* x_nchw, const float* flow, float* out_nchw,
                    int B, int C, int H, int W, b200_stream_t stream);

/* f4  convex_upsample (models/utils.py:201-214; caller RPEFlow_core.py:424 with scale_factor 4): RAFT's convex upsampling.
 *   flow : [B,2,H,W];  mask : [B,9*s*s,H,W] (logits; channel = (k*s + i)*s + j, k = 3x3 tap)  ->  out : [B,2,s*H,s*W]
 *   out[b,c,y*s+i,x*s+j] = sum_k softmax_k(mask[b,:,y,x])[k,i,j] * s * flow[b,c,y+k/3-1,x+k%3-1]   (zeros outside)
 * s in {2,4,8}; out 16-byte aligned.
 */
B200_API int b200_convex_upsample(const float* flow, const float* mask, float* out,
                         int B, int H, int W, int scale, b200_stream_t stream);

/* f3 / f4 backwards (decoder_bwd.cu).  Shared rules:
 *   - inputs, sizes and limits exactly as given to the matching forward; grad_* has the forward output's shape;
 *   - a gradient output passed as NULL is not computed and not written; every other one is overwritten (the entry
 *     zero-fills what it accumulates, with cudaMemsetAsync on `stream`);
 *   - empty calls accept NULL pointers; bad arguments return B200_EINVAL before anything touches a device;
 *   - no host synchronisation and no allocation (the calls can be captured in a CUDA graph).
 * Taps, weights and softmax are recomputed from the inputs with the forward's own fp32 operations.
 *
 * backwarp2d: dx [B,C,H,W] is scattered with float atomics (not bit-reproducible); dflow [B,2,H,W] is reduced over the
 * channels in a fixed order.  The flow gradient follows ATen's grid_sampler_2d backward with border padding: it is 0
 * where the un-clamped sample coordinate is <= 0 or >= size - 1 (a sample exactly on the border counts as clipped).
 */
B200_API int b200_backwarp2d_bwd(const float* x_nchw, const float* flow, const float* grad_out_nchw,
                        float* dx_nchw, float* dflow, int B, int C, int H, int W, b200_stream_t stream);

/* convex_upsample: dflow [B,2,H,W], dmask [B,9*s*s,H,W]; grad_out [B,2,s*H,s*W], 16-byte aligned.  Two passes, no
 * atomics: both gradients are bit-reproducible.  scratch : >= b200_convex_upsample_bwd_scratch_floats(B,H,W,s) floats
 * (per low-res pixel the 9 taps' partial flow gradients); needed only when dflow is not NULL.
 */
B200_API int64_t b200_convex_upsample_bwd_scratch_floats(int B, int H, int W, int scale);
B200_API int b200_convex_upsample_bwd(const float* flow, const float* mask, const float* grad_out,
                             float* dflow, float* dmask, float* scratch,
                             int B, int H, int W, int scale, b200_stream_t stream);

/* a2  backward of a1.
 * Replaces: correlation.cpp:24-35 (correlation_backward_cuda) + correlation_backward_kernel.cu:4-89;
 *           binding `_correlation_backward_cuda` (correlation.cpp:40), called from wrapper.py:31.
 *   grad_out : [B,(2md+1)^2,H,W] NCHW contiguous; in1,in2 : NHWC;  gin1,gin2 : [B,C,H,W] **NCHW** (as the
 *   reference; wrapper.py:34-35 permutes them back to NHWC).
 */
B200_API int b200_corr2d_bwd(const float* grad_out_nchw, const float* in1_nhwc, const float* in2_nhwc,
                    float* gin1_nchw, float* gin2_nchw,
                    int B, int C, int H, int W, int md, b200_stream_t stream);

/* a2 on NCHW maps: the backward of b200_corr2d_fwd_nchw with no permutes on either side.
 *   grad_out : [B,81,H,W];  in1, in2 : [B,C,H,W] NCHW contiguous;  gin1, gin2 : [B,C,H,W] NCHW.  Any alignment, any W.
 *   - a gradient passed as NULL is neither computed nor written; every element of a requested one is written;
 *   - B = 0, or both gradients NULL, is a no-op that accepts NULL pointers; bad sizes, null inputs and grids beyond
 *     2^31 - 1 tiles return B200_EINVAL before anything touches a device;
 *   - no atomics (bit-reproducible), no allocation and no host synchronisation (the call can be captured in a graph).
 * Limits: md == 4; any other displacement returns B200_ENOSUP (permute the inputs and call b200_corr2d_bwd).  Sums in
 * the order of b200_corr2d_bwd's md = 4 tiled kernel, so where that one runs (C % 4 == 0, W % 4 == 0, 16-byte aligned
 * pointers) both entries return the same bits.
 */
B200_API int b200_corr2d_bwd_nchw(const float* grad_out_nchw, const float* in1_nchw, const float* in2_nchw,
                         float* gin1_nchw, float* gin2_nchw, int B, int C, int H, int W, int md, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * a3  furthest point sampling.
 * Replaces: furthest_point_sampling.cpp:5-16 + furthest_point_sampling_kernel.cu:34-85; binding
 *           `_furthest_point_sampling_cuda` (furthest_point_sampling.cpp:20), called from wrapper.py:101.
 *   xyz : [B,N,3] fp32 contiguous        idx : [B,n_samples] int64
 * Rule (SURVEY §8a): idx[0]=0; dist_i = min(dist_i, ((dx*dx+dy*dy)+dz*dz)) in non-fused fp32, init 1e10;
 * next = argmax(dist), LOWEST index on ties  == the reference torch fallback (wrapper.py:83-96) bit for bit.
 * Requires N > n_samples >= 1 (wrapper.py:98 asserts it).  No scratch needed (distances live in registers).
 * Limits: N <= 65536 (B200_ENOSUP otherwise: call b200_fps_large, which takes any N).
 */
B200_API int b200_fps(const float* xyz, int64_t* idx, int B, int N, int n_samples, b200_stream_t stream);

/* a3 for clouds of any size (the reference's kernel, furthest_point_sampling_kernel.cu:34-85, keeps its running
 * distances in the global `dists_temp` and takes any N; b200_fps stops at 65536 points).  Same rule, same result as
 * b200_fps bit for bit: a pruned scan over one 8-CTA thread-block cluster per cloud, on a Morton-sorted copy of the
 * cloud in the caller's scratch (fps_large.cu).
 *   xyz : [B,N,3] fp32 contiguous        idx : [B,n_samples] int64
 *   scratch : >= b200_fps_scratch_bytes(B,N) bytes, 256-byte aligned; its contents on entry do not matter.
 * Requires N > n_samples >= 1; short or misaligned scratch -> B200_EINVAL.  B = 0 is a no-op (NULL pointers allowed).
 * No host synchronisation and no allocation: capturable in a CUDA graph.
 */
B200_API int64_t b200_fps_scratch_bytes(int B, int N);                 /* -1 for B < 0 or N < 1 */
B200_API int b200_fps_large(const float* xyz, int64_t* idx, void* scratch, int64_t scratch_bytes, int B, int N,
                            int n_samples, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * a4  k nearest neighbours (brute-force exact).
 * Replaces: k_nearest_neighbor.cpp:6-24 + k_nearest_neighbor_kernel.cu:8-112; binding
 *           `_k_nearest_neighbor_cuda` (k_nearest_neighbor.cpp:28), called from wrapper.py:125.
 *   input : [B,M,D] fp32, query : [B,Q,D] fp32, D in {2,3}        idx : [B,Q,k] int64
 * Rule (SURVEY §8a): d = ((dx*dx+dy*dy)+dz*dz) non-fused fp32; result sorted by (d ascending, index
 * ascending); 1 <= k <= 32 (the reference silently overruns its 32-slot arrays beyond that -> B200_EINVAL
 * here).  If M < k the trailing slots are 0 (the reference zero-initialises, k_nearest_neighbor.cpp:16).
 */
B200_API int b200_knn(const float* input_xyz, const float* query_xyz, int64_t* idx,
             int B, int M, int Q, int D, int k, b200_stream_t stream);

/* a4, production path: the same search with the same bit-exact result, but over a uniform cell grid built from the
 * inputs (exact early termination, brute force only as the limit case; see csrc/knn_grid.cu for the bound).
 *   scratch : >= b200_knn_scratch_bytes(B,M,Q,D,k) bytes, 256-byte aligned (cell-ordered copies of the inputs and,
 *             for D=3, of the queries; per-cloud cell table).  Contents are undefined afterwards.
 */
B200_API int64_t b200_knn_scratch_bytes(int B, int M, int Q, int D, int k);
B200_API int b200_knn_grid(const float* input_xyz, const float* query_xyz, int64_t* idx,
                  void* scratch, int64_t scratch_bytes,
                  int B, int M, int Q, int D, int k, b200_stream_t stream);

/* The same search on CHANNEL-FIRST clouds: input_xyz [B,D,M], query_xyz [B,D,Q] — the layout every model call site
 * passes (models/csrc/wrapper.py:119-122 transposes + copies them per call; this entry reads them as they are). */
B200_API int b200_knn_grid_cf(const float* input_xyz, const float* query_xyz, int64_t* idx, void* scratch,
                              int64_t scratch_bytes, int B, int M, int Q, int D, int k, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * a6  batched index gathers.  Elements are 4 bytes wide and moved bit-exactly (fp32 or int32 data).
 * Replaces: models/utils.py:119-137 (batch_indexing_channel_first) and :101-116 (.._channel_last).
 *   channel-first: data [B,C,N], idx [B,I] int64 -> out [B,C,I]   out[b,c,i] = data[b,c,idx[b,i]]
 *   channel-last : data [B,N,C], idx [B,I] int64 -> out [B,I,C]   out[b,i,:] = data[b,idx[b,i],:]
 * Negative indices wrap once (idx+N) as torch indexing does; anything else out of range -> B200_EINVAL is
 * NOT detected on the device (no sync) — such indices are clamped and counted in *bad_count if non-NULL.
 */
B200_API int b200_gather_cf(const void* data, const int64_t* idx, void* out,
                   int B, int C, int N, int64_t I, int* bad_count, b200_stream_t stream);
B200_API int b200_gather_cl(const void* data, const int64_t* idx, void* out,
                   int B, int C, int N, int64_t I, int* bad_count, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * a7  image -> point bilinear projection gather.
 * Replaces: models/utils.py:288-294 (grid_sample_wrapper = normalise + F.grid_sample(bilinear,
 *           align_corners=True, zero padding)).
 *   feat : [B,C,H,W] NCHW fp32;  xy : [B,2,N] (x row then y row, level-pixel units)  ->  out : [B,C,N]
 * Coordinates take the reference's round trip: xn = 2*x/(W-1)-1 ; ix = ((xn+1)/2)*(W-1)  (fp32).
 */
B200_API int b200_grid_sample_pts(const float* feat_nchw, const float* xy, float* out,
                         int B, int C, int H, int W, int N, b200_stream_t stream);

/* a6 / a7 backwards (decoder_bwd.cu): the gradients of grid_sample_wrapper (F.grid_sample, models/utils.py:288-294) and
 * of batch_indexing_channel_first / _last (torch.gather / advanced indexing, models/utils.py:119-137, :101-116).
 * Rules as for the f3 / f4 backwards above: inputs and sizes exactly as given to the matching forward, grad_out has the
 * forward output's shape; every gradient is overwritten (zero-filled with cudaMemsetAsync on `stream`, then accumulated);
 * empty calls accept NULL pointers; bad arguments return B200_EINVAL before anything touches a device; no host
 * synchronisation and no allocation (capturable in a CUDA graph).  Scattered gradients are summed with float atomics:
 * not bit-reproducible.
 *
 * grid_sample_pts: dfeat [B,C,H,W], dxy [B,2,N]; either may be NULL (not computed, not written).  Taps are recomputed
 * with the forward's own fp32 operations.  dxy follows ATen's grid_sampler_2d backward with zero padding (out-of-image
 * taps read 0, nothing is clipped), reduced over the channels in a fixed order.  Where the forward finds no tap inside
 * the image — the point lies outside it, or a coordinate is huge (|.| >= 1e9 after the round trip) or not finite, or
 * W = 1 / H = 1 makes the round trip 0/0 — dxy is 0 (ATen gives 0 or NaN there).
 */
B200_API int b200_grid_sample_pts_bwd(const float* feat_nchw, const float* xy, const float* grad_out, float* dfeat_nchw,
                             float* dxy, int B, int C, int H, int W, int N, b200_stream_t stream);

/* gathers: fp32 only.  ddata [B,C,N] (cf) / [B,N,C] (cl) receives grad_out [B,C,I] / [B,I,C] at the element the forward
 * read: negative indices wrap once, out-of-range ones clamp (the forward's rule; nothing is counted here).  The
 * channel-last entry adds whole 16-byte rows (red.global.add.v4.f32) when C % 4 == 0 and both pointers are 16-byte
 * aligned. */
B200_API int b200_gather_cf_bwd(const float* grad_out, const int64_t* idx, float* ddata,
                       int B, int C, int N, int64_t I, b200_stream_t stream);
B200_API int b200_gather_cl_bwd(const float* grad_out, const int64_t* idx, float* ddata,
                       int B, int C, int N, int64_t I, b200_stream_t stream);

/* a8  point -> image projection with nearest-neighbour correlation.
 * Replaces: models/utils.py:297-317 (project_feat_with_nn_corr) with nn_indices supplied
 *           (models/RPEFlow_core.py:329-330 always supplies them).
 *   xy [B,2,N]; feat2d [B,C2,H,W]; feat3d [B,C3,N]; nn [B,H*W] int64 -> out [B,C3+3,H,W]
 *   out[:,0:2] = xy[:,nn]-pixel ; out[:,2] = mean_c( bilinear(feat2d, xy[:,nn])[c] * feat2d[c,pixel] ) ;
 *   out[:,3:]  = feat3d[:,nn]
 *   scratch : >= b200_project_nn_corr_scratch_floats(B, C2, C3, N) floats, 16-byte aligned (one point-major row per
 *             point: feat2d sampled at the point, then the point's feat3d channels; each part padded to 4 floats).
 */
B200_API int64_t b200_project_nn_corr_scratch_floats(int B, int C2, int C3, int N);
B200_API int b200_project_nn_corr(const float* xy, const float* feat2d_nchw, const float* feat3d,
                         const int64_t* nn, float* out, float* scratch,
                         int B, int C2, int C3, int H, int W, int N, b200_stream_t stream);

/* a8 + a7 in one pass.  Same as b200_project_nn_corr; additionally, when sampled_cf != NULL, writes
 *   sampled_cf [B,C2,N] = bilinear(feat2d, xy)   == grid_sample_wrapper(feat2d, xy) (models/utils.py:288-294),
 * the tensor the 2D->3D fuser asks for right after the 3D->2D one with the same map and points
 * (models/RPEFlow_core.py:31+53, :80+107, :134+157): the feature map is sampled once, not twice.
 */
B200_API int b200_project_nn_corr_sampled(const float* xy, const float* feat2d_nchw, const float* feat3d,
                         const int64_t* nn, float* out, float* scratch, float* sampled_cf,
                         int B, int C2, int C3, int H, int W, int N, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * f1  PointConv forward (SURVEY §8f rank 1), both PointConvDownSampling and PointConvNoSampling (= sampled_xyz is xyz).
 * Replaces: models/pointconv.py:33-61 and :90-122 after their k_nearest_neighbor call (gathers, weight net,
 *           torch.matmul(weights, knn_features), nn.Linear(16*(C+3), out), LeakyReLU(0.1); norm = None).
 *   xyz [B,3,N], feat [B,C,N], sampled_xyz [B,3,S] (channel-first fp32), knn [B,S,16] int64 into xyz -> out [B,Cout,S]
 *   weights (row-major [out,in]): weight_net Wa [8,3], ba [8], Wb [16,8], bb [16]; linear L [Cout, 16*(C+3)], bias [Cout]
 *   scratch : >= b200_pointconv_scratch_floats(B,C,Cout,N) floats, 16-byte aligned.
 *   precision: 1 = TF32 tensor cores (tcgen05), 2 (and 0) = 3xTF32 (fp32-level accuracy).
 *   knn indices are local to each sample.  A negative index wraps once (j + N, as torch indexing does) and whatever is
 *   still outside [0, N-1] is clamped to it: -1 reads point N-1, -N-3 reads point 0, N or more reads point N-1.  No
 *   error is reported for such indices.
 * Limits: k == 16, Cout <= 256 (B200_ENOSUP otherwise).
 */
typedef struct b200_pointconv_weights {
    const float *Wa, *ba, *Wb, *bb, *L, *bias;
} b200_pointconv_weights;
B200_API int64_t b200_pointconv_scratch_floats(int B, int C, int Cout, int N);
B200_API int b200_pointconv_fwd(const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                       const b200_pointconv_weights* w, float* out, float* scratch,
                       int B, int C, int Cout, int N, int S, int k, int precision, b200_stream_t stream);

/* f1 for training: the same call without the activation.  Same arguments and scratch as b200_pointconv_fwd; writes
 *   out [B,Cout,S] = y, the nn.Linear output (models/pointconv.py before norm_fn / activation_fn), so that a caller can
 *   apply any norm and activation itself.  LeakyReLU(0.1) of it equals b200_pointconv_fwd bit for bit.
 * Limits: k == 16, Cout <= 256, N <= 65536 (B200_ENOSUP otherwise).
 */
B200_API int b200_pointconv_fwd_linear(const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                       const b200_pointconv_weights* w, float* out, float* scratch,
                       int B, int C, int Cout, int N, int S, int k, int precision, b200_stream_t stream);

/* f1 backward: gradients of b200_pointconv_fwd_linear with respect to both clouds, the features and the six parameters.
 * Replaces the autograd graph of models/pointconv.py:33-61 / :90-122 up to the Linear output.  M and the weight net are
 * recomputed from the inputs; the two Linear-sized contractions (dM = dy.L, dL = dy^T.M) run on tcgen05 tensor cores
 * (3xTF32), the rest in fp32.
 *   inputs, knn, w, B..k : exactly as given to the forward
 *   grad_y  : [B,Cout,S] channel-first, the gradient of y
 *   grads   : output pointers, same shapes as the tensors they differentiate (xyz [B,3,N], feat [B,C,N], sampled_xyz
 *             [B,3,S], weights as in b200_pointconv_weights).  NULL = not needed: its work is skipped and it is not
 *             written.  Every non-NULL output is overwritten.  For PointConvNoSampling (sampled_xyz = xyz) the caller
 *             adds the xyz and sampled_xyz gradients.
 *   scratch : >= b200_pointconv_bwd_scratch_floats(B,C,Cout,N,S) floats, 16-byte aligned.  It holds the point-major
 *             feature rows and their gradient (2 x B*N*roundup16(C+3) floats) and per-chunk M / dM images of at most
 *             32 MB each, whatever the batch.
 * Gradients of xyz, feat and sampled_xyz are summed with float atomics, so they are not bit-reproducible from run to
 * run; the parameter gradients are (per-CTA partials, fixed-order reduction).  No host synchronisation, no allocation.
 * Limits: k == 16, Cout <= 256, N <= 65536 (B200_ENOSUP otherwise).  B = 0 or S = 0 is a no-op; C = 0 is valid.
 */
typedef struct b200_pointconv_grads {
    float *xyz, *feat, *sampled_xyz;
    float *Wa, *ba, *Wb, *bb, *L, *bias;
} b200_pointconv_grads;
B200_API int64_t b200_pointconv_bwd_scratch_floats(int B, int C, int Cout, int N, int S);
B200_API int b200_pointconv_bwd(const float* xyz, const float* feat, const float* sampled_xyz, const int64_t* knn,
                       const b200_pointconv_weights* w, const float* grad_y, const b200_pointconv_grads* grads,
                       float* scratch, int B, int C, int Cout, int N, int S, int k, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * f2  inverse-distance interpolation over k nearest neighbours (SURVEY §8f rank 2).
 * Replaces: models/utils.py:140-156 (knn_interpolation) after its k_nearest_neighbor call — the two
 *           batch_indexing gathers, norm, clamp(1e-8), reciprocal, normalisation and weighted sum; backwarp_3d
 *           (:159-169) is the same op on (xyz1+flow, -flow).
 *   input_xyz [B,3,M], input_feat [B,C,M], query_xyz [B,3,Q]  (channel-first fp32), knn_idx [B,Q,k] int64 -> out [B,C,Q]
 * Every operation is rounded separately in the reference's order (bit-exact vs the oracle).  1 <= k <= 8 (the model uses 3).
 */
B200_API int b200_knn_interpolate(const float* input_xyz, const float* input_feat, const float* query_xyz,
                         const int64_t* knn_idx, float* out, int B, int C, int M, int Q, int k,
                         b200_stream_t stream);

/* f2 backward (decoder_bwd.cu), under the rules of the f3 / f4 backwards above.  knn_idx gets the forward's treatment
 * (negative indices wrap once, out-of-range ones are clamped), so every gradient lands where the forward read.
 *   d_input_xyz [B,3,M] and d_input_feat [B,C,M] are scattered with float atomics (not bit-reproducible);
 *   d_query_xyz [B,3,Q] is written once per query.  The distance clamp at 1e-8 passes no gradient (torch's clamp_min
 *   backward), so a query that coincides with one of its neighbours gives that pair no xyz gradient.
 * When only d_input_feat is requested the channel reduction the xyz gradients need is skipped.
 */
B200_API int b200_knn_interpolate_bwd(const float* input_xyz, const float* input_feat, const float* query_xyz,
                             const int64_t* knn_idx, const float* grad_out,
                             float* d_input_xyz, float* d_input_feat, float* d_query_xyz,
                             int B, int C, int M, int Q, int k, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * a5  3-D point cost volume (pwc3d_core.Correlation3D.forward), forward only.
 * Replaces: models/pwc3d_core.py:69-117 with both KNN index sets supplied by the caller
 *           (b200_knn(xyz2 as input, xyz1 as query) for knn12; knn11 as RPEFlow_core.py:331 computes it).
 *   xyz1 [B,3,N1], feat1 [B,Cin,N1], xyz2 [B,3,N2], feat2 [B,Cin,N2]        (channel-first fp32)
 *   knn12 [B,N1,k] int64 into cloud 2; knn11 [B,N1,k] int64 into cloud 1    -> out [B,Cout,N1]
 *   weights (row-major [out,in], the nn.Conv2d 1x1 weights squeezed):
 *     cost_mlp : W1 [Cout, 2*Cin+3], b1[Cout], W2 [Cout,Cout], b2[Cout]     LeakyReLU(0.1) after each
 *     weight_net{1,2}: Wa[8,3],ba[8], Wb[8,8],bb[8], Wc[Cout,8],bc[Cout]    ReLU after each (incl. last)
 *   packed as struct b200_corr3d_weights (device pointers).
 *   scratch : >= b200_corr3d_scratch_floats(B,Cin,Cout,N1,N2,k) floats.
 *   knn indices are local to each sample and are clamped to [0, N-1] of the cloud they index (N2 for knn12, N1 for
 *   knn11): a negative index reads point 0 (it does not wrap), N or more reads point N-1.  No error is reported.
 *   precision: 0 = fp32 FFMA everywhere; 1 = TF32 tensor cores (tcgen05) for the Cout x Cout layer,
 *              fp32 accumulate (what cuDNN does for the reference's 1x1 convs under torch's default
 *              allow_tf32); 2 = 3xTF32 split (tensor cores, ~fp32 accuracy).
 */
typedef struct b200_corr3d_weights {
    const float *W1, *b1, *W2, *b2;
    const float *n1_Wa, *n1_ba, *n1_Wb, *n1_bb, *n1_Wc, *n1_bc;   /* weight_net1 (self neighbours)  */
    const float *n2_Wa, *n2_ba, *n2_Wb, *n2_bb, *n2_Wc, *n2_bc;   /* weight_net2 (cross neighbours) */
} b200_corr3d_weights;

B200_API int64_t b200_corr3d_scratch_floats(int B, int Cin, int Cout, int N1, int N2, int k);
B200_API int b200_corr3d_fwd(const float* xyz1, const float* feat1, const float* xyz2, const float* feat2,
                    const int64_t* knn12, const int64_t* knn11, const b200_corr3d_weights* w,
                    float* out, float* scratch,
                    int B, int Cin, int Cout, int N1, int N2, int k, int precision, b200_stream_t stream);

/* a5 backward: gradients of b200_corr3d_fwd with respect to both clouds, both feature maps and the 16 parameters.
 * Replaces the autograd graph of models/pwc3d_core.py:69-117 (fp32 FFMA arithmetic, whatever precision the forward used).
 *   inputs, knn12, knn11, w, B..k : exactly as given to the forward
 *   grad_out    : [B,Cout,N1] channel-first, the gradient of `out`
 *   fwd_scratch : the forward's scratch, unchanged since the forward returned (its point-major P [B,N1,Cout] is read)
 *   grads       : output pointers, same shapes as the tensors they differentiate (xyz [B,3,N], feat [B,Cin,N], weights
 *                 [out,in] / [out]).  NULL = not needed: its work is skipped and it is not written.  Every non-NULL
 *                 output is overwritten (the callee zero-fills what it accumulates).
 *   scratch     : >= b200_corr3d_bwd_scratch_floats(B,Cin,Cout,N1,N2,k) floats, 16-byte aligned.
 * Only the 3->8->8 part of weight_net1 (n1_Wa, n1_ba, n1_Wb, n1_bb) is bit-reproducible from run to run.  Every other
 * gradient depends on float-atomic sums whose order varies: dP, dG2, the clouds, the split-K dW1 / db1, and the
 * per-CTA shared-memory sums of the weight-net output layers, W1's xyz columns and b2.  No host synchronisation, no
 * allocation.  b200_corr3d_bwd_det below computes the same gradients without float atomics.
 */
typedef struct b200_corr3d_grads {
    float *xyz1, *feat1, *xyz2, *feat2;
    float *W1, *b1, *W2, *b2;
    float *n1_Wa, *n1_ba, *n1_Wb, *n1_bb, *n1_Wc, *n1_bc;
    float *n2_Wa, *n2_ba, *n2_Wb, *n2_bb, *n2_Wc, *n2_bc;
} b200_corr3d_grads;

B200_API int64_t b200_corr3d_bwd_scratch_floats(int B, int Cin, int Cout, int N1, int N2, int k);
B200_API int b200_corr3d_bwd(const float* xyz1, const float* feat1, const float* xyz2, const float* feat2,
                    const int64_t* knn12, const int64_t* knn11, const b200_corr3d_weights* w,
                    const float* grad_out, const float* fwd_scratch, const b200_corr3d_grads* grads, float* scratch,
                    int B, int Cin, int Cout, int N1, int N2, int k, b200_stream_t stream);

/* a5 backward without float atomics: the same arguments, checks and outputs as b200_corr3d_bwd, except
 *   scratch : >= b200_corr3d_bwd_det_scratch_bytes(B,Cin,Cout,N1,N2,k) BYTES, 16-byte aligned, allocated by the caller.
 *             It holds b200_corr3d_bwd's scratch, a row buffer of B*N1*k*((Cout+3)&~3) floats (dP rows, then dz1 rows),
 *             B*N1*k float4 offset-gradient rows, the inverse index lists of knn11 and knn12 and the sort's workspace.
 *             The size function needs a CUDA device (it asks cub for the sort's workspace); it returns a negative value
 *             and sets b200_last_error() when that fails.  B*N1*k and B*N2 must be below 2^31.
 * Sum-order contract.  Every output is the same, bit for bit, on every run, whatever the scheduling of the CTAs and
 * whatever else runs on the device.  The four input gradients (xyz1, feat1, xyz2, feat2) of a sample do not depend on
 * the other samples of the batch.  Indices are first clamped as the forward clamps them (m < 0 -> 0, m >= N -> N-1).
 * Every gradient that b200_corr3d_bwd scatters over the knn rows (dP and dxyz1 over knn11; dG2, hence feat2 and W1's
 * feat2 columns, and dxyz2 over knn12) is, for each element, a sum over the rows r = i*k + s that point at it, taken
 * in ascending r and added in fp32 starting from +0.0.  Each dxyz1[i] is
 *     ((sum of the pulled +de rows of knn11, ascending r) - (own de over s, ascending s)) - (own t over s, ascending s)
 * with e = xyz1[m] - xyz1[i] (weight_net1) and t = dd + de the offset gradient of d = xyz2[j] - xyz1[i] (cost_mlp
 * layer 1 and weight_net2).  Weight gradients are fixed-order sums of per-tile, per-warp and per-split partials, so
 * they are reproducible but, like the atomic path's, depend on the whole batch.  No sum order depends on which
 * gradients are requested: a call that asks for a subset returns the same bits as a call that asks for all of them.
 * Sequence: knn11 / knn12 inverted (cub::DeviceRadixSort on key b*N + index, stable) -> pass 1 -> pull over knn11
 * (dP, dxyz1) -> pass 2 -> pull over knn12 (dG2, dxyz2) -> per-CTA partial sums -> linear backward (split-K partials
 * summed in ascending split order).  No host synchronisation, no allocation.
 */
B200_API int64_t b200_corr3d_bwd_det_scratch_bytes(int B, int Cin, int Cout, int N1, int N2, int k);
B200_API int b200_corr3d_bwd_det(const float* xyz1, const float* feat1, const float* xyz2, const float* feat2,
                    const int64_t* knn12, const int64_t* knn11, const b200_corr3d_weights* w,
                    const float* grad_out, const float* fwd_scratch, const b200_corr3d_grads* grads, float* scratch,
                    int B, int Cin, int Cout, int N1, int N2, int k, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * a9 event voxel grid, integer pixels + temporal bilinear (FlyingThings3D / EKubric).
 * Replaces: event_utils.py:109-128 (eventsToVoxel/eventsToVoxelTorch) -> :23-39, :264-303, :211-261, :162-208.
 *   events : [n,4] fp32 rows (x,y,t,p), time-sorted        vox : [bins*(polarity?2:1), H, W] fp32
 *   The kernel zero-fills vox itself.  status[0] counts events whose truncated pixel is outside the grid
 *   (the reference raises IndexError there; negative pixels in [-W,-1]/[-H,-1] wrap like torch indexing).
 *   polarity=1: channels [0,bins) count p>0 events, [bins,2*bins) count p<=0 events (both weight +1).
 *   polarity=0: one grid, weight = p (event_utils.py:247).
 *   A zero-length window (first and last timestamps equal) makes the reference's normalised time 0/0 = NaN, which its
 *   clamp keeps: every event then puts NaN into all channels at its pixel (with polarity=1, in both grids).
 */
B200_API int b200_event_voxel_int(const float* events, int64_t n, float* vox, int bins, int H, int W,
                         int polarity, int* status, b200_stream_t stream);

/* a10 event voxel grid, float pixels + tri-linear splat (DSEC).
 * Replaces: dsec.py:570-604 (eventsToVoxelInter) + :536-568 (eventsToVoxelInterTorch).
 *   x,y : [n] fp32 (rectified pixel coords); t : [n] int64 (microseconds, sorted); p : [n] fp32
 *   vox : [bins*(polarity?2:1), H, W]; scratch : >= 8 ints (first/last index of each polarity subset).
 */
B200_API int b200_event_voxel_trilinear(const float* x, const float* y, const int64_t* t, const float* p, int64_t n,
                               float* vox, int bins, int H, int W, int polarity, int* scratch,
                               b200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif  /* B200FLOW_H_ */
