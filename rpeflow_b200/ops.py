"""Host-side mirror of the reference's operator API for the cost-volume hot path.

Same names, argument meaning and return types as ``models/csrc/wrapper.py`` of danqu130/RPEFlow
(``correlation2d`` :55-72, ``furthest_point_sampling`` :75-103, ``k_nearest_neighbor`` :106-127,
``squared_distance`` :40-52, ``CorrelationFunction`` :18-37) and as the three pybind modules it imports
(``_correlation_forward_cuda`` / ``_correlation_backward_cuda`` correlation.cpp:38-41,
``_furthest_point_sampling_cuda`` furthest_point_sampling.cpp:19-21, ``_k_nearest_neighbor_cuda``
k_nearest_neighbor.cpp:27-29), but every op runs a hand-written sm_100a kernel through the C-ABI of
include/b200flow.h.  PyTorch is only used to own device memory and name the stream.

Differences from the reference, all deliberate:
* CUDA only.  There is no torch/CPU fallback: CPU tensors raise RuntimeError.
* Launches go to torch's *current* stream on the tensor's device (the reference uses the legacy default stream).
* ``k > 32`` raises (the reference overruns its 32-slot arrays); CUDA launch errors are reported.
* Exactness rules for FPS/KNN are the ones stated in include/b200flow.h.
"""
import torch

from . import _lib
from ._lib import check, lib

__all__ = [
    "correlation2d", "furthest_point_sampling", "k_nearest_neighbor", "squared_distance", "CorrelationFunction",
    "Correlation2dNCHWFunction",
    "_correlation_forward_cuda", "_correlation_backward_cuda", "_furthest_point_sampling_cuda",
    "_k_nearest_neighbor_cuda", "knn_bruteforce",
]


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _require(cond, msg):
    if not cond:
        raise RuntimeError(msg)          # what TORCH_CHECK raises on the reference side


def _cuda_f32(t, name):
    _require(isinstance(t, torch.Tensor), f"{name} must be a tensor")
    _require(t.is_cuda, f"{name} must be a CUDA tensor")
    _require(t.dtype == torch.float32, f"{name} must be a float tensor")
    _require(t.is_contiguous(), f"{name} must be a contiguous tensor")


# ------------------------------------------------------------------------------------------ extension-level API
def _correlation_forward_cuda(input1, input2, max_displacement):
    """input1/input2 [B,H,W,C] NHWC -> [B,(2md+1)^2,H,W]  (replaces correlation.cpp:11-22)."""
    _cuda_f32(input1, "input1")
    _cuda_f32(input2, "input2")
    _require(input1.shape == input2.shape and input1.dim() == 4, "input1/input2 must both be [B,H,W,C]")
    B, H, W, C = input1.shape
    md = int(max_displacement)
    out = torch.empty((B, (2 * md + 1) ** 2, H, W), dtype=torch.float32, device=input1.device)
    with torch.cuda.device(input1.device):
        check(lib.b200_corr2d_fwd(input1.data_ptr(), input2.data_ptr(), out.data_ptr(), B, C, H, W, md,
                                  _stream(input1)), "b200_corr2d_fwd")
    return out


def _correlation_backward_cuda(grad_output, input1, input2, max_displacement):
    """-> (grad_input1, grad_input2), both [B,C,H,W] NCHW as the reference (correlation.cpp:24-35)."""
    _cuda_f32(input1, "input1")
    _cuda_f32(input2, "input2")
    grad_output = grad_output.contiguous().float()      # the reference forgets this check (SURVEY §8b)
    B, H, W, C = input1.shape
    md = int(max_displacement)
    _require(tuple(grad_output.shape) == (B, (2 * md + 1) ** 2, H, W), "grad_output has the wrong shape")
    g1 = torch.empty((B, C, H, W), dtype=torch.float32, device=input1.device)
    g2 = torch.empty_like(g1)
    with torch.cuda.device(input1.device):
        check(lib.b200_corr2d_bwd(grad_output.data_ptr(), input1.data_ptr(), input2.data_ptr(), g1.data_ptr(),
                                  g2.data_ptr(), B, C, H, W, md, _stream(input1)), "b200_corr2d_bwd")
    return g1, g2


FPS_CLUSTER_MAX_N = 65536     # b200_fps holds a cloud of up to 8 x 8192 points in a cluster's registers


def _furthest_point_sampling_cuda(points_xyz, n_samples):
    """points_xyz [B,N,3] -> [B,n_samples] int64 (replaces furthest_point_sampling.cpp:5-16).  Clouds of more than 65536
    points (or whatever b200_fps of this build declines with B200_ENOSUP) take b200_fps_large with a scratch buffer."""
    _cuda_f32(points_xyz, "points_xyz")
    _require(points_xyz.dim() == 3 and points_xyz.shape[2] == 3, "points_xyz must be [B,N,3]")
    B, N, _ = points_xyz.shape
    out = torch.empty((B, int(n_samples)), dtype=torch.int64, device=points_xyz.device)
    with torch.cuda.device(points_xyz.device):
        if N <= FPS_CLUSTER_MAX_N:
            rc = lib.b200_fps(points_xyz.data_ptr(), out.data_ptr(), B, N, int(n_samples), _stream(points_xyz))
            if rc != _lib.B200_ENOSUP:
                check(rc, "b200_fps")
                return out
        nbytes = lib.b200_fps_scratch_bytes(B, N)
        scratch = torch.empty((max(nbytes, 256),), dtype=torch.uint8, device=points_xyz.device)  # torch blocks are 512-B aligned
        check(lib.b200_fps_large(points_xyz.data_ptr(), out.data_ptr(), scratch.data_ptr(), nbytes, B, N, int(n_samples),
                                 _stream(points_xyz)), "b200_fps_large")
    return out


def _knn_check(input_xyz, query_xyz):
    _cuda_f32(input_xyz, "input_xyz")
    _cuda_f32(query_xyz, "query_xyz")
    _require(input_xyz.dim() == 3 and query_xyz.dim() == 3 and input_xyz.shape[0] == query_xyz.shape[0]
             and input_xyz.shape[2] == query_xyz.shape[2], "input_xyz/query_xyz must be [B,M,D]/[B,Q,D]")


def _k_nearest_neighbor_cuda(input_xyz, query_xyz, k, channel_first=False):
    """input [B,M,D], query [B,Q,D] -> [B,Q,k] int64 (replaces k_nearest_neighbor.cpp:6-24).  Exact search over a
    cell grid (b200_knn_grid); bit-identical to the brute-force scan of knn_bruteforce().
    channel_first=True: input [B,D,M], query [B,D,Q] read as they are (b200_knn_grid_cf)."""
    _knn_check(input_xyz, query_xyz) if not channel_first else (_cuda_f32(input_xyz, "input_xyz"), _cuda_f32(query_xyz, "query_xyz"))
    if channel_first:
        _require(input_xyz.dim() == 3 and query_xyz.dim() == 3 and input_xyz.shape[:2] == query_xyz.shape[:2],
                 "input_xyz/query_xyz must be [B,D,M]/[B,D,Q]")
        B, D, M = input_xyz.shape
        Q = query_xyz.shape[2]
    else:
        B, M, D = input_xyz.shape
        Q = query_xyz.shape[1]
    out = torch.empty((B, Q, int(k)), dtype=torch.int64, device=query_xyz.device)
    nbytes = lib.b200_knn_scratch_bytes(B, M, Q, D, int(k))
    scratch = torch.empty((max(nbytes, 256),), dtype=torch.uint8, device=query_xyz.device)     # torch blocks are 512-B aligned
    fn, name = (lib.b200_knn_grid_cf, "b200_knn_grid_cf") if channel_first else (lib.b200_knn_grid, "b200_knn_grid")
    with torch.cuda.device(query_xyz.device):
        check(fn(input_xyz.data_ptr(), query_xyz.data_ptr(), out.data_ptr(), scratch.data_ptr(), nbytes,
                 B, M, Q, D, int(k), _stream(query_xyz)), name)
    return out


def knn_bruteforce(input_xyz, query_xyz, k):
    """Same contract through the brute-force kernels (b200_knn): every query scans every input."""
    _knn_check(input_xyz, query_xyz)
    B, M, D = input_xyz.shape
    Q = query_xyz.shape[1]
    out = torch.empty((B, Q, int(k)), dtype=torch.int64, device=query_xyz.device)
    with torch.cuda.device(query_xyz.device):
        check(lib.b200_knn(input_xyz.data_ptr(), query_xyz.data_ptr(), out.data_ptr(), B, M, Q, D, int(k),
                           _stream(query_xyz)), "b200_knn")
    return out


# ------------------------------------------------------------------------------------------ wrapper-level API
class CorrelationFunction(torch.autograd.Function):
    """NHWC in, NCHW out; gradients returned NHWC (wrapper.py:18-37)."""

    @staticmethod
    def forward(ctx, input1, input2, max_displacement):
        ctx.save_for_backward(input1, input2)
        ctx.max_displacement = max_displacement
        return _correlation_forward_cuda(input1, input2, max_displacement)

    @staticmethod
    def backward(ctx, grad_output):
        input1, input2 = ctx.saved_tensors
        g1, g2 = _correlation_backward_cuda(grad_output, input1, input2, ctx.max_displacement)
        return g1.permute(0, 2, 3, 1).contiguous(), g2.permute(0, 2, 3, 1).contiguous(), None


def _no_fallback(name, *tensors):
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError(f"rpeflow_b200.{name}: CUDA tensors required — this build has no CPU/torch fallback")


def _corr2d_fwd_nchw(a, b, md, negative_slope):
    """b200_corr2d_fwd_nchw[_leaky] on contiguous fp32 NCHW maps; None when the call is outside its limits."""
    B, C, H, W = a.shape
    out = torch.empty((B, (2 * md + 1) ** 2, H, W), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        if negative_slope is None:
            rc = lib.b200_corr2d_fwd_nchw(a.data_ptr(), b.data_ptr(), out.data_ptr(), B, C, H, W, md, _stream(a))
            name = "b200_corr2d_fwd_nchw"
        else:
            rc = lib.b200_corr2d_fwd_nchw_leaky(a.data_ptr(), b.data_ptr(), out.data_ptr(), B, C, H, W, md, float(negative_slope),
                                                _stream(a))
            name = "b200_corr2d_fwd_nchw_leaky"
    if rc == _lib.B200_ENOSUP:            # md != 4 or rows TMA cannot address (W % 4 != 0): the NHWC entry takes them
        return None
    check(rc, name)
    return out


def _correlation2d_nchw(input1, input2, max_displacement, negative_slope):
    """The single-pass NCHW route (b200_corr2d_fwd_nchw[_leaky]); None when the call is outside its limits."""
    needs_grad = torch.is_grad_enabled() and (input1.requires_grad or input2.requires_grad)
    md = int(max_displacement)
    if needs_grad or not 1 <= md <= 4 or input1.dim() != 4 or input1.shape != input2.shape:
        return None
    return _corr2d_fwd_nchw(input1.contiguous().float(), input2.contiguous().float(), md, negative_slope)


class Correlation2dNCHWFunction(torch.autograd.Function):
    """correlation2d with a graph: NCHW in, NCHW out, gradients in the inputs' dtypes.

    The forward runs the kernels of the no-grad call (b200_corr2d_fwd_nchw inside its limits, else permute +
    b200_corr2d_fwd), so both forwards are bit-identical.  It saves the caller's NCHW inputs, no copies.  At md = 4 the
    backward reads them as they are (b200_corr2d_bwd_nchw, no permutes); other displacements permute the saved inputs
    for b200_corr2d_bwd, which writes NCHW gradients."""

    @staticmethod
    def forward(ctx, input1, input2, max_displacement):
        _no_fallback("Correlation2dNCHWFunction", input1, input2)
        md = int(max_displacement)
        _require(input1.dim() == 4 and input1.shape == input2.shape, "input1/input2 must both be [B,C,H,W]")
        a, b = input1.contiguous().float(), input2.contiguous().float()
        out = _corr2d_fwd_nchw(a, b, md, None) if 1 <= md <= 4 else None
        if out is None:
            out = _correlation_forward_cuda(a.permute(0, 2, 3, 1).contiguous(), b.permute(0, 2, 3, 1).contiguous(), md)
        ctx.save_for_backward(input1, input2)
        ctx.max_displacement = md
        return out

    @staticmethod
    def backward(ctx, grad_output):
        input1, input2 = ctx.saved_tensors
        md = ctx.max_displacement
        need1, need2 = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        a, b = input1.contiguous().float(), input2.contiguous().float()
        grad_output = grad_output.contiguous().float()
        if md == 4:
            B, C, H, W = a.shape
            _require(tuple(grad_output.shape) == (B, 81, H, W), "grad_output has the wrong shape")
            g1 = torch.empty_like(a) if need1 else None
            g2 = torch.empty_like(b) if need2 else None
            with torch.cuda.device(a.device):
                check(lib.b200_corr2d_bwd_nchw(grad_output.data_ptr(), a.data_ptr(), b.data_ptr(),
                                               g1.data_ptr() if need1 else None, g2.data_ptr() if need2 else None,
                                               B, C, H, W, md, _stream(a)), "b200_corr2d_bwd_nchw")
        else:
            g1, g2 = _correlation_backward_cuda(grad_output, a.permute(0, 2, 3, 1).contiguous(),
                                                b.permute(0, 2, 3, 1).contiguous(), md)
        return (g1.to(input1.dtype) if need1 else None), (g2.to(input2.dtype) if need2 else None), None


def correlation2d(input1, input2, max_displacement, cpp_impl=True):
    """input1, input2 [B,C,H,W] -> [B,(2md+1)^2,H,W] (wrapper.py:55-72). cpp_impl is accepted and ignored.

    Without autograd (inference; the reference evaluates under torch.no_grad) and for md = 4, W % 4 == 0 the cost
    volume is computed straight from the NCHW maps (b200_corr2d_fwd_nchw): the wrapper's two permutes are gone.  When
    autograd needs a graph, Correlation2dNCHWFunction runs the same forward and a backward without permutes.
    Otherwise: permute to NHWC and go through CorrelationFunction exactly as wrapper.py:68-70 does."""
    _no_fallback("correlation2d", input1, input2)
    out = _correlation2d_nchw(input1, input2, max_displacement, None)
    if out is not None:
        return out
    needs_grad = torch.is_grad_enabled() and (input1.requires_grad or input2.requires_grad)
    if needs_grad and input1.dim() == 4 and input1.shape == input2.shape:
        return Correlation2dNCHWFunction.apply(input1, input2, max_displacement)
    input1 = input1.permute(0, 2, 3, 1).contiguous().float()
    input2 = input2.permute(0, 2, 3, 1).contiguous().float()
    return CorrelationFunction.apply(input1, input2, max_displacement)


def correlation2d_leaky(input1, input2, max_displacement, negative_slope=0.1):
    """leaky_relu(correlation2d(input1, input2, md), negative_slope) — the expression of RPEFlow_core.py:362 — with the
    activation as the epilogue of the correlation kernel (SURVEY §8f rank 3).  Outside the single-pass route's limits
    (autograd, md != 4, W % 4 != 0) it is the two-op composition."""
    _no_fallback("correlation2d_leaky", input1, input2)
    if not 0.0 <= float(negative_slope) <= 1.0:
        raise RuntimeError("rpeflow_b200.correlation2d_leaky: negative_slope must be in [0, 1]")
    out = _correlation2d_nchw(input1, input2, max_displacement, negative_slope)
    if out is not None:
        return out
    return torch.nn.functional.leaky_relu(correlation2d(input1, input2, max_displacement), float(negative_slope))


def warp_correlate(feat1_2d, feat2_2d, flow_2d, max_displacement=4, negative_slope=0.1, l2_budget_bytes=48 << 20):
    """RPEFlow_core.py:351+362 as one call: leaky_relu(correlation2d(feat1, backwarp_2d(feat2, flow, 'border'), md), slope).

    The warped map is an intermediate nobody else reads, so the batch is walked in chunks whose warped maps fit the
    L2 budget: each chunk's backwarp output is still L2-resident when the correlation's TMA loads ask for it and the
    map never makes the round trip through HBM.  flow_2d None = the coarsest level (no warp, RPEFlow_core.py:346)."""
    from .projection import backwarp_2d
    _no_fallback("warp_correlate", feat1_2d, feat2_2d)
    if flow_2d is None:
        return correlation2d_leaky(feat1_2d, feat2_2d, max_displacement, negative_slope)
    B = feat1_2d.shape[0]
    per_sample = feat2_2d[0].numel() * 4
    chunk = max(1, min(B, int(l2_budget_bytes // max(per_sample, 1))))
    if chunk >= B:
        return correlation2d_leaky(feat1_2d, backwarp_2d(feat2_2d, flow_2d, "border"), max_displacement, negative_slope)
    outs = []
    for i in range(0, B, chunk):
        warped = backwarp_2d(feat2_2d[i:i + chunk], flow_2d[i:i + chunk], "border")
        outs.append(correlation2d_leaky(feat1_2d[i:i + chunk], warped, max_displacement, negative_slope))
    return torch.cat(outs, dim=0)


def furthest_point_sampling(xyz, n_samples, cpp_impl=True):
    """xyz [B,N,3] -> [B,n_samples] int64 (wrapper.py:75-103)."""
    assert xyz.shape[2] == 3 and xyz.shape[1] > n_samples        # wrapper.py:98
    _no_fallback("furthest_point_sampling", xyz)
    return _furthest_point_sampling_cuda(xyz.contiguous(), n_samples).to(torch.int64)


def k_nearest_neighbor(input_xyz, query_xyz, k, cpp_impl=True):
    """[B,N,D] or [B,D,N] (D<=3, sniffed like wrapper.py:119-122) -> [B,Q,k] int64 (wrapper.py:106-127)."""
    _no_fallback("k_nearest_neighbor", input_xyz, query_xyz)
    if input_xyz.shape[1] <= 3:                          # channel-first: read in place, no transpose().contiguous() passes
        assert query_xyz.shape[1] == input_xyz.shape[1]
        return _k_nearest_neighbor_cuda(input_xyz.contiguous(), query_xyz.contiguous(), k, channel_first=True)
    return _k_nearest_neighbor_cuda(input_xyz.contiguous(), query_xyz.contiguous(), k)


def squared_distance(xyz1, xyz2):
    """[B,N1,D],[B,N2,D] -> [B,N1,N2]; kept for API completeness (wrapper.py:40-52); not on the CUDA hot path."""
    assert xyz1.shape[-1] == xyz2.shape[-1] and xyz1.shape[-1] <= 3
    dist = -2 * torch.matmul(xyz1, xyz2.permute(0, 2, 1))
    dist += torch.sum(xyz1 ** 2, -1).unsqueeze(2)
    dist += torch.sum(xyz2 ** 2, -1).unsqueeze(1)
    return dist
