"""Drop-in replacements for the reference's gather / projection helpers (models/utils.py of danqu130/RPEFlow).

Same signatures and return shapes as ``batch_indexing_channel_first`` (:119-137), ``batch_indexing_channel_last``
(:101-116), ``grid_sample_wrapper`` (:288-294) and ``project_feat_with_nn_corr`` (:297-317); each is one or two
sm_100a kernels behind include/b200flow.h.  The first three are differentiable like the reference's ``torch.gather``,
advanced indexing and ``F.grid_sample``: when autograd needs a graph they go through
``BatchIndexingChannelFirstFunction``, ``BatchIndexingChannelLastFunction`` and ``GridSampleFunction`` (the same
forward kernel, bit for bit, and b200_gather_cf_bwd / b200_gather_cl_bwd / b200_grid_sample_pts_bwd); otherwise they
run the forward kernel alone.  Their backwards scatter with float atomics and raise under
``torch.use_deterministic_algorithms(True)``.  ``project_feat_with_nn_corr`` is forward only: the reference defines
it under ``torch.no_grad()`` (models/utils.py:297).

The decoder ops ``knn_interpolation`` / ``backwarp_3d`` (:140-169), ``backwarp_2d`` (:186-198) and ``convex_upsample``
(:201-214) also have backwards.  Under ``torch.no_grad()``, or when no input requires grad, they run their forward
kernel alone; when autograd needs a graph they go through ``KnnInterpolationFunction``, ``Backwarp2dFunction`` and
``ConvexUpsampleFunction`` (the same forward kernel, bit for bit, and b200_*_bwd).  The first two sum gradients with
float atomics and raise under ``torch.use_deterministic_algorithms(True)``; convex_upsample's backward is
bit-reproducible and runs there too.
"""
import torch
from torch.autograd.function import once_differentiable

from ._lib import check, lib, require_dense

__all__ = ["batch_indexing_channel_first", "batch_indexing_channel_last", "grid_sample_wrapper", "backwarp_2d", "convex_upsample",
           "project_feat_with_nn_corr", "knn_interpolation", "backwarp_3d", "KnnInterpolationFunction",
           "Backwarp2dFunction", "ConvexUpsampleFunction", "BatchIndexingChannelFirstFunction",
           "BatchIndexingChannelLastFunction", "GridSampleFunction"]


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _require_cuda(what, *tensors):
    if not all(t.is_cuda for t in tensors):
        raise RuntimeError(f"rpeflow_b200.{what}: CUDA tensors required — no CPU/torch fallback")


def _needs_graph(*tensors):
    return torch.is_grad_enabled() and any(t.requires_grad for t in tensors)


def _refuse_nondeterministic(what):
    if torch.are_deterministic_algorithms_enabled():
        raise RuntimeError(f"rpeflow_b200.{what}: the backward sums gradients with float atomics and is not "
                           "deterministic; torch.use_deterministic_algorithms(True) is set")


def _prep_data(data, name):
    if not data.is_cuda:
        raise RuntimeError(f"rpeflow_b200.{name}: CUDA tensors required — no CPU/torch fallback")
    if data.element_size() != 4:
        raise RuntimeError(f"rpeflow_b200.{name}: only 4-byte element types are supported (got {data.dtype})")
    return data.contiguous()


def _prep_idx(idx, device):
    return idx.to(device=device, dtype=torch.int64).contiguous()


# Deliberate deviation from the reference: the gather kernels wrap negative indices once (python / advanced-indexing
# semantics; torch.gather itself raises on them) and CLAMP out-of-range ones instead of raising, because raising needs a
# device-to-host sync per call.  With B200_CHECK_INDICES=1 every gather counts the indices it had to clamp and raises
# IndexError like torch.gather does (one sync per call: a debugging aid for corrupt KNN / FPS outputs, not for production).
import os as _os
CHECK_INDICES = _os.environ.get("B200_CHECK_INDICES", "0") not in ("", "0")


def _bad_counter(device):
    return torch.zeros((1,), dtype=torch.int32, device=device) if CHECK_INDICES else None


def _raise_if_bad(counter, what, n):
    if counter is not None:
        bad = int(counter.item())
        if bad:
            raise IndexError(f"rpeflow_b200.{what}: {bad} indices are out of range for a dimension of size {n}")


def _gather_run(data, idx, channel_last):
    """data [B,C,N] (or [B,N,C] when channel_last), idx [B,I] int64 -> [B,C,I] (or [B,I,C])."""
    B, I = idx.shape
    if channel_last:
        _, N, C = data.shape
        out, fn, what = torch.empty((B, I, C), dtype=data.dtype, device=data.device), lib.b200_gather_cl, "b200_gather_cl"
    else:
        _, C, N = data.shape
        out, fn, what = torch.empty((B, C, I), dtype=data.dtype, device=data.device), lib.b200_gather_cf, "b200_gather_cf"
    bad = _bad_counter(data.device)
    with torch.cuda.device(data.device):
        check(fn(data.data_ptr(), idx.data_ptr(), out.data_ptr(), B, C, N, I, bad.data_ptr() if bad is not None else None,
                 _stream(data)), what)
    _raise_if_bad(bad, "batch_indexing_channel_last" if channel_last else "batch_indexing_channel_first", N)
    return out


def _gather_forward(ctx, data, idx, channel_last):
    what = "BatchIndexingChannelLastFunction" if channel_last else "BatchIndexingChannelFirstFunction"
    _require_cuda(what, data, idx)
    _refuse_nondeterministic("batch_indexing_channel_last" if channel_last else "batch_indexing_channel_first")
    require_dense(what, data=data, idx=idx)
    if data.dim() != 3 or idx.dim() != 2 or idx.shape[0] != data.shape[0]:
        raise ValueError(f"{what}: needs data [B,{'N,C' if channel_last else 'C,N'}] and idx [B,I]")
    ctx.save_for_backward(idx)
    ctx.data_shape = data.shape
    return _gather_run(data, idx, channel_last)


def _gather_backward(ctx, grad_out, channel_last):
    if not ctx.needs_input_grad[0]:
        return None, None
    idx, = ctx.saved_tensors
    B, I = idx.shape
    if channel_last:
        _, N, C = ctx.data_shape
        fn, what = lib.b200_gather_cl_bwd, "b200_gather_cl_bwd"
    else:
        _, C, N = ctx.data_shape
        fn, what = lib.b200_gather_cf_bwd, "b200_gather_cf_bwd"
    g = grad_out.contiguous().float()
    ddata = torch.empty(ctx.data_shape, dtype=torch.float32, device=idx.device)
    with torch.cuda.device(idx.device):
        check(fn(g.data_ptr(), idx.data_ptr(), ddata.data_ptr(), B, C, N, I, _stream(idx)), what)
    return ddata, None


class BatchIndexingChannelFirstFunction(torch.autograd.Function):
    """apply(data [B,C,N], idx [B,I]) -> [B,C,I]; contiguous CUDA fp32 data, int64 indices.  Forward is b200_gather_cf,
    backward b200_gather_cf_bwd: a scatter-add into a zero-filled [B,C,N] at the element each output read (the
    forward's wrap-and-clamp rule).  Only the indices and the data's shape are saved, never the data.  The scatter sums
    with float atomics, so this raises under torch.use_deterministic_algorithms(True)."""

    @staticmethod
    def forward(ctx, data, idx):
        return _gather_forward(ctx, data, idx, False)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        return _gather_backward(ctx, grad_out, False)


class BatchIndexingChannelLastFunction(torch.autograd.Function):
    """apply(data [B,N,C], idx [B,I]) -> [B,I,C]: b200_gather_cl, backward b200_gather_cl_bwd (scatter-add of whole
    rows); otherwise as BatchIndexingChannelFirstFunction."""

    @staticmethod
    def forward(ctx, data, idx):
        return _gather_forward(ctx, data, idx, True)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        return _gather_backward(ctx, grad_out, True)


def _batch_indexing(data, idx, channel_last):
    B = data.shape[0]
    flat_idx = idx.view(B, idx.numel() // max(B, 1))
    if _needs_graph(data):
        fn = BatchIndexingChannelLastFunction if channel_last else BatchIndexingChannelFirstFunction
        return fn.apply(data, flat_idx)
    return _gather_run(data, flat_idx, channel_last)


def batch_indexing_channel_first(batched_data, batched_indices):
    """[B,C,N], [B,I1..Im] -> [B,C,I1..Im] (bit-exact move of 4-byte elements).  Differentiable in the data
    (BatchIndexingChannelFirstFunction) when autograd needs a graph."""
    assert batched_data.shape[0] == batched_indices.shape[0]
    data = _prep_data(batched_data, "batch_indexing_channel_first")
    if data.dim() != 3:
        raise RuntimeError("batch_indexing_channel_first expects data of shape [B,C,N]")
    idx = _prep_idx(batched_indices, data.device)
    B, C, _ = data.shape
    return _batch_indexing(data, idx, False).view([B, C] + list(idx.shape[1:]))


def batch_indexing_channel_last(batched_data, batched_indices):
    """[B,N,C] (or [B,N]), [B,I1..Im] -> [B,I1..Im,C] (or [B,I1..Im]).  Differentiable in the data
    (BatchIndexingChannelLastFunction) when autograd needs a graph."""
    assert batched_data.shape[0] == batched_indices.shape[0]
    data = _prep_data(batched_data, "batch_indexing_channel_last")
    flat = data.dim() == 2
    if flat:
        data = data.unsqueeze(-1)
    if data.dim() != 3:
        raise RuntimeError("batch_indexing_channel_last expects data of shape [B,N,C] or [B,N]")
    idx = _prep_idx(batched_indices, data.device)
    B, _, C = data.shape
    out = _batch_indexing(data, idx, True)
    shape = [B] + list(idx.shape[1:])
    return out.view(shape) if flat else out.view(shape + [C])


class _SampleMemo:
    """Samples that project_feat_with_nn_corr(xy, feat_2d, ...) has already taken: bilinear(feat_2d, xy) as [B,C,N].

    The model samples the same map at the same points twice in four of its five fuser pairs per level — the 3D->2D fuser
    calls project_feat_with_nn_corr(xy, feat_2d, ...) and the 2D->3D fuser then calls grid_sample_wrapper(feat_2d, xy)
    (RPEFlow_core.py:31+53, :80+107, :134+157).  The first call's sampler kernel writes that second result as a by-product
    (b200_project_nn_corr_sampled); it is parked here and handed out ONCE to the next grid_sample_wrapper call with the
    same (map, points).  An entry holds references to both key tensors — their storage cannot be recycled while it is
    parked — and records their version counters, so an in-place write to either one invalidates it.  A handful of
    entries (a level has four pairs in flight) bounds what is kept alive."""

    def __init__(self, capacity=6):
        self.capacity = capacity
        self.entries = []
        self.hits = self.misses = 0

    @staticmethod
    def _key(t):
        return (t.data_ptr(), tuple(t.shape), tuple(t.stride()), t.dtype, t._version)

    def put(self, feat_2d, xy, sampled):
        self.entries.append((feat_2d, self._key(feat_2d), xy, self._key(xy), sampled))
        del self.entries[:-self.capacity]

    def take(self, feat_2d, xy):
        kf, kx = self._key(feat_2d), self._key(xy)
        for i in range(len(self.entries) - 1, -1, -1):
            f, f_key, x, x_key, sampled = self.entries[i]
            if f_key == kf and x_key == kx and self._key(f) == kf and self._key(x) == kx:
                del self.entries[i]
                self.hits += 1
                return sampled
        self.misses += 1
        return None

    def clear(self):
        self.entries.clear()


SAMPLE_MEMO = _SampleMemo()


def _grid_sample_run(feat, pts):
    B, C, H, W = feat.shape
    N = pts.shape[2]
    out = torch.empty((B, C, N), dtype=torch.float32, device=feat.device)
    with torch.cuda.device(feat.device):
        check(lib.b200_grid_sample_pts(feat.data_ptr(), pts.data_ptr(), out.data_ptr(), B, C, H, W, N,
                                       _stream(feat)), "b200_grid_sample_pts")
    return out


class GridSampleFunction(torch.autograd.Function):
    """apply(feat_2d [B,C,H,W], xy [B,2,N]), contiguous CUDA fp32.  Forward is b200_grid_sample_pts, backward
    b200_grid_sample_pts_bwd (ATen's zero-padding gradients; a point with no tap inside the image gets a zero xy
    gradient); gradients autograd does not ask for are not computed.  The map gradient is summed with float atomics,
    so this raises under torch.use_deterministic_algorithms(True)."""

    @staticmethod
    def forward(ctx, feat_2d, xy):
        _require_cuda("GridSampleFunction", feat_2d, xy)
        _refuse_nondeterministic("grid_sample_wrapper")
        require_dense("GridSampleFunction", feat_2d=feat_2d, xy=xy)
        ctx.save_for_backward(feat_2d, xy)
        return _grid_sample_run(feat_2d, xy)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        feat, xy = ctx.saved_tensors
        dfeat = torch.empty_like(feat) if ctx.needs_input_grad[0] else None
        dxy = torch.empty_like(xy) if ctx.needs_input_grad[1] else None
        if dfeat is None and dxy is None:
            return None, None
        B, C, H, W = feat.shape
        N = xy.shape[2]
        g = grad_out.contiguous().float()
        with torch.cuda.device(feat.device):
            check(lib.b200_grid_sample_pts_bwd(feat.data_ptr(), xy.data_ptr(), g.data_ptr(),
                                               dfeat.data_ptr() if dfeat is not None else None,
                                               dxy.data_ptr() if dxy is not None else None, B, C, H, W, N, _stream(feat)),
                  "b200_grid_sample_pts_bwd")
        return dfeat, dxy


def grid_sample_wrapper(feat_2d, xy):
    """feat_2d [B,C,H,W], xy [B,2,N] (pixels) -> [B,C,N]; bilinear, align_corners=True, zero padding.
    Differentiable in both (GridSampleFunction) when autograd needs a graph.  Otherwise, if project_feat_with_nn_corr
    has just sampled this very map at these very points, its result is returned (see _SampleMemo) and no kernel runs;
    a call that needs a graph runs the kernel and leaves that parked result in place."""
    if not (feat_2d.is_cuda and xy.is_cuda):
        raise RuntimeError("rpeflow_b200.grid_sample_wrapper: CUDA tensors required — no CPU/torch fallback")
    if _needs_graph(feat_2d, xy):
        return GridSampleFunction.apply(feat_2d.contiguous().float(), xy.contiguous().float())
    parked = SAMPLE_MEMO.take(feat_2d, xy)
    if parked is not None:
        return parked
    return _grid_sample_run(feat_2d.contiguous().float(), xy.contiguous().float())


def _backwarp2d_run(feat, flow):
    B, C, H, W = feat.shape
    out = torch.empty_like(feat)
    with torch.cuda.device(feat.device):
        check(lib.b200_backwarp2d(feat.data_ptr(), flow.data_ptr(), out.data_ptr(), B, C, H, W, _stream(feat)),
              "b200_backwarp2d")
    return out


class Backwarp2dFunction(torch.autograd.Function):
    """apply(x [B,C,H,W], flow [B,2,H,W]), contiguous CUDA fp32.  Forward is b200_backwarp2d (border padding), backward
    b200_backwarp2d_bwd; gradients autograd does not ask for are not computed.  dx is summed with float atomics, so
    this raises under torch.use_deterministic_algorithms(True)."""

    @staticmethod
    def forward(ctx, x, flow):
        _require_cuda("Backwarp2dFunction", x, flow)
        _refuse_nondeterministic("backwarp_2d")
        require_dense("Backwarp2dFunction", x=x, flow=flow)
        ctx.save_for_backward(x, flow)
        return _backwarp2d_run(x, flow)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        x, flow = ctx.saved_tensors
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dflow = torch.empty_like(flow) if ctx.needs_input_grad[1] else None
        if dx is None and dflow is None:
            return None, None
        B, C, H, W = x.shape
        g = grad_out.contiguous().float()
        with torch.cuda.device(x.device):
            check(lib.b200_backwarp2d_bwd(x.data_ptr(), flow.data_ptr(), g.data_ptr(),
                                          dx.data_ptr() if dx is not None else None,
                                          dflow.data_ptr() if dflow is not None else None, B, C, H, W, _stream(x)),
                  "b200_backwarp2d_bwd")
        return dx, dflow


def backwarp_2d(x, flow12, padding_mode="border"):
    """x [B,C,H,W], flow12 [B,2,H,W] -> x sampled at (pixel + flow), bilinear, align_corners=True (models/utils.py:186-198).
    The model only ever passes padding_mode='border' (RPEFlow_core.py:351); other modes are not built.  Differentiable
    in x and flow12 (Backwarp2dFunction) when autograd needs a graph."""
    _require_cuda("backwarp_2d", x, flow12)
    if padding_mode != "border":
        raise RuntimeError("rpeflow_b200.backwarp_2d: only padding_mode='border' is built (the mode RPEFlow uses)")
    assert x.shape[-2:] == flow12.shape[-2:]                       # models/utils.py:193
    feat = x.contiguous().float()
    flow = flow12.contiguous().float()
    if _needs_graph(feat, flow):
        return Backwarp2dFunction.apply(feat, flow)
    return _backwarp2d_run(feat, flow)


def _convex_upsample_run(f, m, s):
    B, _, H, W = f.shape
    out = torch.empty((B, 2, H * s, W * s), dtype=torch.float32, device=f.device)
    with torch.cuda.device(f.device):
        check(lib.b200_convex_upsample(f.data_ptr(), m.data_ptr(), out.data_ptr(), B, H, W, s, _stream(f)),
              "b200_convex_upsample")
    return out


class ConvexUpsampleFunction(torch.autograd.Function):
    """apply(flow [B,2,H,W], mask [B,9*s*s,H,W], s), contiguous CUDA fp32.  Forward is b200_convex_upsample, backward
    b200_convex_upsample_bwd: two fixed-order passes without atomics, so the gradients are bit-reproducible and the
    op runs under torch.use_deterministic_algorithms(True)."""

    @staticmethod
    def forward(ctx, flow, mask, s):
        _require_cuda("ConvexUpsampleFunction", flow, mask)
        require_dense("ConvexUpsampleFunction", flow=flow, mask=mask)
        ctx.save_for_backward(flow, mask)
        ctx.s = s
        return _convex_upsample_run(flow, mask, s)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        flow, mask = ctx.saved_tensors
        s = ctx.s
        dflow = torch.empty_like(flow) if ctx.needs_input_grad[0] else None
        dmask = torch.empty_like(mask) if ctx.needs_input_grad[1] else None
        if dflow is None and dmask is None:
            return None, None, None
        B, _, H, W = flow.shape
        g = grad_out.contiguous().float()
        if g.data_ptr() % 16:                                        # the kernel reads grad_out with 16-byte loads
            g = g.clone()
        scratch = torch.empty((max(1, lib.b200_convex_upsample_bwd_scratch_floats(B, H, W, s)),), dtype=torch.float32,
                              device=flow.device) if dflow is not None else None
        with torch.cuda.device(flow.device):
            check(lib.b200_convex_upsample_bwd(flow.data_ptr(), mask.data_ptr(), g.data_ptr(),
                                               dflow.data_ptr() if dflow is not None else None,
                                               dmask.data_ptr() if dmask is not None else None,
                                               scratch.data_ptr() if scratch is not None else None, B, H, W, s,
                                               _stream(flow)), "b200_convex_upsample_bwd")
        return dflow, dmask, None


def convex_upsample(flow, mask, scale_factor=8):
    """flow [B,2,H,W], mask [B,9*s*s,H,W] -> [B,2,s*H,s*W]: convex combination of the 3x3 neighbourhood with softmax
    weights (models/utils.py:201-214).  Differentiable in flow and mask (ConvexUpsampleFunction) when autograd needs a
    graph."""
    _require_cuda("convex_upsample", flow, mask)
    s = int(scale_factor)
    B, C, H, W = flow.shape
    if C != 2 or s not in (2, 4, 8) or tuple(mask.shape) != (B, 9 * s * s, H, W):
        raise RuntimeError("rpeflow_b200.convex_upsample: needs flow [B,2,H,W], mask [B,9*s*s,H,W], s in {2,4,8}")
    f, m = flow.contiguous().float(), mask.contiguous().float()
    if _needs_graph(f, m):
        return ConvexUpsampleFunction.apply(f, m, s)
    return _convex_upsample_run(f, m, s)


@torch.no_grad()
def project_feat_with_nn_corr(xy, feat_2d, feat_3d, nn_indices=None, keep_samples=True):
    """xy [B,2,N], feat_2d [B,C2,H,W], feat_3d [B,C3,N], nn_indices [B,H*W] -> [B,C3+3,H,W].
    keep_samples: also keep bilinear(feat_2d, xy) as [B,C2,N] for the grid_sample_wrapper(feat_2d, xy) call that
    follows in the model (one extra 4*C2*N-byte write instead of a second pass over the map)."""
    if not (xy.is_cuda and feat_2d.is_cuda and feat_3d.is_cuda):
        raise RuntimeError("rpeflow_b200.project_feat_with_nn_corr: CUDA tensors required — no CPU/torch fallback")
    f2 = feat_2d.contiguous().float()
    f3 = feat_3d.contiguous().float()
    pts = xy.contiguous().float()
    B, C2, H, W = f2.shape
    C3, N = f3.shape[1], f3.shape[2]
    if nn_indices is None:                              # models/utils.py:304-305: nearest projected point per pixel
        from .ops import k_nearest_neighbor
        ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float32, device=f2.device),
                                torch.arange(W, dtype=torch.float32, device=f2.device), indexing="ij")
        grid = torch.stack([xs, ys], 0).reshape(1, 2, H * W).expand(B, 2, H * W)
        nn_indices = k_nearest_neighbor(pts, grid, k=1)[..., 0]
    else:
        assert tuple(nn_indices.shape) == (B, H * W)
    nn = _prep_idx(nn_indices, f2.device)
    out = torch.empty((B, C3 + 3, H, W), dtype=torch.float32, device=f2.device)
    scratch = torch.empty((max(1, lib.b200_project_nn_corr_scratch_floats(B, C2, C3, N)),), dtype=torch.float32, device=f2.device)
    sampled = torch.empty((B, C2, N), dtype=torch.float32, device=f2.device) if keep_samples else None
    with torch.cuda.device(f2.device):
        check(lib.b200_project_nn_corr_sampled(pts.data_ptr(), f2.data_ptr(), f3.data_ptr(), nn.data_ptr(), out.data_ptr(),
                                               scratch.data_ptr(), sampled.data_ptr() if keep_samples else None,
                                               B, C2, C3, H, W, N, _stream(f2)), "b200_project_nn_corr")
    if keep_samples:
        SAMPLE_MEMO.put(feat_2d, xy, sampled)
    return out


def _knn_interpolate_run(xin, feat, xq, idx):
    B, C, M = feat.shape
    Q, k = xq.shape[2], idx.shape[2]
    out = torch.empty((B, C, Q), dtype=torch.float32, device=xin.device)
    with torch.cuda.device(xin.device):
        check(lib.b200_knn_interpolate(xin.data_ptr(), feat.data_ptr(), xq.data_ptr(), idx.data_ptr(), out.data_ptr(),
                                       B, C, M, Q, k, _stream(xin)), "b200_knn_interpolate")
    return out


class KnnInterpolationFunction(torch.autograd.Function):
    """apply(input_xyz [B,3,M], input_feat [B,C,M], query_xyz [B,3,Q], knn_idx [B,Q,k] int64), contiguous CUDA fp32.
    Forward is b200_knn_interpolate, backward b200_knn_interpolate_bwd (gradients of all three point tensors; those
    autograd does not ask for are not computed).  The input gradients are summed with float atomics, so this raises
    under torch.use_deterministic_algorithms(True)."""

    @staticmethod
    def forward(ctx, input_xyz, input_feat, query_xyz, knn_idx):
        _require_cuda("KnnInterpolationFunction", input_xyz, input_feat, query_xyz, knn_idx)
        _refuse_nondeterministic("knn_interpolation")
        require_dense("KnnInterpolationFunction", input_xyz=input_xyz, input_feat=input_feat, query_xyz=query_xyz,
                      knn_idx=knn_idx)
        ctx.save_for_backward(input_xyz, input_feat, query_xyz, knn_idx)
        return _knn_interpolate_run(input_xyz, input_feat, query_xyz, knn_idx)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        xin, feat, xq, idx = ctx.saved_tensors
        need = ctx.needs_input_grad
        grads = [torch.empty_like(t) if need[n] else None for n, t in enumerate((xin, feat, xq))]
        if all(g is None for g in grads):
            return None, None, None, None
        B, C, M = feat.shape
        Q, k = xq.shape[2], idx.shape[2]
        g = grad_out.contiguous().float()
        ptr = [t.data_ptr() if t is not None else None for t in grads]
        with torch.cuda.device(xin.device):
            check(lib.b200_knn_interpolate_bwd(xin.data_ptr(), feat.data_ptr(), xq.data_ptr(), idx.data_ptr(),
                                               g.data_ptr(), *ptr, B, C, M, Q, k, _stream(xin)),
                  "b200_knn_interpolate_bwd")
        return (*grads, None)


def knn_interpolation(input_xyz, input_features, query_xyz, k=3, knn_indices=None):
    """input_xyz [B,3,M], input_features [B,C,M], query_xyz [B,3,Q] -> [B,C,Q] (models/utils.py:140-156): the k-nearest
    search (cell-grid KNN) followed by ONE kernel for gathers + inverse-distance weights + weighted sum.
    Differentiable in all three point tensors (KnnInterpolationFunction) when autograd needs a graph; the neighbour
    search itself carries no gradient, as in the reference."""
    _require_cuda("knn_interpolation", input_xyz, input_features, query_xyz)
    from .ops import k_nearest_neighbor
    xin, feat, xq = (t.contiguous().float() for t in (input_xyz, input_features, query_xyz))
    if knn_indices is None:
        knn_indices = k_nearest_neighbor(xin.detach(), xq.detach(), k)        # [B,Q,k]
    idx = _prep_idx(knn_indices, xin.device)
    B, C, M = feat.shape
    Q = xq.shape[2]
    assert tuple(idx.shape) == (B, Q, k) and xin.shape == (B, 3, M)
    if _needs_graph(xin, feat, xq):
        return KnnInterpolationFunction.apply(xin, feat, xq, idx)
    return _knn_interpolate_run(xin, feat, xq, idx)


def backwarp_3d(xyz1, xyz2, flow12, k=3):
    """models/utils.py:159-169: xyz2 + interpolation of -flow12 from the warped cloud xyz1 + flow12.  Differentiable in
    all three (autograd composes KnnInterpolationFunction with the add and the negation)."""
    return xyz2 + knn_interpolation(xyz1 + flow12, -flow12, xyz2, k)
