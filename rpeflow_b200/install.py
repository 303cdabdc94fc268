"""Wire the sm_100a kernels into an UNMODIFIED checkout of danqu130/RPEFlow.

    import sys; sys.path.insert(0, "/path/to/RPEFlow")
    import rpeflow_b200.install as b200; b200.install()
    from models.RPEFlow import RPEFlow                          # wrapper.py now finds its three extensions
    ...
    b200.uninstall()                                            # puts every re-bound name back (A/B runs in one process)

What ``install()`` does
1. the three extension modules: before ``models.csrc`` is imported it registers ``models.csrc._correlation_cuda``,
   ``models.csrc._furthest_point_sampling_cuda`` and ``models.csrc._k_nearest_neighbor_cuda`` in ``sys.modules`` (the
   shims in rpeflow_b200/shims), so the byte-for-byte unchanged ``models/csrc/wrapper.py:4-8`` imports them; if
   ``wrapper`` is already imported it sets the four symbols wrapper.py bound at import time instead;
2. (``patch_python=True``) re-binds the pure-python hot ops that have no extension boundary in the reference —
   ``correlation2d`` / ``k_nearest_neighbor`` / ``furthest_point_sampling`` (no permute / transpose passes),
   ``batch_indexing_channel_{first,last}``, ``grid_sample_wrapper``, ``project_feat_with_nn_corr``,
   ``knn_interpolation``, ``backwarp_3d``, ``backwarp_2d``, ``convex_upsample`` (models/utils.py) in every module that
   imported them by name, the ``forward`` of ``Correlation3D`` (models/pwc3d_core.py:69), ``PointConvDownSampling`` /
   ``PointConvNoSampling`` (models/pointconv.py:33,90) and ``CorrFeatureFuser3D`` (RPEFlow_core.py:104: samples the cost
   volume and the two flow channels without building the 83-channel map), and optionally the two voxelisers.

Every re-bound callable decides PER CALL: the CUDA kernel runs only when all tensor arguments are fp32 (or index)
CUDA tensors, autograd does not need a graph through the op, and the arguments are inside what the kernel was
built for; anything else goes to the reference's own function, untouched.  ``stats()`` counts both routes per op.

``install(train=...)`` additionally sends calls that DO need a graph to this library's forward and backward, unless
``torch.use_deterministic_algorithms(True)`` is set and the op's backward sums with float atomics: those go to the
reference.  ``train`` is a collection of op names from ``TRAINABLE``:
- "Correlation3D": ``pwc3d.Correlation3DFunction``, b200_corr3d_fwd / b200_corr3d_bwd.  Under deterministic mode its
  backward is b200_corr3d_bwd_det, which has no atomics, so this one also trains here under deterministic mode;
- "PointConv": ``PointConvDownSampling`` / ``PointConvNoSampling`` through ``pointconv.PointConvFunction``,
  b200_pointconv_fwd_linear / b200_pointconv_bwd, followed by the module's own ``norm_fn`` and ``activation_fn``, so a
  training-mode BatchNorm1d or SyncBatchNorm runs as the reference runs it;
- "knn_interpolation" (it also governs ``backwarp_3d``): ``projection.KnnInterpolationFunction``,
  b200_knn_interpolate / b200_knn_interpolate_bwd;
- "backwarp_2d": ``projection.Backwarp2dFunction``, b200_backwarp2d / b200_backwarp2d_bwd;
- "convex_upsample": ``projection.ConvexUpsampleFunction``, b200_convex_upsample / b200_convex_upsample_bwd.  Its
  backward has no atomics, so this one also trains here under deterministic mode;
- "correlation2d" (lowercase, like the function): ``ops.Correlation2dNCHWFunction``, b200_corr2d_fwd_nchw / b200_corr2d_bwd_nchw on the model's NCHW maps
  with no permutes (other displacements: b200_corr2d_fwd / b200_corr2d_bwd).  No atomics either: it also trains under
  deterministic mode;
- "grid_sample_wrapper": ``projection.GridSampleFunction``, b200_grid_sample_pts / b200_grid_sample_pts_bwd;
- "batch_indexing_channel_first" / "batch_indexing_channel_last": ``projection.BatchIndexingChannelFirstFunction`` /
  ``BatchIndexingChannelLastFunction``, b200_gather_cf / b200_gather_cf_bwd and b200_gather_cl / b200_gather_cl_bwd
  (4-byte data only: gathers of 2-byte data keep going to the reference).
A call takes the train route when it needs a graph, its op is in ``train``, every floating tensor is CUDA fp32 and its
arguments are inside what the kernels were built for; ``stats()`` counts it as "b200".  ``train=True`` means
{"Correlation3D"}.
"""
import importlib
import sys

import torch

from . import events, ops, pointconv, projection, pwc3d
from .shims import _correlation_cuda, _furthest_point_sampling_cuda, _k_nearest_neighbor_cuda

_SHIMS = {
    "models.csrc._correlation_cuda": _correlation_cuda,
    "models.csrc._furthest_point_sampling_cuda": _furthest_point_sampling_cuda,
    "models.csrc._k_nearest_neighbor_cuda": _k_nearest_neighbor_cuda,
}
_MISSING = object()
_SAVED = []            # (object, attribute, previous value) in the order they were replaced
_ADDED_MODULES = []    # sys.modules keys registered by install()
_STATS = {}
_OBSERVER = None
_TRAIN = frozenset()   # ops whose calls that need a graph run this library's autograd Functions (install(train=...))
TRAINABLE = ("Correlation3D", "PointConv", "knn_interpolation", "backwarp_2d", "convex_upsample", "correlation2d",
             "grid_sample_wrapper", "batch_indexing_channel_first", "batch_indexing_channel_last")


def stats(reset=False):
    """{op: {"b200": calls that ran this library's kernels, "reference": calls handed back to the reference}}."""
    out = {k: dict(v) for k, v in _STATS.items()}
    if reset:
        _STATS.clear()
    return out


def set_observer(fn):
    """fn(op_name, args, kwargs, result) after every call that ran a kernel of this library (tests record call sites)."""
    global _OBSERVER
    _OBSERVER = fn


def _count(name, route):
    _STATS.setdefault(name, {"b200": 0, "reference": 0})[route] += 1


def _set(obj, name, value):
    _SAVED.append((obj, name, getattr(obj, name, _MISSING)))
    setattr(obj, name, value)


def _tensors(args, kwargs):
    for a in list(args) + list(kwargs.values()):
        if isinstance(a, torch.Tensor):
            yield a


def _kernel_ok(tensors, float_dtypes=(torch.float32,), graph_ok=False):
    """All CUDA, floating tensors fp32, and (unless graph_ok) no autograd graph needed through the op."""
    need_graph = torch.is_grad_enabled() and not graph_ok
    for t in tensors:
        if not t.is_cuda:
            return False
        if t.is_floating_point():
            if t.dtype not in float_dtypes:
                return False
            if need_graph and t.requires_grad:
                return False
        elif t.dtype == torch.bool or t.is_complex():
            return False
    return True


def _dispatch(name, fast, slow, extra_ok=None, train=None, atomics=True):
    """Per-call choice between this library's kernel (fast) and the reference's own function (slow).  train: the
    TRAINABLE name under which a call that needs a graph may still run fast (whose autograd Function then builds it);
    atomics: that op's backward sums with float atomics, so deterministic mode sends such calls to the reference."""
    def op(*args, **kwargs):
        tensors = list(_tensors(args, kwargs))

        def fits():
            return extra_ok is None or extra_ok(*args, **kwargs)
        if _kernel_ok(tensors) and fits():
            _count(name, "b200")
            out = fast(*args, **kwargs)
            if _OBSERVER is not None:
                _OBSERVER(name, args, kwargs, out)
            return out
        if (train in _TRAIN and _kernel_ok(tensors, graph_ok=True)
                and not (atomics and torch.are_deterministic_algorithms_enabled()) and fits()):
            _count(name, "b200")
            return fast(*args, **kwargs)
        _count(name, "reference")
        return slow(*args, **kwargs)
    op.__name__ = getattr(slow, "__name__", name)
    op.__doc__ = fast.__doc__
    op._b200_reference = slow
    return op


# ------------------------------------------------------------------------------------------ extension level
def register_extension_shims():
    """models.csrc._{correlation,furthest_point_sampling,k_nearest_neighbor}_cuda -> rpeflow_b200/shims.  If the reference's
    wrapper module has already run its import block, the four names it bound are replaced in place."""
    wrapper = sys.modules.get("models.csrc.wrapper")
    for name, mod in _SHIMS.items():
        if sys.modules.get(name) is not mod:
            _SAVED.append((sys.modules, name, sys.modules.get(name, _MISSING)))
            sys.modules[name] = mod
    if wrapper is not None:
        _set(wrapper, "_correlation_forward_cuda", ops._correlation_forward_cuda)
        _set(wrapper, "_correlation_backward_cuda", ops._correlation_backward_cuda)
        _set(wrapper, "_furthest_point_sampling_cuda", ops._furthest_point_sampling_cuda)
        _set(wrapper, "_k_nearest_neighbor_cuda", ops._k_nearest_neighbor_cuda)


# ------------------------------------------------------------------------------------------ module forwards
def _needs_graph(module, *tensors):
    return torch.is_grad_enabled() and (any(t.requires_grad for t in tensors if isinstance(t, torch.Tensor))
                                        or any(p.requires_grad for p in module.parameters()))


def _all_cuda_f32(*tensors):
    return all(t.is_cuda and t.dtype == torch.float32 for t in tensors if isinstance(t, torch.Tensor) and t.is_floating_point())


def _corr3d_forward(self, xyz1, feat1, xyz2, feat2, knn_indices_1in1=None):
    """Correlation3D.forward (pwc3d_core.py:69-117) through b200_corr3d_fwd when no graph is needed."""
    import torch.nn as nn
    plain = all(isinstance(c.norm_fn, nn.Identity) for mlp in (self.cost_mlp, self.weight_net1, self.weight_net2) for c in mlp.convs)
    fits = _all_cuda_f32(xyz1, feat1, xyz2, feat2) and plain and self.k <= 32 and feat1.shape[1] <= 512
    if fits and "Correlation3D" in _TRAIN and _needs_graph(self, xyz1, feat1, xyz2, feat2):
        _count("Correlation3D.forward", "b200")
        knn12 = ops.k_nearest_neighbor(input_xyz=xyz2.detach(), query_xyz=xyz1.detach(), k=self.k)
        if knn_indices_1in1 is None:
            knn_indices_1in1 = ops.k_nearest_neighbor(input_xyz=xyz1.detach(), query_xyz=xyz1.detach(), k=self.k)
        return pwc3d.correlation3d(xyz1, feat1, xyz2, feat2, pwc3d.param_weights(self), knn12, knn_indices_1in1,
                                   getattr(self, "b200_precision", 2))
    if _needs_graph(self, xyz1, feat1, xyz2, feat2) or not fits:
        _count("Correlation3D.forward", "reference")
        return self._b200_reference_forward(xyz1, feat1, xyz2, feat2, knn_indices_1in1)
    _count("Correlation3D.forward", "b200")
    knn12 = ops.k_nearest_neighbor(input_xyz=xyz2, query_xyz=xyz1, k=self.k)
    if knn_indices_1in1 is None:
        knn_indices_1in1 = ops.k_nearest_neighbor(input_xyz=xyz1, query_xyz=xyz1, k=self.k)
    out = pwc3d.correlation3d_forward(xyz1, feat1, xyz2, feat2, pwc3d.pack_weights(self), knn12, knn_indices_1in1,
                                      getattr(self, "b200_precision", 2))
    if _OBSERVER is not None:
        _OBSERVER("k_nearest_neighbor", (xyz2, xyz1, self.k), {}, knn12)
        _OBSERVER("Correlation3D.forward", (xyz1, feat1, xyz2, feat2, knn_indices_1in1), {}, out)
    return out


def _pointconv_body_ok(self):
    """The PointConv body (gathers, weight net, matmul, Linear) is what the kernels were built for: k = 16, at most 256
    output channels, a weight net without norm and with LeakyReLU(0.1)."""
    import torch.nn as nn
    if self.k != 16 or self.linear.out_features > 256:
        return False
    return all(isinstance(c.norm_fn, nn.Identity) and isinstance(c.relu_fn, nn.LeakyReLU)
               and abs(c.relu_fn.negative_slope - 0.1) <= 1e-12 for c in self.weight_net.convs)


def _pointconv_train(self, xyz, tensors):
    """True when this call needs a graph and goes to pointconv.PointConvFunction (install(train={"PointConv", ...}))."""
    return ("PointConv" in _TRAIN and _needs_graph(self, *tensors) and _all_cuda_f32(*tensors)
            and xyz.shape[2] <= 65536 and not torch.are_deterministic_algorithms_enabled() and _pointconv_body_ok(self))


def _pointconv_weights(self):
    """Weights for b200_pointconv_fwd, or None when the module is outside what the kernel was built for: the body of
    _pointconv_body_ok, then the module's own LeakyReLU(0.1), which the kernel applies.  An eval-mode BatchNorm1d after
    the Linear layer (the feature pyramid's norm, conf/test/things.yaml: pwc3d.norm.feature_pyramid) is an affine map per
    output channel and is folded into the Linear weights."""
    import torch.nn as nn
    if not _pointconv_body_ok(self) or not isinstance(self.activation_fn, nn.LeakyReLU) \
            or abs(self.activation_fn.negative_slope - 0.1) > 1e-12:
        return None
    w = pointconv.pack_pointconv_weights(self)
    bn = self.norm_fn
    if isinstance(bn, nn.Identity):
        return w
    if isinstance(bn, nn.BatchNorm1d) and not bn.training and bn.track_running_stats and bn.running_mean is not None:
        scale = torch.rsqrt(bn.running_var.float() + bn.eps)
        shift = -bn.running_mean.float() * scale
        if bn.affine:
            scale = scale * bn.weight.detach().float()
            shift = shift * bn.weight.detach().float() + bn.bias.detach().float()
        w["L"] = (w["L"] * scale[:, None]).contiguous()
        w["bias"] = (w["bias"] * scale + shift).contiguous()
        return w
    return None


def _pointconv_apply(self, xyz, features, sampled_xyz, knn):
    """The Linear output y of the module's PointConv body through pointconv.PointConvFunction (trains the parameters)."""
    w = pointconv.param_weights(self)
    params = [w[n].contiguous() for n in pointconv.PointConvWeights.NAMES]
    return pointconv.PointConvFunction.apply(xyz.contiguous(), features.contiguous(), sampled_xyz.contiguous(),
                                             knn.to(torch.int64).contiguous(), getattr(self, "b200_precision", 2), *params)


def _pointconv_down_forward(self, xyz, features, sampled_xyz):
    if _pointconv_train(self, xyz, (xyz, features, sampled_xyz)):
        _count("PointConvDownSampling.forward", "b200")
        knn = ops.k_nearest_neighbor(xyz.detach(), sampled_xyz.detach(), self.k)
        y = _pointconv_apply(self, xyz, features, sampled_xyz, knn)
        return self.activation_fn(self.norm_fn(y))
    w = None if (_needs_graph(self, xyz, features, sampled_xyz) or not _all_cuda_f32(xyz, features, sampled_xyz)) \
        else _pointconv_weights(self)
    if w is None:
        _count("PointConvDownSampling.forward", "reference")
        return self._b200_reference_forward(xyz, features, sampled_xyz)
    _count("PointConvDownSampling.forward", "b200")
    knn = ops.k_nearest_neighbor(xyz, sampled_xyz, self.k)
    out = pointconv.pointconv_forward(xyz, features, sampled_xyz, knn, w, getattr(self, "b200_precision", 2))
    if _OBSERVER is not None:
        _OBSERVER("k_nearest_neighbor", (xyz, sampled_xyz, self.k), {}, knn)
        _OBSERVER("PointConvDownSampling.forward", (xyz, features, sampled_xyz), {}, out)
    return out


def _pointconv_nosample_forward(self, xyz, features, knn_indices=None):
    if _pointconv_train(self, xyz, (xyz, features)):
        _count("PointConvNoSampling.forward", "b200")
        knn = knn_indices[:, :, :self.k] if knn_indices is not None else \
            ops.k_nearest_neighbor(xyz.detach(), xyz.detach(), self.k)
        y = _pointconv_apply(self, xyz, features, xyz, knn)          # autograd adds the two xyz gradients
        return self.activation_fn(self.norm_fn(y))
    w = None if (_needs_graph(self, xyz, features) or not _all_cuda_f32(xyz, features)) else _pointconv_weights(self)
    if w is None:
        _count("PointConvNoSampling.forward", "reference")
        return self._b200_reference_forward(xyz, features, knn_indices)
    _count("PointConvNoSampling.forward", "b200")
    knn = knn_indices[:, :, :self.k] if knn_indices is not None else ops.k_nearest_neighbor(xyz, xyz, self.k)
    out = pointconv.pointconv_forward(xyz, features, xyz, knn, w, getattr(self, "b200_precision", 2))
    if _OBSERVER is not None:
        _OBSERVER("PointConvNoSampling.forward", (xyz, features, knn), {}, out)
    return out


def _corr_fuser3d_forward(self, xy, feat_corr_2d, feat_corr_3d, efeat_2d, last_flow_3d, last_flow_2d_to_3d):
    """CorrFeatureFuser3D.forward (RPEFlow_core.py:104-120), same arithmetic.  Sampling is per channel, so instead of
    building cat[cost volume, 2 flow channels] (83 x H x W) and sampling that, the cost volume — already sampled at xy by
    CorrFeatureFuser2D's project_feat_with_nn_corr — and the two flow channels are sampled separately and only the small
    [B,83,N] result is concatenated."""
    gs = sys.modules[type(self).__module__].grid_sample_wrapper          # the per-call dispatcher bound by patch_python_ops
    with torch.no_grad():                                                 # the reference samples under no_grad too (:105)
        feat_2d_to_3d = torch.cat([gs(feat_corr_2d, xy), gs(last_flow_2d_to_3d, xy)], dim=1)
        efeat_2d_to_3d = gs(efeat_2d, xy)
        feat_2d_to_3d[:, -2:] -= last_flow_3d[:, :2]
    latent_loss, _, _, _ = self.mi(feat_corr_3d, self.head_2d(feat_2d_to_3d), efeat_2d_to_3d)
    out = self.mlps(torch.cat([feat_2d_to_3d, efeat_2d_to_3d], dim=1))
    out = self.fuse(feat_corr_3d, out)
    return out, latent_loss


def _rebind_forward(cls, fwd):
    if "_b200_reference_forward" not in cls.__dict__:
        _set(cls, "_b200_reference_forward", cls.forward)
        _set(cls, "forward", fwd)


# ------------------------------------------------------------------------------------------ python-level ops
_MODULES = ("models.utils", "models.RPEFlow_core", "models.pwc2d_core", "models.pwc3d_core", "models.pointconv",
            "models.losses3d", "models.RPEFlow", "models.csrc", "models.csrc.wrapper")


def patch_python_ops(patch_events=True, only=None):
    """only: optional set of names (function names as in models/utils.py / wrapper.py, or "Correlation3D", "PointConv",
    "CorrFeatureFuser3D") — re-bind just those (ablations, staged roll-out); None = everything."""
    want = (lambda n: True) if only is None else (lambda n: n in only)
    mutils = importlib.import_module("models.utils")
    wrapper = importlib.import_module("models.csrc.wrapper")
    ref = {n: getattr(mutils, n) for n in ("batch_indexing_channel_first", "batch_indexing_channel_last", "grid_sample_wrapper",
                                           "project_feat_with_nn_corr", "knn_interpolation", "backwarp_3d", "backwarp_2d",
                                           "convex_upsample")}
    ref.update({n: getattr(wrapper, n) for n in ("correlation2d", "k_nearest_neighbor", "furthest_point_sampling")})
    ref = {n: getattr(f, "_b200_reference", f) for n, f in ref.items()}        # idempotent: never wrap a wrapper

    # fast routes and their argument limits, with the reference's own parameter names (call sites use keywords)
    def correlation2d(input1, input2, max_displacement, cpp_impl=True):
        return ops.correlation2d(input1, input2, max_displacement)

    def correlation2d_ok(input1, input2, max_displacement, cpp_impl=True):
        # odd ranks go to the reference wrapper and its torch loop (md > 4 is served by the plain any-displacement kernels)
        return cpp_impl and 1 <= int(max_displacement) <= 64 and input1.dim() == 4 and input1.shape == input2.shape

    def k_nearest_neighbor(input_xyz, query_xyz, k, cpp_impl=True):
        return ops.k_nearest_neighbor(input_xyz, query_xyz, k)

    def k_nearest_neighbor_ok(input_xyz, query_xyz, k, cpp_impl=True):
        if not (cpp_impl and 1 <= int(k) <= 32 and input_xyz.dim() == 3 and query_xyz.dim() == 3):
            return False
        d = input_xyz.shape[1] if input_xyz.shape[1] <= 3 else input_xyz.shape[2]            # wrapper.py:119 layout sniffing
        return d in (2, 3)

    def furthest_point_sampling(xyz, n_samples, cpp_impl=True):
        return ops.furthest_point_sampling(xyz, n_samples)

    def furthest_point_sampling_ok(xyz, n_samples, cpp_impl=True):
        return cpp_impl and xyz.dim() == 3 and xyz.shape[2] == 3 and n_samples < xyz.shape[1]

    def knn_interpolation(input_xyz, input_features, query_xyz, k=3):
        """models/utils.py:140-156: the k-nearest search, then gathers + inverse-distance weights + weighted sum in one kernel."""
        idx = ops.k_nearest_neighbor(input_xyz.detach(), query_xyz.detach(), k)
        if _OBSERVER is not None:
            _OBSERVER("k_nearest_neighbor", (input_xyz, query_xyz, k), {}, idx)
        return projection.knn_interpolation(input_xyz, input_features, query_xyz, k, knn_indices=idx)

    def backwarp_3d(xyz1, xyz2, flow12, k=3):
        """models/utils.py:159-169."""
        return xyz2 + knn_interpolation(xyz1 + flow12, -flow12, xyz2, k)

    def four_byte(batched_data, batched_indices):
        return batched_data.element_size() == 4 and not batched_indices.is_floating_point()

    replaced = {
        "correlation2d": _dispatch("correlation2d", correlation2d, ref["correlation2d"], correlation2d_ok, train="correlation2d",
                                   atomics=False),
        "k_nearest_neighbor": _dispatch("k_nearest_neighbor", k_nearest_neighbor, ref["k_nearest_neighbor"], k_nearest_neighbor_ok),
        "furthest_point_sampling": _dispatch("furthest_point_sampling", furthest_point_sampling, ref["furthest_point_sampling"],
                                             furthest_point_sampling_ok),
        "batch_indexing_channel_first": _dispatch(
            "batch_indexing_channel_first", projection.batch_indexing_channel_first, ref["batch_indexing_channel_first"],
            lambda batched_data, batched_indices: batched_data.dim() == 3 and four_byte(batched_data, batched_indices),
            train="batch_indexing_channel_first"),
        "batch_indexing_channel_last": _dispatch(
            "batch_indexing_channel_last", projection.batch_indexing_channel_last, ref["batch_indexing_channel_last"],
            lambda batched_data, batched_indices: batched_data.dim() in (2, 3) and four_byte(batched_data, batched_indices),
            train="batch_indexing_channel_last"),
        "grid_sample_wrapper": _dispatch("grid_sample_wrapper", projection.grid_sample_wrapper, ref["grid_sample_wrapper"],
                                         train="grid_sample_wrapper"),
        "project_feat_with_nn_corr": _dispatch("project_feat_with_nn_corr", projection.project_feat_with_nn_corr,
                                               ref["project_feat_with_nn_corr"]),
        "knn_interpolation": _dispatch("knn_interpolation", knn_interpolation, ref["knn_interpolation"],
                                       lambda input_xyz, input_features, query_xyz, k=3: k <= 8, train="knn_interpolation"),
        "backwarp_3d": _dispatch("backwarp_3d", backwarp_3d, ref["backwarp_3d"], lambda xyz1, xyz2, flow12, k=3: k <= 8,
                                 train="knn_interpolation"),
        "backwarp_2d": _dispatch("backwarp_2d", projection.backwarp_2d, ref["backwarp_2d"],
                                 lambda x, flow12, padding_mode: padding_mode == "border", train="backwarp_2d"),
        "convex_upsample": _dispatch("convex_upsample", projection.convex_upsample, ref["convex_upsample"],
                                     lambda flow, mask, scale_factor=8: scale_factor in (2, 4, 8) and flow.shape[1] == 2,
                                     train="convex_upsample", atomics=False),
    }
    for modname in _MODULES:
        try:
            mod = importlib.import_module(modname)
        except Exception:
            continue
        for name, fn in replaced.items():
            if hasattr(mod, name) and want(name):
                _set(mod, name, fn)
    if want("PointConv"):
        pcm = importlib.import_module("models.pointconv")
        _rebind_forward(pcm.PointConvDownSampling, _pointconv_down_forward)
        _rebind_forward(pcm.PointConvNoSampling, _pointconv_nosample_forward)
    if want("Correlation3D"):
        core3 = importlib.import_module("models.pwc3d_core")
        _rebind_forward(core3.Correlation3D, _corr3d_forward)
    if want("CorrFeatureFuser3D"):
        try:
            core = importlib.import_module("models.RPEFlow_core")
            _rebind_forward(core.CorrFeatureFuser3D, _corr_fuser3d_forward)
        except Exception:                                # the fuser is an optimisation, not a requirement
            pass
    if patch_events:
        try:
            _set(importlib.import_module("event_utils"), "eventsToVoxel", events.eventsToVoxel)
        except Exception:
            pass
        try:
            dsec = importlib.import_module("dsec")
            _set(dsec.DSECTrain, "eventsToVoxelInter",
                 lambda self, ev, num_bins, height, width, event_polarity=False:
                 events.eventsToVoxelInter(ev, num_bins, height, width, event_polarity))
        except Exception:
            pass


def install(patch_python=True, patch_events=False, only=None, extensions=True, train=False):
    """train: the ops whose calls that need an autograd graph run this library's forward and backward instead of the
    reference's torch code — a collection of names from TRAINABLE ("Correlation3D": pwc3d.Correlation3DFunction;
    "PointConv": pointconv.PointConvFunction under the module's own norm and activation; "knn_interpolation" (with
    backwarp_3d), "backwarp_2d", "convex_upsample", "grid_sample_wrapper", "batch_indexing_channel_first",
    "batch_indexing_channel_last": the projection module's autograd Functions; "correlation2d":
    ops.Correlation2dNCHWFunction).  True means
    {"Correlation3D"}; False (the default) routes every such call to the reference."""
    global _TRAIN
    if isinstance(train, bool):
        names = {"Correlation3D"} if train else set()
    elif isinstance(train, str):
        names = {train}
    else:
        names = set(train)
    unknown = names - set(TRAINABLE)
    if unknown:
        raise ValueError(f"install(train=...): unknown op(s) {sorted(unknown)}; choose from {TRAINABLE}")
    _TRAIN = frozenset(names)
    if extensions:
        register_extension_shims()
    if patch_python:
        patch_python_ops(patch_events=patch_events, only=only)


def uninstall():
    """Undo install(): every replaced attribute and sys.modules entry gets its previous value back."""
    global _TRAIN
    _TRAIN = frozenset()
    while _SAVED:
        obj, name, old = _SAVED.pop()
        if obj is sys.modules:
            if old is _MISSING:
                sys.modules.pop(name, None)
            else:
                sys.modules[name] = old
        elif old is _MISSING:
            try:
                delattr(obj, name)
            except AttributeError:
                pass
        else:
            setattr(obj, name, old)
    wrapper = sys.modules.get("models.csrc.wrapper")       # imported while the shims were registered: unbind its four symbols
    if wrapper is not None:
        for name in ("_correlation_forward_cuda", "_correlation_backward_cuda", "_furthest_point_sampling_cuda",
                     "_k_nearest_neighbor_cuda"):
            if getattr(wrapper, name, None) is getattr(ops, name):
                setattr(wrapper, name, None)
    projection.SAMPLE_MEMO.clear()
