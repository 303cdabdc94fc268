"""Drop-in for ``models/pointconv.py`` (danqu130/RPEFlow): ``PointConvDownSampling`` (:7-61) and
``PointConvNoSampling`` (:64-122) — SURVEY §8f rank 1.

Both classes keep the reference's constructor and ``state_dict`` keys (``weight_net.convs.{0,1}.conv_fn.{weight,bias}``,
``linear.{weight,bias}``), so released checkpoints load unchanged.  ``forward`` is the cell-grid KNN (b200_knn_grid)
followed by the fused tcgen05 kernel of ``b200_pointconv_fwd``: gathers, weight net, the [16 x k].[k x (C+3)] product,
the Linear layer and the LeakyReLU in one pass, no [B,S,k,*] tensor in memory.

By default the modules are forward-only: ``forward`` refuses to run while gradients are enabled for any input or
parameter that requires them.  ``PointConv*(..., differentiable=True)`` and the functional ``pointconv`` train through
``PointConvFunction`` instead: its forward is ``b200_pointconv_fwd_linear`` (the Linear output, before the activation)
and its backward ``b200_pointconv_bwd`` (gradients of both clouds, the features and the six parameters; only the inputs,
the indices and the weights are kept for it).  Built for the configuration the model uses: ``norm=None``,
``activation='leaky_relu'``, ``k=16``.
"""
import ctypes

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd.function import once_differentiable

from ._lib import PointConvGrads, PointConvWeights, check, lib, require_dense
from .ops import k_nearest_neighbor

__all__ = ["PointConvDownSampling", "PointConvNoSampling", "PointConvFunction", "pointconv", "pointconv_forward",
           "pack_pointconv_weights", "param_weights"]


class _Conv(nn.Module):
    def __init__(self, cin, cout):
        super().__init__()
        self.conv_fn = nn.Conv2d(cin, cout, 1)


class _MLP(nn.Module):
    def __init__(self, cin, widths):
        super().__init__()
        chans = [cin] + list(widths)
        self.convs = nn.ModuleList(_Conv(a, b) for a, b in zip(chans[:-1], chans[1:]))


def pack_pointconv_weights(module):
    """dict name -> contiguous fp32 tensors in the order of b200_pointconv_weights."""
    def wb(conv):
        w = conv.conv_fn.weight
        return w.detach().reshape(w.shape[0], w.shape[1]).contiguous().float(), conv.conv_fn.bias.detach().contiguous().float()
    out = {}
    out["Wa"], out["ba"] = wb(module.weight_net.convs[0])
    out["Wb"], out["bb"] = wb(module.weight_net.convs[1])
    out["L"] = module.linear.weight.detach().contiguous().float()
    out["bias"] = module.linear.bias.detach().contiguous().float()
    return out


def param_weights(module):
    """dict name -> the module's own parameters as [out,in] / [out] views (gradients land on the parameters)."""
    def wb(conv):
        w = conv.conv_fn.weight
        return w.view(w.shape[0], w.shape[1]), conv.conv_fn.bias
    out = {}
    out["Wa"], out["ba"] = wb(module.weight_net.convs[0])
    out["Wb"], out["bb"] = wb(module.weight_net.convs[1])
    out["L"], out["bias"] = module.linear.weight, module.linear.bias
    return out


def _pointconv_run(xyz, features, sampled_xyz, knn, weights, precision, entry):
    """b200_pointconv_fwd (entry "b200_pointconv_fwd") or b200_pointconv_fwd_linear on prepared tensors."""
    B, C, N = features.shape
    S, k = sampled_xyz.shape[2], knn.shape[2]
    cout = weights["L"].shape[0]
    assert tuple(weights["L"].shape) == (cout, 16 * (C + 3)) and tuple(knn.shape) == (B, S, k)
    keep = {n: weights[n].to(xyz.device) for n in PointConvWeights.NAMES}
    w = PointConvWeights(**{n: keep[n].data_ptr() for n in PointConvWeights.NAMES})
    out = torch.empty((B, cout, S), dtype=torch.float32, device=xyz.device)
    scratch = torch.empty((lib.b200_pointconv_scratch_floats(B, C, cout, N),), dtype=torch.float32, device=xyz.device)
    with torch.cuda.device(xyz.device):
        check(getattr(lib, entry)(xyz.data_ptr(), features.data_ptr(), sampled_xyz.data_ptr(), knn.data_ptr(),
                                  ctypes.byref(w), out.data_ptr(), scratch.data_ptr(), B, C, cout, N, S, k,
                                  int(precision), torch.cuda.current_stream(xyz.device).cuda_stream), entry)
    return out


def pointconv_forward(xyz, features, sampled_xyz, knn_indices, weights, precision=2):
    """xyz [B,3,N], features [B,C,N], sampled_xyz [B,3,S], knn_indices [B,S,16] -> [B,out,S]; all CUDA."""
    if not (xyz.is_cuda and features.is_cuda and sampled_xyz.is_cuda):
        raise RuntimeError("rpeflow_b200.pointconv_forward: CUDA tensors required — no CPU/torch fallback")
    xyz, features, sampled_xyz = (t.contiguous().float() for t in (xyz, features, sampled_xyz))
    knn = knn_indices.to(torch.int64).contiguous()
    return _pointconv_run(xyz, features, sampled_xyz, knn, weights, precision, "b200_pointconv_fwd")


class PointConvFunction(torch.autograd.Function):
    """apply(xyz, features, sampled_xyz, knn, precision, *6 weights in PointConvWeights.NAMES order) -> y [B,out,S].

    y is the Linear output, before any norm or activation.  Tensors are CUDA, contiguous fp32 (knn int64 [B,S,16]).
    Forward is b200_pointconv_fwd_linear: LeakyReLU(0.1) of y equals pointconv_forward bit for bit.  Only the inputs,
    the indices and the weights are saved.  Backward is b200_pointconv_bwd; gradients autograd does not ask for are
    not computed.  The gradients of the clouds and the features are summed with float atomics, so this raises under
    torch.use_deterministic_algorithms(True)."""

    @staticmethod
    def forward(ctx, xyz, features, sampled_xyz, knn, precision, *params):
        if torch.are_deterministic_algorithms_enabled():
            raise RuntimeError("rpeflow_b200.pointconv: the backward sums gradients with float atomics and is not "
                               "deterministic; torch.use_deterministic_algorithms(True) is set")
        # a non-contiguous or non-fp32 argument used to be read through its raw pointer: silently wrong y and gradients
        require_dense("PointConvFunction", xyz=xyz, features=features, sampled_xyz=sampled_xyz, knn=knn,
                      **dict(zip(PointConvWeights.NAMES, params)))
        out =_pointconv_run(xyz, features, sampled_xyz, knn, dict(zip(PointConvWeights.NAMES, params)), precision,
                             "b200_pointconv_fwd_linear")
        ctx.save_for_backward(xyz, features, sampled_xyz, knn, *params)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y):
        xyz, features, sampled_xyz, knn, *params = ctx.saved_tensors
        need = ctx.needs_input_grad
        inputs = (xyz, features, sampled_xyz)
        grads_in = [torch.empty_like(t) if need[n] else None for n, t in enumerate(inputs)]
        grads_w = [torch.empty_like(p) if need[5 + n] else None for n, p in enumerate(params)]
        if not any(g is not None for g in grads_in + grads_w):
            return (None,) * (5 + len(params))
        B, C, N = features.shape
        S, k = sampled_xyz.shape[2], knn.shape[2]
        cout = params[4].shape[0]
        grad_y = grad_y.contiguous().float()
        w = PointConvWeights(**{n: p.data_ptr() for n, p in zip(PointConvWeights.NAMES, params)})
        g = PointConvGrads(**{n: (t.data_ptr() if t is not None and t.numel() > 0 else None)
                              for n, t in zip(PointConvGrads.NAMES, grads_in + grads_w)})
        scratch = torch.empty((lib.b200_pointconv_bwd_scratch_floats(B, C, cout, N, S),), dtype=torch.float32,
                              device=xyz.device)
        with torch.cuda.device(xyz.device):
            check(lib.b200_pointconv_bwd(xyz.data_ptr(), features.data_ptr(), sampled_xyz.data_ptr(), knn.data_ptr(),
                                         ctypes.byref(w), grad_y.data_ptr(), ctypes.byref(g), scratch.data_ptr(),
                                         B, C, cout, N, S, k, torch.cuda.current_stream(xyz.device).cuda_stream),
                  "b200_pointconv_bwd")
        return (*grads_in, None, None, *grads_w)


def pointconv(xyz, features, sampled_xyz, knn_indices, weights, precision=2):
    """Differentiable pointconv_forward: LeakyReLU(0.1) of PointConvFunction.  weights = dict name -> [out,in] / [out]
    tensors (param_weights(module) for a module's own parameters).  Gradients flow to xyz, features, sampled_xyz and the
    weights; the forward arithmetic is the one precision selects (1 TF32, 2 3xTF32), the backward is 3xTF32 / fp32."""
    if not (xyz.is_cuda and features.is_cuda and sampled_xyz.is_cuda):
        raise RuntimeError("rpeflow_b200.pointconv: CUDA tensors required — no CPU/torch fallback")
    xyz, features, sampled_xyz = (t.contiguous().float() for t in (xyz, features, sampled_xyz))
    knn = knn_indices.to(torch.int64).contiguous()
    params = [weights[n].contiguous().float() for n in PointConvWeights.NAMES]
    y = PointConvFunction.apply(xyz, features, sampled_xyz, knn, int(precision), *params)
    return F.leaky_relu(y, 0.1)


class _PointConv(nn.Module):
    def __init__(self, in_channels, out_channels, norm=None, activation='leaky_relu', k=16, precision=2,
                 differentiable=False):
        """differentiable=True: under grad, forward trains through PointConvFunction (b200_pointconv_bwd) instead of
        raising."""
        super().__init__()
        if norm is not None or activation != 'leaky_relu':
            raise NotImplementedError("rpeflow_b200 PointConv is built for norm=None, activation='leaky_relu' (what RPEFlow uses)")
        self.k = k
        self.precision = precision
        self.differentiable = differentiable
        self.weight_net = _MLP(3, [8, 16])
        self.linear = nn.Linear(16 * (in_channels + 3), out_channels)

    def _train(self, *tensors):
        """True: run through PointConvFunction; raises when a graph is needed and the module is forward-only."""
        if not (torch.is_grad_enabled() and (any(t.requires_grad for t in tensors) or
                                             any(p.requires_grad for p in self.parameters()))):
            return False
        if self.differentiable:
            return True
        if tensors[1].requires_grad or any(p.requires_grad for p in self.parameters()):
            raise RuntimeError("rpeflow_b200 PointConv is forward-only; run it under torch.no_grad() "
                               "(training keeps models.pointconv)")
        return False


class PointConvDownSampling(_PointConv):
    def forward(self, xyz, features, sampled_xyz):
        """xyz [B,3,N], features [B,C,N], sampled_xyz [B,3,S] -> [B,out,S] (pointconv.py:33-61)."""
        if self._train(xyz, features, sampled_xyz):
            knn = k_nearest_neighbor(xyz.detach(), sampled_xyz.detach(), self.k)
            return pointconv(xyz, features, sampled_xyz, knn, param_weights(self), self.precision)
        knn = k_nearest_neighbor(xyz, sampled_xyz, self.k)                       # pointconv.py:46
        return pointconv_forward(xyz, features, sampled_xyz, knn, pack_pointconv_weights(self), self.precision)


class PointConvNoSampling(_PointConv):
    def forward(self, xyz, features, knn_indices=None):
        """xyz [B,3,N], features [B,C,N], knn_indices [B,N,>=k] or None -> [B,out,N] (pointconv.py:90-122)."""
        train = self._train(xyz, features)
        if knn_indices is not None:
            assert knn_indices.shape[:2] == torch.Size([xyz.shape[0], xyz.shape[2]]) and knn_indices.shape[2] >= self.k
            knn_indices = knn_indices[:, :, :self.k]
        else:
            knn_indices = k_nearest_neighbor(xyz.detach(), xyz.detach(), self.k)   # pointconv.py:107
        if train:                                   # xyz is both clouds: autograd adds the two gradients
            return pointconv(xyz, features, xyz, knn_indices, param_weights(self), self.precision)
        return pointconv_forward(xyz, features, xyz, knn_indices, pack_pointconv_weights(self), self.precision)
