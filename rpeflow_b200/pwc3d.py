"""Drop-in for ``models/pwc3d_core.py::Correlation3D`` (danqu130/RPEFlow, :60-117): the 3-D point cost volume.

``Correlation3D`` below keeps the reference's constructor, parameter tree and ``state_dict`` keys
(``cost_mlp.convs.{0,1}.conv_fn.{weight,bias}``, ``weight_net{1,2}.convs.{0,1,2}.conv_fn.{weight,bias}``) so
released checkpoints load unchanged, and the same ``forward(xyz1, feat1, xyz2, feat2, knn_indices_1in1=None)``.
The whole forward is the fused sm_100a path of ``b200_corr3d_fwd`` (+ ``b200_knn`` for the neighbour search).

By default the module is forward-only: ``forward`` refuses to run while gradients are enabled for any input/parameter
that requires them.  ``Correlation3D(..., differentiable=True)`` and the functional ``correlation3d`` train through
``Correlation3DFunction`` instead, whose backward is ``b200_corr3d_bwd`` (gradients of both clouds, both feature maps
and all 16 parameters; only the inputs, the indices and the forward's per-point ``P`` rows are kept for it), or
``b200_corr3d_bwd_det`` under ``torch.use_deterministic_algorithms(True)``: no float atomics, bit-reproducible.
"""
import ctypes

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from ._lib import B200Error, Corr3dGrads, Corr3dWeights, check, lib, require_dense
from .ops import k_nearest_neighbor

__all__ = ["Correlation3D", "Correlation3DFunction", "correlation3d", "correlation3d_forward", "pack_weights",
           "param_weights", "build_pc_pyramid"]


class _Conv(nn.Module):
    """1x1 Conv2d + activation with the reference's attribute names (models/utils.py:37-64, norm=None)."""

    def __init__(self, cin, cout):
        super().__init__()
        self.conv_fn = nn.Conv2d(cin, cout, 1)


class _MLP(nn.Module):
    """models/utils.py:84-98 (MLP2d): only the parameter container is needed here."""

    def __init__(self, cin, widths):
        super().__init__()
        chans = [cin] + list(widths)
        self.convs = nn.ModuleList(_Conv(a, b) for a, b in zip(chans[:-1], chans[1:]))


def pack_weights(module):
    """dict name -> contiguous fp32 [out,in] / [out] tensors in the order of b200_corr3d_weights."""
    def wb(conv):
        w = conv.conv_fn.weight
        return w.detach().reshape(w.shape[0], w.shape[1]).contiguous().float(), conv.conv_fn.bias.detach().contiguous().float()
    out = {}
    out["W1"], out["b1"] = wb(module.cost_mlp.convs[0])
    out["W2"], out["b2"] = wb(module.cost_mlp.convs[1])
    for tag, net in (("n1", module.weight_net1), ("n2", module.weight_net2)):
        for letter, conv in zip("abc", net.convs):
            out[f"{tag}_W{letter}"], out[f"{tag}_b{letter}"] = wb(conv)
    return out


def param_weights(module):
    """dict name -> the module's own parameters as [out,in] / [out] views (gradients land on the parameters)."""
    def wb(conv):
        w = conv.conv_fn.weight
        return w.view(w.shape[0], w.shape[1]), conv.conv_fn.bias
    out = {}
    out["W1"], out["b1"] = wb(module.cost_mlp.convs[0])
    out["W2"], out["b2"] = wb(module.cost_mlp.convs[1])
    for tag, net in (("n1", module.weight_net1), ("n2", module.weight_net2)):
        for letter, conv in zip("abc", net.convs):
            out[f"{tag}_W{letter}"], out[f"{tag}_b{letter}"] = wb(conv)
    return out


def _corr3d_run(xyz1, feat1, xyz2, feat2, weights, knn12, knn11, precision):
    """b200_corr3d_fwd on prepared tensors (contiguous fp32, int64 indices) -> (out, the scratch it leaves P in)."""
    B, Cin, N1 = feat1.shape
    N2 = feat2.shape[2]
    k = knn12.shape[2]
    Cout = weights["W2"].shape[0]
    assert tuple(weights["W1"].shape) == (Cout, 2 * Cin + 3)
    assert tuple(knn11.shape) == (B, N1, k) and tuple(knn12.shape) == (B, N1, k)
    keep = {n: weights[n].to(xyz1.device) for n in Corr3dWeights.NAMES}
    w = Corr3dWeights(**{n: keep[n].data_ptr() for n in Corr3dWeights.NAMES})
    out = torch.empty((B, Cout, N1), dtype=torch.float32, device=xyz1.device)
    n_scratch = lib.b200_corr3d_scratch_floats(B, Cin, Cout, N1, N2, k)
    scratch = torch.empty((n_scratch,), dtype=torch.float32, device=xyz1.device)
    with torch.cuda.device(xyz1.device):
        check(lib.b200_corr3d_fwd(xyz1.data_ptr(), feat1.data_ptr(), xyz2.data_ptr(), feat2.data_ptr(),
                                  knn12.data_ptr(), knn11.data_ptr(), ctypes.byref(w), out.data_ptr(),
                                  scratch.data_ptr(), B, Cin, Cout, N1, N2, k, int(precision),
                                  torch.cuda.current_stream(xyz1.device).cuda_stream), "b200_corr3d_fwd")
    return out, scratch


def correlation3d_forward(xyz1, feat1, xyz2, feat2, weights, knn12, knn11, precision=2):
    """Functional form: all tensors CUDA fp32; weights = dict from pack_weights(); returns [B,Cout,N1].

    precision: arithmetic of the Cout x Cout cost_mlp layer — 0 = fp32 FFMA, 1 = TF32 tensor cores (tcgen05; what cuDNN
    does for the reference's 1x1 convs under torch's default allow_tf32), 2 = 3xTF32 tensor cores (default; within the
    fp32 path's 1e-4 tolerance).  Shapes the tensor-core kernel does not cover (k != 16, Cout % 32 != 0) run fp32."""
    xyz1, feat1, xyz2, feat2 = (t.contiguous().float() for t in (xyz1, feat1, xyz2, feat2))
    if not xyz1.is_cuda:
        raise RuntimeError("rpeflow_b200.correlation3d_forward: CUDA tensors required — no CPU/torch fallback")
    knn12 = knn12.to(torch.int64).contiguous()
    knn11 = knn11.to(torch.int64).contiguous()
    return _corr3d_run(xyz1, feat1, xyz2, feat2, weights, knn12, knn11, precision)[0]


class Correlation3DFunction(torch.autograd.Function):
    """apply(xyz1, feat1, xyz2, feat2, knn12, knn11, precision, *16 weights in Corr3dWeights.NAMES order).

    Tensors are CUDA, contiguous fp32 (indices int64).  Forward is b200_corr3d_fwd, the same call as
    correlation3d_forward (bit-identical output); its scratch is kept for the backward, which reads P from it.
    Backward is fp32; gradients autograd does not ask for are not computed.  It is b200_corr3d_bwd, which sums
    gradients with float atomics, or, when torch.are_deterministic_algorithms_enabled() is true as the backward runs,
    b200_corr3d_bwd_det: no atomics, every gradient the same bit for bit on every run, and each sample's input gradients
    independent of the rest of the batch (the sum order is stated in include/b200flow.h)."""

    @staticmethod
    def forward(ctx, xyz1, feat1, xyz2, feat2, knn12, knn11, precision, *params):
        # a non-contiguous or non-fp32 argument used to be read through its raw pointer: silently wrong out and gradients
        require_dense("Correlation3DFunction", xyz1=xyz1, feat1=feat1, xyz2=xyz2, feat2=feat2, knn12=knn12, knn11=knn11,
                      **dict(zip(Corr3dWeights.NAMES, params)))
        out, scratch =_corr3d_run(xyz1, feat1, xyz2, feat2, dict(zip(Corr3dWeights.NAMES, params)), knn12, knn11,
                                   precision)
        ctx.save_for_backward(xyz1, feat1, xyz2, feat2, knn12, knn11, scratch, *params)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        xyz1, feat1, xyz2, feat2, knn12, knn11, scratch, *params = ctx.saved_tensors
        need = ctx.needs_input_grad
        inputs = (xyz1, feat1, xyz2, feat2)
        grads_in = [torch.empty_like(t) if need[n] else None for n, t in enumerate(inputs)]
        grads_w = [torch.empty_like(p) if need[7 + n] else None for n, p in enumerate(params)]
        if not any(g is not None for g in grads_in + grads_w):
            return (None,) * (7 + len(params))
        B, Cin, N1 = feat1.shape
        N2 = feat2.shape[2]
        k = knn12.shape[2]
        Cout = params[2].shape[0]
        grad_out = grad_out.contiguous().float()
        w = Corr3dWeights(**{n: p.data_ptr() for n, p in zip(Corr3dWeights.NAMES, params)})
        g = Corr3dGrads(**{n: (t.data_ptr() if t is not None else None)
                           for n, t in zip(Corr3dGrads.NAMES, grads_in + grads_w)})
        with torch.cuda.device(xyz1.device):
            if torch.are_deterministic_algorithms_enabled():
                entry = "b200_corr3d_bwd_det"
                nbytes = lib.b200_corr3d_bwd_det_scratch_bytes(B, Cin, Cout, N1, N2, k)
                if nbytes < 0:
                    raise B200Error(f"b200_corr3d_bwd_det_scratch_bytes failed: {lib.b200_last_error().decode()}")
                bwd_scratch = torch.empty((nbytes,), dtype=torch.uint8, device=xyz1.device)
            else:
                entry = "b200_corr3d_bwd"
                bwd_scratch = torch.empty((lib.b200_corr3d_bwd_scratch_floats(B, Cin, Cout, N1, N2, k),),
                                          dtype=torch.float32, device=xyz1.device)
            check(getattr(lib, entry)(xyz1.data_ptr(), feat1.data_ptr(), xyz2.data_ptr(), feat2.data_ptr(),
                                      knn12.data_ptr(), knn11.data_ptr(), ctypes.byref(w), grad_out.data_ptr(),
                                      scratch.data_ptr(), ctypes.byref(g), bwd_scratch.data_ptr(), B, Cin, Cout, N1, N2, k,
                                      torch.cuda.current_stream(xyz1.device).cuda_stream), entry)
        return (*grads_in, None, None, None, *grads_w)


def correlation3d(xyz1, feat1, xyz2, feat2, weights, knn12, knn11, precision=2):
    """Differentiable correlation3d_forward: weights = dict name -> [out,in] / [out] tensors (param_weights(module)
    for a module's own parameters).  Gradients flow to the clouds, the feature maps and the weights through
    Correlation3DFunction; the forward arithmetic is the one precision selects, the backward is fp32."""
    if not xyz1.is_cuda:
        raise RuntimeError("rpeflow_b200.correlation3d: CUDA tensors required — no CPU/torch fallback")
    xyz1, feat1, xyz2, feat2 = (t.contiguous().float() for t in (xyz1, feat1, xyz2, feat2))
    knn12 = knn12.to(torch.int64).contiguous()
    knn11 = knn11.to(torch.int64).contiguous()
    params = [weights[n].contiguous().float() for n in Corr3dWeights.NAMES]
    return Correlation3DFunction.apply(xyz1, feat1, xyz2, feat2, knn12, knn11, int(precision), *params)


class Correlation3D(nn.Module):
    def __init__(self, in_channels, out_channels, k=16, precision=2, differentiable=False):
        """differentiable=True: under grad, forward trains through Correlation3DFunction (b200_corr3d_bwd) instead of
        raising."""
        super().__init__()
        self.k = k
        self.precision = precision
        self.differentiable = differentiable
        self.cost_mlp = _MLP(3 + 2 * in_channels, [out_channels, out_channels])
        self.weight_net1 = _MLP(3, [8, 8, out_channels])
        self.weight_net2 = _MLP(3, [8, 8, out_channels])

    def forward(self, xyz1, feat1, xyz2, feat2, knn_indices_1in1=None):
        """xyz* [B,3,N], feat* [B,C,N], knn_indices_1in1 [B,N,k] or None -> [B,Cout,N]."""
        if self.differentiable and torch.is_grad_enabled() and (
                any(t.requires_grad for t in (xyz1, feat1, xyz2, feat2)) or any(p.requires_grad for p in self.parameters())):
            knn12 = k_nearest_neighbor(input_xyz=xyz2.detach(), query_xyz=xyz1.detach(), k=self.k)
            if knn_indices_1in1 is None:
                knn_indices_1in1 = k_nearest_neighbor(input_xyz=xyz1.detach(), query_xyz=xyz1.detach(), k=self.k)
            else:
                assert knn_indices_1in1.shape == torch.Size([feat1.shape[0], feat1.shape[2], self.k])
            return correlation3d(xyz1, feat1, xyz2, feat2, param_weights(self), knn12, knn_indices_1in1, self.precision)
        if torch.is_grad_enabled() and (feat1.requires_grad or feat2.requires_grad or
                                        any(p.requires_grad for p in self.parameters())):
            raise RuntimeError("rpeflow_b200.Correlation3D is forward-only; run it under torch.no_grad() "
                               "(training keeps models.pwc3d_core.Correlation3D)")
        knn12 = k_nearest_neighbor(input_xyz=xyz2, query_xyz=xyz1, k=self.k)        # pwc3d_core.py:81
        if knn_indices_1in1 is None:
            knn_indices_1in1 = k_nearest_neighbor(input_xyz=xyz1, query_xyz=xyz1, k=self.k)   # :104
        else:
            assert knn_indices_1in1.shape == torch.Size([feat1.shape[0], feat1.shape[2], self.k])
        return correlation3d_forward(xyz1, feat1, xyz2, feat2, pack_weights(self), knn12, knn_indices_1in1,
                                     self.precision)


def build_pc_pyramid(pc1, pc2, n_samples_list):
    """models/pwc3d_core.py:8-28: one FPS call on cat[pc1,pc2] for max(n_samples_list); levels are prefixes."""
    from .ops import furthest_point_sampling
    from .projection import batch_indexing_channel_first
    batch_size, _, n_points = pc1.shape
    both = torch.cat([pc1, pc2], dim=0)
    picked = furthest_point_sampling(both.transpose(1, 2), max(n_samples_list))
    idx1, idx2 = picked[:batch_size], picked[batch_size:]
    lv0 = torch.arange(n_points, device=pc1.device)[None, :].expand(batch_size, n_points)
    xyzs1, xyzs2, ids1, ids2 = [pc1], [pc2], [lv0], [lv0]
    for n in n_samples_list:
        ids1.append(idx1[:, :n])
        ids2.append(idx2[:, :n])
        xyzs1.append(batch_indexing_channel_first(pc1, idx1[:, :n]))
        xyzs2.append(batch_indexing_channel_first(pc2, idx2[:, :n]))
    return xyzs1, xyzs2, ids1, ids2
