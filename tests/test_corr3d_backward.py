"""Correlation3D backward (b200_corr3d_bwd, pwc3d.Correlation3DFunction, install(train=True)).

CPU: the C-ABI at version 8 agrees with the header, b200_corr3d_bwd rejects bad arguments without touching a device,
and the new entry points refuse CPU tensors.

GPU (-m gpu): all 20 gradients (both clouds, both feature maps, 16 parameters) against fp64 CPU autograd through
oracle.torch_ref.correlation3d with the same knn indices, at max|diff| <= 1e-4 * max|ref| per tensor; gradient subsets;
the training-mode forward equals the no-grad forward bit for bit; a module optimiser step; CUDA-graph capture; and,
when a reference tree is staged, the unmodified RPEFlow with Correlation3D trained through this library.
"""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import rpeflow_b200 as b200
from rpeflow_b200 import _lib, pwc3d
from rpeflow_b200._lib import Corr3dGrads, Corr3dWeights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200flow.h")
DEV = torch.device("cuda", 0)
BAR = 1e-4
GRAD_NAMES = ("xyz1", "feat1", "xyz2", "feat2") + Corr3dWeights.NAMES


# ------------------------------------------------------------------------------------------------- CPU
def test_abi8_header_and_signature_table_agree():
    text = open(HEADER).read()
    declared = sorted(set(re.findall(r"^B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(", text, flags=re.M)))
    assert "b200_corr3d_bwd" in declared and "b200_corr3d_bwd_scratch_floats" in declared
    assert sorted(_lib.SIGNATURES) == declared
    assert _lib.ABI_VERSION == 8 and _lib.lib.b200_abi_version() == 8
    assert "b200_corr3d_grads" in text and len(Corr3dGrads.NAMES) == 20


def _fake_structs():
    one = ctypes.c_void_p(16)              # never dereferenced: argument checks come first
    w = Corr3dWeights(**{n: 16 for n in Corr3dWeights.NAMES})
    g = Corr3dGrads(**{n: 16 for n in Corr3dGrads.NAMES})
    return one, w, g


def test_bwd_rejects_bad_arguments_without_a_gpu():
    lib = _lib.lib
    one, w, g = _fake_structs()
    args = lambda **kw: dict(dict(xyz1=one, scratch=one, B=1, k=16, w=w), **kw)

    def call(xyz1, scratch, B, k, w):
        return lib.b200_corr3d_bwd(xyz1, one, one, one, one, one, ctypes.byref(w) if w is not None else None, one, one,
                                   ctypes.byref(g), scratch, B, 8, 8, 64, 64, k, None)
    assert call(**args(k=33)) == -1 and b"k must be in [1,32]" in lib.b200_last_error()
    assert call(**args(k=0)) == -1
    assert call(**args(xyz1=None)) == -1 and b"null pointer" in lib.b200_last_error()
    assert call(**args(w=None)) == -1
    assert call(**args(scratch=ctypes.c_void_p(20))) == -1 and b"16-byte aligned" in lib.b200_last_error()
    w_null = Corr3dWeights(**{n: 16 for n in Corr3dWeights.NAMES})
    w_null.n2_bc = None
    assert call(**args(w=w_null)) == -1 and b"null weight pointer" in lib.b200_last_error()
    assert lib.b200_corr3d_bwd(one, one, one, one, one, one, ctypes.byref(w), one, one, ctypes.byref(g), one,
                               1, 8, 513, 64, 64, 16, None) == -1
    assert b"exceeds 512" in lib.b200_last_error()
    # B = 0 is a no-op that accepts null data pointers, like the forward
    assert lib.b200_corr3d_bwd(None, None, None, None, None, None, ctypes.byref(w), None, None, ctypes.byref(g), None,
                               0, 8, 8, 64, 64, 16, None) == 0
    assert lib.b200_corr3d_bwd_scratch_floats(2, 32, 32, 100, 100, 16) > lib.b200_corr3d_scratch_floats(2, 32, 32, 100, 100, 16)


def test_new_entry_points_have_no_cpu_fallback():
    x = torch.rand(1, 3, 64)
    f = torch.rand(1, 8, 64, requires_grad=True)
    knn = torch.zeros(1, 64, 4, dtype=torch.int64)
    mod = b200.Correlation3D(8, 8, k=4, differentiable=True)
    with pytest.raises(RuntimeError, match="no CPU"):
        b200.correlation3d(x, f, x, f, pwc3d.param_weights(mod), knn, knn)
    with pytest.raises(RuntimeError, match="no CPU"):
        mod(x, f, x, f)


# ------------------------------------------------------------------------------------------------- GPU helpers
def _cloud(B, N, gen, dup):
    if not dup:
        return torch.rand(B, 3, N, generator=gen)
    base = torch.rand(B, 3, max(1, N // 8), generator=gen)         # every point appears ~8 times
    pick = torch.randint(0, base.shape[2], (B, N), generator=gen)
    return torch.gather(base, 2, pick[:, None, :].expand(B, 3, N)).contiguous()


def _case(B, Cin, Cout, N1, N2, k, seed, dup=False):
    """CPU fp32 inputs, weights of a fresh module, knn indices from this library, and a fixed upstream gradient."""
    gen = torch.Generator().manual_seed(seed)
    xyz1 = _cloud(B, N1, gen, dup)
    xyz2 = (_cloud(B, N2, gen, dup) if N2 != N1 else xyz1 + 0.05 * torch.randn(B, 3, N1, generator=gen))
    f1, f2 = torch.randn(B, Cin, N1, generator=gen), torch.randn(B, Cin, N2, generator=gen)
    torch.manual_seed(seed)
    mod = b200.Correlation3D(Cin, Cout, k=k)
    w = {n: v.clone() for n, v in pwc3d.pack_weights(mod).items()}
    knn12 = b200.k_nearest_neighbor(xyz2.to(DEV), xyz1.to(DEV), k).cpu()
    knn11 = b200.k_nearest_neighbor(xyz1.to(DEV), xyz1.to(DEV), k).cpu()
    grad = torch.randn(B, Cout, N1, generator=gen)
    c = dict(xyz1=xyz1, feat1=f1, xyz2=xyz2, feat2=f2, w=w, knn12=knn12, knn11=knn11, grad=grad, k=k, mod=mod)
    c["grad"] = grad * (~_near_kink_points(c))[:, None, :]
    return c


def _near_kink_points(c, tau=2e-7):
    """[B,N1] bool: query points whose gradient passes through a pre-activation within tau * (that layer's max) of a
    ReLU / LeakyReLU kink in the fp64 forward.  There fp32 and fp64 may pick different slopes, so the gradient is not
    defined to fp32 accuracy; the tests give these points a zero upstream gradient (a handful per case)."""
    import torch.nn.functional as F
    from oracle import torch_ref
    x1, f1, x2, f2 = (c[n].double() for n in ("xyz1", "feat1", "xyz2", "feat2"))
    w = {n: v.double() for n, v in c["w"].items()}
    knn12, knn11 = c["knn12"], c["knn11"]
    B, _, N1 = f1.shape
    k = knn12.shape[2]

    def near(pre):                                      # [B,C,N,k] -> [B,N] rows with a pre-activation close to 0
        return (pre.abs() < tau * pre.abs().max()).any(dim=3).any(dim=1)

    def net(x, tag, flags):
        for letter in "abc":
            x = F.conv2d(x, w[f"{tag}_W{letter}"][:, :, None, None], w[f"{tag}_b{letter}"])
            flags.append(near(x))
            x = F.relu(x)

    d = torch_ref.batch_indexing_channel_first(x2, knn12) - x1.unsqueeze(-1)
    stacked = torch.cat([f1.unsqueeze(-1).expand(-1, -1, -1, k), torch_ref.batch_indexing_channel_first(f2, knn12), d], 1)
    z1 = F.conv2d(stacked, w["W1"][:, :, None, None], w["b1"])
    z2 = F.conv2d(F.leaky_relu(z1, 0.1), w["W2"][:, :, None, None], w["b2"])
    flags1 = [near(z1), near(z2)]
    net(d, "n2", flags1)
    stage1 = torch.stack(flags1).any(dim=0)                                  # [B,N1] points whose P is fragile
    flags2 = []
    net(torch_ref.batch_indexing_channel_first(x1, knn11) - x1.unsqueeze(-1), "n1", flags2)
    via_p = torch.gather(stage1, 1, knn11.reshape(B, -1)).reshape(B, N1, k).any(dim=2)
    return torch.stack(flags2).any(dim=0) | via_p


def _oracle_grads(c):
    """fp64 CPU autograd of the reference op graph (oracle.torch_ref.correlation3d) with the same indices."""
    from oracle import torch_ref
    leaves = {n: c[n].double().requires_grad_(True) for n in ("xyz1", "feat1", "xyz2", "feat2")}
    wts = {n: v.double().requires_grad_(True) for n, v in c["w"].items()}
    out = torch_ref.correlation3d(leaves["xyz1"], leaves["feat1"], leaves["xyz2"], leaves["feat2"], wts, k=c["k"],
                                  knn11=c["knn11"], knn12=c["knn12"])
    out.backward(c["grad"].double())
    got = {n: t.grad for n, t in leaves.items()}
    got.update({n: t.grad for n, t in wts.items()})
    return out.detach(), got


def _gpu_run(c, want=GRAD_NAMES, precision=2):
    leaves = {n: c[n].to(DEV).requires_grad_(n in want) for n in ("xyz1", "feat1", "xyz2", "feat2")}
    wts = {n: v.to(DEV).requires_grad_(n in want) for n, v in c["w"].items()}
    out = b200.correlation3d(leaves["xyz1"], leaves["feat1"], leaves["xyz2"], leaves["feat2"], wts, c["knn12"].to(DEV),
                             c["knn11"].to(DEV), precision)
    out.backward(c["grad"].to(DEV))
    got = {n: t.grad for n, t in leaves.items()}
    got.update({n: t.grad for n, t in wts.items()})
    return out.detach(), got


def _worst(got, ref):
    scale = ref.abs().max().item()
    diff = (got.double().cpu() - ref.double()).abs().max().item()
    return diff / scale if scale > 0 else (0.0 if diff == 0 else float("inf"))


CASES = {
    "C32_N4096": (2, 32, 32, 4096, 4096, 16, False),
    "C64_N2048": (2, 64, 64, 2048, 2048, 16, False),
    "C96_N1024": (2, 96, 96, 1024, 1024, 16, False),
    "C128_N512": (2, 128, 128, 512, 512, 16, False),
    "C192_N256": (2, 192, 192, 256, 256, 16, False),
    "Cin20_Cout36": (2, 20, 36, 300, 300, 16, False),
    "k4": (2, 32, 32, 500, 500, 4, False),
    "N2_below_k": (2, 16, 24, 70, 10, 16, False),
    "duplicates": (2, 32, 32, 512, 512, 16, True),
}


# ------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_all_gradients_vs_fp64_oracle(name):
    c = _case(*CASES[name][:6], seed=len(name), dup=CASES[name][6])
    ref_out, ref = _oracle_grads(c)
    out, got = _gpu_run(c)
    assert _worst(out, ref_out) <= BAR
    ratios = {n: _worst(got[n], ref[n]) / BAR for n in GRAD_NAMES}
    print(f"\n[{name}] worst max|diff| / (1e-4 max|ref|): " + " ".join(f"{n}={r:.3g}" for n, r in ratios.items()))
    bad = {n: r for n, r in ratios.items() if not r <= 1.0}
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("subset", [Corr3dWeights.NAMES, ("feat1", "feat2"), ("xyz2",), ("xyz1",)])
def test_gradient_subsets_match_the_full_run(subset):
    c = _case(2, 32, 40, 600, 600, 16, seed=3)
    _, full = _gpu_run(c)
    _, part = _gpu_run(c, want=subset)
    for n in GRAD_NAMES:
        if n in subset:
            assert part[n] is not None and _worst(part[n], full[n].cpu()) <= BAR, n
        else:
            assert part[n] is None, n


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_training_forward_is_bit_identical_to_no_grad(precision):
    c = _case(2, 64, 64, 2048, 2048, 16, seed=5)
    args = [c[n].to(DEV) for n in ("xyz1", "feat1", "xyz2", "feat2")]
    w = {n: v.to(DEV) for n, v in c["w"].items()}
    knn12, knn11 = c["knn12"].to(DEV), c["knn11"].to(DEV)
    with torch.no_grad():
        plain = pwc3d.correlation3d_forward(*args, w, knn12, knn11, precision)
    leaves = [a.clone().requires_grad_(True) for a in args]
    trained = b200.correlation3d(*leaves, {n: v.clone().requires_grad_(True) for n, v in w.items()}, knn12, knn11, precision)
    assert trained.requires_grad and torch.equal(trained.detach(), plain)


@pytest.mark.gpu
def test_module_optimiser_step_matches_the_oracle_step():
    C, N, k, lr = 48, 700, 16, 0.1
    c = _case(2, C, C, N, N, k, seed=11)
    mod = c["mod"].to(DEV)
    mod_default = b200.Correlation3D(C, C, k=k).to(DEV)
    x1, f1, x2, f2 = (c[n].to(DEV) for n in ("xyz1", "feat1", "xyz2", "feat2"))
    with pytest.raises(RuntimeError):
        mod_default(x1, f1, x2, f2)                         # the default module stays forward-only
    mod.differentiable = True
    params = {n: (v._base if v._base is not None else v) for n, v in pwc3d.param_weights(mod).items()}
    before = {n: p.detach().clone() for n, p in params.items()}
    opt = torch.optim.SGD(mod.parameters(), lr=lr)
    out = mod(x1, f1, x2, f2, c["knn11"].to(DEV))
    (out * c["grad"].to(DEV)).sum().backward()
    opt.step()
    _, ref = _oracle_grads(c)
    for n in Corr3dWeights.NAMES:
        step = (params[n].detach() - before[n]).reshape(ref[n].shape)
        assert _worst(step, -lr * ref[n]) <= BAR, n


@pytest.mark.gpu
def test_cuda_graph_replay_matches_eager_gradients():
    c = _case(2, 64, 64, 1024, 1024, 16, seed=13)
    leaves = {n: c[n].to(DEV).requires_grad_(True) for n in ("xyz1", "feat1", "xyz2", "feat2")}
    wts = {n: v.to(DEV).requires_grad_(True) for n, v in c["w"].items()}
    knn12, knn11, grad = c["knn12"].to(DEV), c["knn11"].to(DEV), c["grad"].to(DEV)
    every = list(leaves.values()) + list(wts.values())

    def step():
        out = b200.correlation3d(leaves["xyz1"], leaves["feat1"], leaves["xyz2"], leaves["feat2"], wts, knn12, knn11)
        out.backward(grad)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            for t in every:
                t.grad = None
            step()
    torch.cuda.current_stream().wait_stream(side)
    eager = [t.grad.clone() for t in every]
    for t in every:
        t.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for t in every:
        t.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    for e, t in zip(eager, every):
        assert _worst(t.grad, e.cpu()) <= BAR


# ------------------------------------------------------------------------------------------------- real model
def _reference_root():
    from refmodel_util import reference_root
    return reference_root()


@pytest.mark.gpu
@pytest.mark.skipif(_reference_root() is None,
                    reason="no reference tree (stage one with `make -C oracle reftree REF=<RPEFlow checkout>`)")
def test_reference_model_gradients_with_correlation3d_trained_here():
    """Unmodified RPEFlow, eval mode, grad enabled, loss = fixed random weighting of flow_2d / flow_3d.  Arm T:
    install(train=True); arm R: install().  The arms differ only in Correlation3D's route."""
    from rpeflow_b200 import refhost
    import rpeflow_b200.install as inst

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    model = refhost.build_rpeflow(_reference_root(), device=DEV, install=False, seed=0)
    inputs = {k: v.to(DEV) for k, v in refhost.synthetic_model_inputs(1, height=256, width=448, n_points=4096, seed=0).items()}
    gen = torch.Generator().manual_seed(0)
    mix = {}

    def arm(train):
        inst.install(train=train)
        inst.stats(reset=True)
        try:
            model.zero_grad(set_to_none=True)
            out = model.forward(inputs, is_Train=False)
            loss = 0.0
            for key in ("flow_2d", "flow_3d"):
                t = out[key][0] if isinstance(out[key], (list, tuple)) else out[key]
                if key not in mix:
                    mix[key] = torch.randn(t.shape, generator=gen).to(DEV)
                loss = loss + (t * mix[key]).sum()
            loss.backward()
            torch.cuda.synchronize()
            grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
            flows = {key: (out[key][0] if isinstance(out[key], (list, tuple)) else out[key]).detach().clone()
                     for key in ("flow_2d", "flow_3d")}
            return flows, grads, inst.stats()
        finally:
            inst.uninstall()

    flows_t, grads_t, st_t = arm(True)
    flows_r, grads_r, st_r = arm(False)
    assert st_t["Correlation3D.forward"] == {"b200": 5, "reference": 0}, st_t["Correlation3D.forward"]
    assert st_r["Correlation3D.forward"] == {"b200": 0, "reference": 5}, st_r["Correlation3D.forward"]
    for key in flows_t:
        assert _worst(flows_t[key], flows_r[key].cpu()) <= 1e-3, key
    assert grads_t.keys() == grads_r.keys() and len(grads_t) > 0
    for n in grads_r:
        assert _worst(grads_t[n], grads_r[n].cpu()) <= 1e-3, n
