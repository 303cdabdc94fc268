"""PointConv backward (b200_pointconv_fwd_linear, b200_pointconv_bwd, pointconv.PointConvFunction,
install(train={"PointConv", ...})).

CPU: the new C-ABI entries agree with the header at ABI 8, reject bad arguments without touching a device, and the new
Python entry points refuse CPU tensors; the default modules still refuse to run under grad.

GPU (-m gpu): all nine gradients (xyz, features, sampled_xyz, Wa, ba, Wb, bb, L, bias) against fp64 CPU autograd of
oracle.torch_ref.pointconv's Linear output with the same knn indices, at max|diff| <= 1e-4 * max|ref| per tensor;
gradient subsets; the training forward against b200_pointconv_fwd bit for bit; a module optimiser step; CUDA-graph
capture; BatchNorm1d (training mode) composed after the body; deterministic mode; and, when a reference tree is staged,
the unmodified RPEFlow with its 20 PointConv bodies and 5 cost volumes trained through this library.
"""
import ctypes
import os
import re

import pytest
import torch
import torch.nn.functional as F

import rpeflow_b200 as b200
from rpeflow_b200 import _lib, pointconv
from rpeflow_b200._lib import PointConvGrads, PointConvWeights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200flow.h")
DEV = torch.device("cuda", 0)
BAR = 1e-4
INPUTS = ("xyz", "feat", "sampled_xyz")
GRAD_NAMES = INPUTS + PointConvWeights.NAMES


# ------------------------------------------------------------------------------------------------- CPU
def test_new_symbols_in_header_and_signature_table_at_abi8():
    text = open(HEADER).read()
    declared = sorted(set(re.findall(r"^B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(", text, flags=re.M)))
    for name in ("b200_pointconv_fwd_linear", "b200_pointconv_bwd", "b200_pointconv_bwd_scratch_floats"):
        assert name in declared and name in _lib.SIGNATURES
    assert sorted(_lib.SIGNATURES) == declared
    assert _lib.ABI_VERSION == 8 and _lib.lib.b200_abi_version() == 8
    assert "b200_pointconv_grads" in text and len(PointConvGrads.NAMES) == 9


def _fake():
    one = ctypes.c_void_p(16)              # never dereferenced: argument checks come first
    w = PointConvWeights(**{n: 16 for n in PointConvWeights.NAMES})
    g = PointConvGrads(**{n: 16 for n in PointConvGrads.NAMES})
    return one, w, g


def test_bwd_rejects_bad_arguments_without_a_gpu():
    lib = _lib.lib
    one, w, g = _fake()

    def call(xyz=one, scratch=one, w=w, B=1, C=8, Cout=32, N=64, S=32, k=16):
        return lib.b200_pointconv_bwd(xyz, one, one, one, ctypes.byref(w) if w is not None else None, one, ctypes.byref(g),
                                      scratch, B, C, Cout, N, S, k, None)
    assert call(k=8) == -3 and b"k = 16" in lib.b200_last_error()
    assert call(Cout=257) == -3
    assert call(N=65537) == -3
    assert call(xyz=None) == -1 and b"null pointer" in lib.b200_last_error()
    assert call(w=None) == -1
    w_null = PointConvWeights(**{n: 16 for n in PointConvWeights.NAMES})
    w_null.bias = None
    assert call(w=w_null) == -1 and b"null weight pointer" in lib.b200_last_error()
    assert call(scratch=ctypes.c_void_p(20)) == -1 and b"16-byte aligned" in lib.b200_last_error()
    assert call(Cout=0) == -1
    # B = 0 is a no-op that accepts null data pointers
    assert lib.b200_pointconv_bwd(None, None, None, None, ctypes.byref(w), None, ctypes.byref(g), None,
                                  0, 8, 32, 64, 32, 16, None) == 0
    assert lib.b200_pointconv_bwd_scratch_floats(2, 32, 32, 4096, 2048) > 0


def test_fwd_linear_rejects_bad_arguments_without_a_gpu():
    lib = _lib.lib
    one, w, _ = _fake()

    def call(xyz=one, scratch=one, B=1, Cout=32, N=64, k=16):
        return lib.b200_pointconv_fwd_linear(xyz, one, one, one, ctypes.byref(w), one, scratch, B, 8, Cout, N, 32, k, 2, None)
    assert call(k=8) == -3
    assert call(Cout=257) == -3
    assert call(N=65537) == -3
    assert call(xyz=None) == -1
    assert call(scratch=ctypes.c_void_p(20)) == -1
    assert lib.b200_pointconv_fwd_linear(None, None, None, None, ctypes.byref(w), None, None, 0, 8, 32, 64, 32, 16, 2, None) == 0


def test_new_entry_points_have_no_cpu_fallback():
    x = torch.rand(1, 3, 64)
    f = torch.rand(1, 8, 64, requires_grad=True)
    knn = torch.zeros(1, 64, 16, dtype=torch.int64)
    mod = b200.PointConvNoSampling(8, 16, differentiable=True)
    with pytest.raises(RuntimeError, match="no CPU"):
        pointconv.pointconv(x, f, x, knn, pointconv.param_weights(mod))
    with pytest.raises(RuntimeError, match="no CPU"):
        mod(x, f, knn)


def test_default_modules_still_raise_under_grad():
    x = torch.rand(1, 3, 64)
    f = torch.rand(1, 8, 64)
    with pytest.raises(RuntimeError, match="forward-only"):
        b200.PointConvDownSampling(8, 16)(x, f, x[:, :, :32])
    with pytest.raises(RuntimeError, match="forward-only"):
        b200.PointConvNoSampling(8, 16)(x, f)


def test_install_train_rejects_unknown_op_names():
    import rpeflow_b200.install as inst
    with pytest.raises(ValueError, match="unknown op"):
        inst.install(train={"PointConv", "Correlation2D"})


class _UpstreamConv(torch.nn.Module):
    def __init__(self, cin, cout, slope):
        super().__init__()
        self.conv_fn, self.norm_fn, self.relu_fn = torch.nn.Conv2d(cin, cout, 1), torch.nn.Identity(), torch.nn.LeakyReLU(slope)


class _UpstreamPointConv(torch.nn.Module):
    """The attributes install reads from models/pointconv.py's PointConvDownSampling / PointConvNoSampling."""
    def __init__(self, C, Cout, weight_net_slope):
        super().__init__()
        self.k = 16
        self.weight_net = torch.nn.Module()
        self.weight_net.convs = torch.nn.ModuleList([_UpstreamConv(3, 8, weight_net_slope), _UpstreamConv(8, 16, weight_net_slope)])
        self.linear = torch.nn.Linear(16 * (C + 3), Cout)
        self.norm_fn, self.activation_fn = torch.nn.Identity(), torch.nn.LeakyReLU(0.1)


@pytest.mark.parametrize("slope,accepted", [(0.1, True), (0.2, False)])
def test_install_takes_only_the_kernels_weight_net_slope(slope, accepted):
    """The kernels apply LeakyReLU(0.1) inside the weight net: a module whose weight net uses another slope is refused by
    the inference route (_pointconv_weights) and the training route (_pointconv_body_ok) alike, so it runs the reference."""
    import rpeflow_b200.install as inst
    mod = _UpstreamPointConv(8, 32, slope)
    assert inst._pointconv_body_ok(mod) is accepted
    assert (inst._pointconv_weights(mod) is not None) is accepted


# ------------------------------------------------------------------------------------------------- GPU helpers
def _cloud(B, N, gen, dup):
    if not dup:
        return torch.rand(B, 3, N, generator=gen)
    base = torch.rand(B, 3, max(1, N // 8), generator=gen)         # every point appears ~8 times
    pick = torch.randint(0, base.shape[2], (B, N), generator=gen)
    return torch.gather(base, 2, pick[:, None, :].expand(B, 3, N)).contiguous()


def _case(B, C, Cout, N, S, seed, dup=False, nosample=False):
    """CPU fp32 inputs, the weights of a fresh module, knn indices from this library and a fixed upstream gradient.
    nosample: sampled_xyz is xyz itself (PointConvNoSampling)."""
    gen = torch.Generator().manual_seed(seed)
    xyz = _cloud(B, N, gen, dup)
    feat = torch.randn(B, C, N, generator=gen)
    sampled = xyz if nosample else xyz[:, :, torch.randperm(N, generator=gen)[:S]].contiguous()
    torch.manual_seed(seed)
    mod = b200.PointConvDownSampling(C, Cout)
    w = {n: v.clone() for n, v in pointconv.pack_pointconv_weights(mod).items()}
    knn = b200.k_nearest_neighbor(xyz.to(DEV), sampled.to(DEV), 16).cpu()
    grad = torch.randn(B, Cout, sampled.shape[2], generator=gen)
    c = dict(xyz=xyz, feat=feat, sampled_xyz=sampled, w=w, knn=knn, grad=grad, nosample=nosample, mod=mod)
    c["grad"] = grad * (~_near_kink_points(c))[:, None, :]
    return c


def _near_kink_points(c, tau=2e-7):
    """[B,S] bool: sampled points with a weight-net pre-activation within tau * (that layer's max) of the LeakyReLU
    kink in the fp64 forward.  There fp32 and fp64 may pick different slopes, so the gradient is not defined to fp32
    accuracy; the tests give these points a zero upstream gradient."""
    from oracle import torch_ref
    xyz, sampled = c["xyz"].double(), c["sampled_xyz"].double()
    w = {n: v.double() for n, v in c["w"].items()}
    rel = torch_ref.batch_indexing_channel_first(xyz, c["knn"]) - sampled[:, :, :, None]           # [B,3,S,k]
    z1 = F.conv2d(rel, w["Wa"][:, :, None, None], w["ba"])
    z2 = F.conv2d(F.leaky_relu(z1, 0.1), w["Wb"][:, :, None, None], w["bb"])
    near = lambda z: (z.abs() < tau * z.abs().max()).any(dim=3).any(dim=1)
    return near(z1) | near(z2)


def _oracle(c, post=False):
    """fp64 CPU autograd of oracle.torch_ref.pointconv with the same indices: the Linear output y (the oracle's
    LeakyReLU inverted) or, with post=True, the oracle's own output; returns (output, gradients)."""
    from oracle import torch_ref
    xyz = c["xyz"].double().requires_grad_(True)
    leaves = {"xyz": xyz, "feat": c["feat"].double().requires_grad_(True)}
    leaves["sampled_xyz"] = xyz if c["nosample"] else c["sampled_xyz"].double().requires_grad_(True)
    wts = {n: v.double().requires_grad_(True) for n, v in c["w"].items()}
    out = torch_ref.pointconv(leaves["xyz"], leaves["feat"], leaves["sampled_xyz"], wts, k=16, knn=c["knn"])
    if not post:
        out = torch.where(out > 0, out, out * 10.0)
    out.backward(c["grad"].double())
    got = {n: (t.grad if not (c["nosample"] and n == "sampled_xyz") else None) for n, t in leaves.items()}
    got.update({n: t.grad for n, t in wts.items()})
    return out.detach(), got


def _gpu_leaves(c, want=GRAD_NAMES):
    xyz = c["xyz"].to(DEV).requires_grad_("xyz" in want)
    leaves = {"xyz": xyz, "feat": c["feat"].to(DEV).requires_grad_("feat" in want)}
    leaves["sampled_xyz"] = xyz if c["nosample"] else c["sampled_xyz"].to(DEV).requires_grad_("sampled_xyz" in want)
    wts = {n: v.to(DEV).requires_grad_(n in want) for n, v in c["w"].items()}
    return leaves, wts


def _linear(leaves, wts, knn, precision=2):
    params = [wts[n] for n in PointConvWeights.NAMES]
    return pointconv.PointConvFunction.apply(leaves["xyz"], leaves["feat"], leaves["sampled_xyz"], knn, precision, *params)


def _gpu_run(c, want=GRAD_NAMES, precision=2):
    leaves, wts = _gpu_leaves(c, want)
    out = _linear(leaves, wts, c["knn"].to(DEV), precision)
    out.backward(c["grad"].to(DEV))
    got = {n: t.grad for n, t in leaves.items()}
    if c["nosample"]:
        got["sampled_xyz"] = None
    got.update({n: t.grad for n, t in wts.items()})
    return out.detach(), got


def _worst(got, ref):
    scale = ref.abs().max().item()
    diff = (got.double().cpu() - ref.double()).abs().max().item()
    return diff / scale if scale > 0 else (0.0 if diff == 0 else float("inf"))


# name: (B, C, Cout, N, S, dup, nosample)
CASES = {
    "down0": (2, 32, 32, 8192, 4096, False, False),
    "down1": (2, 64, 64, 4096, 2048, False, False),
    "down2": (2, 96, 96, 2048, 1024, False, False),
    "down3": (2, 128, 128, 1024, 512, False, False),
    "down4": (2, 192, 192, 512, 256, False, False),
    "est1_1024": (2, 195, 128, 1024, 1024, False, True),
    "est2_1024": (2, 128, 128, 1024, 1024, False, True),
    "est2_256": (2, 128, 128, 256, 256, False, True),
    "C0": (2, 0, 32, 600, 300, False, False),
    "Cout24": (2, 20, 24, 700, 350, False, False),
    "duplicates": (2, 32, 32, 1024, 512, True, False),
    "N_below_16": (2, 8, 16, 10, 6, False, False),
}


# ------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_all_gradients_vs_fp64_oracle(name):
    B, C, Cout, N, S, dup, nosample = CASES[name]
    c = _case(B, C, Cout, N, S, seed=len(name), dup=dup, nosample=nosample)
    ref_out, ref = _oracle(c)
    out, got = _gpu_run(c)
    assert _worst(out, ref_out) <= BAR
    names = [n for n in GRAD_NAMES if ref[n] is not None and ref[n].numel() > 0]
    ratios = {n: _worst(got[n], ref[n]) / BAR for n in names}
    print(f"\n[{name}] worst max|diff| / (1e-4 max|ref|): " + " ".join(f"{n}={r:.3g}" for n, r in ratios.items()))
    bad = {n: r for n, r in ratios.items() if not r <= 1.0}
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("subset", [("Wa", "ba", "Wb", "bb"), ("L", "bias"), ("feat",), ("xyz",), ("sampled_xyz",)])
def test_gradient_subsets_match_the_full_run(subset):
    c = _case(2, 48, 40, 1200, 600, seed=3)
    _, full = _gpu_run(c)
    _, part = _gpu_run(c, want=subset)
    for n in GRAD_NAMES:
        if n in subset:
            assert part[n] is not None and _worst(part[n], full[n].cpu()) <= BAR, n
        else:
            assert part[n] is None, n


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [1, 2])
def test_training_forward_is_bit_identical_to_the_fused_forward(precision):
    c = _case(2, 64, 64, 4096, 2048, seed=5)
    x, f, s, knn = (c[n].to(DEV) for n in ("xyz", "feat", "sampled_xyz", "knn"))
    w = {n: v.to(DEV) for n, v in c["w"].items()}
    with torch.no_grad():
        fused = pointconv.pointconv_forward(x, f, s, knn, w, precision)
    trained = pointconv.pointconv(x.clone().requires_grad_(True), f.clone().requires_grad_(True), s, knn,
                                  {n: v.clone().requires_grad_(True) for n, v in w.items()}, precision)
    assert trained.requires_grad and torch.equal(trained.detach(), fused)


@pytest.mark.gpu
def test_module_optimiser_step_matches_the_oracle_step():
    C, Cout, N, S, lr = 48, 64, 1500, 700, 0.1
    c = _case(2, C, Cout, N, S, seed=11)
    mod = c["mod"].to(DEV)
    x, f, s = (c[n].to(DEV) for n in ("xyz", "feat", "sampled_xyz"))
    with pytest.raises(RuntimeError):
        b200.PointConvDownSampling(C, Cout).to(DEV)(x, f, s)       # the default module stays forward-only
    mod.differentiable = True
    params = {n: (v._base if v._base is not None else v) for n, v in pointconv.param_weights(mod).items()}
    before = {n: p.detach().clone() for n, p in params.items()}
    opt = torch.optim.SGD(mod.parameters(), lr=lr)
    out = mod(x, f, s)
    ref_out, ref = _oracle(c, post=True)
    keep = (ref_out.abs() > 2e-7 * ref_out.abs().max()).to(torch.float32)   # skip outputs on the final LeakyReLU kink
    (out * (c["grad"] * keep).to(DEV)).sum().backward()
    opt.step()
    c["grad"] = c["grad"] * keep
    _, ref = _oracle(c, post=True)
    for n in PointConvWeights.NAMES:
        step = (params[n].detach() - before[n]).reshape(ref[n].shape)
        assert _worst(step, -lr * ref[n]) <= BAR, n


@pytest.mark.gpu
def test_cuda_graph_replay_matches_eager_gradients():
    c = _case(2, 64, 64, 2048, 1024, seed=13)
    leaves, wts = _gpu_leaves(c)
    knn, grad = c["knn"].to(DEV), c["grad"].to(DEV)
    every = list(leaves.values()) + list(wts.values())

    def step():
        _linear(leaves, wts, knn).backward(grad)

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


@pytest.mark.gpu
def test_training_batchnorm_composition_matches_fp64_autograd():
    """PointConvFunction -> BatchNorm1d (training mode, batch statistics) -> LeakyReLU(0.1), as install(train=
    {"PointConv"}) runs a pyramid level with norm='batch_norm', against fp64 autograd of the same composition."""
    from oracle import torch_ref
    c = _case(2, 32, 64, 1024, 512, seed=17)
    assert not _near_kink_points(c).any()                  # BN couples all points: this seed has no weight-net kink
    gen = torch.Generator().manual_seed(17)
    gamma, beta = 1.0 + 0.1 * torch.randn(64, generator=gen), 0.1 * torch.randn(64, generator=gen)
    grad = torch.randn(2, 64, 512, generator=gen)

    def arm(double):
        dev, dt = (torch.device("cpu"), torch.float64) if double else (DEV, torch.float32)
        bn = torch.nn.BatchNorm1d(64).to(dev, dt).train()
        with torch.no_grad():
            bn.weight.copy_(gamma)
            bn.bias.copy_(beta)
        leaves = {n: c[n].to(dev, dt).requires_grad_(True) for n in INPUTS}
        wts = {n: v.to(dev, dt).requires_grad_(True) for n, v in c["w"].items()}
        if double:
            post = torch_ref.pointconv(leaves["xyz"], leaves["feat"], leaves["sampled_xyz"], wts, k=16, knn=c["knn"])
            y = torch.where(post > 0, post, post * 10.0)
        else:
            y = _linear(leaves, wts, c["knn"].to(DEV))
        y.retain_grad()
        out = F.leaky_relu(bn(y), 0.1)
        return out, y, leaves, wts, bn

    ref_out, *_ = arm(True)
    keep = (ref_out.abs() > 2e-7 * ref_out.abs().max()).to(torch.float64)
    got, ref = {}, {}
    for double, store in ((True, ref), (False, got)):
        out, y, leaves, wts, bn = arm(double)
        out.backward((grad * keep).to(out.device, out.dtype))
        store.update({n: t.grad for n, t in leaves.items()})
        store.update({n: t.grad for n, t in wts.items()})
        store["bn_weight"], store["bn_bias"] = bn.weight.grad, bn.bias.grad
        store["out"] = out.detach()
        store["dy_abs_sum"] = y.grad.abs().sum(dim=(0, 2))
    # Training-mode BatchNorm subtracts the batch mean of each channel, so dbias = sum_{b,s} dy is exactly zero: the
    # fp64 reference is rounding noise (~1e-13) and a bar relative to it is meaningless.  A sum of fp32 terms that
    # cancel is exact to a fraction of the terms' magnitudes, so dbias is held to 1e-4 of max_o sum_{b,s} |dy[o]|.
    assert (got["bias"].double().cpu() - ref["bias"]).abs().max().item() <= BAR * ref["dy_abs_sum"].max().item()
    for n in ref:
        if n not in ("bias", "dy_abs_sum"):
            assert _worst(got[n], ref[n]) <= BAR, n


@pytest.mark.gpu
def test_deterministic_mode_makes_the_direct_api_raise():
    c = _case(1, 16, 32, 256, 128, seed=19)
    leaves, wts = _gpu_leaves(c)
    torch.use_deterministic_algorithms(True)
    try:
        with pytest.raises(RuntimeError, match="deterministic"):
            pointconv.pointconv(leaves["xyz"], leaves["feat"], leaves["sampled_xyz"], c["knn"].to(DEV), wts)
    finally:
        torch.use_deterministic_algorithms(False)


# ------------------------------------------------------------------------------------------------- real model
def _reference_root():
    from refmodel_util import reference_root
    return reference_root()


@pytest.mark.gpu
@pytest.mark.skipif(_reference_root() is None,
                    reason="no reference tree (stage one with `make -C oracle reftree REF=<RPEFlow checkout>`)")
def test_reference_model_gradients_with_pointconv_trained_here():
    """Unmodified RPEFlow, eval mode, grad enabled, loss = fixed random weighting of flow_2d / flow_3d.  Arm T:
    install(train={"Correlation3D", "PointConv"}); arm R: install()."""
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

    flows_t, grads_t, st_t = arm({"Correlation3D", "PointConv"})
    flows_r, grads_r, _ = arm(False)
    pc = [st_t.get(n, {"b200": 0, "reference": 0}) for n in ("PointConvDownSampling.forward", "PointConvNoSampling.forward")]
    assert sum(s["b200"] for s in pc) == 20 and sum(s["reference"] for s in pc) == 0, pc
    assert st_t["Correlation3D.forward"] == {"b200": 5, "reference": 0}, st_t["Correlation3D.forward"]
    for key in flows_t:
        assert _worst(flows_t[key], flows_r[key].cpu()) <= 1e-3, key
    assert grads_t.keys() == grads_r.keys() and len(grads_t) > 0
    for n in grads_r:
        assert _worst(grads_t[n], grads_r[n].cpu()) <= 1e-3, n
