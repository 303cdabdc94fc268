"""correlation2d's backward on NCHW maps (b200_corr2d_bwd_nchw, ops.Correlation2dNCHWFunction, install(train=...)).

CPU: the new entry agrees with the header at ABI 8 and rejects bad arguments without touching a device; a host program
compiled against corr2d_bwd_nchw_index.cuh walks every address the kernel forms (sources in range, zero-filled pieces at
the base, 16-byte pieces aligned, every output element written once); CPU tensors raise; install takes the name.

GPU (-m gpu): the same bits as b200_corr2d_bwd on permuted inputs wherever that entry takes its md = 4 tiled kernel;
the CPU oracle at ragged channel counts, narrow and misaligned maps; NULL gradients, poisoned outputs, repeatability;
and through autograd: training forward == no-grad forward, gradients against fp64 autograd of oracle.torch_ref,
fp16 / bf16 and strided inputs, other displacements, KAT-corr, CUDA-graph capture and the install() routing.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import rpeflow_b200 as b200
import rpeflow_b200.install as inst
from rpeflow_b200 import _lib
from rpeflow_b200.workload import CONFIGS, LEVEL_CHANNELS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200flow.h")
CSRC = os.path.join(ROOT, "rpeflow_b200", "csrc")
DEV = torch.device("cuda", 0)
FP32_BAR = 2e-5                   # max|got - ref| / max|ref| against fp64, as tests/test_decoder_backward.py
HALF_BAR = {torch.float16: FP32_BAR + 2.0 ** -11, torch.bfloat16: FP32_BAR + 2.0 ** -8}


def _level_shapes():
    """(C, H, W) of the model's five correlation levels in every workload."""
    shapes = {}
    for name in ("things", "dsec", "hd"):
        for lvl, c in zip(range(1, 6), LEVEL_CHANNELS):
            shapes[f"{name}_l{lvl}"] = (c,) + CONFIGS[name].level_hw(lvl)
    return shapes


LEVELS = _level_shapes()
# every shape where b200_corr2d_bwd takes its tiled kernel (C % 4 == 0, W % 4 == 0), at B = 2
TILED = {n: s for n, s in LEVELS.items() if s[2] % 4 == 0}
TILED.update({"ragged_36x11x44": (36, 11, 44), "ragged_8x9x12": (8, 9, 12)})
# the oracle cases: levels with W % 4 != 0, C neither a multiple of 4 nor of 32, maps smaller than one tile
ORACLE = {n: s for n, s in LEVELS.items() if s[2] % 4 != 0}
ORACLE.update({"c7_5x3": (7, 5, 3), "c20_13x50": (20, 13, 50), "c36_11x44": (36, 11, 44), "c100_9x20": (100, 9, 20),
               "tiny_3x1x1": (3, 1, 1), "tiny_12x6x20": (12, 6, 20), "tiny_33x7x9": (33, 7, 9)})


# ------------------------------------------------------------------------------------------------- CPU
def test_new_symbol_in_header_and_signature_table_at_abi8():
    import re
    text = open(HEADER).read()
    declared = sorted(set(re.findall(r"^B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(", text, flags=re.M)))
    assert "b200_corr2d_bwd_nchw" in declared and "b200_corr2d_bwd_nchw" in _lib.SIGNATURES
    assert sorted(_lib.SIGNATURES) == declared
    assert _lib.ABI_VERSION == 8 and _lib.lib.b200_abi_version() == 8


def test_corr2d_bwd_nchw_rejects_bad_arguments_without_a_gpu():
    lib = _lib.lib
    one = ctypes.c_void_p(16)              # never dereferenced: argument checks come first

    def call(g=one, a=one, b=one, g1=one, g2=one, B=1, C=8, H=8, W=8, md=4):
        return lib.b200_corr2d_bwd_nchw(g, a, b, g1, g2, B, C, H, W, md, None)
    for bad in ({"B": -1}, {"C": 0}, {"H": 0}, {"W": 0}, {"W": -3}):
        assert call(**bad) == -1 and b"bad sizes" in lib.b200_last_error(), bad
    for md in (0, -1, 65):
        assert call(md=md) == -1 and b"max_displacement" in lib.b200_last_error()
    for bad in ({"g": None}, {"a": None}, {"b": None}, {"g": None, "g2": None}, {"a": None, "g1": None}):
        assert call(**bad) == -1 and b"null pointer" in lib.b200_last_error(), bad
    assert call(B=1 << 20, H=1 << 13, W=1 << 13) == -1 and b"grid limit" in lib.b200_last_error()
    assert call(B=65536, H=1 << 12, W=1 << 12) == -1
    for md in (1, 2, 3, 5, 64):
        assert call(md=md) == _lib.B200_ENOSUP and b"needs md=4" in lib.b200_last_error()
    assert lib.b200_corr2d_bwd_nchw(None, None, None, None, None, 0, 8, 8, 8, 4, None) == 0
    assert lib.b200_corr2d_bwd_nchw(None, None, None, None, None, 3, 8, 8, 8, 4, None) == 0


def _audit_shapes():
    shapes = [(2,) + s for s in LEVELS.values()]
    shapes += [(2,) + s for s in list(TILED.values()) + list(ORACLE.values())]
    shapes += [(3, 5, 7, 11), (1, 33, 40, 250), (2, 16, 12, 17), (1, 64, 8, 32), (1, 65, 9, 33)]
    return sorted(set(shapes))


def test_every_address_of_the_kernel_is_in_range(tmp_path):
    cxx = shutil.which(os.environ.get("CXX", "c++")) or shutil.which("g++") or shutil.which("clang++")
    if cxx is None:
        pytest.skip("no host C++ compiler")
    exe = str(tmp_path / "audit")
    subprocess.run([cxx, "-O2", "-std=c++17", "-I", CSRC, os.path.join(ROOT, "tests", "corr2d_bwd_nchw_audit.cpp"), "-o", exe],
                   check=True)
    args = [str(v) for s in _audit_shapes() for v in s]
    res = subprocess.run([exe] + args, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert f"{len(_audit_shapes())} shapes, 0 failures" in res.stdout


def test_new_entry_points_have_no_cpu_fallback():
    a = torch.rand(1, 4, 8, 8, requires_grad=True)
    b = torch.rand(1, 4, 8, 8, requires_grad=True)
    for call in (lambda: b200.correlation2d(a, b, 4), lambda: b200.Correlation2dNCHWFunction.apply(a, b, 4),
                 lambda: b200.correlation2d_leaky(a, b, 4)):
        with pytest.raises(RuntimeError, match="no CPU"):
            call()


def test_install_train_takes_correlation2d():
    assert "correlation2d" in inst.TRAINABLE and "Correlation2D" not in inst.TRAINABLE
    try:
        inst.install(patch_python=False, extensions=False, train={"correlation2d"})
        assert inst._TRAIN == {"correlation2d"}
        inst.install(patch_python=False, extensions=False, train="correlation2d")
        assert inst._TRAIN == {"correlation2d"}
        inst.install(patch_python=False, extensions=False, train=True)
        assert inst._TRAIN == {"Correlation3D"}
        with pytest.raises(ValueError, match="unknown op"):
            inst.install(patch_python=False, extensions=False, train={"Correlation2D"})
    finally:
        inst.uninstall()


# ------------------------------------------------------------------------------------------------- GPU helpers
def _case(B, C, H, W, seed, md=4):
    gen = torch.Generator().manual_seed(seed)
    f1 = torch.randn(B, C, H, W, generator=gen)
    f2 = torch.randn(B, C, H, W, generator=gen)
    go = torch.randn(B, (2 * md + 1) ** 2, H, W, generator=gen)
    return f1, f2, go


def _offset(t):
    """The same values at a 4-byte storage offset (not 16-byte aligned)."""
    pad = torch.zeros(t.numel() + 1, device=DEV)
    return pad[1:].view(t.shape).copy_(t)


def _bwd_nchw(go, f1, f2, want=(1, 2), out=None):
    """b200_corr2d_bwd_nchw on device tensors; out: optional (g1, g2) buffers to write into."""
    B, C, H, W = f1.shape
    g1, g2 = out if out is not None else (torch.empty_like(f1), torch.empty_like(f2))
    rc = _lib.lib.b200_corr2d_bwd_nchw(go.data_ptr(), f1.data_ptr(), f2.data_ptr(),
                                       g1.data_ptr() if 1 in want else None, g2.data_ptr() if 2 in want else None,
                                       B, C, H, W, 4, torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "b200_corr2d_bwd_nchw")
    return g1, g2


def _bwd_nhwc(go, f1, f2):
    return b200.ops._correlation_backward_cuda(go, f1.permute(0, 2, 3, 1).contiguous(), f2.permute(0, 2, 3, 1).contiguous(), 4)


def _worst(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape
    if ref.numel() == 0:
        return 0.0
    return (got - ref).abs().max().item() / max(ref.abs().max().item(), 1e-30)


def _nhwc_np(t):
    return t.permute(0, 2, 3, 1).contiguous().numpy()


# ------------------------------------------------------------------------------------------------- entry level
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(TILED))
def test_same_bits_as_the_tiled_nhwc_backward(name):
    C, H, W = TILED[name]
    f1, f2, go = (t.to(DEV) for t in _case(2, C, H, W, seed=C + H + W))
    g1, g2 = _bwd_nchw(go, f1, f2)
    r1, r2 = _bwd_nhwc(go, f1, f2)
    assert torch.equal(g1, r1) and torch.equal(g2, r2)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ORACLE))
def test_against_the_cpu_oracle(name):
    from oracle import spec
    C, H, W = ORACLE[name]
    f1, f2, go = _case(2, C, H, W, seed=C * H + W)
    w1, w2 = spec.corr2d_bwd(go.numpy(), _nhwc_np(f1), _nhwc_np(f2), 4)
    g1, g2 = _bwd_nchw(go.to(DEV), f1.to(DEV), f2.to(DEV))
    np.testing.assert_allclose(g1.cpu().numpy(), w1, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(g2.cpu().numpy(), w2, rtol=1e-5, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 36, 11, 44), (2, 32, 16, 64), (1, 20, 13, 50), (2, 7, 5, 3)])
@pytest.mark.parametrize("which", ["inputs", "grad_out", "outputs"])
def test_four_byte_offset_pointers_against_the_cpu_oracle(shape, which):
    from oracle import spec
    B, C, H, W = shape
    f1, f2, go = _case(B, C, H, W, seed=W + len(which))
    w1, w2 = spec.corr2d_bwd(go.numpy(), _nhwc_np(f1), _nhwc_np(f2), 4)
    a, b, g = f1.to(DEV), f2.to(DEV), go.to(DEV)
    out = None
    if which == "inputs":
        a, b = _offset(a), _offset(b)
    elif which == "grad_out":
        g = _offset(g)
    else:
        out = (_offset(torch.full_like(a, float("nan"))), _offset(torch.full_like(b, float("nan"))))
    g1, g2 = _bwd_nchw(g, a, b, out=out)
    np.testing.assert_allclose(g1.cpu().numpy(), w1, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(g2.cpu().numpy(), w2, rtol=1e-5, atol=1e-5)


@pytest.mark.gpu
def test_empty_batch():
    f1, f2, go = (t.to(DEV) for t in _case(0, 8, 9, 12, seed=1))
    g1, g2 = _bwd_nchw(go, f1, f2)
    assert g1.shape == (0, 8, 9, 12) and g2.shape == (0, 8, 9, 12)
    a, b = f1.requires_grad_(True), f2.requires_grad_(True)
    out = b200.correlation2d(a, b, 4)
    out.backward(go)
    assert a.grad.shape == a.shape and b.grad.shape == b.shape


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 7, 5, 3), (2, 36, 11, 44), (2, 100, 9, 20), (3, 32, 18, 30), (1, 64, 9, 33)])
def test_poisoned_outputs_are_fully_overwritten_and_single_gradients_match(shape):
    B, C, H, W = shape
    f1, f2, go = (t.to(DEV) for t in _case(B, C, H, W, seed=sum(shape)))
    nan = lambda: torch.full((B, C, H, W), float("nan"), device=DEV)      # noqa: E731
    g1, g2 = _bwd_nchw(go, f1, f2, out=(nan(), nan()))
    assert bool(torch.isfinite(g1).all()) and bool(torch.isfinite(g2).all())
    only1 = _bwd_nchw(go, f1, f2, want=(1,), out=(nan(), nan()))
    assert torch.equal(only1[0], g1) and bool(torch.isnan(only1[1]).all())
    only2 = _bwd_nchw(go, f1, f2, want=(2,), out=(nan(), nan()))
    assert torch.equal(only2[1], g2) and bool(torch.isnan(only2[0]).all())


@pytest.mark.gpu
def test_repeatable_bits_also_in_deterministic_mode():
    f1, f2, go = (t.to(DEV) for t in _case(2, 64, 72, 120, seed=11))
    first = _bwd_nchw(go, f1, f2)
    second = _bwd_nchw(go, f1, f2)
    assert all(torch.equal(x, y) for x, y in zip(first, second))
    grads = []
    for deterministic in (False, True):
        torch.use_deterministic_algorithms(deterministic)
        try:
            a, b = f1.clone().requires_grad_(True), f2.clone().requires_grad_(True)
            b200.correlation2d(a, b, 4).backward(go)
            grads.append((a.grad, b.grad))
        finally:
            torch.use_deterministic_algorithms(False)
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])
    assert torch.equal(grads[0][0], first[0]) and torch.equal(grads[0][1], first[1])


# ------------------------------------------------------------------------------------------------- autograd
FWD_SHAPES = [(2, 32, 36, 60), (2, 128, 18, 30), (2, 192, 9, 15), (2, 7, 5, 3), (1, 32, 144, 240)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", FWD_SHAPES)
@pytest.mark.parametrize("op", ["correlation2d", "correlation2d_leaky"])
def test_training_forward_is_bit_identical_to_no_grad(shape, op):
    fn = getattr(b200, op)
    f1, f2, _ = _case(*shape, seed=3)
    a, b = f1.to(DEV).requires_grad_(True), f2.to(DEV).requires_grad_(True)
    with torch.no_grad():
        plain = fn(a, b, 4)
    train = fn(a, b, 4)
    assert train.grad_fn is not None and plain.grad_fn is None
    assert torch.equal(train.detach(), plain)


def _ref_fns():
    from oracle import torch_ref
    import torch.nn.functional as F
    return {
        "correlation2d": (lambda input1, input2: b200.correlation2d(input1, input2, 4),
                          lambda input1, input2: torch_ref.correlation2d(input1, input2, 4)),
        "correlation2d_leaky": (lambda input1, input2: b200.correlation2d_leaky(input1, input2, 4, 0.1),
                                lambda input1, input2: F.leaky_relu(torch_ref.correlation2d(input1, input2, 4), 0.1)),
    }


def _grads(fn, inputs, grad, dev, dtype, want=None):
    leaves = {n: t.detach().to(dev, dtype).requires_grad_(want is None or n in want) for n, t in inputs.items()}
    out = fn(**leaves)
    out.backward(grad.to(dev, out.dtype))
    return {n: t.grad for n, t in leaves.items()}


def _check(got, ref, bar=FP32_BAR, masks=None):
    for n, r in ref.items():
        assert got[n] is not None and bool(torch.isfinite(got[n]).all()), n
        g = got[n].detach().double().cpu()
        if masks and n in masks:
            g, r = g * masks[n], r * masks[n]
        assert _worst(g, r) <= bar, (n, _worst(g, r))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 32, 36, 60), (2, 128, 18, 30), (2, 20, 13, 50), (2, 7, 5, 3)])
@pytest.mark.parametrize("op", ["correlation2d", "correlation2d_leaky"])
def test_autograd_gradients_vs_fp64(shape, op):
    fn, ref = _ref_fns()[op]
    f1, f2, go = _case(*shape, seed=5)
    inputs = {"input1": f1, "input2": f2}
    got = _grads(fn, inputs, go, DEV, torch.float32)
    _check(got, _grads(ref, inputs, go, "cpu", torch.float64))


def _off_integer(flow):
    """[B,1,H,W] True where neither fp64 sample coordinate is within 1e-4 px of an integer: the flow gradient of the
    bilinear warp jumps there, and the fp32 forward may floor differently (see tests/test_decoder_backward.py)."""
    B, _, H, W = flow.shape
    gx = torch.arange(W, dtype=torch.float64).view(1, 1, W) + flow[:, 0].double()
    gy = torch.arange(H, dtype=torch.float64).view(1, H, 1) + flow[:, 1].double()
    return (((gx - gx.round()).abs() > 1e-4) & ((gy - gy.round()).abs() > 1e-4)).unsqueeze(1)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 32, 36, 60), (2, 128, 18, 30)])
def test_warp_correlate_gradients_vs_fp64(shape):
    from oracle import torch_ref
    import torch.nn.functional as F
    B, C, H, W = shape
    f1, f2, go = _case(B, C, H, W, seed=8)
    flow = 3.0 * torch.randn(B, 2, H, W, generator=torch.Generator().manual_seed(9))
    inputs = {"feat1": f1, "feat2": f2, "flow": flow}

    def ours(feat1, feat2, flow):
        return b200.warp_correlate(feat1, feat2, flow, 4, 0.1)

    def ref(feat1, feat2, flow):
        return F.leaky_relu(torch_ref.correlation2d(feat1, torch_ref.backwarp_2d(feat2, flow, "border"), 4), 0.1)
    got = _grads(ours, inputs, go, DEV, torch.float32)
    _check(got, _grads(ref, inputs, go, "cpu", torch.float64), masks={"flow": _off_integer(flow)})


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("shape", [(2, 32, 36, 60), (2, 20, 13, 50)])
def test_half_precision_inputs(dtype, shape):
    fn, ref = _ref_fns()["correlation2d"]
    f1, f2, go = _case(*shape, seed=6)
    rounded = {"input1": f1.to(dtype).float(), "input2": f2.to(dtype).float()}
    got = _grads(fn, rounded, go, DEV, dtype)
    assert all(g.dtype == dtype for g in got.values())
    _check(got, _grads(ref, rounded, go, "cpu", torch.float64), bar=HALF_BAR[dtype])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 32, 36, 60), (2, 20, 13, 50)])
def test_non_contiguous_inputs(shape):
    fn, ref = _ref_fns()["correlation2d"]
    f1, f2, go = _case(*shape, seed=7)
    leaves = {n: t.to(DEV).transpose(-1, -2).contiguous().transpose(-1, -2).requires_grad_(True)
              for n, t in (("input1", f1), ("input2", f2))}
    assert not leaves["input1"].is_contiguous()
    fn(**leaves).backward(go.to(DEV))
    _check({n: t.grad for n, t in leaves.items()}, _grads(ref, {"input1": f1, "input2": f2}, go, "cpu", torch.float64))


@pytest.mark.gpu
@pytest.mark.parametrize("md", [2, 5])
def test_other_displacements_through_the_nhwc_backward(md):
    from oracle import torch_ref
    f1, f2, go = _case(2, 24, 13, 20, seed=md, md=md)
    inputs = {"input1": f1, "input2": f2}
    got = _grads(lambda input1, input2: b200.correlation2d(input1, input2, md), inputs, go, DEV, torch.float32)
    _check(got, _grads(lambda input1, input2: torch_ref.correlation2d(input1, input2, md), inputs, go, "cpu", torch.float64))
    subset = _grads(lambda input1, input2: b200.correlation2d(input1, input2, md), inputs, go, DEV, torch.float32,
                    want=("input2",))
    assert subset["input1"] is None and torch.equal(subset["input2"], got["input2"])


@pytest.mark.gpu
def test_gradient_subsets_at_md4():
    f1, f2, go = _case(2, 36, 11, 44, seed=12)
    inputs = {"input1": f1, "input2": f2}
    fn = _ref_fns()["correlation2d"][0]
    full = _grads(fn, inputs, go, DEV, torch.float32)
    for n in inputs:
        part = _grads(fn, inputs, go, DEV, torch.float32, want=(n,))
        assert torch.equal(part[n], full[n]) and all(part[m] is None for m in inputs if m != n)


@pytest.mark.gpu
def test_kat_corr_through_autograd():
    """KAT-corr (correlation_test.cpp:44-60,82-89): rand B=32, C=128, 144x240, md=4, both gradients through autograd
    against the naive libtorch path, mean|d| < 1e-6."""
    from oracle import torch_ref
    torch.manual_seed(0)
    B, C, H, W, md = 32, 128, 144, 240, 4
    f1 = torch.rand(B, C, H, W).to(DEV).requires_grad_(True)
    f2 = torch.rand(B, C, H, W).to(DEV).requires_grad_(True)
    go = torch.rand(B, 81, H, W).to(DEV)
    b200.correlation2d(f1, f2, md).backward(go)
    for s in range(0, B, 8):
        x1 = f1.detach()[s:s + 8].clone().requires_grad_(True)
        x2 = f2.detach()[s:s + 8].clone().requires_grad_(True)
        torch_ref.correlation2d(x1, x2, md).backward(go[s:s + 8])
        assert (x1.grad - f1.grad[s:s + 8]).abs().mean().item() < 1e-6
        assert (x2.grad - f2.grad[s:s + 8]).abs().mean().item() < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 32, 36, 60), (2, 128, 18, 30)])
def test_cuda_graph_replay_matches_eager_gradients(shape):
    f1, f2, go = _case(*shape, seed=13)
    leaves = [f1.to(DEV).requires_grad_(True), f2.to(DEV).requires_grad_(True)]
    g = go.to(DEV)

    def step():
        b200.correlation2d(leaves[0], leaves[1], 4).backward(g)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            for t in leaves:
                t.grad = None
            step()
    torch.cuda.current_stream().wait_stream(side)
    eager = [t.grad.clone() for t in leaves]
    for t in leaves:
        t.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for t in leaves:
        t.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    for e, t in zip(eager, leaves):
        assert torch.equal(t.grad, e)


# ------------------------------------------------------------------------------------------------- install()
@pytest.mark.gpu
def test_install_routes_graph_building_calls_by_the_train_set():
    f1, f2, _ = _case(2, 32, 36, 60, seed=14)
    a, b = f1.to(DEV).requires_grad_(True), f2.to(DEV).requires_grad_(True)

    def fast(input1, input2, max_displacement, cpp_impl=True):
        return b200.correlation2d(input1, input2, max_displacement)
    called = []

    def slow(input1, input2, max_displacement, cpp_impl=True):
        called.append(1)
        return None
    try:
        for train, route in ((set(), "reference"), ({"Correlation3D"}, "reference"), (True, "reference"),
                             ({"correlation2d"}, "b200"), (set(inst.TRAINABLE), "b200")):
            inst.install(patch_python=False, extensions=False, train=train)
            inst.stats(reset=True)
            routed = inst._dispatch("correlation2d", fast, slow, train="correlation2d", atomics=False)
            for deterministic in (False, True):
                torch.use_deterministic_algorithms(deterministic)
                try:
                    out = routed(a, b, 4)
                finally:
                    torch.use_deterministic_algorithms(False)
                if route == "b200":
                    assert out.grad_fn is not None
            assert inst.stats()["correlation2d"] == {"b200": 2 if route == "b200" else 0,
                                                     "reference": 2 if route == "reference" else 0}, train
            inst.uninstall()
        assert len(called) == 6
    finally:
        inst.uninstall()


def _reference_root():
    from refmodel_util import reference_root
    return reference_root()


@pytest.mark.gpu
@pytest.mark.skipif(_reference_root() is None,
                    reason="no reference tree (stage one with `make -C oracle reftree REF=<RPEFlow checkout>`)")
def test_reference_model_with_correlation2d_trained_here():
    """Unmodified RPEFlow, eval mode, grad enabled, loss = fixed random weighting of flow_2d / flow_3d.  Arm T:
    install(train=TRAINABLE); arm R: the same without "correlation2d"."""
    from rpeflow_b200 import refhost

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

    flows_t, grads_t, st_t = arm(set(inst.TRAINABLE))
    flows_r, grads_r, st_r = arm(set(inst.TRAINABLE) - {"correlation2d"})
    assert st_t["correlation2d"] == {"b200": 5, "reference": 0}, st_t["correlation2d"]
    assert st_r["correlation2d"]["reference"] == 5, st_r["correlation2d"]
    for key in flows_t:
        assert _worst(flows_t[key], flows_r[key]) <= 1e-3, key
    assert grads_t.keys() == grads_r.keys() and len(grads_t) > 0
    for n in grads_r:
        assert _worst(grads_t[n], grads_r[n]) <= 1e-3, n
