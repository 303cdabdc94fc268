"""Backwards of the decoder ops knn_interpolation / backwarp_3d, backwarp_2d (border) and convex_upsample
(b200_knn_interpolate_bwd, b200_backwarp2d_bwd, b200_convex_upsample_bwd; projection.*Function; install(train=...)).

CPU: the new C-ABI entries agree with the header at ABI 8 and reject bad arguments without touching a device; the new
Python entry points refuse CPU tensors; install(train=...) takes the new names.

GPU (-m gpu): every gradient against fp64 CPU autograd of oracle.torch_ref on the same inputs and indices, normwise per
tensor, max|got - ref| <= 2e-5 * max|ref| (the bar tests/test_backward_reference.py derives for fp32 sums of this
length); the cases the kernels can get wrong (repeated neighbours, scatter collisions, unselected points, zero
distances, clamped indices, samples pushed off the image, padded taps, saturated softmax); gradient subsets; the
training forward against the no-grad forward bit for bit; fp16 / bf16 and strided inputs; deterministic mode; CUDA-graph
capture; and, when a reference tree is staged, the unmodified RPEFlow with every decoder op trained here.
"""
import ctypes
import os
import re
import zlib

import pytest
import torch

import rpeflow_b200 as b200
from rpeflow_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200flow.h")
DEV = torch.device("cuda", 0)
NEW = ("b200_knn_interpolate_bwd", "b200_backwarp2d_bwd", "b200_convex_upsample_bwd",
       "b200_convex_upsample_bwd_scratch_floats")
FP32_BAR = 2e-5
# fp16 / bf16: the public functions up-cast, so the only added error is the final rounding of each gradient to the
# input dtype (one unit roundoff of the entry); the reference runs on the same rounded inputs.
HALF_BAR = {torch.float16: FP32_BAR + 2.0 ** -11, torch.bfloat16: FP32_BAR + 2.0 ** -8}
# backwarp_2d samples where the fp32 forward puts the sample: pixel + flow, then the round trip 2*g/(W-1)-1 ->
# ((g+1)/2)*(W-1), which together move a coordinate by up to ~1.1e-5 px at W = 240 (the fp64 reference does not).  The
# flow gradient jumps where a coordinate crosses an integer (the bilinear cell changes), so fp32 and fp64 may floor
# differently within that distance of an integer: pixels within INT_TAU of one are left out of the dflow check.
# Elsewhere the shift only perturbs the bilinear weights; emulating the fp32 coordinates in fp64 gives at most 8.5e-6
# (dx) and 1.4e-5 (dflow) of max|ref| at the 144 x 240 level, inside FP32_BAR.
INT_TAU = 1e-4
ZERO_REF = 1e-12


# ------------------------------------------------------------------------------------------------- CPU
def test_new_symbols_in_header_and_signature_table_at_abi8():
    text = open(HEADER).read()
    declared = sorted(set(re.findall(r"^B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(", text, flags=re.M)))
    for name in NEW:
        assert name in declared and name in _lib.SIGNATURES
    assert sorted(_lib.SIGNATURES) == declared
    assert _lib.ABI_VERSION == 8 and _lib.lib.b200_abi_version() == 8


def test_knn_interpolate_bwd_rejects_bad_arguments_without_a_gpu():
    lib = _lib.lib
    one = ctypes.c_void_p(16)              # never dereferenced: argument checks come first

    def call(xyz=one, idx=one, g=one, B=1, C=8, M=64, Q=32, k=3):
        return lib.b200_knn_interpolate_bwd(xyz, one, one, idx, g, None, None, None, B, C, M, Q, k, None)
    assert call(k=0) == -1 and b"k must be in [1,8]" in lib.b200_last_error()
    assert call(k=9) == -1
    assert call(M=0) == -1 and b"bad sizes" in lib.b200_last_error()
    assert call(B=-1) == -1 and call(Q=-1) == -1 and call(C=-1) == -1
    assert call(B=65536) == -1
    for bad in ({"xyz": None}, {"idx": None}, {"g": None}):
        assert call(**bad) == -1 and b"null pointer" in lib.b200_last_error()
    for empty in ({"B": 0}, {"C": 0}, {"Q": 0}):
        assert lib.b200_knn_interpolate_bwd(None, None, None, None, None, None, None, None,
                                            empty.get("B", 1), empty.get("C", 8), 64, empty.get("Q", 32), 3, None) == 0


def test_backwarp2d_bwd_rejects_bad_arguments_without_a_gpu():
    lib = _lib.lib
    one = ctypes.c_void_p(16)

    def call(x=one, flow=one, g=one, B=1, C=4, H=8, W=8):
        return lib.b200_backwarp2d_bwd(x, flow, g, None, None, B, C, H, W, None)
    assert call(H=0) == -1 and b"bad sizes" in lib.b200_last_error()
    assert call(W=0) == -1 and call(B=-1) == -1 and call(C=-1) == -1
    assert call(H=65536, W=65536) == -1 and b"too large" in lib.b200_last_error()
    for bad in ({"x": None}, {"flow": None}, {"g": None}):
        assert call(**bad) == -1 and b"null pointer" in lib.b200_last_error()
    assert lib.b200_backwarp2d_bwd(None, None, None, None, None, 0, 4, 8, 8, None) == 0
    assert lib.b200_backwarp2d_bwd(None, None, None, None, None, 2, 0, 8, 8, None) == 0


def test_convex_upsample_bwd_rejects_bad_arguments_without_a_gpu():
    lib = _lib.lib
    one = ctypes.c_void_p(16)

    def call(flow=one, g=one, dflow=None, scratch=None, B=1, H=8, W=8, s=4):
        return lib.b200_convex_upsample_bwd(flow, one, g, dflow, None, scratch, B, H, W, s, None)
    for s in (0, 1, 3, 16):
        assert call(s=s) == -1 and b"scale_factor must be 2, 4 or 8" in lib.b200_last_error()
    assert call(H=0) == -1 and call(W=0) == -1 and call(B=-1) == -1
    assert call(flow=None) == -1 and b"null pointer" in lib.b200_last_error()
    assert call(g=None) == -1
    assert call(dflow=one, scratch=None) == -1 and b"scratch" in lib.b200_last_error()
    assert call(g=ctypes.c_void_p(20)) == -1 and b"16-byte aligned" in lib.b200_last_error()
    assert lib.b200_convex_upsample_bwd(None, None, None, None, None, None, 0, 8, 8, 4, None) == 0
    for B, H, W, s in ((1, 1, 1, 2), (2, 144, 240, 4), (8, 9, 13, 8)):
        assert lib.b200_convex_upsample_bwd_scratch_floats(B, H, W, s) >= 18 * B * H * W


def test_new_entry_points_have_no_cpu_fallback():
    xyz = torch.rand(1, 3, 16, requires_grad=True)
    feat = torch.rand(1, 4, 16, requires_grad=True)
    idx = torch.zeros(1, 16, 3, dtype=torch.int64)
    x, flow = torch.rand(1, 4, 8, 8, requires_grad=True), torch.zeros(1, 2, 8, 8, requires_grad=True)
    mask = torch.rand(1, 36, 8, 8, requires_grad=True)
    for call in (lambda: b200.knn_interpolation(xyz, feat, xyz, 3, knn_indices=idx),
                 lambda: b200.backwarp_3d(xyz, xyz, xyz),
                 lambda: b200.backwarp_2d(x, flow, "border"),
                 lambda: b200.convex_upsample(flow, mask, 2),
                 lambda: b200.KnnInterpolationFunction.apply(xyz, feat, xyz, idx),
                 lambda: b200.Backwarp2dFunction.apply(x, flow),
                 lambda: b200.ConvexUpsampleFunction.apply(flow, mask, 2)):
        with pytest.raises(RuntimeError, match="no CPU"):
            call()


def test_install_train_takes_the_decoder_op_names():
    import rpeflow_b200.install as inst
    assert {"knn_interpolation", "backwarp_2d", "convex_upsample"} <= set(inst.TRAINABLE)
    try:
        inst.install(patch_python=False, extensions=False, train={"knn_interpolation", "backwarp_2d", "convex_upsample"})
        assert inst._TRAIN == {"knn_interpolation", "backwarp_2d", "convex_upsample"}
        inst.install(patch_python=False, extensions=False, train=True)
        assert inst._TRAIN == {"Correlation3D"}
        inst.install(patch_python=False, extensions=False)
        assert inst._TRAIN == frozenset()
        with pytest.raises(ValueError, match="unknown op"):
            inst.install(patch_python=False, extensions=False, train={"convex_upsample", "backwarp_3d"})
    finally:
        inst.uninstall()


# ------------------------------------------------------------------------------------------------- GPU helpers
def _poison_allocator(nbytes=64 << 20):
    """Leave NaN-filled blocks in the CUDA caching allocator, so that an output the kernel fails to write shows."""
    blocks = [torch.full((n,), float("nan"), device=DEV) for n in (nbytes // 4, 1 << 16, 1 << 12, 256)]
    del blocks


def _worst(got, ref):
    """max|got - ref| / max|ref|.  A reference that is zero up to fp64 rounding (max|ref| < ZERO_REF: with k = 1 the
    normalised weight is 1 and the xyz gradients vanish, but fp64 leaves ~1e-16 of noise) is compared absolutely."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape
    scale = ref.abs().max().item() if ref.numel() else 0.0
    err = (got - ref).abs().max().item() if ref.numel() else 0.0
    return err / scale if scale >= ZERO_REF else err


def _check(got, ref, bar=FP32_BAR, masks=None):
    """masks: {name: bool tensor broadcastable to the gradient}, entries outside it are not compared."""
    for n, r in ref.items():
        assert got[n] is not None, n
        assert bool(torch.isfinite(got[n]).all()), n
        g = got[n].detach().double().cpu()
        if masks and n in masks:
            g, r = g * masks[n], r * masks[n]
        assert _worst(g, r) <= bar, (n, _worst(g, r))


def _ref_grads(fn, inputs, grad):
    """fp64 CPU autograd of fn(**inputs): {name: gradient}."""
    leaves = {n: t.detach().cpu().double().requires_grad_(True) for n, t in inputs.items()}
    out = fn(**leaves)
    got = torch.autograd.grad(out, list(leaves.values()), grad.detach().cpu().double(), allow_unused=True)
    return {n: (g if g is not None else torch.zeros_like(leaves[n])) for n, g in zip(leaves, got)}


def _gpu_grads(fn, inputs, grad, want=None, dtype=torch.float32):
    leaves = {n: t.detach().to(DEV, dtype).requires_grad_(want is None or n in want) for n, t in inputs.items()}
    _poison_allocator()
    out = fn(**leaves)
    out.backward(grad.to(DEV, out.dtype))
    torch.cuda.synchronize()
    return {n: t.grad for n, t in leaves.items()}, out.detach()


# ------------------------------------------------------------------------------------------------- knn_interpolation
def _clamped(idx, M):
    j = torch.where(idx < 0, idx + M, idx)
    return j.clamp(0, M - 1)


def _knn_case(B, C, M, Q, k, seed, kind="random"):
    gen = torch.Generator().manual_seed(seed)
    xin = torch.rand(B, 3, M, generator=gen)
    feat = torch.randn(B, C, M, generator=gen)
    xq = torch.rand(B, 3, Q, generator=gen)
    idx = torch.randint(0, M, (B, Q, k), generator=gen)
    if kind == "m_lt_k":                              # what the KNN returns for M < k: trailing zero indices
        idx = torch.zeros(B, Q, k, dtype=torch.int64)
        idx[:, :, :M] = torch.stack([torch.randperm(M, generator=gen) for _ in range(B * Q)]).view(B, Q, M)
    elif kind == "collision":                         # every query selects the same k points
        idx = torch.arange(5, 5 + k).view(1, 1, k).expand(B, Q, k).contiguous()
    elif kind == "unused":                            # points >= M // 2 are selected by no query
        idx = torch.randint(0, M // 2, (B, Q, k), generator=gen)
    elif kind == "coincide":                          # query q sits on point 2q, its first neighbour; odd points otherwise
        assert M >= 2 * Q
        xq = xin[:, :, 0:2 * Q:2].clone()
        idx = 2 * torch.randint(0, M // 2, (B, Q, k), generator=gen) + 1
        idx[:, :, 0] = 2 * torch.arange(Q)
    elif kind == "out_of_range":
        idx = torch.randint(-2 * M, 2 * M, (B, Q, k), generator=gen)
    grad = torch.randn(B, C, Q, generator=gen)
    return {"input_xyz": xin, "input_features": feat, "query_xyz": xq}, idx, grad


def _knn_ref(idx, M):
    from oracle import torch_ref
    j = _clamped(idx, M)
    return lambda input_xyz, input_features, query_xyz: torch_ref.knn_interpolation(
        input_xyz, input_features, query_xyz, idx.shape[2], knn_indices=j)


def _knn_gpu(idx):
    i = idx.to(DEV)
    return lambda input_xyz, input_features, query_xyz: b200.knn_interpolation(
        input_xyz, input_features, query_xyz, idx.shape[2], knn_indices=i)


KNN_CASES = {f"k{k}_C{C}": (2, C, 300, 257, k, "random") for k in (1, 3, 8) for C in (0, 1, 3, 64, 192)}
KNN_CASES.update({
    "level_4to3_C128": (2, 128, 256, 512, 3, "random"), "level_2to1_C64": (2, 64, 2048, 4096, 3, "random"),
    "flow_4096to8192": (2, 3, 4096, 8192, 3, "random"), "backwarp3d_2048": (2, 3, 2048, 2048, 3, "random"),
    "m_lt_k": (2, 16, 2, 100, 3, "m_lt_k"), "m1_k8": (2, 5, 1, 50, 8, "m_lt_k"),
    "collision": (2, 32, 64, 3000, 3, "collision"), "unused": (2, 8, 400, 300, 3, "unused"),
    "coincide": (2, 16, 600, 256, 3, "coincide"), "out_of_range": (2, 8, 100, 200, 4, "out_of_range"),
})


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(KNN_CASES))
def test_knn_interpolation_gradients_vs_fp64(name):
    B, C, M, Q, k, kind = KNN_CASES[name]
    inputs, idx, grad = _knn_case(B, C, M, Q, k, seed=zlib.crc32(name.encode()) % 1000, kind=kind)
    got, out = _gpu_grads(_knn_gpu(idx), inputs, grad)
    _check(got, _ref_grads(_knn_ref(idx, M), inputs, grad))
    if kind == "unused":
        for n in ("input_xyz", "input_features"):
            assert bool((got[n][:, :, M // 2:] == 0).all()), n
    if kind == "coincide":
        even = got["input_xyz"][:, :, 0:2 * Q:2]
        assert bool((even == 0).all())                 # r = 0 gives that pair (the only one reading point 2q) no xyz grad
        near = inputs["input_features"][:, :, 0:2 * Q:2].to(DEV)
        assert _worst(out, near) <= 1e-6               # the coincident neighbour takes weight ~1


@pytest.mark.gpu
@pytest.mark.parametrize("subset", [("input_features",), ("input_xyz",), ("query_xyz",), ("input_xyz", "query_xyz")])
def test_knn_interpolation_gradient_subsets(subset):
    inputs, idx, grad = _knn_case(2, 64, 512, 1024, 3, seed=5)
    full, _ = _gpu_grads(_knn_gpu(idx), inputs, grad)
    part, _ = _gpu_grads(_knn_gpu(idx), inputs, grad, want=subset)
    for n in inputs:
        if n in subset:
            assert _worst(part[n], full[n]) <= FP32_BAR, n
        else:
            assert part[n] is None, n


@pytest.mark.gpu
def test_backwarp_3d_gradients_reach_all_three_inputs():
    from oracle import torch_ref
    gen = torch.Generator().manual_seed(7)
    B, N = 2, 2048
    xyz1 = torch.rand(B, 3, N, generator=gen)
    xyz2 = xyz1 + 0.02 * torch.randn(B, 3, N, generator=gen)
    flow = 0.02 * torch.randn(B, 3, N, generator=gen)
    grad = torch.randn(B, 3, N, generator=gen)
    inputs = {"xyz1": xyz1, "xyz2": xyz2, "flow12": flow}
    idx = b200.k_nearest_neighbor((xyz1 + flow).to(DEV), xyz2.to(DEV), 3).cpu()     # what backwarp_3d searches with

    def ref(xyz1, xyz2, flow12):
        return xyz2 + torch_ref.knn_interpolation(xyz1 + flow12, -flow12, xyz2, 3, knn_indices=idx)
    got, _ = _gpu_grads(lambda **t: b200.backwarp_3d(**t), inputs, grad)
    assert got["flow12"] is not None
    _check(got, _ref_grads(ref, inputs, grad))


# ------------------------------------------------------------------------------------------------- backwarp_2d
def _bw_case(B, C, H, W, seed, kind="random"):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, H, W, generator=gen)
    if kind == "random":
        flow = 3.0 * torch.randn(B, 2, H, W, generator=gen)
    elif kind == "zero":
        flow = torch.zeros(B, 2, H, W)
    else:                                             # "outside": every sample pushed past a corner, all four sides
        sx = torch.where(torch.arange(W) < W // 2, -1.0, 1.0).view(1, W).expand(H, W)
        sy = torch.where(torch.arange(H) < H // 2, -1.0, 1.0).view(H, 1).expand(H, W)
        flow = torch.stack([sx * (W + 3.5), sy * (H + 2.5)]).unsqueeze(0).expand(B, 2, H, W).contiguous()
    return {"x": x, "flow12": flow}, torch.randn(B, C, H, W, generator=gen)


def _bw_ref(x, flow12):
    from oracle import torch_ref
    return torch_ref.backwarp_2d(x, flow12, "border")


def _bw_gpu(x, flow12):
    return b200.backwarp_2d(x, flow12, "border")


def _off_integer(flow):
    """[B,H,W] True where neither fp64 sample coordinate is within INT_TAU of an integer."""
    B, _, H, W = flow.shape
    gx = torch.arange(W, dtype=torch.float64).view(1, 1, W) + flow[:, 0].double()
    gy = torch.arange(H, dtype=torch.float64).view(1, H, 1) + flow[:, 1].double()
    return ((gx - gx.round()).abs() > INT_TAU) & ((gy - gy.round()).abs() > INT_TAU)


def _bw_masks(inputs):
    return {"flow12": _off_integer(inputs["flow12"]).unsqueeze(1)}


BW_CASES = {"level4_C128": (2, 128, 18, 30), "level3_C96": (2, 96, 36, 60), "level2_C64": (2, 64, 72, 120),
            "level1_C32": (1, 32, 144, 240), "odd_C5": (3, 5, 17, 23), "H2": (2, 3, 2, 9), "W2": (2, 3, 7, 2)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BW_CASES))
@pytest.mark.parametrize("kind", ["random", "zero", "outside"])
def test_backwarp_2d_gradients_vs_fp64(name, kind):
    B, C, H, W = BW_CASES[name]
    inputs, grad = _bw_case(B, C, H, W, seed=zlib.crc32(name.encode()) % 1000, kind=kind)
    got, _ = _gpu_grads(_bw_gpu, inputs, grad)
    ref = _ref_grads(_bw_ref, inputs, grad)
    _check(got, ref, masks=_bw_masks(inputs))
    dflow = got["flow12"].cpu()
    if kind == "outside":
        assert bool((dflow == 0).all())
    elif kind == "zero":
        assert bool((dflow[:, 0, :, 0] == 0).all() and (dflow[:, 0, :, W - 1] == 0).all())
        assert bool((dflow[:, 1, 0, :] == 0).all() and (dflow[:, 1, H - 1, :] == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("subset", [("x",), ("flow12",)])
def test_backwarp_2d_gradient_subsets(subset):
    inputs, grad = _bw_case(2, 32, 36, 60, seed=9)
    full, _ = _gpu_grads(_bw_gpu, inputs, grad)
    part, _ = _gpu_grads(_bw_gpu, inputs, grad, want=subset)
    for n in inputs:
        if n in subset:
            assert _worst(part[n], full[n]) <= FP32_BAR, n
        else:
            assert part[n] is None, n


# ------------------------------------------------------------------------------------------------- convex_upsample
def _cu_case(B, H, W, s, seed, kind="random"):
    gen = torch.Generator().manual_seed(seed)
    flow = 4.0 * torch.randn(B, 2, H, W, generator=gen)
    mask = torch.randn(B, 9 * s * s, H, W, generator=gen)
    if kind == "onehot":
        hot = torch.randint(0, 9, (B, 1, s, s, H, W), generator=gen)
        mask = 80.0 * torch.nn.functional.one_hot(hot, 9).squeeze(1).permute(0, 5, 1, 2, 3, 4).reshape(B, 9 * s * s, H, W).float()
    elif kind == "pm80":
        mask = 80.0 * torch.sign(mask)
    return {"flow": flow, "mask": mask}, torch.randn(B, 2, H * s, W * s, generator=gen)


def _cu_ref(s):
    from oracle import torch_ref
    return lambda flow, mask: torch_ref.convex_upsample(flow, mask, s)


def _cu_gpu(s):
    return lambda flow, mask: b200.convex_upsample(flow, mask, s)


CU_CASES = {"s2": (2, 9, 13, 2, "random"), "s4": (2, 9, 13, 4, "random"), "s8": (2, 9, 13, 8, "random"),
            "1x1_s4": (2, 1, 1, 4, "random"), "1xW_s8": (2, 1, 7, 8, "random"), "1xW_s2": (3, 1, 5, 2, "random"),
            "level1_s4": (2, 144, 240, 4, "random"), "onehot80_s4": (2, 12, 20, 4, "onehot"),
            "pm80_s4": (2, 12, 20, 4, "pm80"), "pm80_s8": (1, 6, 5, 8, "pm80")}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CU_CASES))
def test_convex_upsample_gradients_vs_fp64(name):
    B, H, W, s, kind = CU_CASES[name]
    inputs, grad = _cu_case(B, H, W, s, seed=zlib.crc32(name.encode()) % 1000, kind=kind)
    got, _ = _gpu_grads(_cu_gpu(s), inputs, grad)
    _check(got, _ref_grads(_cu_ref(s), inputs, grad))


@pytest.mark.gpu
def test_convex_upsample_is_bit_reproducible_and_runs_in_deterministic_mode():
    inputs, grad = _cu_case(2, 36, 60, 4, seed=3)
    first, _ = _gpu_grads(_cu_gpu(4), inputs, grad)
    torch.use_deterministic_algorithms(True)
    try:
        second, _ = _gpu_grads(_cu_gpu(4), inputs, grad)
    finally:
        torch.use_deterministic_algorithms(False)
    for n in inputs:
        assert torch.equal(first[n], second[n]), n


@pytest.mark.gpu
@pytest.mark.parametrize("subset", [("flow",), ("mask",)])
def test_convex_upsample_gradient_subsets(subset):
    inputs, grad = _cu_case(2, 18, 30, 4, seed=4)
    full, _ = _gpu_grads(_cu_gpu(4), inputs, grad)
    part, _ = _gpu_grads(_cu_gpu(4), inputs, grad, want=subset)
    for n in inputs:
        assert torch.equal(part[n], full[n]) if n in subset else part[n] is None, n


# ------------------------------------------------------------------------------------------------- all three
def _ops():
    """name -> (inputs, grad, gpu fn, fp64 reference fn)."""
    kin, idx, kg = _knn_case(2, 64, 512, 1024, 3, seed=21)
    bin_, bg = _bw_case(2, 32, 36, 60, seed=22)
    cin, cg = _cu_case(2, 18, 30, 4, seed=23)
    return {"knn_interpolation": (kin, kg, _knn_gpu(idx), _knn_ref(idx, 512)),
            "backwarp_2d": (bin_, bg, _bw_gpu, _bw_ref),
            "convex_upsample": (cin, cg, _cu_gpu(4), _cu_ref(4))}


def _masks(op, inputs):
    return _bw_masks(inputs) if op == "backwarp_2d" else None


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["knn_interpolation", "backwarp_2d", "convex_upsample"])
def test_training_forward_is_bit_identical_to_no_grad(op):
    inputs, _, fn, _ = _ops()[op]
    leaves = {n: t.to(DEV).requires_grad_(True) for n, t in inputs.items()}
    with torch.no_grad():
        plain = fn(**leaves)
    train = fn(**leaves)
    assert train.grad_fn is not None and plain.grad_fn is None
    assert torch.equal(train.detach(), plain)


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["knn_interpolation", "backwarp_2d", "convex_upsample"])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_precision_inputs(op, dtype):
    inputs, grad, fn, ref = _ops()[op]
    rounded = {n: t.to(dtype).float() for n, t in inputs.items()}
    got, _ = _gpu_grads(fn, rounded, grad, dtype=dtype)
    for n in got:
        assert got[n].dtype == dtype, n
    _check(got, _ref_grads(ref, rounded, grad), bar=HALF_BAR[dtype], masks=_masks(op, rounded))


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["knn_interpolation", "backwarp_2d", "convex_upsample"])
def test_non_contiguous_inputs(op):
    inputs, grad, fn, ref = _ops()[op]
    leaves = {}
    for n, t in inputs.items():                      # the same values behind a transposed layout
        base = t.to(DEV).transpose(-1, -2).contiguous().transpose(-1, -2)
        assert not base.is_contiguous() or t.shape[-1] == 1
        leaves[n] = base.requires_grad_(True)
    _poison_allocator()
    fn(**leaves).backward(grad.to(DEV))
    _check({n: t.grad for n, t in leaves.items()}, _ref_grads(ref, inputs, grad), masks=_masks(op, inputs))


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["knn_interpolation", "backwarp_2d"])
def test_atomic_backwards_raise_in_deterministic_mode_and_install_routes_them_to_the_reference(op):
    import rpeflow_b200.install as inst
    inputs, _, fn, _ = _ops()[op]
    leaves = {n: t.to(DEV).requires_grad_(True) for n, t in inputs.items()}
    fast = {"knn_interpolation": lambda input_xyz, input_features, query_xyz, k=3:
            b200.knn_interpolation(input_xyz, input_features, query_xyz, k),
            "backwarp_2d": lambda x, flow12, padding_mode="border": b200.backwarp_2d(x, flow12, padding_mode)}[op]
    called = []

    def slow(*args, **kwargs):
        called.append(op)
        return None
    try:
        inst.install(patch_python=False, extensions=False, train=set(inst.TRAINABLE))
        inst.stats(reset=True)
        routed = inst._dispatch(op, fast, slow, train=op)
        torch.use_deterministic_algorithms(True)
        try:
            with pytest.raises(RuntimeError, match="deterministic"):
                fn(**leaves)
            routed(*leaves.values())
        finally:
            torch.use_deterministic_algorithms(False)
        assert called == [op] and inst.stats()[op] == {"b200": 0, "reference": 1}
        out = routed(*leaves.values())
        assert out.grad_fn is not None and inst.stats()[op] == {"b200": 1, "reference": 1}
    finally:
        inst.uninstall()


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["knn_interpolation", "backwarp_2d", "convex_upsample"])
def test_cuda_graph_replay_matches_eager_gradients(op):
    inputs, grad, fn, _ = _ops()[op]
    leaves = [t.to(DEV).requires_grad_(True) for t in inputs.values()]
    g = grad.to(DEV)

    def step():
        fn(**dict(zip(inputs, leaves))).backward(g)

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
        if op == "convex_upsample":
            assert torch.equal(t.grad, e)
        else:
            assert _worst(t.grad, e) <= FP32_BAR


# ------------------------------------------------------------------------------------------------- real model
def _reference_root():
    from refmodel_util import reference_root
    return reference_root()


DECODER_OPS = {"knn_interpolation": 9, "backwarp_3d": 4, "backwarp_2d": 4, "convex_upsample": 1}


@pytest.mark.gpu
@pytest.mark.skipif(_reference_root() is None,
                    reason="no reference tree (stage one with `make -C oracle reftree REF=<RPEFlow checkout>`)")
def test_reference_model_gradients_with_the_decoder_trained_here():
    """Unmodified RPEFlow, eval mode, grad enabled, loss = fixed random weighting of flow_2d / flow_3d.  Arm T:
    install(train=TRAINABLE); arm R: install(train={"Correlation3D", "PointConv"})."""
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

    flows_t, grads_t, st_t = arm(set(inst.TRAINABLE))
    flows_r, grads_r, st_r = arm({"Correlation3D", "PointConv"})
    for op, calls in DECODER_OPS.items():
        t, r = st_t.get(op, {"b200": 0, "reference": 0}), st_r.get(op, {"b200": 0, "reference": 0})
        assert t["reference"] == 0 and t["b200"] == calls, (op, t)
        assert r["b200"] + r["reference"] == calls, (op, r)
    for op in ("knn_interpolation", "backwarp_2d", "convex_upsample"):
        assert st_r[op]["reference"] > 0, (op, st_r[op])        # the model needs these graphs
    print("backwarp_3d routes without its train route:", st_r.get("backwarp_3d"))
    for key in flows_t:
        assert _worst(flows_t[key], flows_r[key]) <= 1e-3, key
    assert grads_t.keys() == grads_r.keys() and len(grads_t) > 0
    for n in grads_r:
        assert _worst(grads_t[n], grads_r[n]) <= 1e-3, n
