"""Backwards of the projection gathers grid_sample_wrapper and batch_indexing_channel_{first,last}
(b200_grid_sample_pts_bwd, b200_gather_cf_bwd, b200_gather_cl_bwd; projection.GridSampleFunction,
BatchIndexingChannelFirstFunction, BatchIndexingChannelLastFunction; install(train=...)).

CPU: the new C-ABI entries agree with the header at ABI 8 and reject bad arguments without touching a device; the new
Functions and the graph path of the public functions refuse CPU tensors; install(train=...) takes the three names and
routes graph-building calls by them (checked against stand-in reference modules).

GPU (-m gpu): every gradient against fp64 CPU autograd of F.grid_sample / torch.gather / advanced indexing
(oracle.torch_ref) on the same inputs, normwise per tensor, max|got - ref| <= 2e-5 * max|ref| (the bar
tests/test_backward_reference.py derives for fp32 sums of this length), at the model's call shapes and at ragged ones;
the cases the kernels can get wrong (pixel centres and the border, points partly or wholly outside the image,
non-finite coordinates, atomic collisions, unsampled pixels and unread columns, duplicate / wrapped / clamped indices,
multi-dimensional and int32 indices, flat channel-last data, batch-local indices); gradient subsets; the training
forward against the no-grad forward bit for bit; the sample memo; fp16 / bf16 and strided inputs; CUDA-graph capture;
deterministic mode.
"""
import ctypes
import os
import re
import sys
import types
import zlib

import pytest
import torch

import rpeflow_b200 as b200
from rpeflow_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200flow.h")
DEV = torch.device("cuda", 0)
NEW = ("b200_grid_sample_pts_bwd", "b200_gather_cf_bwd", "b200_gather_cl_bwd")
OPS = ("grid_sample_wrapper", "batch_indexing_channel_first", "batch_indexing_channel_last")
FP32_BAR = 2e-5
# fp16 / bf16: the public function up-casts, so the only added error is the final rounding of each gradient to the
# input dtype; the reference runs on the same rounded inputs.
HALF_BAR = {torch.float16: FP32_BAR + 2.0 ** -11, torch.bfloat16: FP32_BAR + 2.0 ** -8}
# The fp32 forward samples at the round trip 2*x/(W-1)-1 -> ((g+1)/2)*(W-1) of x, which moves a coordinate by up to
# ~1.1e-5 px at W = 240 (the fp64 reference does not).  The xy gradient jumps where a coordinate crosses an integer (the
# bilinear cell changes), so fp32 and fp64 may floor differently within that distance of an integer: points within
# INT_TAU of one are left out of the xy check (as in tests/test_decoder_backward.py).
INT_TAU = 1e-4
ZERO_REF = 1e-12


# ------------------------------------------------------------------------------------------------- CPU
def test_new_symbols_in_header_and_signature_table_at_abi8():
    text = open(HEADER).read()
    declared = sorted(set(re.findall(r"^B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(", text, flags=re.M)))
    for name in NEW:
        assert name in declared and name in _lib.SIGNATURES and name in _lib.KERNELS_PER_CALL
    assert sorted(_lib.SIGNATURES) == declared
    assert _lib.ABI_VERSION == 8 and _lib.lib.b200_abi_version() == 8


def test_grid_sample_pts_bwd_rejects_bad_arguments_without_a_gpu():
    lib = _lib.lib
    one = ctypes.c_void_p(16)              # never dereferenced: argument checks come first

    def call(feat=one, xy=one, g=one, B=1, C=4, H=8, W=8, N=16):
        return lib.b200_grid_sample_pts_bwd(feat, xy, g, None, None, B, C, H, W, N, None)
    assert call(H=0) == -1 and b"bad sizes" in lib.b200_last_error()
    assert call(W=0) == -1 and call(B=-1) == -1 and call(C=-1) == -1 and call(N=-1) == -1
    assert call(H=65536, W=65536) == -1 and b"too large" in lib.b200_last_error()
    assert call(B=65536) == -1
    for bad in ({"feat": None}, {"xy": None}, {"g": None}):
        assert call(**bad) == -1 and b"null pointer" in lib.b200_last_error()
    for B, C, N in ((0, 4, 16), (2, 0, 16), (2, 4, 0)):
        assert lib.b200_grid_sample_pts_bwd(None, None, None, None, None, B, C, 8, 8, N, None) == 0


@pytest.mark.parametrize("entry", ["b200_gather_cf_bwd", "b200_gather_cl_bwd"])
def test_gather_bwd_rejects_bad_arguments_without_a_gpu(entry):
    lib = _lib.lib
    fn = getattr(lib, entry)
    one = ctypes.c_void_p(16)

    def call(g=one, idx=one, d=one, B=1, C=4, N=8, I=16):
        return fn(g, idx, d, B, C, N, I, None)
    assert call(N=0) == -1 and b"bad sizes" in lib.b200_last_error()
    assert call(B=-1) == -1 and call(C=-1) == -1 and call(I=-1) == -1
    assert call(B=65536) == -1 and b"grid limit" in lib.b200_last_error()
    assert call(I=1 << 45) == -1 and b"grid limit" in lib.b200_last_error()
    for bad in ({"g": None}, {"idx": None}, {"d": None}):
        assert call(**bad) == -1 and b"null pointer" in lib.b200_last_error()
    for B, C in ((0, 4), (2, 0)):
        assert fn(None, None, None, B, C, 8, 16, None) == 0


def test_new_entry_points_have_no_cpu_fallback():
    feat, xy = torch.rand(1, 4, 8, 8, requires_grad=True), torch.rand(1, 2, 16, requires_grad=True)
    data_cf, data_cl = torch.rand(1, 4, 16, requires_grad=True), torch.rand(1, 16, 4, requires_grad=True)
    idx = torch.zeros(1, 5, dtype=torch.int64)
    for call in (lambda: b200.grid_sample_wrapper(feat, xy),
                 lambda: b200.batch_indexing_channel_first(data_cf, idx),
                 lambda: b200.batch_indexing_channel_last(data_cl, idx),
                 lambda: b200.GridSampleFunction.apply(feat, xy),
                 lambda: b200.BatchIndexingChannelFirstFunction.apply(data_cf, idx),
                 lambda: b200.BatchIndexingChannelLastFunction.apply(data_cl, idx)):
        with pytest.raises(RuntimeError, match="no CPU"):
            call()


def test_install_train_takes_the_projection_op_names():
    import rpeflow_b200.install as inst
    assert set(OPS) <= set(inst.TRAINABLE)
    try:
        inst.install(patch_python=False, extensions=False, train=set(OPS))
        assert inst._TRAIN == set(OPS)
        inst.install(patch_python=False, extensions=False, train=True)
        assert inst._TRAIN == {"Correlation3D"}
        with pytest.raises(ValueError, match="unknown op"):
            inst.install(patch_python=False, extensions=False, train={"grid_sample_wrapper", "project_feat_with_nn_corr"})
    finally:
        inst.uninstall()


def _stand_in_reference(monkeypatch, calls):
    """models / models.utils / models.csrc / models.csrc.wrapper modules carrying device-agnostic torch versions of the
    reference's functions (each call recorded), so install() can re-bind them without a reference checkout."""
    def recorded(name, fn):
        def f(*args, **kwargs):
            calls.append(name)
            return fn(*args, **kwargs)
        f.__name__ = name
        return f
    utils = types.ModuleType("models.utils")
    for name, fn in (("grid_sample_wrapper", _ref_grid_sample), ("batch_indexing_channel_first", _ref_gather_cf),
                     ("batch_indexing_channel_last", _ref_gather_cl)):
        setattr(utils, name, recorded(name, fn))
    for name in ("project_feat_with_nn_corr", "knn_interpolation", "backwarp_3d", "backwarp_2d", "convex_upsample"):
        setattr(utils, name, recorded(name, lambda *a, **k: None))
    wrapper = types.ModuleType("models.csrc.wrapper")
    for name in ("correlation2d", "k_nearest_neighbor", "furthest_point_sampling"):
        setattr(wrapper, name, recorded(name, lambda *a, **k: None))
    for name, mod in (("models", types.ModuleType("models")), ("models.csrc", types.ModuleType("models.csrc")),
                      ("models.utils", utils), ("models.csrc.wrapper", wrapper)):
        monkeypatch.setitem(sys.modules, name, mod)
    return utils


@pytest.mark.parametrize("op", OPS)
def test_install_routes_graph_calls_by_train_name_on_cpu_tensors(monkeypatch, op):
    """On CPU tensors every call goes to the reference whatever `train` says (the kernels need CUDA)."""
    import rpeflow_b200.install as inst
    calls = []
    utils = _stand_in_reference(monkeypatch, calls)
    args = _small_args(op, torch.device("cpu"))
    try:
        inst.install(extensions=False, only=set(OPS), train={op})
        inst.stats(reset=True)
        out = getattr(utils, op)(*args)
        assert out.grad_fn is not None and calls == [op]
        assert inst.stats()[op] == {"b200": 0, "reference": 1}
    finally:
        inst.uninstall()


# ------------------------------------------------------------------------------------------------- references
def _ref_grid_sample(feat_2d, xy):
    from oracle import torch_ref
    return torch_ref.grid_sample_wrapper(feat_2d, xy)


def _ref_gather_cf(data, idx):
    from oracle import torch_ref
    return torch_ref.batch_indexing_channel_first(data, idx)


def _ref_gather_cl(data, idx):
    """oracle.torch_ref.batch_indexing_channel_last with the batch index made on the data's device."""
    nb = data.shape[0]
    b = torch.arange(nb, device=data.device).view([nb] + [1] * (idx.dim() - 1)).expand_as(idx)
    return data[b, idx.to(torch.int64)]


def _small_args(op, dev):
    gen = torch.Generator().manual_seed(1)
    if op == "grid_sample_wrapper":
        return (torch.randn(2, 3, 7, 9, generator=gen).to(dev).requires_grad_(True),
                (torch.rand(2, 2, 20, generator=gen) * 6).to(dev))
    idx = torch.randint(0, 10, (2, 6), generator=gen).to(dev)
    shape = (2, 3, 10) if op == "batch_indexing_channel_first" else (2, 10, 3)
    return torch.randn(*shape, generator=gen).to(dev).requires_grad_(True), idx


# ------------------------------------------------------------------------------------------------- GPU helpers
def _poison_allocator(nbytes=64 << 20):
    """Leave NaN-filled blocks in the CUDA caching allocator, so that an output the kernel fails to write shows."""
    blocks = [torch.full((n,), float("nan"), device=DEV) for n in (nbytes // 4, 1 << 16, 1 << 12, 256)]
    del blocks


def _worst(got, ref):
    """max|got - ref| / max|ref|; a reference that is zero up to fp64 rounding is compared absolutely."""
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
    """fp64 CPU autograd of fn(**inputs) over the floating inputs: {name: gradient}."""
    leaves = {n: t.detach().cpu().double().requires_grad_(True) if t.is_floating_point() else t.cpu()
              for n, t in inputs.items()}
    floats = [n for n, t in leaves.items() if t.is_floating_point()]
    out = fn(**leaves)
    got = torch.autograd.grad(out, [leaves[n] for n in floats], grad.detach().cpu().double(), allow_unused=True)
    return {n: (g if g is not None else torch.zeros_like(leaves[n])) for n, g in zip(floats, got)}


def _gpu_grads(fn, inputs, grad, want=None, dtype=torch.float32):
    leaves = {n: t.detach().to(DEV, dtype).requires_grad_(want is None or n in want) if t.is_floating_point()
              else t.to(DEV) for n, t in inputs.items()}
    _poison_allocator()
    out = fn(**leaves)
    out.backward(grad.to(DEV, out.dtype))
    torch.cuda.synchronize()
    return {n: t.grad for n, t in leaves.items() if t.is_floating_point()}, out.detach()


# ------------------------------------------------------------------------------------------------- grid_sample_wrapper
def _gs_gpu(feat_2d, xy):
    return b200.grid_sample_wrapper(feat_2d, xy)


def _gs_points(B, H, W, N, kind, gen):
    x = torch.rand(B, N, generator=gen) * (W + 1.0) - 1.0          # "random": a margin of one pixel past every side
    y = torch.rand(B, N, generator=gen) * (H + 1.0) - 1.0
    if kind == "centres":                                              # pixel centres, the border rows / columns included
        x = torch.randint(0, W, (B, N), generator=gen).float()
        y = torch.randint(0, H, (B, N), generator=gen).float()
        x[:, 0::7], y[:, 1::7] = float(W - 1), float(H - 1)
        x[:, 2::7], y[:, 3::7] = 0.0, 0.0
    elif kind == "outside":                                            # a third partly outside, a third wholly outside
        x = torch.rand(B, N, generator=gen) * (W + 6.0) - 3.0
        y = torch.rand(B, N, generator=gen) * (H + 6.0) - 3.0
        x[:, 0::3] = torch.where(torch.rand(B, (N + 2) // 3, generator=gen) < 0.5, -2.5, W + 1.5)
    elif kind == "nonfinite":                                          # every fourth point non-finite or huge
        bad = torch.tensor([float("nan"), float("inf"), -float("inf"), 3e9, -1e12])
        pick = torch.randint(0, 5, (B, (N + 3) // 4), generator=gen)
        x[:, 0::4] = bad[pick]
        y[:, 1::4] = bad[pick[:, :len(range(1, N, 4))]]
    elif kind == "collide":                                            # every point in one cell: 4 pixels take every tap
        x[:] = min(3, W - 2) + 0.25
        y[:] = min(2, H - 2) + 0.5
    elif kind == "unused":                                             # nothing right of the middle column or below row H/2
        x = torch.rand(B, N, generator=gen) * (W // 2 - 1)
        y = torch.rand(B, N, generator=gen) * (H // 2 - 1)
    return torch.stack([x, y], 1)


def _gs_case(B, C, H, W, N, seed, kind="random"):
    gen = torch.Generator().manual_seed(seed)
    feat = torch.randn(B, C, H, W, generator=gen)
    xy = _gs_points(B, H, W, N, kind, gen)
    return {"feat_2d": feat, "xy": xy}, torch.randn(B, C, N, generator=gen)


def _finite_points(xy):
    """[B,1,N] True where the forward finds a finite coordinate (the rest gets a zero xy gradient by definition)."""
    return (torch.isfinite(xy) & (xy.abs() < 1e9)).all(1, keepdim=True)


def _off_integer(xy):
    """[B,1,N] True where neither coordinate lies within INT_TAU of an integer (and both are finite)."""
    x = xy.double()
    return (((x - x.round()).abs() > INT_TAU) & torch.isfinite(x)).all(1, keepdim=True)


def _gs_reference(inputs, grad):
    """fp64 autograd of F.grid_sample.  Non-finite or huge points are moved far outside the image first, which is what the
    forward does with them (no tap inside the image); ATen itself gives NaN or 0 for those."""
    xy = inputs["xy"]
    moved = torch.where(_finite_points(xy).expand_as(xy), xy, torch.full_like(xy, -1e6))
    return _ref_grads(_ref_grid_sample, {"feat_2d": inputs["feat_2d"], "xy": moved}, grad)


GS_SHAPES = {"l1_C32": (2, 32, 144, 240, 4096), "l2_C64": (2, 64, 72, 120, 2048), "l3_C96": (2, 96, 36, 60, 1024),
             "l4_C128": (2, 128, 18, 30, 512), "l5_C192": (2, 192, 9, 15, 256), "cost_C81": (2, 81, 72, 120, 2048),
             "dec_C96": (2, 96, 144, 240, 4096), "odd_C5": (3, 5, 17, 23, 301), "odd_C33": (2, 33, 31, 47, 1000),
             "tiny": (2, 1, 2, 3, 77)}
GS_CASES = {f"{s}_random": (s, "random") for s in GS_SHAPES}
GS_CASES.update({f"{s}_{k}": (s, k) for s in ("l2_C64", "odd_C5", "tiny")
                 for k in ("centres", "outside", "nonfinite", "collide")})
GS_CASES.update({"l3_C96_unused": ("l3_C96", "unused"), "odd_C33_unused": ("odd_C33", "unused")})


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GS_CASES))
def test_grid_sample_gradients_vs_fp64(name):
    shape, kind = GS_CASES[name]
    B, C, H, W, N = GS_SHAPES[shape]
    inputs, grad = _gs_case(B, C, H, W, N, seed=zlib.crc32(name.encode()) % 1000, kind=kind)
    got, out = _gpu_grads(_gs_gpu, inputs, grad)
    _check(got, _gs_reference(inputs, grad), masks={"xy": _off_integer(inputs["xy"])})
    dxy, dfeat = got["xy"].cpu(), got["feat_2d"].cpu()
    if kind == "nonfinite":
        assert bool((dxy * ~_finite_points(inputs["xy"]) == 0).all())
        assert bool((out.cpu() * ~_finite_points(inputs["xy"]) == 0).all())
    if kind == "outside":
        far = (inputs["xy"][:, 0] <= -2.0) | (inputs["xy"][:, 0] >= W + 1.0)
        assert bool((dxy[:, :, :][far.unsqueeze(1).expand_as(dxy)] == 0).all())
    if kind == "unused":
        assert bool((dfeat[:, :, :, W // 2:] == 0).all() and (dfeat[:, :, H // 2:, :] == 0).all())
    if kind == "collide":
        x0, y0 = min(3, W - 2), min(2, H - 2)
        assert bool((dfeat[:, :, y0:y0 + 2, x0:x0 + 2] != 0).all()) and int((dfeat != 0).sum()) == B * C * 4


@pytest.mark.gpu
@pytest.mark.parametrize("subset", [("feat_2d",), ("xy",)])
def test_grid_sample_gradient_subsets(subset):
    inputs, grad = _gs_case(2, 32, 36, 60, 1024, seed=9)
    full, _ = _gpu_grads(_gs_gpu, inputs, grad)
    part, _ = _gpu_grads(_gs_gpu, inputs, grad, want=subset)
    for n in inputs:
        if n in subset:
            assert _worst(part[n], full[n]) <= FP32_BAR, n
        else:
            assert part[n] is None, n


@pytest.mark.gpu
def test_grid_sample_after_project_feat_builds_a_graph_and_leaves_the_memo_entry():
    from rpeflow_b200.projection import SAMPLE_MEMO
    inputs, grad = _gs_case(2, 32, 36, 60, 1024, seed=11)
    feat = inputs["feat_2d"].to(DEV).requires_grad_(True)
    xy = inputs["xy"].to(DEV).requires_grad_(True)
    f3 = torch.randn(2, 16, 1024, device=DEV)
    nn_idx = torch.randint(0, 1024, (2, 36 * 60), device=DEV)
    SAMPLE_MEMO.clear()
    try:
        b200.project_feat_with_nn_corr(xy, feat, f3, nn_idx)
        parked, hits = len(SAMPLE_MEMO.entries), SAMPLE_MEMO.hits
        assert parked == 1
        out = b200.grid_sample_wrapper(feat, xy)
        assert out.grad_fn is not None
        assert len(SAMPLE_MEMO.entries) == parked and SAMPLE_MEMO.hits == hits
        out.backward(grad.to(DEV))
        _check({"feat_2d": feat.grad, "xy": xy.grad}, _gs_reference(inputs, grad), masks={"xy": _off_integer(inputs["xy"])})
        with torch.no_grad():
            again = b200.grid_sample_wrapper(feat, xy)
        assert SAMPLE_MEMO.hits == hits + 1 and torch.equal(again, out.detach())
    finally:
        SAMPLE_MEMO.clear()


# ------------------------------------------------------------------------------------------------- gathers
def _wrapped(idx, N):
    j = torch.where(idx < 0, idx + N, idx)
    return j.clamp(0, N - 1)


def _gather_case(B, C, N, ishape, seed, kind="random", flat=False, channel_last=False):
    gen = torch.Generator().manual_seed(seed)
    if channel_last:
        data = torch.randn(B, N, generator=gen) if flat else torch.randn(B, N, C, generator=gen)
    else:
        data = torch.randn(B, C, N, generator=gen)
    if kind == "random":
        idx = torch.randint(0, N, (B, *ishape), generator=gen)
    elif kind == "perm":                                               # distinct indices per sample (FPS-like)
        idx = torch.stack([torch.randperm(N, generator=gen)[:ishape[0]] for _ in range(B)])
    elif kind == "dups":                                               # heavy duplicates: 20 distinct columns
        idx = torch.randint(0, 20, (B, *ishape), generator=gen)
    elif kind == "collide":                                            # every output reads one element
        idx = torch.full((B, *ishape), 7, dtype=torch.int64)
    elif kind == "wrap_clamp":                                         # negative (wrapped once) and out of range (clamped)
        idx = torch.randint(-2 * N, 2 * N, (B, *ishape), generator=gen)
    elif kind == "unused":                                             # columns >= N // 2 are read by nobody
        idx = torch.randint(0, N // 2, (B, *ishape), generator=gen)
    out_shape = ([B] + list(ishape) + ([] if flat else [C])) if channel_last else [B, C] + list(ishape)
    return data, idx, torch.randn(*out_shape, generator=gen)


def _gather_check(data, idx, grad, channel_last, idx_dtype=torch.int64, kind="random"):
    N = data.shape[1] if channel_last else data.shape[2]
    fn = b200.batch_indexing_channel_last if channel_last else b200.batch_indexing_channel_first
    ref = _ref_gather_cl if channel_last else _ref_gather_cf
    got, out = _gpu_grads(lambda data, idx: fn(data, idx), {"data": data, "idx": idx.to(idx_dtype)}, grad)
    j = _wrapped(idx, N)
    assert torch.equal(out.cpu(), ref(data, j))
    _check(got, _ref_grads(lambda data, idx: ref(data, idx), {"data": data, "idx": j}, grad))
    if kind == "unused":
        d = got["data"].cpu()
        assert bool(((d[:, N // 2:] if channel_last else d[:, :, N // 2:]) == 0).all())
    return got


GATHER_CF = {"pyramid_xyz_8192to4096": (2, 3, 8192, (4096,), "perm"), "feat_C64_knn16": (2, 64, 4096, (1024, 16), "random"),
             "ragged_C5": (3, 5, 77, (1001,), "random"), "dups_C32": (2, 32, 500, (3000,), "dups"),
             "collide_C8": (2, 8, 50, (4000,), "collide"), "wrap_clamp_C7": (2, 7, 100, (13, 17), "wrap_clamp"),
             "unused_C16": (2, 16, 400, (900,), "unused"), "flat_index_B1": (1, 3, 64, (), "random")}
GATHER_CL = {"xyz_C3_knn16": (2, 3, 8192, (4096, 16), "random", False), "feat_C64_knn16": (2, 64, 2048, (1024, 16), "random", False),
             "ragged_C5": (3, 5, 77, (1001,), "random", False), "C4_dups": (2, 4, 300, (5000,), "dups", False),
             "C128_collide": (2, 128, 50, (700,), "collide", False), "wrap_clamp_C8": (2, 8, 100, (13, 17), "wrap_clamp", False),
             "unused_C12": (2, 12, 400, (900,), "unused", False), "flat_BN": (2, 1, 1000, (3000,), "random", True),
             "flat_BN_wrap": (3, 1, 333, (20, 30), "wrap_clamp", True)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GATHER_CF))
def test_gather_channel_first_gradients_vs_fp64(name):
    B, C, N, ishape, kind = GATHER_CF[name]
    data, idx, grad = _gather_case(B, C, N, ishape, zlib.crc32(name.encode()) % 1000, kind)
    _gather_check(data, idx, grad, False, kind=kind)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GATHER_CL))
def test_gather_channel_last_gradients_vs_fp64(name):
    B, C, N, ishape, kind, flat = GATHER_CL[name]
    data, idx, grad = _gather_case(B, C, N, ishape, zlib.crc32(name.encode()) % 1000, kind, flat, channel_last=True)
    _gather_check(data, idx, grad, True, kind=kind)


@pytest.mark.gpu
@pytest.mark.parametrize("channel_last", [False, True])
def test_gather_int32_indices_and_batch_local_indices(channel_last):
    B, C, N = 4, 8, 257
    data, idx, grad = _gather_case(B, C, N, (600,), 31, "wrap_clamp", channel_last=channel_last)
    got = _gather_check(data, idx, grad, channel_last, idx_dtype=torch.int32)
    # sample b reads only its own data: its gradient equals a one-sample call on that sample
    for b in (0, B - 1):
        one, _ = _gpu_grads(lambda data, idx: (b200.batch_indexing_channel_last if channel_last else
                                               b200.batch_indexing_channel_first)(data, idx),
                            {"data": data[b:b + 1], "idx": idx[b:b + 1]}, grad[b:b + 1])
        assert _worst(one["data"], got["data"][b:b + 1]) <= FP32_BAR


@pytest.mark.gpu
def test_gather_cl_bwd_vector_and_scalar_stores_agree():
    """C % 4 == 0 with aligned pointers takes the red.global.add.v4.f32 path; grad_out one float past a 16-byte boundary
    takes the scalar one.  Both sum the same values into the same elements."""
    lib = _lib.lib
    B, N, C, I = 2, 300, 8, 4000
    gen = torch.Generator().manual_seed(3)
    idx = torch.randint(-N, N, (B, I), generator=gen)
    grad = torch.randn(B, I, C, generator=gen)
    outs = []
    for off in (0, 1):
        g = torch.empty(B * I * C + 4, device=DEV)[off:off + B * I * C]
        g.copy_(grad.view(-1))
        d = torch.full((B, N, C), float("nan"), device=DEV)
        assert lib.b200_gather_cl_bwd(g.data_ptr(), idx.to(DEV).data_ptr(), d.data_ptr(), B, C, N, I,
                                      torch.cuda.current_stream().cuda_stream) == 0
        torch.cuda.synchronize()
        outs.append(d)
    ref = _ref_grads(_ref_gather_cl, {"data": torch.zeros(B, N, C), "idx": _wrapped(idx, N)}, grad)["data"]
    for d in outs:
        assert _worst(d, ref) <= FP32_BAR


# ------------------------------------------------------------------------------------------------- all three
def _ops():
    """name -> (inputs, grad, gpu fn, fp64 reference fn, xy mask or None)."""
    gin, gg = _gs_case(2, 32, 36, 60, 1024, seed=21)
    cf_data, cf_idx, cf_g = _gather_case(2, 16, 600, (700, 3), 22, "wrap_clamp")
    cl_data, cl_idx, cl_g = _gather_case(2, 12, 600, (900,), 23, "dups", channel_last=True)
    return {
        "grid_sample_wrapper": (gin, gg, _gs_gpu, _ref_grid_sample, {"xy": _off_integer(gin["xy"])}),
        "batch_indexing_channel_first": ({"data": cf_data, "idx": cf_idx}, cf_g,
                                         lambda data, idx: b200.batch_indexing_channel_first(data, idx),
                                         lambda data, idx: _ref_gather_cf(data, _wrapped(idx, 600)), None),
        "batch_indexing_channel_last": ({"data": cl_data, "idx": cl_idx}, cl_g,
                                        lambda data, idx: b200.batch_indexing_channel_last(data, idx), _ref_gather_cl, None),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("op", OPS)
def test_training_forward_is_bit_identical_to_no_grad(op):
    inputs, _, fn, _, _ = _ops()[op]
    leaves = {n: t.to(DEV).requires_grad_(True) if t.is_floating_point() else t.to(DEV) for n, t in inputs.items()}
    with torch.no_grad():
        plain = fn(**leaves)
    train = fn(**leaves)
    assert train.grad_fn is not None and plain.grad_fn is None
    assert torch.equal(train.detach(), plain)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_grid_sample_half_precision_inputs(dtype):
    inputs, grad, fn, ref, masks = _ops()["grid_sample_wrapper"]
    rounded = {n: t.to(dtype).float() for n, t in inputs.items()}
    got, _ = _gpu_grads(fn, rounded, grad, dtype=dtype)
    for n in got:
        assert got[n].dtype == dtype, n
    _check(got, _ref_grads(ref, rounded, grad), bar=HALF_BAR[dtype], masks={"xy": _off_integer(rounded["xy"])})


@pytest.mark.gpu
@pytest.mark.parametrize("op", OPS)
def test_non_contiguous_inputs(op):
    inputs, grad, fn, ref, masks = _ops()[op]
    leaves = {}
    for n, t in inputs.items():                      # the same values behind a transposed layout
        base = t.to(DEV).transpose(-1, -2).contiguous().transpose(-1, -2)
        assert not base.is_contiguous()
        leaves[n] = base.requires_grad_(True) if t.is_floating_point() else base
    _poison_allocator()
    fn(**leaves).backward(grad.to(DEV))
    got = {n: t.grad for n, t in leaves.items() if t.is_floating_point()}
    _check(got, _ref_grads(ref, inputs, grad), masks=masks)


@pytest.mark.gpu
@pytest.mark.parametrize("op", OPS)
def test_cuda_graph_replay_matches_eager_gradients(op):
    inputs, grad, fn, _, _ = _ops()[op]
    named = {n: t.to(DEV).requires_grad_(True) if t.is_floating_point() else t.to(DEV) for n, t in inputs.items()}
    leaves = [t for t in named.values() if t.is_floating_point()]
    g = grad.to(DEV)

    def step():
        fn(**named).backward(g)

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
        assert _worst(t.grad, e) <= FP32_BAR


@pytest.mark.gpu
@pytest.mark.parametrize("op", OPS)
def test_deterministic_mode_raises_and_install_routes_to_the_reference(monkeypatch, op):
    import rpeflow_b200.install as inst
    fn = getattr(b200, op)
    leaves = _small_args(op, DEV)                    # valid indices: the reference's torch.gather would reject others
    calls = []
    utils = _stand_in_reference(monkeypatch, calls)
    try:
        inst.install(extensions=False, only=set(OPS), train={op})
        inst.stats(reset=True)
        torch.use_deterministic_algorithms(True)
        try:
            with pytest.raises(RuntimeError, match="deterministic"):
                fn(*leaves)
            getattr(utils, op)(*leaves)
        finally:
            torch.use_deterministic_algorithms(False)
        assert calls == [op] and inst.stats()[op] == {"b200": 0, "reference": 1}
        out = getattr(utils, op)(*leaves)
        assert out.grad_fn is not None and calls == [op] and inst.stats()[op] == {"b200": 1, "reference": 1}
    finally:
        inst.uninstall()


@pytest.mark.gpu
@pytest.mark.parametrize("op", OPS)
def test_install_train_routes_graph_calls_here_only_when_named(monkeypatch, op):
    import rpeflow_b200.install as inst
    args = _small_args(op, DEV)
    others = set(OPS) - {op}
    for train, want in ((set(OPS), {"b200": 1, "reference": 0}), (others, {"b200": 0, "reference": 1})):
        calls = []
        utils = _stand_in_reference(monkeypatch, calls)
        try:
            inst.install(extensions=False, only=set(OPS), train=train)
            inst.stats(reset=True)
            out = getattr(utils, op)(*args)
            assert out.grad_fn is not None and inst.stats()[op] == want, (train, inst.stats())
            assert calls == ([] if want["b200"] else [op])
            with torch.no_grad():
                getattr(utils, op)(*args)
            assert inst.stats()[op]["b200"] == want["b200"] + 1
        finally:
            inst.uninstall()
    if op != "grid_sample_wrapper":                  # 2-byte data: always the reference
        calls = []
        utils = _stand_in_reference(monkeypatch, calls)
        try:
            inst.install(extensions=False, only=set(OPS), train=set(OPS))
            inst.stats(reset=True)
            getattr(utils, op)(args[0].detach().half().requires_grad_(True), args[1])
            assert inst.stats()[op] == {"b200": 0, "reference": 1} and calls == [op]
        finally:
            inst.uninstall()
