"""Correlation3D and PointConv backward kernels against float64 references written in this file.

The references below gather with advanced indexing and redo the arithmetic with matmuls in float64 on the CPU; they
share no code with the library or with oracle.torch_ref, and their gradients come from torch.autograd.grad.  The
neighbour indices are made here too (not by the library's KNN), so the tests can aim at the cases where gather-based
backward kernels go wrong:

- shapes at the kernels' tile edges (read from corr3d_bwd.cu / pointconv_bwd.cu, see the case tables);
- scatter collisions: every query selecting the same point, duplicate indices inside a neighbourhood;
- points that no query selects, whose gradients must be exactly zero (the output buffers are handed out of a
  NaN-poisoned caching allocator, so stale memory shows);
- indices at the first and last valid point of each batch, B > 1 with batch-local indices;
- fp16 / bf16 inputs, non-contiguous inputs, the run-to-run reproducibility include/b200flow.h states, and gradcheck.

Every comparison is max|got - ref| <= bar * max|ref| for each gradient tensor (normwise, as fp32 sums of terms of both
signs have no useful elementwise relative error).  Query points whose gradient passes through a pre-activation within
KINK_TAU of that layer's largest magnitude of a ReLU/LeakyReLU kink get a zero upstream gradient: there fp32 and fp64 may
take different slopes, so the gradient is not defined to fp32 accuracy.
"""
import pytest
import torch

import rpeflow_b200 as b200
from rpeflow_b200 import pointconv, pwc3d
from rpeflow_b200._lib import Corr3dWeights, PointConvWeights

DEV = torch.device("cuda", 0)

# fp32 bar.  Both backwards compute in fp32 (FFMA, or 3xTF32 with fp32 accumulation for PointConv's dM = dy.L and
# dL = dy^T.M); a sum of n fp32 terms carries a rounding error of about sqrt(n) * 2^-24 of the terms' magnitude and
# at most n * 2^-24.  The longest sums here are dL over B*S <= 9003 points and dW2 over B*N1*k <= 72000 rows, i.e.
# sqrt(n) * 2^-24 <= 1.6e-5, and every gradient is a chain of two to four such sums.  The sums run over terms of
# both signs whose magnitude is at most that of the result's largest entry, so 2e-5 of max|ref| bounds the error
# with some margin while an error of one lost or doubled term of a 16-long neighbourhood (~6%) is four orders over.
# Measured on a B200: at most 6e-6 over every case of this file.
FP32_BAR = 2e-5
# fp16 / bf16 inputs: the wrappers up-cast to fp32, so the arithmetic is the fp32 path above and the only added error
# is the final rounding of each gradient to the input dtype, at most one unit roundoff u (2^-11 fp16, 2^-8 bf16) of
# the entry.  The reference runs on the same rounded inputs, so input rounding is not an error.  Accumulating in the
# input dtype instead would cost about sqrt(n) * u over the n >= 2000 terms that reach one point in these cases
# (the collision case puts all of them on one address), i.e. > 40 u: far over this bar.
HALF_BAR = {torch.float16: FP32_BAR + 2.0 ** -11, torch.bfloat16: FP32_BAR + 2.0 ** -8}
KINK_TAU = 1e-6
PC_GRADS = ("xyz", "feat", "sampled_xyz") + PointConvWeights.NAMES
C3_GRADS = ("xyz1", "feat1", "xyz2", "feat2") + Corr3dWeights.NAMES


# ------------------------------------------------------------------------------------------------- references
def _lrelu(x):
    return torch.where(x > 0, x, 0.1 * x)


def _relu(x):
    return torch.where(x > 0, x, torch.zeros_like(x))


def _near_kink(z, dims, tau):
    """bool over the leading dims of z: some entry within tau * max|z| of 0."""
    near = z.abs() < tau * z.abs().max()
    return near.flatten(dims).any(dim=dims)


def ref_pointconv(xyz, feat, sampled, knn, w, tau=KINK_TAU):
    """LeakyReLU(0.1) of PointConv's Linear output, [B,Cout,S], and a [B,Cout,S] mask of the outputs whose gradient is
    defined to fp32 accuracy.  xyz [B,3,N], feat [B,C,N], sampled [B,3,S], knn [B,S,k] local to each batch."""
    B = xyz.shape[0]
    bi = torch.arange(B)[:, None, None]
    rel = xyz.transpose(1, 2)[bi, knn] - sampled.transpose(1, 2)[:, :, None, :]        # [B,S,k,3]
    z1 = rel @ w["Wa"].T + w["ba"]
    z2 = _lrelu(z1) @ w["Wb"].T + w["bb"]                                               # [B,S,k,16]
    rows = torch.cat([xyz, feat], 1).transpose(1, 2)[bi, knn]                           # [B,S,k,C+3]
    mixed = (_lrelu(z2).transpose(2, 3) @ rows).flatten(2)                              # [B,S,16*(C+3)], w-major
    y = (mixed @ w["L"].T + w["bias"]).transpose(1, 2)                                  # [B,Cout,S]
    ok = ~(_near_kink(z1, 2, tau) | _near_kink(z2, 2, tau))[:, None, :] & (y.abs() >= tau * y.abs().max())
    return _lrelu(y), ok


def ref_corr3d(xyz1, feat1, xyz2, feat2, knn12, knn11, w, tau=KINK_TAU):
    """Correlation3D output [B,Cout,N1] and a [B,Cout,N1] mask of the outputs whose gradient is defined to fp32
    accuracy.  knn12 [B,N1,k] into cloud 2, knn11 [B,N1,k] into cloud 1, both local to each batch."""
    B, _, N1 = feat1.shape
    k = knn12.shape[2]
    bi = torch.arange(B)[:, None, None]
    p1 = xyz1.transpose(1, 2)
    d = xyz2.transpose(1, 2)[bi, knn12] - p1[:, :, None, :]                             # [B,N1,k,3]
    f1 = feat1.transpose(1, 2)[:, :, None, :].expand(-1, -1, k, -1)
    x = torch.cat([f1, feat2.transpose(1, 2)[bi, knn12], d], -1)                        # [B,N1,k,2Cin+3]
    z1 = x @ w["W1"].T + w["b1"]
    z2 = _lrelu(z1) @ w["W2"].T + w["b2"]
    flags = [_near_kink(z1, 2, tau), _near_kink(z2, 2, tau)]

    def weight_net(v, tag, flags):
        for letter in "abc":
            v = v @ w[f"{tag}_W{letter}"].T + w[f"{tag}_b{letter}"]
            flags.append(_near_kink(v, 2, tau))
            v = _relu(v)
        return v                                                                        # [B,N1,k,Cout]

    P = (weight_net(d, "n2", flags) * _lrelu(z2)).sum(2)                                # [B,N1,Cout]
    fragile_p = torch.stack(flags).any(0)                                               # [B,N1]
    flags1 = []
    w1 = weight_net(p1[bi, knn11] - p1[:, :, None, :], "n1", flags1)
    out = (w1 * P[bi, knn11]).sum(2).transpose(1, 2)                                    # [B,Cout,N1]
    fragile = torch.stack(flags1).any(0) | fragile_p[bi, knn11].any(2)
    return out, ~fragile[:, None, :].expand_as(out)


def ref_grads(fn, inputs, weights, grad):
    """fp64 CPU autograd of fn(*inputs, weights) with upstream grad * (its own kink mask): (mask, {name: gradient})."""
    leaves = {n: t.detach().to(torch.float64).requires_grad_(True) for n, t in inputs.items()}
    wts = {n: t.detach().to(torch.float64).requires_grad_(True) for n, t in weights.items()}
    out, ok = fn(*leaves.values(), wts)
    g = grad.to(torch.float64) * ok
    names = list(leaves) + list(wts)
    got = torch.autograd.grad(out, list(leaves.values()) + list(wts.values()), g)
    return ok, dict(zip(names, got))


# ------------------------------------------------------------------------------------------------- cases
def _uniform(gen, shape, fan_in):
    bound = fan_in ** -0.5                             # the default init of nn.Conv2d / nn.Linear
    return (torch.rand(shape, generator=gen, dtype=torch.float64) * 2 - 1) * bound


def _indices(kind, B, Q, k, N, gen):
    """[B,Q,k] int64 neighbour indices into a cloud of N points (local to each batch)."""
    if kind == "random":                               # k > N repeats indices too
        return torch.randint(0, N, (B, Q, k), generator=gen)
    if kind == "same":                                 # every neighbour of every query: the batch's last point
        return torch.full((B, Q, k), N - 1, dtype=torch.int64)
    if kind == "dups":                                 # each neighbourhood draws its k indices from 3 points
        pool = torch.randint(0, N, (B, Q, 3), generator=gen)
        return torch.gather(pool, 2, torch.randint(0, 3, (B, Q, k), generator=gen))
    if kind == "edges":                                # only the first and the last valid index of each batch
        return torch.where(torch.rand(B, Q, k, generator=gen) < 0.5, 0, N - 1)
    if kind == "even":                                 # odd points are never selected
        return 2 * torch.randint(0, (N + 1) // 2, (B, Q, k), generator=gen)
    raise ValueError(kind)


def pc_case(B, C, Cout, N, S, knn="random", seed=0):
    gen = torch.Generator().manual_seed(seed)
    inputs = {"xyz": torch.rand(B, 3, N, generator=gen), "feat": torch.randn(B, C, N, generator=gen),
              "sampled_xyz": torch.rand(B, 3, S, generator=gen)}
    w = {"Wa": _uniform(gen, (8, 3), 3), "ba": _uniform(gen, (8,), 3), "Wb": _uniform(gen, (16, 8), 8),
         "bb": _uniform(gen, (16,), 8), "L": _uniform(gen, (Cout, 16 * (C + 3)), 16 * (C + 3)),
         "bias": _uniform(gen, (Cout,), 16 * (C + 3))}
    w = {n: t.float() for n, t in w.items()}
    return inputs, w, _indices(knn, B, S, 16, N, gen), torch.randn(B, Cout, S, generator=gen)


def c3_case(B, Cin, Cout, N1, N2, k, knn="random", seed=0):
    gen = torch.Generator().manual_seed(seed)
    inputs = {"xyz1": torch.rand(B, 3, N1, generator=gen), "feat1": torch.randn(B, Cin, N1, generator=gen),
              "xyz2": torch.rand(B, 3, N2, generator=gen), "feat2": torch.randn(B, Cin, N2, generator=gen)}
    w = {"W1": _uniform(gen, (Cout, 2 * Cin + 3), 2 * Cin + 3), "b1": _uniform(gen, (Cout,), 2 * Cin + 3),
         "W2": _uniform(gen, (Cout, Cout), Cout), "b2": _uniform(gen, (Cout,), Cout)}
    for tag in ("n1", "n2"):
        for letter, (o, i) in zip("abc", ((8, 3), (8, 8), (Cout, 8))):
            w[f"{tag}_W{letter}"], w[f"{tag}_b{letter}"] = _uniform(gen, (o, i), i), _uniform(gen, (o,), i)
    w = {n: t.float() for n, t in w.items()}
    knn12 = _indices(knn, B, N1, k, N2, gen)
    knn11 = _indices(knn, B, N1, k, N1, gen)
    return inputs, w, knn12, knn11, torch.randn(B, Cout, N1, generator=gen)


def _poison_allocator(nbytes=64 << 20):
    """Leave NaN-filled blocks in the CUDA caching allocator, so that an output the kernel fails to write shows."""
    blocks = [torch.full((n,), float("nan"), device=DEV) for n in (nbytes // 4, 1 << 16, 1 << 12, 256)]
    del blocks


def gpu_pointconv(inputs, w, knn, grad, dtype=torch.float32, want=PC_GRADS):
    """pointconv.pointconv on the GPU (inputs and weights in dtype), backward of grad: {name: gradient or None}."""
    leaves = {n: t.to(DEV, dtype).requires_grad_(n in want) for n, t in inputs.items()}
    wts = {n: t.to(DEV, dtype).requires_grad_(n in want) for n, t in w.items()}
    _poison_allocator()
    out = pointconv.pointconv(leaves["xyz"], leaves["feat"], leaves["sampled_xyz"], knn.to(DEV), wts)
    out.backward(grad.to(DEV, out.dtype))
    torch.cuda.synchronize()
    return {n: t.grad for n, t in list(leaves.items()) + list(wts.items())}


def gpu_corr3d(inputs, w, knn12, knn11, grad, dtype=torch.float32, want=C3_GRADS):
    leaves = {n: t.to(DEV, dtype).requires_grad_(n in want) for n, t in inputs.items()}
    wts = {n: t.to(DEV, dtype).requires_grad_(n in want) for n, t in w.items()}
    _poison_allocator()
    out = b200.correlation3d(leaves["xyz1"], leaves["feat1"], leaves["xyz2"], leaves["feat2"], wts, knn12.to(DEV),
                             knn11.to(DEV))
    out.backward(grad.to(DEV, out.dtype))
    torch.cuda.synchronize()
    return {n: t.grad for n, t in list(leaves.items()) + list(wts.items())}


def assert_close(got, ref, bar, label, dtype=torch.float32):
    """max|got - ref| <= bar * max|ref| per gradient; an all-zero reference must be matched exactly."""
    ratios = {}
    for n, r in ref.items():
        g = got[n]
        assert g is not None and tuple(g.shape) == tuple(r.shape), f"{label}: {n} missing or misshaped"
        assert g.dtype == dtype, f"{label}: grad {n} is {g.dtype}, its input is {dtype}"
        diff = (g.detach().double().cpu() - r).abs().max().item() if r.numel() else 0.0
        scale = r.abs().max().item() if r.numel() else 0.0
        ratios[n] = diff / scale if scale > 0 else (0.0 if diff == 0 else float("inf"))
    print(f"\n[{label}] max|diff| / max|ref|: " + " ".join(f"{n}={v:.2g}" for n, v in ratios.items()))
    bad = {n: v for n, v in ratios.items() if not v <= bar}
    assert not bad, f"{label}: over {bar:g} of max|ref|: {bad}"


def check_pointconv(case, label, dtype=torch.float32, bar=FP32_BAR):
    inputs, w, knn, grad = case
    if dtype != torch.float32:                         # the reference sees the same rounded values
        inputs = {n: t.to(dtype).float() for n, t in inputs.items()}
        w = {n: t.to(dtype).float() for n, t in w.items()}
    ok, ref = ref_grads(lambda x, f, s, wt: ref_pointconv(x, f, s, knn, wt), inputs, w, grad)
    got = gpu_pointconv(inputs, w, knn, grad * ok, dtype)
    assert_close(got, ref, bar, label, dtype)
    return got, ref


def check_corr3d(case, label, dtype=torch.float32, bar=FP32_BAR):
    inputs, w, knn12, knn11, grad = case
    if dtype != torch.float32:
        inputs = {n: t.to(dtype).float() for n, t in inputs.items()}
        w = {n: t.to(dtype).float() for n, t in w.items()}
    ok, ref = ref_grads(lambda x1, f1, x2, f2, wt: ref_corr3d(x1, f1, x2, f2, knn12, knn11, wt), inputs, w, grad)
    got = gpu_corr3d(inputs, w, knn12, knn11, grad * ok, dtype)
    assert_close(got, ref, bar, label, dtype)
    return got, ref


# ------------------------------------------------------------------------------------------------- CPU
def test_references_compute_the_model_operations():
    """The references here are the model's operations: fp64 forward equal to oracle.torch_ref's op graph."""
    from oracle import torch_ref
    inputs, w, knn, _ = pc_case(2, 5, 7, 40, 30, seed=1)
    d = {n: t.double() for n, t in inputs.items()}
    wd = {n: t.double() for n, t in w.items()}
    want = torch_ref.pointconv(d["xyz"], d["feat"], d["sampled_xyz"], wd, k=16, knn=knn)
    torch.testing.assert_close(ref_pointconv(d["xyz"], d["feat"], d["sampled_xyz"], knn, wd)[0], want,
                               rtol=1e-12, atol=1e-12)
    inputs, w, knn12, knn11, _ = c3_case(2, 5, 7, 30, 20, 4, seed=1)
    d = {n: t.double() for n, t in inputs.items()}
    wd = {n: t.double() for n, t in w.items()}
    want = torch_ref.correlation3d(d["xyz1"], d["feat1"], d["xyz2"], d["feat2"], wd, k=4, knn11=knn11, knn12=knn12)
    torch.testing.assert_close(ref_corr3d(*d.values(), knn12, knn11, wd)[0], want, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------------------- PointConv
# pointconv_bwd.cu: k = 16 only; the dM / dL GEMMs take 128-point x 128-column tiles and K blocks of 16 (over Cout for
# dM, over the chunk's points for dL); the point kernel runs 4 points per CTA and walks Cp = roundup16(C+3) channels in
# blocks of 32; points are walked in chunks of floor(32 MB / (64 Cp) / 128) * 128 that run across batch boundaries.
# name: (B, C, Cout, N, S)
PC_SHAPES = {
    "N1_S1": (1, 8, 32, 1, 1),                  # one point, one query: every index is 0
    "B3_S7_C13": (3, 13, 64, 50, 7),             # C+3 = 16: no channel padding
    "S127_C1": (1, 1, 64, 300, 127),             # one short of a GEMM point tile
    "B3_S128_C3": (3, 3, 128, 300, 128),         # exactly one tile per batch
    "B3_S129_C29_Cout129": (3, 29, 129, 400, 129),   # C+3 = 32: one channel block; Cout one over a 128-row tile
    "B3_S3001_C30": (3, 30, 64, 4000, 3001),     # C+3 = 33 spills into a second channel block; prime S
    "C195_Cout128": (2, 195, 128, 600, 333),     # the flow estimator's first body
    "C64_Cout1": (1, 64, 1, 200, 77),            # dM's K = Cout = 1: a single, mostly empty K block
    "C96_Cout256": (1, 96, 256, 300, 150),       # the largest Cout
    "B3_two_chunks_C509": (3, 509, 40, 500, 400),    # Cp = 512: 1024-point chunks, B*S = 1200 -> 1024 + 176
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PC_SHAPES))
def test_pointconv_gradients_at_tile_edges(name):
    check_pointconv(pc_case(*PC_SHAPES[name], seed=len(name)), name)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["same", "dups", "edges"])
def test_pointconv_gradients_with_colliding_neighbours(kind):
    """same: the 3*300*16 neighbour slots of all queries all name the last point of their batch."""
    check_pointconv(pc_case(3, 24, 64, 200, 300, knn=kind, seed=3), kind)


@pytest.mark.gpu
def test_pointconv_unselected_points_get_exactly_zero():
    got, _ = check_pointconv(pc_case(3, 21, 64, 301, 500, knn="even", seed=4), "even")
    for n in ("xyz", "feat"):
        assert torch.count_nonzero(got[n][:, :, 1::2]) == 0, n


# ------------------------------------------------------------------------------------------------- Correlation3D
# corr3d_bwd.cu: k in [1, 32] (register arrays of 4, 8, 16 or 32); the stage-2 pass takes 16 points per tile, the stage-1
# pass floor(128 / k) points (halved while its shared memory exceeds 200 KB, so 4 at Cout = 192), channels padded to 4;
# a warp-wide reduction is used only when Cout % 32 == 0; the linear backward tiles are 64 x 64 with 16-deep K blocks.
# name: (B, Cin, Cout, N1, N2, k)
C3_SHAPES = {
    "N1_k1": (1, 8, 16, 1, 1, 1),
    "B3_N7_k5_Cout5": (3, 3, 5, 7, 9, 5),         # Cout padded 5 -> 8
    "N15_Cin1_Cout33": (1, 1, 33, 15, 40, 16),    # one short of a stage-2 tile; no warp reduction
    "B3_N16": (3, 32, 32, 16, 16, 16),
    "B3_N17_k17_Cin17": (3, 17, 64, 17, 30, 17),  # one over a stage-2 tile; k = 17 on the 32-row path
    "k32": (2, 64, 64, 100, 120, 32),
    "k4_N129": (2, 20, 36, 129, 64, 4),           # one over two linear-backward tiles
    "B3_N1500": (3, 32, 64, 1500, 1300, 16),      # the model's k and a level-5-like width; N1 % 8 != 0
    "C192": (1, 192, 192, 203, 190, 16),          # the widest level: 4-point stage-1 tiles, N1 % 4 != 0
    "Cout3_N2_below_k": (2, 5, 3, 50, 10, 16),    # every neighbourhood repeats indices
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(C3_SHAPES))
def test_corr3d_gradients_at_tile_edges(name):
    check_corr3d(c3_case(*C3_SHAPES[name], seed=len(name)), name)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["same", "dups", "edges"])
def test_corr3d_gradients_with_colliding_neighbours(kind):
    """same: all 3*150*16 slots of knn12 name the last point of cloud 2, all of knn11 the last point of cloud 1."""
    check_corr3d(c3_case(3, 16, 32, 150, 120, 16, knn=kind, seed=3), kind)


@pytest.mark.gpu
def test_corr3d_unselected_points_get_exactly_zero():
    """Cloud-2 points outside knn12 get no gradient.  (Every cloud-1 point is a query, so its gradients are not 0.)"""
    got, _ = check_corr3d(c3_case(3, 16, 32, 150, 121, 16, knn="even", seed=4), "even")
    for n in ("xyz2", "feat2"):
        assert torch.count_nonzero(got[n][:, :, 1::2]) == 0, n


# ------------------------------------------------------------------------------------------------- dtypes, layouts
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("op", ["pointconv", "corr3d"])
def test_reduced_precision_inputs(op, dtype):
    """~2000 queries per batch select each point ~64 times (pointconv) / ~16 times per cloud (corr3d)."""
    if op == "pointconv":
        check_pointconv(pc_case(2, 32, 64, 500, 2000, seed=5), f"pointconv-{dtype}", dtype, HALF_BAR[dtype])
    else:
        check_corr3d(c3_case(2, 32, 64, 2000, 1800, 16, seed=5), f"corr3d-{dtype}", dtype, HALF_BAR[dtype])


def _strided(t, how):
    """A non-contiguous CUDA leaf holding t's values: "T" transposes the last two dims of storage, "batch" slices every
    other batch of a larger tensor, "chan" is a channel slice."""
    if how == "T":
        v = t.transpose(-1, -2).contiguous().to(DEV).transpose(-1, -2)
    elif how == "batch":
        big = torch.zeros((2 * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype)
        big[::2] = t
        v = big.to(DEV)[::2]
    else:
        big = torch.zeros((t.shape[0], t.shape[1] + 2) + tuple(t.shape[2:]), dtype=t.dtype)
        big[:, 1:-1] = t
        v = big.to(DEV)[:, 1:-1]
    assert not v.is_contiguous()
    return v.requires_grad_(t.is_floating_point())


@pytest.mark.gpu
def test_pointconv_non_contiguous_inputs():
    inputs, w, knn, grad = pc_case(3, 20, 48, 300, 200, seed=7)
    ok, ref = ref_grads(lambda x, f, s, wt: ref_pointconv(x, f, s, knn, wt), inputs, w, grad)
    leaves = {"xyz": _strided(inputs["xyz"], "T"), "feat": _strided(inputs["feat"], "batch"),
              "sampled_xyz": _strided(inputs["sampled_xyz"], "chan")}
    wts = {n: (_strided(t, "T") if t.dim() == 2 else t.to(DEV).requires_grad_(True)) for n, t in w.items()}
    knn32 = _strided(knn.to(torch.int32), "T")
    out = pointconv.pointconv(leaves["xyz"], leaves["feat"], leaves["sampled_xyz"], knn32, wts)
    out.backward(_strided(grad * ok, "T").detach())
    assert_close({n: t.grad for n, t in list(leaves.items()) + list(wts.items())}, ref, FP32_BAR, "strided")
    # the autograd Function itself takes dense fp32 only, and says so instead of reading the wrong memory
    params = [wts[n] for n in PointConvWeights.NAMES]
    with pytest.raises(ValueError, match="contiguous"):
        pointconv.PointConvFunction.apply(leaves["xyz"], leaves["feat"], leaves["sampled_xyz"], knn.to(DEV), 2, *params)
    dense = [p.detach().contiguous() for p in params]
    with pytest.raises(ValueError, match="int64"):
        pointconv.PointConvFunction.apply(*(t.detach().contiguous() for t in leaves.values()), knn32.contiguous(), 2,
                                          *dense)


@pytest.mark.gpu
def test_corr3d_non_contiguous_inputs():
    inputs, w, knn12, knn11, grad = c3_case(3, 12, 32, 200, 150, 16, seed=7)
    ok, ref = ref_grads(lambda x1, f1, x2, f2, wt: ref_corr3d(x1, f1, x2, f2, knn12, knn11, wt), inputs, w, grad)
    leaves = {"xyz1": _strided(inputs["xyz1"], "T"), "feat1": _strided(inputs["feat1"], "batch"),
              "xyz2": _strided(inputs["xyz2"], "chan"), "feat2": _strided(inputs["feat2"], "T")}
    wts = {n: (_strided(t, "T") if t.dim() == 2 else t.to(DEV).requires_grad_(True)) for n, t in w.items()}
    k12, k11 = _strided(knn12, "batch"), _strided(knn11.to(torch.int32), "T")
    out = b200.correlation3d(*leaves.values(), wts, k12, k11)
    out.backward(_strided(grad * ok, "T").detach())
    assert_close({n: t.grad for n, t in list(leaves.items()) + list(wts.items())}, ref, FP32_BAR, "strided")
    params = [wts[n] for n in Corr3dWeights.NAMES]
    with pytest.raises(ValueError, match="contiguous"):
        pwc3d.Correlation3DFunction.apply(*leaves.values(), knn12.to(DEV), knn11.to(DEV), 2, *params)
    with pytest.raises(ValueError, match="float32"):
        pwc3d.Correlation3DFunction.apply(*(t.detach().contiguous().half() for t in leaves.values()), knn12.to(DEV),
                                          knn11.to(DEV), 2, *(p.detach().contiguous() for p in params))


@pytest.mark.gpu
def test_unsupported_neighbour_counts_raise():
    inputs, w, knn, grad = pc_case(1, 8, 16, 40, 20, seed=8)
    args = [inputs[n].to(DEV).requires_grad_(True) for n in ("xyz", "feat", "sampled_xyz")]
    with pytest.raises(RuntimeError, match="k = 16"):
        pointconv.pointconv(*args, knn[:, :, :8].to(DEV), {n: t.to(DEV) for n, t in w.items()})
    inputs, w, knn12, knn11, grad = c3_case(1, 8, 16, 40, 40, 33, seed=8)
    args = [t.to(DEV).requires_grad_(True) for t in inputs.values()]
    with pytest.raises(RuntimeError, match=r"k must be in \[1,32\]"):
        b200.correlation3d(*args, {n: t.to(DEV) for n, t in w.items()}, knn12.to(DEV), knn11.to(DEV))


# ------------------------------------------------------------------------------------------------- determinism
@pytest.mark.gpu
def test_pointconv_parameter_gradients_are_bit_reproducible():
    """include/b200flow.h: the six parameter gradients are per-CTA partials reduced in a fixed order, so two runs agree
    bit for bit.  xyz, feat and sampled_xyz are summed with float atomics whose order varies from run to run, so they
    are only held to the tolerance.  B*S = 9000 > the 8192-point chunk of C = 48: two chunks."""
    case = pc_case(3, 48, 64, 2000, 3000, seed=11)
    first, ref = check_pointconv(case, "run 1")
    second, _ = check_pointconv(case, "run 2")
    for n in PointConvWeights.NAMES:
        assert torch.equal(first[n], second[n]), n


@pytest.mark.gpu
def test_corr3d_weight_net1_hidden_gradients_are_bit_reproducible():
    """include/b200flow.h: weight_net1's 3->8->8 gradients are thread-owned sums of values computed without atomics,
    reduced in a fixed order, so two runs agree bit for bit.  Every other gradient reads a float-atomic sum (dP, dG2,
    the clouds, split-K dW1 / db1, the shared-memory Wc / bc / W1c / b2 partials), so it is only held to the tolerance."""
    case = c3_case(3, 32, 64, 1500, 1300, 16, seed=11)
    first, _ = check_corr3d(case, "run 1")
    second, _ = check_corr3d(case, "run 2")
    for n in ("n1_Wa", "n1_ba", "n1_Wb", "n1_bb"):
        assert torch.equal(first[n], second[n]), n


# ------------------------------------------------------------------------------------------------- gradcheck
def _kink_free(ref, tau, seeds, make):
    """The first case from make(seed) whose pre-activations all lie farther than tau * (their layer's max) from a kink,
    so that finite differences of step << tau do not cross one."""
    for seed in seeds:
        case = make(seed)
        _, ok = ref(case, tau)
        if bool(ok.all()):
            return case
    raise AssertionError("no kink-free case")


@pytest.mark.gpu
def test_pointconv_gradcheck():
    """The kernels compute in fp32 only: pointconv() takes fp64 leaves but casts them to fp32, so this gradcheck uses
    a loose step and tolerance.  eps = 1e-4; fp32 rounding of the outputs (~1e-7 of max|y| ~ 0.9, a few roundings) over
    2 eps gives ~1e-3 of noise, hence atol = 5e-3, rtol = 1e-2.  The case has no pre-activation within 2e-3 of its layer's max of a kink, 20x the
    largest shift a step causes, and the check of two backward runs allows the atomics' rounding (nondet_tol)."""
    def make(seed):
        inputs, w, knn, _ = pc_case(1, 2, 3, 6, 2, seed=seed)
        return {n: t.double() for n, t in inputs.items()}, {n: t.double() for n, t in w.items()}, knn

    def ref(case, tau):
        x, w, knn = case
        out, ok = ref_pointconv(x["xyz"], x["feat"], x["sampled_xyz"], knn, w, tau)
        return out, ok & (out.abs().max() > 0.5)

    x, w, knn = _kink_free(ref, 2e-3, range(200), make)
    leaves = [t.to(DEV).requires_grad_(True) for t in list(x.values()) + [w[n] for n in PointConvWeights.NAMES]]
    knn = knn.to(DEV)

    def fn(*ts):
        return pointconv.pointconv(ts[0], ts[1], ts[2], knn, dict(zip(PointConvWeights.NAMES, ts[3:])))
    assert torch.autograd.gradcheck(fn, leaves, eps=1e-4, atol=5e-3, rtol=1e-2, nondet_tol=1e-5)


@pytest.mark.gpu
def test_corr3d_gradcheck():
    """As test_pointconv_gradcheck (fp32 arithmetic behind fp64 leaves, eps = 1e-4) on a case small enough to have no
    pre-activation near a kink: B = 1, N1 = 2, N2 = 3, k = 2, Cin = 2, Cout = 3.  Its outputs are ~0.1, so the fp32
    noise of a difference quotient is ~1e-4: atol = 1e-3, rtol = 1e-2."""
    def make(seed):
        inputs, w, knn12, knn11, _ = c3_case(1, 2, 3, 2, 3, 2, seed=seed)
        return {n: t.double() for n, t in inputs.items()}, {n: t.double() for n, t in w.items()}, knn12, knn11

    def ref(case, tau):
        x, w, knn12, knn11 = case
        out, ok = ref_corr3d(*x.values(), knn12, knn11, w, tau)
        return out, ok & (out.abs().max() > 0.1)           # skip cases whose ReLU nets are all but dead

    x, w, knn12, knn11 = _kink_free(ref, 2e-3, range(500), make)
    leaves = [t.to(DEV).requires_grad_(True) for t in list(x.values()) + [w[n] for n in Corr3dWeights.NAMES]]
    knn12, knn11 = knn12.to(DEV), knn11.to(DEV)

    def fn(*ts):
        return b200.correlation3d(*ts[:4], dict(zip(Corr3dWeights.NAMES, ts[4:])), knn12, knn11)
    assert torch.autograd.gradcheck(fn, leaves, eps=1e-4, atol=1e-3, rtol=1e-2, nondet_tol=1e-5)
