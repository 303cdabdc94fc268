"""Correlation3D and PointConv forward kernels against the float64 references of test_backward_reference.py.

The references (ref_corr3d, ref_pointconv), the case builders and the NaN-poisoning allocator are imported from
test_backward_reference.py, so forward and backward are held to one float64 definition of each operation.  Every case
below names the route it is meant to reach, read from the eligibility code of the library:

- Correlation3D (corr3d.cu b200_corr3d_fwd): "v2<NW,DEPTH>" = corr3d_v2.cu, taken when Cin == Cout, precision 2, k = 16
  and C % 32 == 0 with 32 <= C <= 192 (corr3d_v2_eligible; NW,DEPTH = 4,1 up to C = 128, 8,2 above); otherwise
  "tc<SPLIT>" = corr3d_stage1_tc_kernel at precision 1 (SPLIT 0) or 2 (SPLIT 1) when k = 16 and Cout % 32 == 0 with
  Cout <= 256 (corr3d_stage1_tc_eligible); otherwise "fp32<KMAX>" = corr3d_stage1_kernel<4/8/16/32> by k (launch_stage1).
- PointConv (pointconv.cu b200_pointconv_fwd): "v2<MODE,WIDE>" = pointconv_v2_kernel<MODE,WIDE>: MODE 0 at precision 1
  (TF32), MODE 1 at precisions 0 and 2 when roundup32(Cout) <= 128 (3xTF32, B halves stacked along N), MODE 2 above
  (three MMAs, shallower ring); WIDE = N > 65536 (uint32 neighbour indices instead of uint16, which leave room for one
  ring stage fewer at some widths: a single stage at MODE 2 with Cout = 256).
test_every_case_reaches_its_route checks each claim against the kernels torch.profiler sees launched.

Comparison.  Per sample b: max|got - ref| <= bar * max|ref| over that sample's outputs (normwise: fp32 sums of terms of
both signs have no useful elementwise relative error; per sample, so that one broken sample of small scale is not hidden
by a large one).  Outputs are handed out of a NaN-poisoned caching allocator (so is the scratch: Fpm, Limg, A1/G2/P and
the v2 weight images), so an output the kernel does not write, or a padding row or column read before it is written,
shows as NaN and fails the bar.

fp32-class bar (Correlation3D precisions 0 and 2, PointConv precisions 0 and 2): FP32_BAR = 2e-5.  These routes compute
in fp32 FFMA, or in 3xTF32 on tcgen05: a = hi + lo with hi = a truncated to TF32 (10 explicit mantissa bits) and lo = a - hi
exact, and a.b ~ hi.hi + hi.lo + lo.hi accumulated in fp32.  The dropped lo.lo term and the truncation of lo to TF32
when it is an operand are each below 2^-20 of |a.b|, so a product carries < 3 * 2^-20 ~ 3e-6 relative error, of either
sign from product to product except for a small systematic shrink.  The outputs are sums of n such products (n = Cin,
Cout <= 512, k <= 32 for Correlation3D, 16 * (C+3) <= 8192 for PointConv's Linear); a sum of n random-sign terms is
itself ~ sqrt(n) times a term, the same growth as its accumulated error, so the error stays ~1e-6 of max|y| per layer,
and the two to four chained layers add, not multiply.  2e-5 leaves margin over that, while one lost or doubled term of a
16-neighbour sum (~6 %) or a wrong bias is three orders of magnitude over it.

Long tensor-core contractions (PointConv's Linear, K = 16 * (C+3) up to 8192): on top of the bar, K / 8 * 2^-23 of max|y|.
tcgen05.mma adds each k-step of 8 products to the fp32 accumulator with a truncation of up to 2^-23 (mean 2^-24) of the
running sum, always towards zero, so over K / 8 steps these errors add up linearly instead of cancelling.  Measured on a
B200 the 3xTF32 error of PointConv grows just so: ~8e-9 * K of max|y| (6.6e-6 at C = 30, 2.7e-5 at C = 195, 5.9e-5 to
7.3e-5 at C = 509), i.e. (K / 8) * 2^-24 within the spread of the data.  Correlation3D's tcgen05 contractions have
K <= 256, where the term is below 4e-6 and inside the bar.  The accumulation is the tensor cores' own; splitting the
Linear's K loop over several accumulators would shrink it, and this term with it.

TF32 bar (precision 1: Correlation3D's Cout x Cout layer W2.h1 on tcgen05, PointConv's Linear on tcgen05; everything else
fp32): TF32_BAR = 2^-8 ~ 3.9e-3.  The tensor cores read only the top 10 mantissa bits of an fp32 operand, i.e. each
operand is truncated by a relative amount uniform in [0, 2^-10), so a product is shrunk by a relative amount in [0, 2^-9):
mean 2^-10, standard deviation 2^-10 / sqrt(6) ~ 4e-4.  A sum y = sum t_i is then off by ~ -2^-10 * y (the mean, a
fraction of y itself) plus a zero-mean part of standard deviation ~ 4e-4 * sqrt(sum t_i^2), and sqrt(sum t_i^2) is of the
order of a typical |y|, below max|y| of the sample.  That is ~ 2^-10 + 3 * 4e-4 ~ 2.2e-3 of max|y| at three standard
deviations; the ReLU / LeakyReLU and the positive-weighted neighbour sums after the layer do not enlarge it normwise.
The bar is 2^-8, about 1.8 times that, and still 15 times below one lost neighbour term.

Measured on a B200 at its 1000 W power limit (largest ratio per route and precision over every case of this file):
  Correlation3D  v2<4,1> p2 4.6e-6, v2<8,2> p2 5.3e-6, tc<1> p2 2.8e-6, tc<0> p1 2.3e-3, fp32<4/8/16/32> p0/p1/p2 9.3e-7
  PointConv      v2<1,false> p0/p2 5.1e-5 (C = 509; 3.7e-6 up to C = 29), v2<2,false> p0/p2 7.3e-5 (C = 509; 6.7e-6 at
                 C = 30), v2<1,true> p0/p2 4.6e-6 (C = 29), v2<2,true> p0/p2 7.1e-6 (C = 30), v2<0,false> p1 1.0e-3,
                 v2<0,true> p1 9.0e-4

Exact properties, bit for bit: a batched call equals the B single-sample calls (at the benchmark's batch of 148, where
every persistent v2 CTA runs dozens of items); b200_pointconv_fwd equals LeakyReLU(0.1) of b200_pointconv_fwd_linear;
PointConv precision 0 equals precision 2.  Permuting the neighbours inside each neighbourhood changes only the order of
the fp32 sums, so it is held to the route's bar.  Out-of-range neighbour indices follow the rules include/b200flow.h
states: Correlation3D clamps to [0, N-1]; PointConv wraps a negative index once (+N) and then clamps.
"""
import functools
import re
import zlib

import pytest
import torch
import torch.nn.functional as F

from rpeflow_b200 import pointconv, pwc3d
from rpeflow_b200._lib import B200Error
from rpeflow_b200.workload import LEVEL_CHANNELS, PYRAMID_POINTS
from test_backward_reference import DEV, _indices, _poison_allocator, _uniform, ref_corr3d, ref_pointconv

FP32_BAR = 2e-5
TF32_BAR = 2.0 ** -8
TF32_ROUTES = {("corr3d", "tc<0>"), ("pointconv", "v2<0,false>"), ("pointconv", "v2<0,true>")}
MEASURED = {}                                           # (op, route, precision) -> largest ratio seen


# ------------------------------------------------------------------------------------------------- cases
def _seed(name):
    return zlib.crc32(name.encode())


def c3_inputs(B, Cin, Cout, N1, N2, k, kind, seed):
    gen = torch.Generator().manual_seed(seed)
    inputs = {"xyz1": torch.rand(B, 3, N1, generator=gen), "feat1": torch.randn(B, Cin, N1, generator=gen),
              "xyz2": torch.rand(B, 3, N2, generator=gen), "feat2": torch.randn(B, Cin, N2, generator=gen)}
    w = {"W1": _uniform(gen, (Cout, 2 * Cin + 3), 2 * Cin + 3), "b1": _uniform(gen, (Cout,), 2 * Cin + 3),
         "W2": _uniform(gen, (Cout, Cout), Cout), "b2": _uniform(gen, (Cout,), Cout)}
    for tag in ("n1", "n2"):
        for letter, (o, i) in zip("abc", ((8, 3), (8, 8), (Cout, 8))):
            w[f"{tag}_W{letter}"], w[f"{tag}_b{letter}"] = _uniform(gen, (o, i), i), _uniform(gen, (o,), i)
    w = {n: t.float() for n, t in w.items()}
    return inputs, w, _indices(kind, B, N1, k, N2, gen), _indices(kind, B, N1, k, N1, gen)


def pc_inputs(B, C, Cout, N, S, kind, seed):
    gen = torch.Generator().manual_seed(seed)
    inputs = {"xyz": torch.rand(B, 3, N, generator=gen), "feat": torch.randn(B, C, N, generator=gen),
              "sampled_xyz": torch.rand(B, 3, S, generator=gen)}
    w = {"Wa": _uniform(gen, (8, 3), 3), "ba": _uniform(gen, (8,), 3), "Wb": _uniform(gen, (16, 8), 8),
         "bb": _uniform(gen, (16,), 8), "L": _uniform(gen, (Cout, 16 * (C + 3)), 16 * (C + 3)),
         "bias": _uniform(gen, (Cout,), 16 * (C + 3))}
    return inputs, {n: t.float() for n, t in w.items()}, _indices(kind, B, S, 16, N, gen)


def _f64(d):
    return {n: t.double() for n, t in d.items()}


def c3_reference(inputs, w, knn12, knn11):
    x = _f64(inputs)
    return ref_corr3d(x["xyz1"], x["feat1"], x["xyz2"], x["feat2"], knn12, knn11, _f64(w))[0]


def pc_reference(inputs, w, knn):
    """LeakyReLU(y) from ref_pointconv, and y itself (LeakyReLU(0.1) inverted in float64)."""
    x = _f64(inputs)
    out = ref_pointconv(x["xyz"], x["feat"], x["sampled_xyz"], knn, _f64(w))[0]
    return out, torch.where(out > 0, out, out / 0.1)


def _v2(C):
    return "v2<4,1>" if C <= 128 else "v2<8,2>"


# Correlation3D.  name: ((B, Cin, Cout, N1, N2, k), neighbour kind, {precision: route}).
# v2 tiles: pass 1 takes 128-row tiles of each cloud but sizes its grid from max(N1, N2); pass 2 items are 8 points
# (128 rows), pass 3 items 32 points.  N1 in {1, 7, 9, 31, 33, 129} sits on both sides of those edges; N2 alternates
# between 131 more than N1 (more than one 128-row tile of cloud 2 beyond cloud 1) and 5 (fewer points than k, so every
# neighbourhood repeats indices).  The same shapes run the tcgen05 stage-1 kernel at precision 1 and fp32 at precision 0.
C3_CASES = {}
for _i, _C in enumerate((32, 64, 96, 128, 160, 192)):
    for _j, _N1 in enumerate((1, 7, 9, 31, 33, 129)):
        _N2 = _N1 + 131 if (_i + _j) % 2 else 5
        C3_CASES[f"C{_C}_N1_{_N1}_N2_{_N2}"] = ((3, _C, _C, _N1, _N2, 16), "random",
                                                {0: "fp32<16>", 1: "tc<0>", 2: _v2(_C)})
C3_CASES.update({
    # cloud 2 smaller than cloud 1 by more than a 128-row tile: pass 1's grid is sized by cloud 1
    "C32_N1_300_N2_40": ((3, 32, 32, 300, 40, 16), "random", {0: "fp32<16>", 1: "tc<0>", 2: "v2<4,1>"}),
    "C192_N1_300_N2_40": ((3, 192, 192, 300, 40, 16), "random", {0: "fp32<16>", 1: "tc<0>", 2: "v2<8,2>"}),
    # tcgen05 stage 1 at precision 2: widths above v2's 192, and Cin != Cout
    "C224_N1_33_N2_164": ((3, 224, 224, 33, 164, 16), "random", {0: "fp32<16>", 1: "tc<0>", 2: "tc<1>"}),
    "C256_N1_129_N2_5": ((3, 256, 256, 129, 5, 16), "random", {0: "fp32<16>", 1: "tc<0>", 2: "tc<1>"}),
    "Cin48_Cout64": ((3, 48, 64, 129, 260, 16), "random", {0: "fp32<16>", 1: "tc<0>", 2: "tc<1>"}),
    # fp32 stage 1 (every precision): KMAX = 4 / 8 / 16 / 32 by k; the scalar path for Cout % 4 != 0; fewer points per
    # CTA for wide Cout (TP = 128 / k halved while its shared memory exceeds 200 KB: 8 -> 4 at k = 16, 4 -> 2 at k = 32)
    "k1_Cin1_Cout3": ((3, 1, 3, 40, 30, 1), "random", {0: "fp32<4>", 1: "fp32<4>", 2: "fp32<4>"}),
    "k4_Cout33": ((3, 16, 33, 70, 50, 4), "random", {0: "fp32<4>", 1: "fp32<4>", 2: "fp32<4>"}),
    "k5_Cout5": ((3, 8, 5, 33, 20, 5), "random", {0: "fp32<8>", 1: "fp32<8>", 2: "fp32<8>"}),
    "k8_Cout64": ((3, 32, 64, 129, 60, 8), "random", {0: "fp32<8>", 1: "fp32<8>", 2: "fp32<8>"}),
    "k9_Cin1_Cout32": ((3, 1, 32, 31, 200, 9), "random", {0: "fp32<16>", 1: "fp32<16>", 2: "fp32<16>"}),
    "k16_Cout33_N2_7": ((3, 20, 33, 100, 7, 16), "random", {0: "fp32<16>", 1: "fp32<16>", 2: "fp32<16>"}),
    "k17_Cout96": ((3, 24, 96, 50, 40, 17), "random", {0: "fp32<32>", 1: "fp32<32>", 2: "fp32<32>"}),
    "k16_Cout512": ((2, 64, 512, 70, 90, 16), "random", {0: "fp32<16>", 1: "fp32<16>", 2: "fp32<16>"}),
    "k32_Cout512": ((2, 16, 512, 40, 50, 32), "random", {0: "fp32<32>", 1: "fp32<32>", 2: "fp32<32>"}),
})
for _kind in ("same", "dups", "edges"):           # same: every neighbour is the last point of its cloud
    C3_CASES[f"{_kind}_C32"] = ((3, 32, 32, 150, 200, 16), _kind, {0: "fp32<16>", 1: "tc<0>", 2: "v2<4,1>"})
    C3_CASES[f"{_kind}_k5_Cout5"] = ((3, 8, 5, 60, 40, 5), _kind, {0: "fp32<8>"})

# PointConv, uint16 neighbour indices (N <= 65536).  name: ((B, C, Cout, N, S), neighbour kind, 3xTF32 MODE at precisions
# 0 and 2).
# A CTA takes 120 sampled points (S = 119 / 120 / 121 / 241); channels are padded to Cp = roundup16(C+3) (C = 0 / 13 / 14 /
# 29 / 30 / 195 / 509 -> Cp = 16 / 16 / 32 / 32 / 48 / 208 / 512), out_channels to Npad = roundup32(Cout) (MODE 2 and the
# shallower ring above 128).  N = 65536 is the largest cloud of these; its uint16 neighbour table holds 65535.
PC_CASES = {
    "S1_C0_Cout1": ((3, 0, 1, 50, 1), "random", 1),
    "S119_C13_Cout31": ((3, 13, 31, 300, 119), "random", 1),
    "S120_C14_Cout33": ((3, 14, 33, 300, 120), "random", 1),
    "S121_C29_Cout128": ((3, 29, 128, 400, 121), "random", 1),
    "S241_C30_Cout129": ((3, 30, 129, 500, 241), "random", 2),
    "S121_C195_Cout160": ((2, 195, 160, 300, 121), "random", 2),
    "S119_C509_Cout255": ((2, 509, 255, 200, 119), "random", 2),
    "S241_C13_Cout256": ((3, 13, 256, 400, 241), "random", 2),
    "S1_C509_Cout33": ((2, 509, 33, 20, 1), "random", 1),
    "N65536_edges": ((2, 8, 64, 65536, 241), "edges", 1),
}
for _kind in ("same", "dups", "edges"):
    PC_CASES[f"{_kind}_Cout129"] = ((3, 24, 129, 300, 241), _kind, 2)
    PC_CASES[f"{_kind}_Cout64"] = ((3, 24, 64, 300, 130), _kind, 1)

# PointConv, uint32 neighbour indices (N > 65536, b200_pointconv_fwd only; "edges" reaches index 65536).  Cout = 256: MODE 2
# on a one-stage ring, MODE 0 on three stages; Cout = 128: MODE 1 on two stages, MODE 0 on four.
PC_WIDE = {
    "N65537_S63_C30": ((2, 30, 256, 65537, 63), "random", 2),
    "N65537_S64_C13": ((2, 13, 256, 65537, 64), "edges", 2),
    "N65537_S65_C0": ((2, 0, 256, 65537, 65), "dups", 2),
    "N65537_S121_C29_Cout128": ((2, 29, 128, 65537, 121), "edges", 1),
}


def _pc_routes(mode, wide=False):
    w = "true" if wide else "false"
    return {0: f"v2<{mode},{w}>", 1: f"v2<0,{w}>", 2: f"v2<{mode},{w}>"}


def _pc_case_routes(name):
    return _pc_routes(PC_CASES[name][2]) if name in PC_CASES else _pc_routes(PC_WIDE[name][2], wide=True)


@functools.lru_cache(maxsize=None)
def c3_case(name):
    shape, kind, _ = C3_CASES[name]
    inputs, w, knn12, knn11 = c3_inputs(*shape, kind, _seed(name))
    return inputs, w, knn12, knn11, c3_reference(inputs, w, knn12, knn11)


@functools.lru_cache(maxsize=None)
def pc_case(name):
    shape, kind, _ = PC_CASES[name] if name in PC_CASES else PC_WIDE[name]
    inputs, w, knn = pc_inputs(*shape, kind, _seed(name))
    return (inputs, w, knn) + pc_reference(inputs, w, knn)


# ------------------------------------------------------------------------------------------------- GPU calls
def _dev(d):
    return {n: t.to(DEV) for n, t in d.items()}


def run_corr3d(inputs, w, knn12, knn11, precision):
    """b200_corr3d_fwd; inputs are moved first, so that out and the scratch come out of the poisoned blocks."""
    x, wd, k12, k11 = _dev(inputs), _dev(w), knn12.to(DEV), knn11.to(DEV)
    _poison_allocator()
    out = pwc3d.correlation3d_forward(x["xyz1"], x["feat1"], x["xyz2"], x["feat2"], wd, k12, k11, precision)
    torch.cuda.synchronize()
    return out


def run_pointconv(inputs, w, knn, precision, entry="b200_pointconv_fwd"):
    """b200_pointconv_fwd, or b200_pointconv_fwd_linear (entry), after the same poisoning."""
    x, wd, k = _dev(inputs), _dev(w), knn.to(DEV)
    _poison_allocator()
    out = pointconv._pointconv_run(x["xyz"], x["feat"], x["sampled_xyz"], k, wd, precision, entry)
    torch.cuda.synchronize()
    return out


def sample_ratios(got, ref):
    """max|got - ref| / max|ref| of every sample (dim 0); NaN in got gives NaN."""
    d = (got.detach().double().cpu() - ref).abs().flatten(1).amax(1).tolist()
    s = ref.abs().flatten(1).amax(1).tolist()
    return [0.0 if dd == 0 else (dd / ss if ss > 0 else float("inf")) for dd, ss in zip(d, s)]


def check(op, route, precision, got, ref, label, K=0):
    """Per-sample bar of the route; K = the length of its longest tensor-core contraction (module docstring)."""
    bar = (TF32_BAR if (op, route) in TF32_ROUTES else FP32_BAR) + K / 8 * 2.0 ** -23
    assert tuple(got.shape) == tuple(ref.shape), f"{label}: shape {tuple(got.shape)} != {tuple(ref.shape)}"
    assert bool(torch.isfinite(got).all()), f"{label}: non-finite output (an unwritten element shows as NaN)"
    r = sample_ratios(got, ref)
    key = (op, route, precision)
    MEASURED[key] = max(MEASURED.get(key, 0.0), max(r))
    print(f"\n[{label} {op} {route} p{precision}] per-sample max|diff| / max|ref|: " + " ".join(f"{v:.2g}" for v in r))
    bad = {b: v for b, v in enumerate(r) if not v <= bar}
    assert not bad, f"{label} ({route}, precision {precision}): samples over {bar:g} of max|ref|: {bad}"


def pc_check(route, precision, got, ref, label, inputs):
    """check() for PointConv, whose Linear is a tensor-core contraction over K = 16 * (C+3)."""
    check("pointconv", route, precision, got, ref, label, K=16 * (inputs["feat"].shape[1] + 3))


@pytest.fixture(scope="module", autouse=True)
def _report_measured():
    yield
    if MEASURED:
        print("\nlargest max|diff| / max|ref| per route and precision:")
        for (op, route, p), v in sorted(MEASURED.items()):
            print(f"  {op:9s} {route:9s} p{p}: {v:.3g}")


# ------------------------------------------------------------------------------------------------- CPU
def test_references_agree_with_the_fp32_oracle():
    """The imported float64 references against oracle/spec.c (fp32 C, its own loops) at two small shapes per op."""
    from oracle import spec
    for shape in ((2, 5, 7, 30, 20, 4), (1, 3, 33, 17, 9, 16)):
        inputs, w, knn12, knn11 = c3_inputs(*shape, "random", 11)
        want = spec.corr3d_fwd(*(inputs[n].numpy() for n in ("xyz1", "feat1", "xyz2", "feat2")), knn12.numpy(),
                               knn11.numpy(), {n: t.numpy() for n, t in w.items()})
        r = sample_ratios(torch.from_numpy(want), c3_reference(inputs, w, knn12, knn11))
        assert max(r) <= 1e-5, (shape, r)
    for shape in ((2, 5, 7, 40, 30), (1, 2, 33, 20, 3)):
        inputs, w, knn = pc_inputs(*shape, "random", 12)
        want = spec.pointconv_fwd(inputs["xyz"].numpy(), inputs["feat"].numpy(), inputs["sampled_xyz"].numpy(),
                                  knn.numpy(), {n: t.numpy() for n, t in w.items()})
        r = sample_ratios(torch.from_numpy(want), pc_reference(inputs, w, knn)[0])
        assert max(r) <= 1e-5, (shape, r)


# ------------------------------------------------------------------------------------------------- Correlation3D
C3_IDS = [(n, p) for n, (_, _, routes) in C3_CASES.items() for p in routes]


@pytest.mark.gpu
@pytest.mark.parametrize("name,precision", C3_IDS, ids=[f"{n}-p{p}" for n, p in C3_IDS])
def test_corr3d_forward_vs_float64(name, precision):
    inputs, w, knn12, knn11, ref = c3_case(name)
    got = run_corr3d(inputs, w, knn12, knn11, precision)
    check("corr3d", C3_CASES[name][2][precision], precision, got, ref, name)


# ------------------------------------------------------------------------------------------------- PointConv
PC_IDS = [(n, p) for n in PC_CASES for p in (0, 1, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,precision", PC_IDS, ids=[f"{n}-p{p}" for n, p in PC_IDS])
def test_pointconv_forward_vs_float64(name, precision):
    """b200_pointconv_fwd and b200_pointconv_fwd_linear against the reference; the first is LeakyReLU(0.1) of the
    second bit for bit, and precision 0 is precision 2 bit for bit."""
    inputs, w, knn, ref, ref_linear = pc_case(name)
    route = _pc_case_routes(name)[precision]
    got = run_pointconv(inputs, w, knn, precision)
    pc_check(route, precision, got, ref, name, inputs)
    linear = run_pointconv(inputs, w, knn, precision, "b200_pointconv_fwd_linear")
    pc_check(route, precision, linear, ref_linear, name + " linear", inputs)
    assert torch.equal(got, F.leaky_relu(linear, 0.1)), f"{name}: fwd != LeakyReLU(fwd_linear)"
    if precision == 0:
        assert torch.equal(got, run_pointconv(inputs, w, knn, 2)), f"{name}: precision 0 != precision 2"


WIDE_IDS = [(n, p) for n in PC_WIDE for p in (0, 1, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,precision", WIDE_IDS, ids=[f"{n}-p{p}" for n, p in WIDE_IDS])
def test_pointconv_wide_index_vs_float64(name, precision):
    """Clouds of more than 65536 points: b200_pointconv_fwd only (the _linear entry refuses them)."""
    inputs, w, knn, ref, _ = pc_case(name)
    got = run_pointconv(inputs, w, knn, precision)
    pc_check(_pc_case_routes(name)[precision], precision, got, ref, name, inputs)
    if precision == 0:
        assert torch.equal(got, run_pointconv(inputs, w, knn, 2)), f"{name}: precision 0 != precision 2"
    with pytest.raises(B200Error, match="N <= 65536"):
        run_pointconv(inputs, w, knn, precision, "b200_pointconv_fwd_linear")


# ------------------------------------------------------------------------------------------------- routes
def _kernel_names(fn):
    """Names (with template arguments, no spaces) of the b200:: kernels fn launches, as torch.profiler records them."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        m = re.search(r"b200::(\w+)(<[^<>]*>)?", re.sub(r"\((?:unsigned )?int\)", "", e.name))
        if m:
            names.add((m.group(1) + (m.group(2) or "")).replace(" ", ""))
    return names


C3_ROUTE_KERNELS = {f"fp32<{k}>": {"pointwise_linear_kernel", f"corr3d_stage1_kernel<{k}>", "corr3d_stage2_kernel"}
                    for k in (4, 8, 16, 32)}
C3_ROUTE_KERNELS.update({f"tc<{s}>": {"pointwise_linear_kernel", f"corr3d_stage1_tc_kernel<{s}>", "corr3d_stage2_kernel"}
                         for s in (0, 1)})
C3_ROUTE_KERNELS.update({f"v2<{c}>": {"corr3d_v2_linear_kernel", f"corr3d_v2_stage1_kernel<{c}>", "corr3d_v2_stage2_kernel"}
                         for c in ("4,1", "8,2")})
C3_PREP_KERNELS = {"corr3d_prep_weights", "corr3d_v2_prep_kernel", "corr3d_v2_prep_w1_kernel"}
PC_ROUTE_KERNELS = {f"v2<{m},{w}>": {"pointconv_v2_prep_kernel", f"pointconv_v2_kernel<{m},{w}>"}
                    for m in (0, 1, 2) for w in ("false", "true")}


@pytest.mark.gpu
def test_every_case_reaches_its_route():
    """Each (case, precision) of the tables above launches the kernels of the route it claims, and no other route's; the
    PointConv cases launch every PointConv forward kernel and nothing else."""
    wrong, seen = [], set()
    for name, (_, _, routes) in C3_CASES.items():
        inputs, w, knn12, knn11, _ = c3_case(name)
        for p, route in routes.items():
            got = _kernel_names(lambda: run_corr3d(inputs, w, knn12, knn11, p)) - C3_PREP_KERNELS
            if got != C3_ROUTE_KERNELS[route]:
                wrong.append(f"corr3d {name} p{p}: claims {route}, launched {sorted(got)}")
    for name in list(PC_CASES) + list(PC_WIDE):
        inputs, w, knn, _, _ = pc_case(name)
        for p, route in _pc_case_routes(name).items():
            got = _kernel_names(lambda: run_pointconv(inputs, w, knn, p))
            seen |= got
            if got != PC_ROUTE_KERNELS[route]:
                wrong.append(f"pointconv {name} p{p}: claims {route}, launched {sorted(got)}")
    assert not wrong, "\n".join(wrong)
    every = set().union(*PC_ROUTE_KERNELS.values())
    assert seen == every, sorted(seen ^ every)


# ------------------------------------------------------------------------------------------------- batch invariance
def _split_calls(run, inputs, knns, B):
    """run(inputs_b, knns_b) for each sample b alone, stacked."""
    return torch.cat([run({n: t[b:b + 1].contiguous() for n, t in inputs.items()},
                          [k[b:b + 1].contiguous() for k in knns]) for b in range(B)])


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [2, 1])
@pytest.mark.parametrize("C,N", list(zip(LEVEL_CHANNELS, PYRAMID_POINTS)))
def test_corr3d_batch_of_148_equals_single_sample_calls(C, N, precision):
    """The benchmark's five Correlation3D levels at its batch of 148: the persistent v2 kernels (precision 2) run dozens of
    (sample, tile) items per CTA, so ring wrap, barrier phases and accumulator reuse all occur; none of it may change a
    bit of any sample.  Samples 0, 74 and 147 are also compared with the float64 reference."""
    B = 148
    route = _v2(C) if precision == 2 else "tc<0>"
    inputs, w, knn12, knn11 = c3_inputs(B, C, C, N, N, 16, "random", C + precision)
    batched = run_corr3d(inputs, w, knn12, knn11, precision)
    single = _split_calls(lambda x, k: run_corr3d(x, w, k[0], k[1], precision), inputs, [knn12, knn11], B)
    diff = [b for b in range(B) if not torch.equal(batched[b], single[b])]
    assert not diff, f"samples whose batched result differs from their single-sample call: {diff}"
    for b in (0, B // 2, B - 1):
        one = {n: t[b:b + 1] for n, t in inputs.items()}
        ref = c3_reference(one, w, knn12[b:b + 1], knn11[b:b + 1])
        check("corr3d", route, precision, batched[b:b + 1], ref, f"C{C}_N{N} B148 sample {b}")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [2, 1])
def test_pointconv_batch_of_148_equals_single_sample_calls(precision):
    """The first feature-pyramid PointConv of the benchmark's model (32 -> 64 channels, 4096 -> 2048 points) at 148."""
    B, C, Cout, N, S = 148, 32, 64, 4096, 2048
    inputs, w, knn = pc_inputs(B, C, Cout, N, S, "random", 5 + precision)
    batched = run_pointconv(inputs, w, knn, precision)
    single = _split_calls(lambda x, k: run_pointconv(x, w, k[0], precision), inputs, [knn], B)
    diff = [b for b in range(B) if not torch.equal(batched[b], single[b])]
    assert not diff, f"samples whose batched result differs from their single-sample call: {diff}"
    for b in (0, B // 2, B - 1):
        ref, _ = pc_reference({n: t[b:b + 1] for n, t in inputs.items()}, w, knn[b:b + 1])
        pc_check(_pc_routes(1)[precision], precision, batched[b:b + 1], ref, f"B148 sample {b}", inputs)


# ------------------------------------------------------------------------------------------------- neighbour order
def _permute_neighbours(knn, seed):
    gen = torch.Generator().manual_seed(seed)
    return torch.gather(knn, 2, torch.argsort(torch.rand(knn.shape, generator=gen), dim=2))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C32_N1_129_N2_260", "C192_N1_300_N2_40", "Cin48_Cout64", "k17_Cout96"])
def test_corr3d_neighbour_order_does_not_matter(name):
    inputs, w, knn12, knn11, ref = c3_case(name)
    for p, route in C3_CASES[name][2].items():
        got = run_corr3d(inputs, w, _permute_neighbours(knn12, 1), _permute_neighbours(knn11, 2), p)
        check("corr3d", route, p, got, ref, name + " permuted")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["S241_C30_Cout129", "S121_C29_Cout128", "N65537_S63_C30"])
def test_pointconv_neighbour_order_does_not_matter(name):
    inputs, w, knn, ref, _ = pc_case(name)
    for p, route in _pc_case_routes(name).items():
        pc_check(route, p, run_pointconv(inputs, w, _permute_neighbours(knn, 3), p), ref, name + " permuted", inputs)


# ------------------------------------------------------------------------------------------------- index rules
# Correlation3D: an index outside [0, N-1] of its cloud is clamped to it.  PointConv: a negative index wraps once (+N),
# what is still out of range is clamped.  (include/b200flow.h, at b200_corr3d_fwd and b200_pointconv_fwd.)
def _out_of_range(knn, N):
    bad = knn.clone()
    bad[:, :, 0] = -1
    bad[:, :, 1] = N
    bad[:, 0::2, 2] = -N
    bad[:, 1::2, 2] = -N - 3
    bad[:, :, -1] = N + 5
    return bad


@pytest.mark.gpu
@pytest.mark.parametrize("name,precision", [("C32_N1_300_N2_40", 0), ("C32_N1_300_N2_40", 1), ("C32_N1_300_N2_40", 2),
                                            ("Cin48_Cout64", 2), ("k5_Cout5", 0), ("k32_Cout512", 0)])
def test_corr3d_out_of_range_indices_are_clamped(name, precision):
    inputs, w, knn12, knn11, _ = c3_case(name)
    N1, N2 = inputs["xyz1"].shape[2], inputs["xyz2"].shape[2]
    bad12, bad11 = _out_of_range(knn12, N2), _out_of_range(knn11, N1)
    ref = c3_reference(inputs, w, bad12.clamp(0, N2 - 1), bad11.clamp(0, N1 - 1))
    got = run_corr3d(inputs, w, bad12, bad11, precision)
    check("corr3d", C3_CASES[name][2][precision], precision, got, ref, name + " out-of-range")


@pytest.mark.gpu
@pytest.mark.parametrize("name,precision", [("S121_C29_Cout128", 0), ("S121_C29_Cout128", 1), ("S121_C29_Cout128", 2),
                                            ("S241_C30_Cout129", 2), ("N65537_S63_C30", 1), ("N65537_S63_C30", 2)])
def test_pointconv_out_of_range_indices_wrap_once_then_clamp(name, precision):
    inputs, w, knn, _, _ = pc_case(name)
    N = inputs["xyz"].shape[2]
    bad = _out_of_range(knn, N)
    ref, _ = pc_reference(inputs, w, torch.where(bad < 0, bad + N, bad).clamp(0, N - 1))
    pc_check(_pc_case_routes(name)[precision], precision, run_pointconv(inputs, w, bad, precision), ref, name + " out-of-range", inputs)
