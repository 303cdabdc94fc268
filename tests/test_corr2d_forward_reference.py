"""correlation2d forward kernels against a float64 reference, on every route, at tile and store edges and at the bench batch.

Reference.  ref_corr2d(a, b, md) on NCHW maps in float64: b zero-padded by md, out[:, t] = sum_c a * b_shift / C for every
shift t = (dy + md) * (2md+1) + (dx + md), and S[:, t] = sum_c |a * b_shift| / C beside it.  It runs on the device of its
inputs: float64 on the GPU for the GPU tests, on the CPU for the CPU checks against oracle/spec.c and oracle/torch_ref.py.

Routes (read from the eligibility code; route_of() is the Python mirror, test_every_case_reaches_its_route checks every
claim against the b200:: kernels torch.profiler sees):
- b200_corr2d_fwd (NHWC in): md > 4 -> "any" = corr2d_fwd_any_kernel (warp per output, lanes over channels, shuffle
  tree).  md = 4, C % 4 == 0 and in1 / in2 16-byte aligned -> corr2d_fwd_tma_kernel, "tma.v4" when W % 4 == 0 and out is
  16-byte aligned (float4 stores after a neighbour shuffle), else "tma.scalar".  Otherwise, md 1..4 -> "cp<md,VEC>" =
  corr2d_fwd_kernel<md, C % 4 == 0 && inputs 16-byte aligned> (cp.async or scalar loads; a strip stores float2 pairs when
  W is even, the strip is inside the map and out is 8-byte aligned, else scalars).
- b200_corr2d_fwd_nchw[_leaky] (NCHW in): B200_ENOSUP, with the output untouched, unless md = 4, W % 4 == 0 and all
  three pointers are 16-byte aligned.  Then "diag" = corr2d_fwd_diag_kernel (48 x 8 tiles, 8-channel stages, 4-stage
  ring) when corr2d_diag_preferred(W), else "nchw32" = corr2d_fwd_nchw_kernel (32 x 8 tiles, 16-channel stages, 3-stage
  ring, row shift +4 split by channels over warps 8 and 9 with a two-buffer hand-over).
The mirror leaves out two refusals of the TMA kernel that no test can build: a per-sample map of 2^40 bytes or more,
and a driver without cuTensorMapEncodeTiled.  They are the only calls that reach corr2d_fwd_kernel<4,true> (md = 4 with
C % 4 == 0 and aligned inputs is the TMA kernel's otherwise), so that one of the twelve forward kernels is not launched
here; it is corr2d_fwd_kernel<3,true> with a wider halo.

Bar, elementwise: |got - ref| <= (C + 2) * 2^-24 * S * (1 + 1e-3).  Every route sums C fp32 products in some tree (one
chain, an (even, odd) channel pair of chains, chains split over two warps, a 32-lane shuffle tree; fused or not; the
zero-filled padding channels add exact zeros), so each product passes through at most C roundings, and the final
/ C or * fl(1/C) adds at most two more: Higham's gamma_{C+2} <= (C + 2) * 2^-24 * (1 + 1e-3) for C + 2 <= 16777 bounds
the error relative to S, whatever the order.  The bar is rigorous and cannot flake; inputs stay far from subnormals.
test_bar_has_teeth shows that dropping one channel's term breaks it on at least 99 % of the outputs of every case.
Leaky outputs are held to leaky(ref) (the slope rounded to fp32 as the kernel holds it) at bar + 2^-24 * |ref|: leaky_relu
is 1-Lipschitz for slopes in [0, 1] and its product adds one rounding.

Outputs are written into NaN-filled buffers with guard elements before and after, so an output a kernel skips fails the
bar and a store outside the tensor shows in the guards.  Pointer alignment is set by 4- and 8-byte offsets into such
buffers, which is how the misaligned routes are reached.

Inputs: randn per element times a per-channel scale 2^U(-6, 6) (independently for in1 and in2) times a per-sample scale
2^U(-2, 2), so that a stage reading past C or into the next sample shows.  Kind "cancel": the second half of the channels
repeats the first half of in1 and negates that of in2 (times 1 + 2^-10 * randn), so every output sits near 0 while S
does not.

Not tested: non-finite inputs.  The any kernel skips displacements outside the image, while the tiled kernels multiply
by the zero-filled halo, so an inf there gives NaN on the tiled routes and not on the any route.

Exact properties, bit for bit: the bench's five correlation levels (CONFIGS["things"], LEVEL_CHANNELS) at BENCH_BATCH
equal the 148 single-sample calls, for correlation2d and correlation2d_leaky; correlation2d_leaky == leaky_relu of
correlation2d on the same route for slopes 0, 0.1, 0.5 and 1.  The NCHW entry and the NHWC entry at md = 4 are both held
to the bar, not to each other's bits (the cp.async kernel divides by C, the others multiply by fl(1/C)).

Measured on a B200 at its 1000 W power limit (largest |got - ref| / bar per route over every case of this file):
  diag 0.63 (leaky 0.57), nchw32 0.49 (leaky 0.43), tma.v4 0.27, tma.scalar 0.36 (leaky 0.064), any 0.59,
  cp<1,true> 0.18, cp<1,false> 0.30, cp<2,true> 0.30, cp<2,false> 0.38, cp<3,true> 0.22, cp<3,false> 0.16, cp<4,false> 0.50
Value-only faults that the file catches (each fails the cases of its route): warp 8 of corr2d_fwd_nchw_kernel dropping
warp 9's partial sums or reading the other hand-over buffer, the diag store swapping the pair halves of odd pixels, and
the cp.async epilogue dividing by C + 1.
"""
import functools
import zlib

import pytest
import torch
import torch.nn.functional as F

import rpeflow_b200 as b200
from rpeflow_b200 import _lib
from rpeflow_b200.workload import BENCH_BATCH, CONFIGS, LEVEL_CHANNELS
from test_backward_reference import DEV, _poison_allocator
from test_forward_reference import _kernel_names

U = 2.0 ** -24
GUARD = 64                                              # NaN floats before and after every output buffer
MEASURED = {}                                           # route -> largest |got - ref| / bar seen


# ------------------------------------------------------------------------------------------------- reference and bar
def ref_corr2d(a, b, md):
    """a, b [B,C,H,W] float64 -> (out, S), both [B,(2md+1)^2,H,W]: the mean over channels of a * b shifted by (dy, dx)
    with zero padding, and the mean of its absolute values."""
    B, C, H, W = a.shape
    D = 2 * md + 1
    bp = F.pad(b, (md, md, md, md))
    out = a.new_empty(B, D * D, H, W)
    S = a.new_empty(B, D * D, H, W)
    for r in range(D):
        for c in range(D):
            p = a * bp[:, :, r:r + H, c:c + W]
            out[:, r * D + c] = p.sum(1) / C
            S[:, r * D + c] = p.abs().sum(1) / C
    return out, S


def bar_of(C, S):
    return (C + 2) * U * S * (1 + 1e-3)


def leaky64(x, slope):
    """leaky_relu in float64 with the slope the kernel holds (fp32)."""
    s = float(torch.tensor(slope, dtype=torch.float32))
    return torch.where(x >= 0, x, x * s)


def check_bar(route, got, ref, S, C, label, slope=None):
    """Elementwise bar of the module docstring; records the largest ratio per route."""
    assert tuple(got.shape) == tuple(ref.shape), f"{label}: shape {tuple(got.shape)} != {tuple(ref.shape)}"
    bar = bar_of(C, S)
    if slope is not None:
        ref = leaky64(ref, slope)
        bar = bar + U * ref.abs()
    diff = (got.to(ref.device).double() - ref).abs()
    ratio = torch.where(bar > 0, diff / bar.clamp_min(1e-300), torch.where(diff == 0, 0.0, float("inf")))
    worst = ratio.max().item()                          # NaN when an output is NaN (unwritten)
    key = route + (" leaky" if slope is not None else "")
    if worst == worst:
        MEASURED[key] = max(MEASURED.get(key, 0.0), worst)
    print(f"\n[{label} {key}] max |got - ref| / bar = {worst:.3g}")
    bad = ~(diff <= bar)
    n = int(bad.sum())
    if n:
        idx = bad.nonzero()[0].tolist()
        raise AssertionError(f"{label} ({key}): {n} of {bad.numel()} outputs over the bar, first at {idx}: "
                             f"got {got[tuple(idx)].item()!r}, ref {ref[tuple(idx)].item()!r}, bar {bar[tuple(idx)].item():.3g}")


@pytest.fixture(scope="module", autouse=True)
def _report_measured():
    yield
    if MEASURED:
        print("\nlargest |got - ref| / bar per route:")
        for route, v in sorted(MEASURED.items()):
            print(f"  {route:16s} {v:.3g}")


# ------------------------------------------------------------------------------------------------- inputs
def make_inputs(B, C, H, W, seed, kind="scaled"):
    """fp32 NCHW (a, b) on the CPU, as the module docstring describes."""
    gen = torch.Generator().manual_seed(seed)
    half = C // 2 if kind == "cancel" else C

    def ch():
        return 2.0 ** (torch.rand(1, half, 1, 1, generator=gen, dtype=torch.float64) * 12 - 6)
    smp = 2.0 ** (torch.rand(B, 1, 1, 1, generator=gen, dtype=torch.float64) * 4 - 2)
    a = torch.randn(B, half, H, W, generator=gen, dtype=torch.float64) * ch() * smp
    b = torch.randn(B, half, H, W, generator=gen, dtype=torch.float64) * ch() * smp
    if kind == "cancel":
        assert C % 2 == 0
        jitter = 1 + 2.0 ** -10 * torch.randn(B, half, H, W, generator=gen, dtype=torch.float64)
        a, b = torch.cat([a, a], 1), torch.cat([b, -b * jitter], 1)
    return a.float(), b.float()


# ------------------------------------------------------------------------------------------------- route mirror
def _ceil_div(a, b):
    return -(-a // b)


def diag_preferred(W):
    """corr2d_diag.cu corr2d_diag_preferred, in the same double arithmetic."""
    w48 = _ceil_div(W, 48) * 48 / W
    w32 = _ceil_div(W, 32) * 32 / W
    return w48 <= 1.2 * w32


def _align(off):
    """Alignment in bytes of a float pointer at `off` floats from a 16-byte aligned base (at most 16)."""
    return 16 if off % 4 == 0 else (8 if off % 2 == 0 else 4)


def route_of(entry, C, H, W, md, in_off=0, out_off=0):
    """The route b200_corr2d_fwd ("nhwc") or b200_corr2d_fwd_nchw[_leaky] ("nchw") takes (see the module docstring)."""
    in_ok = _align(in_off) == 16
    if entry == "nchw":
        if md != 4 or W % 4 or not in_ok or _align(out_off) != 16:
            return "enosup"
        return "diag" if diag_preferred(W) else "nchw32"
    if md > 4:
        return "any"
    if md == 4 and C % 4 == 0 and in_ok:
        return "tma.v4" if W % 4 == 0 and _align(out_off) == 16 else "tma.scalar"
    return f"cp<{md},{'true' if C % 4 == 0 and in_ok else 'false'}>"


def kernel_of(route):
    if route.startswith("tma"):
        return "corr2d_fwd_tma_kernel"
    if route.startswith("cp<"):
        return "corr2d_fwd_kernel" + route[2:]
    return {"any": "corr2d_fwd_any_kernel", "diag": "corr2d_fwd_diag_kernel", "nchw32": "corr2d_fwd_nchw_kernel"}[route]


def bench_route(C, H, W):
    """Route of ops.correlation2d on contiguous fp32 NCHW maps at md = 4 without autograd."""
    r = route_of("nchw", C, H, W, 4)
    return route_of("nhwc", C, H, W, 4) if r == "enosup" else r


FORWARD_KERNELS = ({f"corr2d_fwd_kernel<{m},{v}>" for m in (1, 2, 3, 4) for v in ("true", "false")}
                   | {"corr2d_fwd_tma_kernel", "corr2d_fwd_nchw_kernel", "corr2d_fwd_diag_kernel", "corr2d_fwd_any_kernel"})
UNREACHABLE = {"corr2d_fwd_kernel<4,true>"}             # module docstring: calls no test can build


# ------------------------------------------------------------------------------------------------- cases
# name: (entry, B, C, H, W, md, in_off, out_off, kind, route).  B = None: a persistence case, whose batch is chosen at run
# time so that the tiles exceed twice the SM count and do not divide evenly over the grid (one CTA per SM).
CASES = {}


def _add(name, entry, B, C, H, W, md, route, in_off=0, out_off=0, kind="scaled"):
    assert name not in CASES
    CASES[name] = (entry, B, C, H, W, md, in_off, out_off, kind, route)


# diag: every W % 48 residue (both strip parities of the float4 + float2 stores at the ragged edge), heights with
# H % 8 in 1..7 and H < 8 (the row pairs and the warps at the ends of the diagonal), channel tails of the 8-channel stage
_DIAG_W = (96, 100, 104, 108, 112, 68, 72, 76, 80, 36, 40, 44)
_DIAG_H = (9, 1, 2, 3, 13, 5, 7, 17, 6, 15, 11, 8)
_DIAG_C = (8, 1, 5, 7, 9, 15, 17, 33, 81, 16, 24, 40)
for _W, _H, _C in zip(_DIAG_W, _DIAG_H, _DIAG_C):
    _add(f"diag_W{_W}_H{_H}_C{_C}", "nchw", 2 + _W % 2, _C, _H, _W, 4, "diag")
# nchw32: every W % 32 residue, the 16-channel stage's tails, and W = 156 (the diag_preferred tie, decided by rounding)
_N32_W = (32, 4, 8, 12, 16, 20, 24, 28, 52, 56, 60, 64, 156)
_N32_H = (8, 3, 9, 1, 14, 23, 5, 16, 7, 2, 12, 19, 10)
_N32_C = (16, 1, 5, 7, 9, 15, 17, 33, 81, 32, 31, 48, 12)
for _W, _H, _C in zip(_N32_W, _N32_H, _N32_C):
    _add(f"nchw32_W{_W}_H{_H}_C{_C}", "nchw", 2, _C, _H, _W, 4, "nchw32")
# TMA: every W % 24 residue (W % 4 != 0 stores scalars), vector and scalar stores with W % 4 == 0 (out 16- / 8- / 4-byte
# aligned), channel tails of the 32-channel stage
_TMA_C = (4, 8, 12, 28, 36, 60, 96, 100)
for _r in range(24):
    _W, _H, _C = 24 + _r, (1, 3, 5, 8, 9, 12, 15, 17)[_r % 8], _TMA_C[_r % len(_TMA_C)]
    _off = (0, 2, 1)[_r // 4 % 3] if _W % 4 == 0 else 0
    _add(f"tma_W{_W}_H{_H}_C{_C}_out{_off}", "nhwc", 2, _C, _H, _W, 4, route_of("nhwc", _C, _H, _W, 4, 0, _off), out_off=_off)
_add("tma_W96_H16_C68_out0", "nhwc", 3, 68, 16, 96, 4, "tma.v4")
_add("tma_W96_H16_C68_out2", "nhwc", 3, 68, 16, 96, 4, "tma.scalar", out_off=2)
# cp.async kernel: md 1..3 with VEC on and off, md 4 with C % 4 == 0 and unaligned inputs; odd W, strips that end past W
# (xs + 6 > W), float2 stores (W even, out 8-byte aligned) and scalar ones (out 4-byte aligned), 2md+1 > H, W
_add("cp1_vec_W26_H11_C12_out2", "nhwc", 2, 12, 11, 26, 1, "cp<1,true>", out_off=2)
_add("cp1_vec_W1_H1_C4", "nhwc", 2, 4, 1, 1, 1, "cp<1,true>")
_add("cp1_W13_H5_C7", "nhwc", 2, 7, 5, 13, 1, "cp<1,false>")
_add("cp1_unaligned_W30_H9_C8", "nhwc", 2, 8, 9, 30, 1, "cp<1,false>", in_off=1)
_add("cp2_vec_W50_H7_C36", "nhwc", 2, 36, 7, 50, 2, "cp<2,true>")
_add("cp2_vec_W48_H16_C16_out1", "nhwc", 3, 16, 16, 48, 2, "cp<2,true>", out_off=1)
_add("cp2_W23_H10_C17", "nhwc", 2, 17, 10, 23, 2, "cp<2,false>")
_add("cp2_W3_H2_C5", "nhwc", 2, 5, 2, 3, 2, "cp<2,false>")
_add("cp3_vec_W29_H13_C20", "nhwc", 2, 20, 13, 29, 3, "cp<3,true>")
_add("cp3_vec_W48_H8_C64_out1", "nhwc", 2, 64, 8, 48, 3, "cp<3,true>", out_off=1)
_add("cp3_W31_H6_C33", "nhwc", 2, 33, 6, 31, 3, "cp<3,false>")
_add("cp3_unaligned_W7_H3_C16", "nhwc", 2, 16, 3, 7, 3, "cp<3,false>", in_off=1)
_add("cp4_unaligned_W44_H17_C16_out2", "nhwc", 2, 16, 17, 44, 4, "cp<4,false>", in_off=1, out_off=2)
_add("cp4_unaligned_W24_H8_C32", "nhwc", 2, 32, 8, 24, 4, "cp<4,false>", in_off=1)
_add("cp4_W35_H9_C81", "nhwc", 2, 81, 9, 35, 4, "cp<4,false>")
_add("cp4_W5_H4_C3", "nhwc", 2, 3, 4, 5, 4, "cp<4,false>")
# any md: 2md+1 beyond H and / or W, C > 32 (each lane sums several channels) and C < 32 (idle lanes)
_add("any_md5_W40_H6_C33", "nhwc", 2, 33, 6, 40, 5, "any")
_add("any_md5_W11_H11_C3", "nhwc", 2, 3, 11, 11, 5, "any")
_add("any_md7_W9_H20_C70", "nhwc", 2, 70, 20, 9, 7, "any")
_add("any_md12_W12_H10_C100", "nhwc", 2, 100, 10, 12, 12, "any", in_off=1, out_off=1)
_add("any_md12_W30_H30_C40", "nhwc", 2, 40, 30, 30, 12, "any")
# near-total cancellation on each family
_add("cancel_diag_W100_H9_C32", "nchw", 2, 32, 9, 100, 4, "diag", kind="cancel")
_add("cancel_nchw32_W60_H11_C34", "nchw", 2, 34, 11, 60, 4, "nchw32", kind="cancel")
_add("cancel_tma_W50_H9_C64", "nhwc", 2, 64, 9, 50, 4, "tma.scalar", kind="cancel")
_add("cancel_cp2_W20_H7_C18", "nhwc", 2, 18, 7, 20, 2, "cp<2,false>", kind="cancel")
_add("cancel_any_md6_W15_H8_C66", "nhwc", 2, 66, 8, 15, 6, "any", kind="cancel")
# persistence: tiles > 2 x SMs, not a multiple of the grid; nchunks = ceil(C / stage channels) takes every value modulo
# the ring depth (diag: 8 channels, 4 stages; nchw32: 16 channels, 3 stages, and every CTA runs both hand-over buffers;
# TMA: 32 channels, 2 stages)
for _C in (8, 16, 24, 32, 40):
    _add(f"persist_diag_C{_C}", "nchw", None, _C, 20, 100, 4, "diag")
for _C in (16, 32, 48, 64):
    _add(f"persist_nchw32_C{_C}", "nchw", None, _C, 20, 60, 4, "nchw32")
for _C in (32, 64, 96):
    _add(f"persist_tma_C{_C}", "nhwc", None, _C, 13, 52, 4, "tma.v4")
_add("persist_tma_scalar_C64", "nhwc", None, 64, 13, 50, 4, "tma.scalar")

TILE = {"diag": (48, 8), "nchw32": (32, 8), "tma.v4": (24, 8), "tma.scalar": (24, 8)}


def tiles_per_sample(route, H, W):
    tw, th = TILE[route]
    return _ceil_div(W, tw) * _ceil_div(H, th)


def persist_batch(per_sample, sms):
    """Smallest batch whose tile count exceeds 2 x sms and is not a multiple of sms."""
    B = 1
    while B * per_sample <= 2 * sms or (B * per_sample) % sms == 0:
        B += 1
    return B


@functools.lru_cache(maxsize=None)
def _sm_count():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def case_batch(name, on_gpu):
    entry, B, C, H, W, md, in_off, out_off, kind, route = CASES[name]
    if B is None:
        B = persist_batch(tiles_per_sample(route, H, W), _sm_count()) if on_gpu else 2
    return B


def _seed(name):
    return zlib.crc32(name.encode())


# ------------------------------------------------------------------------------------------------- GPU calls
def _placed(x, off):
    """x copied to the device at `off` floats past a fresh (512-byte aligned) allocation."""
    buf = torch.empty(x.numel() + off, dtype=torch.float32, device=DEV)
    return buf[off:off + x.numel()].view(x.shape).copy_(x)


def run_entry(entry, a, b, md, in_off=0, out_off=0, slope=None):
    """The C entry on CPU NCHW inputs: "nhwc" (b200_corr2d_fwd on permuted copies) or "nchw" (b200_corr2d_fwd_nchw, or
    _leaky with slope).  Returns (return code, NCHW output view, guard buffer); the output starts as NaN."""
    B, C, H, W = a.shape
    D = 2 * md + 1
    if entry == "nhwc":
        a, b = a.permute(0, 2, 3, 1).contiguous(), b.permute(0, 2, 3, 1).contiguous()
    x1, x2 = _placed(a, in_off), _placed(b, in_off)
    n = B * D * D * H * W
    buf = torch.full((GUARD + out_off + n + GUARD,), float("nan"), device=DEV)
    out = buf[GUARD + out_off:GUARD + out_off + n].view(B, D * D, H, W)
    st = torch.cuda.current_stream().cuda_stream
    lib = _lib.lib
    if entry == "nhwc":
        rc = lib.b200_corr2d_fwd(x1.data_ptr(), x2.data_ptr(), out.data_ptr(), B, C, H, W, md, st)
    elif slope is None:
        rc = lib.b200_corr2d_fwd_nchw(x1.data_ptr(), x2.data_ptr(), out.data_ptr(), B, C, H, W, md, st)
    else:
        rc = lib.b200_corr2d_fwd_nchw_leaky(x1.data_ptr(), x2.data_ptr(), out.data_ptr(), B, C, H, W, md, float(slope), st)
    torch.cuda.synchronize()
    return rc, out, torch.cat([buf[:GUARD + out_off], buf[GUARD + out_off + n:]])


def run_checked(entry, a, b, md, in_off=0, out_off=0, slope=None, label=""):
    rc, out, guard = run_entry(entry, a, b, md, in_off, out_off, slope)
    _lib.check(rc, f"{label} {entry}")
    assert bool(torch.isnan(guard).all()), f"{label}: a store landed outside the output tensor"
    return out


@functools.lru_cache(maxsize=4)
def gpu_case(name):
    """(a, b) on the CPU, (ref, S) on the GPU in float64."""
    entry, _, C, H, W, md, _, _, kind, _ = CASES[name]
    a, b = make_inputs(case_batch(name, True), C, H, W, _seed(name), kind)
    return (a, b) + ref_corr2d(a.to(DEV, torch.float64), b.to(DEV, torch.float64), md)


# ------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("md", [1, 2, 3, 4, 5])
def test_reference_agrees_with_the_oracles(md):
    """ref_corr2d against oracle/spec.c (fp32 C loops, NHWC) and oracle/torch_ref.correlation2d (torch, float64 here)."""
    from oracle import spec, torch_ref
    for B, C, H, W in ((2, 3, 5, 7), (1, 17, 9, 4), (2, 8, 3, 12)):
        a, b = make_inputs(B, C, H, W, md * 100 + C)
        ref, S = ref_corr2d(a.double(), b.double(), md)
        want = torch.from_numpy(spec.corr2d_fwd(a.permute(0, 2, 3, 1).numpy(), b.permute(0, 2, 3, 1).numpy(), md))
        assert bool(((want.double() - ref).abs() <= bar_of(C, S)).all()), (md, B, C, H, W)
        assert bool(((torch_ref.correlation2d(a.double(), b.double(), md) - ref).abs() <= 1e-12 * S).all())
        assert bool((S >= ref.abs()).all())


@pytest.mark.parametrize("name", sorted(CASES))
def test_bar_has_teeth(name):
    """Dropping the term of one channel (the one of largest scale, kept in every sample) moves at least 99 % of the
    outputs with S > 0 over the bar, at the case's C, shape and values (two samples on the CPU)."""
    entry, _, C, H, W, md, _, _, kind, _ = CASES[name]
    a, b = make_inputs(min(case_batch(name, False), 2), C, H, W, _seed(name), kind)
    a, b = a.double(), b.double()
    ref, S = ref_corr2d(a, b, md)
    k = int((a.abs().mean((0, 2, 3)) * b.abs().mean((0, 2, 3))).argmax())
    dropped = a.clone()
    dropped[:, k] = 0
    wrong, _ = ref_corr2d(dropped, b, md)
    live = S > 0
    over = ((wrong - ref).abs() > bar_of(C, S)) & live
    frac = over.sum().item() / max(live.sum().item(), 1)
    assert live.any() and frac >= 0.99, f"{name}: only {frac:.4f} of the outputs move over the bar"


def test_route_mirror_unit_checks():
    # the NCHW entry: the widths corr2d_nchw_kernel takes (everything else with W % 4 == 0 is the diag kernel)
    assert [W for W in range(4, 400, 4) if route_of("nchw", 8, 8, W, 4) == "nchw32"] == \
        [4, 8, 12, 16, 20, 24, 28, 32, 52, 56, 60, 64, 156]
    for W in (30, 15, 6, 2):
        assert route_of("nchw", 8, 8, W, 4) == "enosup"
    for md in (1, 2, 3, 5):
        assert route_of("nchw", 8, 8, 48, md) == "enosup"
    assert route_of("nchw", 8, 8, 48, 4, in_off=1) == "enosup" and route_of("nchw", 8, 8, 48, 4, out_off=2) == "enosup"
    # the NHWC entry
    assert route_of("nhwc", 8, 8, 48, 5) == "any" and route_of("nhwc", 3, 8, 48, 64) == "any"
    assert route_of("nhwc", 8, 8, 48, 4) == "tma.v4"
    assert route_of("nhwc", 8, 8, 48, 4, out_off=2) == "tma.scalar" and route_of("nhwc", 8, 8, 50, 4) == "tma.scalar"
    assert route_of("nhwc", 8, 8, 48, 4, in_off=1) == "cp<4,false>" and route_of("nhwc", 9, 8, 48, 4) == "cp<4,false>"
    assert route_of("nhwc", 8, 8, 48, 3) == "cp<3,true>" and route_of("nhwc", 8, 8, 48, 3, in_off=2) == "cp<3,false>"
    assert route_of("nhwc", 8, 8, 48, 1, out_off=1) == "cp<1,true>"
    # the bench's five levels: diag, diag, nchw32, then W % 4 != 0 -> permute + the TMA kernel with scalar stores
    routes = [bench_route(c, *CONFIGS["things"].level_hw(lvl)) for lvl, c in zip(range(1, 6), LEVEL_CHANNELS)]
    assert routes == ["diag", "diag", "nchw32", "tma.scalar", "tma.scalar"]
    # every case claims the route the mirror computes, and the claims cover every reachable forward kernel
    for name, (entry, _, C, H, W, md, in_off, out_off, _, route) in CASES.items():
        assert route_of(entry, C, H, W, md, in_off, out_off) == route, name
    assert {kernel_of(r) for *_, r in CASES.values()} == FORWARD_KERNELS - UNREACHABLE
    assert persist_batch(9, 148) * 9 > 296 and persist_batch(9, 148) * 9 % 148


# ------------------------------------------------------------------------------------------------- GPU: every case
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_forward_vs_float64(name):
    entry, _, C, H, W, md, in_off, out_off, kind, route = CASES[name]
    a, b, ref, S = gpu_case(name)
    got = run_checked(entry, a, b, md, in_off, out_off, label=name)
    check_bar(route, got, ref, S, C, name)
    if entry == "nchw":
        leaky = run_checked(entry, a, b, md, in_off, out_off, slope=0.1, label=name)
        check_bar(route, leaky, ref, S, C, name, slope=0.1)


@pytest.mark.gpu
def test_every_case_reaches_its_route():
    """Each case launches exactly the kernel of the route it claims; the claims cover every forward kernel a call can
    reach (module docstring for corr2d_fwd_kernel<4,true>)."""
    wrong, seen = [], set()
    for name, (entry, B, C, H, W, md, in_off, out_off, kind, route) in CASES.items():
        a, b = make_inputs(2 if B is None else B, C, H, W, 1, kind)
        got = _kernel_names(lambda: run_entry(entry, a, b, md, in_off, out_off))
        seen |= got
        if got != {kernel_of(route)}:
            wrong.append(f"{name}: claims {route} ({kernel_of(route)}), launched {sorted(got)}")
    for lvl, C in zip(range(1, 6), LEVEL_CHANNELS):
        H, W = CONFIGS["things"].level_hw(lvl)
        a, b = (t.to(DEV) for t in make_inputs(1, C, H, W, lvl))
        got = _kernel_names(lambda: b200.correlation2d(a, b, 4))
        if got != {kernel_of(bench_route(C, H, W))}:
            wrong.append(f"bench level {lvl}: claims {bench_route(C, H, W)}, launched {sorted(got)}")
    assert not wrong, "\n".join(wrong)
    assert seen == FORWARD_KERNELS - UNREACHABLE, sorted(seen ^ (FORWARD_KERNELS - UNREACHABLE))


@pytest.mark.gpu
@pytest.mark.parametrize("in_off,out_off", [(0, 1), (0, 2), (1, 0), (2, 0)])
@pytest.mark.parametrize("md,W", [(4, 48), (4, 30), (3, 48)])
def test_nchw_entry_refuses_and_leaves_the_output_untouched(md, W, in_off, out_off):
    """B200_ENOSUP outside md = 4, W % 4 == 0 and 16-byte aligned pointers; not one output element is written."""
    a, b = make_inputs(2, 16, 9, W, 3)
    if md == 4 and W % 4 == 0:
        assert route_of("nchw", 16, 9, W, md, in_off, out_off) == "enosup"
    for slope in (None, 0.1):
        rc, out, guard = run_entry("nchw", a, b, md, in_off, out_off, slope)
        assert rc == _lib.B200_ENOSUP, rc
        assert bool(torch.isnan(out).all()) and bool(torch.isnan(guard).all())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["diag_W100_H1_C1", "diag_W72_H7_C17", "nchw32_W60_H12_C31", "nchw32_W156_H10_C12",
                                  "persist_diag_C40", "persist_nchw32_C48"])
def test_leaky_is_leaky_relu_of_the_plain_call(name):
    """correlation2d_leaky == leaky_relu(correlation2d) bit for bit on the NCHW routes, slopes 0, 0.1, 0.5, 1."""
    entry, _, C, H, W, md, _, _, kind, route = CASES[name]
    a, b, ref, S = gpu_case(name)
    a, b = a.to(DEV), b.to(DEV)
    plain = b200.correlation2d(a, b, md)
    check_bar(route, plain, ref, S, C, name + " ops")
    for slope in (0.0, 0.1, 0.5, 1.0):
        leaky = b200.correlation2d_leaky(a, b, md, slope)
        assert torch.equal(leaky, F.leaky_relu(plain, slope)), f"{name}: slope {slope}"


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,H,W", [(2, 32, 20, 100), (2, 33, 9, 60), (3, 64, 12, 56), (2, 96, 17, 240)])
def test_nchw_entry_and_nhwc_entry_both_meet_the_bar(B, C, H, W):
    """md = 4: b200_corr2d_fwd_nchw and b200_corr2d_fwd on the permuted maps, each against float64."""
    a, b = make_inputs(B, C, H, W, B * C + H + W)
    ref, S = ref_corr2d(a.to(DEV, torch.float64), b.to(DEV, torch.float64), 4)
    for entry in ("nchw", "nhwc"):
        route = route_of(entry, C, H, W, 4)
        check_bar(route, run_checked(entry, a, b, 4, label=f"{entry} B{B}_C{C}_H{H}_W{W}"), ref, S, C,
                  f"{entry} B{B}_C{C}_H{H}_W{W}")


# ------------------------------------------------------------------------------------------------- GPU: bench batch
@pytest.mark.gpu
@pytest.mark.parametrize("lvl", [1, 2, 3, 4, 5])
def test_bench_levels_at_bench_batch_equal_single_sample_calls(lvl):
    """The bench's correlation levels at BENCH_BATCH: correlation2d and correlation2d_leaky(0.1) of the batch equal the
    single-sample calls bit for bit; samples 0, B/2 and B-1 also meet the float64 bar."""
    C = LEVEL_CHANNELS[lvl - 1]
    H, W = CONFIGS["things"].level_hw(lvl)
    route = bench_route(C, H, W)
    B = BENCH_BATCH
    a, b = make_inputs(B, C, H, W, 1000 + lvl)
    a, b = a.to(DEV), b.to(DEV)
    for slope in (None, 0.1):
        call = (lambda x, y: b200.correlation2d(x, y, 4)) if slope is None else \
            (lambda x, y: b200.correlation2d_leaky(x, y, 4, slope))
        _poison_allocator(4 * B * 81 * H * W)
        batched = call(a, b)
        torch.cuda.synchronize()
        diff = []
        for i in range(B):
            _poison_allocator(4 * 81 * H * W)
            if not torch.equal(batched[i:i + 1], call(a[i:i + 1], b[i:i + 1])):
                diff.append(i)
        assert not diff, f"level {lvl} slope {slope}: samples whose batched result differs from their single call: {diff}"
        for i in (0, B // 2, B - 1):
            ref, S = ref_corr2d(a[i:i + 1].double(), b[i:i + 1].double(), 4)
            check_bar(route, batched[i:i + 1], ref, S, C, f"level {lvl} B{B} sample {i}", slope=slope)
        del batched
