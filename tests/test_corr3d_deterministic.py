"""Correlation3D backward without float atomics (b200_corr3d_bwd_det, deterministic mode).

CPU: the new entries are in the header and the signature table; b200_corr3d_bwd_det rejects what b200_corr3d_bwd
rejects, with the same messages; B = 0 is a no-op; and the SASS of the deterministic kernels (DET instantiations, the
pull kernel, the split-K reduce, the inverse-index kernels) has no RED(G) / ATOM(G) / ATOMS instruction, while the atomic
path's kernels do.

GPU (-m gpu): all 20 gradients against fp64 autograd of oracle.torch_ref.correlation3d at test_corr3d_backward's bar for
every one of its CASES, also through b200.correlation3d and Correlation3D(differentiable=True) under
torch.use_deterministic_algorithms(True); bitwise repeatability (one run next to a long kernel on a second stream);
batch invariance of the input gradients; index edge cases; gradient subsets equal to the full run bit for bit;
agreement with the atomic path; install(train={"Correlation3D"}) routing; CUDA-graph replay.
"""
import contextlib
import ctypes
import os
import re
import shutil
import subprocess

import pytest
import torch

import rpeflow_b200 as b200
from rpeflow_b200 import _lib, pwc3d
from rpeflow_b200._lib import Corr3dGrads, Corr3dWeights
from test_corr3d_backward import BAR, CASES, GRAD_NAMES, _case, _near_kink_points, _oracle_grads, _worst

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200flow.h")
DEV = torch.device("cuda", 0)
INPUTS = ("xyz1", "feat1", "xyz2", "feat2")


# ------------------------------------------------------------------------------------------------- CPU
def test_det_entries_are_declared_and_bound():
    text = open(HEADER).read()
    declared = sorted(set(re.findall(r"^B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(", text, flags=re.M)))
    for name in ("b200_corr3d_bwd_det", "b200_corr3d_bwd_det_scratch_bytes"):
        assert name in declared and name in _lib.SIGNATURES
    assert _lib.SIGNATURES["b200_corr3d_bwd_det"] == _lib.SIGNATURES["b200_corr3d_bwd"]
    assert "b200_corr3d_bwd_det" in _lib.KERNELS_PER_CALL
    assert _lib.ABI_VERSION == 8 and _lib.lib.b200_abi_version() == 8


def _calls(entry):
    one = ctypes.c_void_p(16)              # never dereferenced: argument checks come first
    g = Corr3dGrads(**{n: 16 for n in Corr3dGrads.NAMES})

    def call(xyz1=one, scratch=one, B=1, k=16, w="ok", Cout=8):
        ws = Corr3dWeights(**{n: 16 for n in Corr3dWeights.NAMES})
        if w == "null_field":
            ws.n2_bc = None
        wp = None if w is None else ctypes.byref(ws)
        rc = entry(xyz1, one, one, one, one, one, wp, one, one, ctypes.byref(g), scratch, B, 8, Cout, 64, 64, k, None)
        return rc, _lib.lib.b200_last_error()
    return call


@pytest.mark.parametrize("bad", [dict(k=33), dict(k=0), dict(xyz1=None), dict(w=None),
                                 dict(scratch=ctypes.c_void_p(20)), dict(w="null_field"), dict(Cout=513), dict(B=-1),
                                 dict(B=65536)])
def test_det_rejects_what_the_atomic_entry_rejects(bad):
    rc_a, msg_a = _calls(_lib.lib.b200_corr3d_bwd)(**bad)
    rc_d, msg_d = _calls(_lib.lib.b200_corr3d_bwd_det)(**bad)
    assert rc_a == rc_d == -1
    assert msg_a.startswith(b"b200_corr3d_bwd: ") and msg_d.startswith(b"b200_corr3d_bwd_det: ")
    assert msg_d[len(b"b200_corr3d_bwd_det: "):] == msg_a[len(b"b200_corr3d_bwd: "):]


def test_det_batch_zero_is_a_no_op():
    w = Corr3dWeights(**{n: 16 for n in Corr3dWeights.NAMES})
    g = Corr3dGrads(**{n: 16 for n in Corr3dGrads.NAMES})
    assert _lib.lib.b200_corr3d_bwd_det(None, None, None, None, None, None, ctypes.byref(w), None, None, ctypes.byref(g),
                                        None, 0, 8, 8, 64, 64, 16, None) == 0
    assert _lib.lib.b200_corr3d_bwd_det_scratch_bytes(0, 8, 8, 64, 64, 16) == 0


def _cuobjdump():
    found = shutil.which("cuobjdump")
    if found:
        return found
    for home in (os.environ.get("CUDA_HOME"), "/usr/local/cuda"):
        if home and os.path.exists(os.path.join(home, "bin", "cuobjdump")):
            return os.path.join(home, "bin", "cuobjdump")
    return None


def _sass_by_kernel():
    tool = _cuobjdump()
    if tool is None:
        pytest.skip("cuobjdump not found")
    text = subprocess.run([tool, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in text.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur is not None:
            out[cur].append(line)
    return out


ATOMIC = re.compile(r"\b(RED|REDG|ATOM|ATOMG|ATOMS)\b")     # sm_100 spells the global forms REDG / ATOMG


def test_deterministic_kernels_have_no_atomic_instructions():
    sass = _sass_by_kernel()
    # mangled names: <true> is ILb1E, <false> ILb0E
    det = [n for n in sass if re.search(r"corr3d_bwd_stage[12]_kernelI(Li\d+E)?Lb1E", n)
           or re.search(r"linear_bwd_w_kernelILb1E", n)
           or re.search(r"(corr3d_det_pull|corr3d_det_keys|corr3d_det_offsets|linear_bwd_w_reduce)_kernel", n)]
    assert len(det) == 10, det            # stage2<true>, stage1<4|8|16|32, true>, w<true>, w reduce, pull, keys, offsets
    for n in det:
        hits = [l.strip() for l in sass[n] if ATOMIC.search(l)]
        assert not hits, (n, hits[:3])
    atomic = [n for n in sass if re.search(r"corr3d_bwd_stage[12]_kernelI(Li\d+E)?Lb0E", n)
              or re.search(r"linear_bwd_w_kernelILb0E", n)]
    assert len(atomic) == 6, atomic
    for n in atomic:                      # the scan sees the atomics the other path does use
        assert any(ATOMIC.search(l) for l in sass[n]), n


# ------------------------------------------------------------------------------------------------- GPU helpers
@contextlib.contextmanager
def deterministic():
    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(before)


def _det_run(c, want=GRAD_NAMES, det=True, precision=2, side_kernel=None):
    """b200.correlation3d forward + backward; det selects deterministic mode for both."""
    leaves = {n: c[n].to(DEV).requires_grad_(n in want) for n in INPUTS}
    wts = {n: v.to(DEV).requires_grad_(n in want) for n, v in c["w"].items()}
    knn12, knn11, grad = c["knn12"].to(DEV), c["knn11"].to(DEV), c["grad"].to(DEV)
    with deterministic() if det else contextlib.nullcontext():
        out = b200.correlation3d(leaves["xyz1"], leaves["feat1"], leaves["xyz2"], leaves["feat2"], wts, knn12, knn11,
                                 precision)
        if side_kernel is not None:
            side_kernel()
        out.backward(grad)
    got = {n: t.grad for n, t in leaves.items()}
    got.update({n: t.grad for n, t in wts.items()})
    return out.detach(), got


def _assert_within_bar(got, ref, names=GRAD_NAMES, tag=""):
    ratios = {n: _worst(got[n], ref[n]) / BAR for n in names}
    print(f"\n[{tag}] worst max|diff| / (1e-4 max|ref|): " + " ".join(f"{n}={r:.3g}" for n, r in ratios.items()))
    bad = {n: r for n, r in ratios.items() if not r <= 1.0}
    assert not bad, bad


def _assert_equal(a, b, names=GRAD_NAMES):
    for n in names:
        assert torch.equal(a[n], b[n]), n


# ------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_all_gradients_vs_fp64_oracle(name):
    c = _case(*CASES[name][:6], seed=len(name), dup=CASES[name][6])
    ref_out, ref = _oracle_grads(c)
    out, got = _det_run(c)
    assert _worst(out, ref_out) <= BAR
    _assert_within_bar(got, ref, tag=name)


@pytest.mark.gpu
def test_module_differentiable_in_deterministic_mode():
    C, N, k = 48, 700, 16
    c = _case(2, C, C, N, N, k, seed=11)
    mod = c["mod"].to(DEV)
    mod.differentiable = True
    x1, f1, x2, f2 = (c[n].to(DEV).requires_grad_(True) for n in INPUTS)
    with deterministic():
        out = mod(x1, f1, x2, f2, c["knn11"].to(DEV))
        out.backward(c["grad"].to(DEV))
    _, ref = _oracle_grads(c)
    got = dict(zip(INPUTS, (x1.grad, f1.grad, x2.grad, f2.grad)))
    params = {n: (v._base if v._base is not None else v) for n, v in pwc3d.param_weights(mod).items()}
    got.update({n: params[n].grad.reshape(ref[n].shape) for n in Corr3dWeights.NAMES})
    _assert_within_bar(got, ref, tag="module")


@pytest.mark.gpu
def test_bitwise_repeatable_also_next_to_a_busy_stream():
    c = _case(2, 64, 64, 2048, 2048, 16, seed=21)
    _, first = _det_run(c)
    _, second = _det_run(c)
    side = torch.cuda.Stream()
    big = torch.ones(1 << 26, device=DEV)

    def busy():                           # unrelated kernels (~10 ms in all) on a second stream during the backward
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(150):
                big.mul_(1.0)
    _, third = _det_run(c, side_kernel=busy)
    torch.cuda.synchronize()
    _assert_equal(first, second)
    _assert_equal(first, third)


@pytest.mark.gpu
def test_input_gradients_do_not_depend_on_the_rest_of_the_batch():
    c = _case(4, 32, 40, 900, 800, 16, seed=23)
    _, full = _det_run(c)
    for b in range(4):
        one = dict(c)
        for n in INPUTS + ("knn12", "knn11", "grad"):
            one[n] = c[n][b:b + 1].contiguous()
        _, alone = _det_run(one)
        for n in INPUTS:
            assert torch.equal(full[n][b:b + 1], alone[n]), (b, n)


def _edge_case(kind, k=16):
    if kind == "identical_clouds":            # every query has the same neighbour list
        c = _case(2, 16, 24, 64, 64, k, seed=31)
        for n in ("xyz1", "xyz2"):
            c[n] = c[n][:, :, :1].expand(-1, -1, 64).contiguous() + 0.0
        c["knn11"] = torch.arange(k).expand(2, 64, k).contiguous()
        c["knn12"] = c["knn11"].clone()
        return c
    if kind == "one_point_for_all_rows":
        c = _case(2, 16, 24, 200, 150, k, seed=32)
        c["knn11"] = torch.full_like(c["knn11"], 7)
        c["knn12"] = torch.full_like(c["knn12"], 5)
        return c
    if kind == "N2_below_k":
        return _case(2, 16, 24, 70, 10, k, seed=33)
    if kind == "out_of_range":
        c = _case(2, 16, 24, 300, 250, k, seed=34)
        gen = torch.Generator().manual_seed(34)
        for n, N in (("knn11", 300), ("knn12", 250)):
            c[n] = torch.randint(-40, N + 40, c[n].shape, generator=gen)
        return c
    if kind == "N1_is_1":
        return _case(2, 16, 24, 1, 40, k, seed=35)
    raise KeyError(kind)


EDGES = ["identical_clouds", "one_point_for_all_rows", "N2_below_k", "out_of_range", "N1_is_1", "k1", "k4", "k16", "k32"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", EDGES)
def test_index_edge_cases(kind):
    c = _case(2, 16, 24, 300, 280, int(kind[1:]), seed=36) if kind.startswith("k") else _edge_case(kind)
    ref_c = dict(c)
    if kind == "out_of_range":                # the reference gathers what the kernels read: clamped indices
        ref_c["knn11"] = c["knn11"].clamp(0, c["feat1"].shape[2] - 1)
        ref_c["knn12"] = c["knn12"].clamp(0, c["feat2"].shape[2] - 1)
    c["grad"] = ref_c["grad"] = c["grad"] * (~_near_kink_points(ref_c))[:, None, :]
    ref_out, ref = _oracle_grads(ref_c)
    out, first = _det_run(c)
    _, second = _det_run(c)
    assert _worst(out, ref_out) <= BAR
    _assert_within_bar(first, ref, tag=kind)
    _assert_equal(first, second)


@pytest.mark.gpu
@pytest.mark.parametrize("subset", [Corr3dWeights.NAMES, ("feat1", "feat2"), ("xyz2",), ("xyz1",), ("W1",), ("b1", "xyz2")])
def test_gradient_subsets_equal_the_full_run(subset):
    c = _case(2, 32, 40, 600, 600, 16, seed=3)
    _, full = _det_run(c)
    _, part = _det_run(c, want=subset)
    for n in GRAD_NAMES:
        if n in subset:
            assert part[n] is not None and torch.equal(part[n], full[n]), n
        else:
            assert part[n] is None, n


@pytest.mark.gpu
def test_deterministic_and_atomic_paths_agree_on_the_same_forward():
    c = _case(2, 64, 64, 2048, 2048, 16, seed=5)
    leaves = {n: c[n].to(DEV).requires_grad_(True) for n in INPUTS}
    wts = {n: v.to(DEV).requires_grad_(True) for n, v in c["w"].items()}
    every = list(leaves.values()) + list(wts.values())
    out = b200.correlation3d(leaves["xyz1"], leaves["feat1"], leaves["xyz2"], leaves["feat2"], wts, c["knn12"].to(DEV),
                             c["knn11"].to(DEV))
    grad = c["grad"].to(DEV)
    got = []
    for det in (False, True):
        for t in every:
            t.grad = None
        with deterministic() if det else contextlib.nullcontext():
            out.backward(grad, retain_graph=True)
        got.append({n: t.grad.clone() for n, t in zip(GRAD_NAMES, list(leaves.values()) + [wts[n] for n in Corr3dWeights.NAMES])})
    _assert_within_bar(got[1], {n: v.double().cpu() for n, v in got[0].items()}, tag="det vs atomic")


@pytest.mark.gpu
def test_install_trains_correlation3d_in_deterministic_mode():
    import torch.nn as nn
    import rpeflow_b200.install as inst

    class Conv(nn.Module):                    # the reference's layer shape: conv_fn plus an identity norm
        def __init__(self, cin, cout):
            super().__init__()
            self.conv_fn = nn.Conv2d(cin, cout, 1)
            self.norm_fn = nn.Identity()

    class MLP(nn.Module):
        def __init__(self, cin, widths):
            super().__init__()
            chans = [cin] + list(widths)
            self.convs = nn.ModuleList(Conv(a, b) for a, b in zip(chans[:-1], chans[1:]))

    class RefCorrelation3D(nn.Module):        # stands in for models.pwc3d_core.Correlation3D
        def __init__(self, cin, cout, k):
            super().__init__()
            self.k = k
            self.cost_mlp = MLP(3 + 2 * cin, [cout, cout])
            self.weight_net1 = MLP(3, [8, 8, cout])
            self.weight_net2 = MLP(3, [8, 8, cout])

        def _b200_reference_forward(self, *args):
            raise AssertionError("reference route")

    c = _case(2, 32, 32, 500, 500, 16, seed=41)
    mod = RefCorrelation3D(32, 32, 16).to(DEV)
    mod.load_state_dict(c["mod"].state_dict())
    x1, f1, x2, f2 = (c[n].to(DEV).requires_grad_(True) for n in INPUTS)
    knn11, grad = c["knn11"].to(DEV), c["grad"].to(DEV)

    def run(train):
        saved, inst._TRAIN = inst._TRAIN, frozenset(train)
        inst.stats(reset=True)
        try:
            for t in (x1, f1, x2, f2, *mod.parameters()):
                t.grad = None
            with deterministic():
                inst._corr3d_forward(mod, x1, f1, x2, f2, knn11).backward(grad)
        finally:
            inst._TRAIN = saved
        return inst.stats(), [t.grad.clone() for t in (x1, f1, x2, f2)]

    st, via_install = run({"Correlation3D"})
    assert st["Correlation3D.forward"] == {"b200": 1, "reference": 0}
    _, direct = _det_run(c, want=INPUTS)
    for n, g in zip(INPUTS, via_install):
        assert torch.equal(g, direct[n]), n
    with pytest.raises(AssertionError, match="reference route"):
        run(set())
    assert inst.stats()["Correlation3D.forward"] == {"b200": 0, "reference": 1}


@pytest.mark.gpu
def test_cuda_graph_replay_matches_eager_gradients_bit_for_bit():
    c = _case(2, 64, 64, 1024, 1024, 16, seed=13)
    leaves = {n: c[n].to(DEV).requires_grad_(True) for n in INPUTS}
    wts = {n: v.to(DEV).requires_grad_(True) for n, v in c["w"].items()}
    knn12, knn11, grad = c["knn12"].to(DEV), c["knn11"].to(DEV), c["grad"].to(DEV)
    every = list(leaves.values()) + list(wts.values())

    def step():
        out = b200.correlation3d(leaves["xyz1"], leaves["feat1"], leaves["xyz2"], leaves["feat2"], wts, knn12, knn11)
        out.backward(grad)

    with deterministic():
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
        assert torch.equal(t.grad, e)


def _direct_det_bwd(x, w, knn12, knn11, grad, names, guard=4 << 20):
    """b200_corr3d_bwd_det called directly, only the gradients in names requested (NaN-filled first).  The scratch is
    exactly b200_corr3d_bwd_det_scratch_bytes long and followed by a guard band that must stay untouched."""
    xyz1, feat1, xyz2, feat2 = x
    _, fwd = pwc3d._corr3d_run(xyz1, feat1, xyz2, feat2, w, knn12, knn11, 2)
    B, Cin, N1 = feat1.shape
    N2, k, Cout = feat2.shape[2], knn12.shape[2], w["W2"].shape[0]
    shapes = dict(zip(INPUTS, x), **w)
    grads = {n: torch.full_like(shapes[n], float("nan")) for n in names}
    nbytes = _lib.lib.b200_corr3d_bwd_det_scratch_bytes(B, Cin, Cout, N1, N2, k)
    assert nbytes > 0
    buf = torch.full((nbytes + guard,), 0x5A, dtype=torch.uint8, device=DEV)
    ws = Corr3dWeights(**{n: w[n].data_ptr() for n in Corr3dWeights.NAMES})
    gs = Corr3dGrads(**{n: (grads[n].data_ptr() if n in grads else None) for n in Corr3dGrads.NAMES})
    _lib.check(_lib.lib.b200_corr3d_bwd_det(xyz1.data_ptr(), feat1.data_ptr(), xyz2.data_ptr(), feat2.data_ptr(),
                                            knn12.data_ptr(), knn11.data_ptr(), ctypes.byref(ws), grad.data_ptr(),
                                            fwd.data_ptr(), ctypes.byref(gs), buf.data_ptr(), B, Cin, Cout, N1, N2, k,
                                            torch.cuda.current_stream().cuda_stream), "b200_corr3d_bwd_det")
    torch.cuda.synchronize()
    assert bool((buf[nbytes:] == 0x5A).all()), "write past the end of the scratch"
    return grads


@pytest.mark.gpu
@pytest.mark.parametrize("B,Cin,Cout,N1,N2,k", [(1, 128, 64, 37888, 1000, 1), (16, 64, 64, 4096, 1024, 16)])
def test_w1_without_b1_stays_inside_the_scratch_and_equals_the_full_run(B, Cin, Cout, N1, N2, k):
    """Cin % 64 == 0 and N2 << N1: the split-K plan of the feat1 half of dW1 is the one with the bias column whether or
    not db1 is asked for, so the partial buffer fits and the W1-only and b1-only runs sum in the full run's order."""
    gen = torch.Generator().manual_seed(B + Cin)
    x = [torch.rand(B, 3, N1, generator=gen), torch.randn(B, Cin, N1, generator=gen),
         torch.rand(B, 3, N2, generator=gen), torch.randn(B, Cin, N2, generator=gen)]
    x = [t.to(DEV) for t in x]
    knn12 = torch.randint(0, N2, (B, N1, k), generator=gen).to(DEV)
    knn11 = torch.randint(0, N1, (B, N1, k), generator=gen).to(DEV)
    grad = torch.randn(B, Cout, N1, generator=gen).to(DEV)
    torch.manual_seed(0)
    w = {n: v.to(DEV) for n, v in pwc3d.pack_weights(pwc3d.Correlation3D(Cin, Cout, k=k)).items()}
    full = _direct_det_bwd(x, w, knn12, knn11, grad, GRAD_NAMES)
    for names in (("W1",), ("b1",), ("W1", "feat2")):
        part = _direct_det_bwd(x, w, knn12, knn11, grad, names)
        for n in names:
            assert torch.equal(part[n], full[n]), (names, n)
