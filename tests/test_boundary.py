"""CPU-only checks of the drop-in boundary: the C-ABI library loads, exports exactly what include/b200flow.h
declares, rejects bad arguments without touching a GPU, the product never imports the oracle, and the shims
satisfy the unmodified reference wrapper's import block (when a reference tree is staged under oracle/_ref)."""
import ctypes
import glob
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200flow.h")
REFERENCE = os.path.join(ROOT, "oracle", "_ref", "reference")      # `make -C oracle reftree REF=<RPEFlow checkout>`


def declared_symbols():
    text = open(HEADER).read()
    return sorted(set(re.findall(r"^B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(", text, flags=re.M)))


def test_library_exports_every_declared_symbol():
    from rpeflow_b200 import _lib
    names = declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(_lib.lib, n), f"{n} declared in b200flow.h but not exported"
    assert sorted(_lib.SIGNATURES) == names, "ctypes signature table and header disagree"
    assert _lib.lib.b200_abi_version() == _lib.ABI_VERSION
    assert b"sm_100a" in _lib.lib.b200_build_info()


def test_library_contains_sm100a_code_only():
    out = subprocess.run(["cuobjdump", "-lelf", os.path.join(ROOT, "rpeflow_b200", "libb200flow.so")],
                         capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = set(re.findall(r"sm_\d+a?", out.stdout))
    assert archs == {"sm_100a"}, archs


def test_argument_errors_are_reported_without_a_gpu():
    from rpeflow_b200 import _lib
    lib = _lib.lib
    one = ctypes.c_void_p(16)              # never dereferenced: argument checks come first
    assert lib.b200_knn(one, one, one, 1, 10, 10, 3, 33, None) == -1
    assert b"k must be in [1,32]" in lib.b200_last_error()
    assert lib.b200_knn(one, one, one, 1, 10, 10, 4, 3, None) == -1
    assert lib.b200_fps(one, one, 1, 100, 100, None) == -1
    assert b"N > n_samples" in lib.b200_last_error()
    assert lib.b200_fps(one, one, 1, 100000, 10, None) == -3
    assert lib.b200_corr2d_fwd(one, one, one, 1, 8, 4, 4, 65, None) == -1          # md in [1,64]: 5..64 take the plain kernel
    assert lib.b200_corr2d_fwd(None, one, one, 1, 8, 4, 4, 4, None) == -1
    assert lib.b200_event_voxel_int(one, 0, one, 5, 4, 4, 1, one, None) == -1
    assert lib.b200_corr3d_scratch_floats(2, 32, 32, 100, 100, 16) >= 3 * 2 * 100 * 32


def test_host_mirror_has_no_cpu_fallback():
    import rpeflow_b200 as b200
    x = torch.rand(1, 3, 64)
    with pytest.raises(RuntimeError, match="no CPU"):
        b200.k_nearest_neighbor(x, x, 4)
    with pytest.raises(RuntimeError, match="no CPU"):
        b200.correlation2d(torch.rand(1, 4, 8, 8), torch.rand(1, 4, 8, 8), 4)
    with pytest.raises(RuntimeError, match="no CPU"):
        b200.furthest_point_sampling(torch.rand(1, 64, 3), 8)
    with pytest.raises(RuntimeError, match="no CPU"):
        b200.grid_sample_wrapper(torch.rand(1, 4, 8, 8), torch.rand(1, 2, 5))
    with pytest.raises(RuntimeError):
        b200.ops._k_nearest_neighbor_cuda(x, x, 4)


def test_product_never_touches_the_oracle():
    pkg = os.path.join(ROOT, "rpeflow_b200")
    for base, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(base, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "liboracle" not in text and "/root/reference" not in text, f


ASYNC_PTX = ("mbarrier.", "tcgen05.", "cp.async.bulk", "fence.proxy", "fence.mbarrier_init", "bar.sync")


def test_kernels_call_the_async_ptx_helpers():
    """mbarrier, bulk/TMA copy, tcgen05, proxy-fence and named-barrier PTX is written once, in csrc/sm100_async.cuh
    (one bounded mbarrier wait for every kernel); no kernel file spells it out in a string literal of its own."""
    found = []
    for path in sorted(glob.glob(os.path.join(ROOT, "rpeflow_b200", "csrc", "*.cu"))):
        code = re.sub(r"/\*.*?\*/", lambda m: "\n" * m.group().count("\n"), open(path).read(), flags=re.S)
        for n, line in enumerate(code.split("\n"), 1):
            for tok in re.finditer(r'"(?:[^"\\\n]|\\.)*"|//.*', line):      # the first "//" outside a string ends the code
                if tok.group().startswith("//"):
                    break
                found += [f"{os.path.basename(path)}:{n}: {line.strip()}" for op in ASYNC_PTX if op in tok.group()]
    assert not found, "inline async PTX outside sm100_async.cuh:\n" + "\n".join(found)


ENVIRONMENT = {"B200FLOW_LIB", "B200_CHECK_INDICES", "B200_PROJECT_ROUTE"}


def test_environment_selects_no_kernel():
    """The inputs choose every kernel, not the process's environment.  The library reads only B200FLOW_LIB (load another
    build of libb200flow.so), B200_CHECK_INDICES (validate indices that come from outside the library) and
    B200_PROJECT_ROUTE (run the two-pass projection on a map the tiled route takes, so that both can be compared on one
    input); the native code reads only the last."""
    native = set()
    for path in sorted(glob.glob(os.path.join(ROOT, "rpeflow_b200", "csrc", "*.cu*"))):
        code = re.sub(r"/\*.*?\*/|//[^\n]*", "", open(path).read(), flags=re.S)
        for m in re.finditer(r"\bgetenv\b\s*(?:\(\s*\"(\w+)\")?", code):
            native.add(m.group(1) or f"{os.path.basename(path)}: {code[m.start():m.start() + 40]}")
    assert native <= {"B200_PROJECT_ROUTE"}, sorted(native)
    python = set()
    for path in sorted(glob.glob(os.path.join(ROOT, "rpeflow_b200", "**", "*.py"), recursive=True)):
        code = re.sub(r"#[^\n]*", "", open(path).read())
        for m in re.finditer(r"\b(?:environ|getenv)\b(?:(?:\.get\s*\(|\s*\[|\s*\()\s*([\"'])(\w+)\1)?", code):
            python.add(m.group(2) or f"{os.path.relpath(path, ROOT)}: {code[m.start():m.start() + 40]}")
    assert python <= ENVIRONMENT, sorted(python)


def test_same_names_as_the_reference_wrapper():
    import rpeflow_b200.ops as ops
    for n in ("correlation2d", "furthest_point_sampling", "k_nearest_neighbor", "squared_distance",
              "CorrelationFunction", "_correlation_forward_cuda", "_correlation_backward_cuda",
              "_furthest_point_sampling_cuda", "_k_nearest_neighbor_cuda"):
        assert hasattr(ops, n)
    from rpeflow_b200.shims import _correlation_cuda, _furthest_point_sampling_cuda, _k_nearest_neighbor_cuda
    assert _correlation_cuda._correlation_forward_cuda is ops._correlation_forward_cuda
    assert _furthest_point_sampling_cuda._furthest_point_sampling_cuda is ops._furthest_point_sampling_cuda
    assert _k_nearest_neighbor_cuda._k_nearest_neighbor_cuda is ops._k_nearest_neighbor_cuda


@pytest.mark.skipif(not os.path.isdir(os.path.join(REFERENCE, "models")), reason="no reference tree staged under oracle/_ref")
def test_unmodified_reference_wrapper_picks_up_the_shims():
    code = f"""
import sys
sys.dont_write_bytecode = True
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {REFERENCE!r})
import rpeflow_b200.install as inst
inst.install(patch_python=True)
import models.csrc.wrapper as w
import rpeflow_b200.ops as ops
assert w._correlation_forward_cuda is ops._correlation_forward_cuda
assert w._correlation_backward_cuda is ops._correlation_backward_cuda
assert w._furthest_point_sampling_cuda is ops._furthest_point_sampling_cuda
assert w._k_nearest_neighbor_cuda is ops._k_nearest_neighbor_cuda
import models.RPEFlow_core as core, models.pwc3d_core as p3
assert core.grid_sample_wrapper.__name__ == 'grid_sample_wrapper' and core.grid_sample_wrapper is not None
assert hasattr(p3.Correlation3D, '_b200_reference_forward')
# CPU tensors still take the reference's own torch path (no GPU here): results unchanged
import torch
x = torch.rand(1, 3, 50)
assert w.k_nearest_neighbor(x, x, 3).shape == (1, 50, 3)
m = p3.Correlation3D(8, 8, k=4)
assert m(x, torch.rand(1, 8, 50), x, torch.rand(1, 8, 50)).shape == (1, 8, 50)
# widened rows (SURVEY 8f): PointConv, knn_interpolation, backwarp_3d, correlation2d are re-bound too and keep working on CPU
import models.pointconv as pc, models.utils as mu
assert hasattr(pc.PointConvDownSampling, '_b200_reference_forward') and hasattr(pc.PointConvNoSampling, '_b200_reference_forward')
assert pc.PointConvNoSampling(8, 8)(x, torch.rand(1, 8, 50)).shape == (1, 8, 50)
assert pc.PointConvDownSampling(8, 8)(x, torch.rand(1, 8, 50), x[:, :, :20]).shape == (1, 8, 20)
assert mu.knn_interpolation(x, torch.rand(1, 5, 50), torch.rand(1, 3, 70)).shape == (1, 5, 70)
assert core.correlation2d(torch.rand(1, 4, 8, 8), torch.rand(1, 4, 8, 8), 4).shape == (1, 81, 8, 8)
assert mu.backwarp_2d(torch.rand(1, 4, 8, 8), torch.rand(1, 2, 8, 8), 'border').shape == (1, 4, 8, 8)
assert mu.convex_upsample(torch.rand(1, 2, 4, 4), torch.rand(1, 144, 4, 4), 4).shape == (1, 2, 16, 16)
print('SHIMS-OK')
"""
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert "SHIMS-OK" in out.stdout, out.stdout + out.stderr
    assert "Failed to load" not in out.stdout
