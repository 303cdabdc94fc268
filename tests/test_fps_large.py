"""Furthest point sampling on clouds of more than 65536 points (b200_fps_large, fps_large.cu): index-identical to the C
oracle (oracle/spec.c::orc_fps) at every size, through every layer from the C-ABI to install().

Where the oracle's O(N * S) scan is too slow for the CPU (S = N / 8 on clouds of 1 M points and more), the picks are
compared with a full scan written in torch on the GPU: one elementwise kernel per fp32 operation of the distance rule
(so no contraction), torch.minimum, and torch.argmax (first occurrence = lowest index).  That scan is itself checked
against the oracle in test_torch_full_scan_is_the_oracle.
"""
import ctypes
import sys
import types

import numpy as np
import pytest
import torch

from oracle import spec

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import rpeflow_b200 as b200
    from rpeflow_b200 import _lib
    DEV = torch.device("cuda", 0)


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def fps(xyz, S):
    return b200.ops._furthest_point_sampling_cuda(xyz if isinstance(xyz, torch.Tensor) else cu(xyz), S)


def uniform(rng, B, N):
    return rng.random((B, N, 3), dtype=np.float32)


def ft3d(rng, B, N):
    """FlyingThings3D-shaped: a 30 x 17 x 90 box in front of the camera, as the bench clouds (workload.py)."""
    return (rng.random((B, N, 3), dtype=np.float32) * np.array([30, 17, 90], np.float32)
            + np.array([-15, -8, 22], np.float32)).astype(np.float32)


def torch_full_scan(xyz, S):
    """[B,N,3] CUDA -> [B,S] int64 by the reference's own loop (wrapper.py:83-96) with the stated rule."""
    B, N, _ = xyz.shape
    x, y, z = xyz[..., 0], xyz[..., 1], xyz[..., 2]
    dist = torch.full((B, N), 1e10, device=xyz.device)
    out = torch.empty((B, S), dtype=torch.int64, device=xyz.device)
    cur = torch.zeros(B, dtype=torch.int64, device=xyz.device)
    ar = torch.arange(B, device=xyz.device)
    for s in range(S):
        out[:, s] = cur
        c = xyz[ar, cur]                                          # [B,3]
        dx, dy, dz = x - c[:, 0:1], y - c[:, 1:2], z - c[:, 2:3]
        d = torch.add(torch.mul(dx, dx), torch.mul(dy, dy))
        d = torch.add(d, torch.mul(dz, dz))
        dist = torch.minimum(dist, d)
        cur = torch.argmax(dist, dim=1)
    return out


# ------------------------------------------------------------------------------------------------- oracle exactness
@pytest.mark.parametrize("N", [65537, 100003, 262144, 1048576, 4194304])
def test_small_s_vs_oracle(N):
    rng = np.random.default_rng(N)
    xyz = np.concatenate([uniform(rng, 1, N), ft3d(rng, 1, N)])
    S = 300
    np.testing.assert_array_equal(fps(xyz, S).cpu().numpy(), spec.fps(xyz, S))


@pytest.mark.parametrize("N", [65537, 100003, 262144])
def test_s_is_n_over_8_vs_oracle(N):
    rng = np.random.default_rng(N + 1)
    xyz = np.concatenate([ft3d(rng, 1, N), uniform(rng, 1, N)])
    np.testing.assert_array_equal(fps(xyz, N // 8).cpu().numpy(), spec.fps(xyz, N // 8))


def test_torch_full_scan_is_the_oracle():
    rng = np.random.default_rng(7)
    xyz = ft3d(rng, 2, 70001)
    xyz[:, 100:140] = xyz[:, 0:40]
    np.testing.assert_array_equal(torch_full_scan(cu(xyz), 2000).cpu().numpy(), spec.fps(xyz, 2000))


@pytest.mark.parametrize("N", [1048576, 4194304])
def test_s_is_n_over_8_vs_full_scan(N):
    g = torch.Generator(device=DEV).manual_seed(N)
    xyz = torch.rand(1, N, 3, device=DEV, generator=g) * torch.tensor([30.0, 17.0, 90.0], device=DEV)
    got = fps(xyz, N // 8)
    assert torch.equal(got, torch_full_scan(xyz, N // 8))


def test_s_is_n_minus_1():
    rng = np.random.default_rng(66000)
    xyz = uniform(rng, 1, 66000)
    np.testing.assert_array_equal(fps(xyz, 65999).cpu().numpy(), spec.fps(xyz, 65999))


def _adversarial(N, rng):
    dup = ft3d(rng, 1, N)[0]
    dup[-5000:] = dup[:5000]                                      # duplicates of the first points at the end of the cloud
    far = ft3d(rng, 1, N)[0]
    far[N - 2000:] = far[:2000] + np.float32(1e-3)                # near copies placed in the last CTA's slot range by distance
    same = np.full((N, 3), 1.5, np.float32)
    line = np.zeros((N, 3), np.float32); line[:, 0] = rng.random(N, dtype=np.float32)
    plane = rng.random((N, 3), dtype=np.float32); plane[:, 2] = 0.25
    clus = (rng.random((N, 3), dtype=np.float32) * 0.01 + rng.integers(0, 4, (N, 1)).astype(np.float32)).astype(np.float32)
    clus[[7, N // 2, N - 3]] = [[50.0, 0, 0], [0, -40.0, 0], [0, 0, 60.0]]   # far outliers
    k = int(np.ceil(N ** (1 / 3)))
    lat = (np.stack(np.meshgrid(*[np.arange(k, dtype=np.float32)] * 3, indexing="ij"), -1).reshape(-1, 3)[:N]
           * np.float32(2.0 ** -11))                              # exact distance ties
    rng.shuffle(lat)
    return {"dup": dup, "near-copies": far, "identical": same, "line": line, "plane": plane, "clusters+outliers": clus,
            "lattice": np.ascontiguousarray(lat)}


def test_adversarial_clouds_vs_oracle():
    rng = np.random.default_rng(11)
    clouds = _adversarial(70000, rng)
    xyz = np.stack(list(clouds.values()))
    S = 3000
    got, want = fps(xyz, S).cpu().numpy(), spec.fps(xyz, S)
    for i, name in enumerate(clouds):
        np.testing.assert_array_equal(got[i], want[i], err_msg=name)


def test_padding_slots_ignore_old_scratch_contents():
    """Above 81920 points the sorted points live in scratch; its padding slots must not inherit indices left there by
    earlier work.  Identical points make every row's maximum 0, the case where a stale padding index would win."""
    N = 100003
    need = b200._lib.lib.b200_fps_scratch_bytes(1, N)
    junk = torch.randint(0, 50, (need // 4 + 4096,), dtype=torch.int32, device=DEV)    # small "indices" everywhere
    del junk
    xyz = np.full((1, N, 3), 2.5, np.float32)
    xyz[0, 777] = 3.0
    np.testing.assert_array_equal(fps(xyz, 64).cpu().numpy(), spec.fps(xyz, 64))


def test_ties_across_ctas():
    """Exact copies of points that sort into the first CTA's range, spread over every other CTA's range by a shuffle:
    ties between CTAs go to the lowest original index."""
    rng = np.random.default_rng(3)
    N = 131072
    xyz = ft3d(rng, 1, N)[0]
    order = np.argsort(xyz[:, 2])                                 # z-slabs: far apart in Morton order
    xyz[order[-4000:]] = xyz[order[:4000]]
    xyz = xyz[None]
    np.testing.assert_array_equal(fps(xyz, 5000).cpu().numpy(), spec.fps(xyz, 5000))


# ------------------------------------------------------------------------------------------------- properties
def test_prefix_property():
    g = torch.Generator(device=DEV).manual_seed(2)
    xyz = torch.rand(2, 200000, 3, device=DEV, generator=g)
    full = fps(xyz, 6000)
    for s in (1, 2, 1234, 5999):
        assert torch.equal(full[:, :s], fps(xyz, s))


def test_batch_under_cluster_waves():
    """40 clouds x 8 CTAs: more clusters than fit at once, so they run in waves; each cloud as its own call."""
    g = torch.Generator(device=DEV).manual_seed(40)
    xyz = torch.rand(40, 70000, 3, device=DEV, generator=g) * torch.tensor([30.0, 17.0, 90.0], device=DEV)
    xyz[5, 1000:3000] = xyz[5, 0]
    got = fps(xyz, 1500)
    assert torch.equal(got, torch.cat([fps(xyz[b:b + 1].contiguous(), 1500) for b in range(40)]))
    np.testing.assert_array_equal(got[:3].cpu().numpy(), spec.fps(xyz[:3].cpu().numpy(), 1500))
    assert fps(torch.empty(0, 70000, 3, device=DEV), 10).shape == (0, 10)


# ------------------------------------------------------------------------------------------------- every layer
def test_ops_and_shim_agree():
    from rpeflow_b200.shims import _furthest_point_sampling_cuda as shim
    g = torch.Generator(device=DEV).manual_seed(9)
    xyz = torch.rand(2, 80000, 3, device=DEV, generator=g)
    a = b200.furthest_point_sampling(xyz, 700)
    assert a.dtype == torch.int64
    assert torch.equal(a, shim._furthest_point_sampling_cuda(xyz, 700))
    assert torch.equal(a, b200.furthest_point_sampling(xyz.transpose(1, 2).contiguous().transpose(1, 2), 700))


def test_install_counts_large_clouds_as_b200(monkeypatch):
    """install() re-binds wrapper.furthest_point_sampling; with stand-in reference modules (no checkout needed) a call on
    a 100000-point cloud runs this library's kernels."""
    import rpeflow_b200.install as inst
    ref_calls = []
    models, utils, csrc, wrapper = (types.ModuleType(n) for n in ("models", "models.utils", "models.csrc", "models.csrc.wrapper"))
    for n in ("batch_indexing_channel_first", "batch_indexing_channel_last", "grid_sample_wrapper", "project_feat_with_nn_corr",
              "knn_interpolation", "backwarp_3d", "backwarp_2d", "convex_upsample"):
        setattr(utils, n, lambda *a, **k: None)
    for n in ("correlation2d", "k_nearest_neighbor"):
        setattr(wrapper, n, lambda *a, **k: None)
    wrapper.furthest_point_sampling = lambda xyz, n_samples, cpp_impl=True: ref_calls.append(n_samples)
    models.utils, models.csrc, csrc.wrapper = utils, csrc, wrapper
    for name, mod in (("models", models), ("models.utils", utils), ("models.csrc", csrc), ("models.csrc.wrapper", wrapper)):
        monkeypatch.setitem(sys.modules, name, mod)
    g = torch.Generator(device=DEV).manual_seed(1)
    xyz = torch.rand(1, 100000, 3, device=DEV, generator=g)
    try:
        inst.install(patch_python=True, extensions=False, only={"furthest_point_sampling"})
        inst.stats(reset=True)
        got = wrapper.furthest_point_sampling(xyz, 500)
        assert inst.stats()["furthest_point_sampling"] == {"b200": 1, "reference": 0} and not ref_calls
        np.testing.assert_array_equal(got.cpu().numpy(), spec.fps(xyz.cpu().numpy(), 500))
    finally:
        inst.uninstall()
        inst.stats(reset=True)


def test_build_pc_pyramid_large_pair():
    g = torch.Generator(device=DEV).manual_seed(4)
    pc1 = torch.rand(1, 3, 131072, device=DEV, generator=g)
    pc2 = torch.rand(1, 3, 131072, device=DEV, generator=g)
    xyzs1, xyzs2, ids1, ids2 = b200.build_pc_pyramid(pc1, pc2, [8192, 4096, 1024, 256])
    assert [x.shape[-1] for x in xyzs1] == [131072, 8192, 4096, 1024, 256]
    for lvl in range(2, 5):
        assert torch.equal(ids1[lvl], ids1[1][:, :ids1[lvl].shape[1]])
        assert torch.equal(ids2[lvl], ids2[1][:, :ids2[lvl].shape[1]])
    assert torch.equal(xyzs2[2], torch.gather(pc2, 2, ids2[2].unsqueeze(1).expand(-1, 3, -1)))
    both = torch.cat([pc1, pc2]).transpose(1, 2).contiguous().cpu().numpy()
    want = spec.fps(both, 8192)
    np.testing.assert_array_equal(ids1[1].cpu().numpy(), want[:1])
    np.testing.assert_array_equal(ids2[1].cpu().numpy(), want[1:])


# ------------------------------------------------------------------------------------------------- errors, robustness
def test_scratch_checked_through_ctypes():
    lib = _lib.lib
    B, N, S = 1, 70000, 100
    xyz = torch.rand(B, N, 3, device=DEV)
    out = torch.zeros(B, S, dtype=torch.int64, device=DEV)
    need = lib.b200_fps_scratch_bytes(B, N)
    assert need > B * N * 20 and lib.b200_fps_scratch_bytes(-1, N) == -1
    scratch = torch.empty(need + 256, dtype=torch.uint8, device=DEV)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.b200_fps_large(xyz.data_ptr(), out.data_ptr(), scratch.data_ptr(), need - 1, B, N, S, stream) == -1
    assert b"scratch too small" in lib.b200_last_error()
    assert lib.b200_fps_large(xyz.data_ptr(), out.data_ptr(), scratch.data_ptr() + 4, need, B, N, S, stream) == -1
    assert b"aligned" in lib.b200_last_error()
    assert lib.b200_fps_large(xyz.data_ptr(), out.data_ptr(), None, need, B, N, S, stream) == -1
    assert lib.b200_fps_large(xyz.data_ptr(), out.data_ptr(), scratch.data_ptr(), need, B, N, N, stream) == -1
    assert lib.b200_fps_large(None, None, None, 0, 0, N, S, stream) == 0              # B = 0: nothing to do
    assert lib.b200_fps(xyz.data_ptr(), out.data_ptr(), B, N, S, stream) == _lib.B200_ENOSUP
    assert b"b200_fps_large" in lib.b200_last_error()
    assert torch.count_nonzero(out) == 0                                              # no rejected call wrote anything
    assert lib.b200_fps_large(xyz.data_ptr(), out.data_ptr(), scratch.data_ptr(), need, B, N, S, stream) == 0
    np.testing.assert_array_equal(out.cpu().numpy(), spec.fps(xyz.cpu().numpy(), S))


def test_host_layer_errors():
    x = torch.rand(1, 70000, 3, device=DEV)
    with pytest.raises(RuntimeError):
        b200.ops._furthest_point_sampling_cuda(x.cpu(), 10)
    with pytest.raises(RuntimeError, match="N > n_samples"):
        b200.ops._furthest_point_sampling_cuda(x, 70000)
    with pytest.raises(AssertionError):
        b200.furthest_point_sampling(x, 70000)                                        # wrapper.py:98
    with pytest.raises(RuntimeError):
        b200.furthest_point_sampling(x.cpu(), 10)


def test_non_finite_rows_finish_in_range():
    rng = np.random.default_rng(12)
    N = 90000
    xyz = uniform(rng, 3, N)
    xyz[0, 10:20] = np.nan
    xyz[1, 30:40, 1] = np.inf
    xyz[1, 50:60, 2] = -np.inf
    xyz[2, 0] = np.nan                                                                # the first centre itself
    xyz[2, 5000:5100] = np.nan
    got = fps(xyz, 4000).cpu().numpy()
    assert got.shape == (3, 4000) and got.min() >= 0 and got.max() < N


# ------------------------------------------------------------------------------------------------- CUDA graphs
def test_cuda_graph_capture_replays_eager():
    lib = _lib.lib
    B, N, S = 2, 150000, 2000
    g = torch.Generator(device=DEV).manual_seed(21)
    xyz = torch.rand(B, N, 3, device=DEV, generator=g)
    out = torch.full((B, S), -1, dtype=torch.int64, device=DEV)
    need = lib.b200_fps_scratch_bytes(B, N)
    scratch = torch.empty(need, dtype=torch.uint8, device=DEV)                      # allocated before capture
    eager = fps(xyz, S)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            rc = lib.b200_fps_large(xyz.data_ptr(), out.data_ptr(), scratch.data_ptr(), need, B, N, S,
                                    ctypes.c_void_p(side.cuda_stream))
    assert rc == 0
    scratch.fill_(0xAB)                                                               # the replay does not rely on old contents
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
    xyz.copy_(torch.rand(B, N, 3, device=DEV, generator=g))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, fps(xyz, S))
