"""GPU parity tests: the sm_100a kernels, called through the python host layer -> ctypes -> C-ABI
(include/b200flow.h), against (1) the golden fixtures produced by the unmodified reference, (2) the CPU oracle
(oracle/spec.c) on seeded inputs, (3) the reference's own CUDA kernels when oracle/_ref was built, and
(4) size-independent properties at BASELINE.json's full sizes.

Bars (SURVEY §8a): FPS/KNN indices and gathers bit-exact; corr2d |d| <= 1e-6 + 1e-5|ref|; projection gathers
1e-5; event voxels 1e-5*max(1,count); Correlation3D fp32 path 1e-4 relative to the output scale.
"""
import numpy as np
import pytest
import torch

from oracle import refcuda, spec, torch_ref

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import rpeflow_b200 as b200
    from rpeflow_b200 import events as b200_events
    DEV = torch.device("cuda", 0)


def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def nhwc(a):
    return np.ascontiguousarray(np.transpose(a, (0, 2, 3, 1)))


# ------------------------------------------------------------------------------------------------- KNN
@pytest.mark.parametrize("name", ["knn3d", "knn3d_k3_cf", "knn2d"])
def test_knn_golden_inputs_exact_vs_oracle(golden, name):
    g = golden(name)
    k = int(g["k"])
    got = b200.k_nearest_neighbor(cu(g["input"]), cu(g["query"]), k).cpu().numpy()
    inp, qry = g["input"], g["query"]
    if inp.shape[1] <= 3:
        inp, qry = np.transpose(inp, (0, 2, 1)), np.transpose(qry, (0, 2, 1))
    np.testing.assert_array_equal(got, spec.knn(inp, qry, k))
    assert got.dtype == np.int64 and got.shape == g["idx"].shape
    # vs the reference's torch fallback: only near-ties may differ (checked in test_oracle_golden for the oracle)
    assert np.mean(got != g["idx"]) < 0.01


@pytest.mark.parametrize("B,M,Q,D,k", [
    (2, 1000, 513, 3, 16), (1, 37, 5, 3, 32), (3, 5, 9, 3, 8), (2, 2500, 300, 3, 3), (1, 4096, 1000, 2, 16),
    (2, 700, 1500, 2, 1), (1, 3000, 70, 3, 1), (1, 1, 4, 3, 1), (1, 1025, 33, 3, 2), (4, 256, 256, 3, 16),
])
def test_knn_random_exact(B, M, Q, D, k):
    rng = np.random.default_rng(B * 1000 + M + Q + k)
    inp = rng.random((B, M, D), dtype=np.float32)
    qry = rng.random((B, Q, D), dtype=np.float32)
    got = b200.ops._k_nearest_neighbor_cuda(cu(inp), cu(qry), k).cpu().numpy()
    np.testing.assert_array_equal(got, spec.knn(inp, qry, k))


def test_knn_ties_and_duplicates_lowest_index_first():
    rng = np.random.default_rng(5)
    base = rng.random((1, 400, 3), dtype=np.float32)
    inp = np.concatenate([base, base[:, :100], base[:, :50]], axis=1)        # 5 % + exact duplicates
    inp = np.round(inp * 8) / 8                                               # coarse lattice: many exact distance ties
    qry = inp[:, ::3].copy()
    for k in (1, 3, 16, 32):
        got = b200.ops._k_nearest_neighbor_cuda(cu(inp), cu(qry), k).cpu().numpy()
        np.testing.assert_array_equal(got, spec.knn(inp, qry, k))


def test_knn_ids_magnitudes_exact():
    """IDS-like coordinate magnitudes (x in +-15, y in +-9, z in [100,120]) where fp32 rounding bites (SURVEY §7)."""
    rng = np.random.default_rng(6)
    pts = rng.random((2, 4096, 3), dtype=np.float32) * np.float32([30, 18, 20]) + np.float32([-15, -9, 100])
    got = b200.ops._k_nearest_neighbor_cuda(cu(pts), cu(pts[:, :2048]), 16).cpu().numpy()
    np.testing.assert_array_equal(got, spec.knn(pts, pts[:, :2048], 16))


def test_knn_kat_reference_test_main():
    """KAT-knn (k_nearest_neighbor_test.cpp:25-38): manual_seed(0), rand[8,8192,3] x2, k=16."""
    torch.manual_seed(0)
    inp = torch.rand(8, 8192, 3)
    qry = torch.rand(8, 8192, 3)
    got = b200.ops._k_nearest_neighbor_cuda(inp.to(DEV), qry.to(DEV), 16)
    want = spec.knn(inp.numpy(), qry.numpy(), 16)
    np.testing.assert_array_equal(got.cpu().numpy(), want)
    # the reference main only prints the mismatch count against its expanded-formula naive path; bound it here
    naive = torch_ref.k_nearest_neighbor(inp[:2].to(DEV), qry[:2].to(DEV), 16)
    assert (naive != got[:2]).float().mean().item() < 2e-3


def test_knn_full_size_properties():
    """cfg3 scale (B=32, 4096 points, k=16) — properties + a sampled exact check."""
    g = torch.Generator().manual_seed(3)
    pts = torch.rand(32, 4096, 3, generator=g)
    dev = pts.to(DEV)
    idx = b200.ops._k_nearest_neighbor_cuda(dev, dev, 16)
    assert idx.shape == (32, 4096, 16) and idx.dtype == torch.int64
    assert torch.equal(idx[:, :, 0], torch.arange(4096, device=DEV).expand(32, 4096))      # a point is its own nearest
    nb = torch.gather(dev.unsqueeze(1).expand(32, 4096, 4096, 3), 2, idx.unsqueeze(-1).expand(-1, -1, -1, 3))
    d = ((nb - dev.unsqueeze(2)) ** 2).sum(-1)
    assert bool((d[:, :, 1:] >= d[:, :, :-1]).all())                                            # ascending
    sel = [0, 7, 31]
    np.testing.assert_array_equal(idx[sel].cpu().numpy(), spec.knn(pts[sel].numpy(), pts[sel].numpy(), 16))


def _knn_adversarial_cases():
    """Inputs chosen to break a cell-grid search: duplicates, clusters + far outliers, degenerate extents, queries
    far outside the inputs' bounding box, huge offsets (coarse fp32 spacing), tiny extents, M < k, inf/NaN."""
    rng = np.random.default_rng(77)
    cases = {}
    a = rng.random((2, 3000, 3), dtype=np.float32)
    a[:, 1500:] = a[:, :1500]                                        # every point twice
    cases["duplicates"] = (a, a[:, ::3].copy(), 16)
    c = (rng.standard_normal((1, 4000, 3)) * 0.01).astype(np.float32)
    c[0, :5] = np.float32([[50, 50, 50], [-80, 3, 1], [0, 0, 900], [1e4, -1e4, 0], [7, 7, 7]])     # outliers blow up the box
    cases["cluster_outliers"] = (c, c[:, :600].copy(), 16)
    pl = rng.random((1, 2048, 3), dtype=np.float32)
    pl[..., 2] = 3.25                                                # planar cloud: one zero extent
    cases["planar"] = (pl, rng.random((1, 300, 3), dtype=np.float32), 8)
    ln = np.zeros((1, 1500, 3), np.float32)
    ln[..., 0] = rng.random((1, 1500), dtype=np.float32)             # points on a line
    cases["line"] = (ln, ln[:, :200].copy() + np.float32([0, 0.1, 0]), 3)
    cases["all_identical"] = (np.full((1, 500, 3), 2.5, np.float32), rng.random((1, 40, 3), dtype=np.float32), 16)
    far = rng.random((1, 2000, 3), dtype=np.float32)
    cases["queries_outside"] = (far, (rng.random((1, 500, 3), dtype=np.float32) * 40 - 20).astype(np.float32), 16)
    off = (rng.random((1, 3000, 3), dtype=np.float32) + np.float32(4096.0)).astype(np.float32)   # spacing 2^-11: many exact ties
    cases["large_offset_ties"] = (off, off[:, :500].copy(), 16)
    tiny = (rng.random((1, 1000, 3), dtype=np.float32) * np.float32(1e-12)).astype(np.float32)
    cases["tiny_extent"] = (tiny, tiny[:, :100].copy(), 4)
    cases["m_less_than_k"] = (rng.random((2, 7, 3), dtype=np.float32), rng.random((2, 50, 3), dtype=np.float32), 16)
    lat = np.stack(np.meshgrid(np.arange(16), np.arange(16), np.arange(16), indexing="ij"), -1).reshape(1, -1, 3).astype(np.float32)
    cases["integer_lattice_ties"] = (lat, lat[:, ::7].copy(), 32)    # equidistant neighbours everywhere
    px = rng.random((2, 4096, 2), dtype=np.float32) * np.float32([239, 143])
    ys, xs = np.meshgrid(np.arange(144, dtype=np.float32), np.arange(240, dtype=np.float32), indexing="ij")
    grid = np.broadcast_to(np.stack([xs, ys], -1).reshape(1, -1, 2), (2, 144 * 240, 2)).copy()
    cases["pixels_to_points_2d"] = (px, grid, 1)
    half = px.copy()
    half[..., 0] *= 0.25                                             # projected points cover a quarter of the image
    cases["pixels_sparse_cover_2d"] = (half, grid, 1)
    sk = rng.random((1, 5000, 3), dtype=np.float32) * np.float32([30, 17, 90]) + np.float32([-15, -8.5, 22])
    cases["ids_shaped_cross"] = (sk, (sk[:, :2048] + rng.standard_normal((1, 2048, 3)).astype(np.float32) * 0.3).astype(np.float32), 16)
    return cases


@pytest.mark.parametrize("name", sorted(_knn_adversarial_cases()))
def test_knn_grid_adversarial_exact(name):
    inp, qry, k = _knn_adversarial_cases()[name]
    want = spec.knn(inp, qry, k)
    got = b200.ops._k_nearest_neighbor_cuda(cu(inp), cu(qry), k).cpu().numpy()         # cell-grid search
    np.testing.assert_array_equal(got, want)
    brute = b200.ops.knn_bruteforce(cu(inp), cu(qry), k).cpu().numpy()                  # every query scans every input
    np.testing.assert_array_equal(brute, want)


def test_knn_grid_nonfinite_inputs_match_bruteforce():
    rng = np.random.default_rng(3)
    inp = rng.random((1, 600, 3), dtype=np.float32)
    inp[0, 5] = np.float32([np.inf, 0, 0])
    inp[0, 9] = np.float32([np.nan, 1, 1])
    qry = rng.random((1, 64, 3), dtype=np.float32)
    got = b200.ops._k_nearest_neighbor_cuda(cu(inp), cu(qry), 8).cpu().numpy()
    brute = b200.ops.knn_bruteforce(cu(inp), cu(qry), 8).cpu().numpy()
    np.testing.assert_array_equal(got, brute)
    assert not np.isin(got, [5, 9]).any()                            # an inf/NaN distance never enters a list


@pytest.mark.parametrize("B,M,Q,D,k", [(2, 1000, 513, 3, 16), (1, 4096, 1000, 2, 16), (2, 700, 1500, 2, 1), (1, 1025, 33, 3, 2)])
def test_knn_bruteforce_random_exact(B, M, Q, D, k):
    rng = np.random.default_rng(B * 1000 + M + Q + k)
    inp = rng.random((B, M, D), dtype=np.float32)
    qry = rng.random((B, Q, D), dtype=np.float32)
    np.testing.assert_array_equal(b200.ops.knn_bruteforce(cu(inp), cu(qry), k).cpu().numpy(), spec.knn(inp, qry, k))


def test_knn_errors():
    x = torch.rand(1, 10, 3, device=DEV)
    with pytest.raises(RuntimeError):
        b200.ops._k_nearest_neighbor_cuda(x, x, 33)                # reference would overrun its 32 slots
    with pytest.raises(RuntimeError):
        b200.ops._k_nearest_neighbor_cuda(x.cpu(), x.cpu(), 3)     # TORCH_CHECK is_cuda
    with pytest.raises(RuntimeError):
        b200.ops._k_nearest_neighbor_cuda(x.transpose(1, 2), x, 3)  # TORCH_CHECK is_contiguous
    with pytest.raises(RuntimeError):
        b200.ops._k_nearest_neighbor_cuda(x.double(), x.double(), 3)


# ------------------------------------------------------------------------------------------------- FPS
def test_fps_golden(golden):
    g = golden("fps")
    got = b200.furthest_point_sampling(cu(g["xyz"]), int(g["n_samples"]))
    assert got.dtype == torch.int64
    np.testing.assert_array_equal(got.cpu().numpy(), g["idx"])


def test_fps_kat_reference_test_main():
    """KAT-fps (furthest_point_sampling_test.cpp:34-44,63): manual_seed(0), rand[64,4096,3], 1024 samples, exact."""
    torch.manual_seed(0)
    xyz = torch.rand(64, 4096, 3)
    got = b200.ops._furthest_point_sampling_cuda(xyz.to(DEV), 1024).cpu().numpy()
    np.testing.assert_array_equal(got, spec.fps(xyz.numpy(), 1024))


@pytest.mark.parametrize("B,N,S", [(4, 8192, 4096), (2, 777, 300), (3, 1000, 999), (1, 513, 64), (2, 4097, 100),
                                   (2, 10000, 400), (2, 20000, 400), (1, 40000, 300), (1, 32768, 4096), (1, 2, 1)])
def test_fps_sizes_exact(B, N, S):
    rng = np.random.default_rng(N + S)
    xyz = rng.random((B, N, 3), dtype=np.float32)
    if N > 100:
        xyz[:, 50:60] = xyz[:, 0:10]                       # duplicates: sampled-with-replacement clouds
    got = b200.ops._furthest_point_sampling_cuda(cu(xyz), S).cpu().numpy()
    np.testing.assert_array_equal(got, spec.fps(xyz, S))


def _fps_adversarial_clouds():
    rng = np.random.default_rng(5)
    N = 3000
    dup = rng.random((N, 3), dtype=np.float32); dup[1000:2000] = dup[:1000]            # sampled with replacement
    clus = (rng.random((N, 3), dtype=np.float32) * 0.01 + rng.integers(0, 3, (N, 1)).astype(np.float32)); clus[7] = 50.0
    plane = rng.random((N, 3), dtype=np.float32); plane[:, 2] = 0.25
    line = np.zeros((N, 3), np.float32); line[:, 0] = rng.random(N, dtype=np.float32)
    same = np.full((N, 3), 1.5, np.float32)
    lattice = np.stack(np.meshgrid(*[np.arange(15, dtype=np.float32)] * 3, indexing="ij"), -1).reshape(-1, 3)[:N]   # exact ties
    ft3d = rng.random((N, 3), dtype=np.float32) * np.array([30, 17, 90], np.float32) + np.array([-15, -8, 22], np.float32)
    big = (rng.random((N, 3), dtype=np.float32) - 0.5) * 2e4
    return {"dup": dup, "clusters+outlier": clus, "plane": plane, "line": line, "identical": same,
            "lattice": np.ascontiguousarray(lattice), "ft3d": ft3d, "large": big}


def test_fps_pruned_scan_exact():
    """The bounding-box pruned kernel (N <= 8192) returns the full scan's indices on every cloud, as the oracle computes
    them."""
    clouds = _fps_adversarial_clouds()
    xyz = np.stack(list(clouds.values()))
    S = 1500
    want = spec.fps(xyz, S)
    got = b200.ops._furthest_point_sampling_cuda(cu(xyz), S).cpu().numpy()
    for i, name in enumerate(clouds):
        np.testing.assert_array_equal(got[i], want[i], err_msg=name)
    # full-size clouds (config 1): all 4096 picks
    g = torch.Generator().manual_seed(12)
    big = torch.rand(6, 8192, 3, generator=g) * torch.tensor([30.0, 17.0, 90.0])
    got = b200.ops._furthest_point_sampling_cuda(big.to(DEV), 4096).cpu().numpy()
    np.testing.assert_array_equal(got, spec.fps(big.numpy(), 4096))


def test_fps_forced_cluster():
    """The cloud size forces a cluster of 2, 4 or 8 CTAs on clouds of more than 8192 points: both sides of each size
    boundary, a ragged last CTA, and duplicates of the first CTA's points in the last one (ties between CTAs go to the
    lowest index)."""
    for N in (8193, 16384, 16385, 32768, 32769, 50001, 65536):
        rng = np.random.default_rng(N)
        xyz = rng.random((2, N, 3), dtype=np.float32) * np.array([30.0, 17.0, 90.0], dtype=np.float32)
        xyz[:, 50:60] = xyz[:, 0:10]
        xyz[:, -10:] = xyz[:, 0:10]
        want = spec.fps(xyz, 600)
        got = b200.ops._furthest_point_sampling_cuda(cu(xyz), 600).cpu().numpy()
        np.testing.assert_array_equal(got, want, err_msg=f"N={N}")


def test_fps_two_clouds_per_sm_variant():
    """Coordinates in shared memory, two clouds per SM (taken above 4096 points when a call has more clouds than SMs):
    same picks as the oracle, with and without padding slots, and as the register-resident kernel that calls of at
    most one cloud per SM take."""
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    rng = np.random.default_rng(31)
    for n in (8192, 5003):
        xyz = (rng.random((sms + 1, n, 3), dtype=np.float32) * np.array([40.0, 25.0, 80.0], dtype=np.float32)).astype(np.float32)
        xyz[1, 100:400] = xyz[1, 7]                                     # duplicates: index tie-breaks
        want = spec.fps(xyz, 700)
        np.testing.assert_array_equal(b200.ops._furthest_point_sampling_cuda(cu(xyz), 700).cpu().numpy(), want)
    g = torch.Generator().manual_seed(5)
    many = (torch.rand(300, 8192, 3, generator=g) * torch.tensor([30.0, 17.0, 90.0])).to(DEV)
    a = b200.ops._furthest_point_sampling_cuda(many, 4096)
    parts = [b200.ops._furthest_point_sampling_cuda(c, 4096) for c in many.split(sms)]
    assert torch.equal(a, torch.cat(parts))


def test_fps_pyramid_prefix_property():
    """build_pc_pyramid (pwc3d_core.py:8-28): levels are prefixes of one 4096-long list; cfg3 batch."""
    g = torch.Generator().manual_seed(4)
    pc1 = torch.rand(8, 3, 8192, generator=g).to(DEV)
    pc2 = torch.rand(8, 3, 8192, generator=g).to(DEV)
    xyzs1, xyzs2, ids1, ids2 = b200.build_pc_pyramid(pc1, pc2, [4096, 2048, 1024, 512, 256])
    assert [x.shape[-1] for x in xyzs1] == [8192, 4096, 2048, 1024, 512, 256]
    for lvl in range(2, 6):
        assert torch.equal(ids1[lvl], ids1[1][:, :ids1[lvl].shape[1]])
    assert torch.equal(xyzs2[3], torch.gather(pc2, 2, ids2[3].unsqueeze(1).expand(-1, 3, -1)))
    for b in range(8):                                     # sampled indices are distinct for distinct points
        assert ids1[1][b].unique().numel() == 4096


def test_fps_errors():
    x = torch.rand(2, 100, 3, device=DEV)
    with pytest.raises(AssertionError):
        b200.furthest_point_sampling(x, 100)               # wrapper.py:98
    with pytest.raises(RuntimeError):
        b200.ops._furthest_point_sampling_cuda(x, 100)
    with pytest.raises(RuntimeError):
        b200.ops._furthest_point_sampling_cuda(x.cpu(), 10)


# ------------------------------------------------------------------------------------------------- corr2d
CORR_TOL = dict(rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_corr2d_golden(golden, tag):
    g = golden("corr2d_" + tag)
    md = int(g["md"])
    f1 = cu(g["feat1"]).requires_grad_(True)
    f2 = cu(g["feat2"]).requires_grad_(True)
    out = b200.correlation2d(f1, f2, md)
    np.testing.assert_allclose(out.detach().cpu().numpy(), g["out"], **CORR_TOL)
    out.backward(cu(g["grad_out"]))
    np.testing.assert_allclose(f1.grad.cpu().numpy(), g["grad1"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(f2.grad.cpu().numpy(), g["grad2"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("C,H,W", [(32, 144, 240), (64, 72, 120), (96, 36, 60), (128, 18, 30), (192, 9, 15),
                                   (32, 128, 160), (20, 13, 50), (7, 5, 3)])
def test_corr2d_pyramid_levels_vs_oracle(C, H, W):
    """cfg2 level shapes (B reduced to 2 for the CPU oracle) + odd shapes."""
    rng = np.random.default_rng(C + H)
    f1 = rng.standard_normal((2, H, W, C), dtype=np.float32)
    f2 = rng.standard_normal((2, H, W, C), dtype=np.float32)
    got = b200.ops._correlation_forward_cuda(cu(f1), cu(f2), 4).cpu().numpy()
    want = spec.corr2d_fwd(f1, f2, 4)
    np.testing.assert_allclose(got, want, **CORR_TOL)
    assert np.mean(np.abs(got - want)) < 1e-6             # correlation_test.cpp:82-83


@pytest.mark.parametrize("C,H,W", [(32, 144, 240), (64, 72, 120), (96, 36, 60), (128, 18, 28), (36, 11, 44), (8, 9, 12),
                                   (20, 13, 50), (7, 5, 3), (30, 9, 20)])
def test_corr2d_backward_levels_vs_oracle(C, H, W):
    """a2 at the pyramid shapes: the register-tiled kernel (md = 4, C % 4 == 0, W % 4 == 0) and the simple one (the other
    shapes: (20, 13, 50), (7, 5, 3), (30, 9, 20)) against the CPU oracle; ragged tiles and tiles larger than the map
    included."""
    rng = np.random.default_rng(C * H + W)
    f1 = rng.standard_normal((2, H, W, C), dtype=np.float32)
    f2 = rng.standard_normal((2, H, W, C), dtype=np.float32)
    go = rng.standard_normal((2, 81, H, W), dtype=np.float32)
    w1, w2 = spec.corr2d_bwd(go, f1, f2, 4)
    g1, g2 = b200.ops._correlation_backward_cuda(cu(go), cu(f1), cu(f2), 4)
    np.testing.assert_allclose(g1.cpu().numpy(), w1, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(g2.cpu().numpy(), w2, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("B,C,H,W,md", [(2, 19, 11, 14, 5), (1, 40, 20, 16, 7)])
def test_corr2d_large_displacements_vs_oracle(B, C, H, W, md):
    """max_displacement > 4 (the reference kernels take any; ADVICE r1): the plain any-displacement kernels, forward through
    correlation2d() and both gradients through autograd, against the CPU oracle."""
    rng = np.random.default_rng(md * 100 + C)
    f1 = rng.standard_normal((B, C, H, W), dtype=np.float32)
    f2 = rng.standard_normal((B, C, H, W), dtype=np.float32)
    go = rng.standard_normal((B, (2 * md + 1) ** 2, H, W), dtype=np.float32)
    a, b = cu(f1).requires_grad_(True), cu(f2).requires_grad_(True)
    out = b200.correlation2d(a, b, md)
    np.testing.assert_allclose(out.detach().cpu().numpy(), spec.corr2d_fwd(nhwc(f1), nhwc(f2), md), **CORR_TOL)
    out.backward(cu(go))
    g1, g2 = spec.corr2d_bwd(go, nhwc(f1), nhwc(f2), md)
    np.testing.assert_allclose(a.grad.cpu().numpy(), g1, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(b.grad.cpu().numpy(), g2, rtol=1e-5, atol=1e-5)
    with torch.no_grad():
        np.testing.assert_allclose(b200.correlation2d(cu(f1), cu(f2), md).cpu().numpy(), out.detach().cpu().numpy(), rtol=0, atol=0)


@pytest.mark.parametrize("B,C,H,W,md", [(3, 128, 18, 30, 4), (5, 192, 9, 15, 4), (2, 5, 7, 11, 4), (2, 20, 13, 50, 4), (1, 8, 6, 10, 2),
                                        (2, 12, 9, 15, 1), (1, 33, 40, 250, 3), (2, 16, 12, 17, 4)])
def test_corr2d_wrapper_call_on_narrow_maps_vs_oracle(B, C, H, W, md):
    """correlation2d on NCHW maps whose rows TMA cannot address (W % 4 != 0: levels 4 and 5 of every configuration) and
    other displacements (b200_corr2d_fwd_nchw answers B200_ENOSUP, the host mirror permutes and calls b200_corr2d_fwd) against the CPU oracle,
    with and without the fused LeakyReLU, contiguous and 4-byte-offset (unaligned) inputs."""
    rng = np.random.default_rng(B * 1000 + C + H + W)
    f1 = rng.standard_normal((B, C, H, W), dtype=np.float32)
    f2 = rng.standard_normal((B, C, H, W), dtype=np.float32)
    want = spec.corr2d_fwd(nhwc(f1), nhwc(f2), md)
    got = b200.correlation2d(cu(f1), cu(f2), md)
    np.testing.assert_allclose(got.cpu().numpy(), want, **CORR_TOL)
    if md == 4:
        leaky = b200.correlation2d_leaky(cu(f1), cu(f2), md, 0.1)
        np.testing.assert_allclose(leaky.cpu().numpy(), np.where(want > 0, want, 0.1 * want), **CORR_TOL)
    pad1 = torch.zeros(f1.size + 1, device=DEV)
    pad2 = torch.zeros(f2.size + 1, device=DEV)
    u1 = pad1[1:].view(B, C, H, W).copy_(cu(f1))                       # storage offset of 4 bytes
    u2 = pad2[1:].view(B, C, H, W).copy_(cu(f2))
    np.testing.assert_allclose(b200.correlation2d(u1, u2, md).cpu().numpy(), want, **CORR_TOL)


def test_corr2d_kat_reference_test_main():
    """KAT-corr (correlation_test.cpp:44-60,82-89): rand B=32,C=128,144x240, md=4; fwd + both grads, mean|d|<1e-6.
    Inputs drawn on the CPU generator (the reference draws on the device, which is not reproducible)."""
    torch.manual_seed(0)
    B, C, H, W, md = 32, 128, 144, 240, 4
    f1 = torch.rand(B, C, H, W).to(DEV)
    f2 = torch.rand(B, C, H, W).to(DEV)
    go = torch.rand(B, 81, H, W).to(DEV)
    a = f1.permute(0, 2, 3, 1).contiguous()
    b = f2.permute(0, 2, 3, 1).contiguous()
    out = b200.ops._correlation_forward_cuda(a, b, md)
    g1, g2 = b200.ops._correlation_backward_cuda(go, a, b, md)
    for s in range(0, B, 8):                              # naive libtorch path of the reference, in slices (memory)
        x1 = f1[s:s + 8].clone().requires_grad_(True)
        x2 = f2[s:s + 8].clone().requires_grad_(True)
        naive = torch_ref.correlation2d(x1, x2, md)
        naive.backward(go[s:s + 8])
        assert (naive - out[s:s + 8]).abs().mean().item() < 1e-6
        assert (x1.grad - g1[s:s + 8]).abs().mean().item() < 1e-6
        assert (x2.grad - g2[s:s + 8]).abs().mean().item() < 1e-6
        torch.testing.assert_close(out[s:s + 8], naive.detach(), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("op", ["knn", "fps", "corr2d"])
def test_kat_vs_reference_cuda_kernels(op):
    """The inputs of the three KAT tests above through the reference's own CUDA kernels, the kernels this library
    replaces (oracle/_ref/libref_kernels.so, compiled from an upstream RPEFlow checkout by
    `make -C oracle ref REF=<checkout>`): KNN within the near-tie rate, FPS exactly, corr2d forward and both gradients."""
    if not refcuda.available():
        pytest.skip("reference CUDA kernels not built (make -C oracle ref REF=<RPEFlow checkout>)")
    torch.manual_seed(0)
    if op == "knn":
        inp, qry = torch.rand(8, 8192, 3).to(DEV), torch.rand(8, 8192, 3).to(DEV)
        got = b200.ops._k_nearest_neighbor_cuda(inp, qry, 16)
        assert (refcuda.knn(inp, qry, 16) != got).float().mean().item() < 2e-3
    elif op == "fps":
        xyz = torch.rand(64, 4096, 3).to(DEV)
        got = b200.ops._furthest_point_sampling_cuda(xyz, 1024).cpu().numpy()
        np.testing.assert_array_equal(got, refcuda.fps(xyz, 1024).cpu().numpy())   # the reference test demands exact equality
    else:
        B, C, H, W, md = 32, 128, 144, 240, 4
        f1, f2, go = torch.rand(B, C, H, W)[:4], torch.rand(B, C, H, W)[:4], torch.rand(B, 81, H, W)[:4]   # KAT draw order
        a = f1.permute(0, 2, 3, 1).contiguous().to(DEV)
        b = f2.permute(0, 2, 3, 1).contiguous().to(DEV)
        go = go.contiguous().to(DEV)
        torch.testing.assert_close(b200.ops._correlation_forward_cuda(a, b, md), refcuda.corr2d_fwd(a, b, md), rtol=1e-5, atol=1e-6)
        g1, g2 = b200.ops._correlation_backward_cuda(go, a, b, md)
        r1, r2 = refcuda.corr2d_bwd(go, a, b, md)
        torch.testing.assert_close(g1, r1, rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(g2, r2, rtol=1e-5, atol=1e-5)


def test_corr2d_linearity_property():
    g = torch.Generator().manual_seed(8)
    a, b, c = (torch.randn(8, 32, 144, 240, generator=g).to(DEV) for _ in range(3))
    lhs = b200.correlation2d(a, b + 2 * c, 4)
    rhs = b200.correlation2d(a, b, 4) + 2 * b200.correlation2d(a, c, 4)
    torch.testing.assert_close(lhs, rhs, rtol=1e-4, atol=1e-5)
    centre = b200.correlation2d(a, a, 4)[:, 40]           # zero displacement = mean of squares
    torch.testing.assert_close(centre, (a * a).mean(1), rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------------- gathers / projection
def test_gathers_golden_and_random(golden):
    g = golden("gather_cf")
    got = b200.batch_indexing_channel_first(cu(g["data"]), cu(g["idx"]))
    assert torch.equal(got.cpu(), torch.from_numpy(g["out"]))
    g = golden("gather_cl")
    got = b200.batch_indexing_channel_last(cu(g["data"]), cu(g["idx"]))
    assert torch.equal(got.cpu(), torch.from_numpy(g["out"]))
    gen = torch.Generator().manual_seed(11)
    for (B, C, N, shape) in [(4, 64, 2048, (2048, 16)), (2, 3, 8192, (4096,)), (1, 33, 100, (7, 3, 2)), (2, 128, 512, (512, 16))]:
        data = torch.randn(B, C, N, generator=gen).to(DEV)
        idx = torch.randint(0, N, (B,) + shape, generator=gen).to(DEV)
        want = torch_ref.batch_indexing_channel_first(data, idx)
        assert torch.equal(b200.batch_indexing_channel_first(data, idx), want)
        assert torch.equal(b200.batch_indexing_channel_first(data, idx.int()), want)         # any int dtype
        dl = data.transpose(1, 2).contiguous()
        assert torch.equal(b200.batch_indexing_channel_last(dl, idx), torch_ref.batch_indexing_channel_last(dl.cpu(), idx.cpu()).to(DEV))
    neg = torch.tensor([[-1, 0, -5]], device=DEV)
    data = torch.arange(10., device=DEV).view(1, 1, 10)
    assert b200.batch_indexing_channel_first(data, neg).flatten().tolist() == [9.0, 0.0, 5.0]
    ints = torch.arange(40, dtype=torch.int32, device=DEV).view(2, 2, 10)                     # int32 payloads move bit-exactly
    assert torch.equal(b200.batch_indexing_channel_first(ints, torch.tensor([[3], [4]], device=DEV)),
                       torch.tensor([[[3], [13]], [[24], [34]]], dtype=torch.int32, device=DEV))


def test_grid_sample_golden_and_levels(golden):
    g = golden("grid_sample")
    got = b200.grid_sample_wrapper(cu(g["feat"]), cu(g["xy"])).cpu().numpy()
    np.testing.assert_allclose(got, g["out"], rtol=1e-5, atol=1e-5)
    gen = torch.Generator().manual_seed(12)
    for (B, C, H, W, N) in [(2, 32, 144, 240, 4096), (2, 83, 72, 120, 2048), (1, 192, 9, 15, 256), (1, 5, 2, 2, 9)]:
        feat = torch.randn(B, C, H, W, generator=gen)
        xy = torch.rand(B, 2, N, generator=gen) * torch.tensor([W + 4.0, H + 4.0]).view(1, 2, 1) - 2.0
        want = spec.grid_sample_pts(feat.numpy(), xy.numpy())
        got = b200.grid_sample_wrapper(feat.to(DEV), xy.to(DEV))
        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-5, atol=1e-5)
        # ATen's CUDA path: the same torch ops on the GPU divide by the python scalar (W-1) as x * (1/(W-1)), so the
        # pixel coordinate differs from the CPU reference (true division, = our rule) by 1-2 ulp(|x|) ~ 3e-5 px;
        # times the feature gradient that is ~1e-4 absolute.  Looser bar, cross-check only.
        lib_ref = torch_ref.grid_sample_wrapper(feat.to(DEV), xy.to(DEV))
        torch.testing.assert_close(got, lib_ref, rtol=1e-4, atol=5e-4)


def test_project_nn_corr_golden_and_levels(golden):
    g = golden("project_nn_corr")
    got = b200.project_feat_with_nn_corr(cu(g["xy"]), cu(g["feat2d"]), cu(g["feat3d"]), cu(g["nn"]))
    np.testing.assert_allclose(got.cpu().numpy(), g["out"], rtol=1e-5, atol=1e-5)
    gen = torch.Generator().manual_seed(13)
    for (B, C2, C3, H, W, N) in [(2, 32, 32, 144, 240, 4096), (1, 81, 34, 72, 120, 2048), (1, 96, 64, 18, 30, 512), (1, 6, 5, 3, 4, 7)]:
        f2 = torch.randn(B, C2, H, W, generator=gen).to(DEV)
        f3 = torch.randn(B, C3, N, generator=gen).to(DEV)
        xy = (torch.rand(B, 2, N, generator=gen) * torch.tensor([W + 2.0, H + 2.0]).view(1, 2, 1) - 1.0).to(DEV)
        auto = b200.project_feat_with_nn_corr(xy, f2, f3)                                      # nn computed by our KNN (k=1, 2-D)
        grid = torch_ref.pixel_grid(B, H, W).to(DEV)
        nn = b200.k_nearest_neighbor(xy, grid.contiguous(), 1)[..., 0]
        got = b200.project_feat_with_nn_corr(xy, f2, f3, nn)
        assert torch.equal(auto, got)
        want = spec.project_nn_corr(xy.cpu().numpy(), f2.cpu().numpy(), f3.cpu().numpy(), nn.cpu().numpy())
        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-5, atol=1e-5)
        assert torch.equal(got[:, 3:].reshape(B, C3, -1), torch_ref.batch_indexing_channel_first(f3, nn))   # feat3d part is a pure gather


@pytest.mark.parametrize("case", ["dense", "sparse", "crowded", "outside", "random_nn", "odd_channels", "small_map"])
def test_project_nn_corr_tiled_route_equals_two_pass_and_oracle(case, monkeypatch):
    """The single-pass tiled route (project_tile.cu) on inputs that stress its window logic: sparse clouds (nearest point
    outside the 4-pixel halo -> per-tap global reads), every point in one tile (more points than threads), points far
    outside the image / non-finite coordinates, arbitrary nn indices, channel counts that are no multiple of the 8-channel
    stage, maps smaller than a tile.  Bars: 1e-5 vs the oracle (SURVEY §8a); output AND sampled tensor bit-identical to
    the two-pass kernels (same operation order)."""
    from rpeflow_b200 import projection
    gen = torch.Generator().manual_seed(500 + len(case))
    B, C2, C3, H, W, N = {"dense": (3, 32, 32, 144, 240, 4096), "sparse": (2, 16, 8, 72, 120, 40), "crowded": (2, 24, 12, 48, 128, 1500),
                          "outside": (2, 16, 16, 36, 60, 600), "random_nn": (2, 16, 20, 40, 64, 300),
                          "odd_channels": (2, 81, 34, 72, 120, 2048), "small_map": (3, 13, 7, 5, 8, 30)}[case]
    f2 = torch.randn(B, C2, H, W, generator=gen).to(DEV)
    f3 = torch.randn(B, C3, N, generator=gen).to(DEV)
    xy = torch.rand(B, 2, N, generator=gen) * torch.tensor([W - 1.0, H - 1.0]).view(1, 2, 1)
    if case == "crowded":
        xy = xy * torch.tensor([30.0 / W, 10.0 / H]).view(1, 2, 1) + torch.tensor([70.0, 18.0]).view(1, 2, 1)   # all inside one tile
    if case == "outside":
        xy = xy * 3.0 - torch.tensor([W * 1.0, H * 1.0]).view(1, 2, 1)
        xy[0, 0, :5] = torch.tensor([float("nan"), float("inf"), -float("inf"), 1e30, -1e30])
        xy[1, 1, 7] = float("nan")
    xy = xy.to(DEV)
    grid = torch_ref.pixel_grid(B, H, W).to(DEV)
    if case == "random_nn":
        nn = torch.randint(0, N, (B, H * W), generator=gen).to(DEV)
    elif case == "outside":
        finite = torch.nan_to_num(xy, nan=1e6, posinf=1e6, neginf=-1e6).clamp(-1e6, 1e6)
        nn = b200.k_nearest_neighbor(finite, grid.contiguous(), 1)[..., 0]
    else:
        nn = b200.k_nearest_neighbor(xy, grid.contiguous(), 1)[..., 0]
    res = {}
    for route in ("two_pass", "tiled"):
        monkeypatch.setenv("B200_PROJECT_ROUTE", route)
        projection.SAMPLE_MEMO.clear()
        out = b200.project_feat_with_nn_corr(xy, f2, f3, nn)
        res[route] = (out, projection.SAMPLE_MEMO.take(f2, xy))
        bare = b200.project_feat_with_nn_corr(xy, f2, f3, nn, keep_samples=False)
        assert torch.equal(bare.view(torch.int32), out.view(torch.int32))
    monkeypatch.delenv("B200_PROJECT_ROUTE")
    projection.SAMPLE_MEMO.clear()
    for a, b in zip(res["two_pass"], res["tiled"]):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))                # bit patterns: NaN-safe comparison
    plain = b200.grid_sample_wrapper(f2, xy)
    assert torch.equal(plain.view(torch.int32), res["tiled"][1].view(torch.int32))
    if case != "outside":                                                            # the C oracle is not asked about NaN coordinates
        want = spec.project_nn_corr(xy.cpu().numpy(), f2.cpu().numpy(), f3.cpu().numpy(), nn.cpu().numpy())
        np.testing.assert_allclose(res["tiled"][0].cpu().numpy(), want, rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(res["tiled"][1].cpu().numpy(), spec.grid_sample_pts(f2.cpu().numpy(), xy.cpu().numpy()), rtol=1e-5, atol=1e-5)


def test_projection_sampler_serves_the_following_grid_sample_bit_exactly():
    """project_feat_with_nn_corr(xy, f, ...) parks bilinear(f, xy); grid_sample_wrapper(f, xy) issued right after must return
    exactly what the stand-alone sampling kernel returns, exactly once, and never after an in-place write to f or xy."""
    from rpeflow_b200 import projection
    gen = torch.Generator().manual_seed(21)
    for (B, C2, C3, H, W, N) in [(2, 32, 32, 144, 240, 4096), (1, 81, 34, 72, 120, 2048), (2, 96, 64, 36, 60, 1024), (1, 7, 5, 9, 15, 31)]:
        f2 = torch.randn(B, C2, H, W, generator=gen).to(DEV)
        f3 = torch.randn(B, C3, N, generator=gen).to(DEV)
        xy = (torch.rand(B, 2, N, generator=gen) * torch.tensor([W + 2.0, H + 2.0]).view(1, 2, 1) - 1.0).to(DEV)
        projection.SAMPLE_MEMO.clear()
        plain = b200.grid_sample_wrapper(f2, xy)                       # memo empty: the stand-alone kernel
        h0 = projection.SAMPLE_MEMO.hits
        b200.project_feat_with_nn_corr(xy, f2, f3)
        served = b200.grid_sample_wrapper(f2, xy)
        assert projection.SAMPLE_MEMO.hits == h0 + 1
        assert torch.equal(served, plain)
        again = b200.grid_sample_wrapper(f2, xy)                       # handed out once only
        assert projection.SAMPLE_MEMO.hits == h0 + 1 and torch.equal(again, plain) and again.data_ptr() != served.data_ptr()
        b200.project_feat_with_nn_corr(xy, f2, f3)
        f2[:, 0].mul_(2.0)                                             # in-place write invalidates the parked samples
        fresh = b200.grid_sample_wrapper(f2, xy)
        assert projection.SAMPLE_MEMO.hits == h0 + 1
        np.testing.assert_allclose(fresh.cpu().numpy(), spec.grid_sample_pts(f2.cpu().numpy(), xy.cpu().numpy()), rtol=1e-5, atol=1e-5)
        b200.project_feat_with_nn_corr(xy, f2, f3)
        other = xy.clone()
        assert torch.equal(b200.grid_sample_wrapper(f2, other), fresh) and projection.SAMPLE_MEMO.hits == h0 + 1   # other tensor: no hit
    projection.SAMPLE_MEMO.clear()


# ------------------------------------------------------------------------------------------------- Correlation3D
def _corr3d_inputs(B, C, N, k, seed):
    gen = torch.Generator().manual_seed(seed)
    xyz1 = torch.rand(B, 3, N, generator=gen)
    xyz2 = xyz1 + 0.05 * torch.randn(B, 3, N, generator=gen)
    f1 = torch.randn(B, C, N, generator=gen)
    f2 = torch.randn(B, C, N, generator=gen)
    torch.manual_seed(seed)
    mod = b200.Correlation3D(C, C, k=k).eval()
    return xyz1, f1, xyz2, f2, mod


@pytest.mark.parametrize("tag", ["a", "b"])
def test_corr3d_golden(golden, tag):
    g = golden("corr3d_" + tag)
    w = {n[2:]: cu(g[n]) for n in g if n.startswith("w_")}
    got = b200.correlation3d_forward(cu(g["xyz1"]), cu(g["feat1"]), cu(g["xyz2"]), cu(g["feat2"]), w,
                                     cu(g["knn12"]), cu(g["knn11"]))
    scale = np.abs(g["out"]).max()
    np.testing.assert_allclose(got.cpu().numpy(), g["out"], rtol=1e-4, atol=1e-4 * scale)


@pytest.mark.parametrize("C,N", [(32, 4096), (64, 2048), (96, 1024), (128, 512), (192, 256), (20, 100)])
def test_corr3d_levels_vs_oracle_and_module(C, N):
    xyz1, f1, xyz2, f2, mod = _corr3d_inputs(2, C, N, 16, C)
    mod = mod.to(DEV)
    with torch.no_grad():
        got = mod(xyz1.to(DEV), f1.to(DEV), xyz2.to(DEV), f2.to(DEV))
    knn11 = b200.k_nearest_neighbor(xyz1.to(DEV), xyz1.to(DEV), 16).cpu()
    knn12 = b200.k_nearest_neighbor(xyz2.to(DEV), xyz1.to(DEV), 16).cpu()
    w = {n: v.cpu() for n, v in b200.pwc3d.pack_weights(mod).items()}
    want = spec.corr3d_fwd(xyz1.numpy(), f1.numpy(), xyz2.numpy(), f2.numpy(), knn12.numpy(), knn11.numpy(),
                           {n: v.numpy() for n, v in w.items()})
    scale = np.abs(want).max()
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-4, atol=1e-4 * scale)
    lib_ref = torch_ref.correlation3d(xyz1, f1, xyz2, f2, w, k=16, knn11=knn11, knn12=knn12).numpy()     # torch fp32 CPU
    np.testing.assert_allclose(got.cpu().numpy(), lib_ref, rtol=1e-4, atol=1e-4 * scale)


@pytest.mark.parametrize("precision,tol", [(2, 1e-4), (1, 5e-3)])
@pytest.mark.parametrize("C,N", [(32, 4096), (64, 2048), (96, 1024), (128, 512), (192, 256), (32, 37)])
def test_corr3d_tensor_core_paths_vs_oracle(C, N, precision, tol):
    """tcgen05 path of the Cout x Cout layer: precision 2 (3xTF32) meets the fp32 bar (1e-4 of the output scale),
    precision 1 (TF32 operands, what cuDNN does for the reference under torch's default allow_tf32) 5e-3."""
    xyz1, f1, xyz2, f2, mod = _corr3d_inputs(2, C, N, 16, C)
    knn11 = b200.k_nearest_neighbor(xyz1.to(DEV), xyz1.to(DEV), 16)
    knn12 = b200.k_nearest_neighbor(xyz2.to(DEV), xyz1.to(DEV), 16)
    w = b200.pwc3d.pack_weights(mod)
    wd = {n: v.to(DEV) for n, v in w.items()}
    got = b200.pwc3d.correlation3d_forward(xyz1.to(DEV), f1.to(DEV), xyz2.to(DEV), f2.to(DEV), wd, knn12, knn11, precision)
    want = spec.corr3d_fwd(xyz1.numpy(), f1.numpy(), xyz2.numpy(), f2.numpy(), knn12.cpu().numpy(), knn11.cpu().numpy(),
                           {n: v.numpy() for n, v in w.items()})
    scale = np.abs(want).max()
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=tol, atol=tol * scale)
    fp32 = b200.pwc3d.correlation3d_forward(xyz1.to(DEV), f1.to(DEV), xyz2.to(DEV), f2.to(DEV), wd, knn12, knn11, 0)
    np.testing.assert_allclose(got.cpu().numpy(), fp32.cpu().numpy(), rtol=tol, atol=tol * scale)


def test_corr3d_is_forward_only_and_keeps_state_dict_keys():
    _, f1, _, _, mod = _corr3d_inputs(1, 8, 32, 4, 1)
    keys = set(mod.state_dict().keys())
    assert "cost_mlp.convs.0.conv_fn.weight" in keys and "weight_net2.convs.2.conv_fn.bias" in keys and len(keys) == 16
    mod = mod.to(DEV)
    x = torch.rand(1, 3, 32, device=DEV)
    with pytest.raises(RuntimeError):
        mod(x, f1.to(DEV), x, f1.to(DEV))                  # grad enabled + parameters require grad


# ------------------------------------------------------------------------------------------------- events
@pytest.mark.parametrize("name,pol", [("event_voxel_pol", True), ("event_voxel_nopol", False)])
def test_event_voxel_golden(golden, name, pol):
    g = golden(name)
    got = b200.eventsToVoxel(g["events"], num_bins=int(g["bins"]), height=int(g["H"]), width=int(g["W"]), event_polarity=pol)
    assert got.dtype == np.float32 and got.shape == g["vox"].shape
    cnt = np.maximum(1.0, np.abs(g["vox"]))
    assert np.all(np.abs(got - g["vox"]) <= 1e-5 * cnt)


def test_event_voxel_cfg1_size():
    """cfg1: 1 M events on 540x960, 10 bins x 2 polarities."""
    rng = np.random.default_rng(21)
    n, H, W = 1_000_000, 540, 960
    ev = np.zeros((n, 4), np.float32)
    ev[:, 0] = rng.integers(0, W, n)
    ev[:, 1] = rng.integers(0, H, n)
    ev[:, 2] = np.sort(rng.random(n, dtype=np.float32))
    ev[:, 3] = rng.choice(np.float32([-1, 1]), n)
    got = b200.eventsToVoxel(ev, num_bins=10, height=H, width=W, event_polarity=True)
    want, bad = spec.event_voxel_int(ev, 10, H, W, True)
    assert bad == 0
    assert np.all(np.abs(got - want) <= 1e-5 * np.maximum(1.0, want))
    assert abs(float(got.sum(dtype=np.float64)) - n) < 1e-3 * n ** 0.5 + 1.0          # sum(voxel) == n (SURVEY a9)
    assert abs(float(got[:10].sum(dtype=np.float64)) - float((ev[:, 3] > 0).sum())) < 2.0
    auto = b200.eventsToVoxel(ev, num_bins=10, event_polarity=True)                      # height/width inferred
    assert auto.shape == (20, int(ev[:, 1].max()) + 1, int(ev[:, 0].max()) + 1)


def test_event_voxel_out_of_range_raises():
    ev = np.float32([[0, 0, 0.0, 1], [50, 2, 0.5, 1], [1, 1, 1.0, -1]])
    with pytest.raises(IndexError):
        b200.eventsToVoxel(ev, num_bins=5, height=10, width=10, event_polarity=True)
    ev[1, 0] = -1                                         # torch negative-index wrap: column W-1
    got = b200.eventsToVoxel(ev, num_bins=5, height=10, width=10, event_polarity=True)
    want, bad = spec.event_voxel_int(ev, 5, 10, 10, True)
    assert bad == 0 and np.allclose(got, want, atol=1e-6) and got[:, 2, 9].sum() > 0


@pytest.mark.parametrize("name,pol", [("event_trilinear_pol", True), ("event_trilinear_nopol", False)])
def test_event_trilinear_golden(golden, name, pol):
    g = golden(name)
    ev = {k: g[k] for k in ("x", "y", "t", "p")}
    got = b200.eventsToVoxelInter(ev, int(g["bins"]), int(g["H"]), int(g["W"]), event_polarity=pol)
    assert np.all(np.abs(got - g["vox"]) <= 1e-5 * np.maximum(1.0, np.abs(g["vox"])))


def test_event_trilinear_cfg4_size():
    rng = np.random.default_rng(22)
    n, H, W = 1_500_000, 480, 640
    ev = {"x": (rng.random(n) * (W - 1)).astype(np.float32), "y": (rng.random(n) * (H - 1)).astype(np.float32),
          "t": np.sort(rng.integers(0, 100_000, n)).astype(np.int64), "p": rng.integers(0, 2, n).astype(np.uint8)}
    got = b200.eventsToVoxelInter(ev, 10, H, W, event_polarity=True)
    want = spec.event_voxel_trilinear(ev["x"], ev["y"], ev["t"], ev["p"], 10, H, W, True)
    assert np.all(np.abs(got - want) <= 1e-5 * np.maximum(1.0, np.abs(want)))
    # interior events splat total weight 1 each: the grid sums to (almost) n
    assert abs(float(got.sum(dtype=np.float64)) - n) < 0.02 * n


# ------------------------------------------------------------------------------------------------- knn_interpolation (§8f rank 2)
def test_knn_interpolation_golden_and_levels(golden):
    g = golden("knn_interpolation")
    got = b200.knn_interpolation(cu(g["input_xyz"]), cu(g["input_feat"]), cu(g["query_xyz"]), 3)
    np.testing.assert_allclose(got.cpu().numpy(), g["out"], rtol=1e-6, atol=1e-6)          # the reference's own output
    warp = b200.backwarp_3d(cu(g["input_xyz"]), cu(g["xyz2"]), cu(g["flow12"]), 3)
    np.testing.assert_allclose(warp.cpu().numpy(), g["backwarp"], rtol=1e-6, atol=1e-6)
    gen = torch.Generator().manual_seed(4)
    for (B, C, M, Q, k) in [(2, 64, 2048, 4096, 3), (1, 3, 256, 512, 3), (2, 5, 40, 33, 8), (1, 192, 256, 512, 1)]:
        xin = torch.rand(B, 3, M, generator=gen) * 10
        feat = torch.randn(B, C, M, generator=gen)
        xq = torch.rand(B, 3, Q, generator=gen) * 10
        xq[:, :, :3] = xin[:, :, :3]                                                          # coincident points: clamp(1e-8)
        idx = b200.k_nearest_neighbor(xin.to(DEV), xq.to(DEV), k)
        got = b200.knn_interpolation(xin.to(DEV), feat.to(DEV), xq.to(DEV), k, knn_indices=idx)
        want = spec.knn_interpolate(xin.numpy(), feat.numpy(), xq.numpy(), idx.cpu().numpy())
        np.testing.assert_array_equal(got.cpu().numpy(), want)                                # every op rounded as the oracle does
        ref = torch_ref.knn_interpolation(xin, feat, xq, k, knn_indices=idx.cpu())
        np.testing.assert_allclose(got.cpu().numpy(), ref.numpy(), rtol=1e-5, atol=1e-5)
    with pytest.raises(RuntimeError):
        b200.knn_interpolation(xin, feat, xq, 3)                                              # CPU tensors: no fallback


# ------------------------------------------------------------------------------------------------- backwarp_2d + corr2d + leaky (§8f rank 3)
def test_warp2d_golden(golden):
    g = golden("warp2d")
    warped = b200.backwarp_2d(cu(g["f2"]), cu(g["flow"]), "border")
    np.testing.assert_allclose(warped.cpu().numpy(), g["warped"], rtol=1e-5, atol=1e-5)       # the reference's own output
    cost = b200.warp_correlate(cu(g["f1"]), cu(g["f2"]), cu(g["flow"]), 4, 0.1)
    np.testing.assert_allclose(cost.cpu().numpy(), g["cost"], rtol=1e-5, atol=1e-5)
    with pytest.raises(RuntimeError):
        b200.backwarp_2d(cu(g["f2"]), cu(g["flow"]), "zeros")                                  # only the mode RPEFlow uses
    with pytest.raises(RuntimeError):
        b200.backwarp_2d(torch.from_numpy(g["f2"]), torch.from_numpy(g["flow"]))               # CPU tensors: no fallback


@pytest.mark.parametrize("B,C,H,W", [(3, 32, 144, 240), (2, 64, 72, 120), (2, 96, 36, 60), (1, 5, 9, 16), (2, 33, 18, 28),
                                     (1, 1, 1, 4), (1, 3, 2, 8), (1, 8, 70, 52), (1, 12, 5, 100)])
def test_warp_correlate_vs_oracle(B, C, H, W):
    """Level shapes of config 1 (both corr2d tilings) and ragged ones; flows large enough to leave the image."""
    gen = torch.Generator().manual_seed(H * W + C)
    f1 = torch.randn(B, C, H, W, generator=gen)
    f2 = torch.randn(B, C, H, W, generator=gen)
    flow = 4.0 * torch.randn(B, 2, H, W, generator=gen)
    warped = b200.backwarp_2d(f2.to(DEV), flow.to(DEV))
    want_w = spec.backwarp2d_border(f2.numpy(), flow.numpy())
    np.testing.assert_allclose(warped.cpu().numpy(), want_w, rtol=1e-5, atol=1e-5)
    ref_w = torch_ref.backwarp_2d(f2, flow, "border")
    np.testing.assert_allclose(warped.cpu().numpy(), ref_w.numpy(), rtol=1e-5, atol=1e-5)
    # the fused activation is exactly leaky_relu of the unfused cost volume, on both tilings and on the NHWC fallback
    plain = b200.correlation2d(f1.to(DEV), warped, 4)
    leaky = b200.correlation2d_leaky(f1.to(DEV), warped, 4, 0.1)
    assert torch.equal(leaky, torch.nn.functional.leaky_relu(plain, 0.1))
    assert torch.equal(b200.correlation2d_leaky(f1.to(DEV), warped, 4, 1.0), plain)
    # whole expression vs the oracle, chunked (warped map kept L2-sized) and unchunked
    want = spec.corr2d_fwd(nhwc(f1.numpy()), nhwc(want_w), 4)
    want = np.where(want > 0, want, np.float32(0.1) * want)
    for budget in (48 << 20, 1):
        got = b200.warp_correlate(f1.to(DEV), f2.to(DEV), flow.to(DEV), 4, 0.1, l2_budget_bytes=budget)
        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-5, atol=2e-6)
    none = b200.warp_correlate(f1.to(DEV), f2.to(DEV), None, 4, 0.1)                           # coarsest level: no warp
    assert torch.equal(none, b200.correlation2d_leaky(f1.to(DEV), f2.to(DEV), 4, 0.1))


# ------------------------------------------------------------------------------------------------- convex_upsample (§8f rank 4)
@pytest.mark.parametrize("s", [4, 8])
def test_convex_upsample_golden(golden, s):
    g = golden("convex_upsample_s%d" % s)
    got = b200.convex_upsample(cu(g["flow"]), cu(g["mask"]), s)
    np.testing.assert_allclose(got.cpu().numpy(), g["out"], rtol=1e-5, atol=1e-5)             # the reference's own output


@pytest.mark.parametrize("B,H,W,s", [(2, 144, 240, 4), (1, 120, 160, 4), (2, 17, 23, 8), (3, 10, 7, 2)])
def test_convex_upsample_vs_oracle(B, H, W, s):
    gen = torch.Generator().manual_seed(H + W + s)
    flow = 4.0 * torch.randn(B, 2, H, W, generator=gen)
    mask = 2.0 * torch.randn(B, 9 * s * s, H, W, generator=gen)
    got = b200.convex_upsample(flow.to(DEV), mask.to(DEV), s).cpu().numpy()
    np.testing.assert_allclose(got, spec.convex_upsample(flow.numpy(), mask.numpy(), s), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(got, torch_ref.convex_upsample(flow, mask, s).numpy(), rtol=1e-5, atol=1e-5)
    # a one-hot mask copies the chosen neighbour (times s): exact property, size independent
    hot = torch.full((B, 9, s * s, H, W), -1e4)
    hot[:, 4] = 1e4                                                                          # centre tap
    got = b200.convex_upsample(flow.to(DEV), hot.reshape(B, 9 * s * s, H, W).to(DEV), s)
    want = (flow * s).repeat_interleave(s, dim=2).repeat_interleave(s, dim=3)
    assert torch.equal(got.cpu(), want)
    with pytest.raises(RuntimeError):
        b200.convex_upsample(flow, mask, s)                                                  # CPU tensors: no fallback


# ------------------------------------------------------------------------------------------------- empty inputs
def test_empty_batches_and_queries():
    """Batch 0 / zero queries: every entry point returns a correctly shaped empty result (torch semantics; the reference's
    unchecked zero-size launches end the same way)."""
    z = lambda *shape: torch.zeros(shape, device=DEV)
    assert b200.correlation2d(z(0, 8, 12, 16), z(0, 8, 12, 16), 4).shape == (0, 81, 12, 16)
    assert b200.ops._correlation_forward_cuda(z(0, 12, 16, 8), z(0, 12, 16, 8), 4).shape == (0, 81, 12, 16)
    g1, g2 = b200.ops._correlation_backward_cuda(z(0, 81, 12, 16), z(0, 12, 16, 8), z(0, 12, 16, 8), 4)
    assert g1.shape == (0, 8, 12, 16) and g2.shape == (0, 8, 12, 16)
    assert b200.ops._furthest_point_sampling_cuda(z(0, 100, 3), 10).shape == (0, 10)
    assert b200.ops._k_nearest_neighbor_cuda(z(0, 50, 3), z(0, 20, 3), 4).shape == (0, 20, 4)
    assert b200.ops._k_nearest_neighbor_cuda(torch.rand(2, 50, 3, device=DEV), z(2, 0, 3), 4).shape == (2, 0, 4)
    assert b200.grid_sample_wrapper(z(0, 4, 6, 8), z(0, 2, 5)).shape == (0, 4, 5)
    assert b200.grid_sample_wrapper(torch.rand(2, 4, 6, 8, device=DEV), z(2, 2, 0)).shape == (2, 4, 0)
    assert b200.backwarp_2d(z(0, 4, 6, 8), z(0, 2, 6, 8)).shape == (0, 4, 6, 8)
    assert b200.convex_upsample(z(0, 2, 3, 4), z(0, 144, 3, 4), 4).shape == (0, 2, 12, 16)
    assert b200.batch_indexing_channel_first(z(0, 4, 9), torch.zeros(0, 5, dtype=torch.int64, device=DEV)).shape == (0, 4, 5)
    with pytest.raises((RuntimeError, IndexError)):                 # the reference indexes events[-1]: no events is an error there too
        b200_events.events_to_voxel_device(z(0, 4), 5, 6, 8, True)


# ------------------------------------------------------------------------------------------------- wrapper-level behaviour
def test_wrapper_level_views_and_dtypes():
    """The python mirrors accept what the reference wrappers accept: non-contiguous views, float64 feature maps
    (wrapper.py:68-69 casts to float), channel-first or channel-last clouds (wrapper.py:108-115), any int index dtype."""
    g = torch.Generator().manual_seed(21)
    f1 = torch.randn(2, 16, 24, 32, generator=g).to(DEV)
    f2 = torch.randn(2, 16, 24, 32, generator=g).to(DEV)
    base = b200.correlation2d(f1, f2, 4)
    nhwc1, nhwc2 = f1.permute(0, 2, 3, 1).contiguous(), f2.permute(0, 2, 3, 1).contiguous()
    assert torch.equal(b200.correlation2d(nhwc1.permute(0, 3, 1, 2), nhwc2.permute(0, 3, 1, 2), 4), base)   # permuted views
    torch.testing.assert_close(b200.correlation2d(f1.double(), f2.double(), 4), base, rtol=1e-6, atol=1e-6)
    assert b200.correlation2d(f1.double(), f2.double(), 4).dtype == torch.float32
    pts = torch.rand(2, 500, 3, generator=g).to(DEV)
    qry = torch.rand(2, 70, 3, generator=g).to(DEV)
    cl = b200.k_nearest_neighbor(pts, qry, 8)
    cf = b200.k_nearest_neighbor(pts.transpose(1, 2), qry.transpose(1, 2), 8)                  # [B,3,M]: auto-transposed
    assert torch.equal(cl, cf)
    assert torch.equal(b200.k_nearest_neighbor(pts.transpose(1, 2).contiguous(), qry.transpose(1, 2).contiguous(), 8), cl)
    data = torch.randn(2, 5, 500, generator=g).to(DEV)
    want = b200.batch_indexing_channel_first(data, cl)
    assert torch.equal(b200.batch_indexing_channel_first(data, cl.to(torch.int32)), want)
    ref = torch.gather(data.unsqueeze(2).expand(-1, -1, 70, -1), 3, cl.unsqueeze(1).expand(-1, 5, -1, -1))   # [B,C,Q,k]
    assert torch.equal(want, ref)
    xy = (torch.rand(2, 70, 2, generator=g) * torch.tensor([31.0, 23.0])).to(DEV)
    a = b200.grid_sample_wrapper(f1, xy.transpose(1, 2))                                       # non-contiguous [B,2,N] view
    assert torch.equal(a, b200.grid_sample_wrapper(f1, xy.transpose(1, 2).contiguous()))
    flow = torch.randn(2, 24, 32, 2, generator=g).to(DEV)
    assert torch.equal(b200.backwarp_2d(f2, flow.permute(0, 3, 1, 2)), b200.backwarp_2d(f2, flow.permute(0, 3, 1, 2).contiguous()))


# ------------------------------------------------------------------------------------------------- PointConv (§8f rank 1)
@pytest.mark.parametrize("precision,tol", [(2, 1e-4), (1, 5e-3)])
@pytest.mark.parametrize("tag", ["down", "nosample"])
def test_pointconv_golden(golden, tag, precision, tol):
    g = golden("pointconv_" + tag)
    w = {n[2:]: cu(g[n]) for n in g if n.startswith("w_")}
    got = b200.pointconv_forward(cu(g["xyz"]), cu(g["feat"]), cu(g["sampled"]), cu(g["knn"]), w, precision)
    scale = np.abs(g["out"]).max()
    np.testing.assert_allclose(got.cpu().numpy(), g["out"], rtol=tol, atol=tol * scale)      # the reference's own output


@pytest.mark.parametrize("C,cout,N,S", [(32, 32, 8192, 4096), (64, 64, 4096, 2048), (192, 192, 512, 256), (35, 64, 300, 300),
                                         (0, 16, 100, 37), (32, 64, 70000, 512)])     # N > 65536: uint32 indices
def test_pointconv_modules_vs_oracle(C, cout, N, S):
    gen = torch.Generator().manual_seed(C + N)
    B = 2
    xyz = torch.rand(B, 3, N, generator=gen) * 5
    feat = torch.randn(B, C, N, generator=gen)
    torch.manual_seed(7)
    if S == N:
        mod = b200.PointConvNoSampling(C, cout).to(DEV).eval()
        with torch.no_grad():
            got = mod(xyz.to(DEV), feat.to(DEV))
        sampled = xyz
    else:
        mod = b200.PointConvDownSampling(C, cout).to(DEV).eval()
        sampled = xyz[:, :, :S].contiguous()
        with torch.no_grad():
            got = mod(xyz.to(DEV), feat.to(DEV), sampled.to(DEV))
    knn = b200.k_nearest_neighbor(xyz.to(DEV), sampled.to(DEV), 16).cpu()
    w = {n: v.cpu() for n, v in b200.pointconv.pack_pointconv_weights(mod).items()}
    want = spec.pointconv_fwd(xyz.numpy(), feat.numpy(), sampled.numpy(), knn.numpy(), {n: v.numpy() for n, v in w.items()})
    scale = np.abs(want).max()
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-4, atol=1e-4 * scale)
    assert set(mod.state_dict()) == {"weight_net.convs.0.conv_fn.weight", "weight_net.convs.0.conv_fn.bias",
                                     "weight_net.convs.1.conv_fn.weight", "weight_net.convs.1.conv_fn.bias",
                                     "linear.weight", "linear.bias"}
    with pytest.raises(RuntimeError):
        mod(xyz.to(DEV), feat.to(DEV).requires_grad_(True), *([] if S == N else [sampled.to(DEV)]))
