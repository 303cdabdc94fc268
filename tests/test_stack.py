"""The cost-volume stack runner: input grouping / stage order on CPU, and on the GPU that the CUDA-graph replay
(single fused graph and per-input-group graphs fed by the HostFeeder) reproduces the eager kernel-by-kernel run."""
import pytest
import torch

from rpeflow_b200.stack import (CONFIGS, INPUT_GROUPS, CostVolumeStack, GraphedStack, HostFeeder, group_tensors,
                                make_host_inputs, tensors_nbytes, to_device)


def test_input_groups_cover_every_tensor_once():
    host = make_host_inputs(CONFIGS["tiny"], 2)
    groups = group_tensors(host)
    assert list(groups) == INPUT_GROUPS
    ids = [id(t) for g in groups.values() for t in g]
    assert len(ids) == len(set(ids))
    assert sum(t.numel() * t.element_size() for g in groups.values() for t in g) == tensors_nbytes(host)
    # dependency order of the copies: point data first, the largest activations (level 1) last
    assert INPUT_GROUPS[0] == "points" and INPUT_GROUPS[-1] == "lvl1"
    assert sum(t.numel() for t in groups["lvl1"]) > sum(t.numel() for t in groups["lvl2"])


def test_segments_follow_the_copy_order():
    stack = CostVolumeStack.__new__(CostVolumeStack)         # no device needed to list the segments
    assert [g for g, _ in CostVolumeStack.segments(stack)] == INPUT_GROUPS


def _same(a, b):
    if isinstance(a, torch.Tensor):
        return torch.equal(a, b)
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(_same(a[k], b[k]) for k in a)
    return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))


@pytest.mark.gpu
def test_graph_replay_and_feeder_match_eager_run():
    dev = torch.device("cuda", 0)
    cfg = CONFIGS["tiny"]
    host = make_host_inputs(cfg, 2, pin=True)
    stack = CostVolumeStack(cfg, dev)
    x = to_device(host, dev)
    stack.concurrent = False
    want, _ = stack.run(x)                                   # kernel by kernel, one stream
    want = {k: v for k, v in want.items() if k != "event_voxel"}      # atomics: order-dependent last ulp
    from test_event_voxel_reference import check_cells, ref_int
    refs = [ref_int(host["events"][i].numpy(), cfg.event_bins, cfg.height, cfg.width, True) for i in range(2)]

    def voxels_match(out):                                   # instead, every sample cell by cell against the reference
        for i, R in enumerate(refs):
            check_cells(out["event_voxel"][i].cpu().numpy(), R, "stack tiny graph", f"sample {i}")
    stack.concurrent = True
    ints_w, flts_w = stack.checksum(stack.run(x)[0])

    fused = GraphedStack(stack, x, fused=True)
    for _ in range(2):
        out = fused.replay()
    torch.cuda.synchronize()
    assert _same({k: v for k, v in out.items() if k != "event_voxel"}, want)
    voxels_match(out)
    assert torch.equal(fused.checksum[0], ints_w)
    torch.testing.assert_close(fused.checksum[1], flts_w, rtol=1e-6, atol=1e-3)

    feeder = HostFeeder(host, dev, depth=2)                  # per-group graphs, inputs streamed from pinned memory
    runners = [GraphedStack(stack, slot, fused=False) for slot in feeder.slots]
    main = torch.cuda.current_stream()
    for step in range(3):
        slot = step % 2
        evs = feeder.issue(slot)
        out = runners[slot].replay(wait=lambda g, evs=evs: main.wait_event(evs[g]))
        main.synchronize()
        assert _same({k: v for k, v in out.items() if k != "event_voxel"}, want)
        voxels_match(out)
        assert torch.equal(runners[slot].checksum[0], ints_w)

    # external inputs only (point clouds + raw events) streamed per step, the feature maps shared from the resident set
    del runners, feeder
    ext = HostFeeder(host, dev, depth=2, resident=x)
    assert 0 < ext.nbytes < sum(t.numel() * t.element_size() for ts in __import__("rpeflow_b200.stack", fromlist=["x"]).group_tensors(host).values() for t in ts)
    assert all(sl["pcs"].data_ptr() != x["pcs"].data_ptr() and sl["feat2d"] is x["feat2d"] for sl in ext.slots)
    runners = [GraphedStack(stack, slot, fused=False) for slot in ext.slots]
    for step in range(3):
        slot = step % 2
        ext.slots[slot]["pcs"].fill_(float("nan"))           # poison the per-slot buffer: the copy must refill it
        main.synchronize()
        evs = ext.issue(slot)
        out = runners[slot].replay(wait=lambda g, evs=evs: main.wait_event(evs[g]))
        main.synchronize()
        assert _same({k: v for k, v in out.items() if k != "event_voxel"}, want)
        voxels_match(out)
        assert torch.equal(runners[slot].checksum[0], ints_w)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dsec", "hd", "hd_scaled"])
def test_other_baseline_configs_run_and_index_ops_stay_exact(name):
    """BASELINE.json configs[3] (DSEC-shaped: 640x480, tri-linear voxels) and configs[4] (1920x1080, 32768 points: FPS
    over a 4-CTA cluster, KNN over 32768 inputs): one frame pair through the whole stack; FPS and a sample of the KNN
    results are compared with the CPU oracle, float outputs must be finite and the voxel grid is held cell by cell to the
    float64 reference of test_event_voxel_reference.py."""
    import numpy as np
    from oracle import spec
    dev = torch.device("cuda", 0)
    cfg = CONFIGS[name]
    host = make_host_inputs(cfg, 1)
    stack = CostVolumeStack(cfg, dev)
    out, _ = stack.run(to_device(host, dev))
    torch.cuda.synchronize()
    pcs = host["pcs"]
    both = torch.cat([pcs[:, :3], pcs[:, 3:]], 0).transpose(1, 2).contiguous().numpy()
    np.testing.assert_array_equal(out["fps_idx"].cpu().numpy(), spec.fps(both, max(cfg.pyramid)))
    idx1 = out["fps_idx"][0].cpu()
    for lvl in (1, 4):
        n = cfg.pyramid[lvl - 1]
        xyz = pcs[0, :3][:, idx1[:n]].t().contiguous().numpy()[None]
        want = spec.knn(xyz, xyz[:, :64], 16)
        np.testing.assert_array_equal(out["knn_self"][lvl][:, :64].cpu().numpy(), want)
    for lvl in range(1, 6):
        for t in [out["corr2d"][lvl], out["corr3d"][lvl]] + out["proj"][lvl] + out["sample"][lvl]:
            assert bool(torch.isfinite(t).all())
    from test_event_voxel_reference import check_cells, ref_int, ref_trilinear
    if name == "dsec":
        R = ref_trilinear(host["ev_x"][0].numpy(), host["ev_y"][0].numpy(), host["ev_t"][0].numpy(), host["ev_p"][0].numpy(),
                          cfg.event_bins, cfg.height, cfg.width, True)
    else:
        R = ref_int(host["events"][0].numpy(), cfg.event_bins, cfg.height, cfg.width, True)
    check_cells(out["event_voxel"][0].cpu().numpy(), R, "stack " + name, name)


@pytest.mark.gpu
def test_bench_batch_graph_replay_matches_the_oracle_on_first_and_last_sample():
    """The shapes bench.py times: one CUDA-graph replay of the whole census over the bench batch (148 frame pairs: persistent
    corr2d CTAs walking thousands of tiles, 296-cloud FPS with two clouds per SM, multi-tile Correlation3D CTAs).  The first
    and the last sample of every output are compared with the CPU oracle: indices exactly, floats at the SURVEY §8a
    tolerances."""
    import numpy as np
    from oracle import spec
    from rpeflow_b200 import pwc3d
    dev = torch.device("cuda", 0)
    cfg = CONFIGS["things"]
    from rpeflow_b200.workload import BENCH_BATCH
    B = BENCH_BATCH
    host = make_host_inputs(cfg, B)
    stack = CostVolumeStack(cfg, dev)
    x = to_device(host, dev)
    g = GraphedStack(stack, x, fused=True, with_checksum=False)
    out = g.replay()
    torch.cuda.synchronize()
    hs, ws = cfg.sensor
    both = torch.cat([host["pcs"][:, :3], host["pcs"][:, 3:]], 0).transpose(1, 2).contiguous().numpy()
    for i in (0, B - 1):
        sel = [i, B + i]
        fps = out["fps_idx"][sel].cpu().numpy()
        np.testing.assert_array_equal(fps, spec.fps(both[sel], max(cfg.pyramid)))
        pc1, pc2 = host["pcs"][i, :3].numpy(), host["pcs"][i, 3:].numpy()
        ev = host["events"][i].numpy()
        want_vox, bad = spec.event_voxel_int(ev, cfg.event_bins, cfg.height, cfg.width, True)
        vox = out["event_voxel"][i].cpu().numpy()
        assert bad == 0 and np.all(np.abs(vox - want_vox) <= 1e-5 * np.maximum(1.0, want_vox))
        for lvl in range(1, 6):
            n = cfg.pyramid[lvl - 1]
            h, w = cfg.level_hw(lvl)
            xyz1 = np.ascontiguousarray(pc1[:, fps[0, :n]])[None]                    # [1,3,n]
            xyz2 = np.ascontiguousarray(pc2[:, fps[1, :n]])[None]
            x1n, x2n = np.ascontiguousarray(xyz1.transpose(0, 2, 1)), np.ascontiguousarray(xyz2.transpose(0, 2, 1))
            knn11 = spec.knn(x1n, x1n, cfg.k)
            np.testing.assert_array_equal(out["knn_self"][lvl][i:i + 1].cpu().numpy(), knn11)
            knn12 = spec.knn(x2n, x1n, cfg.k)
            f1_3d, f2_3d = host["feat3d"][lvl][0][i:i + 1].numpy(), host["feat3d"][lvl][1][i:i + 1].numpy()
            wts = {k: v.cpu().numpy() for k, v in stack.corr3d[lvl].items()}
            want = spec.corr3d_fwd(xyz1, f1_3d, xyz2, f2_3d, knn12, knn11, wts)
            got = out["corr3d"][lvl][i:i + 1].cpu().numpy()
            np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * np.abs(want).max())
            f1_2d, f2_2d = host["feat2d"][lvl][0][i:i + 1], host["feat2d"][lvl][1][i:i + 1]
            want = spec.corr2d_fwd(f1_2d.permute(0, 2, 3, 1).contiguous().numpy(), f2_2d.permute(0, 2, 3, 1).contiguous().numpy(), 4)
            cost2d = out["corr2d"][lvl][i:i + 1].cpu().numpy()
            np.testing.assert_allclose(cost2d, want, rtol=1e-5, atol=1e-6)
            # projections / samplers of this level: xy as the stack derives them, nn from the oracle's 2-D search
            xy1_t = torch.from_numpy(pc1[:, fps[0, :n]])[None]
            px = (xy1_t[:, 0:1] + (ws - 1) / 2) * ((w - 1) / (ws - 1))                # the stack's own torch arithmetic
            py = (xy1_t[:, 1:2] + (hs - 1) / 2) * ((h - 1) / (hs - 1))
            xy1 = torch.cat([px, py], 1).numpy()
            ys, xs = np.meshgrid(np.arange(h, dtype=np.float32), np.arange(w, dtype=np.float32), indexing="ij")
            grid = np.stack([xs, ys], -1).reshape(1, h * w, 2)
            nn1 = spec.knn(np.ascontiguousarray(xy1.transpose(0, 2, 1)), grid, 1)[..., 0]
            p = out["proj"][lvl]
            want = spec.project_nn_corr(xy1, f1_2d.numpy(), f1_3d, nn1)
            np.testing.assert_allclose(p[0][i:i + 1].cpu().numpy(), want, rtol=1e-5, atol=1e-5)
            dec_2d, dec_3d = host["flowfeat"][lvl][0][i:i + 1].numpy(), host["flowfeat"][lvl][1][i:i + 1].numpy()
            want = spec.project_nn_corr(xy1, dec_2d, dec_3d, nn1)
            np.testing.assert_allclose(p[3][i:i + 1].cpu().numpy(), want, rtol=1e-5, atol=1e-5)
            s = out["sample"][lvl]
            np.testing.assert_allclose(s[0][i:i + 1].cpu().numpy(), spec.grid_sample_pts(f1_2d.numpy(), xy1), rtol=1e-5, atol=1e-5)
            np.testing.assert_allclose(s[4][i:i + 1].cpu().numpy(), spec.grid_sample_pts(dec_2d, xy1), rtol=1e-5, atol=1e-5)
            np.testing.assert_allclose(s[2][i:i + 1, :81].cpu().numpy(), spec.grid_sample_pts(cost2d, xy1), rtol=1e-5, atol=1e-5)
            np.testing.assert_allclose(s[3][i:i + 1].cpu().numpy(), spec.grid_sample_pts(host["efeat2d"][lvl][i:i + 1].numpy(), xy1),
                                       rtol=1e-5, atol=1e-5)
