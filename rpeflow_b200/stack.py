"""The cost-volume stack: one replay of the hot-op census of a RPEFlow forward pass for a batch of frame pairs.

This is the workload behind BASELINE.json's metric (frame-pairs/s through corr2d + KNN/FPS + 3-D cost volume +
projection gathers + event voxels).  The census follows the reference call by call (SURVEY §3.1; file:line in
danqu130/RPEFlow):

  event voxel grid                      1x  event_utils.py:109 (things/kubric) or dsec.py:570 (dsec)
  build_pc_pyramid                      1x FPS on cat[pc1,pc2] -> 4096, 10 xyz gathers      pwc3d_core.py:8-28
  FeaturePyramid3D (2 clouds)          10x KNN k=16 (8192->4096 ... 512->256)               pointconv.py:46
  decode, level 5..1 (RPEFlow_core.py:307-395)
      2x KNN 2-D k=1 (pixel grid -> projected points)   :329-330        1x KNN self k=16      :331
      2x project_feat_with_nn_corr (C_l, C_l)           :334-335        2x grid_sample (C_l)  :336-337
      [l<5] 2x KNN k=3 (knn_interpolation, backwarp_3d) :354-358
      Correlation3D (KNN cross k=16 inside)             :361            correlation2d md=4    :362
      project_feat_with_nn_corr (81, C_l+2)             :373            2x grid_sample (83, C_l event)  :376
      project_feat_with_nn_corr (96, 64)                :394            grid_sample (96)      :395
  final upsampling                      5x KNN k=3 (N_{l+1} -> N_l)                          :429-430

= 1 voxelisation, 1 FPS, 43 KNN, 5 corr2d, 5 Correlation3D, 20 project_feat_with_nn_corr (whose internal
grid_sample is fused) + 25 stand-alone grid_sample_wrapper (the 83-channel one is issued as 81 + 2 channels).  Everything between those calls (convolutions,
attention, flow heads) is out of scope, so the feature maps the ops consume are synthetic activations.
"""
import os

import torch

from . import events as _events
from . import ops, projection, pwc3d
from .workload import (CONFIGS, LEVEL_CHANNELS, PYRAMID_POINTS, StackConfig, _map_tensors, census_work,  # noqa: F401
                       make_host_inputs, tensors_nbytes, to_device)


class _OpTimer:
    """CUDA-event brackets per op group, recorded on the launching (current) stream."""

    def __init__(self, enabled):
        self.enabled = enabled
        self.spans = {}

    def __call__(self, name, fn, *args, **kwargs):
        if not self.enabled:
            return fn(*args, **kwargs)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn(*args, **kwargs)
        b.record()
        self.spans.setdefault(name, []).append((a, b))
        return out

    def totals_ms(self):
        """name -> (total ms, number of brackets); call after a synchronize."""
        return {k: (sum(a.elapsed_time(b) for a, b in v), len(v)) for k, v in self.spans.items()}


class CostVolumeStack:
    def __init__(self, cfg, device, seed=0):
        self.cfg = cfg
        self.device = torch.device(device)
        torch.manual_seed(seed)                       # "random-init weights" (BASELINE.json configs[0])
        self.corr3d = {}
        for lvl, c in zip(range(1, 6), LEVEL_CHANNELS):
            mod = pwc3d.Correlation3D(c, c, k=cfg.k)
            self.corr3d[lvl] = {n: v.to(self.device) for n, v in pwc3d.pack_weights(mod).items()}
        self._grids = {}
        self.concurrent = True        # independent op groups on side streams (parallel branches under graph capture)
        self.max_streams = 3          # batch 148: 1 / 2 / 3 / 6 / 10 = 27.23 / 26.76 / 26.12 / 26.82 / 27.11 ms per step
        # streams the per-sample voxelisations are dealt onto: 2 pays for the RED-issue-bound tri-linear voxeliser (dsec step
        # 28.66 -> 27.83 ms at batch 148), not for the integer one (things: 26.77 -> 27.04 ms with 2, 27.7 with 3)
        self.voxel_lanes = 2 if cfg.name == "dsec" else 1

    def pixel_grid(self, batch, h, w):
        key = (batch, h, w)
        if key not in self._grids:                    # mesh_grid cache of the reference (models/utils.py:172-183)
            ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float32, device=self.device),
                                    torch.arange(w, dtype=torch.float32, device=self.device), indexing="ij")
            self._grids[key] = torch.stack([xs, ys], 0).reshape(1, 2, h * w).expand(batch, 2, h * w).contiguous()
        return self._grids[key]                       # [B,2,HW] channel-first, as RPEFlow_core.py:326-327 passes it

    def voxelise(self, x, lanes=1):
        """One voxel grid per sample (the reference voxelises sample by sample in the dataset's __getitem__).  lanes > 1 deals
        the samples round-robin onto that many side streams (parallel branches under graph capture): the zero fill of one
        sample's grid (HBM-write bound) then overlaps the RED scatter of another's (atomic-throughput bound), while each
        grid still stays L2-resident between its own fill and scatter."""
        cfg = self.cfg
        nb = x["ev_x"].shape[0] if cfg.name == "dsec" else x["events"].shape[0]
        grids = torch.empty((nb, 2 * cfg.event_bins, cfg.height, cfg.width), dtype=torch.float32, device=self.device)

        def one(i):
            if cfg.name == "dsec":
                _events.events_to_voxel_trilinear_device(x["ev_x"][i], x["ev_y"][i], x["ev_t"][i], x["ev_p"][i],
                                                         cfg.event_bins, cfg.height, cfg.width, True, out=grids[i])
            else:
                _events.events_to_voxel_device(x["events"][i], cfg.event_bins, cfg.height, cfg.width, True,
                                               check_range=False, out=grids[i])
        lanes = max(1, min(int(lanes), nb))
        if lanes == 1:
            for i in range(nb):
                one(i)
            return grids
        main = torch.cuda.current_stream(self.device)
        pool = self.__dict__.setdefault("_voxel_streams", [])
        while len(pool) < lanes:
            pool.append(torch.cuda.Stream(device=self.device))
        for st in pool[:lanes]:
            st.wait_stream(main)
        for j, st in enumerate(pool[:lanes]):
            with torch.cuda.stream(st):
                for i in range(j, nb, lanes):
                    one(i)
        for st in pool[:lanes]:
            main.wait_stream(st)
        return grids

    # ---- the census, split into stages by the input group each one needs -------------------------------------
    #   "points" : point clouds + per-point features  -> FPS, pyramid gathers, all 43 KNN searches, 5 Correlation3D
    #   "events" : raw events                         -> voxel grid
    #   "lvl<l>" : the 2-D activations of level l      -> correlation2d, projections, samplers of that level
    # Ops inside a stage keep the reference's call order; stages only depend on "points" (and on their own group),
    # so a feeder can stream the big 2-D activations in while the point work is already running.
    def _parallel(self, T, sections):
        """Run independent groups of ops.  Serially when timing per op (or when concurrency is off); otherwise each
        group on its own side stream, forked from and joined back to the current stream — inside a CUDA-graph
        capture these become parallel branches, which is what keeps the SMs busy through the many small launches
        (32-CTA grid builds, coarse pyramid levels)."""
        if not self.concurrent or T.enabled or len(sections) < 2:
            for fn in sections:
                fn()
            return
        main = torch.cuda.current_stream(self.device)
        streams = self._streams(min(len(sections), self.max_streams))
        for st in streams:
            st.wait_stream(main)
        for i, fn in enumerate(sections):
            with torch.cuda.stream(streams[i % len(streams)]):
                fn()
        for st in streams:
            main.wait_stream(st)

    def _streams(self, n):
        pool = self.__dict__.setdefault("_stream_pool", [])
        while len(pool) < n:
            pool.append(torch.cuda.Stream(device=self.device))
        return pool[:n]

    def _stage_points(self, x, S, T):
        cfg = self.cfg
        B = x["pcs"].shape[0]
        hs, ws = cfg.sensor
        pc1, pc2 = x["pcs"][:, :3].contiguous(), x["pcs"][:, 3:].contiguous()
        both = torch.cat([pc1, pc2], dim=0).transpose(1, 2).contiguous()                    # pwc3d_core.py:12-13
        picked = T("fps", ops.furthest_point_sampling, both, max(cfg.pyramid))
        S["out"]["fps_idx"] = picked
        idx1, idx2 = picked[:B], picked[B:]
        xyzs1, xyzs2 = [pc1], [pc2]
        for n in cfg.pyramid:
            xyzs1.append(T("gather_xyz", projection.batch_indexing_channel_first, pc1, idx1[:, :n]))
            xyzs2.append(T("gather_xyz", projection.batch_indexing_channel_first, pc2, idx2[:, :n]))
        S["xyzs1"], S["xyzs2"] = xyzs1, xyzs2

        def pyramid(xyzs):                                                                   # FeaturePyramid3D, pointconv.py:46
            for lvl in range(5):
                T("knn_pyramid_k16", ops.k_nearest_neighbor, xyzs[lvl], xyzs[lvl + 1], cfg.k)

        def pixels(lvl):                                                                     # RPEFlow_core.py:316-330
            h, w = cfg.level_hw(lvl)

            def to_pixels(xyz):
                px = (xyz[:, 0:1] + (ws - 1) / 2) * ((w - 1) / (ws - 1))
                py = (xyz[:, 1:2] + (hs - 1) / 2) * ((h - 1) / (hs - 1))
                return torch.cat([px, py], dim=1)
            xy1, xy2 = to_pixels(xyzs1[lvl]), to_pixels(xyzs2[lvl])
            grid = self.pixel_grid(B, h, w)
            nn1 = T("knn_2d_k1", ops.k_nearest_neighbor, xy1, grid, 1)                                   # :329
            nn2 = T("knn_2d_k1", ops.k_nearest_neighbor, xy2, grid, 1)                                   # :330
            S[lvl] = {"xy1": xy1, "xy2": xy2, "nn1": nn1[..., 0], "nn2": nn2[..., 0]}

        def cost3d(lvl):
            xyz1, xyz2 = xyzs1[lvl], xyzs2[lvl]
            f1_3d, f2_3d = x["feat3d"][lvl][0], x["feat3d"][lvl][1]
            knn11 = T("knn_self_k16", ops.k_nearest_neighbor, xyz1, xyz1, cfg.k)                         # :331
            S["out"]["knn_self"][lvl] = knn11
            knn12 = T("knn_cross_k16", ops.k_nearest_neighbor, xyz2, xyz1, cfg.k)                        # pwc3d_core.py:81
            S["out"]["corr3d"][lvl] = T("corr3d", pwc3d.correlation3d_forward, xyz1, f1_3d, xyz2, f2_3d, self.corr3d[lvl],
                                        knn12, knn11, cfg.precision)                                     # :361

        def interp(lvl):
            if lvl < 5:                                                                       # :354-358 (k=3 searches only)
                T("knn_interp_k3", ops.k_nearest_neighbor, xyzs1[lvl + 1], xyzs1[lvl], 3)
                T("knn_interp_k3", ops.k_nearest_neighbor, xyzs1[lvl], xyzs2[lvl], 3)
            T("knn_interp_k3", ops.k_nearest_neighbor, xyzs1[lvl], xyzs1[lvl - 1], 3)         # final upsampling, :429-430

        sections = [lambda: pyramid(xyzs1), lambda: pyramid(xyzs2)]
        for lvl in range(5, 0, -1):
            sections += [lambda lvl=lvl: pixels(lvl), lambda lvl=lvl: cost3d(lvl), lambda lvl=lvl: interp(lvl)]
        self._parallel(T, sections)

    def _stage_events(self, x, S, T):
        lanes = self.voxel_lanes if (self.concurrent and not T.enabled) else 1
        S["out"]["event_voxel"] = T("event_voxel", self.voxelise, x, lanes)

    def _stage_corr2d(self, x, S, T, lvl):
        f1_2d, f2_2d = x["feat2d"][lvl]
        S["out"]["corr2d"][lvl] = T("corr2d_L%d" % lvl, ops.correlation2d, f1_2d, f2_2d, self.cfg.max_displacement)   # :362

    def _stage_level(self, x, S, T, lvl):
        L = S[lvl]
        xy1, xy2, nn1, nn2 = L["xy1"], L["xy2"], L["nn1"], L["nn2"]
        xyz1 = S["xyzs1"][lvl]
        f1_2d, f2_2d = x["feat2d"][lvl]
        f1_3d, f2_3d = x["feat3d"][lvl]
        ef_2d = x["efeat2d"][lvl]
        dec_2d, dec_3d = x["flowfeat"][lvl]
        cost2d, cost3d = S["out"]["corr2d"][lvl], S["out"]["corr3d"][lvl]
        p, s = [None] * 4, [None] * 5
        PR, GS = projection.project_feat_with_nn_corr, projection.grid_sample_wrapper

        def a():
            p[0] = T("project_nn_corr_L%d" % lvl, PR, xy1, f1_2d, f1_3d, nn1)                                        # :334
            s[0] = T("grid_sample_L%d" % lvl, GS, f1_2d, xy1)                                                        # :336
            s[3] = T("grid_sample_L%d" % lvl, GS, ef_2d, xy1)                                                        # :108

        def b():
            p[1] = T("project_nn_corr_L%d" % lvl, PR, xy2, f2_2d, f2_3d, nn2)                                        # :335
            s[1] = T("grid_sample_L%d" % lvl, GS, f2_2d, xy2)                                                        # :337

        def c():
            flow3d_to_2d = xyz1[:, :2]                                                        # stand-in for the 2 flow channels
            p[2] = T("project_nn_corr_L%d" % lvl, PR, xy1, cost2d, torch.cat([cost3d, flow3d_to_2d], dim=1), nn1)    # :373 / :80
            # :376 / :107 samples cat[cost volume, 2 flow channels] (83 ch); sampling is per channel, so the two parts are
            # sampled separately and only the small [B,83,N] result is concatenated (the 83-channel map is never built)
            s[2] = torch.cat([T("grid_sample_L%d" % lvl, GS, cost2d, xy1),
                              T("grid_sample_L%d" % lvl, GS, f1_2d[:, :2].contiguous(), xy1)], dim=1)

        def d():
            p[3] = T("project_nn_corr_L%d" % lvl, PR, xy1, dec_2d, dec_3d, nn1)                                      # :394
            s[4] = T("grid_sample_L%d" % lvl, GS, dec_2d, xy1)                                                       # :395
        # Large maps take the tiled projection route (csrc/project_tile.cu): a persistent kernel that owns every SM, so
        # side streams only interleave its prep / post launches with another call's tile kernel (measured: level 1
        # 2.62 ms on four streams, 2.35 ms in sequence); the small levels need the concurrency to fill the GPU.
        h, w = f1_2d.shape[-2:]
        if h * w >= 4096 and os.environ.get("B200_PROJECT_ROUTE") != "two_pass":
            a(); b(); c(); d()
        else:
            self._parallel(T, [a, b, c, d])
        S["out"]["proj"][lvl], S["out"]["sample"][lvl] = p, s

    @staticmethod
    def _new_state():
        return {"out": {"corr2d": {}, "corr3d": {}, "proj": {}, "sample": {}, "knn_self": {}}}

    def segments(self):
        """[(input group, fn(x, S, T))] in execution order."""
        segs = [("points", self._stage_points), ("events", self._stage_events)]
        for lvl in range(5, 0, -1):
            def level(x, S, T, lvl=lvl):
                self._stage_corr2d(x, S, T, lvl)
                self._stage_level(x, S, T, lvl)
            segs.append(("lvl%d" % lvl, level))
        return segs

    @torch.no_grad()
    def run(self, x, timed=False, wait=None, overlap=False):
        """x: device inputs (to_device(make_host_inputs(...))).  Returns (outputs dict, _OpTimer).

        wait(group): called before the first op that reads input group `group` (a feeder makes the current stream
        wait for that group's host->device copy there).  overlap=True runs the ops that need no point data (voxel
        grid, the five correlation2d) on a second stream next to the FPS/KNN chain, which is a 64-CTA latency chain
        and leaves most SMs idle."""
        T = _OpTimer(timed)
        S = self._new_state()
        wait = wait or (lambda group: None)
        if overlap and not timed:
            main = torch.cuda.current_stream(self.device)
            side = self._side_stream()
            side.wait_stream(main)
            with torch.cuda.stream(side):
                wait("events")
                self._stage_events(x, S, T)
                for lvl in range(5, 0, -1):
                    wait("lvl%d" % lvl)
                    self._stage_corr2d(x, S, T, lvl)
            wait("points")
            self._stage_points(x, S, T)
            main.wait_stream(side)
            for lvl in range(5, 0, -1):
                self._stage_level(x, S, T, lvl)
        else:
            for group, fn in self.segments():
                wait(group)
                fn(x, S, T)
        return S["out"], T

    def _side_stream(self):
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(device=self.device)
        return self._side

    @staticmethod
    def checksum(out):
        """Small device vector summarising every output: exact int64 sums for index results, fp64 sums for floats."""
        ints = [out["fps_idx"].sum()] + [out["knn_self"][l].sum() for l in sorted(out["knn_self"])]
        flts = [out["event_voxel"].double().sum()]
        for l in sorted(out["corr2d"]):
            flts += [out["corr2d"][l].double().sum(), out["corr3d"][l].double().sum()]
            flts += [t.double().sum() for t in out["proj"][l]] + [t.double().sum() for t in out["sample"][l]]
        return torch.stack(ints).to(torch.float64), torch.stack(flts)


INPUT_GROUPS = ["points", "events", "lvl5", "lvl4", "lvl3", "lvl2", "lvl1"]      # host->device copy order of a feeder


def group_tensors(x):
    """{group: [tensors]} for an input tree (host or device), in the order a feeder copies them."""
    g = {name: [] for name in INPUT_GROUPS}
    g["points"].append(x["pcs"])
    for lvl in range(5, 0, -1):
        g["points"] += [x["feat3d"][lvl][0], x["feat3d"][lvl][1], x["flowfeat"][lvl][1]]
        g["lvl%d" % lvl] += [x["feat2d"][lvl][0], x["feat2d"][lvl][1], x["efeat2d"][lvl], x["flowfeat"][lvl][0]]
    g["events"] += [x[k] for k in ("events", "ev_x", "ev_y", "ev_t", "ev_p") if k in x]
    return g


class HostFeeder:
    """Streams one step's inputs from pinned host memory into one of `depth` preallocated device input sets on a
    copy stream, group by group in dependency order (small point data first, the level-1 activations last), and
    records one event per group so the compute stream only waits for what the next stage reads."""

    EXTERNAL = ("pcs", "events", "ev_x", "ev_y", "ev_t", "ev_p")      # what reaches the path from outside the model

    def __init__(self, host, device, depth=2, resident=None):
        """`resident`: a device input tree; when given, only the EXTERNAL inputs (point clouds, raw events) get per-slot device
        buffers and per-step copies, everything else (the feature maps the model computes on the device) is shared from it."""
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(device=self.device)
        if resident is None:
            self.slots = [_map_tensors(host, lambda t: torch.empty(t.shape, dtype=t.dtype, device=self.device))
                          for _ in range(depth)]
        else:
            self.slots = [{k: (v.clone() if k in self.EXTERNAL else v) for k, v in resident.items()} for _ in range(depth)]
        src = group_tensors(host)
        self.plan = []
        for slot in self.slots:
            dst = group_tensors(slot)
            own = None if resident is None else {slot[k].data_ptr() for k in self.EXTERNAL if k in slot}
            self.plan.append([(name, [(d, s_) for d, s_ in zip(dst[name], src[name]) if own is None or d.data_ptr() in own])
                              for name in INPUT_GROUPS])
        self.nbytes = sum(s_.numel() * s_.element_size() for _, pairs in self.plan[0] for _, s_ in pairs)

    def issue(self, slot, after=None):
        """Enqueue the copies into device set `slot` (after event `after`, e.g. the last compute that read that
        set).  Returns {group: event}."""
        events = {}
        with torch.cuda.stream(self.stream):
            if after is not None:
                self.stream.wait_event(after)
            for name, pairs in self.plan[slot]:
                for dst, src in pairs:
                    dst.copy_(src, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.stream)
                events[name] = ev
        return events


class GraphedStack:
    """CUDA-graph capture of CostVolumeStack over a fixed device input set: the ~900 launches of a step become one
    graph replay (fused=True: a single graph with the two-stream overlap of CostVolumeStack.run) or one replay per
    input group (fused=False: a feeder's copy events are waited on between replays).  Outputs are static tensors
    owned by the graphs' memory pool."""

    def __init__(self, stack, x, fused=True, with_checksum=True):
        self.stack, self.x, self.fused = stack, x, fused
        self.graphs = []
        self.out = None
        self.checksum = None
        warm = torch.cuda.Stream(device=stack.device)
        warm.wait_stream(torch.cuda.current_stream(stack.device))
        with torch.cuda.stream(warm):                 # eager warm-up: allocator, pixel-grid cache, function attributes
            stack.run(x, overlap=fused)
        torch.cuda.current_stream(stack.device).wait_stream(warm)
        torch.cuda.synchronize(stack.device)
        pool = torch.cuda.graph_pool_handle()
        T = _OpTimer(False)
        with torch.no_grad():
            if fused:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool):
                    self.out, _ = stack.run(x, overlap=True)
                    if with_checksum:
                        self.checksum = stack.checksum(self.out)
                self.graphs.append((None, g))
            else:
                S = stack._new_state()
                segs = stack.segments()
                for n, (group, fn) in enumerate(segs):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, pool=pool):
                        fn(x, S, T)
                        if with_checksum and n == len(segs) - 1:
                            self.checksum = stack.checksum(S["out"])
                    self.graphs.append((group, g))
                self._state = S                       # keeps every intermediate tensor of the pool alive
                self.out = S["out"]

    def replay(self, wait=None):
        for group, g in self.graphs:
            if wait is not None and group is not None:
                wait(group)
            g.replay()
        return self.out
