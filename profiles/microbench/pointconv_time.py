"""PointConv forward (b200_pointconv_fwd) at the 20 call shapes of one RPEFlow forward (config 1), batch 74 by default:
time per call for precision 2 (3xTF32) and 1 (TF32).  For an A/B comparison, run it once per build with B200FLOW_LIB
pointing at the other library (profiles/build_variant.sh)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import rpeflow_b200 as b200
from rpeflow_b200 import ops, pointconv as pc
B = int(os.environ.get("BATCH", "74"))
dev = "cuda"
SHAPES = [("down0", 32, 32, 8192, 4096, 2), ("down1", 64, 64, 4096, 2048, 2), ("down2", 96, 96, 2048, 1024, 2),
          ("down3", 128, 128, 1024, 512, 2), ("down4", 192, 192, 512, 256, 2)]
for n in (4096, 2048, 1024, 512, 256):
    SHAPES += [(f"est1_{n}", 195, 128, n, n, 1), (f"est2_{n}", 128, 128, n, n, 1)]
only = os.environ.get("ONLY")
if only: SHAPES = [s for s in SHAPES if s[0] in only.split(",")]
tot = [0.0, 0.0]
for (name, C, cout, N, S, mult) in SHAPES:
    xyz = torch.rand(B, 3, N, device=dev) * 10
    feat = torch.randn(B, C, N, device=dev)
    samp = xyz[:, :, :S].contiguous()
    knn = ops.k_nearest_neighbor(xyz, samp, 16)
    torch.manual_seed(0)
    w = {n: v.to(dev) for n, v in pc.pack_pointconv_weights(pc.PointConvDownSampling(C, cout)).items()}
    res = []
    for prec in (2, 1):
        for _ in range(2): b200.pointconv_forward(xyz, feat, samp, knn, w, prec)
        ts = []
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); b200.pointconv_forward(xyz, feat, samp, knn, w, prec); e1.record(); e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        res.append(min(ts))
    gf = 2.0 * B * S * (16 * (C + 3) * cout + 16 * 16 * (C + 3)) / 1e9
    tot[0] += mult * res[0]; tot[1] += mult * res[1]
    print(f"{name:10s} C={C}->{cout} N={N} S={S} B={B} x{mult}: 3xTF32 {res[0]:.3f} ms ({gf/res[0]:.0f} dense GFLOP/ms)  TF32 {res[1]:.3f} ms")
print(f"20 calls of one forward: 3xTF32 {tot[0]:.2f} ms, TF32 {tot[1]:.2f} ms")
