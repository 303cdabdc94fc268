"""Correlation3D at the five pyramid levels, batch 74 (the bench batch): device time per call, L2 flushed between calls.
For an A/B comparison, run it once per build with B200FLOW_LIB pointing at the other library (profiles/build_variant.sh)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
import rpeflow_b200 as b200
from rpeflow_b200 import pwc3d

dev = torch.device("cuda", 0)
B = int(os.environ.get("BATCH", "74"))
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
tot = 0.0
LEVELS = [(32, 4096), (64, 2048), (96, 1024), (128, 512), (192, 256)]
if os.environ.get("LEVELS"):
    LEVELS = [LEVELS[int(i)] for i in os.environ["LEVELS"].split(",")]
for C, N in LEVELS:
    torch.manual_seed(0)
    mod = pwc3d.Correlation3D(C, C, k=16)
    w = {n: v.to(dev) for n, v in pwc3d.pack_weights(mod).items()}
    xyz1 = torch.rand(B, 3, N, device=dev); xyz2 = xyz1 + 0.02 * torch.randn(B, 3, N, device=dev)
    f1 = torch.randn(B, C, N, device=dev); f2 = torch.randn(B, C, N, device=dev)
    knn11 = b200.k_nearest_neighbor(xyz1, xyz1, 16); knn12 = b200.k_nearest_neighbor(xyz2, xyz1, 16)
    fn = lambda: pwc3d.correlation3d_forward(xyz1, f1, xyz2, f2, w, knn12, knn11, 2)
    for _ in range(3): fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(7):
        flush.zero_(); a.record(); fn(); b.record(); b.synchronize(); ms.append(a.elapsed_time(b))
    ms.sort(); tot += ms[3]
    print(f"C={C:3d} N={N:4d} B={B}: {ms[3]*1e3:8.1f} us", flush=True)
print(f"total {tot:.3f} ms")
