"""PointConv forward + backward at the 20 call shapes of one RPEFlow forward (those of pointconv_time.py: down0-4 twice,
est1 / est2 at 4096 ... 256 points), batch 8 (a training batch) and 74.

Arm a: this library (pointconv.PointConvFunction -> b200_pointconv_fwd_linear + b200_pointconv_bwd), then LeakyReLU.
Arm b: torch autograd of oracle.torch_ref.pointconv on the same GPU inputs and knn indices (the reference's op graph:
       gathers, weight-net 1x1 convs, torch.matmul, F.linear), once with TF32 off and once at torch's defaults (cuDNN
       TF32 on, matmul TF32 off); both settings are recorded.
Per shape and batch: device time of one forward + backward of all nine gradients (CUDA events, 3 warm-up calls, median
of 7, L2 flushed by overwriting a 256 MB buffer before every timed call), the peak torch.cuda.max_memory_allocated
increase over one call, and the FLOPs of the body counted from shapes (forward, recompute and backward; see flops())
with the resulting rate.  GPU name and power limit are read in the same run (read-only query).
Usage: python profiles/microbench/pointconv_bwd_time.py [--out FILE.json] [--batches 8,74] [--only down0,est1_4096]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import rpeflow_b200 as b200  # noqa: E402
from oracle import torch_ref  # noqa: E402
from rpeflow_b200 import pointconv as pc  # noqa: E402

K = 16
SHAPES = [("down0", 32, 32, 8192, 4096, 2), ("down1", 64, 64, 4096, 2048, 2), ("down2", 96, 96, 2048, 1024, 2),
          ("down3", 128, 128, 1024, 512, 2), ("down4", 192, 192, 512, 256, 2)]
for _n in (4096, 2048, 1024, 512, 256):
    SHAPES += [(f"est1_{_n}", 195, 128, _n, _n, 1), (f"est2_{_n}", 128, 128, _n, _n, 1)]


def flops(B, C, Cout, S):
    """2 x multiply-adds of the body per call: forward (weight net, M = W.F, y = L.M), backward (weight net and M
    recomputed, dM = dy.L, dL = dy^T.M, dW = dM.F^T, dF = W^T.dM, weight-net backward counted as twice its forward)."""
    rows, c3 = B * S, C + 3
    linear = rows * 16 * c3 * Cout
    mix = rows * 16 * K * c3
    wnet = rows * K * (3 * 8 + 8 * 16)
    return 2 * (linear + mix + wnet                      # forward
                + mix + wnet                             # recompute of W and M in the backward
                + 2 * linear + 2 * mix + 2 * wnet)       # dM, dL; dW, dF; weight-net backward


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else None
    except Exception as e:                              # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def measure(fn, flush, reps=7, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        flush.zero_()
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    ms.sort()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    return ms[len(ms) // 2], ms, peak


class _tf32:
    def __init__(self, cudnn, matmul):
        self.want = (cudnn, matmul)

    def __enter__(self):
        self.old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.want

    def __exit__(self, *exc):
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.old


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batches", default="8,74")
    ap.add_argument("--only", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pointconv_bwd_time.py measures on a GPU; none is visible")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    defaults = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    shapes = [s for s in SHAPES if args.only is None or s[0] in args.only.split(",")]
    result = {"gpu": gpu_info(), "k": K, "reps": 7, "warmup": 3, "l2_flush_bytes": 256 << 20, "torch": torch.__version__,
              "reference_tf32_default": {"cudnn_allow_tf32": defaults[0], "matmul_allow_tf32": defaults[1]},
              "library_precision": 2, "rows": []}
    for B in (int(b) for b in args.batches.split(",")):
        for name, C, Cout, N, S, mult in shapes:
            torch.manual_seed(0)
            w = {n: v.to(dev).requires_grad_(True)
                 for n, v in pc.pack_pointconv_weights(pc.PointConvDownSampling(C, Cout)).items()}
            xyz = torch.rand(B, 3, N, device=dev) * 10
            feat = torch.randn(B, C, N, device=dev)
            nosample = name.startswith("est")
            sampled = xyz if nosample else xyz[:, :, :S].contiguous()
            knn = b200.k_nearest_neighbor(xyz, sampled, K)
            x = xyz.clone().requires_grad_(True)
            f = feat.clone().requires_grad_(True)
            s = x if nosample else sampled.clone().requires_grad_(True)
            grad = torch.randn(B, Cout, S, device=dev)
            every = [x, f] + ([] if nosample else [s]) + list(w.values())

            def arm_a():
                for t in every:
                    t.grad = None
                pc.pointconv(x, f, s, knn, w).backward(grad)

            def arm_b():
                for t in every:
                    t.grad = None
                torch_ref.pointconv(x, f, s, w, k=K, knn=knn).backward(grad)

            ta, sa, ma = measure(arm_a, flush)
            with _tf32(False, False):
                tb, sb, mb = measure(arm_b, flush)
            with _tf32(*defaults):
                tc, sc, mc = measure(arm_b, flush)
            fl = flops(B, C, Cout, S)
            row = {"shape": name, "calls_per_forward": mult, "B": B, "C": C, "Cout": Cout, "N": N, "S": S,
                   "library_ms": ta, "reference_fp32_ms": tb, "reference_default_tf32_ms": tc,
                   "speedup_vs_fp32": tb / ta, "speedup_vs_default": tc / ta,
                   "library_peak_mem_bytes": ma, "reference_fp32_peak_mem_bytes": mb,
                   "reference_default_peak_mem_bytes": mc, "flops": fl, "library_tflops": fl / (ta * 1e-3) / 1e12,
                   "library_ms_all": sa, "reference_fp32_ms_all": sb, "reference_default_ms_all": sc}
            result["rows"].append(row)
            print(f"{name:10s} B={B:3d} C={C:3d}->{Cout:3d} N={N:5d} S={S:5d}: library {ta:8.3f} ms  reference fp32 "
                  f"{tb:8.3f} ms (x{tb/ta:5.2f})  default {tc:8.3f} ms (x{tc/ta:5.2f})  mem {ma/2**20:8.1f} / "
                  f"{mb/2**20:8.1f} / {mc/2**20:8.1f} MiB  {row['library_tflops']:.2f} TFLOP/s", flush=True)
            del x, f, s, every, w
            torch.cuda.empty_cache()
    for B in sorted({r["B"] for r in result["rows"]}):
        rows = [r for r in result["rows"] if r["B"] == B]
        tot = {k: sum(r["calls_per_forward"] * r[k] for r in rows)
               for k in ("library_ms", "reference_fp32_ms", "reference_default_tf32_ms")}
        result.setdefault("totals_per_forward", {})[str(B)] = tot
        print(f"B={B}: 20 calls forward + backward: library {tot['library_ms']:.2f} ms, reference fp32 "
              f"{tot['reference_fp32_ms']:.2f} ms, reference default {tot['reference_default_tf32_ms']:.2f} ms")
    print(json.dumps(result["gpu"]))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
