"""Correlation3D forward + backward at the five pyramid levels, k = 16, batch 8 (a training batch) and 74.

Arm a: this library (pwc3d.correlation3d -> b200_corr3d_fwd + b200_corr3d_bwd).
Arm b: torch autograd of oracle.torch_ref.correlation3d on the same GPU inputs and knn indices (the reference's op
       graph: concat, cuDNN 1x1 convs under torch's TF32 defaults, recorded in the output, gathers and reductions).
Per level and batch: device time of one forward + backward (CUDA events, 3 warm-up calls, median of 7, L2 flushed by
overwriting a 256 MB buffer before every timed call), the peak torch.cuda.max_memory_allocated increase over one call,
FFMA FLOPs of arm a counted from shapes and the resulting rate.  GPU name and power limit are read in the same run
(read-only query).  Usage: python profiles/microbench/corr3d_bwd_time.py [--out FILE.json] [--batches 8,74]
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
from rpeflow_b200 import pwc3d  # noqa: E402

LEVELS = [(32, 4096), (64, 2048), (96, 1024), (128, 512), (192, 256)]
K = 16


def ffma_flops(B, C, N, k=K):
    """FLOPs (2 per FFMA) of arm a's forward + backward, from shapes: per-point linears, the Cout x Cout layer three
    times in the backward (z2 recomputed, dW2, W2^T dz2) and once in the forward, the per-row channel terms (layer-1
    offset, both weight nets' last layer forward and backward), and the 3->8->8 weight-net layers."""
    rows = B * N * k
    linear = B * 2 * N * C * C                          # A1 + G2 (Cin = Cout = C)
    fwd = linear + rows * (C * C + 3 * C + 8 * C + 8 * C + 2 * 88)
    bwd = (linear                                       # A1 / G2 recomputed
           + rows * 3 * C * C                           # z2, dW2, dh1
           + rows * (3 * C + 3 * C + 3 * 8 * C + 3 * 8 * C + 2 * C)   # layer-1 offset, weight nets (fwd + 2 bwd), dP/dv
           + rows * 2 * (88 + 150)                      # 3->8->8 forward and backward, both weight nets
           + 3 * linear)                                # dfeat1, dfeat2, dW1a + dW1b
    return 2 * (fwd + bwd)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batches", default="8,74")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("corr3d_bwd_time.py measures on a GPU; none is visible")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"gpu": gpu_info(), "k": K, "reps": 7, "warmup": 3, "l2_flush_bytes": 256 << 20,
              "torch": torch.__version__, "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32,
              "matmul_allow_tf32": torch.backends.cuda.matmul.allow_tf32, "rows": []}
    for B in (int(b) for b in args.batches.split(",")):
        for C, N in LEVELS:
            torch.manual_seed(0)
            mod = pwc3d.Correlation3D(C, C, k=K)
            w = {n: v.to(dev).requires_grad_(True) for n, v in pwc3d.pack_weights(mod).items()}
            xyz1 = torch.rand(B, 3, N, device=dev)
            xyz2 = xyz1 + 0.02 * torch.randn(B, 3, N, device=dev)
            f1, f2 = torch.randn(B, C, N, device=dev), torch.randn(B, C, N, device=dev)
            knn11 = b200.k_nearest_neighbor(xyz1, xyz1, K)
            knn12 = b200.k_nearest_neighbor(xyz2, xyz1, K)
            leaves = [t.clone().requires_grad_(True) for t in (xyz1, f1, xyz2, f2)]
            grad = torch.randn(B, C, N, device=dev)
            every = leaves + list(w.values())

            def arm_a():
                for t in every:
                    t.grad = None
                b200.correlation3d(*leaves, w, knn12, knn11).backward(grad)

            def arm_b():
                for t in every:
                    t.grad = None
                torch_ref.correlation3d(*leaves, w, k=K, knn11=knn11, knn12=knn12).backward(grad)

            ta, sa, ma = measure(arm_a, flush)
            tb, sb, mb = measure(arm_b, flush)
            fl = ffma_flops(B, C, N)
            row = {"B": B, "C": C, "N": N, "library_ms": ta, "reference_autograd_ms": tb, "speedup": tb / ta,
                   "library_peak_mem_bytes": ma, "reference_peak_mem_bytes": mb, "library_ffma_flops": fl,
                   "library_tflops": fl / (ta * 1e-3) / 1e12, "library_ms_all": sa, "reference_ms_all": sb}
            result["rows"].append(row)
            print(f"B={B:3d} C={C:3d} N={N:4d}: library {ta*1e3:9.1f} us  reference {tb*1e3:9.1f} us  x{tb/ta:5.2f}  "
                  f"mem {ma/2**20:8.1f} / {mb/2**20:8.1f} MiB  {row['library_tflops']:.2f} TFLOP/s", flush=True)
            del leaves, every, w
            torch.cuda.empty_cache()
    print(json.dumps(result["gpu"]))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
