"""correlation2d forward + backward under autograd at the model's level shapes, batch 8 (a training batch) and 74.

Shapes (C, H x W): the five levels of `things` (32 144x240, 64 72x120, 96 36x60, 128 18x30, 192 9x15) and level 1 of
`dsec` (32 128x160), md = 4.

Arm A: b200.correlation2d on the NCHW maps, i.e. ops.Correlation2dNCHWFunction (b200_corr2d_fwd_nchw or the NHWC
       forward, b200_corr2d_bwd_nchw; no permutes).
Arm B: what the reference's wrapper does with this library's extension shims: permute both maps to NHWC, then
       ops.CorrelationFunction (b200_corr2d_fwd / b200_corr2d_bwd, NCHW gradients permuted to NHWC and back by autograd).
Arm C: torch autograd of oracle.torch_ref.correlation2d (the reference's libtorch path); skipped where it runs out of
       memory.
Kernels alone: b200_corr2d_bwd_nchw on the NCHW maps against b200_corr2d_bwd on NHWC copies of the same data, both
       gradients.
Per shape and batch: device time (CUDA events, 3 warm-up calls, minimum of 10, L2 flushed by overwriting a 256 MB
buffer before every timed call) and the torch.cuda.max_memory_allocated increase over one forward + backward.  GPU
name and power limit are read in the same run (read-only query).
Usage: python profiles/microbench/corr2d_train_time.py [--out FILE.json] [--batches 8,74]
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
from rpeflow_b200 import _lib  # noqa: E402
from oracle import torch_ref  # noqa: E402

REPS, WARM = 10, 3
SHAPES = [("things_l1", 32, 144, 240), ("things_l2", 64, 72, 120), ("things_l3", 96, 36, 60), ("things_l4", 128, 18, 30),
          ("things_l5", 192, 9, 15), ("dsec_l1", 32, 128, 160)]


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else None
    except Exception as e:                              # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def measure(fn, flush):
    for _ in range(WARM):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(REPS):
        flush.zero_()
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return {"ms": min(ms), "ms_all": ms, "peak_mem_bytes": torch.cuda.max_memory_allocated() - base}


def train_call(fn, leaves, grad):
    def call():
        for t in leaves:
            t.grad = None
        fn().backward(grad)
    return call


def wrapper_route(a, b):
    """models/csrc/wrapper.py:68-70 with this library's shims behind CorrelationFunction."""
    return b200.CorrelationFunction.apply(a.permute(0, 2, 3, 1).contiguous().float(), b.permute(0, 2, 3, 1).contiguous().float(), 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batches", default="8,74")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("corr2d_train_time.py measures on a GPU; none is visible")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lib, stream = _lib.lib, torch.cuda.current_stream().cuda_stream
    result = {"gpu": gpu_info(), "reps": REPS, "warmup": WARM, "statistic": "min", "l2_flush_bytes": 256 << 20,
              "torch": torch.__version__, "md": 4, "rows": []}
    for B in (int(b) for b in args.batches.split(",")):
        for name, C, H, W in SHAPES:
            torch.manual_seed(0)
            a = torch.randn(B, C, H, W, device=dev).requires_grad_(True)
            b = torch.randn(B, C, H, W, device=dev).requires_grad_(True)
            grad = torch.randn(B, 81, H, W, device=dev)
            row = {"shape": name, "B": B, "C": C, "H": H, "W": W}
            row["A_function"] = measure(train_call(lambda: b200.correlation2d(a, b, 4), [a, b], grad), flush)
            row["B_wrapper_route"] = measure(train_call(lambda: wrapper_route(a, b), [a, b], grad), flush)
            try:
                row["C_torch_ref"] = measure(train_call(lambda: torch_ref.correlation2d(a, b, 4), [a, b], grad), flush)
            except torch.cuda.OutOfMemoryError:
                row["C_torch_ref"] = None
            torch.cuda.empty_cache()
            ad, bd = a.detach(), b.detach()
            an, bn = ad.permute(0, 2, 3, 1).contiguous(), bd.permute(0, 2, 3, 1).contiguous()
            g1, g2 = torch.empty_like(ad), torch.empty_like(bd)
            row["kernel_bwd_nchw"] = measure(lambda: _lib.check(lib.b200_corr2d_bwd_nchw(
                grad.data_ptr(), ad.data_ptr(), bd.data_ptr(), g1.data_ptr(), g2.data_ptr(), B, C, H, W, 4, stream),
                "b200_corr2d_bwd_nchw"), flush)
            ref1, ref2 = g1.clone(), g2.clone()
            row["kernel_bwd_nhwc"] = measure(lambda: _lib.check(lib.b200_corr2d_bwd(
                grad.data_ptr(), an.data_ptr(), bn.data_ptr(), g1.data_ptr(), g2.data_ptr(), B, C, H, W, 4, stream),
                "b200_corr2d_bwd"), flush)
            row["kernel_same_bits"] = bool(torch.equal(ref1, g1) and torch.equal(ref2, g2))
            row["A_over_B_time"] = row["A_function"]["ms"] / row["B_wrapper_route"]["ms"]
            result["rows"].append(row)
            c = row["C_torch_ref"]
            print(f"{name:10s} B={B:3d}: A {row['A_function']['ms']:8.3f} ms  B {row['B_wrapper_route']['ms']:8.3f} ms  "
                  f"C {c['ms'] if c else float('nan'):8.3f} ms | mem A {row['A_function']['peak_mem_bytes'] / 2**20:8.1f} "
                  f"B {row['B_wrapper_route']['peak_mem_bytes'] / 2**20:8.1f} MiB | bwd kernels nchw "
                  f"{row['kernel_bwd_nchw']['ms']:.3f} nhwc {row['kernel_bwd_nhwc']['ms']:.3f} ms "
                  f"(same bits: {row['kernel_same_bits']})", flush=True)
            del a, b, grad, ad, bd, an, bn, g1, g2, ref1, ref2
            torch.cuda.empty_cache()
    result["shapes_where_A_is_not_faster_than_B"] = [f"{r['shape']} B={r['B']}" for r in result["rows"]
                                                     if r["A_over_B_time"] >= 1.0]
    print(json.dumps(result["gpu"]), "A not faster than B at:", result["shapes_where_A_is_not_faster_than_B"])
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
