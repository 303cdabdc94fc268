"""Correlation3D forward + backward at the five pyramid levels, k = 16, batch 8 and 74: the atomic backward, the
deterministic one, and torch autograd of the reference graph under deterministic mode.

Arm atomic: pwc3d.correlation3d -> b200_corr3d_fwd + b200_corr3d_bwd.
Arm det:    the same call under torch.use_deterministic_algorithms(True) -> b200_corr3d_fwd + b200_corr3d_bwd_det.
Arm torch:  torch autograd of oracle.torch_ref.correlation3d under torch.use_deterministic_algorithms(True) on the same
            GPU inputs and knn indices (cuDNN 1x1 convs under torch's TF32 defaults, recorded in the output).
Per level and batch: device time of one forward + backward (CUDA events, 3 warm-up calls, median of 7, L2 flushed by
overwriting a 256 MB buffer before every timed call) and the peak torch.cuda.max_memory_allocated increase over one
call.  GPU name and power limit are read in the same run (read-only query).
Usage: python profiles/microbench/corr3d_det_time.py [--out FILE.json] [--batches 8,74]
"""
import argparse
import json
import os
import sys

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")      # cuBLAS refuses deterministic mode without it
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch  # noqa: E402

import rpeflow_b200 as b200  # noqa: E402
from corr3d_bwd_time import LEVELS, K, gpu_info, measure  # noqa: E402
from oracle import torch_ref  # noqa: E402
from rpeflow_b200 import pwc3d  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batches", default="8,74")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("corr3d_det_time.py measures on a GPU; none is visible")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"gpu": gpu_info(), "k": K, "reps": 7, "warmup": 3, "l2_flush_bytes": 256 << 20,
              "torch": torch.__version__, "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32, "rows": []}
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

            def arm(det, ref=False):
                def run():
                    for t in every:
                        t.grad = None
                    torch.use_deterministic_algorithms(det)
                    try:
                        if ref:
                            out = torch_ref.correlation3d(*leaves, w, k=K, knn11=knn11, knn12=knn12)
                        else:
                            out = b200.correlation3d(*leaves, w, knn12, knn11)
                        out.backward(grad)
                    finally:
                        torch.use_deterministic_algorithms(False)
                return run

            row = {"B": B, "C": C, "N": N}
            for name, fn in (("atomic", arm(False)), ("det", arm(True)), ("torch_det", arm(True, ref=True))):
                t, all_ms, peak = measure(fn, flush)
                row[f"{name}_ms"], row[f"{name}_ms_all"], row[f"{name}_peak_mem_bytes"] = t, all_ms, peak
            result["rows"].append(row)
            print(f"B={B:3d} C={C:3d} N={N:4d}: atomic {row['atomic_ms']*1e3:9.1f} us  det {row['det_ms']*1e3:9.1f} us  "
                  f"torch(det) {row['torch_det_ms']*1e3:9.1f} us  mem {row['atomic_peak_mem_bytes']/2**20:7.1f} / "
                  f"{row['det_peak_mem_bytes']/2**20:7.1f} / {row['torch_det_peak_mem_bytes']/2**20:7.1f} MiB", flush=True)
            del leaves, every, w
            torch.cuda.empty_cache()
    print(json.dumps(result["gpu"]))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
