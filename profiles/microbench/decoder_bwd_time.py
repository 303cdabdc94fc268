"""Forward + backward of the decoder ops at the call shapes of one RPEFlow forward, batch 8 (a training batch) and 74.

  knn_interpolation, k = 3: the level-up calls N_{l+1} -> N_l for l = 4..1 (C = 3 for flows, 64 and 128 for features),
                            backwarp_3d's N_l -> N_l (C = 3), the five final flow upsamplings 256 -> 512 ... 4096 -> 8192
                            (C = 3);
  backwarp_2d (border):     (C, H x W) = (128, 18x30), (96, 36x60), (64, 72x120), (32, 144x240);
  convex_upsample:          144 x 240, s = 4.

Arm a: this library (projection.knn_interpolation / backwarp_2d / convex_upsample through their autograd Functions).
Arm b: torch autograd of oracle.torch_ref's functions on the same GPU inputs (knn_interpolation with the same, valid,
       neighbour indices).  torch_ref.backwarp_2d builds its pixel grid on the CPU, so arm b runs the same ops with the
       grid made on the device (ref_backwarp_2d below).
Per shape and batch: device time of one forward + backward of every input gradient (CUDA events, 3 warm-up calls,
minimum of 10, L2 flushed by overwriting a 256 MB buffer before every timed call), the torch.cuda.max_memory_allocated
increase over one call, and the algorithmic bytes of forward + backward (bytes(); each tensor read or written once,
zero-fills of scattered outputs counted) over the library's time as a fraction of the 6.54 TB/s copy peak (DESIGN §5).
GPU name and power limit are read in the same run (read-only query).
Usage: python profiles/microbench/decoder_bwd_time.py [--out FILE.json] [--batches 8,74] [--ops knn,backwarp_2d,convex]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import rpeflow_b200 as b200  # noqa: E402
from oracle import torch_ref  # noqa: E402

COPY_PEAK = 6.54e12          # B/s, DESIGN §5
REPS, WARM = 10, 3
LEVELS = [8192, 4096, 2048, 1024, 512, 256]          # N_0 ... N_5


def knn_shapes():
    out = []
    for l in range(4, 0, -1):
        for C in (3, 64, 128):
            out.append((f"up_l{l + 1}to{l}_C{C}", C, LEVELS[l + 1], LEVELS[l]))
    for l in range(4, 0, -1):
        out.append((f"backwarp3d_l{l}", 3, LEVELS[l], LEVELS[l]))
    for m in (256, 512, 1024, 2048, 4096):
        out.append((f"final_{m}to{2 * m}", 3, m, 2 * m))
    return out


BW_SHAPES = [("l4", 128, 18, 30), ("l3", 96, 36, 60), ("l2", 64, 72, 120), ("l1", 32, 144, 240)]
CU_SHAPES = [("l1", 144, 240, 4)]


def knn_bytes(B, C, M, Q, k=3):
    fwd = 4 * B * (3 * M + C * M + 3 * Q + C * Q) + 8 * B * Q * k
    bwd = 4 * B * (3 * M + C * M + 3 * Q + C * Q) + 8 * B * Q * k + 4 * B * (2 * C * M + 2 * 3 * M + 3 * Q)
    return fwd + bwd


def bw_bytes(B, C, H, W):
    hw = H * W
    fwd = 4 * B * hw * (C + 2 + C)
    bwd = 4 * B * hw * (C + 2 + C + 2 * C + 2)            # x, flow, grad_out; dx zero-filled then accumulated; dflow
    return fwd + bwd


def cu_bytes(B, H, W, s):
    hw = B * H * W
    fwd = 4 * hw * (9 * s * s + 2 + 2 * s * s)
    bwd = 4 * hw * (18 * s * s + 2 * s * s + 2 + 36 + 2)
    return fwd + bwd


def ref_backwarp_2d(x, flow12):
    """oracle.torch_ref.backwarp_2d with its pixel grid made on x's device."""
    nb, _, h, w = x.shape
    xs = torch.arange(0, w, dtype=torch.float32, device=x.device)[None, None, :].expand(nb, h, w)
    ys = torch.arange(0, h, dtype=torch.float32, device=x.device)[None, :, None].expand(nb, h, w)
    g = torch.stack([xs, ys], 1) + flow12
    gn = torch.zeros_like(g)
    gn[:, 0] = 2.0 * g[:, 0] / (w - 1) - 1.0
    gn[:, 1] = 2.0 * g[:, 1] / (h - 1) - 1.0
    return F.grid_sample(x, gn.permute(0, 2, 3, 1), padding_mode="border", align_corners=True)


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
    return min(ms), ms, torch.cuda.max_memory_allocated() - base


def run(leaves, grad, lib_fn, ref_fn, flush):
    def arm(fn):
        def call():
            for t in leaves:
                t.grad = None
            fn().backward(grad)
        return call
    return measure(arm(lib_fn), flush), measure(arm(ref_fn), flush)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batches", default="8,74")
    ap.add_argument("--ops", default="knn,backwarp_2d,convex")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("decoder_bwd_time.py measures on a GPU; none is visible")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ops = args.ops.split(",")
    result = {"gpu": gpu_info(), "reps": REPS, "warmup": WARM, "statistic": "min", "l2_flush_bytes": 256 << 20,
              "torch": torch.__version__, "copy_peak_bytes_per_s": COPY_PEAK, "rows": []}

    def record(op, shape, B, dims, nbytes, lib, ref):
        (ta, sa, ma), (tb, sb, mb) = lib, ref
        row = {"op": op, "shape": shape, "B": B, **dims, "library_ms": ta, "reference_ms": tb, "speedup": tb / ta,
               "library_peak_mem_bytes": ma, "reference_peak_mem_bytes": mb, "bytes": nbytes,
               "library_copy_peak_fraction": nbytes / (ta * 1e-3) / COPY_PEAK,
               "library_ms_all": sa, "reference_ms_all": sb}
        result["rows"].append(row)
        print(f"{op:17s} {shape:20s} B={B:3d}: library {ta:8.3f} ms  reference {tb:8.3f} ms (x{tb / ta:5.2f})  "
              f"mem {ma / 2**20:8.1f} / {mb / 2**20:8.1f} MiB  {row['library_copy_peak_fraction']:.3f} of copy peak",
              flush=True)

    for B in (int(b) for b in args.batches.split(",")):
        torch.manual_seed(0)
        if "knn" in ops:
            for name, C, M, Q in knn_shapes():
                xin = (torch.rand(B, 3, M, device=dev) * 10).requires_grad_(True)
                feat = torch.randn(B, C, M, device=dev).requires_grad_(True)
                xq = (torch.rand(B, 3, Q, device=dev) * 10).requires_grad_(True)
                idx = b200.k_nearest_neighbor(xin.detach(), xq.detach(), 3)
                grad = torch.randn(B, C, Q, device=dev)
                record("knn_interpolation", name, B, {"C": C, "M": M, "Q": Q, "k": 3}, knn_bytes(B, C, M, Q),
                       *run([xin, feat, xq], grad,
                            lambda: b200.knn_interpolation(xin, feat, xq, 3, knn_indices=idx),
                            lambda: torch_ref.knn_interpolation(xin, feat, xq, 3, knn_indices=idx), flush))
                del xin, feat, xq, idx, grad
        if "backwarp_2d" in ops:
            for name, C, H, W in BW_SHAPES:
                x = torch.randn(B, C, H, W, device=dev).requires_grad_(True)
                flow = (3.0 * torch.randn(B, 2, H, W, device=dev)).requires_grad_(True)
                grad = torch.randn(B, C, H, W, device=dev)
                record("backwarp_2d", name, B, {"C": C, "H": H, "W": W}, bw_bytes(B, C, H, W),
                       *run([x, flow], grad, lambda: b200.backwarp_2d(x, flow, "border"),
                            lambda: ref_backwarp_2d(x, flow), flush))
                del x, flow, grad
        if "convex" in ops:
            for name, H, W, s in CU_SHAPES:
                flow = (4.0 * torch.randn(B, 2, H, W, device=dev)).requires_grad_(True)
                mask = torch.randn(B, 9 * s * s, H, W, device=dev).requires_grad_(True)
                grad = torch.randn(B, 2, H * s, W * s, device=dev)
                record("convex_upsample", name, B, {"H": H, "W": W, "s": s}, cu_bytes(B, H, W, s),
                       *run([flow, mask], grad, lambda: b200.convex_upsample(flow, mask, s),
                            lambda: torch_ref.convex_upsample(flow, mask, s), flush))
                del flow, mask, grad
        torch.cuda.empty_cache()
    for B in sorted({r["B"] for r in result["rows"]}):
        tot = {}
        for op in ("knn_interpolation", "backwarp_2d", "convex_upsample"):
            rows = [r for r in result["rows"] if r["B"] == B and r["op"] == op]
            tot[op] = {"library_ms": sum(r["library_ms"] for r in rows), "reference_ms": sum(r["reference_ms"] for r in rows)}
        result.setdefault("totals_over_listed_shapes", {})[str(B)] = tot
        print(f"B={B}: " + "  ".join(f"{op} {t['library_ms']:.2f} / {t['reference_ms']:.2f} ms" for op, t in tot.items()))
    print(json.dumps(result["gpu"]))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
