"""Forward + backward of the projection gathers at the call shapes of one RPEFlow forward, batch 8 (a training batch)
and 74.

  grid_sample_wrapper:          (C, H x W, N) at pyramid levels 1..5 = (32, 144x240, 4096), (64, 72x120, 2048),
                                (96, 36x60, 1024), (128, 18x30, 512), (192, 9x15, 256), plus the level-1 81-channel cost
                                volume and the 96-channel decoder map (RPEFlow_core.py:336-337, :376, :395);
  batch_indexing_channel_first: the pyramid's xyz gathers [B,3,8192] -> 4096 / 1024 / 256 points (pwc3d_core.py:8-28)
                                and a [B,64,4096] feature gather by a [B,4096,16] neighbour index;
  batch_indexing_channel_last:  [B,4096,3] and [B,4096,64] gathered by a [B,4096,16] neighbour index (the PointConv
                                bodies' gathers, models/pointconv.py).

Arm a: this library (projection.grid_sample_wrapper / batch_indexing_channel_* through their autograd Functions).
Arm b: torch autograd of oracle.torch_ref's functions on the same GPU inputs and indices (torch_ref's channel-last
       gather builds its batch index on the CPU, so arm b runs the same indexing with that index made on the device).
Per shape and batch: device time of one forward + backward of every input gradient (CUDA events, 3 warm-up calls,
minimum of 10, L2 flushed by overwriting a 256 MB buffer before every timed call), the torch.cuda.max_memory_allocated
increase over one call, and the algorithmic bytes of forward + backward (the *_bytes functions below; each tensor read
or written once, zero-fills of scattered outputs counted) over the library's time as a fraction of the 6.54 TB/s copy
peak (DESIGN §5).  GPU name and power limit are read in the same run (read-only query).
Usage: python profiles/microbench/projection_bwd_time.py [--out FILE.json] [--batches 8,74] [--ops grid_sample,gather_cf,gather_cl]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import rpeflow_b200 as b200  # noqa: E402
from oracle import torch_ref  # noqa: E402
from decoder_bwd_time import COPY_PEAK, REPS, WARM, gpu_info, run  # noqa: E402

GS_SHAPES = [("l1_C32", 32, 144, 240, 4096), ("l2_C64", 64, 72, 120, 2048), ("l3_C96", 96, 36, 60, 1024),
             ("l4_C128", 128, 18, 30, 512), ("l5_C192", 192, 9, 15, 256), ("l1_cost_C81", 81, 144, 240, 4096),
             ("l1_dec_C96", 96, 144, 240, 4096)]
CF_SHAPES = [("xyz_8192to4096", 3, 8192, (4096,)), ("xyz_8192to1024", 3, 8192, (1024,)),
             ("xyz_8192to256", 3, 8192, (256,)), ("feat_C64_knn16", 64, 4096, (4096, 16))]
CL_SHAPES = [("xyz_C3_knn16", 3, 4096, (4096, 16)), ("feat_C64_knn16", 64, 4096, (4096, 16))]


def grid_sample_bytes(B, C, H, W, N):
    taps = min(16 * C * N, 4 * C * H * W)
    fwd = 8 * N + 4 * C * N + taps
    bwd = 8 * N + 4 * C * N + taps + 4 * C * H * W + taps + 8 * N    # xy, grad_out, taps for dxy; dfeat zero-fill + scatter; dxy
    return B * (fwd + bwd)


def gather_bytes(B, C, N, I):
    rows = min(4 * C * I, 4 * C * N)                                   # a data element read (scattered to) more than once counts once
    fwd = 8 * I + rows + 4 * C * I
    bwd = 8 * I + 4 * C * I + 4 * C * N + rows                         # idx, grad_out; ddata zero-fill + scatter
    return B * (fwd + bwd)


def ref_gather_cl(data, idx):
    """oracle.torch_ref.batch_indexing_channel_last with its batch index made on the data's device."""
    nb = data.shape[0]
    b = torch.arange(nb, device=data.device).view([nb] + [1] * (idx.dim() - 1)).expand_as(idx)
    return data[b, idx]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batches", default="8,74")
    ap.add_argument("--ops", default="grid_sample,gather_cf,gather_cl")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("projection_bwd_time.py measures on a GPU; none is visible")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ops = args.ops.split(",")
    result = {"gpu": gpu_info(), "reps": REPS, "warmup": WARM, "statistic": "min",
              "l2_flush_bytes": 256 << 20, "torch": torch.__version__, "copy_peak_bytes_per_s": COPY_PEAK, "rows": []}

    def record(op, shape, B, dims, nbytes, lib, ref):
        (ta, sa, ma), (tb, sb, mb) = lib, ref
        row = {"op": op, "shape": shape, "B": B, **dims, "library_ms": ta, "reference_ms": tb, "speedup": tb / ta,
               "library_peak_mem_bytes": ma, "reference_peak_mem_bytes": mb, "bytes": nbytes,
               "library_copy_peak_fraction": nbytes / (ta * 1e-3) / COPY_PEAK,
               "library_ms_all": sa, "reference_ms_all": sb}
        result["rows"].append(row)
        print(f"{op:28s} {shape:16s} B={B:3d}: library {ta:8.3f} ms  reference {tb:8.3f} ms (x{tb / ta:5.2f})  "
              f"mem {ma / 2**20:8.1f} / {mb / 2**20:8.1f} MiB  {row['library_copy_peak_fraction']:.3f} of copy peak",
              flush=True)

    for B in (int(b) for b in args.batches.split(",")):
        torch.manual_seed(0)
        if "grid_sample" in ops:
            for name, C, H, W, N in GS_SHAPES:
                feat = torch.randn(B, C, H, W, device=dev).requires_grad_(True)
                xy = torch.stack([torch.rand(B, N, device=dev) * (W - 1), torch.rand(B, N, device=dev) * (H - 1)], 1)
                xy.requires_grad_(True)
                grad = torch.randn(B, C, N, device=dev)
                record("grid_sample_wrapper", name, B, {"C": C, "H": H, "W": W, "N": N}, grid_sample_bytes(B, C, H, W, N),
                       *run([feat, xy], grad, lambda: b200.grid_sample_wrapper(feat, xy),
                            lambda: torch_ref.grid_sample_wrapper(feat, xy), flush))
                del feat, xy, grad
        for kind, shapes in (("gather_cf", CF_SHAPES), ("gather_cl", CL_SHAPES)):
            if kind not in ops:
                continue
            for name, C, N, ishape in shapes:
                cl = kind == "gather_cl"
                data = torch.randn(*((B, N, C) if cl else (B, C, N)), device=dev).requires_grad_(True)
                idx = torch.randint(0, N, (B, *ishape), device=dev)
                I = idx[0].numel()
                grad = torch.randn(*((B, *ishape, C) if cl else (B, C, *ishape)), device=dev)
                op = "batch_indexing_channel_last" if cl else "batch_indexing_channel_first"
                lib_fn = b200.batch_indexing_channel_last if cl else b200.batch_indexing_channel_first
                ref_fn = ref_gather_cl if cl else torch_ref.batch_indexing_channel_first
                record(op, name, B, {"C": C, "N": N, "I": I}, gather_bytes(B, C, N, I),
                       *run([data], grad, lambda: lib_fn(data, idx), lambda: ref_fn(data, idx), flush))
                del data, idx, grad
        torch.cuda.empty_cache()
    for B in sorted({r["B"] for r in result["rows"]}):
        tot = {}
        for op in ("grid_sample_wrapper", "batch_indexing_channel_first", "batch_indexing_channel_last"):
            rows = [r for r in result["rows"] if r["B"] == B and r["op"] == op]
            if rows:
                tot[op] = {"library_ms": sum(r["library_ms"] for r in rows), "reference_ms": sum(r["reference_ms"] for r in rows)}
        result.setdefault("totals_over_listed_shapes", {})[str(B)] = tot
        print(f"B={B}: " + "  ".join(f"{op} {t['library_ms']:.2f} / {t['reference_ms']:.2f} ms" for op, t in tot.items()))
    print(json.dumps(result["gpu"]))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
