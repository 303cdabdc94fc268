"""PointConv forward (b200_pointconv_fwd) on clouds of more than 65536 points: device time per call, and an A/B against a
second build of the library.

Cases, batch 2, S = N / 2 sampled points, precisions 2 (3xTF32) and 1 (TF32):
  N = 65537, C in {0, 13, 30} x out_channels in {64, 128, 192, 256} (the shapes of tests/test_forward_reference.py's
  uint32-index cases, at every 3xTF32 MODE and ring depth those indices give);
  N = 131072 at the feature pyramid's widths C -> C, C in {32, 64, 96, 128, 192}.
Uniform clouds in a 30 x 17 x 90 box, neighbour indices from b200_knn_grid, weights of a seeded module.

Each case: CUDA events around one call on torch's current stream, 1 warm-up call, minimum and median of REPS calls;
before every call a 256 MB buffer is overwritten, so that no input, scratch or output is still in the 126 MB L2.
`--variant LIB` also times a second build of the library, alternating default / variant runs `--rounds` times (A B A B);
each run is its own process, because the library is chosen at import (B200FLOW_LIB).  Every 64th output column of the
two builds' first runs is compared (max|a - b| / max|b| per case).  GPU name and power limit are read in the same run
(read-only query).
Usage: python profiles/microbench/pointconv_wide_time.py [--out profiles/pointconv_wide_b200.json] [--variant LIB]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REPS = 7
B = 2


def cases():
    out = [(C, cout, 65537) for C in (0, 13, 30) for cout in (64, 128, 192, 256)]
    return out + [(C, C, 131072) for C in (32, 64, 96, 128, 192)]


def worker(dump):
    """Time every case with the library this process loaded; print one JSON list, save sampled outputs to dump."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    from rpeflow_b200 import ops, pointconv as pc
    dev = torch.device("cuda", 0)
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)
    res, saved = [], {}
    for C, cout, N in cases():
        S = N // 2
        g = torch.Generator(device=dev).manual_seed(N + 1000 * C + cout)
        xyz = torch.rand(B, 3, N, device=dev, generator=g) * torch.tensor([30.0, 17.0, 90.0], device=dev).view(1, 3, 1)
        feat = torch.randn(B, C, N, device=dev, generator=g)
        samp = xyz[:, :, :S].contiguous()
        knn = ops.k_nearest_neighbor(xyz, samp, 16)
        torch.manual_seed(C + cout)
        w = {n: v.to(dev) for n, v in pc.pack_pointconv_weights(pc.PointConvDownSampling(C, cout)).items()}
        for prec in (2, 1):
            out = pc.pointconv_forward(xyz, feat, samp, knn, w, prec)
            ts = []
            for _ in range(REPS):
                flush.fill_(1.0)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                pc.pointconv_forward(xyz, feat, samp, knn, w, prec)
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            ts.sort()
            flop = 2.0 * B * S * (16 * (C + 3) * cout + 16 * 16 * (C + 3))
            res.append({"C": C, "out": cout, "N": N, "S": S, "B": B, "precision": prec, "ms_min": ts[0],
                        "ms_median": ts[len(ts) // 2], "dense_tflops_at_min": flop / ts[0] / 1e9})
            saved[f"C{C}_out{cout}_N{N}_p{prec}"] = out[:, :, ::64].cpu().numpy()
    np.savez(dump, **saved)
    print("RESULT " + json.dumps(res))


def run(dump, lib=None):
    env = dict(os.environ)
    if lib:
        env["B200FLOW_LIB"] = os.path.abspath(lib)
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--dump", dump]
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, check=False)
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("RESULT ")]
    if p.returncode != 0 or not line:
        raise RuntimeError(f"worker failed ({p.returncode}):\n{p.stdout[-3000:]}\n{p.stderr[-3000:]}")
    return json.loads(line[0][len("RESULT "):])


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0] if q.returncode == 0 else None
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pointconv_wide_b200.json"))
    ap.add_argument("--variant", default=None)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--dump", default=None)
    a = ap.parse_args()
    if a.worker:
        worker(a.dump)
        return
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("pointconv_wide_time.py needs a GPU")
    report = {"gpu": torch.cuda.get_device_name(0), "gpu_name_power_limit_max_sm_clock": gpu_info(), "reps": REPS,
              "warmup": 1, "method": "CUDA events around one call, 256 MB written before each call (L2 flushed); "
                                     "min and median of REPS calls per case", "runs": []}
    with tempfile.TemporaryDirectory() as tmp:
        dumps = {}
        for r in range(a.rounds):
            for name, lib in (("default", None), ("variant", a.variant)):
                if name == "variant" and not lib:
                    continue
                dump = os.path.join(tmp, f"{name}{r}.npz")
                label = "default" if lib is None else os.path.basename(lib)
                report["runs"].append({"library": label, "round": r, "cases": run(dump, lib)})
                dumps.setdefault(name, dump)
        if "variant" in dumps:
            x, y = np.load(dumps["default"]), np.load(dumps["variant"])
            report["output_vs_variant"] = {k: float(np.abs(x[k].astype(np.float64) - y[k]).max() / np.abs(y[k]).max())
                                           for k in x.files}
    report["gpu_name_power_limit_max_sm_clock_after"] = gpu_info()
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    for run_ in report["runs"]:
        for c in run_["cases"]:
            print(f"{run_['library']:>24s} r{run_['round']} C={c['C']:>3d} out={c['out']:>3d} N={c['N']:>6d} "
                  f"p{c['precision']} {c['ms_min']:8.3f} ms (median {c['ms_median']:.3f})")
    for k, v in report.get("output_vs_variant", {}).items():
        print(f"  {k}: max|default - variant| / max|variant| = {v:.2e}")
    print("wrote", a.out)


if __name__ == "__main__":
    main()
