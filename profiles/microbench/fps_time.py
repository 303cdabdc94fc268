"""Furthest point sampling above 8192 points: device time per call and per dependent iteration.

Cases: (B, N, S) in {1, 8} x {65537, 131072, 1048576} x {4096, N/8} (b200_fps_large), and the sizes where b200_fps's
cluster kernel fps_kernel<CS> ends, 16384 / 32768 / 65536 points with S = 4096, at the `hd` batch of 36 clouds and on a
single cloud.  Uniform clouds in a 30 x 17 x 90 box (FT3D-shaped, as the bench), seeded.

Each case: CUDA events around one call on torch's current stream, 1 warm-up call, minimum of REPS >= 5 calls; the
input is written once and then read by every call (one cloud of 1 M points is 12 MB: it stays in the 126 MB L2, as it
would in a real pyramid build that just wrote it).  ns per dependent iteration = time / (S - 1).
`--variant LIB` also times a second build of the library (profiles/build_variant.sh, e.g. built with
-DB200_FPS_CLUSTER_MAX_N=8192 so that every cloud above 8192 points takes the pruned cluster scan), alternating
default / variant runs `--rounds` times; each run is its own process, because the library is chosen at import
(B200FLOW_LIB).  Index lists of both builds are compared.
Where oracle/_ref was built, the reference's own CUDA kernel (refcuda.fps) runs on the same inputs; its time and whether
its index list equals this library's are recorded.
GPU name and power limit are read in the same run (read-only query).
Usage: python profiles/microbench/fps_time.py [--out profiles/fps_large_b200.json] [--variant LIB] [--rounds 2]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REPS = 5


def cases():
    out = []
    for B in (1, 8):
        for N in (65537, 131072, 1048576):
            for S in (4096, N // 8):
                out.append((B, N, S))
    for N in (16384, 32768, 65536):
        for B in (36, 1):
            out.append((B, N, 4096))
    return out


def worker(only_ref):
    """Time every case with the library this process loaded; print one JSON object."""
    sys.path.insert(0, ROOT)
    import torch
    import rpeflow_b200 as b200
    from oracle import refcuda

    from rpeflow_b200 import _lib
    dev = torch.device("cuda", 0)
    res = []

    def route(N, S):              # b200_fps checks its size limit before it returns on an empty call
        big = N > b200.ops.FPS_CLUSTER_MAX_N or _lib.lib.b200_fps(None, None, 0, N, S, None) == _lib.B200_ENOSUP
        return "b200_fps_large" if big else "b200_fps"

    for B, N, S in cases():
        g = torch.Generator(device=dev).manual_seed(N * 7 + B)
        xyz = torch.rand(B, N, 3, device=dev, generator=g) * torch.tensor([30.0, 17.0, 90.0], device=dev)

        def timed(fn):
            fn()
            torch.cuda.synchronize()
            best = float("inf")
            for _ in range(REPS):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                out = fn()
                b.record()
                torch.cuda.synchronize()
                best = min(best, a.elapsed_time(b))
            return best, out

        row = {"B": B, "N": N, "S": S}
        if not only_ref:
            ms, idx = timed(lambda: b200.ops._furthest_point_sampling_cuda(xyz, S))
            row.update(ms=ms, ns_per_iteration=ms * 1e6 / (S - 1),
                       kernel=route(N, S), idx_sha1=hashlib.sha1(idx.cpu().numpy().tobytes()).hexdigest())
        if only_ref and refcuda.available() and B == 1:
            ms, ridx = timed(lambda: refcuda.fps(xyz, S, sync=False))
            mine = b200.ops._furthest_point_sampling_cuda(xyz, S)
            row.update(ref_cuda_ms=ms, ref_cuda_ns_per_iteration=ms * 1e6 / (S - 1),
                       ref_cuda_index_identical=bool(torch.equal(ridx, mine)))
        res.append(row)
    print("RESULT " + json.dumps(res))


def run(lib=None, only_ref=False):
    env = dict(os.environ)
    if lib:
        env["B200FLOW_LIB"] = os.path.abspath(lib)
    cmd = [sys.executable, os.path.abspath(__file__), "--worker"] + (["--ref"] if only_ref else [])
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, check=False)
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("RESULT ")]
    if p.returncode != 0 or not line:
        raise RuntimeError(f"worker failed ({p.returncode}):\n{p.stdout[-3000:]}\n{p.stderr[-3000:]}")
    return json.loads(line[0][len("RESULT "):])


def gpu_info():
    info = {}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["gpu_name_power_limit_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else None
    except Exception as e:  # noqa: BLE001
        info["gpu_name_power_limit_max_sm_clock"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fps_large_b200.json"))
    ap.add_argument("--variant", default=None)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--ref", action="store_true")
    a = ap.parse_args()
    if a.worker:
        worker(a.ref)
        return
    sys.path.insert(0, ROOT)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("fps_time.py needs a GPU")
    report = {"gpu": torch.cuda.get_device_name(0), **gpu_info(), "reps": REPS, "warmup": 1,
              "method": "CUDA events, minimum of REPS calls per case; inputs L2-resident up to 126 MB", "runs": []}
    for r in range(a.rounds):
        report["runs"].append({"library": "default", "round": r, "cases": run()})
        if a.variant:
            report["runs"].append({"library": os.path.basename(a.variant), "round": r, "cases": run(a.variant)})
    sys.path.insert(0, ROOT)
    from oracle import refcuda
    report["reference_cuda"] = run(only_ref=True) if refcuda.available() else "oracle/_ref not built: not measured"
    report.update(gpu_info_after=gpu_info())
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    for run_ in report["runs"]:
        for c in run_["cases"]:
            print(f"{run_['library']:>24s} r{run_['round']} B={c['B']:>3d} N={c['N']:>8d} S={c['S']:>7d} "
                  f"{c['ms']:9.3f} ms {c['ns_per_iteration']:8.1f} ns/it  {c['kernel']}")
    print("wrote", a.out)


if __name__ == "__main__":
    main()
