"""Multi-start alignment on the device (icp_multistart) against the host-side expansion it replaces
(icp_batch on the pair list repeated K times with numpy-built guesses, then argmin on the host), on
one GPU, in one run.  Prints one JSON document and writes it to --out.

  highres    BASELINE configs[4]: 48 x 4,096-beam scans, consecutive pairs, no per-pair guess,
             32 headings (the inputs of bench.py --workload highres)
  proximity  5,000 x 1,024-beam scans, 20,000 proximity pairs (synth.proximity_pairs), 8 headings

Per workload, with the two arms alternated:
  kernel_ms      device time of the kernels of one call (torch.profiler, CUDA activity, in a profiling
                 pass of its own): the alignment launches, plus expansion and selection for icp_multistart
  host_ms        host-to-host time of one call (median over --reps); the expanded arm includes building
                 the B*K guesses in numpy, and the argmin and gather of the winners
  pcie_bytes     bytes each arm moves across PCIe, computed from the shapes
Both arms run on the same resident scan table, so the table upload is in neither.

Run:  python tools/multistart_bench.py --out multistart_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from icp_slam_b200 import icp as gicp, synth  # noqa: E402


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    name, power, clk = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clk, "torch_name": torch.cuda.get_device_name()}


def workload(name):
    if name == "highres":
        args = argparse.Namespace(workload="highres", scans=48, beams=4096, strong=False, pairs=0)
        scans, pairs_x, _ = bench.workload(args, 0, 1)
        return scans, np.ascontiguousarray(pairs_x[::32]), gicp.heading_starts(32)
    rng = np.random.default_rng(bench.SEED)
    poses = synth.loop_trajectory(5000, step=0.04)
    scans = synth.scans_from_poses(poses, 1024, rng, drop_frac=0.03)
    pairs = synth.proximity_pairs(poses, max_pairs=20000, seed=bench.SEED)
    return scans, pairs, gicp.heading_starts(8)


def expanded_arm(e, pairs, S):
    """What a user without multi-start does: B*K guesses built and sent, B*K results back, argmin."""
    B, K = len(pairs), len(S)
    G = np.broadcast_to(gicp.compose_starts(None, S), (B, K, 3, 3)).reshape(-1, 3, 3)
    res = e.run(np.repeat(pairs, K, axis=0), G, epsilon=bench.EPS, max_iters=bench.MAX_ITERS)
    k = np.argmin(res.error.reshape(B, K), axis=1)
    w = np.arange(B) * K + k
    return res.T[w], res.error[w], res.iters[w], k


def multistart_arm(e, pairs, S):
    ms = e.run_multistart(pairs, S, None, epsilon=bench.EPS, max_iters=bench.MAX_ITERS)
    return ms.T, ms.error, ms.iters, ms.start


def kernel_ms(fn, reps):
    """Device time per call of the library's kernels, from a torch.profiler trace of `reps` calls."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    by = {}
    for ev in prof.key_averages():
        n = ev.key
        if "icp_align_kernel" in n or "multistart_" in n:
            kind = "align" if "icp_align_kernel" in n else ("expand" if "expand" in n else "select")
            by[kind] = by.get(kind, 0.0) + ev.device_time_total / 1e3 / reps
    by["total"] = sum(by.values())
    return by


def run(name, reps, prof_reps):
    scans, pairs, S = workload(name)
    B, K = len(pairs), len(S)
    e = gicp.IcpEngine(0)
    e.set_scans(gicp.ScanTable(scans))
    arms = {"expanded": lambda: expanded_arm(e, pairs, S), "multistart": lambda: multistart_arm(e, pairs, S)}
    out = {n: f() for n, f in arms.items()}                      # warm-up (staging images, allocations)
    same = all(np.array_equal(a, b) for a, b in zip(out["expanded"], out["multistart"]))
    host = {n: [] for n in arms}
    for _ in range(reps):
        for n, f in arms.items():                                  # alternated
            t0 = time.perf_counter()
            f()
            host[n].append((time.perf_counter() - t0) * 1e3)
    kern = {n: kernel_ms(f, prof_reps) for n, f in arms.items()}
    pcie = {"expanded": {"h2d": B * K * (8 + 48), "d2h": B * K * (48 + 8 + 4)},
            "multistart": {"h2d": B * 8 + K * 48, "d2h": B * (48 + 8 + 4 + 4)}}
    return {"pairs": B, "starts": K, "problems": B * K, "scans": len(scans), "beams": int(max(len(s) for s in scans)),
            "results_identical": bool(same),
            "host_ms": {n: {"median": float(np.median(v)), "samples": v} for n, v in host.items()},
            "kernel_ms": kern, "pcie_bytes": pcie,
            "host_saving_frac": 1.0 - float(np.median(host["multistart"])) / float(np.median(host["expanded"]))}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workload", choices=["highres", "proximity", "both"], default="both")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--prof-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    doc = {"gpu": gpu_info(), "epsilon": bench.EPS, "max_iters": bench.MAX_ITERS, "reps": a.reps,
           "prof_reps": a.prof_reps, "workloads": {}}
    for w in (["highres", "proximity"] if a.workload == "both" else [a.workload]):
        doc["workloads"][w] = run(w, a.reps, a.prof_reps)
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
