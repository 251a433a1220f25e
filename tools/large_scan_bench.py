"""Scans beyond one CTA's shared memory: rates and latencies of the large-scan variant of the alignment
kernel (per-CTA device scratch), on one GPU, in one run.  Prints one JSON document and writes it to
--out.

  chains      pairs/s and executed-PDE rate (share of the FP32-pipe peak, bench.py's `roofline`
              definitions) for chains of 16,384 / 32,768 / 65,536-beam scans
  latency     one 16k and one 65k pair, with and without thread-block clusters
  submap      1,024-beam sources onto 16-scan merged targets
  mixed       a 1,024-beam chain on a table holding one 20,000-point scan, against the same chain on
              the table without it (host entry point: split launches; device entry point: every pair
              on the large variant)
  global_cost "large" forced against the default (shared-memory kernel) on the 1,024 and 4,096-beam
              chains, alternated in this run
  c_port      the C oracle (OpenMP, all cores) on a subsample of the 16k chain

Run:  python tools/large_scan_bench.py --out large_scan_bench.json
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

from icp_slam_b200 import icp as gicp, synth  # noqa: E402
from oracle import c_oracle  # noqa: E402

EPS = 0.05


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    name, power, clk = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clk, "torch_name": torch.cuda.get_device_name()}


class Dev:
    """Resident-table runs on the device, timed with CUDA events."""

    def __init__(self, e, scans, pairs, init):
        import torch
        self.torch, self.e = torch, e
        e.set_scans(scans)
        dev = torch.device("cuda", e.device)
        B = len(pairs)
        self.B = B
        self.p = torch.from_numpy(np.ascontiguousarray(pairs, dtype=np.int32)).to(dev)
        self.i = torch.from_numpy(np.ascontiguousarray(init[:, :2, :].reshape(B, 6))).to(dev)
        self.T = torch.empty((B, 6), dtype=torch.float64, device=dev)
        self.err = torch.empty(B, dtype=torch.float64, device=dev)
        self.passes = torch.empty(B, dtype=torch.int32, device=dev)
        self.lens = np.array([len(s) for s in scans], dtype=np.int64)
        self.pairs = np.asarray(pairs)

    def launch(self, exhaustive=False):
        self.e.run_device(self.p, self.i, self.T, self.err, self.passes, epsilon=EPS, exhaustive=exhaustive)

    def time(self, reps, exhaustive=False):
        torch = self.torch
        self.launch(exhaustive)                                  # warm-up
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            self.launch(exhaustive)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps * 1e-3

    def executed(self, exhaustive=False):
        self.e.count_work(True)
        self.launch(exhaustive)
        v = self.e.read_work()
        self.e.count_work(False)
        return v

    def work(self):
        """Distance evaluations of the reference's brute force: passes * N1 * N2 per pair."""
        p = self.passes.cpu().numpy().astype(np.float64)
        return float(np.sum(p * self.lens[self.pairs[:, 0]] * self.lens[self.pairs[:, 1]]))


def pde_peak(e):
    info = e.kernel_info()
    q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.split()[0]
    return info["sm_count"] * 128 * float(q) * 1e6 / 4.0          # bench.py: FP32-pipe lane-slots / 4 per PDE


def chain_entry(e, beams, n_scans, reps, peak, seed):
    scans, pairs, init, _, _ = synth.make_chain_workload(n_scans, beams, seed=seed)
    d = Dev(e, scans, pairs, init)
    t = d.time(reps)
    ex = d.executed()
    work = d.work()
    te = d.time(1, exhaustive=True)
    return {"beams": beams, "pairs": d.B, "kernel_ms": t * 1e3, "pairs_per_s": d.B / t,
            "passes_mean": float(d.passes.float().mean().item()),
            "executed_pde": ex, "executed_tpde_s": ex / t * 1e-12, "frac_fp32_pipe": ex / t / peak,
            "executed_share_of_brute_force": ex / work,
            "exhaustive": {"kernel_ms": te * 1e3, "tpde_s": work / te * 1e-12, "frac_fp32_pipe": work / te / peak}}


def latency(e, beams, seed, reps):
    scans, pairs, init, _, _ = synth.make_chain_workload(2, beams, seed=seed)
    d = Dev(e, scans, pairs, init)
    out = {}
    for name, cl in (("cluster_default", -1), ("single_cta", 0)):
        e.set_tuning("cluster", cl)
        out[name + "_ms"] = d.time(reps) * 1e3
    e.set_tuning("cluster", -1)
    out["points"] = [len(s) for s in scans]
    out["passes"] = int(d.passes.cpu()[0])
    return out


def submap(e, reps, k=16, n_src=64, seed=5):
    rng = np.random.default_rng(seed)
    poses = synth.loop_trajectory(n_src + k, step=0.04)
    scans = synth.scans_from_poses(poses, 1024, rng)
    targets, inits, pairs = [], [], []
    for i in range(n_src):
        M0inv = np.linalg.inv(synth.pose_to_mat(poses[i]))
        parts = [scans[j] @ (M0inv @ synth.pose_to_mat(poses[j]))[:2, :2].T + (M0inv @ synth.pose_to_mat(poses[j]))[:2, 2]
                 for j in range(i, i + k)]
        targets.append(np.ascontiguousarray(np.concatenate(parts)))
        inits.append(M0inv @ synth.pose_to_mat(poses[i + k]))
        pairs.append((i + k, len(scans) + i))
    table = scans + targets
    d = Dev(e, table, np.array(pairs, dtype=np.int32), np.array(inits))
    t = d.time(reps)
    d1 = Dev(e, table, np.array(pairs[:1], dtype=np.int32), np.array(inits[:1]))
    t1 = d1.time(reps)
    return {"source_points": 1024, "target_points_mean": float(np.mean([len(x) for x in targets])),
            "pairs": n_src, "batch_ms": t * 1e3, "pairs_per_s": n_src / t, "one_pair_ms": t1 * 1e3}


def mixed(e, reps, seed=7):
    scans, pairs, init, _, _ = synth.make_chain_workload(2001, 1024, seed=seed)
    long_scan = synth.make_chain_workload(2, 20000, seed=seed + 1)[0][0]
    mixed_scans = scans + [long_scan]
    out = {"pairs": len(pairs), "long_scan_points": len(long_scan)}
    rows = {"plain_host": [], "mixed_host": [], "plain_device": [], "mixed_device": []}
    for _ in range(reps):                                    # alternated
        for name, tab in (("plain", scans), ("mixed", mixed_scans)):
            e.set_scans(tab)
            e.run(pairs, init, epsilon=EPS)
            t0 = time.perf_counter()
            r = e.run(pairs, init, epsilon=EPS)
            rows[name + "_host"].append(time.perf_counter() - t0)
            if name == "plain":
                ref = r
            else:
                assert np.array_equal(r.T, ref.T) and np.array_equal(r.iters, ref.iters)
            d = Dev(e, tab, pairs, init)
            rows[name + "_device"].append(d.time(3))
    for k, v in rows.items():
        out[k + "_ms"] = {"median": float(np.median(v)) * 1e3, "all": [x * 1e3 for x in v]}
    out["note"] = ("host = IcpEngine.run (icpb_run_host: pairs split by length, the short ones on the shared-memory "
                   "kernel, per-pair staging on the mixed table); device = run_device (pairs not seen by the host: "
                   "every pair on the large variant when the table's longest scan does not fit)")
    return out


def global_cost(e, reps, seed=9):
    out = {}
    for beams, n in ((1024, 5000), (4096, 1000)):
        scans, pairs, init, _, _ = synth.make_chain_workload(n, beams, seed=seed)
        d = Dev(e, scans, pairs, init)
        ts = {"default": [], "large": []}
        for _ in range(reps):
            for name, v in (("default", -1), ("large", 1)):
                e.set_tuning("large", v)
                ts[name].append(d.time(5))
        e.set_tuning("large", -1)
        out[str(beams)] = {"pairs": d.B, "default_ms": float(np.median(ts["default"])) * 1e3,
                           "large_ms": float(np.median(ts["large"])) * 1e3,
                           "ratio": float(np.median(ts["large"]) / np.median(ts["default"])),
                           "all_default_ms": [x * 1e3 for x in ts["default"]], "all_large_ms": [x * 1e3 for x in ts["large"]]}
    return out


def c_port(n_pairs=4, seed=161):
    scans, pairs, init, _, _ = synth.make_chain_workload(n_pairs + 1, 16384, seed=seed)
    xy, off = c_oracle.pack(scans)
    t0 = time.perf_counter()
    _, _, passes = c_oracle.icp_batch(xy, off, pairs, init, epsilon=EPS)
    t = time.perf_counter() - t0
    return {"beams": 16384, "pairs": n_pairs, "threads": c_oracle.max_threads(), "seconds": t,
            "pairs_per_s": n_pairs / t, "passes": passes.tolist()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="large_scan_bench.json", help="where the JSON document goes")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "no CUDA device: this tool measures the GPU"
    c_oracle.build()
    e = gicp.IcpEngine()
    res = {"gpu": gpu_info()}
    e.set_scans(synth.make_chain_workload(2, 1024, seed=1)[0])
    peak = pde_peak(e)
    res["pde_peak_tpde_s"] = peak * 1e-12
    res["chains"] = [chain_entry(e, 16384, 33, args.reps, peak, 1),
                     chain_entry(e, 32768, 17, args.reps, peak, 2),
                     chain_entry(e, 65536, 9, args.reps, peak, 3)]
    res["latency"] = {"16k": latency(e, 16384, 4, args.reps), "65k": latency(e, 65536, 5, args.reps)}
    res["submap"] = submap(e, args.reps)
    res["mixed"] = mixed(e, args.reps)
    res["global_cost"] = global_cost(e, args.reps)
    res["c_port"] = c_port()
    res["gpu_after"] = gpu_info()
    e.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
