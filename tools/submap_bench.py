"""Submaps built on the device (IcpEngine.set_submaps) against building them on the host (merge_scans plus
set_scans of the combined table), on one GPU, in one run.  Prints one JSON document and writes it to --out.

Resident table: 5,000 x 1,024-beam scans along the synthetic loop.  Submap sets: windows of 4 and 8 scans
either side, around every 5th scan and around every scan (the members placed by the truth poses).
Per set:
  merge_kernel_ms   device time of submap_merge_kernel per set_submaps call (torch.profiler, a profiling pass of
                    its own), the check pass and the write pass separately
  hbm_fraction      bytes the merge must move (check: 16 B read per point; write: 16 B read + 16 B written) over
                    the kernel time, against 7.7 TB/s (the data-sheet HBM3e bandwidth): the merge is bound by
                    bytes, it does 4 multiplies and 4 adds per 32 bytes
  set_submaps_ms    host-to-host time of one set_submaps call (median over --reps)
  host_way_ms       merge_scans on the host plus set_scans of base + submaps (median over --host-reps)
  first_run_ms      one alignment batch (a source scan onto every submap) right after set_submaps, which also
                    builds the table's staging images when the longest submap fits shared memory; steady_run_ms
                    the same batch again (median)
Quality, on a 2,000-pose loop of 360-beam scans with truth poses: proximity_loop_closures with submap_window
None, 0, 4 and 8, without and with heading_starts(8) -- the number of accepted constraints and their
translation and heading errors against the truth.

With --voxels v1 v2 ... the document is the voxel filter's instead (set_submaps(voxel=)): the same four sets,
each without a filter and with every voxel, on a fresh handle per row.  Per row:
  merged_points, kept_points, longest_merged, longest_submap (kept)
  fits_shared_memory  a batch of the set's pairs plus one scan-to-scan pair runs in one launch (the submaps fit
                      shared memory and the table has staging images) rather than two (split by scan length)
  kernel_ms           device time per set_submaps call of every kernel it launches, by name (torch.profiler, a
                      profiling pass of its own): the merge (check pass, then the write into scratch when
                      filtering), insert, keep, the CUB scan (init + scan), bounds, scatter
  set_submaps_ms      host to host (median over --reps)
  device_bytes_added  device memory the first set_submaps call on the fresh handle took (cudaMemGetInfo before and
                      after): the submap part of the table plus the handle's scratch arena at its peak
  first_run_ms, steady_run_ms   as above
  identical_to_host_way  the table (read back with read_scans) and the alignments equal those of merge_scans(voxel=)
                      followed by set_scans of base + submaps, bit for bit
Quality: proximity_loop_closures from the identity with submap_window 4 and 8, without a filter and with every voxel.

Run:  python tools/submap_bench.py --out submap_bench.json
      python tools/submap_bench.py --voxels 0.01 0.02 0.05 --out submap_voxel_bench.json
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

from icp_slam_b200 import callers, icp as gicp, synth  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
SEED = 20261022


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    name, power, clk = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clk, "torch_name": torch.cuda.get_device_name()}


def merge_kernel_ms(fn, reps):
    """Device time per call of the merge kernel's two launches (check, write), from a torch.profiler trace."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    launches = sorted((ev for ev in prof.events() if "submap_merge_kernel" in ev.name and ev.device_type == DeviceType.CUDA),
                      key=lambda ev: ev.time_range.start)
    # every call launches the check pass, then the write pass
    us = [ev.time_range.elapsed_us() / 1e3 for ev in launches]
    return {"check": float(np.median(us[0::2])), "write": float(np.median(us[1::2])), "launches": len(us)}


def run_set(e, base, poses, w, every, reps, host_reps):
    n = len(base)
    targets = np.arange(0, n, every)
    members = callers.submap_window_members(n, targets, w)
    transforms = callers.submap_window_transforms(poses, targets, members)
    n_pts = int(sum(sum(len(base[s]) for s in m) for m in members))
    e.set_scans(gicp.ScanTable(base))
    ids = e.set_submaps(members, transforms)                                  # warm-up, allocation
    src = np.minimum(targets + w + 1, n - 1)
    pairs = np.stack((src, ids), axis=1).astype(np.int32)
    dev = []
    for _ in range(reps):
        t0 = time.perf_counter()
        e.set_submaps(members, transforms)
        dev.append((time.perf_counter() - t0) * 1e3)
    t0 = time.perf_counter()
    first = e.run(pairs, epsilon=0.05)
    first_ms = (time.perf_counter() - t0) * 1e3
    steady = []
    for _ in range(3):
        t0 = time.perf_counter()
        e.run(pairs, epsilon=0.05)
        steady.append((time.perf_counter() - t0) * 1e3)
    kern = merge_kernel_ms(lambda: e.set_submaps(members, transforms), 3)
    # the host way: same submaps in numpy, the whole combined table uploaded
    host = []
    h = gicp.IcpEngine(0)
    try:
        for _ in range(host_reps):
            t0 = time.perf_counter()
            merged = gicp.merge_scans(base, members, transforms)
            h.set_scans(gicp.ScanTable(list(base) + merged))
            host.append((time.perf_counter() - t0) * 1e3)
        ref = h.run(np.stack((src, np.arange(n, n + len(targets))), axis=1).astype(np.int32), epsilon=0.05)
        same = bool(np.array_equal(ref.T, first.T) and np.array_equal(ref.error, first.error)
                    and np.array_equal(ref.iters, first.iters))
        del merged
    finally:
        h.close()
    e.set_submaps([], [])
    check_b, write_b = 16 * n_pts, 32 * n_pts
    return {"window": w, "every": every, "submaps": len(targets), "members": int(sum(len(m) for m in members)),
            "points": n_pts, "longest_submap": int(max(sum(len(base[s]) for s in m) for m in members)),
            "alignments_identical_to_host_way": same,
            "merge_kernel_ms": kern,
            "hbm_fraction": {"check": check_b / (kern["check"] * 1e-3) / HBM_BYTES_PER_S,
                             "write": write_b / (kern["write"] * 1e-3) / HBM_BYTES_PER_S},
            "merge_bytes": {"check": check_b, "write": write_b},
            "set_submaps_ms": {"median": float(np.median(dev)), "samples": dev},
            "host_way_ms": {"median": float(np.median(host)), "samples": host},
            "first_run_ms": first_ms, "steady_run_ms": float(np.median(steady)), "run_pairs": len(pairs)}


def kernel_ms(fn, reps):
    """Device time per call of every kernel ``fn`` launches, summed by kernel name (torch.profiler), median of reps."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    per_call = []
    for _ in range(reps):
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        t = {}
        for ev in prof.events():
            if ev.device_type == DeviceType.CUDA and "kernel" in ev.name.lower():
                name = next((k for k in ("submap_merge_kernel", "submap_voxel_insert_kernel", "submap_voxel_keep_kernel",
                                         "DeviceScanInitKernel", "DeviceScanKernel", "submap_voxel_bounds_kernel",
                                         "submap_voxel_scatter_kernel") if k in ev.name), ev.name)
                t[name] = t.get(name, 0.0) + ev.time_range.elapsed_us() / 1e3
        per_call.append(t)
    return {k: float(np.median([t.get(k, 0.0) for t in per_call])) for k in per_call[0]}


def run_voxel_set(base, poses, w, every, voxel, reps):
    import torch
    n = len(base)
    targets = np.arange(0, n, every)
    members = callers.submap_window_members(n, targets, w)
    transforms = callers.submap_window_transforms(poses, targets, members)
    merged = [int(sum(len(base[s]) for s in m)) for m in members]
    src = np.minimum(targets + w + 1, n - 1)
    e = gicp.IcpEngine(0)
    try:
        e.set_scans(gicp.ScanTable(base))
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        ids = e.set_submaps(members, transforms, voxel=voxel)
        added = free0 - torch.cuda.mem_get_info()[0]
        kept = e.table.lengths[n:]
        pairs = np.stack((src, ids), axis=1).astype(np.int32)
        dev = []
        for _ in range(reps):
            t0 = time.perf_counter()
            e.set_submaps(members, transforms, voxel=voxel)
            dev.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        first = e.run(pairs, epsilon=0.05)
        first_ms = (time.perf_counter() - t0) * 1e3
        steady = []
        for _ in range(3):
            t0 = time.perf_counter()
            e.run(pairs, epsilon=0.05)
            steady.append((time.perf_counter() - t0) * 1e3)
        n0 = e.launch_count
        e.run(np.concatenate((pairs[:64], [(1, 0)])).astype(np.int32), epsilon=0.05)
        fits = e.launch_count - n0 == 1
        table = e.read_scans(ids)
        kern = kernel_ms(lambda: e.set_submaps(members, transforms, voxel=voxel), 3)
    finally:
        e.close()
    h = gicp.IcpEngine(0)
    try:
        t0 = time.perf_counter()
        host = gicp.merge_scans(base, members, transforms, voxel=voxel)
        h.set_scans(gicp.ScanTable(list(base) + host))
        host_ms = (time.perf_counter() - t0) * 1e3
        ref = h.run(np.stack((src, np.arange(n, n + len(targets))), axis=1).astype(np.int32), epsilon=0.05)
        same = bool(all(a.tobytes() == b.tobytes() for a, b in zip(table, host)) and len(table) == len(host)
                    and np.array_equal(ref.T, first.T) and np.array_equal(ref.error, first.error)
                    and np.array_equal(ref.iters, first.iters))
        del host
    finally:
        h.close()
    return {"window": w, "every": every, "voxel": voxel, "submaps": len(targets),
            "merged_points": int(sum(merged)), "kept_points": int(kept.sum()),
            "longest_merged": max(merged), "longest_submap": int(kept.max()), "fits_shared_memory": fits,
            "identical_to_host_way": same, "kernel_ms": kern,
            "set_submaps_ms": {"median": float(np.median(dev)), "samples": dev},
            "host_way_ms": host_ms, "device_bytes_added": int(added),
            "first_run_ms": first_ms, "steady_run_ms": float(np.median(steady)), "run_pairs": len(pairs)}


def voxel_quality(n_poses, voxels):
    rng = np.random.default_rng(SEED)
    poses = synth.loop_trajectory(n_poses, step=0.2)
    scans = synth.scans_from_poses(poses, 360, rng, drop_frac=0.03)
    M = callers.poses_to_mats(poses)
    out = {"poses": n_poses, "beams": 360, "candidates": int(len(callers.proximity_candidates(poses)))}
    for w in (4, 8):
        for v in [None] + list(voxels):
            got, _ = callers.proximity_loop_closures(poses, scans, submap_window=w, submap_voxel=v)
            dt = [float(np.hypot(*(T[:2, 2] - (np.linalg.inv(M[i]) @ M[j])[:2, 2]))) for i, j, T in got]
            dth = [float(abs((np.arctan2(T[1, 0], T[0, 0]) - (poses[j, 2] - poses[i, 2]) + np.pi) % (2 * np.pi)
                             - np.pi)) for i, j, T in got]
            out[f"window_{w}/voxel_{v}"] = {
                "accepted": len(got),
                "dt_m": {"median": float(np.median(dt)) if dt else None, "max": max(dt) if dt else None},
                "dtheta_rad": {"median": float(np.median(dth)) if dth else None, "max": max(dth) if dth else None}}
    return out


def quality(n_poses):
    rng = np.random.default_rng(SEED)
    poses = synth.loop_trajectory(n_poses, step=0.2)
    scans = synth.scans_from_poses(poses, 360, rng, drop_frac=0.03)
    M = callers.poses_to_mats(poses)
    out = {"poses": n_poses, "beams": 360, "candidates": int(len(callers.proximity_candidates(poses)))}
    for starts_name, starts in (("identity", None), ("heading_starts_8", gicp.heading_starts(8))):
        for w in (None, 0, 4, 8):
            got, _ = callers.proximity_loop_closures(poses, scans, starts=starts, submap_window=w)
            dt = [float(np.hypot(*(T[:2, 2] - (np.linalg.inv(M[i]) @ M[j])[:2, 2]))) for i, j, T in got]
            dth = [float(abs((np.arctan2(T[1, 0], T[0, 0]) - (poses[j, 2] - poses[i, 2]) + np.pi) % (2 * np.pi)
                             - np.pi)) for i, j, T in got]
            out[f"{starts_name}/window_{w}"] = {
                "accepted": len(got),
                "dt_m": {"median": float(np.median(dt)) if dt else None, "max": max(dt) if dt else None},
                "dtheta_rad": {"median": float(np.median(dth)) if dth else None, "max": max(dth) if dth else None}}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--scans", type=int, default=5000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=2)
    ap.add_argument("--quality-poses", type=int, default=2000)
    ap.add_argument("--voxels", type=float, nargs="*", default=None,
                    help="voxel filter cell sizes (m): write the voxel filter's document instead")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rng = np.random.default_rng(SEED)
    poses = synth.loop_trajectory(a.scans, step=0.04)
    base = synth.scans_from_poses(poses, 1024, rng, drop_frac=0.03)
    if a.voxels is not None:
        doc = {"gpu": gpu_info(), "scans": a.scans, "beams": 1024, "reps": a.reps, "voxels": a.voxels, "sets": []}
        for w in (4, 8):
            for every in (5, 1):
                for v in [None] + a.voxels:
                    doc["sets"].append(run_voxel_set(base, poses, w, every, v, a.reps))
                    print(json.dumps(doc["sets"][-1]), flush=True)
        doc["quality"] = voxel_quality(a.quality_poses, a.voxels)
        doc["gpu_after"] = gpu_info()
        text = json.dumps(doc, indent=1)
        print(text)
        if a.out:
            with open(a.out, "w") as f:
                f.write(text + "\n")
        return
    doc = {"gpu": gpu_info(), "scans": a.scans, "beams": 1024, "reps": a.reps, "host_reps": a.host_reps, "sets": []}
    e = gicp.IcpEngine(0)
    try:
        for w in (4, 8):
            for every in (5, 1):
                doc["sets"].append(run_set(e, base, poses, w, every, a.reps, a.host_reps))
                print(json.dumps(doc["sets"][-1]), flush=True)
    finally:
        e.close()
    doc["quality"] = quality(a.quality_poses)
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
