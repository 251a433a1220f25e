#!/usr/bin/env python
"""Benchmark of the batched ICP hot path: ICP scan-pair alignments / second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workloads (BASELINE.json configs; `--workload`):
  chain      configs[1], the headline: the full odometry ICP chain over a 5,000-scan synthetic indoor
             trajectory, 1,024-beam scans, pairs (i, i-1) with the odometry initial guess, epsilon 0.05,
             max_iters 100 (reference scripts/main.py:240-247).  One step = one pass of the hot path
             over the whole 4,999-pair batch.  With N GPUs every rank aligns its OWN chain: weak scaling.
  proximity  configs[2]: every pair of the trajectory within 1 m and at least 2 m along the path
             (~100,000 pairs, identity initial guess).  ONE pair list, sharded over the ranks in
             interleaved blocks against a replicated scan table: strong scaling.
  allpairs   configs[3] in miniature (--scans 600 by default): every pair i<j, decoded on the device
             from a linear index, interleaved blocks per rank: strong scaling.
  highres    configs[4]: 4,096-beam scans, 32 initial headings per pair.
On every multi-GPU run the exchange of the constraint records is fused into the alignment kernel: its
epilogue stores each finished pair's 64-byte record into every rank's gather buffer over NVLink peer
memory (icp_slam_b200.dist.FusedGather); one symmetric-memory barrier follows, no collective.

`value`     device-timed: scan table, pairs and initial guesses already resident in HBM.
`e2e`       the same step through the public host API, IcpEngine.align, fed what the reference feeds
            its fan-out: `lidar_points`, a Python list of separate pageable (m_i, 2) float64 arrays
            (reference src/dataloader.py:110-112), plus the pair list and (B, 3, 3) initial guesses in
            host memory; results (and, on N GPUs, every rank's gathered records) back in host memory.
`roofline`  FP32-pipe view of the timed kernel: `frac` is the share of the pipe's lane-slots the
            kernel actually used (executed distance evaluations x 4 slots); the algorithmic speed-up
            of the pruning and the exhaustive variant (the one the pipe roofline bounds) sit beside it.
`cpu_baseline` the C port of the reference algorithm (oracle/icp_oracle.c) on all host cores, and the
            unmodified numpy reference under joblib when it can be imported on this machine.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "icp_scan_pair_alignments_per_sec"
UNIT = "pairs/s"
SEED = 467002
EPS, MAX_ITERS = 0.05, 100
DUMP_BYTES = 64_000_000                                      # cap on what --dump-outputs writes
# counters of the timed kernel from a committed `ncu --set full` capture of this same command
# (written by tools/ncu_summary.py; carries the commit it was taken at)
NCU_SUMMARY = os.path.join(ROOT, "profiles", "r02_align_ncu_summary.json")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="chain", choices=["chain", "proximity", "allpairs", "highres"])
    ap.add_argument("--scans", type=int, default=0, help="scans of the trajectory (default: per workload)")
    ap.add_argument("--beams", type=int, default=0, help="beams per scan (default: per workload)")
    ap.add_argument("--pairs", type=int, default=0, help="cap on the pair count of the non-chain workloads")
    ap.add_argument("--block", type=int, default=256, help="interleaved block of the strong-scaling partition")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target wall time of the CPU sample")
    ap.add_argument("--exhaustive", action="store_true", help="run the timed steps with pruning off (profiling)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the e2e leg (profiling runs)")
    ap.add_argument("--no-sustained", action="store_true", help="skip the sustained-clock segment")
    ap.add_argument("--no-exhaustive", action="store_true", help="skip the pruning-off launches (long workloads)")
    ap.add_argument("--threads", type=int, default=0, help="tuning: cap on the CTA width (icpb_set_tuning)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    dflt = {"chain": (5000, 1024), "proximity": (5000, 1024), "allpairs": (600, 1024), "highres": (48, 4096)}
    args.scans = args.scans or dflt[args.workload][0]
    args.beams = args.beams or dflt[args.workload][1]
    args.strong = args.workload in ("proximity", "allpairs")
    return args


def config_of(args, world):
    """The workload description both arms print (same function, same strings)."""
    name = {"chain": f"odometry ICP chain, {args.scans} scans x {args.beams} beams, pairs (i, i-1), odometry "
                     f"initial guess (BASELINE configs[1]); every GPU its own chain",
            "proximity": f"proximity loop-closure candidates of a {args.scans}-scan x {args.beams}-beam trajectory, "
                         f"identity initial guess (BASELINE configs[2]); one pair list sharded over the GPUs",
            "allpairs": f"all pairs i<j of {args.scans} scans x {args.beams} beams, identity initial guess "
                        f"(BASELINE configs[3]); one index space sharded over the GPUs",
            "highres": f"32-start heading sweep, {args.scans} scans x {args.beams} beams (BASELINE configs[4])"}
    return {"workload": name[args.workload], "scans": args.scans, "beams": args.beams,
            "epsilon": EPS, "max_iters": MAX_ITERS, "n_gpus": world,
            "l2": "GPU arm: L2 flushed between timed steps (768 MB fill, outside the timed events)"}


def workload(args, rank, world):
    """Synthetic scans + pair list + initial guesses.  `chain`/`highres`: every rank its own stretch of
    the trajectory (weak scaling); `proximity`/`allpairs`: the same table and pair list on every rank."""
    from icp_slam_b200 import synth
    own = 0 if args.strong else rank
    rng_seed = SEED + 1000 * own
    rng = np.random.default_rng(rng_seed)
    phase = own / max(world, 1)
    if args.workload == "chain":            # configs[1]: scripts/main.py:239-247
        poses = synth.loop_trajectory(args.scans, step=0.04, start_phase=phase)
        scans = synth.scans_from_poses(poses, args.beams, rng, drop_frac=0.03)
        odo = synth.odometry_from_truth(poses, rng)
        idx = np.arange(1, args.scans)
        pairs = np.stack((idx, idx - 1), axis=1).astype(np.int32)
        init = np.stack([synth.pose_to_mat(odo[i] - odo[i - 1]) for i in idx])
    elif args.workload == "proximity":      # configs[2]: all pairs within 1 m, >= 2 m along the path
        poses = synth.loop_trajectory(args.scans, step=0.04, start_phase=phase)
        scans = synth.scans_from_poses(poses, args.beams, rng, drop_frac=0.03)
        pairs = synth.proximity_pairs(poses, max_pairs=args.pairs or 100000, seed=rng_seed)
        init = None
    elif args.workload == "allpairs":       # configs[3]: exhaustive i<j, source j onto target i
        poses = synth.loop_trajectory(args.scans, step=180.0 / args.scans, start_phase=phase)
        scans = synth.scans_from_poses(poses, args.beams, rng, drop_frac=0.03)
        ij = synth.all_pairs_decode(np.arange(synth.all_pairs_count(args.scans)), args.scans)
        pairs = np.stack((ij[:, 1], ij[:, 0]), axis=1).astype(np.int32)
        init = None
    else:                                   # configs[4]: high-resolution scans, multi-start heading sweep
        k_starts = 32
        poses = synth.loop_trajectory(args.scans, step=0.04, start_phase=phase)
        scans = synth.scans_from_poses(poses, args.beams, rng, drop_frac=0.03)
        idx = np.repeat(np.arange(1, args.scans), k_starts)
        pairs = np.stack((idx, idx - 1), axis=1).astype(np.int32)
        th = np.tile(-np.pi + 2 * np.pi * np.arange(k_starts) / k_starts, args.scans - 1)
        init = np.stack([synth.pose_to_mat((0.0, 0.0, t)) for t in th])
    return scans, pairs, init


class ClockSampler:
    """SM clock and throttle reasons polled through NVML every ~2 ms during the timed region (the timed
    region of the headline workload is tens of milliseconds: nvidia-smi's 100 ms loop sees two samples)."""

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.t = index, [], False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:                                    # noqa: BLE001
            self.nv = None

    def _loop(self):
        nv, h = self.nv, self.h
        while not self.stop_flag:
            try:
                self.rows.append((time.time(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)))
            except Exception:                                # noqa: BLE001
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()

    def window(self, t0, t1):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"]}
        nv = self.nv
        names = (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown),
                 ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown),
                 ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap))
        sm, reasons = [], set()
        for ts, mhz, bits in list(self.rows):
            if t0 <= ts <= t1:
                sm.append(mhz)
                reasons |= {n for n, b in names if bits & b}
        mx = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": mx, "reasons": ["no samples in the timed region"]}
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(min(sm)), "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        self.stop_flag = True


_ALL_CPUS = None


def bind_to_gpu_numa_node(index):
    """One process per GPU: run this rank's host threads on the CPUs next to its GPU, so the pinned
    staging buffers (first touch) and the copy-engine reads stay on the local memory controller and
    PCIe root.  Returns a short description for the JSON line; never fatal."""
    global _ALL_CPUS
    try:
        _ALL_CPUS = os.sched_getaffinity(0)
        import pynvml
        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        cpus = sorted(os.sched_getaffinity(0))
        return f"{len(cpus)} cpus ({cpus[0]}-{cpus[-1]})"
    except Exception as exc:                                  # noqa: BLE001
        return f"unbound ({type(exc).__name__})"


def identity_init(n):
    return np.broadcast_to(np.eye(3), (n, 3, 3)).copy()


def dump_outputs(out_dir, rows, T6, err, passes):
    """--dump-outputs: what the last timed step returned, one float64 .npy per array: T (n, 6), the top
    two rows of each 3x3 transform; error (n,); passes (n,); rows (n,), each row's index in the step's
    problem list.  The inputs are seeded, so two builds run with the same arguments can be compared file
    by file.  Past 64 MB, a seeded sample of the rows (the same rows on every run)."""
    rows = np.asarray(rows)
    keep = (DUMP_BYTES - 4096) // (9 * 8)                     # 9 float64 per row; 4096: the .npy headers
    sel = np.arange(len(rows))
    if len(rows) > keep:
        sel = np.sort(np.random.default_rng(SEED).choice(len(rows), keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("T", T6), ("error", err), ("passes", passes), ("rows", rows)):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(np.asarray(a)[sel], dtype=np.float64))


def cpu_port_rate(scans, pairs, init, seconds, threads=0, all_pairs=False):
    """Time the C port of the reference algorithm on a bounded sample of the same workload."""
    from oracle import c_oracle
    c_oracle.build()
    nthr = threads or c_oracle.max_threads()
    xy, off = c_oracle.pack(scans)
    init = identity_init(len(pairs)) if init is None else init
    rng = np.random.default_rng(SEED)
    order = np.arange(len(pairs)) if all_pairs else rng.permutation(len(pairs))
    probe = order[:max(2 * nthr, 8)]
    t = time.perf_counter()
    c_oracle.icp_batch(xy, off, pairs[probe], init[probe], epsilon=EPS, max_iters=MAX_ITERS, n_threads=nthr)
    dt = time.perf_counter() - t
    n = len(pairs) if all_pairs else int(min(len(pairs), max(len(probe), len(probe) * seconds / max(dt, 1e-3))))
    sel = order[:n]
    t = time.perf_counter()
    _, _, passes = c_oracle.icp_batch(xy, off, pairs[sel], init[sel], epsilon=EPS, max_iters=MAX_ITERS, n_threads=nthr)
    dt = time.perf_counter() - t
    return n / dt, nthr, n, dt, float(passes.mean())


def numpy_reference_rate(scans, pairs, init, seconds):
    """The UNMODIFIED reference -- src.icp.icp under joblib.Parallel(n_jobs=-1, backend="loky"), exactly
    the expression of reference scripts/main.py:240-247 -- when its source tree can be imported on this
    machine (baseline/_ref or /root/reference; it is not shipped with this repository, so on a GPU box
    this leg normally reports why it did not run)."""
    for root in (os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if os.path.exists(os.path.join(root, "src", "icp.py")):
            break
    else:
        return {"unavailable": "reference source tree not present on this machine (pure Python, not shipped)"}
    try:
        sys.path.insert(0, root)
        from joblib import Parallel, delayed
        from src import icp as ref_icp                       # the reference's own module, unmodified
        ncpu = os.cpu_count() or 1
        init = identity_init(len(pairs)) if init is None else init
        rng = np.random.default_rng(SEED)
        sel = rng.permutation(len(pairs))[:max(2 * ncpu, 8)]
        hom = lambda s: np.c_[s, np.ones(len(s))]            # noqa: E731  (scripts/main.py:242-243)

        def go(idx):
            with Parallel(n_jobs=-1, backend="loky") as par:
                t = time.perf_counter()
                par(delayed(ref_icp.icp)(hom(scans[pairs[b, 0]]), hom(scans[pairs[b, 1]]), init[b].copy(),
                                         max_iters=MAX_ITERS, epsilon=EPS) for b in idx)
                return time.perf_counter() - t
        dt = go(sel)                                          # includes the worker start-up
        n = int(min(len(pairs), max(len(sel), len(sel) * seconds / max(dt, 1e-3))))
        sel = rng.permutation(len(pairs))[:n]
        dt = go(sel)
        return {"value": n / dt, "unit": UNIT, "cores": ncpu, "kind": "reference",
                "sample": f"{n} pairs (seeded random subsample) in {dt:.1f} s, unmodified src.icp.icp under "
                          f"joblib.Parallel(n_jobs=-1, backend='loky') from {root}"}
    except Exception as exc:                                  # noqa: BLE001
        return {"unavailable": f"{type(exc).__name__}: {exc}"}
    finally:
        if sys.path and sys.path[0] == root:
            sys.path.pop(0)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores.  The
    reference is pure Python and does not travel to the GPU box, so this times its C port
    (oracle/icp_oracle.c, the one place besides cpu_baseline where bench.py executes oracle/) with all
    host threads; a step is one pass over the whole pair list of the chain (4,999 pairs), a seeded
    subsample sized for a few minutes in total for the larger workloads."""
    if rank != 0:
        return
    scans, pairs, init = workload(args, 0, world)
    from oracle import c_oracle
    c_oracle.build()
    nthr = c_oracle.max_threads()
    xy, off = c_oracle.pack(scans)
    init = identity_init(len(pairs)) if init is None else init
    rng = np.random.default_rng(SEED)
    order = rng.permutation(len(pairs))
    probe = order[:max(2 * nthr, 8)]
    t = time.perf_counter()
    c_oracle.icp_batch(xy, off, pairs[probe], init[probe], epsilon=EPS, max_iters=MAX_ITERS, n_threads=nthr)
    dt = time.perf_counter() - t
    budget = 240.0 / max(args.steps + args.warmup, 1)
    n = int(min(len(pairs), max(len(probe), len(probe) * budget / max(dt, 1e-3))))
    if args.workload == "chain" and len(pairs) * dt / len(probe) * (args.steps + args.warmup) < 900.0:
        n = len(pairs)                                        # the whole batch per step, like the GPU arm
    sel = np.arange(len(pairs)) if n == len(pairs) else order[:n]
    for _ in range(args.warmup):
        c_oracle.icp_batch(xy, off, pairs[sel], init[sel], epsilon=EPS, max_iters=MAX_ITERS, n_threads=nthr)
    t = time.perf_counter()
    for _ in range(args.steps):
        T, err, passes = c_oracle.icp_batch(xy, off, pairs[sel], init[sel], epsilon=EPS, max_iters=MAX_ITERS,
                                            n_threads=nthr)
    dt = time.perf_counter() - t
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, sel, c_oracle.to6(T), err, passes)
    rate = n * args.steps / dt
    sample = (f"{n} of {len(pairs)} pairs per step" + ("" if n == len(pairs) else ", seeded random subsample") +
              f", C port oracle/icp_oracle.c on {nthr} threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_of(args, world),
        "details": {"pairs_per_step": n},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": nthr, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    sys.dont_write_bytecode = True                           # the tree may be read-only: no __pycache__ in it
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from icp_slam_b200 import icp as gicp
    from icp_slam_b200 import dist as gdist

    numa = bind_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # NCCL prints its version banner on stdout at communicator creation; keep stdout for the one
    # JSON line by pointing fd 1 at stderr until the result is printed
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    scans, pairs, init = workload(args, rank, world)
    n_total = len(pairs)                                     # problems of this rank's index space
    # ---- partition: weak = everything this rank generated; strong = interleaved blocks of one list ----
    if args.strong and world > 1:
        mine = gdist.shard_indices(n_total, rank, world, args.block)
    else:
        mine = np.arange(n_total)
    B = len(mine)
    pairs_mine = np.ascontiguousarray(pairs[mine])
    init_mine = None if init is None else np.ascontiguousarray(init[mine])
    eng = gicp.IcpEngine(local)
    if args.threads:
        eng.set_tuning("threads", args.threads)
    table = gicp.ScanTable(scans)
    lens = table.lengths
    xy_t, off_t = torch.from_numpy(table.xy).to(dev), torch.from_numpy(table.offsets).to(dev)
    pairs_t = torch.from_numpy(pairs_mine).to(dev)
    init_t = None if init_mine is None else torch.from_numpy(np.ascontiguousarray(init_mine[:, :2, :].reshape(B, 6))).to(dev)
    eng.set_scans_device(xy_t, off_t, table)
    out_T = torch.empty((B, 6), dtype=torch.float64, device=dev)
    out_err = torch.empty(B, dtype=torch.float64, device=dev)
    out_pass = torch.empty(B, dtype=torch.int32, device=dev)
    # the all-pairs index space is decoded on the device: no pair list in HBM at all
    all_pairs_dev = None
    if args.workload == "allpairs":
        all_pairs_dev = gdist.shard_all_pairs(n_total, rank, world, args.block) if world > 1 else (0, n_total, 0, n_total)
    # ---- the exchange step: records of ALL ranks in every rank's buffer, written by the kernels ----
    gather, ep = None, None
    n_global = n_total if args.strong else world * n_total
    if world > 1:
        if args.strong:
            gather = gdist.FusedGather(n_global, device=dev, block=args.block)
            ep = gather.epilogue()
        else:                                                # rank r owns rows r*B .. (r+1)*B - 1
            gather = gdist.FusedGather(n_global, device=dev, block=n_total)
            ep = gather.epilogue()
    flush = torch.empty(192 * 1024 * 1024, dtype=torch.float32, device=dev)     # 768 MB > 126 MB L2

    def launch(exhaustive=False):
        if exhaustive:
            eng.run_device(None if all_pairs_dev else pairs_t, init_t, out_T, out_err, out_pass, epsilon=EPS,
                           max_iters=MAX_ITERS, all_pairs=all_pairs_dev, exhaustive=True)
        else:
            eng.run_device_ex(pairs_t, init_t, out_T, out_err, out_pass, ep, epsilon=EPS, max_iters=MAX_ITERS,
                              all_pairs=all_pairs_dev)

    def step_device():
        launch(args.exhaustive)
        if gather is not None:
            gather.barrier()                                  # every rank's records have landed everywhere

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
    barrier()
    # ---- multi-GPU correctness, outside every timed region: zeroed buffers, one step, and every block
    # of the fused gather compared with an NCCL all_gather of the same records ----
    gather_check = None
    if gather is not None:
        gather.clear()
        step_device()
        torch.cuda.synchronize()
        rec = torch.empty((B, 8), dtype=torch.float64, device=dev)
        rec[:, :6], rec[:, 6], rec[:, 7] = out_T, out_err, out_pass.to(torch.float64)
        counts = [len(gdist.shard_indices(n_global, r, world, gather.block)) for r in range(world)]
        cap = max(counts)
        send = torch.zeros((cap, 8), dtype=torch.float64, device=dev)
        send[:B] = rec
        recv = torch.empty((world * cap, 8), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(recv, send)
        want = torch.empty((n_global, 8), dtype=torch.float64, device=dev)
        for r in range(world):
            idx = torch.from_numpy(gdist.shard_indices(n_global, r, world, gather.block)).to(dev)
            want[idx] = recv[r * cap:r * cap + counts[r]]
        same = bool(torch.equal(gather.records(), want))
        assert same, f"rank {rank}: the fused gather differs from the NCCL all_gather of the same records"
        gather_check = f"fused gather == NCCL all_gather on all {n_global} rows of every rank (buffers zeroed first)"
        barrier()

    launches0 = eng.launch_count
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.time()
    for k in range(args.steps):
        flush.fill_(float(k))                   # evict L2 between timed iterations (outside the events)
        if world > 1:
            dist.barrier()
        ev[k][0].record()
        step_device()
        ev[k][1].record()
    barrier()
    t_wall1 = time.time()
    if args.dump_outputs and rank == 0:                      # before any later launch rewrites the outputs
        if gather is not None and not args.exhaustive:        # every rank's records, as every rank holds them
            rec = gather.records().cpu().numpy()
            dump_outputs(args.dump_outputs, np.arange(n_global), rec[:, :6], rec[:, 6], rec[:, 7])
        else:
            dump_outputs(args.dump_outputs, mine, out_T.cpu().numpy(), out_err.cpu().numpy(),
                         out_pass.cpu().numpy())
    launches = eng.launch_count - launches0
    step_ms = np.array([e[0].elapsed_time(e[1]) for e in ev])
    total_ms = torch.tensor([step_ms.sum()], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_s = float(total_ms.item()) * 1e-3
    clocks = sampler.window(t_wall0, t_wall1) if rank == 0 else None

    # work actually done (exact: passes per pair come back from the kernel)
    passes = out_pass.cpu().numpy().astype(np.int64)
    work = float(np.sum(passes * lens[pairs_mine[:, 0]] * lens[pairs_mine[:, 1]]))  # PDE per step on this rank
    info = eng.kernel_info(B)

    # ---- sustained segment: a few hundred milliseconds of back-to-back steps, for the clock record ----
    sustained = None
    if not args.no_sustained:
        n_sus = max(20, int(0.4 / max(total_s / args.steps, 1e-4)))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.time()
        e0.record()
        for _ in range(n_sus):
            step_device()
        e1.record()
        barrier()
        t1 = time.time()
        sus_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(sus_ms, op=dist.ReduceOp.MAX)
        if rank == 0:
            sustained = {"steps": n_sus, "ms_per_step": float(sus_ms.item()) / n_sus,
                         "value": (n_global if args.strong else world * B) * n_sus / (float(sus_ms.item()) * 1e-3),
                         "l2": "not flushed (steps back to back)", "clocks": sampler.window(t0, t1)}

    # the same kernel with pruning switched off (every source point sweeps every target, the
    # reference's brute force): the variant the FP32-pipe roofline is defined for
    ex_ms = []
    for k in range(0 if args.no_exhaustive else 2 + min(args.steps, 5)):
        flush.fill_(float(k))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch(exhaustive=True)
        e1.record()
        torch.cuda.synchronize()
        if k >= 2:
            ex_ms.append(e0.elapsed_time(e1))
    assert np.array_equal(out_pass.cpu().numpy().astype(np.int64), passes)
    ex_s = float(np.mean(ex_ms)) * 1e-3 if ex_ms else float("nan")
    # kernel alone (no barrier), and one instrumented launch outside every timed region: the distance
    # evaluations actually executed
    k_ms = []
    for k in range(5):
        flush.fill_(float(k))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        torch.cuda.synchronize()
        k_ms.append(e0.elapsed_time(e1))
    kern_s = float(np.mean(k_ms[1:])) * 1e-3
    eng.count_work(True)
    launch()
    executed = float(eng.read_work())
    eng.count_work(False)
    if gather is not None:
        gather.barrier()

    # ---- e2e: the public host API fed the reference's own input form, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        eng2 = gicp.IcpEngine(local)
        # host threads that pack the list into pinned staging: this rank's share of the host's cores
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
        eng2.set_tuning("pack_threads", max(1, min(8, len(_ALL_CPUS or os.sched_getaffinity(0)) // max(local_world, 1))))
        rec_pin = torch.empty((n_global, 8), dtype=torch.float64).pin_memory() if gather is not None else None
        tab_pin = gicp.ScanTable(xy=torch.from_numpy(table.xy).pin_memory().numpy(), offsets=table.offsets)

        def step_host(scan_arg):
            # scans + pairs + initial guesses in host memory -> constraints of ALL ranks in host memory
            res = eng2.align(scan_arg, pairs_mine, init_mine, epsilon=EPS, max_iters=MAX_ITERS, epilogue=ep)
            if gather is not None:
                gather.barrier()
                rec_pin.copy_(gather.records(), non_blocking=True)
                torch.cuda.synchronize()
            return res

        def time_host(scan_arg):
            for _ in range(max(min(args.warmup, 5), 2)):
                res = step_host(scan_arg)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                res = step_host(scan_arg)
            barrier()
            t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t, res

        t_pin, res = time_host(tab_pin)                       # a pre-packed table in pinned memory, for comparison
        t_e2e, res = time_host(scans)                         # the reference's own input form: the e2e number
        h2d = table.xy.nbytes + table.offsets.nbytes + pairs_mine.nbytes + (0 if init_mine is None else B * 48) + 4 * B
        d2h = B * (6 * 8 + 8 + 4) + 4 + (0 if gather is None else n_global * 64)
        e2e = {"value": (n_global if args.strong else world * B) * args.steps / float(t_e2e.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": float(t_e2e.item()) / args.steps * 1e3,
               "input": "lidar_points as the reference holds them: a Python list of separate pageable (m_i, 2) "
                        "float64 arrays, packed into pinned staging by the library's host threads while earlier "
                        "pieces are on the wire",
               "call": "IcpEngine.align -> icpb_align_host_scans" + ("" if gather is None else
                       " with the fused-gather epilogue, symmetric-memory barrier, D2H of all ranks' records"),
               "pinned_table": {"value": (n_global if args.strong else world * B) * args.steps / float(t_pin.item()),
                                "ms_per_step": float(t_pin.item()) / args.steps * 1e3,
                                "input": "the same scans pre-packed as one (sum m_i, 2) table in pinned memory "
                                         "(icpb_align_host_ex): no host packing, one read of host memory per byte"}}
        assert np.array_equal(res.iters, passes.astype(np.int32))
        eng2.close()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        sm_max_mhz = float(peaks.get("sm_max_mhz", 1965.0))
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        sm_count = info["sm_count"]
        pde_peak = sm_count * 128 * sm_max_mhz * 1e6 / 4.0                 # FP32-pipe lane-slots / 4 per PDE
        ncu = None
        try:
            ncu = json.load(open(NCU_SUMMARY))
        except (OSError, ValueError):
            pass
        same_wl = bool(ncu) and ncu.get("workload") == args.workload and ncu.get("scans") == args.scans \
            and ncu.get("beams") == args.beams and world == 1
        alg_bytes = float(np.sum(16.0 * (lens[pairs_mine[:, 0]] + lens[pairs_mine[:, 1]]) + 60.0 + 56.0))
        roofline = {
            "bound": "fp32_pipe", "unit": "TPDE/s",
            "achieved": executed / kern_s * 1e-12, "peak": pde_peak * 1e-12, "frac": executed / kern_s / pde_peak,
            "traffic": (ncu or {}).get("dram_bytes") if same_wl else None,
            "definition": "PDE = one point-pair distance evaluation = 4 FP32-pipe lane-slots (FADD, FADD, FMUL, FFMA); "
                          "peak = SMs*128*sm_max_mhz/4 (clock " + peak_src + "); achieved = distance evaluations the "
                          "timed kernel EXECUTED (counted by an instrumented launch of the same kernel) / its "
                          "average duration; frac = the share of the FP32 pipe's lane-slots it used",
            "kernel_ms": kern_s * 1e3, "executed_pde_per_launch": executed,
            "algorithmic": {"pde_per_launch": work, "executed_share": executed / max(work, 1.0),
                            "speedup_over_exhaustive_sweep": ex_s / kern_s,
                            "note": "passes*N1*N2 is what the reference's brute force evaluates; exact chunk pruning "
                                    "proves the rest unnecessary (bit-identical results, tests/test_gpu_parity.py)"},
            "exhaustive": {"kernel_ms": ex_s * 1e3, "achieved": work / ex_s * 1e-12, "frac": work / ex_s / pde_peak,
                           "pairs_per_s": B / ex_s,
                           "note": "the same kernel with pruning off: every distance executed, the variant the "
                                   "FP32-pipe roofline bounds; with the min tree on the ALU pipe (which all but "
                                   "serialises with packed f32x2 instructions, profiles/r02_micro_pipes.log) the "
                                   "attainable fraction is 0.80"},
            "hbm_view": {"algorithmic_bytes_per_launch": alg_bytes, "achieved_gbs": alg_bytes / kern_s * 1e-9,
                         "peak_gbs": hbm_peak, "frac": alg_bytes / kern_s * 1e-9 / hbm_peak, "peak_source": peak_src},
        }
        if same_wl:
            # what bounds the pruned kernel: pipe-weighted issue cycles (packed f32x2, ALU-pipe and fp64
            # instructions hold their pipe two cycles); counters of a committed capture of this command
            roofline["issue_view"] = {k: ncu[k] for k in ("warp_instructions", "pipe_weighted_cycles_per_smsp",
                                                          "kernel_cycles_elapsed", "frac_of_weighted_issue_peak",
                                                          "source", "commit") if k in ncu}
        cpu = None
        if world == 1 and not args.no_cpu:
            if _ALL_CPUS:
                os.sched_setaffinity(0, _ALL_CPUS)            # the CPU baseline gets every host core back
            rate, nthr, n, dt, mean_pass = cpu_port_rate(scans, pairs, init, args.cpu_seconds)
            cpu = {"value": rate, "unit": UNIT, "cores": nthr, "kind": "port",
                   "sample": f"{n} of {n_total} pairs (seeded random subsample) in {dt:.1f} s, "
                             f"mean {mean_pass:.1f} passes, C port oracle/icp_oracle.c on {nthr} threads",
                   "numpy_reference": numpy_reference_rate(scans, pairs, init, args.cpu_seconds)}
        pairs_per_step = n_global if args.strong else world * B
        line = {
            "metric": METRIC, "value": pairs_per_step * args.steps / total_s, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_s / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_of(args, world),
            "details": {"pairs_per_step": pairs_per_step, "pairs_per_gpu": B, "mean_passes": float(passes.mean()),
                        "collective": ("none" if world == 1 else
                                       "fused: kernel epilogue stores (pairs, 8) f64 records into every rank's buffer "
                                       "over NVLink peer memory at their global rows + symmetric-memory barrier"),
                        "partition": ("one GPU" if world == 1 else
                                      f"interleaved blocks of {args.block} problems" if args.strong else
                                      "every rank its own chain"),
                        "gather_check": gather_check, "kernel": info, "host_affinity": numa},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "sustained": sustained,
        }
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    sampler.stop()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
