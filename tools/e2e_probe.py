#!/usr/bin/env python
"""Host-to-host time of IcpEngine.align on the headline workload for the three input forms: a list of
pageable arrays, a prebuilt ScanList and a pinned table (developer probe; DESIGN.md section 5)."""
import sys, time, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from icp_slam_b200 import icp as gicp, synth
scans, pairs, init, _, _ = synth.make_chain_workload(5000, 1024, seed=467002)
e = gicp.IcpEngine(0)
def tm(f, n=20):
    f(); f()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(n): f()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / n * 1e3
print("align(list) %.3f ms" % tm(lambda: e.align(scans, pairs, init, epsilon=0.05)))
sl = gicp.ScanList(scans)
print("align(ScanList prebuilt) %.3f ms" % tm(lambda: e.align(sl, pairs, init, epsilon=0.05)))
t = gicp.ScanTable(scans); xy = torch.from_numpy(t.xy).pin_memory()
tp = gicp.ScanTable(xy=xy.numpy(), offsets=t.offsets)
print("align(pinned table) %.3f ms" % tm(lambda: e.align(tp, pairs, init, epsilon=0.05)))
