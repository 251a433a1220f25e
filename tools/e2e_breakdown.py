import sys, time, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from icp_slam_b200 import icp as gicp, synth
scans, pairs, init, _, _ = synth.make_chain_workload(5000, 1024, seed=467002)
t = gicp.ScanTable(scans)
xy = torch.from_numpy(t.xy).pin_memory(); off = torch.from_numpy(t.offsets).pin_memory()
tp = gicp.ScanTable(xy=xy.numpy(), offsets=off.numpy())
e = gicp.IcpEngine(0)
def tm(f, n=10):
    f(); f()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(n): f()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / n * 1e3
print("align (pinned scans)      %.3f ms" % tm(lambda: e.align(tp, pairs, init, epsilon=0.05)))
print("align (pageable table)    %.3f ms" % tm(lambda: e.align(t, pairs, init, epsilon=0.05)))
# the reference's own input form: a list of separate pageable (m_i, 2) arrays (src/dataloader.py:110-112)
for nthr in (4, 8, 12, 16):
    e.set_tuning("pack_threads", nthr)
    print("align (list, %d pack thr)  %.3f ms" % (nthr, tm(lambda: e.align(scans, pairs, init, epsilon=0.05))))
e.set_tuning("pack_threads", 0)
print("ScanList(scans)           %.3f ms" % tm(lambda: gicp.ScanList(scans)))
e.set_scans(tp)
print("run only (resident scans) %.3f ms" % tm(lambda: e.run(pairs, init, epsilon=0.05)))
print("set_scans only (pinned)   %.3f ms" % tm(lambda: e.set_scans(tp)))
print("_to6(init)                %.3f ms" % tm(lambda: gicp._to6(init)))
print("_to33                     %.3f ms" % tm(lambda: gicp._to33(np.zeros((4999, 6)))))
for sg in (4, 16, 32, 64):
    e.set_tuning("segments", sg)
    print("align segments=%d          %.3f ms" % (sg, tm(lambda: e.align(tp, pairs, init, epsilon=0.05))))
