"""CPU-side checks: the C-ABI library loads and exports every symbol include/icpb.h declares,
host-side validation raises before anything is launched, and the product never imports the
oracle.  No compute calls (no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "icpb.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(icpb_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from icp_slam_b200 import _lib
    so = _lib.build()
    L = ctypes.CDLL(so)
    syms = declared_symbols()
    assert len(syms) >= 12
    for s in syms:
        assert hasattr(L, s), s
    assert sorted(_lib.EXPORTS) == syms
    L.icpb_abi_version.restype = ctypes.c_int
    assert L.icpb_abi_version() == 2


def test_default_params_match_reference_defaults():
    from icp_slam_b200 import _lib
    p = _lib.default_params()       # pure host function, no CUDA call
    assert (p.epsilon, p.max_iters, p.stopping_thresh, p.rotation_only) == (0.01, 100, 0.0001, 0)
    assert p.hist_cap == 0 and p.corr_stride == 0 and p.pair_mode == 0


def test_param_struct_layout_matches_header():
    from icp_slam_b200 import _lib
    assert ctypes.sizeof(_lib.IcpbParams) == 2 * 8 + 6 * 4 + 3 * 8
    assert ctypes.sizeof(_lib.IcpbKernelInfo) == 8 * 4


def test_no_gpu_fails_loudly():
    """Without a CUDA device the product raises; it never falls back to a CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from icp_slam_b200 import icp as gicp
    a = np.c_[np.random.default_rng(0).uniform(size=(10, 2)), np.ones(10)]
    with pytest.raises((gicp.IcpbError, RuntimeError)):
        gicp.icp(a, a)


def test_host_validation_precedes_launch():
    from icp_slam_b200 import icp as gicp
    a = np.c_[np.random.default_rng(0).uniform(size=(10, 2)), np.ones(10)]
    with pytest.raises(ValueError):
        gicp.icp(a[:0], a)
    with pytest.raises(ValueError):
        gicp.icp(a[:, :2], a)
    with pytest.raises(ValueError):
        gicp.icp(a, a, init_transform=np.eye(4))
    with pytest.raises(ValueError):
        gicp.ScanTable([a[:, :2], a[:0, :2]])
    with pytest.raises(ValueError):
        gicp.ScanTable(xy=a[:, :2], offsets=[0, 4, 4, 10])
    t = gicp.ScanTable([a[:, :2], a[:4, :2]])
    assert t.n_scans == 2 and t.longest == 10 and list(t.offsets) == [0, 10, 14]
    assert gicp.max_passes(100) == 102 and gicp.max_passes(-3) == 1


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "icp-slam-with-loop-closure_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower().replace("no oracle", ""), f


def test_compose_chain_matches_reference_loop():
    """icpb_compose_chain (a host function: runs without a GPU) against the reference's serial
    composition, restated with the golden SE(2) helpers, and against the end-to-end golden."""
    from icp_slam_b200 import callers, synth
    z = np.load(os.path.join(ROOT, "tests", "golden", "slam_golden.npz"))
    got = callers.compose_chain(z["odometry"][0], z["chain_T"])
    np.testing.assert_allclose(got, z["corrected"], rtol=0, atol=1e-12)
    rng = np.random.default_rng(2)
    T = np.stack([synth.pose_to_mat(p) for p in rng.uniform(-0.3, 0.3, size=(400, 3))])
    want = np.zeros((401, 3)); want[0] = (1.0, -2.0, 3.0)
    for i in range(400):
        want[i + 1] = synth.mat_to_pose(synth.pose_to_mat(want[i]) @ T[i])
    np.testing.assert_allclose(callers.compose_chain(want[0], T), want, rtol=0, atol=1e-12)
    assert callers.compose_chain([0, 0, 0], np.zeros((0, 3, 3))).shape == (1, 3)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (runs on host cores, no GPU needed) prints ONE JSON line with the
    contract's keys."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--scans", "40", "--beams", "128"], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"] > 0
    assert "workload" in d["config"]


def test_bench_dump_outputs_reference_arm(tmp_path):
    """`bench.py --dump-outputs DIR` writes the last timed step's results as float64 .npy files; the
    inputs are seeded, so runs with different step counts write the same arrays, and they are what the
    C port returns for the same pairs."""
    import argparse
    import subprocess
    import sys
    from oracle import c_oracle
    sys.path.insert(0, ROOT)
    import bench
    dirs = []
    for steps in (1, 2):
        d = tmp_path / f"s{steps}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps",
                              str(steps), "--warmup", "0", "--scans", "30", "--beams", "128", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr[-2000:]
        dirs.append(d)
    z = [{n: np.load(d / f"{n}.npy") for n in ("T", "error", "passes", "rows")} for d in dirs]
    for n in z[0]:
        assert z[0][n].dtype == np.float64
        np.testing.assert_array_equal(z[0][n], z[1][n])
    assert z[0]["T"].shape == (29, 6) and z[0]["rows"].tolist() == list(range(29))
    args = argparse.Namespace(workload="chain", scans=30, beams=128, strong=False, pairs=0)
    scans, pairs, init = bench.workload(args, 0, 1)
    xy, off = c_oracle.pack(scans)
    T, err, passes = c_oracle.icp_batch(xy, off, pairs, init, epsilon=bench.EPS, max_iters=bench.MAX_ITERS)
    np.testing.assert_array_equal(z[0]["T"], c_oracle.to6(T))
    np.testing.assert_array_equal(z[0]["error"], err)
    np.testing.assert_array_equal(z[0]["passes"], passes)


def test_bench_dump_outputs_samples_past_the_cap(tmp_path, monkeypatch):
    """Past the size cap, --dump-outputs keeps a sorted seeded sample of the rows, the same on every call."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 72 * 100)
    n = 1000
    T6 = np.arange(6 * n, dtype=np.float64).reshape(n, 6)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), np.arange(n), T6, np.arange(n) * 0.5, np.arange(n, dtype=np.int32))
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert len(rows) == 100 and np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "T.npy"), T6[rows.astype(np.int64)])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "passes.npy"), rows)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_BYTES


def test_upload_plan_pieces_end_on_sector_boundaries():
    """icpb_plan_upload (the host logic that cuts the scan table for the streaming upload): pieces
    are contiguous, cover every scan, and every interior boundary sits on an even point offset (a
    32-byte sector of the fp64 table) -- on a 128-byte line when one lies within reach."""
    from icp_slam_b200 import _lib
    L = ctypes.CDLL(_lib.build())
    L.icpb_plan_upload.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]
    rng = np.random.default_rng(11)
    for trial in range(60):
        n = int(rng.integers(1, 6000))
        lens = rng.integers(1, 1200, size=n) if trial % 3 else rng.integers(1, 4, size=n) * 2 + 1   # all-odd lengths too
        off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
        want = int(rng.integers(0, 40))
        ends = np.zeros(64, dtype=np.int64)
        k = ctypes.c_int32()
        rc = L.icpb_plan_upload(off.ctypes.data, n, want, ends.ctypes.data, ctypes.byref(k))
        assert rc == 0 and 1 <= k.value <= 64
        e = ends[:k.value]
        assert e[-1] == n and np.all(np.diff(e) > 0) and e[0] >= 1
        assert np.all(off[e[:-1]] % 2 == 0)                      # interior boundaries: even point offsets
        if want == 0:
            assert k.value <= 18
    # a table of 5,000 x 1,024-point scans: 18 pieces (the first and last two a quarter and a half of
    # a standard one, so the upload starts and ends with short pieces), all on 128-byte lines
    off = (np.arange(5001) * 1024).astype(np.int64)
    ends = np.zeros(64, dtype=np.int64); k = ctypes.c_int32()
    assert L.icpb_plan_upload(off.ctypes.data, 5000, 0, ends.ctypes.data, ctypes.byref(k)) == 0
    assert k.value == 18 and np.all(off[ends[:17]] % 8 == 0)
    sizes = np.diff(np.concatenate(([0], ends[:18])))
    assert sizes[0] < sizes[1] < sizes[2] and sizes[-1] < sizes[-2] < sizes[-3]
    assert L.icpb_plan_upload(off.ctypes.data, 5000, 16, ends.ctypes.data, ctypes.byref(k)) == 0
    assert k.value == 16 and np.ptp(np.diff(np.concatenate(([0], ends[:16])))) <= 1       # explicit count: equal pieces
    assert L.icpb_plan_upload(None, 5000, 0, ends.ctypes.data, ctypes.byref(k)) != 0


def test_epilogue_struct_layout_matches_header():
    """icpb_epilogue as ctypes sees it: 12 fields, 88 bytes, in the header's order."""
    from icp_slam_b200 import _lib
    text = open(os.path.join(ROOT, "include", "icpb.h")).read()
    body = re.search(r"typedef struct icpb_epilogue \{(.*?)\} icpb_epilogue;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [n for decl in body.split(";") for n in re.findall(r"\*?\s*(\w+)\s*(?:,|$)", decl.split(None, 1)[1] if decl.split() else "")
             if n not in ("const", "uint64_t", "int32_t", "int64_t", "double")]
    assert names == [n for n, _ in _lib.IcpbEpilogue._fields_]
    assert ctypes.sizeof(_lib.IcpbEpilogue) == 88


def test_scan_list_helper_describes_a_list_of_arrays():
    """ScanList: pointer + length per scan straight from the caller's arrays (buffer protocol helper,
    no copies), conversions only for elements that are not C-ordered float64."""
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(0)
    scans = [rng.normal(size=(int(m), 2)) for m in rng.integers(1, 400, size=257)]
    sl = gicp.ScanList(scans)
    assert sl.keep is scans and sl.n_scans == 257
    np.testing.assert_array_equal(sl.lens, [len(s) for s in scans])
    np.testing.assert_array_equal(sl.ptrs, [s.ctypes.data for s in scans])
    odd = list(scans)
    odd[10] = np.asfortranarray(scans[10])
    odd[200] = scans[200].astype(np.float32)
    so = gicp.ScanList(odd)
    assert so.keep is not odd and so.ptrs[9] == scans[9].ctypes.data and so.ptrs[10] != odd[10].ctypes.data
    np.testing.assert_array_equal(so.keep[200], scans[200].astype(np.float32).astype(np.float64))
    with pytest.raises(ValueError):
        gicp.ScanList(scans[:3] + [np.zeros((0, 2))])
    with pytest.raises(ValueError):
        gicp.ScanList(scans[:3] + [np.zeros((5, 3))])
    with pytest.raises(ValueError):
        gicp.ScanList([])
    t = gicp.ScanTable.from_lengths(sl.lens)
    assert t.n_scans == 257 and t.longest == int(sl.lens.max())


def test_edge_arrays_keeps_what_the_optimiser_acts_on():
    """Host side of the pose-graph SGD drop-in (no GPU needed): odometry edges (|a-b| == 1) and edges with
    b <= a are left out (reference src/pose_graph_optimization.py:14-16, :20, :28-30, :46), iteration order
    is kept, malformed transforms are named."""
    from icp_slam_b200 import pose_graph_optimization as pgo
    T = np.array([[0.0, -1.0, 2.0], [1.0, 0.0, 3.0], [0.0, 0.0, 1.0]])
    edges = [(0, 1, np.eye(3)), (7, 3, np.eye(3)), (2, 9, T), (4, 5, np.eye(3)), (1, 6, np.eye(3)), (5, 5, np.eye(3))]
    ab, T6 = pgo.edge_arrays(edges)
    assert ab.dtype == np.int32 and ab.tolist() == [[2, 9], [1, 6]]
    np.testing.assert_array_equal(T6, np.stack([T[:2].reshape(6), np.eye(3)[:2].reshape(6)]))
    assert T6.flags["C_CONTIGUOUS"] and T6.dtype == np.float64
    ab0, T0 = pgo.edge_arrays([(0, 1, np.eye(3))])
    assert ab0.shape == (0, 2) and T0.shape == (0, 6)
    bad = np.eye(3); bad[2, 0] = 0.5
    with pytest.raises(ValueError, match=r"edge \(0, 3\).*bottom row"):
        pgo.edge_arrays([(2, 9, T), (0, 3, bad)])
    with pytest.raises(ValueError, match=r"edge \(0, 3\).*shape \(2, 2\)"):
        pgo.edge_arrays([(0, 3, np.eye(2)), (2, 9, T)])
