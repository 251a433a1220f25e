"""The memory a handle owns: its resident scan table and the host copy of the table's offsets.

* An align call rejected for its pairs or guesses leaves the old table in place, also when the rejected
  table is larger than the resident one (so its buffers would have to grow).
* A borrowed table is read again after icpb_set_scans_device: a batch split by scan length uses the
  offsets of the table as it is now, not those of an earlier call.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gicp():
    from icp_slam_b200 import icp as m
    return m


@pytest.fixture(scope="module")
def synth():
    from icp_slam_b200 import synth as m
    return m


def _assert_same(a, b):
    np.testing.assert_array_equal(a.T, b.T)
    np.testing.assert_array_equal(a.error, b.error)
    np.testing.assert_array_equal(a.iters, b.iters)


@pytest.mark.parametrize("form", ["list", "packed"])
def test_rejected_align_keeps_a_smaller_resident_table(gicp, synth, form):
    small, sp, si, _, _ = synth.make_chain_workload(12, 360, seed=71)
    big, bp, bi, _, _ = synth.make_chain_workload(200, 1024, seed=72)   # ~50x the points of `small`
    scans = big if form == "list" else gicp.ScanTable(big)
    bad_pairs = bp.copy()
    bad_pairs[7, 1] = len(big)
    bad_init = bi.copy()
    bad_init[3, 2, 0] = 0.5                                             # not an SE(2) matrix
    e = gicp.IcpEngine()
    try:
        e.set_scans(small)
        ref = e.run(sp, si, epsilon=0.05, max_iters=30)
        calls = {
            "align, pair out of range": lambda: e.align(scans, bad_pairs, bi, epsilon=0.05, max_iters=30),
            "align, bad guess": lambda: e.align(scans, bp, bad_init, epsilon=0.05, max_iters=30),
            "align_accept, pair out of range": lambda: e.align_accept(scans, bad_pairs, 1.0, bi, epsilon=0.05),
            "align_accept, bad guess": lambda: e.align_accept(scans, bp, 1.0, bad_init, epsilon=0.05),
        }
        for name, call in calls.items():
            with pytest.raises(ValueError):
                call()
            assert e.table.n_scans == len(small), name
            _assert_same(e.run(sp, si, epsilon=0.05, max_iters=30), ref)
    finally:
        e.close()


def test_borrowed_table_rewritten_in_place(gicp, synth):
    """A table with two scans beyond shared memory, then the same scans in reverse order written into the
    same tensors: same scan count and point count, the long scans at other indices."""
    import torch
    shorts = synth.make_chain_workload(8, 1024, seed=81)[0]
    longs = synth.make_chain_workload(2, 20000, seed=82)[0]
    first = shorts[:3] + [longs[0]] + shorts[3:6] + [longs[1]] + shorts[6:]
    second = first[::-1]
    n = len(first)
    pairs = np.array([(i + 1, i) for i in range(n - 1)] + [(3, 7), (2, 6)], dtype=np.int32)
    starts = gicp.heading_starts(3)
    t1, t2 = gicp.ScanTable(first), gicp.ScanTable(second)
    assert t1.n_scans == t2.n_scans and len(t1.xy) == len(t2.xy)
    assert not np.array_equal(t1.offsets, t2.offsets)

    fresh = gicp.IcpEngine()
    e = gicp.IcpEngine()
    try:
        dev = torch.device("cuda", e.device)
        xy_t = torch.from_numpy(t1.xy).to(dev)
        off_t = torch.from_numpy(t1.offsets).to(dev)
        torch.cuda.synchronize(dev)
        fresh.set_scans(t1)
        e.set_scans_device(xy_t, off_t, t1)
        _assert_same(e.run(pairs, epsilon=0.05), fresh.run(pairs, epsilon=0.05))

        xy_t.copy_(torch.from_numpy(t2.xy))
        off_t.copy_(torch.from_numpy(t2.offsets))
        torch.cuda.synchronize(dev)
        e.set_scans_device(xy_t, off_t, t2)
        fresh.set_scans(t2)
        _assert_same(e.run(pairs, epsilon=0.05), fresh.run(pairs, epsilon=0.05))
        a = e.run_multistart(pairs, starts, epsilon=0.05, return_all=True)
        b = fresh.run_multistart(pairs, starts, epsilon=0.05, return_all=True)
        _assert_same(a, b)
        np.testing.assert_array_equal(a.start, b.start)
        np.testing.assert_array_equal(a.error_all, b.error_all)
        np.testing.assert_array_equal(a.iters_all, b.iters_all)
    finally:
        e.close()
        fresh.close()
