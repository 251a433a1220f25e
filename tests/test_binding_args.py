"""The argument path of the Python binding, without a GPU: the pair parser, the SE(2) converter, the top-rows
helpers, the batch parameters, result subsets, the device-buffer checks, the table mirror after a failed
upload and the one signature table of the C exports.  Engine methods run on an engine without a handle: their
checks come before any library call, and a library call on it fails like a failed upload."""
import ctypes

import numpy as np
import pytest


@pytest.fixture(scope="module")
def gicp():
    from icp_slam_b200 import icp as m
    return m


@pytest.fixture(scope="module")
def lib():
    from icp_slam_b200 import _lib as m
    return m


@pytest.fixture
def bare(gicp, lib):
    """An IcpEngine whose handle was never created."""
    e = gicp.IcpEngine.__new__(gicp.IcpEngine)
    e._h, e._L, e.device = ctypes.c_void_p(), lib.lib(), 0
    e.table = e._keep = e._base = None
    return e


def _se2(rng, n):
    T = np.zeros((n, 3, 3))
    T[:, :2, :] = rng.normal(size=(n, 2, 3))
    T[:, 2, 2] = 1.0
    return T


def test_pair_parser(gicp):
    a = gicp._pairs([[1, 0], [2, 1]])
    assert a.dtype == np.int32 and a.shape == (2, 2) and a.flags.c_contiguous
    assert gicp._pairs([]).shape == (0, 2)
    for bad in (np.zeros((4, 3)), np.zeros(4), np.zeros((2, 2, 2))):
        with pytest.raises(ValueError, match="pairs has shape"):
            gicp._pairs(bad)


def test_align_accept_rejects_malformed_pairs(gicp, bare):
    """A (4, 3) array is not six pairs: align_accept rejects it like run, run_multistart and align."""
    scans = gicp.ScanTable([np.random.default_rng(1).uniform(size=(5, 2)) for _ in range(4)])
    for bad in (np.zeros((4, 3), dtype=np.int32), np.zeros(4, dtype=np.int32), np.zeros((2, 2, 2), dtype=np.int32)):
        with pytest.raises(ValueError, match="pairs has shape"):
            bare.align_accept(scans, bad, 1.0)


def test_table_known_by_lengths_is_rejected_before_the_library(gicp, bare):
    t = gicp.ScanTable.from_lengths([5, 7])
    with pytest.raises(ValueError, match="only describes a resident table"):
        gicp._upload_args(t)
    bare._L = None                                           # a library call would raise AttributeError
    with pytest.raises(ValueError, match="only describes a resident table"):
        bare.align(t, [[1, 0]])
    with pytest.raises(ValueError, match="only describes a resident table"):
        bare.align_accept(t, [[1, 0]], 1.0)


def test_upload_args_packed_and_list(gicp):
    scans = [np.random.default_rng(2).uniform(size=(n, 2)) for n in (3, 5)]
    packed = gicp.ScanTable(scans)
    table, held, (xy, off, ptrs, lens) = gicp._upload_args(packed)
    assert table is packed and held is packed and ptrs is None and lens is None
    assert xy.value == packed.xy.ctypes.data and off.value == packed.offsets.ctypes.data
    table, held, (xy, off, ptrs, lens) = gicp._upload_args(scans)
    assert isinstance(held, gicp.ScanList) and xy is None and off is None
    assert table.xy is None and list(table.offsets) == [0, 3, 8]
    assert ptrs.value == held.ptrs.ctypes.data and lens.value == held.lens.ctypes.data


def test_se2_converter(gicp):
    rng = np.random.default_rng(3)
    T = _se2(rng, 4)
    for bounds in (True, False):
        T6 = gicp._to6(T, bounds)
        assert T6.shape == (4, 6) and T6.flags.c_contiguous
        np.testing.assert_array_equal(T6, T[:, :2, :].reshape(4, 6))
        np.testing.assert_array_equal(gicp._to6(T[1], bounds), T[1, :2, :].ravel())
        bottom = T.copy()
        bottom[2, 2, 1] = 1e-300
        with pytest.raises(ValueError, match="bottom row"):
            gicp._to6(bottom, bounds)
        nan = T.copy()
        nan[3, 0, 2] = np.nan
        with pytest.raises(ValueError, match="non-finite"):
            gicp._to6(nan, bounds)
        with pytest.raises(ValueError, match="shape"):
            gicp._to6(T[:, :2, :], bounds)
    wide = T.copy()
    wide[0, 0, 1] = 2 * gicp.MAX_GUESS_LINEAR
    far = T.copy()
    far[1, 1, 2] = 2 * gicp.MAX_GUESS_SHIFT
    for beyond in (wide, far):
        with pytest.raises(ValueError, match="bounds"):
            gicp._to6(beyond)
        np.testing.assert_array_equal(gicp._to6(beyond, bounds=False), beyond[:, :2, :].reshape(4, 6))
    with pytest.raises(ValueError, match=r"starts has shape \(4, 2, 3\); expected \(K, 3, 3\)"):
        gicp._mats(T[:, :2, :], None, "starts")
    with pytest.raises(ValueError, match=r"expected \(5, 3, 3\)"):
        gicp._mats(T, 5, "init_transforms")


def test_top_rows_round_trip(gicp):
    rng = np.random.default_rng(4)
    for shape in ((), (1,), (7,), (3, 5)):
        T = _se2(rng, int(np.prod(shape, dtype=int))).reshape(shape + (3, 3))
        T6 = gicp._top_rows(T)
        assert T6.shape == shape + (6,) and T6.flags.c_contiguous and T6.dtype == np.float64
        np.testing.assert_array_equal(gicp._to33(T6), T)
        np.testing.assert_array_equal(gicp._top_rows(gicp._to33(T6)), T6)
    # a strided view of the top rows (the records' first six columns) goes back the same way
    rec = rng.normal(size=(6, 8))
    np.testing.assert_array_equal(gicp._top_rows(gicp._to33(rec[:, :6])), rec[:, :6])


def test_params_batch_fields(gicp):
    p = gicp._params(0.05, 30, 1e-4, False, B=7)
    assert (p.pair_mode, p.k_first, p.k_block, p.k_stride) == (0, 0, 7, 0)
    assert gicp._params(0.05, 30, 1e-4, False, B=0).k_block == 1
    assert gicp._params(0.05, 30, 1e-4, False).k_block == 1
    p = gicp._params(0.05, 30, 1e-4, True, True, B=99, all_pairs=(4096, 4096, 16384, 777))
    assert (p.pair_mode, p.k_first, p.k_block, p.k_stride) == (1, 4096, 4096, 16384)
    assert p.flags == 1 and p.rotation_only == 1 and p.epsilon == 0.05 and p.max_iters == 30
    with pytest.raises(ValueError):
        gicp._params(0.05, 30, 1e-4, False, all_pairs=(0, 1, 0))
    with pytest.raises(ValueError, match="max_iters"):
        gicp._params(0.05, 2.5, 1e-4, False)


def test_take_keeps_the_result_kind(gicp):
    rng = np.random.default_rng(5)
    B, K = 6, 3
    ms = gicp.MultiStartResult(_se2(rng, B), rng.uniform(size=B), np.arange(B, dtype=np.int32),
                               start=np.arange(B, dtype=np.int32) % K, error_all=rng.uniform(size=(B, K)))
    rows = np.array([1, 4, 5])
    sub = ms.take(rows)
    assert type(sub) is gicp.MultiStartResult and len(sub) == 3
    np.testing.assert_array_equal(sub.T, ms.T[rows])
    np.testing.assert_array_equal(sub.error, ms.error[rows])
    np.testing.assert_array_equal(sub.iters, ms.iters[rows])
    np.testing.assert_array_equal(sub.start, ms.start[rows])
    np.testing.assert_array_equal(sub.error_all, ms.error_all[rows])
    assert sub.iters_all is None and sub.history is None and sub.correspondences is None
    br = gicp.BatchResult(ms.T, ms.error, ms.iters)
    sub = br.take(br.error < 0.5)
    assert type(sub) is gicp.BatchResult
    np.testing.assert_array_equal(sub.error, ms.error[ms.error < 0.5])


def test_buffer_checks(gicp):
    torch = pytest.importorskip("torch")
    good = torch.zeros(12, dtype=torch.float64)
    with pytest.raises(ValueError, match="expected torch.float64"):
        gicp._check_buffer(good.float(), torch.float64, 12, "out_T")
    with pytest.raises(ValueError, match="holds 12 elements; expected 6"):
        gicp._check_buffer(good, torch.float64, 6, "out_T")
    with pytest.raises(ValueError, match="not contiguous"):
        gicp._check_buffer(torch.zeros(24, dtype=torch.float64)[::2], torch.float64, 12, "out_T")
    with pytest.raises(ValueError, match="not on a CUDA device"):
        gicp._check_buffer(good, torch.float64, 12, "out_T")


class _DeviceBuffer:
    """Stands in for a contiguous CUDA tensor: the checks read only its dtype, shape and placement."""

    def __init__(self, dtype, *shape):
        self.dtype, self.shape, self.is_cuda = dtype, shape, True

    def numel(self):
        return int(np.prod(self.shape))

    def is_contiguous(self):
        return True


def test_device_launches_check_every_buffer(gicp, bare):
    """run_device and run_device_ex check every buffer before anything is launched; the all-pairs launch
    ignores the pair tensor it is handed."""
    torch = pytest.importorskip("torch")
    B = 4
    good = dict(pairs_t=_DeviceBuffer(torch.int32, B, 2), init_t=_DeviceBuffer(torch.float64, B, 6),
                out_T=_DeviceBuffer(torch.float64, B, 6), out_err=_DeviceBuffer(torch.float64, B),
                out_passes=_DeviceBuffer(torch.int32, B))
    wrong = {"pairs_t": torch.zeros((B, 2), dtype=torch.int64), "init_t": torch.zeros((B, 3, 3), dtype=torch.float64),
             "out_T": torch.zeros((B, 6), dtype=torch.float32), "out_err": torch.zeros(B + 1, dtype=torch.float64),
             "out_passes": torch.zeros(2 * B, dtype=torch.int32)[::2]}
    for name, bad in wrong.items():
        args = list(dict(good, **{name: bad}).values())
        with pytest.raises(ValueError, match=name):
            bare.run_device(*args)
        with pytest.raises(ValueError, match=name):
            bare.run_device_ex(*args, None)
    with pytest.raises(ValueError, match="pairs_t holds 8 elements; expected 16"):    # B from the first dimension
        bare.run_device(_DeviceBuffer(torch.int32, 2 * B), None, *list(good.values())[2:])
    host_T = torch.zeros((B, 6), dtype=torch.float64)
    with pytest.raises(ValueError, match="out_T is not on a CUDA device"):
        bare.run_device_ex(torch.zeros(1), None, host_T, good["out_err"], good["out_passes"], None,
                           all_pairs=(0, B, 0, B))


def test_failed_upload_that_drops_the_table_clears_the_mirror(gicp, bare):
    """When the library has no table after a failed upload, the engine does not name the old one as
    resident, so the next call uploads it again."""
    rng = np.random.default_rng(6)
    old = gicp.ScanTable([rng.uniform(size=(5, 2)) for _ in range(3)])
    bare.table, bare._base = old, old
    assert bare.is_resident(old) and bare.ensure_scans(old) is old
    with pytest.raises(ValueError):
        bare.set_scans(gicp.ScanTable([rng.uniform(size=(5, 2)) for _ in range(3)]))
    assert bare.table is None and bare._keep is None and bare._base is None
    assert not bare.is_resident(old) and not bare.is_resident(None)


def test_every_export_is_declared_once(lib):
    assert lib.EXPORTS == list(lib.SIGNATURES)
    L = lib.lib()
    for name in lib.EXPORTS:
        restype, argtypes = lib.SIGNATURES[name]
        fn = getattr(L, name)
        assert fn.argtypes == argtypes, name
        assert fn.restype is restype, name
