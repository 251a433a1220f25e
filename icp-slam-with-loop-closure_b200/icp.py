"""Drop-in for the reference's ``src/icp.py`` backed by the sm_100a kernels in libicpb.so.

Same names, argument meaning and return contracts as the reference module:

* ``icp(pc1, pc2, init_transform=np.eye(3), epsilon=0.01, max_iters=100,
  stopping_thresh=0.0001, rotation_only=False) -> (transforms, error)``      (src/icp.py:72-97)
* ``icp_iteration(pc1, pc2, previous_transform, rotation_only=False)
  -> (trans_mat, correspondences, error)``                                     (src/icp.py:55-69)
* ``get_correspondences`` / ``get_closest_point``                              (src/icp.py:4-19)
* ``get_transform`` / ``get_error``                                            (src/icp.py:22-52)

plus the batched entry point ``icp_batch`` that replaces the reference's joblib fan-outs
(scripts/main.py:240-247, src/loop_closure_detection.py:134-142,
src/pose_graph_optimization.py:60-68) with one kernel launch, and ``icp_multistart``, which aligns
every pair from K start transforms and keeps the best one (``heading_starts``, ``compose_starts``).

There is no CPU fallback: without libicpb.so and a B200 every call raises.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import IcpbError  # noqa: F401  (re-exported)
from .synth import pose_to_mat

__all__ = ["icp", "icp_iteration", "icp_batch", "icp_multistart", "heading_starts", "compose_starts",
           "get_correspondences", "get_closest_point", "get_transform", "get_error",
           "ScanTable", "ScanList", "IcpEngine", "BatchResult", "MultiStartResult", "engine", "make_epilogue"]


# Input magnitudes the kernel is exact for (include/icpb.h: ICPB_MAX_COORD, ICPB_MAX_GUESS_LINEAR,
# ICPB_MAX_GUESS_SHIFT).  `not (abs(v) <= bound)` is also true for NaN.
MAX_COORD = 1e10
MAX_GUESS_LINEAR = 1e3
MAX_GUESS_SHIFT = 1e12


def _coords_ok(xy) -> bool:
    return bool((np.abs(xy) <= MAX_COORD).all())


# --------------------------------------------------------------------------- scan table
class ScanTable:
    """The reference's ``lidar_points`` (a list of (m_i, 2) float64 arrays,
    src/dataloader.py:110-112) packed as one (sum m_i, 2) array + int64 CSR offsets."""

    def __init__(self, scans=None, xy=None, offsets=None):
        if scans is not None:
            if len(scans) == 0:
                raise ValueError("empty scan list")
            arrs = []
            for k, s in enumerate(scans):
                s = np.asarray(s, dtype=np.float64)
                if s.ndim != 2 or s.shape[1] != 2:
                    raise ValueError(f"scan {k} has shape {s.shape}; expected (m, 2) as get_point_cloud returns")
                if s.shape[0] == 0:
                    raise ValueError(f"scan {k} is empty (the reference's argmin raises on an empty cloud)")
                arrs.append(s)
            lens = np.array([a.shape[0] for a in arrs], dtype=np.int64)
            self.offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
            self.xy = np.ascontiguousarray(np.concatenate(arrs, axis=0))
        else:
            self.xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
            self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
            if self.offsets.ndim != 1 or len(self.offsets) < 2 or self.offsets[0] != 0 \
                    or self.offsets[-1] != len(self.xy) or np.any(np.diff(self.offsets) <= 0):
                raise ValueError("offsets must start at 0, end at len(xy) and be strictly increasing")
        if not _coords_ok(self.xy):
            raise ValueError(f"scan table holds non-finite coordinates or coordinates beyond +-{MAX_COORD:g}")

    @classmethod
    def from_lengths(cls, lengths) -> "ScanTable":
        """A table known only by its scan lengths (the scans themselves live in device memory, uploaded
        from a list of arrays): enough for index validation and result shapes."""
        t = cls.__new__(cls)
        t.xy = None
        t.offsets = np.concatenate(([0], np.cumsum(np.asarray(lengths, dtype=np.int64)))).astype(np.int64)
        return t

    @property
    def n_scans(self) -> int:
        return len(self.offsets) - 1

    @property
    def lengths(self) -> np.ndarray:
        return np.diff(self.offsets)

    @property
    def longest(self) -> int:
        return int(self.lengths.max())


# --------------------------------------------------------------------------- results
@dataclass
class BatchResult:
    """Per-problem results of ``icp_batch``: what B independent ``icp()`` calls return."""
    T: np.ndarray                  # (B, 3, 3) float64 = transforms[-1]
    error: np.ndarray              # (B,) float64  = the returned error
    iters: np.ndarray              # (B,) int32    = len(transforms) - 1 (passes)
    history: np.ndarray | None = None          # (B, cap, 3, 3) = transforms[1:], identity-padded past iters
    correspondences: np.ndarray | None = None  # (B, longest source) int32, -1 padded; last pass

    @property
    def R(self) -> np.ndarray:
        return self.T[:, :2, :2]

    @property
    def t(self) -> np.ndarray:
        return self.T[:, :2, 2]

    def __len__(self):
        return len(self.error)


@dataclass
class MultiStartResult(BatchResult):
    """Per-pair results of ``icp_multistart``: the winning start's ``T``, ``error`` and ``iters``, and
    which start won.  With ``return_all=True`` also every start's error and pass count."""
    start: np.ndarray | None = None            # (B,) int32: the smallest k with the smallest error
    error_all: np.ndarray | None = None        # (B, K) float64
    iters_all: np.ndarray | None = None        # (B, K) int32


def _to6(T) -> np.ndarray:
    T = np.asarray(T, dtype=np.float64)
    if T.shape[-2:] != (3, 3):
        raise ValueError(f"transform has shape {T.shape}; expected (..., 3, 3)")
    if not (np.all(T[..., 2, 0] == 0) and np.all(T[..., 2, 1] == 0) and np.all(T[..., 2, 2] == 1)):
        raise ValueError("transform bottom row must be [0, 0, 1] (an SE(2) matrix)")
    if not (np.all(np.abs(T[..., :2, :2]) <= MAX_GUESS_LINEAR) and np.all(np.abs(T[..., :2, 2]) <= MAX_GUESS_SHIFT)):
        raise ValueError(f"transform holds non-finite values or values beyond the bounds of include/icpb.h "
                         f"(|linear part| <= {MAX_GUESS_LINEAR:g}, |translation| <= {MAX_GUESS_SHIFT:g})")
    return np.ascontiguousarray(T[..., :2, :].reshape(T.shape[:-2] + (6,)))


def _to33(T6: np.ndarray) -> np.ndarray:
    out = np.zeros(T6.shape[:-1] + (3, 3))
    out[..., :2, :] = T6.reshape(T6.shape[:-1] + (2, 3))
    out[..., 2, 2] = 1.0
    return out


def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def _rows6(T, n, name) -> np.ndarray:
    """(n, 3, 3) SE(2)-shaped matrices (n None: any number) -> (n, 6) top rows, with the shape, the
    bottom rows and finiteness checked; the bounds are the library's to check (on the composed guesses)."""
    T = np.asarray(T, dtype=np.float64)
    if T.ndim != 3 or T.shape[1:] != (3, 3) or (n is not None and len(T) != n):
        raise ValueError(f"{name} has shape {T.shape}; expected ({'K' if n is None else n}, 3, 3)")
    if not (np.all(T[..., 2, 0] == 0) and np.all(T[..., 2, 1] == 0) and np.all(T[..., 2, 2] == 1)):
        raise ValueError(f"{name}: bottom row must be [0, 0, 1] (an SE(2) matrix)")
    if not np.isfinite(T).all():
        raise ValueError(f"{name} holds non-finite values")
    return np.ascontiguousarray(T[..., :2, :].reshape(T.shape[:-2] + (6,)))


def heading_starts(k: int) -> np.ndarray:
    """(k, 3, 3) rotations by theta_i = -pi + 2 pi i / k, i = 0 .. k-1 (``pose_to_mat((0, 0, theta_i))``):
    a sweep of k headings for ``icp_multistart``, the guesses of bench.py's highres workload."""
    k = int(k)
    if k < 1:
        raise ValueError("heading_starts needs k >= 1")
    th = -np.pi + 2 * np.pi * np.arange(k) / k
    return np.stack([pose_to_mat((0.0, 0.0, t)) for t in th])


def compose_starts(init, starts) -> np.ndarray:
    """(B, K, 3, 3): the guesses ``icp_multistart`` aligns from, G[p, k] = init[p] @ starts[k], with the
    formula of include/icpb.h -- every product and sum rounded on its own, left to right, so the result
    has the library's bits: ``icp_batch(scans, np.repeat(pairs, K, axis=0), G.reshape(-1, 3, 3))``
    reproduces every problem of a multi-start run.  ``init`` is (B, 3, 3), or None for one identity
    guess (B = 1)."""
    S = np.asarray(starts, dtype=np.float64)
    if S.ndim != 3 or S.shape[1:] != (3, 3):
        raise ValueError(f"starts has shape {S.shape}; expected (K, 3, 3)")
    I = np.eye(3)[None] if init is None else np.asarray(init, dtype=np.float64)
    if I.ndim != 3 or I.shape[1:] != (3, 3):
        raise ValueError(f"init has shape {I.shape}; expected (B, 3, 3)")
    G = np.zeros((len(I), len(S), 3, 3))
    for r in range(2):
        a, c, t = I[:, None, r, 0], I[:, None, r, 1], I[:, None, r, 2]
        G[:, :, r, 0] = a * S[None, :, 0, 0] + c * S[None, :, 1, 0]
        G[:, :, r, 1] = a * S[None, :, 0, 1] + c * S[None, :, 1, 1]
        G[:, :, r, 2] = (a * S[None, :, 0, 2] + c * S[None, :, 1, 2]) + t
    G[:, :, 2, 2] = 1.0
    return G


class ScanList:
    """The reference's ``lidar_points`` as it is -- a sequence of separate (m_i, 2) float64 arrays in
    pageable memory (src/dataloader.py:110-112) -- described by a pointer and a length per scan for
    ``icpb_align_host_scans``.  Nothing is copied unless an element is not a C-ordered float64 array;
    the library packs and checks the coordinates itself, overlapped with the upload."""

    def __init__(self, scans):
        n = len(scans)
        if n == 0:
            raise ValueError("empty scan list")
        self.ptrs = np.empty(n, dtype=np.uint64)
        self.lens = np.empty(n, dtype=np.int64)
        self.keep = scans                      # the arrays must outlive the call
        helper = _lib.pyhelper()
        k = helper.icpb_py_scan_ptrs(scans, _ptr(self.ptrs), _ptr(self.lens), n) if helper else 0
        if k < 0:
            k = 0
        if k < n:                              # elements the helper did not take: convert them one by one
            fixed = list(scans[:k]) if k else []
            for i in range(k, n):
                a = np.ascontiguousarray(scans[i], dtype=np.float64)
                if a.ndim != 2 or a.shape[1] != 2:
                    raise ValueError(f"scan {i} has shape {a.shape}; expected (m, 2) as get_point_cloud returns")
                fixed.append(a)
                self.ptrs[i] = a.ctypes.data
                self.lens[i] = a.shape[0]
            self.keep = fixed
        if (self.lens <= 0).any():
            bad = int(np.argmax(self.lens <= 0))
            raise ValueError(f"scan {bad} is empty (the reference's argmin raises on an empty cloud)")

    @property
    def n_scans(self) -> int:
        return len(self.lens)


def make_epilogue(peer_ptrs_dev=0, n_peers=0, rank=0, row0=0, row_block=0, row_stride=0,
                  accept_thresh=None, accept_rec=0, accept_count=0, accept_peer_ptrs=0,
                  accept_count_peer_ptrs=0, accept_cap=0) -> _lib.IcpbEpilogue:
    """icpb_epilogue from raw device addresses (ints; 0 = not used).  See include/icpb.h."""
    ep = _lib.IcpbEpilogue()
    ep.d_peer_ptrs = int(peer_ptrs_dev) or None
    ep.n_peers, ep.rank = int(n_peers), int(rank)
    ep.row0, ep.row_block, ep.row_stride = int(row0), int(row_block), int(row_stride)
    ep.accept_thresh = float(accept_thresh) if accept_thresh is not None else 0.0
    ep.d_accept_rec = int(accept_rec) or None
    ep.d_accept_count = int(accept_count) or None
    ep.d_accept_peer_ptrs = int(accept_peer_ptrs) or None
    ep.d_accept_count_peer_ptrs = int(accept_count_peer_ptrs) or None
    ep.accept_cap = int(accept_cap)
    return ep


def _params(epsilon, max_iters, stopping_thresh, rotation_only, exhaustive=False) -> _lib.IcpbParams:
    p = _lib.default_params()
    p.flags = _lib.FLAG_EXHAUSTIVE if exhaustive else 0
    p.epsilon = float(epsilon)
    p.stopping_thresh = float(stopping_thresh)
    mi = int(max_iters)
    if mi != max_iters:
        raise ValueError("max_iters must be an integer")
    p.max_iters = max(min(mi, 2 ** 31 - 8), -2)
    p.rotation_only = 1 if rotation_only else 0
    return p


def max_passes(max_iters: int) -> int:
    """Upper bound on passes: ``iteration > max_iters`` is tested after the pass, so the
    reference makes up to max_iters + 2 of them (src/icp.py:88, SURVEY.md section 8a)."""
    return max(int(max_iters) + 2, 1)


# --------------------------------------------------------------------------- engine
def resolve_device(device: int | None) -> int:
    """None -> ICPB_DEVICE, else LOCAL_RANK (one process per GPU), else 0."""
    if device is None:
        device = os.environ.get("ICPB_DEVICE", os.environ.get("LOCAL_RANK", "0"))
    return int(device)


class IcpEngine:
    """One icpb handle: per process and per device (the replacement for a loky worker)."""

    def __init__(self, device: int | None = None):
        self._h = ctypes.c_void_p()
        self._L = _lib.lib()
        self.device = resolve_device(device)
        _lib.check(self._L.icpb_create(self.device, ctypes.byref(self._h)), "icpb_create")
        self.table: ScanTable | None = None
        self._keep = None

    def close(self):
        if self._h:
            self._L.icpb_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_tuning(self, key: str, value: int):
        """Per-handle tuning / test hook (icpb_set_tuning; nothing is read from the environment)."""
        _lib.check(self._L.icpb_set_tuning(self._h, key.encode(), int(value)), "icpb_set_tuning")

    # -- scan table -----------------------------------------------------------------------
    def set_scans(self, scans) -> ScanTable:
        table = scans if isinstance(scans, ScanTable) else ScanTable(scans)
        _lib.check(self._L.icpb_upload_scans(self._h, _ptr(table.xy), _ptr(table.offsets), table.n_scans),
                   "icpb_upload_scans")
        self.table = table
        self._keep = None
        return table

    def set_scans_device(self, xy_t, offsets_t, table: ScanTable):
        """Borrow a scan table already resident in HBM (torch CUDA tensors)."""
        assert xy_t.is_cuda and offsets_t.is_cuda and xy_t.is_contiguous() and offsets_t.is_contiguous()
        _lib.check(self._L.icpb_set_scans_device(self._h, ctypes.c_void_p(xy_t.data_ptr()),
                                                 ctypes.c_void_p(offsets_t.data_ptr()), table.n_scans,
                                                 table.longest), "icpb_set_scans_device")
        self.table = table
        self._keep = (xy_t, offsets_t)

    # -- host-buffer run (the reference-facing call) -----------------------------------------
    def run(self, pairs, init_transforms=None, epsilon=0.01, max_iters=100, stopping_thresh=0.0001,
            rotation_only=False, return_history=False, return_correspondences=False,
            all_pairs: tuple | None = None, exhaustive: bool = False) -> BatchResult:
        """`exhaustive=True` sweeps every target for every source point (the reference's brute
        force) instead of the default exact chunk pruning; the results are identical."""
        if self.table is None:
            raise ValueError("no scan table set")
        p = _params(epsilon, max_iters, stopping_thresh, rotation_only, exhaustive)
        if all_pairs is not None:
            # (k_first, k_block, k_stride, B): linear indices over i<j decoded on the device
            p.pair_mode = 1
            p.k_first, p.k_block, p.k_stride, B = (int(v) for v in all_pairs)
            pairs_a = None
        else:
            pairs_a = np.ascontiguousarray(pairs, dtype=np.int32)
            if pairs_a.size == 0:
                pairs_a = pairs_a.reshape(0, 2)
            if pairs_a.ndim != 2 or pairs_a.shape[1] != 2:
                raise ValueError(f"pairs has shape {pairs_a.shape}; expected (B, 2) of (source, target) scan ids")
            if pairs_a.size and (pairs_a.min() < 0 or pairs_a.max() >= self.table.n_scans):
                raise ValueError("pair index out of range")
            B = len(pairs_a)
            p.k_block = max(B, 1)
        init6 = None
        if init_transforms is not None:
            it = np.asarray(init_transforms, dtype=np.float64)
            if it.shape != (B, 3, 3):
                raise ValueError(f"init_transforms has shape {it.shape}; expected ({B}, 3, 3)")
            init6 = _to6(it)
        cap = max_passes(p.max_iters) if return_history else 0
        if cap > 4096:
            raise ValueError("return_history with max_iters > 4094 is not supported")
        stride = self.table.longest if return_correspondences else 0
        p.hist_cap, p.corr_stride = cap, stride
        T6 = np.empty((B, 6))
        err = np.empty(B)
        passes = np.empty(B, dtype=np.int32)
        hist = np.empty((B, cap, 6)) if cap else None
        corr = np.empty((B, stride), dtype=np.int32) if stride else None
        _lib.check(self._L.icpb_run_host(self._h, _ptr(pairs_a), _ptr(init6), B, ctypes.byref(p),
                                         _ptr(T6), _ptr(err), _ptr(passes), _ptr(hist), _ptr(corr)),
                   "icpb_run_host")
        history = None
        if cap:
            history = _to33(hist)
            pad = np.arange(cap)[None, :] >= passes[:, None]
            history[pad] = np.eye(3)
        return BatchResult(_to33(T6), err, passes, history, corr)

    # -- multi-start run on the resident table ---------------------------------------------------
    def run_multistart(self, pairs, starts, init_transforms=None, epsilon=0.01, max_iters=100,
                       stopping_thresh=0.0001, rotation_only=False, return_all=False,
                       exhaustive: bool = False) -> MultiStartResult:
        """Every pair aligned from ``init[p] @ starts[k]`` for every start k (icpb_run_multistart_host);
        returns the winner per pair (the smallest k with the smallest error).  The library checks the
        composed guesses against its bounds (ValueError)."""
        if self.table is None:
            raise ValueError("no scan table set")
        p = _params(epsilon, max_iters, stopping_thresh, rotation_only, exhaustive)
        pairs_a = np.ascontiguousarray(pairs, dtype=np.int32)
        if pairs_a.size == 0:
            pairs_a = pairs_a.reshape(0, 2)
        if pairs_a.ndim != 2 or pairs_a.shape[1] != 2:
            raise ValueError(f"pairs has shape {pairs_a.shape}; expected (B, 2) of (source, target) scan ids")
        B = len(pairs_a)
        S6 = _rows6(starts, None, "starts")
        K = len(S6)
        init6 = None if init_transforms is None else _rows6(init_transforms, B, "init_transforms")
        T6, err = np.empty((B, 6)), np.empty(B)
        passes, start = np.empty(B, dtype=np.int32), np.empty(B, dtype=np.int32)
        err_all = np.empty((B, K)) if return_all else None
        passes_all = np.empty((B, K), dtype=np.int32) if return_all else None
        _lib.check(self._L.icpb_run_multistart_host(self._h, _ptr(pairs_a), _ptr(init6), B, _ptr(S6), K,
                                                    ctypes.byref(p), _ptr(T6), _ptr(err), _ptr(passes),
                                                    _ptr(start), _ptr(err_all), _ptr(passes_all)),
                   "icpb_run_multistart_host")
        return MultiStartResult(_to33(T6), err, passes, start=start, error_all=err_all, iters_all=passes_all)

    # -- upload + run in one call, upload overlapped with the kernels ---------------------------
    def align(self, scans, pairs, init_transforms=None, epsilon=0.01, max_iters=100, stopping_thresh=0.0001,
              rotation_only=False, exhaustive: bool = False, epilogue: _lib.IcpbEpilogue | None = None) -> BatchResult:
        """Upload + run in one call (icpb_align_host_ex / icpb_align_host_scans): the scan table goes up
        in pieces and every pair starts as soon as both of its scans are on the device.  ``scans`` is a
        ScanTable (packed, ideally pinned) or the reference's own list of (m_i, 2) arrays, which the
        library packs into pinned staging with a few host threads while earlier pieces are on the wire.
        ``epilogue``: fused all-gather / acceptance of the records (multi-GPU, see dist.FusedGather)."""
        p = _params(epsilon, max_iters, stopping_thresh, rotation_only, exhaustive)
        pairs_a = np.ascontiguousarray(pairs, dtype=np.int32)
        if pairs_a.size == 0:
            pairs_a = pairs_a.reshape(0, 2)
        if pairs_a.ndim != 2 or pairs_a.shape[1] != 2:
            raise ValueError(f"pairs has shape {pairs_a.shape}; expected (B, 2) of (source, target) scan ids")
        B = len(pairs_a)
        p.k_block = max(B, 1)
        init33 = None
        if init_transforms is not None:
            # the reference's (B, 3, 3) matrices go to the library as they are: it checks the pair
            # indices, the bottom rows and finiteness while it stages them (ICPB_EINVAL -> ValueError)
            init33 = np.ascontiguousarray(init_transforms, dtype=np.float64)
            if init33.shape != (B, 3, 3):
                raise ValueError(f"init_transforms has shape {init33.shape}; expected ({B}, 3, 3)")
        T33 = np.empty((B, 3, 3))
        err = np.empty(B)
        passes = np.empty(B, dtype=np.int32)
        ep = ctypes.byref(epilogue) if epilogue is not None else None
        prev, self.table = (self.table, self._keep), None
        try:
            table = self._align_call(scans, pairs_a, init33, B, p, T33, err, passes, ep)
        except Exception:
            # rejected before anything was touched (bad pairs / guesses): the old table is still there;
            # failed part-way: the library has dropped it (icpb_scan_count == 0)
            if self._L.icpb_scan_count(self._h) > 0:
                self.table, self._keep = prev
            raise
        self.table, self._keep = table, None
        return BatchResult(T33, err, passes, None, None)

    def align_accept(self, scans, pairs, accept_thresh, init_transforms=None, epsilon=0.01, max_iters=100,
                     stopping_thresh=0.0001, rotation_only=False):
        """`align` for the loop-closure callers: the acceptance test `error < accept_thresh`
        (src/loop_closure_detection.py:35-39, :155-159) and the compaction run in the kernel epilogue and
        only the accepted constraints come back.  Returns (rows, BatchResult): `rows` are ascending
        indices into `pairs`, the BatchResult holds their results."""
        p = _params(epsilon, max_iters, stopping_thresh, rotation_only)
        pairs_a = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        B = len(pairs_a)
        if B == 0:
            return np.zeros(0, dtype=np.int64), BatchResult(np.zeros((0, 3, 3)), np.zeros(0), np.zeros(0, dtype=np.int32))
        p.k_block = B
        init33 = None
        if init_transforms is not None:
            init33 = np.ascontiguousarray(init_transforms, dtype=np.float64)
            if init33.shape != (B, 3, 3):
                raise ValueError(f"init_transforms has shape {init33.shape}; expected ({B}, 3, 3)")
        if isinstance(scans, ScanTable) and self.table is scans:
            # the table is already resident: nothing to upload, so nothing to overlap with -- align on it
            # and filter the (B x 60 byte) results on the host
            res = self.run(pairs_a, init_transforms, epsilon, max_iters, stopping_thresh, rotation_only)
            keep = np.nonzero(res.error < accept_thresh)[0]
            return keep, BatchResult(res.T[keep], res.error[keep], res.iters[keep])
        rows = np.empty(B, dtype=np.int64)
        T33, err, passes = np.empty((B, 3, 3)), np.empty(B), np.empty(B, dtype=np.int32)
        n = ctypes.c_int64()
        prev, self.table = (self.table, self._keep), None
        try:
            if isinstance(scans, ScanTable):
                table, xy, off, ptrs, lens, ns = scans, _ptr(scans.xy), _ptr(scans.offsets), None, None, scans.n_scans
            else:
                sl = scans if isinstance(scans, ScanList) else ScanList(scans)
                table, xy, off, ptrs, lens, ns = ScanTable.from_lengths(sl.lens), None, None, _ptr(sl.ptrs), _ptr(sl.lens), sl.n_scans
            _lib.check(self._L.icpb_align_host_accept(self._h, xy, off, ptrs, lens, ns, _ptr(pairs_a), _ptr(init33), 9, B,
                                                      ctypes.byref(p), float(accept_thresh), B, ctypes.byref(n),
                                                      _ptr(rows), _ptr(T33), 9, _ptr(err), _ptr(passes)),
                       "icpb_align_host_accept")
        except Exception:
            if self._L.icpb_scan_count(self._h) > 0:
                self.table, self._keep = prev
            raise
        self.table, self._keep = table, None
        k = int(n.value)
        return rows[:k].copy(), BatchResult(T33[:k].copy(), err[:k].copy(), passes[:k].copy())

    def _align_call(self, scans, pairs_a, init33, B, p, T33, err, passes, ep):
        if isinstance(scans, ScanTable):
            table = scans
            if table.xy is None:
                raise ValueError("this ScanTable only describes a resident table; pass the scans themselves")
            _lib.check(self._L.icpb_align_host_ex(self._h, _ptr(table.xy), _ptr(table.offsets), table.n_scans,
                                                  _ptr(pairs_a), _ptr(init33), 9, B, ctypes.byref(p),
                                                  _ptr(T33), 9, _ptr(err), _ptr(passes), ep), "icpb_align_host")
        else:
            sl = scans if isinstance(scans, ScanList) else ScanList(scans)
            _lib.check(self._L.icpb_align_host_scans(self._h, _ptr(sl.ptrs), _ptr(sl.lens), sl.n_scans,
                                                     _ptr(pairs_a), _ptr(init33), 9, B, ctypes.byref(p),
                                                     _ptr(T33), 9, _ptr(err), _ptr(passes), ep),
                       "icpb_align_host_scans")
            table = ScanTable.from_lengths(sl.lens)
        return table

    # -- device-buffer run (inputs and outputs resident in HBM; torch tensors) ---------------
    def run_device(self, pairs_t, init_t, out_T, out_err, out_passes, epsilon=0.01, max_iters=100,
                   stopping_thresh=0.0001, rotation_only=False, all_pairs: tuple | None = None,
                   stream=None, exhaustive: bool = False):
        """Asynchronous launch on torch's current stream (or `stream`, a raw cudaStream_t int).
        pairs_t (B,2) int32, init_t (B,6) float64 or None, outputs (B,6) f64, (B,) f64, (B,) i32."""
        import torch
        p = _params(epsilon, max_iters, stopping_thresh, rotation_only, exhaustive)
        if all_pairs is not None:
            p.pair_mode = 1
            p.k_first, p.k_block, p.k_stride, B = (int(v) for v in all_pairs)
        else:
            B = int(pairs_t.shape[0])
            p.k_block = max(B, 1)
            assert pairs_t.dtype == torch.int32 and pairs_t.is_cuda and pairs_t.is_contiguous()
        assert out_T.dtype == torch.float64 and out_T.numel() == 6 * B and out_T.is_contiguous()
        assert out_err.dtype == torch.float64 and out_err.numel() == B
        assert out_passes.dtype == torch.int32 and out_passes.numel() == B
        if init_t is not None:
            assert init_t.dtype == torch.float64 and init_t.numel() == 6 * B and init_t.is_contiguous()
        if stream is None:
            stream = torch.cuda.current_stream(self.device).cuda_stream
        vp = ctypes.c_void_p
        _lib.check(self._L.icpb_run_device(self._h, vp(pairs_t.data_ptr()) if all_pairs is None else None,
                                           vp(init_t.data_ptr()) if init_t is not None else None, B,
                                           ctypes.byref(p), vp(out_T.data_ptr()), vp(out_err.data_ptr()),
                                           vp(out_passes.data_ptr()), None, None, vp(stream)),
                   "icpb_run_device")

    def run_device_ex(self, pairs_t, init_t, out_T, out_err, out_passes, epilogue: _lib.IcpbEpilogue | None,
                      epsilon=0.01, max_iters=100, stopping_thresh=0.0001, rotation_only=False,
                      all_pairs: tuple | None = None, stream=None):
        """`run_device` with kernel epilogues (icpb_run_device_ex): the fused all-gather of the
        constraint records into every rank's buffer and/or the acceptance test + compaction."""
        import torch
        p = _params(epsilon, max_iters, stopping_thresh, rotation_only)
        if all_pairs is not None:
            p.pair_mode = 1
            p.k_first, p.k_block, p.k_stride, B = (int(v) for v in all_pairs)
        else:
            B = int(pairs_t.shape[0])
            p.k_block = max(B, 1)
        if stream is None:
            stream = torch.cuda.current_stream(self.device).cuda_stream
        vp = ctypes.c_void_p
        _lib.check(self._L.icpb_run_device_ex(self._h, vp(pairs_t.data_ptr()) if all_pairs is None else None,
                                              vp(init_t.data_ptr()) if init_t is not None else None, B,
                                              ctypes.byref(p), vp(out_T.data_ptr()), vp(out_err.data_ptr()),
                                              vp(out_passes.data_ptr()),
                                              ctypes.byref(epilogue) if epilogue is not None else None, vp(stream)),
                   "icpb_run_device_ex")

    def run_device_gather(self, pairs_t, init_t, out_T, out_err, out_passes, peer_ptrs_dev: int, n_peers: int,
                          row0: int, epsilon=0.01, max_iters=100, stopping_thresh=0.0001, rotation_only=False,
                          stream=None):
        """`run_device` with the all-gather fused into the kernel: every finished pair's record
        [T(6), error, passes] is stored into every rank's (total, 8) float64 gather buffer at row
        row0 + pair id over NVLink peer memory.  `peer_ptrs_dev` is the device address of the array
        of peer buffer pointers (torch symmetric memory: ``handle.buffer_ptrs_dev``)."""
        ep = make_epilogue(peer_ptrs_dev, n_peers, row0=row0)
        self.run_device_ex(pairs_t, init_t, out_T, out_err, out_passes, ep, epsilon, max_iters, stopping_thresh,
                           rotation_only, stream=stream)

    # -- one pair given as two arrays ------------------------------------------------------------
    def pair(self, src_xy, dst_xy, init6, p: _lib.IcpbParams, want_hist: bool, want_corr: bool):
        src = np.ascontiguousarray(src_xy, dtype=np.float64)
        dst = np.ascontiguousarray(dst_xy, dtype=np.float64)
        cap = max_passes(p.max_iters) if want_hist else 0
        p.hist_cap = cap
        p.corr_stride = len(src) if want_corr else 0
        T6 = np.empty(6)
        err = ctypes.c_double()
        passes = ctypes.c_int32()
        hist = np.zeros((cap, 6)) if cap else None
        corr = np.empty(len(src), dtype=np.int32) if want_corr else None
        _lib.check(self._L.icpb_icp_pair_host(self._h, _ptr(src), len(src), _ptr(dst), len(dst), _ptr(init6),
                                              ctypes.byref(p), _ptr(T6), ctypes.byref(err),
                                              ctypes.byref(passes), _ptr(hist), _ptr(corr)),
                   "icpb_icp_pair_host")
        return T6, err.value, passes.value, hist, corr

    def kernel_info(self, B: int = 0) -> dict:
        info = _lib.IcpbKernelInfo()
        _lib.check(self._L.icpb_get_kernel_info(self._h, B, ctypes.byref(info)), "icpb_get_kernel_info")
        return info.as_dict()

    @property
    def launch_count(self) -> int:
        return int(self._L.icpb_launch_count(self._h))

    def count_work(self, enable: bool = True):
        """Instrumentation: count the distance evaluations launches actually execute."""
        _lib.check(self._L.icpb_count_work(self._h, 1 if enable else 0), "icpb_count_work")

    def read_work(self) -> int:
        v = ctypes.c_uint64()
        _lib.check(self._L.icpb_read_work(self._h, ctypes.byref(v)), "icpb_read_work")
        return int(v.value)


_engines: dict = {}


def engine(device: int | None = None) -> IcpEngine:
    """Lazily created per (process, device): safe to call from loky/fork workers because the
    handle is keyed by pid and created on first use in that process."""
    device = resolve_device(device)                    # engine(None) and engine(0) share one handle
    key = (os.getpid(), device)
    e = _engines.get(key)
    if e is None:
        e = IcpEngine(device)
        _engines[key] = e
    return e


# --------------------------------------------------------------------------- drop-in functions
def _cloud_xy(pc, name: str) -> np.ndarray:
    """(n, 3) homogeneous rows (C- or F-ordered) -> contiguous (n, 2)."""
    pc = np.asarray(pc, dtype=np.float64)
    if pc.ndim != 2 or pc.shape[1] != 3:
        raise ValueError(f"{name} has shape {pc.shape}; expected (n, 3) homogeneous rows (src/icp.py:76)")
    if pc.shape[0] == 0:
        raise ValueError(f"{name} is empty (the reference's argmin raises on an empty cloud)")
    if not np.all(pc[:, 2] == 1.0):
        raise ValueError(f"{name}: the homogeneous column must be all ones")
    xy = np.ascontiguousarray(pc[:, :2])
    if not _coords_ok(xy):
        raise ValueError(f"{name} holds non-finite coordinates or coordinates beyond +-{MAX_COORD:g}")
    return xy


def _check_T(T, name: str):
    if not isinstance(T, np.ndarray) or T.shape != (3, 3):
        raise ValueError(f"{name} must be a 3x3 numpy array")


def icp(pc1, pc2, init_transform=np.eye(3), epsilon=0.01, max_iters=100, stopping_thresh=0.0001,
        rotation_only=False):
    """Reference ``icp`` (src/icp.py:72-97): estimate the SE(2) transform moving ``pc1`` onto
    ``pc2`` ((n, 3) homogeneous clouds).  Returns ``(transforms, error)``: ``transforms`` is the
    list ``[init_transform, T_1, ..., T_k]`` of cumulative 3x3 matrices (``transforms[0]`` is the
    caller's object; under ``rotation_only`` its translation is zeroed in place like the
    reference does, src/icp.py:60-61) and ``error`` the numpy float64 SSE the last pass measured.
    """
    _check_T(init_transform, "init_transform")
    src, dst = _cloud_xy(pc1, "pc1"), _cloud_xy(pc2, "pc2")
    p = _params(epsilon, max_iters, stopping_thresh, rotation_only)
    if max_passes(p.max_iters) > 1 << 20:
        raise ValueError("max_iters too large to return the transform list")
    if rotation_only:
        init_transform[:2, 2] = 0
    T6, err, passes, hist, _ = engine().pair(src, dst, _to6(init_transform), p, True, False)
    tfs = [init_transform] + list(_to33(hist[:passes]))
    return tfs, np.float64(err)


def icp_iteration(pc1, pc2, previous_transform, rotation_only=False):
    """Reference ``icp_iteration`` (src/icp.py:55-69): one pass.  Returns
    ``(trans_mat, correspondences, error)`` with ``correspondences[i]`` the index into ``pc2``
    matched to source point i (int64, like ``np.zeros(n, dtype=int)``, src/icp.py:15)."""
    _check_T(previous_transform, "previous_transform")
    src, dst = _cloud_xy(pc1, "pc1"), _cloud_xy(pc2, "pc2")
    p = _params(np.inf, 0, 0.0, rotation_only)          # error < inf: stop after the first pass
    if rotation_only:
        previous_transform[:2, 2] = 0
    T6, err, passes, _, corr = engine().pair(src, dst, _to6(previous_transform), p, False, True)
    return _to33(T6), corr.astype(np.int64), np.float64(err)


def get_correspondences(pc1, pc2):
    """Reference ``get_correspondences`` (src/icp.py:10-19): nearest target index per source point."""
    _, corr, _ = icp_iteration(pc1, pc2, np.eye(3))
    return corr


def get_closest_point(point, pc):
    """Reference ``get_closest_point`` (src/icp.py:4-7): index of the row of ``pc`` nearest to ``point``."""
    point = np.asarray(point, dtype=np.float64).reshape(1, -1)
    return get_correspondences(point, pc)[0]


def _fit(pc1, pc2):
    a, b = _cloud_xy(pc1, "pc1"), _cloud_xy(pc2, "pc2")
    if len(a) != len(b):
        raise ValueError("pc1 and pc2 must have the same number of rows (pc1[i] corresponds to pc2[i])")
    e = engine()
    T6 = np.empty(6)
    err = ctypes.c_double()
    _lib.check(e._L.icpb_fit_pairs_host(e._h, _ptr(a), _ptr(b), len(a), _ptr(T6), ctypes.byref(err)),
               "icpb_fit_pairs_host")
    return _to33(T6), np.float64(err.value)


def get_transform(pc1, pc2):
    """Reference ``get_transform`` (src/icp.py:22-46): the SE(2) matrix that best moves pc1[i] onto
    pc2[i] (rows correspond)."""
    return _fit(pc1, pc2)[0]


def get_error(pc1, pc2):
    """Reference ``get_error`` (src/icp.py:49-52): sum of squared differences of corresponding rows."""
    return _fit(pc1, pc2)[1]


def icp_batch(scans, pairs, init_transforms=None, epsilon=0.01, max_iters=100, stopping_thresh=0.0001,
              rotation_only=False, return_history=False, return_correspondences=False,
              device: int | None = None) -> BatchResult:
    """B independent ``icp()`` calls in one launch.

    ``scans``: the reference's ``lidar_points`` list of (m_i, 2) float64 arrays (or a ScanTable);
    ``pairs``: (B, 2) int (source scan, target scan); ``init_transforms``: (B, 3, 3) or None for
    identity.  Results equal those of ``icp(np.c_[scans[s], 1], np.c_[scans[d], 1], init, ...)``
    for every pair.
    """
    e = engine(device)
    if isinstance(scans, ScanTable) and e.table is scans:          # already resident
        return e.run(pairs, init_transforms, epsilon, max_iters, stopping_thresh, rotation_only,
                     return_history, return_correspondences)
    if not (return_history or return_correspondences):
        return e.align(scans, pairs, init_transforms, epsilon, max_iters, stopping_thresh, rotation_only)
    e.set_scans(scans)
    return e.run(pairs, init_transforms, epsilon, max_iters, stopping_thresh, rotation_only,
                 return_history, return_correspondences)


def icp_multistart(scans, pairs, starts, init_transforms=None, epsilon=0.01, max_iters=100, stopping_thresh=0.0001,
                   rotation_only=False, return_all=False, device: int | None = None) -> MultiStartResult:
    """Multi-start ``icp_batch``: pair p is aligned from ``init_transforms[p] @ starts[k]`` for every
    start k ((K, 3, 3), e.g. ``heading_starts(32)``; identity guesses when ``init_transforms`` is None)
    and the start with the smallest error wins (``np.argmin``'s rule: the first on ties).  Every start is
    exactly the ``icp()`` call ``icp_batch`` makes for the guess ``compose_starts(init, starts)[p, k]``;
    the expansion and the selection run on the device, so only B results cross PCIe.  ``return_all``
    adds every start's error and pass count, (B, K).  ``scans`` is uploaded unless it is the ScanTable
    already resident on the device."""
    e = engine(device)
    if not (isinstance(scans, ScanTable) and e.table is scans):
        e.set_scans(scans)
    return e.run_multistart(pairs, starts, init_transforms, epsilon, max_iters, stopping_thresh, rotation_only,
                            return_all)
