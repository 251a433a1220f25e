"""ctypes binding of libicpb.so (include/icpb.h).  No CPU fallback: if the CUDA library is
missing or no sm_100 device is present, every entry point raises."""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
SO_PATH = os.environ.get("ICPB_SO") or os.path.join(_HERE, "libicpb.so")   # ICPB_SO: tuning builds

FLAG_EXHAUSTIVE = 1

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared"]

EXPORTS = ["icpb_default_params", "icpb_abi_version", "icpb_create", "icpb_destroy",
           "icpb_upload_scans", "icpb_set_scans_device", "icpb_run_device", "icpb_run_host",
           "icpb_icp_pair_host", "icpb_get_kernel_info", "icpb_launch_count", "icpb_last_error",
           "icpb_count_work", "icpb_read_work", "icpb_align_host", "icpb_align_host_ld", "icpb_plan_upload", "icpb_fit_pairs_host",
           "icpb_proximity_closest", "icpb_proximity_pairs", "icpb_compose_chain",
           "icpb_run_device_gather", "icpb_pose_graph_sgd", "icpb_occupancy_grid_bounds",
           "icpb_occupancy_grid_update", "icpb_run_device_ex", "icpb_align_host_ex", "icpb_align_host_scans",
           "icpb_set_tuning", "icpb_scan_count", "icpb_align_host_accept",
           "icpb_compose_chain_device", "icpb_compose_chain_gpu", "icpb_run_multistart_host"]


class IcpbParams(ctypes.Structure):
    _fields_ = [("epsilon", ctypes.c_double), ("stopping_thresh", ctypes.c_double),
                ("max_iters", ctypes.c_int32), ("rotation_only", ctypes.c_int32),
                ("hist_cap", ctypes.c_int32), ("corr_stride", ctypes.c_int32),
                ("pair_mode", ctypes.c_int32), ("flags", ctypes.c_int32),
                ("k_first", ctypes.c_int64), ("k_block", ctypes.c_int64), ("k_stride", ctypes.c_int64)]


class IcpbEpilogue(ctypes.Structure):
    """icpb_epilogue (include/icpb.h): fused all-gather and acceptance/compaction of the records."""
    _fields_ = [("d_peer_ptrs", ctypes.c_void_p), ("n_peers", ctypes.c_int32), ("rank", ctypes.c_int32),
                ("row0", ctypes.c_int64), ("row_block", ctypes.c_int64), ("row_stride", ctypes.c_int64),
                ("accept_thresh", ctypes.c_double), ("d_accept_rec", ctypes.c_void_p),
                ("d_accept_count", ctypes.c_void_p), ("d_accept_peer_ptrs", ctypes.c_void_p),
                ("d_accept_count_peer_ptrs", ctypes.c_void_p), ("accept_cap", ctypes.c_int64)]


class IcpbKernelInfo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("threads_per_cta", "ctas_per_sm", "sm_count", "grid",
                                              "regs_per_thread", "smem_bytes", "points_per_thread",
                                              "variant")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class IcpbError(RuntimeError):
    pass


def sources():
    c = os.path.join(_HERE, "csrc")
    return [os.path.join(c, "icpb_api.cu")], [os.path.join(c, "icpb_kernels.cuh"),
                                              os.path.join(c, "icpb_candidates.cuh"),
                                              os.path.join(c, "icpb_sgd.cuh"),
                                              os.path.join(c, "icpb_grid.cuh"),
                                              os.path.join(c, "icpb_compose.cuh"),
                                              os.path.join(c, "icpb_multistart.cuh"),
                                              os.path.join(_ROOT, "include", "icpb.h")]


PYHELPER_SRC = os.path.join(_HERE, "csrc", "icpb_pyhelper.c")
PYHELPER_SO = os.path.join(_HERE, "_icpb_pyhelper.so")


def build_pyhelper(force: bool = False) -> str:
    """gcc -> _icpb_pyhelper.so: list of numpy arrays -> pointer / length arrays (buffer protocol)."""
    import sysconfig
    if not force and os.path.exists(PYHELPER_SO) and os.path.getmtime(PYHELPER_SO) >= os.path.getmtime(PYHELPER_SRC):
        return PYHELPER_SO
    import fcntl
    with open(os.path.join(_HERE, ".build.lock"), "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        tmp = f"{PYHELPER_SO}.{os.getpid()}.tmp"
        cmd = ["gcc", "-O2", "-shared", "-fPIC", "-I", sysconfig.get_paths()["include"]]
        try:                                                # numpy's C API when its headers are there
            import numpy
            inc = numpy.get_include()
            if os.path.exists(os.path.join(inc, "numpy", "arrayobject.h")):
                cmd += ["-DICPB_WITH_NUMPY", "-I", inc]
        except ImportError:
            pass
        subprocess.check_call(cmd + ["-o", tmp, PYHELPER_SRC])
        os.replace(tmp, PYHELPER_SO)
    return PYHELPER_SO


_pyhelper = None


def pyhelper():
    """The buffer-protocol helper, or None when it cannot be built (callers then use a Python loop)."""
    global _pyhelper
    if _pyhelper is None:
        try:
            L = ctypes.PyDLL(build_pyhelper())
            L.icpb_py_scan_ptrs.argtypes = [ctypes.py_object, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong]
            L.icpb_py_scan_ptrs.restype = ctypes.c_longlong
            _pyhelper = L
        except (OSError, subprocess.CalledProcessError):
            _pyhelper = False
    return _pyhelper or None


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libicpb.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs, deps = sources()

    def stale():
        newest = max(os.path.getmtime(p) for p in srcs + deps)
        return not os.path.exists(SO_PATH) or os.path.getmtime(SO_PATH) < newest
    if not force and not stale():
        return SO_PATH
    import fcntl
    # several ranks may get here at once: one builds under the lock into a private name and renames
    with open(os.path.join(_HERE, ".build.lock"), "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        if force or stale():
            tmp = f"{SO_PATH}.{os.getpid()}.tmp"
            cmd = ["nvcc"] + NVCC_FLAGS + ["-I", os.path.join(_ROOT, "include"), "-I", os.path.join(_HERE, "csrc"),
                                           "-o", tmp] + srcs
            if verbose:
                cmd += ["-Xptxas", "-v"]
            subprocess.check_call(cmd)
            os.replace(tmp, SO_PATH)
    return SO_PATH


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        # a fresh checkout (the library is not in the history): compile the CUDA library once, in-tree;
        # if that is impossible there is nothing to fall back to
        import shutil
        if "ICPB_SO" in os.environ or shutil.which("nvcc") is None:
            raise IcpbError(f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU fallback)")
        try:
            build()
        except (subprocess.CalledProcessError, OSError) as exc:
            raise IcpbError(f"{SO_PATH} is missing and could not be built ({exc}); there is no CPU fallback") from exc
    L = ctypes.CDLL(SO_PATH)
    vp, i64, i32p, dp = ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p
    L.icpb_default_params.argtypes = [ctypes.POINTER(IcpbParams)]
    L.icpb_default_params.restype = None
    L.icpb_abi_version.restype = ctypes.c_int
    L.icpb_create.argtypes = [ctypes.c_int, ctypes.POINTER(vp)]
    L.icpb_destroy.argtypes = [vp]
    L.icpb_upload_scans.argtypes = [vp, dp, vp, i64]
    L.icpb_set_scans_device.argtypes = [vp, dp, vp, i64, i64]
    L.icpb_run_device.argtypes = [vp, i32p, dp, i64, ctypes.POINTER(IcpbParams), dp, dp, i32p, dp, i32p, vp]
    L.icpb_run_device_gather.argtypes = [vp, i32p, dp, i64, ctypes.POINTER(IcpbParams), dp, dp, i32p, vp,
                                         ctypes.c_int32, i64, vp]
    L.icpb_run_device_ex.argtypes = [vp, i32p, dp, i64, ctypes.POINTER(IcpbParams), dp, dp, i32p,
                                     ctypes.POINTER(IcpbEpilogue), vp]
    L.icpb_align_host_ex.argtypes = [vp, dp, vp, i64, i32p, dp, ctypes.c_int32, i64, ctypes.POINTER(IcpbParams),
                                     dp, ctypes.c_int32, dp, i32p, ctypes.POINTER(IcpbEpilogue)]
    L.icpb_align_host_scans.argtypes = [vp, vp, vp, i64, i32p, dp, ctypes.c_int32, i64, ctypes.POINTER(IcpbParams),
                                        dp, ctypes.c_int32, dp, i32p, ctypes.POINTER(IcpbEpilogue)]
    L.icpb_set_tuning.argtypes = [vp, ctypes.c_char_p, i64]
    L.icpb_align_host_accept.argtypes = [vp, dp, vp, vp, vp, i64, i32p, dp, ctypes.c_int32, i64,
                                         ctypes.POINTER(IcpbParams), ctypes.c_double, i64,
                                         ctypes.POINTER(ctypes.c_int64), vp, dp, ctypes.c_int32, dp, i32p]
    L.icpb_run_host.argtypes = [vp, i32p, dp, i64, ctypes.POINTER(IcpbParams), dp, dp, i32p, dp, i32p]
    L.icpb_run_multistart_host.argtypes = [vp, i32p, dp, i64, dp, ctypes.c_int32, ctypes.POINTER(IcpbParams),
                                           dp, dp, i32p, i32p, dp, i32p]
    L.icpb_align_host.argtypes = [vp, dp, vp, i64, i32p, dp, i64, ctypes.POINTER(IcpbParams), dp, dp, i32p]
    L.icpb_align_host_ld.argtypes = [vp, dp, vp, i64, i32p, dp, ctypes.c_int32, i64, ctypes.POINTER(IcpbParams),
                                     dp, ctypes.c_int32, dp, i32p]
    L.icpb_proximity_closest.argtypes = [vp, dp, dp, i64, ctypes.c_double, ctypes.c_double, i32p, dp]
    L.icpb_proximity_pairs.argtypes = [vp, dp, dp, i64, ctypes.c_double, ctypes.c_double, i64, i32p,
                                       ctypes.POINTER(ctypes.c_int64)]
    L.icpb_compose_chain.argtypes = [dp, dp, i64, dp]
    L.icpb_compose_chain_device.argtypes = [vp, dp, dp, i64, dp, vp]
    L.icpb_compose_chain_gpu.argtypes = [vp, dp, dp, i64, dp]
    L.icpb_pose_graph_sgd.argtypes = [vp, dp, i64, i32p, dp, i64, dp, ctypes.c_int32, ctypes.c_double]
    L.icpb_occupancy_grid_bounds.argtypes = [vp, dp, i64, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                             ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                             ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]
    L.icpb_occupancy_grid_update.argtypes = [vp, dp, i64, vp, i64, i64, ctypes.c_double, ctypes.c_double,
                                             ctypes.c_double, ctypes.c_int32, ctypes.c_int32]
    L.icpb_fit_pairs_host.argtypes = [vp, dp, dp, i64, dp, dp]
    L.icpb_icp_pair_host.argtypes = [vp, dp, i64, dp, i64, dp, ctypes.POINTER(IcpbParams), dp, dp, i32p, dp, i32p]
    L.icpb_get_kernel_info.argtypes = [vp, i64, ctypes.POINTER(IcpbKernelInfo)]
    L.icpb_launch_count.argtypes = [vp]
    L.icpb_launch_count.restype = ctypes.c_int64
    L.icpb_scan_count.argtypes = [vp]
    L.icpb_scan_count.restype = ctypes.c_int64
    L.icpb_last_error.restype = ctypes.c_char_p
    L.icpb_count_work.argtypes = [vp, ctypes.c_int]
    L.icpb_read_work.argtypes = [vp, ctypes.POINTER(ctypes.c_uint64)]
    for name in EXPORTS:
        getattr(L, name)
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().icpb_last_error().decode("utf-8", "replace")
        if rc in (10001, 10002):
            raise ValueError(f"{what}: {msg}")
        raise IcpbError(f"{what}: status {rc}: {msg}")


def default_params() -> IcpbParams:
    p = IcpbParams()
    lib().icpb_default_params(ctypes.byref(p))
    return p
