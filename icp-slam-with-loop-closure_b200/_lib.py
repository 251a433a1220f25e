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


# Every export of include/icpb.h, declared once: name -> (restype, argtypes).  Pointers are void *: numpy
# arrays go in through `ptr`, torch tensors as c_void_p(t.data_ptr()), out-scalars through ctypes.byref.
_v, _i, _i32, _i64, _f64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int32, ctypes.c_int64, ctypes.c_double
_P, _E = ctypes.POINTER(IcpbParams), ctypes.POINTER(IcpbEpilogue)
_f64p, _i64p = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64)
SIGNATURES = {
    "icpb_default_params": (None, [_P]),
    "icpb_abi_version": (_i, []),
    "icpb_create": (_i, [_i, ctypes.POINTER(_v)]),
    "icpb_destroy": (_i, [_v]),
    "icpb_upload_scans": (_i, [_v, _v, _v, _i64]),
    "icpb_set_scans_device": (_i, [_v, _v, _v, _i64, _i64]),
    "icpb_set_submaps": (_i, [_v, _v, _v, _v, _i64]),
    "icpb_set_submaps_voxel": (_i, [_v, _v, _v, _v, _i64, _f64, _v]),
    "icpb_read_scans": (_i, [_v, _i64, _i64, _v]),
    "icpb_run_device": (_i, [_v, _v, _v, _i64, _P, _v, _v, _v, _v, _v, _v]),
    "icpb_run_device_gather": (_i, [_v, _v, _v, _i64, _P, _v, _v, _v, _v, _i32, _i64, _v]),
    "icpb_run_device_ex": (_i, [_v, _v, _v, _i64, _P, _v, _v, _v, _E, _v]),
    "icpb_run_host": (_i, [_v, _v, _v, _i64, _P, _v, _v, _v, _v, _v]),
    "icpb_run_multistart_host": (_i, [_v, _v, _v, _i64, _v, _i32, _P, _v, _v, _v, _v, _v, _v]),
    "icpb_align_host": (_i, [_v, _v, _v, _i64, _v, _v, _i64, _P, _v, _v, _v]),
    "icpb_plan_upload": (_i, [_v, _i64, _i32, _v, _v]),
    "icpb_align_host_ld": (_i, [_v, _v, _v, _i64, _v, _v, _i32, _i64, _P, _v, _i32, _v, _v]),
    "icpb_align_host_ex": (_i, [_v, _v, _v, _i64, _v, _v, _i32, _i64, _P, _v, _i32, _v, _v, _E]),
    "icpb_align_host_scans": (_i, [_v, _v, _v, _i64, _v, _v, _i32, _i64, _P, _v, _i32, _v, _v, _E]),
    "icpb_align_host_accept": (_i, [_v, _v, _v, _v, _v, _i64, _v, _v, _i32, _i64, _P, _f64, _i64, _i64p,
                                    _v, _v, _i32, _v, _v]),
    "icpb_icp_pair_host": (_i, [_v, _v, _i64, _v, _i64, _v, _P, _v, _v, _v, _v, _v]),
    "icpb_fit_pairs_host": (_i, [_v, _v, _v, _i64, _v, _v]),
    "icpb_proximity_closest": (_i, [_v, _v, _v, _i64, _f64, _f64, _v, _v]),
    "icpb_proximity_pairs": (_i, [_v, _v, _v, _i64, _f64, _f64, _i64, _v, _i64p]),
    "icpb_compose_chain": (_i, [_v, _v, _i64, _v]),
    "icpb_compose_chain_device": (_i, [_v, _v, _v, _i64, _v, _v]),
    "icpb_compose_chain_gpu": (_i, [_v, _v, _v, _i64, _v]),
    "icpb_pose_graph_sgd": (_i, [_v, _v, _i64, _v, _v, _i64, _v, _i32, _f64]),
    "icpb_occupancy_grid_bounds": (_i, [_v, _v, _i64, _f64, _f64, _f64, _f64p, _f64p, _i64p, _i64p]),
    "icpb_occupancy_grid_update": (_i, [_v, _v, _i64, _v, _i64, _i64, _f64, _f64, _f64, _i32, _i32]),
    "icpb_get_kernel_info": (_i, [_v, _i64, ctypes.POINTER(IcpbKernelInfo)]),
    "icpb_set_tuning": (_i, [_v, ctypes.c_char_p, _i64]),
    "icpb_launch_count": (_i64, [_v]),
    "icpb_scan_count": (_i64, [_v]),
    "icpb_count_work": (_i, [_v, _i]),
    "icpb_read_work": (_i, [_v, ctypes.POINTER(ctypes.c_uint64)]),
    "icpb_last_error": (ctypes.c_char_p, []),
}
EXPORTS = list(SIGNATURES)


def ptr(a):
    """A numpy array's data as a void * argument (None stays a null pointer)."""
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def sources():
    c = os.path.join(_HERE, "csrc")
    return [os.path.join(c, "icpb_api.cu")], [os.path.join(c, "icpb_kernels.cuh"),
                                              os.path.join(c, "icpb_candidates.cuh"),
                                              os.path.join(c, "icpb_sgd.cuh"),
                                              os.path.join(c, "icpb_grid.cuh"),
                                              os.path.join(c, "icpb_compose.cuh"),
                                              os.path.join(c, "icpb_multistart.cuh"),
                                              os.path.join(c, "icpb_submaps.cuh"),
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
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = restype, argtypes
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
