"""ctypes binding of libgnnpp_b200.so (C ABI in include/gnnpp_b200.h) + in-tree build.

There is NO CPU fallback: if the shared library is missing, cannot be loaded, or a
call fails, a RuntimeError (or AssertionError for shape errors, matching the
reference's `assert`s) is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libgnnpp_b200.so")
SOURCES = ("graph_filter.cu", "graph_filter_tc.cu", "graph_filter_pair.cu", "graph_filter_small.cu", "rollout.cu", "evaluate.cu", "dataset.cu", "feature.cu", "feature_tc.cu", "feature_mma.cu", "train.cu", "planner.cu")
HEADERS = ("common.cuh", "feature.cuh", "tc_common.cuh", "step_inputs.cuh")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include", "gnnpp_b200.h")
INCLUDE_DEBUG = os.path.join(os.path.dirname(PKG_DIR), "include", "gnnpp_b200_debug.h")

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared",
]

GPP_OK = 0
GPP_ERR_INVALID = -1
GPP_ERR_UNSUPPORTED = -2
FEATURE_MAJOR = 0   # [B, G, N]  (reference API layout)
NODE_MAJOR = 1      # [B, N, G]

# every symbol include/gnnpp_b200.h declares
EXPORTED = (
    "gpp_last_error", "gpp_abi_version", "gpp_device_info",
    "gpp_graph_filter_workspace_bytes", "gpp_graph_filter_forward",
    "gpp_graph_filter_backward_workspace_bytes", "gpp_graph_filter_backward",
    "gpp_planner_create", "gpp_planner_destroy", "gpp_planner_set_weights",
    "gpp_planner_forward", "gpp_planner_forward_host",
    "gpp_planner_train_workspace_bytes", "gpp_planner_train_forward", "gpp_planner_train_backward", "gpp_planner_ce_loss", "gpp_rollout_build_inputs", "gpp_rollout_move",
    "gpp_rollout_targets", "gpp_rollout_track", "gpp_rollout_evaluate_finish",
    "gpp_dataset_prepare", "gpp_dataset_batch",
    "gpp_planner_forward_host_async", "gpp_planner_wait", "gpp_planner_forward_async", "gpp_planner_join",
    "gpp_planner_set_profiling", "gpp_planner_get_profile",
    "gpp_planner_set_graph_filter_mode", "gpp_planner_set_feature_mode",
    "gpp_launch_count", "gpp_reset_launch_count",
)
# test / profiling hooks declared in include/gnnpp_b200_debug.h (not part of the drop-in boundary)
DEBUG_EXPORTED = (
    "gpp_debug_set_option", "gpp_debug_umma_selftest", "gpp_debug_tc_timing", "gpp_debug_pair_timing", "gpp_debug_gf_timing",
    "gpp_debug_feature_tc_timing", "gpp_debug_feature_mma_timing", "gpp_debug_feature_timing", "gpp_debug_train_kernel",
)


class PlannerWeights(C.Structure):
    _fields_ = [
        ("conv_w", C.c_void_p * 5), ("conv_b", C.c_void_p * 5),
        ("bn_w", C.c_void_p * 5), ("bn_b", C.c_void_p * 5),
        ("bn_mean", C.c_void_p * 5), ("bn_var", C.c_void_p * 5),
        ("compress_w", C.c_void_p), ("compress_b", C.c_void_p),
        ("gf_w", C.c_void_p), ("gf_b", C.c_void_p),
        ("action_w", C.c_void_p), ("action_b", C.c_void_p),
    ]


class PlannerBnState(C.Structure):
    _fields_ = [("running_mean", C.c_void_p * 5), ("running_var", C.c_void_p * 5)]


class PlannerGrads(C.Structure):
    _fields_ = [
        ("conv_w", C.c_void_p * 5), ("conv_b", C.c_void_p * 5),
        ("bn_w", C.c_void_p * 5), ("bn_b", C.c_void_p * 5),
        ("compress_w", C.c_void_p), ("compress_b", C.c_void_p),
        ("gf_w", C.c_void_p), ("gf_b", C.c_void_p),
        ("action_w", C.c_void_p), ("action_b", C.c_void_p),
    ]


OBJ_DIR = os.path.join(CSRC_DIR, "build")


def _newer(path: str, deps) -> bool:
    """True if `path` is missing or older than any dependency."""
    if not os.path.isfile(path):
        return True
    t = os.path.getmtime(path)
    return any(os.path.getmtime(d) > t for d in deps if os.path.isfile(d))


def _stale() -> bool:
    deps = [os.path.join(CSRC_DIR, s) for s in SOURCES + HEADERS] + [INCLUDE, INCLUDE_DEBUG]
    return _newer(LIB_PATH, deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compiles the CUDA sources for sm_100a into the in-tree shared library: one nvcc -c per
    translation unit (in parallel, only the stale ones), then one link."""
    if not force and not _stale():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdrs = [os.path.join(CSRC_DIR, h) for h in HEADERS] + [INCLUDE, INCLUDE_DEBUG]
    flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, src[:-3] + ".o")
        path = os.path.join(CSRC_DIR, src)
        if force or _newer(obj, [path] + hdrs):
            cmd = [nvcc] + flags + ["-c", "-o", obj, path]
            if verbose:
                print(" ".join(cmd))
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed on %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + objs
    if verbose:
        print(" ".join(cmd))
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB_PATH


_lib = None
_lock = threading.Lock()


def load():
    """Returns the loaded library; raises RuntimeError if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                "gnn_pathplanning_b200: %s is missing -- build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
                "There is no CPU fallback for this package." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        vp, i, sz = C.c_void_p, C.c_int, C.c_size_t
        lib.gpp_last_error.restype = C.c_char_p
        lib.gpp_last_error.argtypes = []
        lib.gpp_abi_version.restype = i
        lib.gpp_device_info.argtypes = [C.POINTER(i)] * 3
        lib.gpp_graph_filter_workspace_bytes.restype = sz
        lib.gpp_graph_filter_workspace_bytes.argtypes = [i, i, i]
        lib.gpp_graph_filter_forward.restype = i
        lib.gpp_graph_filter_forward.argtypes = [vp, vp, i, vp, vp, vp, i, i, i, i, i, i, i, i, vp, vp]
        lib.gpp_graph_filter_backward_workspace_bytes.restype = sz
        lib.gpp_graph_filter_backward_workspace_bytes.argtypes = [i, i, i, i, i]
        lib.gpp_graph_filter_backward.restype = i
        lib.gpp_graph_filter_backward.argtypes = [vp, vp, vp, vp, i, vp, vp, vp, vp,
                                                  i, i, i, i, i, i, i, i, vp, vp]
        lib.gpp_planner_create.restype = i
        lib.gpp_planner_create.argtypes = [C.POINTER(vp), i]
        lib.gpp_planner_destroy.restype = None
        lib.gpp_planner_destroy.argtypes = [vp]
        lib.gpp_planner_set_weights.restype = i
        lib.gpp_planner_set_weights.argtypes = [vp, C.POINTER(PlannerWeights), i, vp]
        lib.gpp_planner_forward.restype = i
        lib.gpp_planner_forward.argtypes = [vp, vp, vp, i, vp, vp, i, i, vp]
        lib.gpp_planner_forward_host.restype = i
        lib.gpp_planner_forward_host.argtypes = [vp, vp, vp, i, vp, i, i]
        lib.gpp_planner_train_workspace_bytes.restype = sz
        lib.gpp_planner_train_workspace_bytes.argtypes = [i, i, i]
        lib.gpp_planner_train_forward.restype = i
        lib.gpp_planner_train_forward.argtypes = [C.POINTER(PlannerWeights), C.POINTER(PlannerBnState), C.c_float,
                                                  vp, vp, i, vp, vp, i, i, i, vp]
        lib.gpp_planner_train_backward.restype = i
        lib.gpp_planner_train_backward.argtypes = [C.POINTER(PlannerWeights), vp, vp, i, vp, vp,
                                                   C.POINTER(PlannerGrads), i, i, i, vp]
        lib.gpp_planner_ce_loss.restype = i
        lib.gpp_planner_ce_loss.argtypes = [vp, vp, i, vp, vp, C.c_float, i, i, vp]
        lib.gpp_rollout_build_inputs.restype = i
        lib.gpp_rollout_build_inputs.argtypes = [vp, vp, vp, i, vp, i, vp, vp, i, vp, i, i, i, vp]
        lib.gpp_rollout_move.restype = i
        lib.gpp_rollout_move.argtypes = [vp, vp, vp, vp, i, vp, vp, vp, vp, vp, vp, vp, vp, i, i, i, i, vp]
        lib.gpp_rollout_targets.restype = i
        lib.gpp_rollout_targets.argtypes = [vp, vp, vp, vp, vp, vp, i, i, i, vp]
        lib.gpp_rollout_track.restype = i
        lib.gpp_rollout_track.argtypes = [vp, vp, vp, vp, i, i, vp]
        lib.gpp_rollout_evaluate_finish.restype = i
        lib.gpp_rollout_evaluate_finish.argtypes = [vp, vp, vp, vp, vp, vp, vp, i, i, vp]
        lib.gpp_dataset_prepare.restype = i
        lib.gpp_dataset_prepare.argtypes = [vp, vp, C.c_double, vp, i, i, vp]
        lib.gpp_dataset_batch.restype = i
        lib.gpp_dataset_batch.argtypes = [vp, vp, vp, vp, vp, i, vp, vp, vp, vp, vp, i, i, i, i, vp]
        lib.gpp_planner_forward_host_async.restype = i
        lib.gpp_planner_forward_host_async.argtypes = [vp, vp, vp, i, vp, i, i, C.POINTER(C.c_ulonglong)]
        lib.gpp_planner_wait.restype = i
        lib.gpp_planner_wait.argtypes = [vp, C.c_ulonglong]
        lib.gpp_planner_forward_async.restype = i
        lib.gpp_planner_forward_async.argtypes = [vp, vp, vp, i, vp, i, i, vp, C.POINTER(C.c_ulonglong)]
        lib.gpp_planner_join.restype = i
        lib.gpp_planner_join.argtypes = [vp, C.c_ulonglong, vp]
        lib.gpp_debug_tc_timing.restype = i
        lib.gpp_debug_tc_timing.argtypes = [C.POINTER(C.c_ulonglong)]
        lib.gpp_debug_pair_timing.restype = i
        lib.gpp_debug_pair_timing.argtypes = [C.POINTER(C.c_ulonglong)]
        lib.gpp_debug_gf_timing.restype = i
        lib.gpp_debug_gf_timing.argtypes = [C.POINTER(C.c_ulonglong)]
        lib.gpp_debug_feature_timing.restype = i
        lib.gpp_debug_feature_timing.argtypes = [C.POINTER(C.c_ulonglong)]
        lib.gpp_debug_feature_tc_timing.restype = i
        lib.gpp_debug_feature_mma_timing.restype = i
        lib.gpp_debug_feature_mma_timing.argtypes = [C.POINTER(C.c_ulonglong)]
        lib.gpp_debug_feature_tc_timing.argtypes = [C.POINTER(C.c_ulonglong)]
        lib.gpp_planner_set_profiling.restype = i
        lib.gpp_planner_set_profiling.argtypes = [vp, i]
        lib.gpp_planner_get_profile.restype = i
        lib.gpp_planner_get_profile.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i)]
        lib.gpp_planner_set_graph_filter_mode.restype = i
        lib.gpp_planner_set_graph_filter_mode.argtypes = [vp, i]
        lib.gpp_planner_set_feature_mode.restype = i
        lib.gpp_planner_set_feature_mode.argtypes = [vp, i]
        lib.gpp_debug_set_option.restype = i
        lib.gpp_debug_set_option.argtypes = [C.c_char_p, i]
        lib.gpp_debug_train_kernel.restype = i
        lib.gpp_debug_train_kernel.argtypes = [i, vp, vp, vp, vp, i, i, i, i, vp]
        lib.gpp_debug_umma_selftest.restype = i
        lib.gpp_debug_umma_selftest.argtypes = [vp, vp, vp, vp]
        lib.gpp_launch_count.restype = C.c_ulonglong
        lib.gpp_launch_count.argtypes = []
        lib.gpp_reset_launch_count.restype = None
        lib.gpp_reset_launch_count.argtypes = []
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc == GPP_OK:
        return
    msg = load().gpp_last_error().decode("utf-8", "replace")
    if rc == GPP_ERR_INVALID:
        raise AssertionError("libgnnpp_b200: " + msg)
    if rc == GPP_ERR_UNSUPPORTED:
        raise NotImplementedError("libgnnpp_b200: " + msg)
    raise RuntimeError("libgnnpp_b200 (status %d): %s" % (rc, msg))


def set_debug_option(name: str, value: int) -> None:
    """Process-wide debug switch of the library (include/gnnpp_b200_debug.h)."""
    check(load().gpp_debug_set_option(name.encode(), int(value)))


def launch_count() -> int:
    return int(load().gpp_launch_count())


def reset_launch_count() -> None:
    load().gpp_reset_launch_count()
