"""Build + load the CUDA C-ABI library (csrc/rlrm_b200.cu -> librlrm_b200.so, in-tree).

There is no CPU fallback: :func:`load` raises if the shared library is missing or a symbol of
include/rlrm_b200.h is not exported, and ``rlrm_create`` itself fails without a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

from . import _abi as abi

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
# RLRM_LIB_PATH: load an alternative build of the library (kernel tuning A/B runs); the default is the in-tree build
LIB_PATH = os.environ.get("RLRM_LIB_PATH") or os.path.join(_PKG, "librlrm_b200.so")
SOURCES = [os.path.join(_PKG, "csrc", "rlrm_b200.cu")]
HEADERS = [os.path.join(_ROOT, "include", "rlrm_b200.h")] + sorted(
    os.path.join(_PKG, "csrc", f) for f in os.listdir(os.path.join(_PKG, "csrc")) if f.endswith(".cuh"))
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC"]

_lib = None


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(f) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    """nvcc cross-compiles for sm_100a; works without a GPU. Serialised with a file lock so that several ranks of one
    job (torchrun) never compile into the same file at once; the library is written to a temporary name and renamed."""
    import fcntl

    with open(LIB_PATH + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if force or is_stale():
                tmp = f"{LIB_PATH}.{os.getpid()}.tmp"
                cmd = [_nvcc(), *NVCC_FLAGS, "-o", tmp, *SOURCES]
                if verbose:
                    cmd.insert(1, "-Xptxas=-v")
                res = subprocess.run(cmd, capture_output=True, text=True)
                if res.returncode != 0:
                    raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
                os.replace(tmp, LIB_PATH)
                if verbose:
                    print(res.stderr)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


def load():
    """ctypes handle with argtypes set; raises RuntimeError when the extension is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if is_stale() and os.path.exists(_nvcc()):
        build()  # missing or older than its sources: rebuild in-tree (there is still no CPU fallback)
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "multiagent-rl-rm_b200 has no CPU fallback."
        )
    L = C.CDLL(LIB_PATH)
    missing = [s for s in abi.EXPORTED_SYMBOLS if not hasattr(L, s)]
    if missing:
        raise RuntimeError(f"{LIB_PATH} does not export {missing}")
    vp, u64, i32, i64 = C.c_void_p, C.c_uint64, C.c_int32, C.c_int64
    L.rlrm_abi_version.restype = C.c_int
    L.rlrm_last_error.restype = C.c_char_p
    L.rlrm_device_count.restype = C.c_int
    L.rlrm_create.argtypes = [C.POINTER(abi.Config), C.POINTER(abi.Tables), C.c_int, C.POINTER(vp)]
    L.rlrm_destroy.argtypes = [vp]
    L.rlrm_set_learner.argtypes = [vp, C.c_double, C.c_double, C.c_double]
    L.rlrm_set_sweep.argtypes = [vp, C.POINTER(abi.Hyper), i32, i64]
    L.rlrm_reset.argtypes = [vp, C.POINTER(abi.State), vp, vp]
    L.rlrm_reset_at.argtypes = [vp, C.POINTER(abi.State), vp, u64, vp]
    L.rlrm_select_action.argtypes = [vp, C.POINTER(abi.State), vp, u64, C.c_int, vp, vp]
    L.rlrm_step.argtypes = [vp, C.POINTER(abi.State), vp, vp, u64, C.c_int, C.POINTER(abi.StepOut), vp]
    L.rlrm_rm_step.argtypes = [vp, i64, vp, vp, vp, vp, vp]
    L.rlrm_rm_step_agent.argtypes = [vp, C.c_int, i64, vp, vp, vp, vp, vp]
    L.rlrm_mdp.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int, vp, vp, vp, vp, vp]
    L.rlrm_value_iteration.argtypes = [C.c_int, i64, C.c_int, vp, vp, vp, vp, C.c_double, C.c_double, C.c_int, C.c_int, vp, vp, vp, vp,
                                       C.POINTER(C.c_int32), vp]
    L.rlrm_update.argtypes = [vp, C.POINTER(abi.State), vp, vp, vp, C.POINTER(abi.StepOut), vp]
    L.rlrm_train.argtypes = [vp, C.POINTER(abi.State), u64, i32, i32, vp, vp]
    L.rlrm_train_host.argtypes = [vp, C.POINTER(abi.State), u64, i32, i32, vp, vp, vp, vp]
    L.rlrm_evaluate.argtypes = [vp, C.POINTER(abi.State), vp, u64, i32, i32, C.c_double, C.c_double, vp]
    L.rlrm_qlambda_materialize.argtypes = [vp, C.POINTER(abi.State), vp, vp]
    L.rlrm_iterate.argtypes = [vp, C.POINTER(abi.State), u64, i32, vp, vp, vp]
    L.rlrm_update_list.argtypes = [vp, C.POINTER(abi.State), i64, i32, vp, vp]
    L.rlrm_update_list_select.argtypes = [vp, C.POINTER(abi.State), i64, i32, vp, vp, vp]
    L.rlrm_merge_replicas.argtypes = [vp, vp, i32, i64, vp, vp]
    L.rlrm_stream_sync.argtypes = [vp, vp]
    L.rlrm_probe_random_gather.argtypes = [C.c_int, vp, i64, i32, i64, i32, vp, vp]
    L.rlrm_launch_count.argtypes = [vp]
    L.rlrm_launch_count.restype = i64
    for name in ("rlrm_create", "rlrm_destroy", "rlrm_set_learner", "rlrm_set_sweep", "rlrm_reset", "rlrm_reset_at", "rlrm_select_action", "rlrm_step",
                 "rlrm_rm_step", "rlrm_rm_step_agent", "rlrm_mdp", "rlrm_value_iteration", "rlrm_update", "rlrm_train", "rlrm_train_host", "rlrm_evaluate", "rlrm_qlambda_materialize",
                 "rlrm_iterate", "rlrm_update_list", "rlrm_update_list_select", "rlrm_merge_replicas", "rlrm_stream_sync", "rlrm_probe_random_gather"):
        getattr(L, name).restype = C.c_int
    if L.rlrm_abi_version() != abi.ABI_VERSION:
        raise RuntimeError("librlrm_b200.so ABI version mismatch: rebuild")
    _lib = L
    return L


class RlrmError(RuntimeError):
    pass


def check(rc: int):
    if rc != 0:
        raise RlrmError(f"rlrm error {rc}: {load().rlrm_last_error().decode()}")
