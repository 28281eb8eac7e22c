"""TEST INFRASTRUCTURE — ctypes front-end of the softmax-exploration oracle (tests/softmax_oracle.c). Not part of the product path.

``SoftmaxOracle(compiled, n_instances, temperature)`` is an ``oracle.Oracle`` (same state arrays, same reset / step / update)
whose ``select_action`` and ``train`` select with rlrm_set_exploration's softmax rule. ``exp`` and ``softmax_thresholds`` expose
the rule's exp and thresholds. The library is compiled with gcc on first use into a temporary directory keyed by the sources.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SOURCES = [os.path.join(_HERE, "softmax_oracle.c"), os.path.join(_ROOT, "oracle", "rlrm_oracle.c"),
            os.path.join(_ROOT, "include", "rlrm_b200.h")]
_CFLAGS = ["-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-std=c11"]
_libs = {}


def lib(real="f32"):
    if real not in _libs:
        key = hashlib.sha256(b"".join(open(p, "rb").read() for p in _SOURCES)).hexdigest()[:16]
        out_dir = os.path.join(tempfile.gettempdir(), f"rlrm_softmax_oracle_{os.getuid()}_{key}")
        path = os.path.join(out_dir, f"libsoftmax_oracle_{real}.so")
        if not os.path.exists(path):
            os.makedirs(out_dir, exist_ok=True)
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run([os.environ.get("CC", "gcc"), *_CFLAGS, f"-DORACLE_REAL={'float' if real == 'f32' else 'double'}",
                            "-o", tmp, _SOURCES[0], "-lm"], check=True, capture_output=True)
            os.replace(tmp, path)  # several test processes may build at once: each writes its own file, the rename is atomic
        L = C.CDLL(path)
        assert L.oracle_real_size() == (4 if real == "f32" else 8)
        _libs[real] = L
    return _libs[real]


def _p(arr):
    return None if arr is None else arr.ctypes.data


def exp(x):
    """rlrm_exp (x <= 0), the exp of the softmax rule; elementwise over an array"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    lib("f64").softmax_exp_array(C.c_int64(x.size), C.c_void_p(_p(x)), C.c_void_p(_p(out)))
    return out


def softmax_thresholds(row, temperature, real="f32"):
    """T_j = ceil(C_j / total * 2^32), j < n - 1, of the softmax rule on the action values `row` (n = len(row)) in the table type
    `real`; the selected action is #{j : w1 >= T_j}"""
    r = np.ascontiguousarray(row, dtype=np.float32 if real == "f32" else np.float64)
    thr = np.zeros(4, dtype=np.uint64)
    n = lib(real).softmax_thresholds(C.c_void_p(_p(r)), C.c_int(r.size), C.c_double(1.0 / float(temperature)), C.c_void_p(_p(thr)))
    return thr[:n].copy()


class SoftmaxOracle(O.Oracle):
    def __init__(self, compiled, n_instances, temperature, real=None, track_visits=False):
        super().__init__(compiled, n_instances, real=real, track_visits=track_visits)
        self.beta = 1.0 / float(temperature)
        self.S_L = lib(self.real)

    def select_action(self, t=0, draws=None, best=False):
        out = np.zeros(self.N * self.A, dtype=np.uint8)
        d = None if draws is None else np.ascontiguousarray(draws, dtype=np.uint32)
        self.S_L.softmax_select_action(C.byref(self.cfg), C.byref(self.tables), C.byref(self.state), C.c_void_p(_p(d)),
                                       C.c_uint64(t), C.c_int(int(best)), C.c_double(self.beta), C.c_void_p(_p(out)))
        return out.reshape(self.N, self.A)

    def train(self, t0, n_iters, learn=True, trace=False):
        tr = np.zeros((n_iters, self.N * self.A), dtype=np.uint32) if trace else None
        rc = self.S_L.softmax_train(C.byref(self.cfg), C.byref(self.tables), C.byref(self.state), C.c_uint64(t0),
                                    C.c_int32(n_iters), C.c_int32(int(learn)), C.c_void_p(_p(tr)), C.c_double(self.beta))
        assert rc == 0, "softmax exploration needs per-instance tables"
        return tr
