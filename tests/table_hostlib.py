"""ctypes wrapper of tests/host/table_harness.cpp: the product's lowering and micro-op interpreter on the CPU, with
tables (test infrastructure).  The shared object is compiled into a temporary directory."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host", "table_harness.cpp")
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="ws_table_harness_"), "table_harness.so")
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", out, SRC], check=True)
        L = C.CDLL(out)
        L.th_new.restype = C.c_void_p
        L.th_new.argtypes = [C.c_int64, C.c_uint64]
        L.th_error.restype = C.c_char_p
        L.th_index_faults.restype = C.c_int64
        for name in ("th_free", "th_error", "th_flush", "th_index_faults", "th_window_ops", "th_score_ops"):
            getattr(L, name).argtypes = [C.c_void_p]
        L.th_col.argtypes = [C.c_void_p, C.c_int]
        L.th_set_plane.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.th_get_plane.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.th_get_logw.argtypes = [C.c_void_p, C.c_void_p]
        L.th_set_replay_uniforms.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.th_table.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.POINTER(C.c_int32)]
        L.th_score.argtypes = [C.c_void_p, C.c_void_p]
        L.th_sample_expr.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


class TableHostStore:
    """Duck-types what the Python front-end needs of DeviceColumnStore (`_lookup`, `_ensure`, `_call`, `_table_id`)."""

    def __init__(self, n, seed=0):
        self.L = lib()
        self.h = C.c_void_p(self.L.th_new(n, seed))
        self.n = n
        self.names, self.widths, self._keep, self._tables = {}, [], [], {}

    def __del__(self):
        if getattr(self, "h", None):
            self.L.th_free(self.h)

    def _lookup(self, name):
        if name in self.names:
            return self.names[name], self.widths[self.names[name]]
        return -1, 0

    def _ensure(self, name, width):
        if name not in self.names:
            self.names[name] = self.L.th_col(self.h, width)
            self.widths.append(width)
        return self.names[name]

    def colnames(self):
        return list(self.names)

    def _table_id(self, tab):
        key = (tab.values.shape, tab.values.tobytes())
        if key not in self._tables:
            tid = C.c_int32()
            assert self.L.th_table(self.h, tab.values.ctypes.data_as(C.c_void_p), tab.values.shape[0], tab.values.shape[1],
                                   C.byref(tid)) == 0
            self._tables[key] = tid.value
        return self._tables[key]

    def _call(self, fn, *args):
        if fn == "ws_resample_async":
            return      # the harness has no resampler: a Resample step never fires here (as with ess_perc_min = 0)
        name = {"ws_assign": "th_assign", "ws_observe_normal": "th_observe_normal", "ws_weight_expr": "th_weight_expr",
                "ws_sample_expr": "th_sample_expr"}[fn]
        rc = getattr(self.L, name)(self.h, *args)
        if rc != 0:
            raise RuntimeError(f"{name} failed ({rc}): {self.L.th_error(self.h).decode()}")

    def setcol(self, name, v):
        v = np.ascontiguousarray(v, dtype=np.float64)
        self.L.th_set_plane(self.h, self._ensure(name, 1), 0, v.ctypes.data_as(C.c_void_p))

    def getcol(self, name):
        out = np.empty(self.n)
        self.L.th_get_plane(self.h, self.names[name], 0, out.ctypes.data_as(C.c_void_p))
        return out

    def logw(self):
        out = np.empty(self.n)
        self.L.th_get_logw(self.h, out.ctypes.data_as(C.c_void_p))
        return out

    def score(self):
        out = np.empty(self.n)
        assert self.L.th_score(self.h, out.ctypes.data_as(C.c_void_p)) == 0
        return out

    def set_uniforms(self, u):
        self._u = np.ascontiguousarray(u, dtype=np.float64)
        self.L.th_set_replay_uniforms(self.h, self._u.ctypes.data_as(C.c_void_p), self._u.size)

    def index_faults(self):
        return self.L.th_index_faults(self.h)

    def window_ops(self):
        return self.L.th_window_ops(self.h)


class TableHostState:
    """Minimal SMCState stand-in so that core.Assign / Sample / Observe / Weight.apply run unchanged."""

    def __init__(self, n, seed=0):
        self.store = TableHostStore(n, seed)
        self.resampled = False
