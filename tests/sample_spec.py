"""Specification of sample(state, n; replace) (include/wsb200.h, above ws_sample_indices) in Python big integers.

The integer weights q_i and the key images come from the host instantiation of the device routines
(csrc/ws_math.cuh: ws_sample_q, ws_sample_key, through tests/host/sample_harness.cpp), so they match the device bit for bit;
the sums, the targets t_k and the selection are exact integer arithmetic here."""
import bisect
import ctypes as C
import hashlib
import itertools
import os
import subprocess
import tempfile

import numpy as np

from oracle import ref

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host", "sample_harness.cpp")
MATH = os.path.join(HERE, "..", "weightedsampling.jl_b200", "csrc", "ws_math.cuh")
_L = None


def _lib():
    """tests/host/sample_harness.cpp built with g++ into a temporary directory (the tree may be read-only), once per
    version of its sources"""
    global _L
    if _L is None:
        h = hashlib.sha256()
        for f in (SRC, MATH):
            with open(f, "rb") as fh:
                h.update(fh.read())
        so = os.path.join(tempfile.gettempdir(), f"wsb200_sample_harness_{h.hexdigest()[:16]}_{os.getuid()}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", tmp, SRC], check=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.hh_sample_q.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_void_p]
        L.hh_sample_targets.argtypes = [C.c_int64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]
        L.hh_sample_keys.argtypes = [C.c_void_p, C.c_int64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]
        _L = L
    return _L


def max_logw(logw):
    """m = the largest log-weight; ValueError where the device returns WS_ENUMERIC"""
    a = np.asarray(logw, dtype=np.float64)
    fin = a[~np.isnan(a)]
    m = float(fin.max()) if fin.size else -np.inf
    if not np.isfinite(m):
        raise ValueError(f"the largest log-weight is {m}")
    return m


def sample_q(logw, m):
    a = np.ascontiguousarray(logw, dtype=np.float64)
    out = np.empty(a.size, dtype=np.uint64)
    _lib().hh_sample_q(a.ctypes.data_as(C.c_void_p), a.size, m, out.ctypes.data_as(C.c_void_p))
    return out


def sample_keys(logw, seed, stream, first=0):
    a = np.ascontiguousarray(logw, dtype=np.float64)
    out = np.empty(a.size, dtype=np.uint64)
    _lib().hh_sample_keys(a.ctypes.data_as(C.c_void_p), a.size, first, stream, seed, out.ctypes.data_as(C.c_void_p))
    return out


def sample_targets_harness(n, seed, stream, T):
    """t_k from the host instantiation of ws_sample_target (checked against `targets`)"""
    out = np.empty(2 * n, dtype=np.uint64)
    _lib().hh_sample_targets(n, stream, seed, T >> 64, T & (2 ** 64 - 1), out.ctypes.data_as(C.c_void_p))
    return [(int(out[2 * k]) << 64) | int(out[2 * k + 1]) for k in range(n)]


def philox_r128(n, seed, stream):
    x, y, z, w = ref.philox4x32_10(np.arange(n, dtype=np.uint64), stream, seed)
    return [(int(a) << 96) | (int(b) << 64) | (int(c) << 32) | int(d) for a, b, c, d in zip(x, y, z, w)]


def targets(n, seed, stream, T):
    """t_k = floor(r_k T / 2^128)"""
    return [(r * T) >> 128 for r in philox_r128(n, seed, stream)]


def select_top(keys, n):
    """the n largest key images in descending order, equal keys to the lower index"""
    keys = np.asarray(keys, dtype=np.uint64)
    order = np.lexsort((np.arange(keys.size), ~keys))
    return order[:n].astype(np.int64)


def sample_indices_spec(logw, seed, stream, n, replace):
    """0-based indices of the draw (GLOBAL indices: `logw` is the whole, unsharded log-weight vector)"""
    m = max_logw(logw)
    if replace:
        q = [int(v) for v in sample_q(logw, m).tolist()]
        Q = list(itertools.accumulate(q))
        T = Q[-1]
        return np.array([bisect.bisect_right(Q, t) for t in targets(n, seed, stream, T)], dtype=np.int64)
    if n > len(logw):
        raise ValueError("n > N without replacement")
    return select_top(sample_keys(logw, seed, stream), n)
