"""Post-run analysis surface (src/utils.jl): ``exp_norm``, ``expectation``, ``@E``, ``log_evidence``,
``sample``.  Reductions over the particles run on the device (``ws_exp_norm``, ``ws_expectation``,
``ws_log_evidence``, ``ws_sample_indices``); only their small results come back to the host.
"""
from __future__ import annotations

import ctypes as C
import inspect

import numpy as np

from . import _lib as L
from .core import SMCState
from .expr import CExprs, Col, lower


def _ctx_of(state_or_store):
    return state_or_store.store if isinstance(state_or_store, SMCState) else state_or_store


def exp_norm(weights, state=None):
    """``exp_norm(weights)`` (resampling.jl:72-77).

    ``exp_norm(state)`` normalises the state's own device-resident log-weights; ``exp_norm(array,
    state)`` runs the same kernels on a caller array (any length), using ``state``'s device/stream.
    """
    if isinstance(weights, SMCState):
        st = weights.store
        out = np.empty(st.n, dtype=np.float64)
        st._call("ws_exp_norm", out.ctypes.data_as(C.c_void_p))
        return out
    if state is None:
        raise TypeError("exp_norm(array) needs the SMCState whose device runs the kernel: exp_norm(array, state)")
    a = np.ascontiguousarray(weights, dtype=np.float64)
    out = np.empty_like(a)
    _ctx_of(state)._call("ws_exp_norm_host", a.ctypes.data_as(C.c_void_p), a.size, out.ctypes.data_as(C.c_void_p))
    return out


def logsumexp(logw, state):
    """``logsumexp(logw)`` (resampling.jl:61-64) on a caller array."""
    a = np.ascontiguousarray(logw, dtype=np.float64)
    out = C.c_double()
    _ctx_of(state)._call("ws_logsumexp_host", a.ctypes.data_as(C.c_void_p), a.size, C.byref(out))
    return out.value


def ess_perc(weights, state=None):
    """``ess_perc(w)`` (resampling.jl:51-54); ``ess_perc(state)`` for the state's own weights."""
    if isinstance(weights, SMCState):
        le, ess = C.c_double(), C.c_double()
        weights.store._call("ws_log_evidence", C.byref(le), C.byref(ess))
        return ess.value
    a = np.ascontiguousarray(weights, dtype=np.float64)
    out = C.c_double()
    _ctx_of(state)._call("ws_ess_perc_host", a.ctypes.data_as(C.c_void_p), a.size, C.byref(out))
    return out.value


def icdf(weights, us, state):
    """``icdf(weights, us)`` (resampling.jl:13-26); returns 0-based ancestor indices."""
    w = np.ascontiguousarray(weights, dtype=np.float64)
    u = np.ascontiguousarray(us, dtype=np.float64)
    if w.shape != u.shape:
        raise ValueError("weights and us must have the same length")
    out = np.empty(w.size, dtype=np.int32)
    nc = C.c_int64()
    _ctx_of(state)._call("ws_icdf_host", w.ctypes.data_as(C.c_void_p), u.ctypes.data_as(C.c_void_p), w.size,
                         out.ctypes.data_as(C.c_void_p), C.byref(nc))
    return out


def resample_indices(weights, state, scheme="stratified", uniforms=None, return_clamped=False):
    """``stratified_resample(weights)`` (resampling.jl:35-43) and the systematic / multinomial
    variants of SURVEY Appendix B, on a caller weight vector; 0-based indices.

    ``uniforms``: the raw r_n in [0,1) (n for stratified, 1 for systematic, n iid for multinomial);
    None draws them from Philox."""
    w = np.ascontiguousarray(weights, dtype=np.float64)
    out = np.empty(w.size, dtype=np.int32)
    nc = C.c_int64()
    up = None
    if uniforms is not None:
        u = np.ascontiguousarray(np.atleast_1d(uniforms), dtype=np.float64)
        up = u.ctypes.data_as(C.c_void_p)
    _ctx_of(state)._call("ws_resample_host", w.ctypes.data_as(C.c_void_p), w.size, L.RESAMPLER[scheme], up,
                         out.ctypes.data_as(C.c_void_p), C.byref(nc))
    return (out, nc.value) if return_clamped else out


def log_evidence(state):
    """``log_evidence(state) = logsumexp(weights) - log N`` (utils.jl:21)."""
    le, ess = C.c_double(), C.c_double()
    state.store._call("ws_log_evidence", C.byref(le), C.byref(ess))
    return le.value


def E(f, state):
    """``@E(f, state)`` (utils.jl:45-68): ``f``'s argument names are particle-variable names."""
    names = list(inspect.signature(f).parameters)
    val = f(*[Col(n) for n in names])
    return expectation(val, state)


def expectation(values, state):
    """``expectation(values, weights)`` (utils.jl:11) with ``values`` a particle expression (or a list
    of up to 8 of them, evaluated in one pass) and the weights those of ``state``."""
    st = state.store
    many = isinstance(values, (list, tuple))
    toks = []
    for v in (values if many else [values]):
        t = lower(v, st)
        if isinstance(t, list):
            raise TypeError("expectation of a vector-valued expression: index a component")
        toks.append(t)
    out = (C.c_double * len(toks))()
    ex = CExprs(toks)
    st._call("ws_expectation", ex.ptr(0), len(toks), out)
    return [out[i] for i in range(len(toks))] if many else out[0]


def sample(state, n, replace=True):
    """``sample(state, n; replace=true)`` (utils.jl:102-118) -> pandas DataFrame of n particles.

    The indices are drawn on the device (``ws_sample_indices``) and only the n drawn rows come to the host.  On a
    sharded state the call is collective: every rank must call it, and every rank gets the same DataFrame."""
    import pandas as pd
    st = state.store
    n = int(n)
    n_all = getattr(st, "n_global", st.n)
    if n <= 0:
        raise ValueError("Number of samples must be positive")
    if not replace and n > n_all:
        raise ValueError(f"Cannot sample {n} particles without replacement from {n_all} particles")
    idx = np.empty(n, dtype=np.int64)
    st._call("ws_sample_indices", n, int(bool(replace)), idx.ctypes.data_as(C.c_void_p))
    rows_call = "ws_col_download_global_rows" if getattr(st, "nranks", 1) > 1 else "ws_col_download_rows"
    data = {}
    for name in st.colnames():
        cid, width = st._lookup(name)
        rows = np.empty((width, n), dtype=np.float64)
        st._call(rows_call, cid, idx.ctypes.data_as(C.c_void_p), n, rows.ctypes.data_as(C.c_void_p))
        data[name] = rows[0] if width == 1 else list(np.ascontiguousarray(rows.T))
    return pd.DataFrame(data)


def to_dataframe(state):
    """``DataFrame(state)`` (utils.jl:83-88): every column plus ``log_weight``."""
    import pandas as pd
    st = state.store
    got = {}
    # newest columns first: a column that is several resampling events behind is read through the
    # composed ancestors, and the composition continues from the one made for the previous (newer) column
    for name in reversed(st.colnames()):
        v = st.getcol(name)
        got[name] = v if v.ndim == 1 else list(v)
    data = {name: got[name] for name in st.colnames()}
    data["log_weight"] = state.weights
    return pd.DataFrame(data)


_SPARK = "▁▂▃▄▅▆▇█"


def _sparkline(counts):
    """utils.jl:128-133: counts scaled so that the largest maps to a full block."""
    counts = np.asarray(counts, dtype=np.float64)
    mx = counts.max() if counts.size else 0.0
    if not (mx > 0):
        return _SPARK[0] * len(counts)
    lv = np.clip(np.ceil(counts / mx * len(_SPARK)).astype(int), 1, len(_SPARK))
    return "".join(_SPARK[k - 1] for k in lv)


def describe(state, cols=None):
    """``describe(state; cols=nothing)`` (utils.jl:183-289) -> DataFrame(variable, mean, median, std, min, max,
    hist, ess).  Every number is computed on the device (``ws_describe``: fused weighted moments, a radix select
    for the StatsBase weighted median, an 8-bin weighted histogram); vector columns are described
    component-wise and have an empty ``hist``, as in the reference."""
    import pandas as pd
    st = state.store
    if st.n == 0:
        raise ValueError("Store cannot be empty")
    names = st.colnames() if cols is None else list(cols)
    for name in names:
        if st._lookup(name)[0] < 0:
            raise ValueError(f"Column {name} not found in store")
    rows = {k: [] for k in ("variable", "mean", "median", "std", "min", "max", "hist", "ess")}
    if not names:
        return pd.DataFrame(rows)
    planes = []
    for name in names:
        cid, width = st._lookup(name)
        planes += [(cid, k) for k in range(width)]
    ca = (C.c_int32 * len(planes))(*[p[0] for p in planes])
    ka = (C.c_int32 * len(planes))(*[p[1] for p in planes])
    out = (L.ws_plane_stats * len(planes))()
    ess = C.c_double()
    st._call("ws_describe", len(planes), ca, ka, out, C.byref(ess))
    i = 0
    for name in names:
        cid, width = st._lookup(name)
        ps = out[i:i + width]
        i += width
        rows["variable"].append(name)
        for f in ("mean", "median", "std", "min", "max"):
            rows[f].append(getattr(ps[0], f) if width == 1 else np.array([getattr(p, f) for p in ps]))
        if width == 1:
            lo, hi = ps[0].min, ps[0].max
            h = list(ps[0].hist)
            rows["hist"].append(_sparkline([sum(h)] * 8 if lo == hi else h))
        else:
            rows["hist"].append("")
        rows["ess"].append(ess.value)
    return pd.DataFrame(rows)
