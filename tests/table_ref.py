"""Reference rules for build-time tables and Categorical (include/wsb200.h: ws_table), next to oracle/ref.py.

`evaluating(...)` lets `oracle.ref.run` evaluate the table expressions of weightedsampling.jl_b200/expr.py
(TableRead, RandCat, CatLogp) with these rules; `hmm_forward` is the exact filter of a hidden Markov model, the
discrete counterpart of `oracle.ref.kalman_filter_evidence`."""
import contextlib
import math

import numpy as np

from oracle import ref


def index_ok(x, n):
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        return (x >= 1.0) & (x <= float(n)) & (x == np.floor(x))


def _log(v):
    # libm's log, as the host side of ws_table forms the log table (log 0 = -Inf, negative -> NaN)
    return math.log(v) if v > 0.0 else (-math.inf if v == 0.0 else math.nan)


def table_read(values, row, col, logp=False):
    """T[row, col] (1-based) per particle -> (values, number of index faults).  logp: log T with a column outside
    1..n_cols giving -Inf and no fault."""
    T = np.asarray(values, dtype=np.float64)
    T = T[None, :] if T.ndim == 1 else T
    src = np.vectorize(_log)(T) if logp else T
    row, col = np.broadcast_arrays(np.asarray(row, dtype=np.float64), np.asarray(col, dtype=np.float64))
    rok, cok = index_ok(row, T.shape[0]), index_ok(col, T.shape[1])
    out = np.full(row.shape, np.nan)
    ok = rok & cok
    out[ok] = src[row[ok].astype(np.int64) - 1, col[ok].astype(np.int64) - 1]
    bad = ~ok
    if logp:
        out[rok & ~cok] = -np.inf
        bad = ~rok
    return out, int(np.sum(bad))


def partial_sums(values):
    """row-wise sequential Float64 sums cp += p[i]"""
    T = np.asarray(values, dtype=np.float64)
    T = T[None, :] if T.ndim == 1 else T
    C = np.empty_like(T)
    for r in range(T.shape[0]):
        cp = 0.0
        for k in range(T.shape[1]):
            cp += float(T[r, k])
            C[r, k] = cp
    return C


def categorical_draw(values, row, u):
    """Distributions 0.25's walk: i = 1, cp = p[1]; while cp <= u && i < K: i += 1, cp += p[i] -> (draws, faults)"""
    C = partial_sums(values)
    K = C.shape[1]
    row, u = np.broadcast_arrays(np.asarray(row, dtype=np.float64), np.asarray(u, dtype=np.float64))
    out = np.full(row.shape, np.nan)
    rok = index_ok(row, C.shape[0])
    for i in np.flatnonzero(rok.ravel()):
        c = C[int(row.flat[i]) - 1]
        k = 1
        while c[k - 1] <= u.flat[i] and k < K:
            k += 1
        out.flat[i] = float(k)
    return out, int(np.sum(~rok))


class Faults:
    n = 0


def _eval(e, st, base):
    k = type(e).__name__
    if k == "TableRead":
        v, f = table_read(e.table.values, _b(base(e.row, st), st), _b(base(e.col, st), st))
        Faults.n += f
        return v
    if k == "CatLogp":
        v, f = table_read(e.p.table.values, _b(base(e.p.row, st), st), _b(base(e.x, st), st), logp=True)
        Faults.n += f
        return v
    if k == "RandCat":
        row = _b(base(e.p.row, st), st)
        v, f = categorical_draw(e.p.table.values, row, st.streams.uniforms(st.n))
        Faults.n += f
        return v
    return base(e, st)


def _b(v, st):
    return np.broadcast_to(np.asarray(v, dtype=np.float64), (st.n,))


@contextlib.contextmanager
def evaluating():
    """oracle.ref evaluates table expressions inside the block (nested expressions included)"""
    orig = ref.eval_expr

    def ev(e, st):
        k = type(e).__name__
        if k in ("TableRead", "CatLogp", "RandCat"):
            return _eval(e, st, ev)
        # the other node types recurse through ref.eval_expr, which is this function while the block is open
        return orig(e, st)

    ref.eval_expr = ev
    Faults.n = 0
    try:
        yield Faults
    finally:
        ref.eval_expr = orig


def hmm_forward(P, pi0, emission_logpdfs):
    """Exact filter of a hidden Markov model whose state at the first observation is distributed as pi0 and then moves
    by s_t ~ P[s_{t-1}, :]; emission_logpdfs[t][k] = log p(y_t | s_t = k + 1).  Returns (log-evidence, filtering
    marginals [T, K]).  (A model that draws s ~ Categorical(p0) and transitions before its first observation passes
    pi0 = p0 @ P.)"""
    P = np.asarray(P, dtype=np.float64)
    pred = np.asarray(pi0, dtype=np.float64)
    logZ, filt = 0.0, []
    for t, lp in enumerate(emission_logpdfs):
        if t > 0:
            pred = filt[-1] @ P
        lp = np.asarray(lp, dtype=np.float64)
        m = float(np.max(lp))
        a = pred * np.exp(lp - m)
        z = float(np.sum(a))
        logZ += math.log(z) + m
        filt.append(a / z)
    return logZ, np.asarray(filt)
