"""sample(state, n; replace) drawn on the device (ws_sample_indices) against its big-integer specification
(tests/sample_spec.py), its statistics, its Philox streams, the rows it returns and the bytes it moves."""
import ctypes as C

import numpy as np
import pytest

import models
import sample_spec as S

pytestmark = pytest.mark.gpu

SIZES = [1, 2049, 65_537, 1_000_003]
KINDS = ["lognormal_0.3", "lognormal_3", "one_hot", "third_inf", "nan", "uniform"]


def _logw(kind, n):
    rng = np.random.default_rng(n)
    if kind.startswith("lognormal"):
        return float(kind.split("_")[1]) * rng.standard_normal(n)
    if kind == "one_hot":
        lw = np.full(n, -np.inf)
        lw[(7 * n) // 11] = 0.5
        return lw
    lw = rng.standard_normal(n)
    if kind == "third_inf":
        lw[rng.random(n) < 1 / 3] = -np.inf
        lw[0] = 0.0
    if kind == "nan":
        lw[rng.random(n) < 0.1] = np.nan
        lw[-1] = 0.0
    return lw


def _state(ws, logw, n=None, seed=21):
    st = ws.SMCState(len(logw) if n is None else n, device=0, seed=seed)
    if logw is not None:
        st.weights = logw
    return st


def _draw(st, n, replace):
    stream, seed = C.c_uint64(), C.c_uint64()
    st.store._call("ws_next_philox_stream", C.byref(stream), C.byref(seed))
    idx = np.empty(n, dtype=np.int64)
    st.store._call("ws_sample_indices", n, int(replace), idx.ctypes.data_as(C.c_void_p))
    return idx, seed.value, stream.value


@pytest.mark.parametrize("n_part", SIZES)
@pytest.mark.parametrize("kind", KINDS)
def test_indices_equal_the_specification(ws, n_part, kind):
    st = _state(ws, _logw(kind, n_part)) if kind != "uniform" else _state(ws, None, n_part)
    lw = st.weights
    # with replacement: more draws than particles for the small sets
    n = min(2 * n_part + 3, 20_000)
    idx, seed, stream = _draw(st, n, True)
    np.testing.assert_array_equal(idx, S.sample_indices_spec(lw, seed, stream, n, True))
    # without replacement: a few, then all of them (a permutation)
    for n in sorted({min(n_part, 1000), n_part}):
        idx, seed, stream = _draw(st, n, False)
        np.testing.assert_array_equal(idx, S.sample_indices_spec(lw, seed, stream, n, False))
        if n == n_part:
            assert np.array_equal(np.sort(idx), np.arange(n_part))


def test_large_total_mass(ws):
    """equal weights at N = 1e6: T = 2^52 N > 2^64"""
    st = _state(ws, np.full(1_000_000, -2.0))
    idx, seed, stream = _draw(st, 50_000, True)
    np.testing.assert_array_equal(idx, S.sample_indices_spec(st.weights, seed, stream, 50_000, True))


def test_errors(ws):
    for lw in (np.full(100, -np.inf), np.full(100, np.nan)):
        st = _state(ws, lw)
        with pytest.raises(ws.WsError) as e:
            _draw(st, 5, True)
        assert e.value.code == -7
        with pytest.raises(ws.WsError) as e:
            _draw(st, 5, False)
        assert e.value.code == -7
    st = _state(ws, np.zeros(10))
    buf = np.empty(16, dtype=np.int64)
    for n, rep in ((0, 1), (-1, 0), (11, 0)):
        with pytest.raises(ws.WsError) as e:
            st.store._call("ws_sample_indices", n, rep, buf.ctypes.data_as(C.c_void_p))
        assert e.value.code == -1


def test_offspring_counts(ws):
    """chi-square of the offspring counts against n w"""
    w = np.random.default_rng(1).random(50) + 0.05
    w /= w.sum()
    st = _state(ws, np.log(w))
    n = 1_000_000
    idx, _, _ = _draw(st, n, True)
    c = np.bincount(idx, minlength=50)
    chi2 = float(((c - n * w) ** 2 / (n * w)).sum())
    assert chi2 < 100.0, chi2  # 49 degrees of freedom: p ~ 3e-5


def test_inclusion_frequencies_without_replacement(ws):
    """n = 2 of 5: the pair (first, second) against the successive-sampling probabilities w_a w_b / (1 - w_a)"""
    w = np.array([0.4, 0.25, 0.15, 0.12, 0.08])
    st = _state(ws, np.log(w))
    reps = 4000
    cnt = np.zeros((5, 5))
    for _ in range(reps):
        idx, _, _ = _draw(st, 2, False)
        cnt[idx[0], idx[1]] += 1
    p = np.array([[0.0 if a == b else w[a] * w[b] / (1 - w[a]) for b in range(5)] for a in range(5)])
    mask = p > 0
    chi2 = float((((cnt - reps * p) ** 2)[mask] / (reps * p[mask])).sum())
    assert chi2 < 60.0, chi2   # 19 degrees of freedom: p ~ 4e-6
    incl = (cnt.sum(0) + cnt.sum(1)) / reps
    exact = p.sum(0) + p.sum(1)
    assert np.abs(incl - exact).max() < 0.04


def test_streams(ws):
    lw = np.random.default_rng(2).standard_normal(5000)
    a = _state(ws, lw, seed=3)
    b = _state(ws, lw, seed=3)
    i1, _, s1 = _draw(a, 100, True)
    i2, _, s2 = _draw(a, 100, True)
    assert s2 == s1 + 1 and not np.array_equal(i1, i2)
    j1, _, _ = _draw(b, 100, True)
    j2, _, _ = _draw(b, 100, True)
    np.testing.assert_array_equal(i1, j1)
    np.testing.assert_array_equal(i2, j2)


def _ssm(ws, n, T):
    rng = np.random.default_rng(7)
    obs = list(np.cumsum(rng.standard_normal(T)))
    st = ws.SMCState(n, ess_perc_min=1.0, device=0, seed=5)
    ws.run(ws.model(models.SSM1D)(obs), st)
    return st


def test_rows_equal_the_columns(ws):
    """every column, including history columns that are genealogy-stale, through ws.sample"""
    st = _ssm(ws, 20_000, 30)
    stale = [nm for nm in st.store.colnames() if st.store._lookup(nm)[0] >= 0 and _behind(st, nm) > 0]
    assert stale, "the history columns should be behind the current order"
    for replace in (True, False):
        stream, seed = C.c_uint64(), C.c_uint64()
        st.store._call("ws_next_philox_stream", C.byref(stream), C.byref(seed))
        df = ws.sample(st, 777, replace=replace)
        idx = S.sample_indices_spec(st.weights, seed.value, stream.value, 777, replace)
        assert list(df.columns) == st.store.colnames()
        for nm in st.store.colnames():
            np.testing.assert_array_equal(df[nm].to_numpy(), st[nm][idx])


def _behind(st, name):
    out = C.c_int64()
    st.store._call("ws_col_events_behind", st.store._lookup(name)[0], C.byref(out))
    return out.value


def test_traffic_is_o_of_n(ws):
    n_part = 10_000_000
    st = _state(ws, np.random.default_rng(4).standard_normal(n_part))
    ws.log_evidence(st)   # the reduction, outside the measured window
    for n, replace in ((1000, True), (1000, False), (100_000, True)):
        before = st.stats()["d2h_bytes"]
        _draw(st, n, replace)
        moved = st.stats()["d2h_bytes"] - before
        assert moved <= 16 * n + 4096, (n, replace, moved)
