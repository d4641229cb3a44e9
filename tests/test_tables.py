"""Build-time tables and the Categorical kernel on the CPU: the product's lowering and interpreter run through
tests/host/table_harness.cpp and are checked value for value against tests/table_ref.py; the front-end checks need
no device at all."""
import math

import numpy as np
import pytest

import wsb200 as ws
from wsb200 import core, expr as E
from table_hostlib import TableHostState
import table_ref as R


def _state(n, **cols):
    st = TableHostState(n)
    for k, v in cols.items():
        st.store.setcol(k, v)
    return st


# ---- table reads ------------------------------------------------------------------------------------------------
def test_table_reads_match_reference_with_faults():
    T = np.arange(1.0, 13.0).reshape(3, 4) * 0.5
    rows = np.array([1, 2, 3, 1.5, 0, 4, np.nan, 2, 3, -1, 1, 3.0])
    cols = np.array([1, 4, 2, 1, 1, 1, 2, 4.0000001, 0, 1, 5, np.nan])
    st = _state(rows.size, r=rows, c=cols)
    core.Assign("v", E.table(T)[E.col("r"), E.col("c")]).apply(st)
    got = st.store.getcol("v")
    want, faults = R.table_read(T, rows, cols)
    np.testing.assert_array_equal(got, want)
    assert faults == 9 and st.store.index_faults() == faults
    assert np.all(np.isfinite(got[:3])) and np.isnan(got[3:]).all()


def test_vector_table_and_constant_index():
    mu = np.array([-1.0, 0.25, 7.5])
    s = np.array([1.0, 2.0, 3.0, 3.0, 0.0, 4.0, 2.5, np.nan])
    st = _state(s.size, s=s)
    core.Assign("m", E.table(mu)[E.col("s")] * 2.0 + 1.0).apply(st)
    core.Assign("k", E.table(mu)[3]).apply(st)
    want, faults = R.table_read(mu, 1.0, s)
    np.testing.assert_array_equal(st.store.getcol("m"), want * 2.0 + 1.0)
    np.testing.assert_array_equal(st.store.getcol("k"), np.full(s.size, 7.5))
    assert st.store.index_faults() == faults == 4


def test_tables_are_deduplicated_by_content():
    st = _state(4, s=np.ones(4))
    a, b = E.table([1.0, 2.0]), E.table(np.array([1.0, 2.0]))
    assert st.store._table_id(a) == st.store._table_id(b)
    assert st.store._table_id(E.table([2.0, 1.0])) != st.store._table_id(a)


# ---- Categorical draws ------------------------------------------------------------------------------------------
def _draw(P, rows, u):
    st = _state(len(u), s=rows)
    st.store.set_uniforms(u)
    core.Sample("x", "Categorical", lambda _s: E.table(P)[E.col("s"), :]).apply(st)
    return st


def test_categorical_draws_on_partial_sums_and_edges():
    P = np.array([[0.1, 0.2, 0.3, 0.4], [0.0, 0.5, 0.0, 0.5], [0.25, 0.25, 0.25, 0.25]])
    C = R.partial_sums(P)
    us, rows = [], []
    for r in range(3):
        for c in C[r]:
            us += [c, np.nextafter(c, 0.0), np.nextafter(c, 1.0)]   # exactly on a partial sum, and either side of it
            rows += [r + 1] * 3
    us += [0.0, np.nextafter(1.0, 0.0), 0.999999]
    rows += [1, 2, 3]
    us, rows = np.clip(np.array(us), 0.0, np.nextafter(1.0, 0.0)), np.array(rows, dtype=float)
    st = _draw(P, rows, us)
    want, faults = R.categorical_draw(P, rows, us)
    np.testing.assert_array_equal(st.store.getcol("x"), want)
    assert faults == 0 and st.store.index_faults() == 0
    # u == C_1 of row 1 walks past the first category (C_k <= u), a zero-probability category is never drawn
    assert want[0] == 2.0 and not np.any((rows == 2) & ((want == 1.0) | (want == 3.0)))


def test_categorical_row_summing_below_one():
    # a row that sums to 1 - ulp: u just below 1 lies beyond C_K, and the walk stops at K
    p = np.array([0.3, 0.3, 0.4])
    p[2] = np.nextafter(1.0, 0.0) - (p[0] + p[1])
    assert R.partial_sums(p)[0, -1] < 1.0
    u = np.array([np.nextafter(1.0, 0.0), R.partial_sums(p)[0, -1], 0.6, 0.3])
    st = _draw(p[None, :], np.ones(4), u)
    want, _ = R.categorical_draw(p, 1.0, u)
    np.testing.assert_array_equal(st.store.getcol("x"), want)
    assert list(want) == [3.0, 3.0, 3.0, 2.0]


def test_categorical_random_rows_match_walk():
    rng = np.random.default_rng(5)
    K, n = 7, 4000
    P = rng.dirichlet(np.ones(K), size=5)
    P[2, 3] = 0.0
    P[2] /= P[2].sum()
    rows = rng.integers(1, 6, size=n).astype(float)
    rows[:3] = [0.0, 6.0, 2.5]           # bad rows: NaN and a fault each
    u = rng.random(n)
    st = _draw(P, rows, u)
    want, faults = R.categorical_draw(P, rows, u)
    np.testing.assert_array_equal(st.store.getcol("x"), want)
    assert faults == 3 and st.store.index_faults() == 3


def test_categorical_constant_vector_and_replay_order():
    p = np.array([0.5, 0.25, 0.25])
    u = np.array([0.1, 0.6, 0.9, 0.5, 0.2, 0.8, 0.74, 0.76])   # two draws of four particles, statement order
    st = _state(4)
    st.store.set_uniforms(u)
    core.Sample("a", "Categorical", lambda _s: p).apply(st)
    core.Sample("b", "Categorical", lambda _s: p).apply(st)
    np.testing.assert_array_equal(st.store.getcol("a"), R.categorical_draw(p, 1.0, u[:4])[0])
    np.testing.assert_array_equal(st.store.getcol("b"), R.categorical_draw(p, 1.0, u[4:])[0])


# ---- Categorical logpdf -----------------------------------------------------------------------------------------
def test_categorical_logpdf_zero_probability_and_out_of_support():
    P = np.array([[0.2, 0.0, 0.8], [0.5, 0.5, 0.0]])
    s = np.array([1, 1, 1, 2, 2, 2, 1, 1, 1, 2.0, 3.0])
    y = np.array([1, 2, 3, 1, 2, 3, 0, 4, 1.5, np.nan, 1.0])
    st = _state(s.size, s=s, y=y)
    core.Observe(E.col("y"), "Categorical", lambda _s: E.table(P)[E.col("s"), :]).apply(st)
    want, faults = R.table_read(P, s, y, logp=True)
    got = st.store.logw()
    np.testing.assert_array_equal(got, want)
    assert got[1] == -np.inf and got[5] == -np.inf and np.all(got[6:10] == -np.inf)
    assert got[0] == math.log(0.2) and faults == 1 and st.store.index_faults() == 1   # only the bad row faults
    np.testing.assert_array_equal(st.store.score(), want)     # the score tape folds the same log-densities


# ---- front end --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", [[0.5, 0.6], [1.2, -0.2], [0.5, 0.5 - 1e-6], [np.nan, 1.0]])
def test_invalid_probability_rows_raise_value_error(bad):
    st = _state(2, s=np.ones(2))
    with pytest.raises(ValueError):
        core.Sample("x", "Categorical", lambda _s: E.table([[0.5, 0.5], bad])[E.col("s"), :]).apply(st)
    with pytest.raises(ValueError):
        core.Sample("x", "Categorical", lambda _s: np.asarray(bad)).apply(st)


def test_probability_rows_within_sqrt_eps_pass():
    st = _state(2, s=np.ones(2))
    st.store.set_uniforms(np.full(2, 0.5))
    core.Sample("x", "Categorical", lambda _s: E.table([[0.5, 0.5 + 1e-9]])[E.col("s"), :]).apply(st)


HMM_SRC = '''
@model function hmm(ys, P, mu, sigma, p0)
    s ~ Categorical(p0)
    for y in ys
        s ~ Categorical(P[s, :])
        y => Normal(mu[s], sigma)
    end
end
'''


def test_model_lowers_table_indices_and_categorical_rows():
    P = np.array([[0.9, 0.1], [0.2, 0.8]])
    mu = np.array([-1.0, 1.0])
    root = ws.model(HMM_SRC)([0.3, -0.5], P, mu, 0.7, np.array([0.5, 0.5]))
    n = 64
    rng = np.random.default_rng(1)
    u = rng.random(3 * n)
    st = TableHostState(n)
    st.store.set_uniforms(u)
    root.apply(st)                            # no UnsupportedModelError: the whole program lowers
    s0 = R.categorical_draw([[0.5, 0.5]], 1.0, u[:n])[0]
    s1 = R.categorical_draw(P, s0, u[n:2 * n])[0]
    s2 = R.categorical_draw(P, s1, u[2 * n:])[0]
    np.testing.assert_array_equal(st.store.getcol("s"), s2)
    lw = (R.table_read(mu, 1.0, s1)[0] - 0.3) / 0.7
    lw2 = (R.table_read(mu, 1.0, s2)[0] + 0.5) / 0.7
    want = -(lw ** 2 + lw2 ** 2) / 2 - 2 * (math.log(0.7) + 0.5 * math.log(2 * math.pi))
    np.testing.assert_allclose(st.store.logw(), want, rtol=1e-13, atol=1e-13)


def test_model_entry_index_and_build_time_matrix_index():
    src = '''
    @model function m(A, k)
        z .= A[s, k] + A[2, 1]
    end
    '''
    A = np.array([[1.0, 2.0], [3.0, 4.0]])
    st = _state(3, s=np.array([1.0, 2.0, 1.0]))
    ws.model(src, particle_vars=("s",))(A, 2).apply(st)
    np.testing.assert_array_equal(st.store.getcol("z"), [5.0, 7.0, 5.0])


def test_particle_index_into_particle_variable_still_unsupported():
    src = '''
    @model function m()
        x .= [1.0, 2.0]
        s .= 1.0
        z .= x[s]
    end
    '''
    with pytest.raises(ws.UnsupportedModelError):
        ws.model(src)()


@pytest.mark.parametrize("name", core._REFERENCE_ONLY_KERNELS)
def test_reference_only_kernels_still_raise(name):
    assert name != "Categorical"
    with pytest.raises(ws.UnsupportedModelError):
        core.resolve_kernel(name)
    with pytest.raises(ws.UnsupportedModelError):
        ws.model(f'''
        @model function m()
            x ~ {name}(1.0)
        end
        ''')()


def test_categorical_is_a_default_kernel():
    assert "Categorical" in ws.default_kernels and "Categorical" not in core._REFERENCE_ONLY_KERNELS


def test_per_particle_probability_vectors_unsupported():
    st = _state(2, a=np.full(2, 0.5))
    with pytest.raises(ws.UnsupportedModelError):
        core.Sample("x", "Categorical", lambda _s: E.Vec([E.col("a"), 1.0 - E.col("a")])).apply(st)


def test_wide_rows_are_accepted_up_to_the_limit():
    K = 2 ** 16
    p = np.full(K, 1.0 / K)
    st = _state(3, s=np.ones(3))
    st.store.set_uniforms(np.array([0.0, 0.5, np.nextafter(1.0, 0.0)]))
    core.Sample("x", "Categorical", lambda _s: p).apply(st)
    np.testing.assert_array_equal(st.store.getcol("x"), R.categorical_draw(p, 1.0, [0.0, 0.5, np.nextafter(1.0, 0.0)])[0])
