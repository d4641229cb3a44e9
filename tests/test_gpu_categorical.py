"""Discrete latent states on the device: tables indexed by particle values and the Categorical kernel, checked
against the oracle under replayed streams, against the exact HMM filter under Philox draws, and on the score-fold
(ws_move), expectation and speculative-block (ws_exec_spec) paths."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import ref
import table_ref as TR

pytestmark = pytest.mark.gpu
REL = 1e-12

HMM = '''
@model function hmm(ys, P, mu, sigma, p0)
    s ~ Categorical(p0)
    for y in ys
        s ~ Categorical(P[s, :])
        y => Normal(mu[s], sigma)
    end
end
'''

HMM_CAT = '''
@model function hmm_cat(ys, P, B, p0)
    s ~ Categorical(p0)
    for y in ys
        s ~ Categorical(P[s, :])
        y => Categorical(B[s, :])
    end
end
'''

SWITCHING = '''
@model function switching(ys, P, a, q, r)
    s ~ Categorical([0.5, 0.5])
    x ~ Normal(0.0, 1.0)
    for y in ys
        s ~ Categorical(P[s, :])
        x ~ Normal(a[s] * x, q[s])
        y => Normal(x, r)
    end
end
'''

MIXTURE = '''
@model function mixture(ys, w, mu, sigma)
    z ~ Categorical(w)
    c ~ Normal(0.0, 1.0)
    for y in ys
        y => Normal(mu[z] + c, sigma)
        if resampled
            c << RW(0.3)
        end
    end
end
'''


def _sticky(K, stay, rng):
    P = rng.dirichlet(np.ones(K), size=K) * (1.0 - stay) + np.eye(K) * stay
    return P / P.sum(axis=1, keepdims=True)


def _ancestors(st):
    a = np.empty(st.store.n, dtype=np.int32)
    st.store._call("ws_ancestors_download", a.ctypes.data_as(C.c_void_p))
    return a


def _replay(ws, root, n, normals=None, uniforms=None, ess=0.5):
    st = ws.SMCState(n, ess_perc_min=ess, device=0)
    st.set_replay(normals=normals, uniforms=uniforms)
    ws.run(root, st)
    ost = ref.OracleState(n, ref.Streams(normals, uniforms), ess_perc_min=ess)
    ost.expr_factory = ws.col      # the score walk binds a Sample's value to a column expression
    with TR.evaluating() as faults:
        ref.run(root, ost)
    assert faults.n == 0
    return st, ost


def _compare(st, ost):
    assert st.store.colnames() == ost.names
    for name in ost.names:
        np.testing.assert_allclose(st[name], ost.cols[name], rtol=REL, atol=REL, err_msg=name)
    np.testing.assert_allclose(st.weights, ost.weights, rtol=REL, atol=REL)
    fired = [e for e in ost.log if e["resampled"]]
    assert len(fired) >= 2 and st.stats()["resamples_done"] == len(fired)
    np.testing.assert_array_equal(_ancestors(st), np.asarray(fired[-1]["ancestors"]))
    assert abs(ws_log_evidence(st) - ref.log_evidence(ost)) <= REL * abs(ref.log_evidence(ost))


def ws_log_evidence(st):
    import wsb200
    return wsb200.log_evidence(st)


def test_hmm_k4_replay_parity(ws):
    rng = np.random.default_rng(11)
    K, T, n = 4, 30, 20_000
    P = _sticky(K, 0.8, rng)
    mu, sigma = np.array([-3.0, -1.0, 1.0, 3.0]), 0.8
    s, ys = 0, []
    for _ in range(T):
        s = rng.choice(K, p=P[s])
        ys.append(mu[s] + sigma * rng.standard_normal())
    root = ws.model(HMM)(ys, P, mu, sigma, np.full(K, 0.25))
    st, ost = _replay(ws, root, n, uniforms=rng.random(n * (2 * T + 2)))
    _compare(st, ost)
    assert set(np.unique(st["s"])) <= {1.0, 2.0, 3.0, 4.0}


def test_regime_switching_lgssm_replay_parity(ws):
    rng = np.random.default_rng(12)
    T, n = 25, 20_000
    P = np.array([[0.95, 0.05], [0.1, 0.9]])
    a, q, r = np.array([0.9, 0.5]), np.array([0.3, 1.5]), 0.5
    x, s, ys = 0.0, 0, []
    for _ in range(T):
        s = rng.choice(2, p=P[s])
        x = a[s] * x + q[s] * rng.standard_normal()
        ys.append(x + r * rng.standard_normal())
    root = ws.model(SWITCHING)(ys, P, a, q, r)
    st, ost = _replay(ws, root, n, normals=rng.standard_normal(n * (T + 1)), uniforms=rng.random(n * (2 * T + 2)))
    _compare(st, ost)


def _hmm_truth(rng, K, T, emit):
    P = _sticky(K, 0.7, rng)
    p0 = np.full(K, 1.0 / K)
    s, ys = rng.choice(K, p=p0), []
    for _ in range(T):
        s = rng.choice(K, p=P[s])
        ys.append(emit(s))
    return P, p0, ys


def _exact_check(ws, root, exact_le, marg, n, seeds):
    les, probs = [], []
    for seed in seeds:
        st = ws.SMCState(n, seed=seed, device=0)
        ws.run(root, st)
        les.append(ws.log_evidence(st))
        probs.append(ws.expectation([ws.col("s").eq(float(k + 1)) for k in range(len(marg))], st))
    les, probs = np.array(les), np.array(probs)
    sd = float(np.std(les, ddof=1))
    # the estimates of independent runs spread by the MC standard error: the mean of R of them is within a few
    # standard errors of the exact value (the small downward bias of log Z-hat is O(1/N))
    assert abs(les.mean() - exact_le) <= 5.0 * sd / math.sqrt(len(les)) + 1e-4, (les, exact_le, sd)
    # E(s == k) at T: binomial standard error of at most 0.5 / sqrt(ESS), ESS >= N / 10 here
    np.testing.assert_allclose(probs.mean(axis=0), marg, atol=5.0 * 0.5 / math.sqrt(n / 10) / math.sqrt(len(seeds)))
    return les, sd


def test_hmm_k3_normal_emissions_exact_answer(ws):
    rng = np.random.default_rng(21)
    K, T, n = 3, 50, 1_000_000
    mu, sigma = np.array([-2.0, 0.0, 2.0]), 1.0
    P, p0, ys = _hmm_truth(rng, K, T, lambda s: mu[s] + sigma * rng.standard_normal())
    emis = [[ref.normal_logpdf(y, mu[k], sigma) for k in range(K)] for y in ys]
    exact_le, filt = TR.hmm_forward(P, p0 @ P, emis)
    root = ws.model(HMM)(ys, P, mu, sigma, p0)
    _exact_check(ws, root, exact_le, filt[-1], n, seeds=[1, 2, 3, 4])


def test_hmm_k3_categorical_emissions_exact_answer(ws):
    rng = np.random.default_rng(22)
    K, T, n = 3, 50, 1_000_000
    B = np.array([[0.7, 0.2, 0.1, 0.0], [0.1, 0.6, 0.2, 0.1], [0.0, 0.1, 0.3, 0.6]])
    P, p0, ys = _hmm_truth(rng, K, T, lambda s: float(rng.choice(4, p=B[s]) + 1))
    emis = [[math.log(B[k, int(y) - 1]) if B[k, int(y) - 1] > 0 else -math.inf for k in range(K)] for y in ys]
    exact_le, filt = TR.hmm_forward(P, p0 @ P, emis)
    root = ws.model(HMM_CAT)(ys, P, B, p0)
    _exact_check(ws, root, exact_le, filt[-1], n, seeds=[5, 6, 7, 8])


def test_move_with_table_reads_in_the_score_tape_replay(ws):
    rng = np.random.default_rng(31)
    T, n = 8, 5_000
    w, mu, sigma = np.array([0.2, 0.3, 0.5]), np.array([-2.0, 0.5, 3.0]), 0.7
    ys = list(0.5 + 0.3 + sigma * rng.standard_normal(T))
    root = ws.model(MIXTURE)(ys, w, mu, sigma)
    st, ost = _replay(ws, root, n, normals=rng.standard_normal(n * (T + 2)), uniforms=rng.random(n * (3 * T + 2)), ess=0.9)
    assert st.stats()["moves_run"] >= 2
    _compare(st, ost)


def test_spec_blocks_with_a_mixture_body_equal_statement_by_statement(ws):
    rng = np.random.default_rng(41)
    T, n = 40, 100_003
    w, mu, sigma = np.array([0.2, 0.3, 0.5]), np.array([-2.0, 0.5, 3.0]), 1.5
    ys = list(0.5 + sigma * rng.standard_normal(T))
    out = []
    for spec in (False, True):
        old = ws.core.SPEC_BLOCKS
        ws.core.SPEC_BLOCKS = spec
        try:
            st = ws.SMCState(n, ess_perc_min=0.5, seed=9, device=0)
            ws.run(ws.model(MIXTURE)(ys, w, mu, sigma), st)
        finally:
            ws.core.SPEC_BLOCKS = old
        out.append((st["z"], st["c"], st.weights, ws.log_evidence(st), st.stats()))
    (za, ca, wa, la, sa), (zb, cb, wb, lb, sb) = out
    assert sb["fused_passes"] < sa["fused_passes"], "the loop should have run in speculative blocks"
    np.testing.assert_array_equal(za, zb)
    np.testing.assert_allclose(cb, ca, rtol=REL, atol=REL)
    np.testing.assert_allclose(wb, wa, rtol=REL, atol=REL)
    assert abs(lb - la) <= REL * abs(la)


def test_expectation_reads_tables(ws):
    n = 10_000
    rng = np.random.default_rng(51)
    st = ws.SMCState(n, device=0)
    s = rng.integers(1, 4, size=n).astype(float)
    st.store.setcol("s", s)
    lw = rng.standard_normal(n)
    st.weights = lw
    mu = ws.table([1.5, -2.0, 0.25])
    got = ws.expectation(mu[ws.col("s")] * ws.col("s"), st)
    wn = np.exp(lw - lw.max())
    wn /= wn.sum()
    assert abs(got - np.sum(wn * np.array([1.5, -2.0, 0.25])[s.astype(int) - 1] * s)) <= 1e-12


def test_run_raises_index_error_after_out_of_range_index(ws):
    src = '''
    @model function bad(mu)
        z ~ Categorical([0.5, 0.5])
        k .= z + 1.0
        m .= mu[k]
    end
    '''
    st = ws.SMCState(1000, seed=3, device=0)
    with pytest.raises(IndexError):
        ws.run(ws.model(src)(np.array([10.0, 20.0])), st)
    m, z = st["m"], st["z"]
    assert np.all(np.isnan(m[z == 2.0])) and np.all(m[z == 1.0] == 20.0)
    good = ws.SMCState(1000, seed=3, device=0)
    ws.run(ws.model(src)(np.array([10.0, 20.0, 30.0])), good)        # in range: no error
    np.testing.assert_array_equal(good["m"], good["z"] * 10.0 + 10.0)
