"""The specification of sample(state, n; replace) (tests/sample_spec.py) on the CPU: against brute force, ties, -inf
and NaN log-weights, and integer masses above 2^64."""
import math

import numpy as np
import pytest

import sample_spec as S
from oracle import ref


def _brute_replace(logw, seed, stream, n):
    """exact inversion with a linear scan over the harness's q, t_k from the harness routine"""
    q = [int(v) for v in S.sample_q(logw, S.max_logw(logw)).tolist()]
    T = sum(q)
    out = []
    for t in S.sample_targets_harness(n, seed, stream, T):
        acc = 0
        for j, qj in enumerate(q):
            acc += qj
            if acc > t:
                out.append(j)
                break
    return np.array(out, dtype=np.int64), q


def _brute_keys(logw, seed, stream):
    """Gumbel keys from Philox in numpy floats (libm log: equal to the device's up to an ulp or two)"""
    n = len(logw)
    x, y, _, _ = ref.philox4x32_10(np.arange(n, dtype=np.uint64), stream, seed)
    v = ((x.astype(np.uint64) << np.uint64(32)) | y.astype(np.uint64)) >> np.uint64(11)
    u = (v.astype(np.float64) + 1.0) * 2.0 ** -53
    e = -np.log(u)
    return np.where(np.isfinite(logw), np.asarray(logw) - np.log(np.maximum(e, 2.0 ** -54)), -np.inf)


@pytest.mark.parametrize("n_part", [1, 2, 7, 300])
@pytest.mark.parametrize("s", [0.3, 3.0])
def test_with_replacement_matches_brute_force(n_part, s):
    logw = s * np.random.default_rng(n_part).standard_normal(n_part)
    idx = S.sample_indices_spec(logw, 5, 9, 400, True)
    brute, q = _brute_replace(logw, 5, 9, 400)
    np.testing.assert_array_equal(idx, brute)
    # q against libm's exp: the device exp is within an ulp or two, so q within one unit
    q_np = np.rint(np.exp(logw - logw.max()) * 2.0 ** 52)
    assert np.abs(np.array(q, dtype=np.float64) - q_np).max() <= 1.0


@pytest.mark.parametrize("n_part", [2, 7, 300])
def test_without_replacement_matches_brute_force(n_part):
    logw = 2.0 * np.random.default_rng(n_part + 1).standard_normal(n_part)
    n = max(1, n_part // 2)
    idx = S.sample_indices_spec(logw, 3, 4, n, False)
    k = _brute_keys(logw, 3, 4)
    brute = np.lexsort((np.arange(n_part), -k))[:n]
    np.testing.assert_array_equal(idx, brute)
    full = S.sample_indices_spec(logw, 3, 4, n_part, False)
    assert sorted(full.tolist()) == list(range(n_part))


def test_targets_are_the_exact_high_product():
    rng = np.random.default_rng(0)
    for T in [1, 2 ** 52, 2 ** 64 - 1, 2 ** 64, 2 ** 64 + 1, 3 * 2 ** 70 + 12345, 2 ** 127 + 5, 2 ** 128 - 1,
              int(rng.integers(1, 2 ** 62)) * int(rng.integers(1, 2 ** 62))]:
        h = S.sample_targets_harness(64, 17, 2, T)
        assert h == S.targets(64, 17, 2, T)
        assert all(0 <= t < T for t in h)


def test_total_mass_above_2_64():
    n_part = 8192                      # equal weights: q = 2^52 each, T = 2^65
    logw = np.full(n_part, -3.5)
    q = S.sample_q(logw, S.max_logw(logw))
    assert (q == np.uint64(2 ** 52)).all()
    idx = S.sample_indices_spec(logw, 1, 1, 20000, True)
    # with equal weights, index_k = floor(r_k N / 2^128)
    expect = [(r * n_part) >> 128 for r in S.philox_r128(20000, 1, 1)]
    np.testing.assert_array_equal(idx, expect)
    counts = np.bincount(idx, minlength=n_part)
    assert counts.sum() == 20000 and counts.max() < 12


def test_non_finite_log_weights():
    logw = np.array([0.0, -np.inf, np.nan, 1.0, -np.inf, np.nan, -2.0])
    finite = {0, 3, 6}
    idx = S.sample_indices_spec(logw, 2, 8, 5000, True)
    assert set(idx.tolist()) <= finite
    # without replacement: the finite ones first (by key), then the others by index
    full = S.sample_indices_spec(logw, 2, 8, 7, False)
    assert set(full[:3].tolist()) == finite and full[3:].tolist() == [1, 2, 4, 5]
    for bad in (np.full(4, -np.inf), np.full(4, np.nan), np.array([0.0, np.inf]), np.array([np.nan, -np.inf])):
        with pytest.raises(ValueError):
            S.sample_indices_spec(bad, 0, 1, 3, True)


def test_ties_go_to_the_lower_index():
    keys = np.array([5, 9, 5, 9, 0, 5, 7], dtype=np.uint64)
    assert S.select_top(keys, 7).tolist() == [1, 3, 6, 0, 2, 5, 4]
    assert S.select_top(keys, 4).tolist() == [1, 3, 6, 0]
    # one-hot: the only drawable particle
    logw = np.full(50, -np.inf)
    logw[17] = 3.0
    assert set(S.sample_indices_spec(logw, 0, 3, 100, True).tolist()) == {17}
    assert S.sample_indices_spec(logw, 0, 3, 3, False).tolist() == [17, 0, 1]


def test_spec_frequencies():
    """chi-square of offspring counts against n w (with replacement)"""
    w = np.array([0.05, 0.1, 0.2, 0.3, 0.35])
    n = 200_000
    idx = S.sample_indices_spec(np.log(w), 12, 6, n, True)
    c = np.bincount(idx, minlength=5)
    chi2 = float(((c - n * w) ** 2 / (n * w)).sum())
    assert chi2 < 20.0, chi2   # 4 degrees of freedom: p ~ 5e-4


def test_weight_far_below_the_largest_is_never_drawn():
    logw = np.array([0.0, -40.0, -36.0])           # 2^-57.7 and 2^-51.9 of the largest
    q = S.sample_q(logw, 0.0)
    assert q[0] == 2 ** 52 and q[1] == 0 and q[2] == int(np.rint(math.exp(-36.0) * 2.0 ** 52))
