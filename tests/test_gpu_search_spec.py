"""Ancestors of the multi-kernel resampler (tile CDF, group offsets, warp-tile search) against the big-integer
specification of the integer slot grid (oracle/ref.py: stratified_ancestors_fixed_point), stratified and systematic.

A warp searches a run of consecutive 256-particle tiles and keeps the Philox blocks of one tile's slot range for the
next (ws_search_kernel's ring, in the upper half of the warp's window); a tile of up to 381 slots is expanded in one
round of twelve slots per lane, a larger one in chunks.  The weights below
give warp tiles whose slot ranges cover 63, 64, 65, 66 and many more Philox blocks (four slots per block), ranges that
skip blocks, an odd number of warp tiles and a partial last tile.
"""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SIZES = [511, 512, 513, 2047, 2049, 65_537, 1_000_003]


def _state(ws, n, **kw):
    # the scan form and the one-kernel step for small sets are chosen when the state is made
    env = {"WSB200_SMALL_RESAMPLE": "0", "WSB200_SCAN": "3pass"}
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return ws.SMCState(n, device=0, **kw)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _check(ws, w, scheme, seed=11):
    from oracle import ref
    st = _state(ws, w.size, seed=seed)
    stream, sd = C.c_uint64(), C.c_uint64()
    st.store._call("ws_next_philox_stream", C.byref(stream), C.byref(sd))
    a, clamped = ws.resample_indices(w, st, scheme, return_clamped=True)
    a_ref, clamped_ref = ref.stratified_ancestors_fixed_point(w, sd.value, stream.value, scheme)
    np.testing.assert_array_equal(a, a_ref)
    assert clamped == clamped_ref


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("s", [0.3, 1.0, 3.0])
@pytest.mark.parametrize("scheme", ["stratified", "systematic"])
def test_log_normal_weights(ws, n, s, scheme):
    w = np.exp(s * np.random.default_rng(n).standard_normal(n))
    _check(ws, w / w.sum(), scheme)


# per warp tile, the mean slot count relative to 256: 0.98, 1.0, 1.02 -> 63 to 66 blocks; 1.2 -> 77; 2.0 -> 128 (beyond
# the ring, and more slots than one expansion round); 0.3 and 0.5 -> ranges shorter than a round of 32 blocks
TILE_SCALES = np.array([0.98, 1.0, 1.02, 1.2, 0.3, 2.0, 0.5])


@pytest.mark.parametrize("n", [2049, 65_537, 1_000_003, 256 * 1001])
@pytest.mark.parametrize("scheme", ["stratified", "systematic"])
def test_tile_slot_ranges(ws, n, scheme):
    tiles = (n + 255) // 256
    c = np.resize(TILE_SCALES, tiles)
    w = np.repeat(c, 256)[:n] * np.exp(0.01 * np.random.default_rng(3).standard_normal(n))
    _check(ws, w / w.sum(), scheme)


@pytest.mark.parametrize("n", [513, 65_537, 1_000_003])
@pytest.mark.parametrize("scheme", ["stratified", "systematic"])
def test_one_hot_and_zero_weights(ws, n, scheme):
    w = np.zeros(n)
    w[n // 3] = 1.0
    _check(ws, w, scheme)
    w = np.exp(np.random.default_rng(5).standard_normal(n))
    w[::3] = 0.0                          # log-weight -inf
    w[n // 2 - 300:n // 2 + 300] = 0.0    # (n > 600) whole warp tiles without offspring
    _check(ws, w / w.sum(), scheme)


@pytest.mark.parametrize("n", [2049, 1_000_003])
@pytest.mark.parametrize("scheme", ["stratified", "systematic"])
def test_log_weights_inside_a_step(ws, n, scheme):
    """log-weights with -inf and a dominant particle, through the tile pass's own exp-normalisation (mode 0)"""
    from oracle import ref
    lw = 1.0 * np.random.default_rng(7).standard_normal(n)
    lw[::5] = -np.inf
    lw[n // 4] = 8.0
    st = _state(ws, n, ess_perc_min=float("inf"), seed=3, resampler=scheme)
    st.store.setcol("id", np.arange(n, dtype=np.float64))
    st.weights = lw
    st.weights_changed = True
    stream, sd = C.c_uint64(), C.c_uint64()
    st.store._call("ws_next_philox_stream", C.byref(stream), C.byref(sd))
    ws.Resample().apply(st)
    a_ref, _ = ref.stratified_ancestors_fixed_point(ref.exp_norm(lw), sd.value, stream.value, scheme)
    np.testing.assert_array_equal(st["id"].astype(np.int64), a_ref)
