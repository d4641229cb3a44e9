"""sample(state, n; replace) on a sharded state: R ranks return the single-GPU global indices and bit-identical
DataFrames.  Needs >= 2 (or 4) GPUs; skipped on a smaller box."""
import ctypes
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 200_003


def _ngpu():
    import wsb200
    n = ctypes.c_int()
    wsb200.load().ws_device_count(ctypes.byref(n))
    return n.value


def _inputs():
    rng = np.random.default_rng(9)
    lw = 2.0 * rng.standard_normal(N)
    lw[rng.random(N) < 0.2] = -np.inf
    a = rng.standard_normal(N)
    a[::7] = -0.0
    a[3::11] = np.frombuffer(np.uint64(0x7FF8_0000_0000_1234).tobytes(), dtype=np.float64)[0]  # a NaN payload
    b = rng.standard_normal((N, 2))
    return lw, a, b


def _draws(ws, st):
    out = []
    for n, rep in ((5000, 1), (3000, 0), (N, 0)):
        idx = np.empty(n, dtype=np.int64)
        st.store._call("ws_sample_indices", n, rep, idx.ctypes.data_as(ctypes.c_void_p))
        out.append(idx)
    df = ws.sample(st, 4000, replace=True)
    df2 = ws.sample(st, 2500, replace=False)
    bits = [np.ascontiguousarray(d["a"].to_numpy()).view(np.uint64) for d in (df, df2)]
    bits += [np.ascontiguousarray(np.stack(d["b"].to_numpy())).view(np.uint64) for d in (df, df2)]
    return out, bits


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import wsb200 as ws
    lw, a, b = _inputs()
    lo, hi = (N * rank) // world, (N * (rank + 1)) // world
    st = ws.sharded_state(N, device=rank, seed=31)
    st.store.setcol("a", a[lo:hi])
    st.store.setcol("b", b[lo:hi])
    st.weights = lw[lo:hi]
    q.put((rank,) + _draws(ws, st))
    dist.barrier()
    dist.destroy_process_group()


def _spawn(target, world, port, *args):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=target, args=(r, world, port, *args, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = sorted((q.get(timeout=300) for _ in range(world)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return out


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_draw_equals_single_gpu(world):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    import wsb200 as ws
    lw, a, b = _inputs()
    single = ws.SMCState(N, device=0, seed=31)
    single.store.setcol("a", a)
    single.store.setcol("b", b)
    single.weights = lw
    idx1, bits1 = _draws(ws, single)
    assert np.array_equal(np.sort(idx1[2]), np.arange(N))
    for o in _spawn(_worker, world, 29960 + world):
        for x, y in zip(o[1], idx1):
            np.testing.assert_array_equal(x, y)
        for x, y in zip(o[2], bits1):
            np.testing.assert_array_equal(x, y)


def _worker_ssm(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import models
    import wsb200 as ws
    st = ws.sharded_state(N, device=rank, seed=13, ess_perc_min=0.8)
    obs = list(np.cumsum(np.random.default_rng(7).standard_normal(20)))
    ws.run(ws.model(models.SSM1D)(obs), st)
    stream, seed = ctypes.c_uint64(), ctypes.c_uint64()
    st.store._call("ws_next_philox_stream", ctypes.byref(stream), ctypes.byref(seed))
    df = ws.sample(st, 3000)
    names = st.store.colnames()
    shards = {nm: st[nm] for nm in names}
    q.put((rank, stream.value, seed.value, st.weights, shards, {nm: df[nm].to_numpy() for nm in names}, list(df.columns)))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_ssm_rows_equal_the_concatenated_shards():
    world = 2
    if _ngpu() < world:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import sample_spec as S
    out = _spawn(_worker_ssm, world, 29990)
    lw = np.concatenate([o[3] for o in out])
    idx = S.sample_indices_spec(lw, out[0][2], out[0][1], 3000, True)
    for o in out:
        assert o[1] == out[0][1] and o[6] == out[0][6]
        for nm in o[6]:
            full = np.concatenate([p[4][nm] for p in out])
            np.testing.assert_array_equal(o[5][nm], full[idx])
