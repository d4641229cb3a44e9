"""sample(state, n; replace) at N = 1e8 particles on one GPU: the device index draw (ws_sample_indices) and the whole
ws.sample (indices + the drawn rows of one column), for log-weights s * z, z standard normal.
usage: python benchmarks/run_sample.py [--n 100000000] [--reps 3] [--out FILE]
Prints one JSON line per (s, replace, n); times are host clock around a call that ends in a device synchronise,
the median of --reps calls after one warm-up call of the same shape.  d2h_bytes: the device-to-host bytes of one call
(ws_get_stats).  The first line names the card and its power limit."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import wsb200 as ws


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        name, power = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the timings stand without it; say so
        return {"gpu": "unknown", "power_limit": f"not read ({type(e).__name__})"}


def timed(fn, st, reps):
    fn()  # warm-up of this shape
    ts, moved = [], []
    for _ in range(reps):
        b = st.stats()["d2h_bytes"]
        t0 = time.perf_counter()
        fn()
        st.sync()
        ts.append(time.perf_counter() - t0)
        moved.append(st.stats()["d2h_bytes"] - b)
    return float(np.median(ts)) * 1e3, int(moved[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = [dict(card(), n_particles=a.n)]
    print(json.dumps(lines[0]), flush=True)
    z = np.random.default_rng(0).standard_normal(a.n)
    for s in (0.5, 3.0):
        st = ws.SMCState(a.n, device=0, seed=1)
        st.store.setcol("x", z)
        st.weights = s * z
        ws.log_evidence(st)  # the log-weight reduction, outside the timed calls
        for replace, ns in ((True, (1_000, 1_000_000, 100_000_000)), (False, (1_000, 1_000_000))):
            for n in ns:
                idx = np.empty(n, dtype=np.int64)
                draw = lambda: st.store._call("ws_sample_indices", n, int(replace), idx.ctypes.data_as(C.c_void_p))
                ms_idx, b_idx = timed(draw, st, a.reps)
                ms_all, b_all = timed(lambda: ws.sample(st, n, replace=replace), st, a.reps)
                rec = dict(s=s, replace=replace, n=n, index_draw_ms=round(ms_idx, 3), sample_ms=round(ms_all, 3),
                           index_draw_d2h_bytes=b_idx, sample_d2h_bytes=b_all, host_path_before="not measured")
                lines.append(rec)
                print(json.dumps(rec), flush=True)
        del st
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
