"""Hidden Markov model filter step on one GPU, against the LGSSM-1D step at the same N.
usage: python benchmarks/run_hmm.py [--n 1000000 100000000] [--k 2 8 64] [--steps 200] [--warmup 20] [--out FILE]

HMM step:      s ~ Categorical(P[s, :]) ; y => Normal(mu[s], 1.0) ; Resample()
LGSSM-1D step: x ~ Normal(0.9 x, 1.0)   ; y => Normal(x, 0.5)     ; Resample()
ess_perc_min = 1.0, so the stratified resample runs every step (as bench.py).  The timed region is `--steps` steps
issued as one run! that continues a filter warmed up by `--warmup` steps; its device time comes from CUDA events on the
library's stream.  hbm_share: SURVEY §8(d)'s 80 bytes per particle-update at 7.7 TB/s over the measured step.
Prints one JSON line per (model, K, N); the first line names the card and its power limit."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import wsb200 as ws

BYTES_PER_UPDATE = 80.0
HBM_BYTES_PER_S = 7.7e12

HMM_INIT = '''
@model function hmm_init(p0)
    s ~ Categorical(p0)
end
'''
HMM_STEP = '''
@model function hmm_step(ys, P, mu)
    for y in ys
        s ~ Categorical(P[s, :])
        y => Normal(mu[s], 1.0)
    end
end
'''
LG_INIT = '''
@model function lg_init()
    x ~ Normal(0.0, 1.0)
end
'''
LG_STEP = '''
@model function lg_step(ys)
    for y in ys
        x ~ Normal(0.9 * x, 1.0)
        y => Normal(x, 0.5)
    end
end
'''


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        name, power = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the timings stand without it; say so
        return {"gpu": "unknown", "power_limit": f"not read ({type(e).__name__})"}


def timed_steps(torch, n, init, step, args_of, steps, warmup):
    state = ws.SMCState(n, ess_perc_min=1.0, seed=1234, device=0)
    sp = C.c_void_p()
    state.store._call("ws_stream", C.byref(sp))
    stream = torch.cuda.ExternalStream(sp.value, device=torch.device("cuda", 0))
    ws.run(init, state)
    ws.run(step(*args_of(warmup)), state)
    state.sync()
    root = step(*args_of(steps))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    ws.run(root, state)
    le = ws.log_evidence(state)
    e1.record(stream)
    state.sync()
    ms = e0.elapsed_time(e1) / steps
    fired = state.stats()["resamples_done"]
    del state
    return ms, le, fired


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, nargs="+", default=[1_000_000, 100_000_000])
    ap.add_argument("--k", type=int, nargs="+", default=[2, 8, 64])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("run_hmm.py measures on a CUDA device; none is available")
    lines = [dict(card(), steps=a.steps, warmup=a.warmup)]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(0)
    ys = rng.standard_normal(a.steps + a.warmup)

    def record(rec, n, ms):
        rec.update(n_particles=n, ms_per_step=round(ms, 4), particle_updates_per_s=n / (ms * 1e-3),
                   hbm_share=round(BYTES_PER_UPDATE * n / HBM_BYTES_PER_S / (ms * 1e-3), 3))
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    for n in a.n:
        ms, le, fired = timed_steps(torch, n, ws.model(LG_INIT)(), ws.model(LG_STEP, particle_vars=("x",)),
                                    lambda t: (list(ys[:t]),), a.steps, a.warmup)
        record(dict(model="lgssm1d", log_evidence=le, resamples=fired), n, ms)
        for K in a.k:
            P = 0.8 * np.eye(K) + 0.2 * rng.dirichlet(np.ones(K), size=K)
            P /= P.sum(axis=1, keepdims=True)
            mu = np.linspace(-2.0, 2.0, K)
            ms, le, fired = timed_steps(torch, n, ws.model(HMM_INIT)(np.full(K, 1.0 / K)), ws.model(HMM_STEP, particle_vars=("s",)),
                                        lambda t: (list(ys[:t]), P, mu), a.steps, a.warmup)
            record(dict(model="hmm", K=K, log_evidence=le, resamples=fired), n, ms)
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
