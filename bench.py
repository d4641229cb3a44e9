#!/usr/bin/env python
"""bench.py — particle-updates/s of the 2-D SSM bootstrap filter (BASELINE.json configs[1]).

A "step" is one time step of the filter-only form of examples/2D_ssm.jl over all N particles:
    x .= x + v ; dv ~ MvNormal([0,0], 0.1 I2) ; v .= v + dv ; o => MvNormal(x, 0.5 I2) ; Resample()
with ess_perc_min = 1.0, so the stratified resample + gather of all six planes runs every step (the
setting of the reference's own benchmark, benchmarks/ssm/WeightedSampling/lgssm1d.jl:26-27).
particle-updates/s = N * steps / time.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--particles N] [--impl reference] [--dump-outputs DIR]

* `value`     device time of the K steps (CUDA events on the library's stream), library timing hooks OFF.
* `e2e`       the same K steps through the public API (wsb200.run of the @model program) with host
              inputs (the observations) and a device->host read of the step result (log-evidence)
              inside the timed region, wall clock.
* `roofline`  the dominant kernel (the fused propagate + observe pass, which also performs the deferred
              ancestor gather) against the measured HBM copy bandwidth; per-kernel times come from a SECOND,
              separately run pass of the same steps with the library's per-kernel CUDA events switched on
              (`ws_set_timing` adds event records, so it stays out of the headline region).
* `sharded_parity` (N > 1)  before the timed region the ranks run a small sharded filter (n = 200 003, T = 12)
              through both exchange paths and rank 0 compares it, particle for particle, with the same filter on
              one GPU.
* `cpu_baseline` / `--impl reference`  the C restatement of the reference's run! (oracle/ws_oracle.c:
              orc_ssm2d_run) on one host core (the reference is single-threaded: TODO.md:28).  Julia is
              not available, so this is "kind: port".
* `--dump-outputs DIR`  after the timed steps, writes what they computed as DIR/<name>.npy (float64): the particle
              columns x, v, dv and the log-weights at a fixed, seeded sample of particles, and the log-evidence.  The
              inputs depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SSM2D_FILTER = '''
@model function ssm2d_filter(obs)
    I2 = [1.0 0.0; 0.0 1.0]
    x .= [0.0, 0.0]
    v .= [1.0, 0.0]
    for o in obs
        x .= x + v
        dv ~ MvNormal([0.0, 0.0], 0.1 * I2)
        v .= v + dv
        o => MvNormal(x, 0.5 * I2)
    end
end
'''

P_PLANES = 6
# algorithmic bytes per particle-update (SURVEY.md §8d, C2 filter-only, Int32 ancestors)
ALG_BYTES_STEP = 224
ALG_BYTES_GATHER = 4 + 16 * P_PLANES          # eager mode only: read ancestor + read/write 6 planes
ALG_BYTES_PASS_EAGER = 8 * (4 + 6) + 16       # propagate+observe: read x,v; write x,v,dv; logw RMW
# deferred gather (default): the fused pass reads x,v THROUGH the ancestors (4 B index), writes x,v,dv and
# writes logw = c + logpdf (after a resample the old log-weights are one scalar c: no read); dv is never
# gathered because it is overwritten before it is read
ALG_BYTES_PASS_LAZY = 4 + 8 * 4 + 8 * 6 + 8
ALG_BYTES_SCAN = 8 + 4                        # read logw, write ancestor
NECESSARY_BYTES_STEP_LAZY = ALG_BYTES_PASS_LAZY + ALG_BYTES_SCAN


def synth_obs(T, seed=42):
    """examples/2D_ssm.jl:19-28 generative process (SURVEY §8d C2 input)."""
    rng = np.random.default_rng(seed)
    x = np.array([0.0, 0.0])
    v = np.array([1.0, 0.0])
    obs = []
    for _ in range(T):
        obs.append(x + 0.5 * rng.standard_normal(2))
        x = x + v
        v = v + 0.1 * rng.standard_normal(2)
    return obs


def measured_traffic(kernel_prefix, n):
    """DRAM bytes per launch of a kernel from the committed ncu --set full capture (profiles/ncu_traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum per particle at N = 2e7), scaled to this run's N."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        t = json.load(f)["kernels"]
    for name, k in t.items():
        if name.startswith(kernel_prefix):
            return k["bytes_per_particle"] * n
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    def __init__(self, device_index):
        super().__init__(daemon=True)
        self.idx = device_index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nm, val in zip(names, out[2:]):
                    if val.strip().lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


PARITY_MODEL = '''
@model function ssm(obs)
    I2 = [1.0 0.0; 0.0 1.0]
    x .= [0.0, 0.0]
    v .= [1.0, 0.0]
    for o in obs
        x .= x + v
        dv ~ MvNormal([0.0, 0.0], 0.1 * I2)
        v .= v + dv
        o => MvNormal(x, 0.5 * I2)
    end
end
'''


def sharded_parity(ws, dist, torch, local_rank, rank, world, n=200_003, T=12):
    """tests/test_gpu_sharded.py::test_sharded_equals_single_gpu inside the bench (the driver's GPU test box has one
    GPU, so this is where the multi-GPU path is checked on the final code): one global filter sharded over the
    ranks == the same filter on one GPU, for the direct (peer-store) and the ncclSend/Recv exchange."""
    import ctypes as C
    rng = np.random.default_rng(3)
    obs = [np.array([t, 0.0]) + 0.7 * rng.standard_normal(2) for t in range(T)]
    root_of = ws.model(PARITY_MODEL)
    out = {"n": n, "T": T, "world": world, "paths": {}}
    single = None
    if rank == 0:
        st1 = ws.SMCState(n, device=local_rank, seed=77, ess_perc_min=1.0)
        ws.run(root_of(obs), st1)
        single = (st1["x"], st1["v"], st1.weights, ws.log_evidence(st1), st1.stats()["resamples_done"])
        del st1
    for path in ("push", "nccl"):
        old = os.environ.get("WSB200_EXCHANGE")
        if path == "nccl":
            os.environ["WSB200_EXCHANGE"] = "nccl"
        else:
            os.environ.pop("WSB200_EXCHANGE", None)
        st = ws.sharded_state(n, device=local_rank, seed=77, ess_perc_min=1.0)
        if old is None:
            os.environ.pop("WSB200_EXCHANGE", None)
        else:
            os.environ["WSB200_EXCHANGE"] = old
        ws.run(root_of(obs), st)
        le = ws.log_evidence(st)
        mig, pushed = C.c_int64(), C.c_int64()
        st.store._call("ws_get_migrated", C.byref(mig))
        st.store._call("ws_get_pushed", C.byref(pushed))
        mine = (rank, st["x"], st["v"], st.weights, le, st.stats()["resamples_done"], mig.value, pushed.value)
        box = [None] * world if rank == 0 else None
        dist.gather_object(mine, box, dst=0)
        del st
        if rank == 0:
            box.sort(key=lambda t: t[0])
            xs = np.concatenate([b[1] for b in box])
            vs = np.concatenate([b[2] for b in box])
            wts = np.concatenate([b[3] for b in box])
            x1, v1, w1, le1, nres1 = single
            bad = ((np.abs(xs - x1) > 1e-9 * (1 + np.abs(x1))).any(axis=1) |
                   (np.abs(vs - v1) > 1e-9 * (1 + np.abs(v1))).any(axis=1) |
                   (np.abs(wts - w1) > 1e-9 * (1 + np.abs(w1))))
            out["paths"][path] = {
                "mismatches": int(bad.sum()), "bit_identical_particles": int(((xs == x1).all(axis=1) & (vs == v1).all(axis=1)).sum()),
                "log_evidence_max_rel_err": float(max(abs(b[4] - le1) for b in box) / abs(le1)),
                "resamples": [int(b[5]) for b in box], "resamples_single_gpu": int(nres1),
                "migrated": int(sum(b[6] for b in box)), "pushed": int(sum(b[7] for b in box))}
    if rank == 0:
        out["mismatches"] = max(p["mismatches"] for p in out["paths"].values())
        out["exchange"] = "push" if out["paths"]["push"]["pushed"] > 0 else "nccl"
    return out


DUMP_PARTICLES = 1_000_000      # 7 float64 values per sampled particle: 56 MB in all, whatever --particles is


def dump_outputs(state, le, out_dir, rank, world):
    """Writes the state a caller of ws.run holds after the timed steps.  The sample of particles is seeded, so it
    depends only on the particle count; rows are read through the deferred ancestors, which leaves the state as it was."""
    import ctypes as C
    st = state.store
    m = min(st.n, DUMP_PARTICLES // world)
    rows = np.sort(np.random.default_rng(0).choice(st.n, size=m, replace=False)).astype(np.int64)
    out = {"log_evidence": np.array([le]), "log_weights": state.weights[rows]}
    for name in ("x", "v", "dv"):
        cid, width = st._lookup(name)
        planes = np.empty((width, m))
        st._call("ws_col_download_rows", cid, rows.ctypes.data_as(C.c_void_p), m, planes.ctypes.data_as(C.c_void_p))
        out[name] = np.ascontiguousarray(planes.T)
    os.makedirs(out_dir, exist_ok=True)
    suffix = "" if world == 1 else f"_rank{rank}"
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def cpu_reference_run(n, steps, seed=1):
    """The reference's run! restated in C (oracle/ws_oracle.c), one core."""
    from oracle import cref
    obs = np.asarray(synth_obs(steps))
    t0 = time.perf_counter()
    le, mean, nres = cref.ssm2d_run(n, obs, seed=seed, ess_perc_min=1.0)
    dt = time.perf_counter() - t0
    return n * steps / dt, dt, le


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.cpu_particles
    # warm-up (page faults, ziggurat tables), then K samples of a bounded run
    cpu_reference_run(min(n, 200_000), 2)
    vals = []
    t_total0 = time.perf_counter()
    for _ in range(max(1, min(args.steps, 3))):
        v, dt, _ = cpu_reference_run(n, args.cpu_steps)
        vals.append(v)
    value = float(np.median(vals))
    ms = 1e3 * n / value
    line = {
        "impl": "reference", "metric": "particle_updates_per_sec", "value": value, "unit": "particle-updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "ssm2d_filter_only_bootstrap (examples/2D_ssm.jl, x overwritten), ess_perc_min=1.0",
                   "particles": n, "time_steps_per_sample": args.cpu_steps},
        "cpu_baseline": {"value": value, "unit": "particle-updates/s", "cores": 1, "kind": "port",
                         "sample": f"{n} particles x {args.cpu_steps} steps, C restatement of run! (oracle/ws_oracle.c), "
                                   f"median of {len(vals)} runs; Julia unavailable"},
        "e2e": {"value": value, "unit": "particle-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.perf_counter() - t_total0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--particles", type=int, default=100_000_000)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-particles", type=int, default=2_000_000)
    ap.add_argument("--cpu-steps", type=int, default=40)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the sharded == single-GPU check that precedes an N > 1 run")
    ap.add_argument("--profile-steps", type=int, default=10, help="steps of the second pass that times each kernel class")
    ap.add_argument("--skew", type=float, default=2.0, help="N > 1: rank skew of the extra migration-heavy Resample (0 = skip it)")
    ap.add_argument("--eager-gather", action="store_true", help="gather every column inside Resample (reference order of work)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed steps computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import wsb200 as ws

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: wsb200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    parity = None
    if world > 1 and not args.no_parity:
        parity = sharded_parity(ws, dist, torch, local_rank, rank, world)
        dist.barrier()

    N = args.particles
    K, W = args.steps, args.warmup
    KP = max(3, min(K, args.profile_steps))        # steps of the per-kernel (timing hooks on) pass
    obs = synth_obs(W + K + KP)
    build = ws.model(SSM2D_FILTER)

    if world > 1:
        # one GLOBAL filter of N * world particles, sharded by slot range; exact global resampling
        state = ws.sharded_state(N * world, ess_perc_min=1.0, seed=1234, device=local_rank)
    else:
        state = ws.SMCState(N, ess_perc_min=1.0, seed=1234, device=local_rank)
    st = state.store
    import ctypes as C
    sp = C.c_void_p()
    st._call("ws_stream", C.byref(sp))
    stream = torch.cuda.ExternalStream(sp.value, device=torch.device("cuda", local_rank))

    # warm-up: initial assigns + W steps (also creates the columns)
    ws.run(build(obs[:W]), state)
    state.sync()
    le0 = ws.log_evidence(state)

    # the timed region continues the same filter with the next K observations (run! on an existing
    # state, as benchmarks/ssm/bench_single_update does).  The continuation model has no initial
    # assigns.
    cont = ws.model('''
    @model function ssm2d_continue(obs)
        I2 = [1.0 0.0; 0.0 1.0]
        for o in obs
            x .= x + v
            dv ~ MvNormal([0.0, 0.0], 0.1 * I2)
            v .= v + dv
            o => MvNormal(x, 0.5 * I2)
        end
    end
    ''', particle_vars=("x", "v", "dv"))

    if args.eager_gather:
        st._call("ws_set_lazy_gather", 0)
    stats0 = state.stats()
    mig0c = C.c_int64()
    st._call("ws_get_migrated", C.byref(mig0c))
    mig0 = mig0c.value
    sampler = ClockSampler(local_rank)
    sampler.start()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the K steps are issued as up to four consecutive run! calls with an event between them: the total is what is
    # reported, the pieces show the spread inside the timed region
    n_chunks = min(4, K)
    cuts = [W + (K * i) // n_chunks for i in range(n_chunks + 1)]
    roots = [cont(obs[a:b]) for a, b in zip(cuts[:-1], cuts[1:])]
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_chunks + 1)]
    barrier()
    t0 = time.perf_counter()
    evs[0].record(stream)
    for i, root in enumerate(roots):
        ws.run(root, state)
        if i + 1 < n_chunks:
            evs[i + 1].record(stream)
    le = ws.log_evidence(state)          # device -> host read of the step result
    evs[n_chunks].record(stream)
    state.sync()
    t1 = time.perf_counter()
    barrier()
    dev_ms = evs[0].elapsed_time(evs[n_chunks])
    wall_ms = (t1 - t0) * 1e3
    chunk_ms_per_step = [evs[i].elapsed_time(evs[i + 1]) / (cuts[i + 1] - cuts[i]) for i in range(n_chunks)]
    clocks = sampler.stop()
    stats1 = state.stats()
    if args.dump_outputs:
        dump_outputs(state, le, args.dump_outputs, rank, world)
    # second pass, NOT part of the headline: the same filter continues for KP steps with per-kernel events on
    st._call("ws_set_timing", 1)
    st._call("ws_reset_kernel_times")
    evp0, evp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evp0.record(stream)
    ws.run(cont(obs[W + K:W + K + KP]), state)
    evp1.record(stream)
    state.sync()
    prof_ms = evp0.elapsed_time(evp1)
    kt = state.kernel_times()
    st._call("ws_set_timing", 0)
    mbx = C.c_int64()
    st._call("ws_get_mailbox_exchanges", C.byref(mbx))
    mailbox_exchanges = int(mbx.value)   # > 0: the small exchanges of the sharded steps went through the mailboxes (0 on one GPU)

    # N > 1: one more step, NOT part of the headline, with the weights skewed ACROSS ranks (rank r's log-weights are
    # lowered by skew * r, so the low ranks hold almost all of the mass): most offspring of the following Resample
    # must cross shard boundaries, which the near-uniform weights of the filter never make them do.  Reported against
    # the NVLink peer bandwidth (770 GB/s per direction, B200_PROFILING.md).
    migration = None
    if world > 1 and args.skew > 0:
        first_ms = None
        for rep in range(2):     # the first such step also sizes the staging / spare buffers for this much migration: warm-up
            p0, m0 = C.c_int64(), C.c_int64()
            st._call("ws_get_pushed", C.byref(p0))
            st._call("ws_get_migrated", C.byref(m0))
            ws.Weight(None, (ws.col("x")[0] * 0.0 - args.skew * rank,)).apply(state)
            state.sync()
            barrier()
            evm0, evm1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            evm0.record(stream)
            ws.Resample().apply(state)
            state.store._call("ws_flush")
            evm1.record(stream)
            state.sync()
            barrier()
            if rep == 0:
                first_ms = evm0.elapsed_time(evm1)
        p1, m1 = C.c_int64(), C.c_int64()
        st._call("ws_get_pushed", C.byref(p1))
        st._call("ws_get_migrated", C.byref(m1))
        t = torch.tensor([evm0.elapsed_time(evm1), float(p1.value - p0.value), float(m1.value - m0.value)], device="cuda", dtype=torch.float64)
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        mig_ms, sent_max, recv_max = float(tmax[0]), float(tmax[1]), float(tmax[2])
        bytes_per_particle = 8 * P_PLANES
        busiest = max(sent_max, recv_max) * bytes_per_particle
        migration = {"skew": args.skew, "ms": mig_ms, "first_ms_this_rank": first_ms, "migrated_particles_total": float(tsum[2]),
                     "sent_particles_busiest_rank": sent_max, "received_particles_busiest_rank": recv_max,
                     "bytes_per_particle": bytes_per_particle,
                     "nvlink_gbs_busiest_rank": busiest / (mig_ms * 1e-3) / 1e9 if mig_ms > 0 else None,
                     "nvlink_peak_gbs_per_direction": 770.0,
                     "nvlink_frac": busiest / (mig_ms * 1e-3) / 1e9 / 770.0 if mig_ms > 0 else None,
                     "note": "one Resample (scan, search, exchange, gather of 6 planes) after rank-skewed weights, second of two such steps; the NVLink "
                             "figure divides the busiest rank's migrated bytes by the WHOLE step time"}
    mig = C.c_int64()
    st._call("ws_get_migrated", C.byref(mig))
    migrated_per_step = (mig.value - mig0) / max(1, K)

    if world > 1:
        t = torch.tensor([dev_ms, wall_ms, migrated_per_step], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms, migrated_per_step = float(t[0]), float(t[1]), float(t[2])

    total_updates = float(N) * K * world
    value = total_updates / (dev_ms * 1e-3)
    e2e = total_updates / (wall_ms * 1e-3)
    launches = stats1["kernel_launches"] - stats0["kernel_launches"]

    peak, peak_src = measured_peaks()
    per_kernel = {}
    eager = args.eager_gather
    pass_bytes = ALG_BYTES_PASS_EAGER if eager else ALG_BYTES_PASS_LAZY
    for name, alg in (("gather", ALG_BYTES_GATHER), ("fused_pass", pass_bytes), ("scan_search", ALG_BYTES_SCAN)):
        k = kt[name]
        if name == "gather" and not eager:
            continue    # deferred gather: this class only stages the few offspring that migrate between ranks
        if k["launches"] > 0 and k["ms"] > 0:
            avg_ms = k["ms"] / max(1, KP)    # per step (a sharded step times the search in two regions)
            gbs = alg * N / (avg_ms * 1e-3) / 1e9
            per_kernel[name] = {"avg_ms": avg_ms, "launches": k["launches"], "alg_bytes_per_particle": alg,
                                "achieved_gbs": gbs, "frac": gbs / peak, "share_of_step": k["ms"] / prof_ms}
    dom = max(per_kernel, key=lambda n: per_kernel[n]["avg_ms"]) if per_kernel else None
    roofline = None
    if dom:
        sl = stats1["sl_passes"] - stats0["sl_passes"]
        vm_name = "ws_vm_sl_kernel<WsSigSsm2d>" if sl > 0 else "ws_vm_kernel"
        scan_form = os.environ.get("WSB200_SCAN", "3pass") if world == 1 else "3pass"
        scan_name = {"chain": "ws_chain_kernel", "1pass": "ws_scan_search_kernel"}.get(
            scan_form, "ws_cdf_tiles_kernel + ws_cdf_group_offsets_kernel + ws_search_kernel")
        roofline = {"bound": "hbm", "kernel": {"gather": "ws_gather_kernel", "fused_pass": vm_name, "scan_search": scan_name}[dom],
                    "achieved": per_kernel[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                    "frac": per_kernel[dom]["frac"],
                    "traffic": measured_traffic({"gather": "ws_gather_kernel", "fused_pass": vm_name.split("<")[0],
                                                 "scan_search": scan_name.split(" ")[0]}[dom], N),
                    "traffic_source": "profiles/ncu_traffic.json (ncu --set full, bytes per particle at N=2e7) x N",
                    "peak_source": peak_src,
                    "per_kernel": per_kernel,
                    "per_kernel_source": f"second pass of {KP} steps with ws_set_timing(1): {prof_ms / KP:.3f} ms/step "
                                         f"(headline, hooks off: {dev_ms / K:.3f} ms/step)",
                    "whole_step": {"alg_bytes_per_particle": ALG_BYTES_STEP,
                                   "achieved_gbs": ALG_BYTES_STEP * N * K / (dev_ms * 1e-3) / 1e9,
                                   "frac": ALG_BYTES_STEP * N * K / (dev_ms * 1e-3) / 1e9 / peak,
                                   "note": "224 B is SURVEY §8(d)'s figure for the reference's order of work (eager "
                                           "6-plane gather); the deferred-gather design only has to move "
                                           f"{NECESSARY_BYTES_STEP_LAZY} B per particle-update",
                                   "necessary_bytes_per_particle": None if eager else NECESSARY_BYTES_STEP_LAZY,
                                   "frac_of_necessary": None if eager else
                                   NECESSARY_BYTES_STEP_LAZY * N * K / (dev_ms * 1e-3) / 1e9 / peak}}

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:   # reported at N = 1 only (rank 0)
            cpu_reference_run(200_000, 2)
            v, dt, _ = cpu_reference_run(args.cpu_particles, args.cpu_steps)
            cpu = {"value": v, "unit": "particle-updates/s", "cores": 1, "kind": "port",
                   "sample": f"{args.cpu_particles} particles x {args.cpu_steps} steps of the same model, C restatement of "
                             f"the reference's run! (oracle/ws_oracle.c), {dt:.1f} s; Julia unavailable in the image"}
        line = {
            "metric": "particle_updates_per_sec", "value": value, "unit": "particle-updates/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "ssm2d_filter_only_bootstrap (BASELINE configs[1]: examples/2D_ssm.jl with x overwritten), "
                                   "ess_perc_min=1.0 (resample + 6-plane gather every step)",
                       "particles_per_gpu": N, "planes": P_PLANES, "resampler": "stratified",
                       "parallelism": "single GPU" if world == 1 else
                       f"{world} ranks: ONE filter of {N * world} particles sharded by slot range; exact global stratified "
                       "resampling; the step's small exchanges ((m,S,Q) triples, CDF masses, slot bounds, barrier) are stored by the "
                       "kernels into peer-mapped mailboxes over NVLink (NCCL collectives as fallback); migrating offspring are written "
                       "straight into the destination rank's planes over NVLink by the gather kernel (ncclSend/Recv as fallback)",
                       "mailbox_exchanges": mailbox_exchanges,
                       "migrated_particles_per_step": migrated_per_step,
                       "l2": "working set 10.4 GB per GPU >> 126 MB L2 (no flush needed)",
                       "log_evidence": le, "log_evidence_after_warmup": le0},
            "roofline": roofline, "cpu_baseline": cpu,
            "e2e": {"value": e2e, "unit": "particle-updates/s", "h2d_bytes_per_step": 16,
                    "d2h_bytes_per_step": int((stats1["d2h_bytes"] - stats0["d2h_bytes"]) / max(1, K))},
            "gpu_launches": int(launches), "clocks": clocks,
            "ms_per_step_chunks": chunk_ms_per_step, "sharded_parity": parity,
            "ess_knife_edge_steps": state.ess_ties(), "migration": migration,
            "fusion": {"fused_passes": stats1["fused_passes"] - stats0["fused_passes"],
                       "fused_statements": stats1["fused_statements"] - stats0["fused_statements"],
                       "straight_line_passes": stats1["sl_passes"] - stats0["sl_passes"],
                       "resamples": stats1["resamples_done"] - stats0["resamples_done"]},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
