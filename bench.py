#!/usr/bin/env python
"""MPC solves/sec of the B200 path on the BASELINE.json workloads.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c1|c2|c3|c4|c5] [--batch B]
                    [--scaling weak|strong] [--impl reference] [--no-cpu-baseline] [--dump-outputs DIR]

Default = configs[2] (C3): 4096 independent CaltechACN 54-EVSE x 288-period instances per GPU.  A step = one pass of the
whole hot path over the batch, as SURVEY.md 8(d) defines a solve: pack -> iterate (to the certified 1e-4 gap) ->
polish -> postprocess (continuous pilot projection).

* `value`  : raw session tables / prices / previous peaks RESIDENT in HBM when the timed region starts; timed = the
             device packer (acb_pack_sessions) + acb_solve_batch (whose epilogue projects the pilots).  K steps are
             enqueued double-buffered on two streams (a production pipeline never drains the GPU between batches), one
             pair of CUDA events around all K.
* `e2e`    : the public batched call BatchedAdaptiveCharging.schedule_async on HOST arrays: staging into pinned memory,
             H2D, pack, solve, projection, D2H of the float64 pilots of every instance; same double buffering.
* `latency`: one AdaptiveChargingOptimization.solve() call (the reference's own usage: one solve per control step) on
             a C1 and a C2 instance, host objects in, numpy out.
* `parity_sample`: 256 instances spread over the batch against oracle optima precomputed by
             tests/golden/make_bench_golden.py (objective within 1e-4 |f*|, violation, energy, bounds).
* `--impl reference`: the CPU oracle (float64 restatement of the reference's cvxpy/ECOS path, which cannot run here:
             cvxpy / ECOS / acnportal are not installed) on ALL host cores, one persistent pool.
* `--dump-outputs DIR`: after the timed steps, what the last timed step of `value` handed to its caller (C4: the last
             control step of the replay) is written as DIR/<name>.npy, float32 or float64, rank 0's instances.  The
             inputs depend on the arguments only, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "mpc_solves_per_sec_1e-4_rel_gap"
UNIT = "solves/s"
BENCH_OBJECTIVE = [("tou_energy_cost", 1.0, {}), ("total_energy", 0.3, {}), ("demand_charge", 1.0 / 30.0, {})]
C1_OBJECTIVE = [("quick_charge", 1.0, {}), ("equal_share", 1e-3, {})]
C5_OBJECTIVE = [("load_flattening", 1.0, {}), ("non_completion_penalty", 100.0, {})]
GOLDEN = os.path.join(ROOT, "tests", "golden", "bench_c3_golden.json")

CONFIGS = {
    "c1": dict(workload="C1: single-phase 30-EVSE network, 30 sessions, T=144, quick_charge + 1e-3*equal_share (BASELINE configs[0])",
               N=30, T=144, M=1, S_max=30, objective=C1_OBJECTIVE, batch=1, horizon=144),
    "c2": dict(workload="C2: CaltechACN three-phase 54-EVSE network, SOC constraints, T=288, tou_energy_cost + 0.3*total_energy + (1/30)*demand_charge (BASELINE configs[1])",
               N=54, T=288, M=8, S_max=54, objective=BENCH_OBJECTIVE, batch=1, horizon=288),
    "c3": dict(workload="C3: batch of independent CaltechACN three-phase 54-EVSE MPC instances, SOC constraints, T=288, "
                        "tou_energy_cost + 0.3*total_energy + (1/30)*demand_charge, randomised sessions/prices (BASELINE configs[2])",
               N=54, T=288, M=8, S_max=54, objective=BENCH_OBJECTIVE, batch=4096, horizon=288),
    "c4": dict(workload="C4: closed-loop warm-started replay of 1024 CaltechACN-shaped sites at 5-minute steps, sites sharded over the GPUs "
                        "(BASELINE configs[3]; a bench step = one control step of every site)",
               N=54, T=288, M=8, S_max=54, objective=BENCH_OBJECTIVE, batch=1024, horizon=128),
    "c5": dict(workload="C5: 1000-EVSE hierarchical three-phase network (86 constraint rows), T=288, load_flattening + 100*non_completion_penalty "
                        "(BASELINE configs[4]; general streaming path)",
               N=1000, T=288, M=86, S_max=1000, objective=C5_OBJECTIVE, batch=128, horizon=288),
}


def objective_components(spec):
    import adacharge_b200 as ab

    return [ab.ObjectiveComponent(getattr(ab, n), c, k) for n, c, k in spec]


def config_dict(cfg, seed, infra):
    from adacharge_b200.generators import config_c1, config_c2, config_c5

    if cfg == "c1":
        return config_c1(seed)
    if cfg == "c5":
        return config_c5(seed, infra=infra)
    return config_c2(seed, infra=infra, price_noise=0.2 if cfg == "c3" else 0.0)


def make_workload(cfg, batch, seed0):
    """Raw host arrays of `batch` synthetic instances (seed = seed0 + index): what an acnportal Interface would hand over."""
    from adacharge_b200.generators import caltech_acn_infrastructure, hierarchical_three_phase_network
    from adacharge_b200.batched import SESSION_FIELDS

    C = CONFIGS[cfg]
    infra = None if cfg == "c1" else (hierarchical_three_phase_network(1000) if cfg == "c5" else caltech_acn_infrastructure())
    S, Tp = C["S_max"], C["horizon"]
    sess = {n: np.zeros((batch, S), dtype=dt) for n, dt in SESSION_FIELDS}
    sess["station"][...] = -1
    prices = np.zeros((batch, Tp))
    prev = np.zeros(batch)
    ext = np.zeros((batch, Tp)) if cfg == "c5" else None
    dc = 15.51
    for b in range(batch):
        d = config_dict(cfg, seed0 + b, infra)
        inf = d["infrastructure_info"]
        index = {sid: i for i, sid in enumerate(inf["station_ids"])}
        for j, s in enumerate(d["active_sessions"]):
            sess["station"][b, j] = index[s["station_id"]]
            sess["arrival_offset"][b, j] = s["arrival"]
            sess["remaining_time"][b, j] = s["departure"] - s["arrival"]
            sess["remaining_demand"][b, j] = s["requested_energy"] - s["energy_delivered"]
            sess["min_rate"][b, j] = s["min_rates"]
            sess["max_rate"][b, j] = s["max_rates"]
        if "prices" in d:
            prices[b] = np.asarray(d["prices"])[:Tp]
        prev[b] = d.get("prev_peak", 0.0)
        if ext is not None:
            ext[b] = np.asarray(d["external_signal"])[:Tp]
        dc = d.get("demand_charge", dc)
        if infra is None:
            infra = inf  # C1 builds its own (identical) single-phase network per seed
    return dict(infra=infra, sessions=sess, prices=prices, prev_peak=prev, external_signal=ext, demand_charge=dc)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def _oracle_one(job):
    cfg, seed = job
    from adacharge_b200.interface import TestingInterface
    from adacharge_b200.generators import caltech_acn_infrastructure, hierarchical_three_phase_network
    from oracle import mpc

    infra = None if cfg == "c1" else (hierarchical_three_phase_network(1000) if cfg == "c5" else caltech_acn_infrastructure())
    d = config_dict(cfg, seed, infra)
    iface = TestingInterface(d)
    S, I = iface.active_sessions(), iface.infrastructure_info()
    spec = [(n, c, dict(k, **({"external_signal": d["external_signal"]} if n == "load_flattening" and "external_signal" in d else {}))) for n, c, k in CONFIGS[cfg]["objective"]]
    t = time.perf_counter()
    if _cpu_kind(cfg) == "reference":  # the unmodified reference (cvxpy front end) where it can run: never in this image
        from oracle import reference_cvxpy

        R = np.asarray(reference_cvxpy.solve_reference(spec, S, I, iface, "SOC", False, None, iface.get_prev_peak()))
    else:
        R = mpc.solve_mpc(spec, S, I, iface, "SOC", False, None, iface.get_prev_peak())
    return time.perf_counter() - t, float(mpc.evaluate_objective(R, spec, I, iface, S, iface.get_prev_peak()))


def _cpu_what(cfg):
    if _cpu_kind(cfg) == "reference":
        return "the unmodified reference's AdaptiveChargingOptimization.solve (cvxpy), loaded by oracle/reference_cvxpy.py"
    return ("oracle/mpc.py float64 interior-point restatement of the reference's cvxpy/ECOS path, which cannot run here "
            "(cvxpy, ecos, acnportal not installed)")


def _cpu_kind(cfg):
    """"reference" when the reference's own solve can run (cvxpy importable, its source present, every objective term of the
    workload defined by it: non_completion_penalty is not), else "port" (oracle/mpc.py)."""
    try:
        from oracle import reference_cvxpy

        if not reference_cvxpy.available():
            return "port"
        ref = reference_cvxpy.load()
        return "reference" if all(hasattr(ref, n) for n, _, _ in CONFIGS[cfg]["objective"]) else "port"
    except Exception:
        return "port"


def _worker_init():
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"


class OraclePool:
    """One persistent pool of single-threaded oracle workers on every host core."""

    def __init__(self, cores=None):
        import multiprocessing as mp

        self.cores = cores or (os.cpu_count() or 1)
        for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[var] = "1"  # inherited by the spawned workers before they import numpy / scipy
        self.pool = mp.get_context("spawn").Pool(self.cores, initializer=_worker_init)

    def run(self, cfg, seeds, budget_s=None):
        """Solves the instances `seeds` of workload `cfg`; with a wall-clock budget the pool is stopped when it runs out
        (the 1000-EVSE instances of C5 take the Python oracle more than five minutes each) and only the completed solves
        count.  Returns (solves per second, wall seconds, results of the completed solves)."""
        t = time.perf_counter()
        jobs = [self.pool.apply_async(_oracle_one, ((cfg, s_),)) for s_ in seeds]
        done = []
        while True:
            done = [j for j in jobs if j.ready()]
            wall = time.perf_counter() - t
            if len(done) == len(jobs) or (budget_s is not None and wall > budget_s):
                break
            time.sleep(0.2)
        self.timed_out = len(done) < len(jobs)
        if self.timed_out:
            self.pool.terminate()
        wall = time.perf_counter() - t
        return len(done) / wall, wall, [j.get() for j in done]

    def close(self):
        if not getattr(self, "timed_out", False):
            self.pool.close()
        self.pool.join()


def run_reference(args):
    """The reference arm: the CPU oracle on all host cores.  A bounded sample of the workload: `rounds` instances per
    core (at most the --steps asked for), all submitted to one persistent pool so that every core stays busy."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = "c3" if args.config == "c4" else args.config  # the replay's instances are C3-shaped
    pool = OraclePool()
    cores = pool.cores
    if args.warmup > 0:
        pool.run("c1", [10_000 + i for i in range(cores)])  # pages the interpreter and scipy in on every worker (small instances)
    per_solve = {"c1": 0.8, "c2": 40.0, "c3": 40.0, "c5": 600.0}[cfg]
    rounds = int(max(1, min(args.steps, 150.0 // per_solve)))
    n = rounds * cores
    value, wall, done = pool.run(cfg, list(range(n)), budget_s=300.0)
    pool.close()
    note = "" if len(done) == n else f"; stopped after {wall:.0f} s with {len(done)} of {n} solves finished (value = finished / wall)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": make_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": _cpu_kind(cfg),
                         "sample": f"{n} instances of the workload (seeds 0..{n - 1}) on one persistent pool of {cores} single-threaded workers "
                                   f"(all host cores), wall {wall:.1f} s{note}; {_cpu_what(cfg)}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def make_config(args, n_gpus):
    C = CONFIGS[args.config]
    per_gpu = args.batch if args.scaling == "weak" else max(1, args.batch // n_gpus)
    return {
        "workload": C["workload"], "instances_per_gpu": per_gpu, "global_instances": per_gpu * n_gpus, "N": C["N"], "T": C["T"], "M": C["M"],
        "parallelism": f"independent instances sharded over {n_gpus} GPU(s), no solve-path collective",
        "tolerances": {"eps_rel": 1e-4, "eps_abs": 1e-5, "violation": 1e-5, "rate_tol_A": 3e-4},
        "l2": "no flush needed: each step reads its raw inputs and writes B x N x Tp float32 rates + float64 pilots "
              "(765 MB at B=4096), several times the 126 MB L2; steps are double-buffered on two streams",
    }


# ----------------------------------------------------------------------------------------------- parity gate
def parity_gate(res, seed0, stride_limit=None):
    """The timed e2e result of rank 0 against the precomputed oracle optima: objective within 1e-4 |f*|, relative
    infrastructure violation, energy over-delivery (kWh), bounds."""
    from adacharge_b200.interface import TestingInterface
    from adacharge_b200.generators import caltech_acn_infrastructure, config_c2
    from oracle import mpc

    if not os.path.exists(GOLDEN):
        return {"instances": 0, "note": "tests/golden/bench_c3_golden.json missing"}
    gold = json.load(open(GOLDEN))
    infra = caltech_acn_infrastructure()
    worst = dict(rel_objective_error=0.0, infrastructure_rel=-1.0, energy_kwh=-1.0, lb=-1.0, ub=-1.0)
    n = fail = 0
    B = res.pilots.shape[0]
    for g in gold["instances"]:
        b = g["seed"] - seed0
        if b < 0 or b >= B:
            continue
        iface = TestingInterface(config_c2(g["seed"], infra=infra, price_noise=0.2))
        S, I = iface.active_sessions(), iface.infrastructure_info()
        T = int(res.T[b])
        R = res.pilots[b, :, :T]
        f = mpc.evaluate_objective(R, BENCH_OBJECTIVE, I, iface, S, iface.get_prev_peak())
        v = mpc.violations(R, S, I, iface)
        rel = abs(f - g["objective"]) / abs(g["objective"])
        worst["rel_objective_error"] = max(worst["rel_objective_error"], rel)
        worst["infrastructure_rel"] = max(worst["infrastructure_rel"], v["infrastructure_rel"])
        worst["energy_kwh"] = max(worst["energy_kwh"], v["energy"])
        worst["lb"], worst["ub"] = max(worst["lb"], v["lb"]), max(worst["ub"], v["ub"])
        ok = rel <= 1e-4 and v["infrastructure_rel"] <= 1e-5 and v["energy"] <= 1e-4 and v["lb"] <= 1e-6 and v["ub"] <= 1e-6 and int(res.status[b]) == 0
        fail += 0 if ok else 1
        n += 1
    return {"instances": n, "failed": fail, "max_rel_objective_error": worst["rel_objective_error"],
            "max_infrastructure_violation_rel": worst["infrastructure_rel"], "max_energy_over_kwh": worst["energy_kwh"],
            "max_lb_violation_A": worst["lb"], "max_ub_violation_A": worst["ub"],
            "bars": {"objective_rel": 1e-4, "infrastructure_rel": 1e-5, "energy_kwh": 1e-4, "bounds_A": 1e-6},
            "source": "oracle optima of every 16th instance of the batch (tests/golden/bench_c3_golden.json, made by tests/golden/make_bench_golden.py)"}


def latency_lines():
    """One AdaptiveChargingOptimization.solve() per call (ada.py:169-175), host objects in, numpy out."""
    import adacharge_b200 as ab
    from adacharge_b200.generators import config_c1, config_c2

    out = {}
    for name, d, spec in (("c1", config_c1(0), C1_OBJECTIVE), ("c2", config_c2(0), BENCH_OBJECTIVE)):
        iface = ab.TestingInterface(d)
        S, I = iface.active_sessions(), iface.infrastructure_info()
        aco = ab.AdaptiveChargingOptimization(objective_components(spec), iface)
        for _ in range(3):
            aco.solve(S, I, prev_peak=iface.get_prev_peak())
        ts = []
        for _ in range(15):
            t = time.perf_counter()
            aco.solve(S, I, prev_peak=iface.get_prev_peak())
            ts.append(time.perf_counter() - t)
        out[name] = {"ms_per_solve_median": float(np.median(ts) * 1e3), "ms_per_solve_min": float(np.min(ts) * 1e3),
                     "iters": aco.last_info["iters"], "call": "AdaptiveChargingOptimization.solve (class defaults: eps_rel 2e-5, rate polish)"}
    return out


# ----------------------------------------------------------------------------------------------- --dump-outputs
DUMP_BYTES = 64 << 20  # what --dump-outputs writes in all, at most


def dump_outputs(out_dir, outs, seed=0):
    """Writes `outs` (name -> tensor whose first axis is the instance) as out_dir/<name>.npy: float32 where the tensor is
    float32, float64 otherwise.  When that would exceed DUMP_BYTES, every array keeps the same fixed, seeded sample of
    instances; instance.npy holds the batch index of each instance written."""
    import torch

    B = len(next(iter(outs.values())))
    itemsize = {name: 4 if t.dtype == torch.float32 else 8 for name, t in outs.items()}
    per_instance = 8 + sum(itemsize[name] * (t.numel() // B) for name, t in outs.items())
    k = min(B, (DUMP_BYTES - 4096) // per_instance)  # (4096: room for the .npy headers)
    idx = np.arange(B) if k == B else np.sort(np.random.default_rng(seed).choice(B, k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "instance.npy"), idx.astype(np.float64))
    for name, t in outs.items():
        a = t[torch.from_numpy(idx).to(t.device)].cpu().numpy()
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float32 if itemsize[name] == 4 else np.float64))


def batch_outputs(bac):
    """The device results of the last call on a BatchedAdaptiveCharging, the fields of its BatchResult."""
    import torch

    def cat(field):
        return torch.cat([field(ch) for ch in bac.chunks])

    return dict(pilots=cat(lambda ch: ch.pilots), status=cat(lambda ch: ch.status), iters=cat(lambda ch: ch.iters),
                T=cat(lambda ch: ch.packed["T"]), stats=cat(lambda ch: ch.stats))


# ----------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None, help="instances per GPU per step (weak) or in total (strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--groups", type=int, default=8, help="c4: independent groups of sites per GPU, each on its own stream")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none to write")
    if args.batch is None:
        args.batch = CONFIGS[args.config]["batch"]
    if args.config == "c4":
        args.scaling = "strong"  # a fixed fleet of sites is sharded
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from adacharge_b200 import _cabi, sharding
    from adacharge_b200.batched import BatchedAdaptiveCharging

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # rank 0 prints exactly one JSON line on stdout.  NCCL writes its version banner to stdout when NCCL_DEBUG is
        # VERSION (the GPU boxes export that) and to NCCL_DEBUG_FILE at WARN/INFO: raise VERSION to WARN, point the
        # log at stderr, and keep fd 1 on stderr while the communicator comes up.
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    _cabi.lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.config == "c4":
        return run_c4(args, world, rank, local, dev, barrier)

    C = CONFIGS[args.config]
    per_gpu = args.batch if args.scaling == "weak" else len(sharding.shard_range(args.batch, rank, world))
    seed0 = rank * per_gpu if args.scaling == "weak" else sharding.shard_range(args.batch, rank, world).start
    W = make_workload(args.config, per_gpu, seed0)
    obj = objective_components(C["objective"])
    kw = dict(prices=W["prices"], prev_peak=W["prev_peak"], external_signal=W["external_signal"])
    steps, warm = args.steps, max(args.warmup, 3)

    def make(chunks):
        return BatchedAdaptiveCharging(obj, W["infra"], 5, batch=per_gpu, max_sessions=C["S_max"], horizon=C["horizon"],
                                       demand_charge=W["demand_charge"], chunks=chunks)

    # ---- value: resident raw inputs -> pack + solve (+ fused projection); two instances on their own streams alternate
    res_a = make(1).upload_raw(W["sessions"], **kw)
    # (the general path synchronises with the host at every convergence check: two objects would only take turns)
    res_b = make(1).upload_raw(W["sessions"], **kw) if args.config != "c5" else res_a
    solve_ev = []

    for k in range(warm):
        (res_a if k % 2 == 0 else res_b).solve_resident()
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        # each object runs on its own stream: step k+1 fills the SMs that the straggler tail of step k leaves idle
        (res_a if k % 2 == 0 else res_b).solve_resident(events=solve_ev, independent=True, start_event=e0 if k < 2 else None)
    res_a.join()
    res_b.join()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    barrier()
    clk = clocks.stop() if rank == 0 else None
    ms = sharding.max_over_ranks(ms, dev)
    if args.dump_outputs and rank == 0:
        # (before the isolated steps below, which solve again into res_a)
        dump_outputs(args.dump_outputs, batch_outputs(res_a if (steps - 1) % 2 == 0 else res_b))
    # the solve kernel alone: isolated steps (one stream, nothing else in flight), CUDA events on the stream the kernel is
    # launched on around acb_solve_batch, and around the whole step for the kernel's share of it
    iso_solve, iso_step = [], []
    for _ in range(3):
        ev = []
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        res_a.solve_resident(events=ev)
        b.record()
        torch.cuda.synchronize()
        iso_step.append(a.elapsed_time(b))
        iso_solve.append(ev[0][0].elapsed_time(ev[0][1]))
    kern_ms, iso_ms = float(np.mean(iso_solve)), float(np.mean(iso_step))
    ch = res_a.chunks[0]
    status = ch.status.cpu().numpy()
    iters = ch.iters.cpu().numpy().astype(np.float64)
    res_b = None
    # ---- e2e: host arrays -> host pilots through the public batched call, double-buffered
    e2e_a = make(4 if args.config != "c5" else 1)
    e2e_b = make(4) if args.config != "c5" else e2e_a
    for k in range(2):
        (e2e_a if k % 2 == 0 else e2e_b).schedule_async(W["sessions"], **kw)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for k in range(steps):
        # (schedule_async first waits until the results of step k-2, which used the same buffers, have landed)
        (e2e_a if k % 2 == 0 else e2e_b).schedule_async(W["sessions"], independent=True, start_event=e0 if k < 2 else None, **kw)
    e2e_a.join()
    e2e_b.join()
    e1.record()
    torch.cuda.synchronize()
    wall_e2e = (time.perf_counter() - t0) * 1e3
    ms_e2e = sharding.max_over_ranks(max(e0.elapsed_time(e1), wall_e2e), dev)
    result = e2e_a.result()
    barrier()

    summary = torch.tensor([float((status == 0).sum()), float(len(status)), iters.sum(), iters.max()], dtype=torch.float64, device=dev)
    tot = torch.stack(sharding.gather_summaries(summary)).cpu().numpy()  # the final gather
    n_total = tot[:, 1].sum()
    value = n_total * steps / (ms / 1e3)
    e2e = n_total * steps / (ms_e2e / 1e3)
    # roofline of the solve kernel: algorithmic bytes per SURVEY.md 8(d) (fp32 state streamed once per iteration)
    N, T, M = C["N"], C["T"], C["M"]
    b_iter = 4 * (4 * N * T + 2 * (2 * M + 2) * T)
    alg_bytes_rank = float(((iters + 1) * b_iter).sum())
    launch_ms = ms / steps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes_rank / (kern_ms / 1e3) / 1e9  # algorithmic bytes of one launch / that launch's duration (isolated)
    traffic = None
    try:
        if args.config == "c5":
            # general path: measured DRAM bytes per instance-iteration (ncu, k_rows + k_cols_it + k_level) x the launch's instance-iterations
            traffic = json.load(open(os.path.join(ROOT, "profiles", "general_path_dram.json")))["dram_bytes_per_instance_iteration"] * float((iters + 1).sum())
        else:
            # measured DRAM bytes per instance (ncu, profiles/) x instances per launch on this rank
            traffic = json.load(open(os.path.join(ROOT, "profiles", "solve_kernel_dram.json")))["dram_bytes_per_instance"] * per_gpu
    except Exception:
        pass
    if rank == 0:
        general = args.config == "c5"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": launch_ms, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": make_config(args, world),
            "timed_region": "device packer (acb_pack_sessions) + acb_solve_batch incl. fused continuous-pilot projection, raw inputs resident; "
                            f"{steps} steps double-buffered on two streams between one pair of CUDA events",
            "solved": int(tot[:, 0].sum()), "instances": int(n_total), "iters_mean": float(tot[:, 2].sum() / n_total), "iters_max": float(tot[:, 3].max()),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 (B200_PROFILING.md)",
                         "kernel": "acb_solve_general (k_rows/k_cols)" if general else "acb_solve_kernel", "algorithmic_bytes_per_iteration": b_iter,
                         "kernel_ms_per_launch": kern_ms, "isolated_step_ms": iso_ms, "kernel_share_of_step": kern_ms / iso_ms,
                         "note": "effective bandwidth: state is on-chip resident, DRAM sees load/store only (SURVEY.md 8(d)); per-GPU figure; "
                                 "launch duration from isolated steps (the timed steps overlap two launches on two streams)"
                                 if not general else "state streamed through HBM/L2 every iteration; per-GPU figure"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(e2e_a.h2d_bytes) * world,
                    "d2h_bytes_per_step": int(e2e_a.d2h_bytes) * world, "ms_per_step": ms_e2e / steps,
                    "call": "BatchedAdaptiveCharging.schedule_async(host session tables, prices, prev_peak) -> host float64 pilots"},
            "gpu_launches": int(steps * res_a.kernel_launches_per_call), "clocks": clk,
        }
        if args.config == "c3":
            line["parity_sample"] = parity_gate(result, seed0)
        if world == 1 and not args.no_latency:
            line["latency"] = latency_lines()
        if world == 1 and not args.no_cpu_baseline:
            pool = OraclePool()
            n = pool.cores
            v, wall, done = pool.run(args.config, list(range(n)), budget_s=120.0)
            pool.close()
            note = "" if len(done) == n else f"; stopped after {wall:.0f} s with {len(done)} of {n} solves finished"
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": pool.cores, "kind": _cpu_kind(args.config),
                                    "sample": f"first {n} instances of the batch, one per core on all {pool.cores} host cores, {_cpu_what(args.config)}, wall {wall:.1f} s{note}"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_c4(args, world, rank, local, dev, barrier):
    """BASELINE configs[3]: closed-loop replay, sites sharded over the ranks; a step = one control step of every site
    (active sessions -> pack -> warm-started solve -> pilots -> simulator update, all on the device, no host sync)."""
    import torch
    import torch.distributed as dist

    from adacharge_b200 import sharding
    from adacharge_b200.generators import caltech_acn_infrastructure
    from adacharge_b200.replay_fast import DeviceFleetReplay

    rng = sharding.shard_range(args.batch, rank, world)
    # Sites are independent closed loops: the rank's sites are cut into groups that advance on their own streams, so
    # that a group's step does not wait for the slowest site of another group (each group is in lockstep internally)
    n_groups = max(1, min(args.groups, len(rng) // 8))
    cuts = [rng.start + round(k * len(rng) / n_groups) for k in range(n_groups + 1)]
    infra = caltech_acn_infrastructure()
    rps = [DeviceFleetReplay(infra, objective_components(BENCH_OBJECTIVE), n_sites=b - a, steps_per_day=288, days=1,
                             seed0=1000, Tp=CONFIGS["c4"]["horizon"], site_offset=a) for a, b in zip(cuts[:-1], cuts[1:])]
    streams = [torch.cuda.Stream(device=dev) for _ in rps]
    t_start = 96  # 8 am: the fleet is filling up (the busiest part of the day for the solver)
    warm = max(args.warmup, 3)

    def run_steps(t0, t1):
        for t in range(t0, t1):
            for rp, st in zip(rps, streams):
                with torch.cuda.stream(st):
                    rp.step(t, want_first=False)

    def summary():
        ss = [rp.summary() for rp in rps]
        return dict(site_steps=sum(x["site_steps"] for x in ss), unsolved=sum(x["unsolved"] for x in ss),
                    iters=sum(x["iters_mean"] * x["site_steps"] for x in ss))

    run_steps(t_start, t_start + warm)
    torch.cuda.synchronize()
    s0 = summary()
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cur = torch.cuda.current_stream(dev)
    t0 = time.perf_counter()
    e0.record(cur)
    for st in streams:
        st.wait_event(e0)
    run_steps(t_start + warm, t_start + warm + args.steps)
    for st in streams:
        cur.wait_stream(st)
    e1.record(cur)
    t_enq = (time.perf_counter() - t0) * 1e3
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    barrier()
    clk = clocks.stop() if rank == 0 else None
    ms = sharding.max_over_ranks(ms, dev)
    if args.dump_outputs and rank == 0:
        # the last control step of every site of the rank (the groups are consecutive ranges of sites) and the peaks so far
        outs = [batch_outputs(rp._bac) for rp in rps]
        outs = {k: torch.cat([o[k] for o in outs]) for k in outs[0]}
        outs["prev_peak"] = torch.cat([rp._d["prev_peak"] for rp in rps])
        dump_outputs(args.dump_outputs, outs)
    s1 = summary()
    summ = torch.tensor([s1["site_steps"] - s0["site_steps"], s1["unsolved"] - s0["unsolved"], s1["iters"] - s0["iters"], t_enq],
                        dtype=torch.float64, device=dev)
    tot = torch.stack(sharding.gather_summaries(summ)).cpu().numpy()
    if rank == 0:
        solves = tot[:, 0].sum()
        value = solves / (ms / 1e3)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": make_config(args, world),
            "timed_region": "closed loop on the device: acb_fleet_sessions + acb_pack_sessions + warm-started acb_solve_batch (fused pilot projection) + "
                            "acb_fleet_apply per control step, CUDA events around all steps, no host synchronisation in between",
            "solved": int(solves - tot[:, 1].sum()), "instances": int(solves), "iters_mean": float(tot[:, 2].sum() / max(solves, 1)),
            "host_enqueue_ms_per_step_max_rank": float(tot[:, 3].max() / args.steps),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "ms_per_step": ms / args.steps,
                    "call": "DeviceFleetReplay.step (the closed loop is end to end by construction: the EV state lives on the device)"},
            "gpu_launches": int(args.steps * 4 * n_groups), "site_groups_per_gpu": n_groups, "clocks": clk,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
