"""Cost of uninterrupted charging (BatchedAdaptiveCharging / DeviceFleetReplay with uninterrupted_charging) against the
same workload without it: C3 (4096 instances) solves per second and mean iterations, C4 steps per second, and the
acb_admit_sessions launch on its own.

    python tools/uninterrupted_cost.py [OUT.json] [--steps K] [--c4-steps K]

One GPU run.  Every timing is CUDA events after warm-up; the two variants of a workload solve the same inputs and are
timed alternately (variant after variant within each step).  With uninterrupted charging the admitted first-period
minimum rules out the on-chip kernel's FAST variant (lb_zero), so most of the difference is FAST against non-FAST.
C3's sessions arrive at their arrival_offset (current_time 0), so that is their absolute arrival.  Prints one JSON
document (and writes it to OUT.json)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import ctypes as C  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from adacharge_b200.batched import BatchedAdaptiveCharging  # noqa: E402

MODES = {"off": dict(), "uninterrupted": dict(uninterrupted_charging=True)}


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def timed(fn, n):
    """Times (ms) of n calls of fn, each between two events on the current stream."""
    out = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def spread(v):
    return dict(mean=float(np.mean(v)), min=float(np.min(v)), max=float(np.max(v)))


def admission_alone(bac, n=20):
    """acb_admit_sessions on the chunk's raw tables as the last step left them, alone on the current stream.  The tables
    are restored before every launch (outside the timed window): the admission permutes them in place."""
    ch = bac.chunks[0]
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    snap = {k: v.clone() for k, v in ch.dev_raw.items()}
    t = []
    for k in range(n + 3):
        for key, v in snap.items():
            ch.dev_raw[key].copy_(v)
        torch.cuda.synchronize()
        t += timed(lambda: bac.admit(ch, st), 1)
    return spread(t[3:])


def c3(steps):
    C_ = bench.CONFIGS["c3"]
    W = bench.make_workload("c3", C_["batch"], 0)
    sess = dict(W["sessions"], arrival=W["sessions"]["arrival_offset"].copy())
    kw = dict(prices=W["prices"], prev_peak=W["prev_peak"])
    obj = bench.objective_components(C_["objective"])
    objs = {m: BatchedAdaptiveCharging(obj, W["infra"], 5, batch=C_["batch"], max_sessions=C_["S_max"], horizon=C_["horizon"],
                                       demand_charge=W["demand_charge"], chunks=1, **f) for m, f in MODES.items()}
    # resident form as bench.py's `value`: raw arrays on the device; the admission permutes them in place, so every
    # timed call starts from a fresh device copy of the staged tables (copied before the timed window)
    def reload(bac):
        ch = bac.chunks[0]
        for key, h in ch.host.items():
            ch.dev_raw[key].copy_(h)
        torch.cuda.synchronize()

    for bac in objs.values():
        bac.upload_raw(sess, **kw)
        bac.solve_resident()  # warm-up
    torch.cuda.synchronize()
    per = {m: [] for m in MODES}
    for _ in range(steps):
        for m, bac in objs.items():
            reload(bac)
            per[m] += timed(bac.solve_resident, 1)
    out = dict(workload=C_["workload"], instances=C_["batch"], steps=steps)
    for m, bac in objs.items():
        ch = bac.chunks[0]
        it, stt = ch.iters.cpu().numpy(), ch.status.cpu().numpy()
        adm = (ch.limits0["min_rate0"].cpu().numpy() > 0).sum() if m != "off" else 0
        out[m] = dict(step_ms=spread(per[m]), solves_per_s=C_["batch"] / (np.mean(per[m]) / 1e3), iters_mean=float(it.mean()),
                      iters_max=int(it.max()), solved=int((stt == 0).sum()), lb_zero=bool(ch.lb_zero), admitted_sessions=int(adm))
    reload(objs["uninterrupted"])
    out["admission_alone_ms"] = admission_alone(objs["uninterrupted"])
    out["ratio"] = out["uninterrupted"]["step_ms"]["mean"] / out["off"]["step_ms"]["mean"]
    del objs
    torch.cuda.empty_cache()
    return out


def c4(steps):
    from adacharge_b200.generators import caltech_acn_infrastructure
    from adacharge_b200.replay_fast import DeviceFleetReplay

    n_sites, t0, warm = bench.CONFIGS["c4"]["batch"], 96, 3  # 8 am, as bench.py's C4
    infra = caltech_acn_infrastructure()
    rps = {m: DeviceFleetReplay(infra, bench.objective_components(bench.BENCH_OBJECTIVE), n_sites=n_sites, steps_per_day=288, days=1, seed0=1000,
                                Tp=bench.CONFIGS["c4"]["horizon"], **f) for m, f in MODES.items()}
    for t in range(t0, t0 + warm):
        for rp in rps.values():
            rp.step(t, want_first=False)
    torch.cuda.synchronize()
    per = {m: [] for m in MODES}
    for t in range(t0 + warm, t0 + warm + steps):
        for m, rp in rps.items():
            per[m] += timed(lambda: rp.step(t, want_first=False), 1)
    out = dict(workload=f"C4: DeviceFleetReplay of {n_sites} CaltechACN-shaped sites, one stream, control steps {t0 + warm}..{t0 + warm + steps - 1}",
               sites=n_sites, steps=steps)
    for m, rp in rps.items():
        s = rp.summary()
        out[m] = dict(step_ms=spread(per[m]), steps_per_s=1e3 / np.mean(per[m]), site_steps=s["site_steps"], unsolved=s["unsolved"],
                      iters_mean=s["iters_mean"])
    out["admission_alone_ms"] = admission_alone(rps["uninterrupted"]._bac)
    out["ratio"] = out["uninterrupted"]["step_ms"]["mean"] / out["off"]["step_ms"]["mean"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?", default=None)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--c4-steps", type=int, default=12, help="control steps of C4 (12 = one hour of 5-minute steps)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = dict(card=card(), c3=c3(a.steps), c4=c4(a.c4_steps))
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
