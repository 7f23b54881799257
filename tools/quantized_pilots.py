"""Cost of quantised pilots (BatchedAdaptiveCharging / DeviceFleetReplay with quantize, reallocate) against continuous
pilots, per step of the C3, C5 and C4 workloads of bench.py, plus the acb_quantize_pilots launch on its own.

    python tools/quantized_pilots.py [OUT.json] [--steps K]

One GPU run.  Every timing is CUDA events after warm-up; the three variants of a workload solve the same inputs and are
timed alternately (variant after variant within each step).  Prints one JSON document (and writes it to OUT.json)."""
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
from adacharge_b200 import _cabi, engine  # noqa: E402
from adacharge_b200.batched import BatchedAdaptiveCharging  # noqa: E402

MODES = {"continuous": dict(), "discrete": dict(quantize=True), "reallocate": dict(quantize=True, reallocate=True)}


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def timed(fn, n):
    """Mean and spread (ms) of n calls of fn, each between two events on the current stream."""
    out = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def launch_alone(bac, mode, n=20):
    """acb_quantize_pilots on the chunk's last solve, alone on the current stream."""
    L, ch = _cabi.lib(), bac.chunks[0]
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def go():
        _cabi.check(L.acb_quantize_pilots(bac.site.handle, mode, C.byref(ch.sessions), float(bac.period), C.byref(ch.batch),
                                          engine._ptr(ch.pilots), st), "acb_quantize_pilots")
    timed(go, 3)
    t = timed(go, n)
    return dict(mean_ms=float(np.mean(t)), min_ms=float(np.min(t)), max_ms=float(np.max(t)))


def batched(cfg, steps):
    C_ = bench.CONFIGS[cfg]
    W = bench.make_workload(cfg, C_["batch"], 0)
    kw = dict(prices=W["prices"], prev_peak=W["prev_peak"], external_signal=W["external_signal"])
    obj = bench.objective_components(C_["objective"])
    objs = {m: BatchedAdaptiveCharging(obj, W["infra"], 5, batch=C_["batch"], max_sessions=C_["S_max"], horizon=C_["horizon"],
                                       demand_charge=W["demand_charge"], chunks=1, **f).upload_raw(W["sessions"], **kw) for m, f in MODES.items()}
    for bac in objs.values():  # warm-up
        bac.solve_resident()
    torch.cuda.synchronize()
    per = {m: [] for m in MODES}
    for _ in range(steps):
        for m, bac in objs.items():
            per[m] += timed(bac.solve_resident, 1)
    rates = {m: bac.chunks[0].rates.cpu().numpy() for m, bac in objs.items()}
    out = dict(workload=C_["workload"], instances=C_["batch"], steps=steps,
               same_schedule=all(np.array_equal(rates["continuous"], r) for r in rates.values()),
               step_ms={m: dict(mean=float(np.mean(v)), min=float(np.min(v)), max=float(np.max(v))) for m, v in per.items()},
               launch_alone={m: launch_alone(objs[m], objs[m].pilot_mode) for m in ("discrete", "reallocate")})
    c = out["step_ms"]["continuous"]["mean"]
    out["ratio_to_continuous"] = {m: out["step_ms"][m]["mean"] / c for m in MODES}
    del objs
    torch.cuda.empty_cache()
    return out


def fleet(steps):
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
               sites=n_sites, steps=steps,
               step_ms={m: dict(mean=float(np.mean(v)), min=float(np.min(v)), max=float(np.max(v))) for m, v in per.items()},
               launch_alone={m: launch_alone(rps[m]._bac, rps[m].pilot_mode) for m in ("discrete", "reallocate")},
               site_steps={m: rp.summary()["site_steps"] for m, rp in rps.items()})
    c = out["step_ms"]["continuous"]["mean"]
    out["ratio_to_continuous"] = {m: out["step_ms"][m]["mean"] / c for m in MODES}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?", default=None)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--c4-steps", type=int, default=12, help="control steps of C4 (12 = one hour of 5-minute steps)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = dict(card=card(), c3=batched("c3", a.steps), c5=batched("c5", max(2, a.steps // 2)), c4=fleet(a.c4_steps))
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
