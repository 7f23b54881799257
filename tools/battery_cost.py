"""Cost and effect of two-stage batteries and the rampdown estimate (DeviceFleetReplay's battery / estimate_max_rate) on the
C4 shape: 1024 CaltechACN-shaped sites, one day of 5-minute steps, bench.py's C4 horizon and objective, simulator on the
device, in three configurations: ideal batteries (the default), batteries, batteries with the estimate.

    python tools/battery_cost.py [OUT_DIR] [--rounds R] [--sites N]

One GPU run.  The three configurations replay the same EVs; each round builds them afresh and runs the day with the
configurations alternated step by step.  Every step is timed with CUDA events around DeviceFleetReplay.step, after a
short warm-up on throwaway replays.  Per configuration: solves (of sites with sessions), uncertified solves, mean
iterations per solve, device time per day, delivered fraction of the requested energy, mean and max peak (kW) and the
pilot energy the batteries did not take, sum over steps and EVSEs of (p - a) * w (kWh; p the applied pilot, a the
battery's current, w kWh per A-period), read back between the timed steps.  Prints one JSON document and writes it to
OUT_DIR/battery_b200.json, with a summary table in OUT_DIR/battery.md."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402

CONFIGS = {"ideal": {}, "battery": dict(battery=True), "battery+estimate": dict(battery=True, estimate_max_rate=True)}


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def make(n_sites, kw):
    from adacharge_b200.generators import caltech_acn_infrastructure
    from adacharge_b200.replay_fast import DeviceFleetReplay

    return DeviceFleetReplay(caltech_acn_infrastructure(), bench.objective_components(bench.BENCH_OBJECTIVE), n_sites=n_sites, steps_per_day=288,
                             days=1, seed0=1000, Tp=bench.CONFIGS["c4"]["horizon"], **kw)


def one_round(n_sites):
    rps = {k: make(n_sites, kw) for k, kw in CONFIGS.items()}
    ms = {k: 0.0 for k in CONFIGS}
    untaken = {k: 0.0 for k in CONFIGS}
    for t in range(288):
        for k, rp in rps.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            rp.step(t, want_first=False)
            b.record()
            torch.cuda.synchronize()
            ms[k] += a.elapsed_time(b)
            if rp.battery:  # every site solved (max_recompute 1): column 0 of this step's pilots is what was applied
                p0 = rp._ch.pilots[:, :, 0].cpu().numpy()
                untaken[k] += float(((p0 - rp.state()["rates"]) * (rp.volt * rp.period / 1e3 / 60)).sum())
    out = {}
    for k, rp in rps.items():
        s, x = rp.summary(), rp.state()
        req, dlv, peak_kw = float(rp.ev_req.sum()), float(x["ev_dlv"].sum()), x["prev_peak"] * rp.volt[0] / 1000
        out[k] = dict(solves=s["solves"], unsolved=s["unsolved"], iters_mean=s["iters_mean"], device_ms_per_day=ms[k],
                      delivered_frac=dlv / req, delivered_kwh=dlv, requested_kwh=req,
                      peak_kw_mean=float(peak_kw.mean()), peak_kw_max=float(peak_kw.max()), untaken_pilot_kwh=untaken[k])
    return out


TABLE = ("| configuration | solves | uncertified | mean iterations | device ms / day (mean, min-max over rounds) | delivered fraction "
         "| peak kW mean / max | pilot energy not taken, kWh |\n|---|---|---|---|---|---|---|---|\n")


def markdown(res):
    r0 = res["rounds"][0]
    rows = []
    for k in CONFIGS:
        r, m = r0[k], res["device_ms_per_day"][k]
        rows.append(f"| {k} | {r['solves']:.0f} | {r['unsolved']:.0f} | {r['iters_mean']:.1f} | {m['mean']:.0f} ({m['min']:.0f}-{m['max']:.0f}) "
                    f"| {r['delivered_frac']:.4f} | {r['peak_kw_mean']:.1f} / {r['peak_kw_max']:.1f} | {r['untaken_pilot_kwh']:.1f} |")
    return (f"Written by `tools/battery_cost.py` ({res['workload']}).\n\nCard: {res['card']['torch_name']}; nvidia-smi name, power limit, max SM clock: "
            f"{res['card']['nvidia_smi']}.\n\nCounts and energies are of the first round (every round replays the same EVs); device time is "
            f"over {len(res['rounds'])} rounds.\n\n" + TABLE + "\n".join(rows) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir", nargs="?", default=None)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--sites", type=int, default=bench.CONFIGS["c4"]["batch"])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    for kw in CONFIGS.values():  # warm-up: module loads, the stream-ordered pool
        rp = make(a.sites, kw)
        for t in range(96, 99):
            rp.step(t, want_first=False)
        del rp
    torch.cuda.synchronize()
    rounds = [one_round(a.sites) for _ in range(a.rounds)]
    res = dict(card=card(), workload=f"C4 shape: DeviceFleetReplay of {a.sites} CaltechACN-shaped sites, one day (288 5-minute steps), Tp "
                                     f"{bench.CONFIGS['c4']['horizon']}, seed0 1000, max_recompute 1, configurations alternated step by step",
               rounds=rounds)
    ms = {k: [r[k]["device_ms_per_day"] for r in rounds] for k in CONFIGS}
    res["device_ms_per_day"] = {k: dict(mean=float(np.mean(v)), min=float(np.min(v)), max=float(np.max(v))) for k, v in ms.items()}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out_dir:
        os.makedirs(a.out_dir, exist_ok=True)
        with open(os.path.join(a.out_dir, "battery_b200.json"), "w") as f:
            f.write(txt + "\n")
        with open(os.path.join(a.out_dir, "battery.md"), "w") as f:
            f.write(markdown(res))


if __name__ == "__main__":
    main()
