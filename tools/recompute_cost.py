"""Cost and effect of event-driven recompute (DeviceFleetReplay's max_recompute) on the C4 shape: 1024 CaltechACN-shaped
sites, one day of 5-minute steps, bench.py's C4 horizon and objective, simulator on the device, at max_recompute 1 (every
step, the default), 3, 12 and None (events only).

    python tools/recompute_cost.py [OUT.json] [--rounds R] [--sites N]

One GPU run.  The four configurations replay the same EVs; each round builds them afresh and runs the day with the
configurations alternated step by step (configuration after configuration within each control step).  Every step is timed
with CUDA events around DeviceFleetReplay.step; after a short warm-up on throwaway replays.  Per configuration: solves
(of sites with sessions), device time per day, mean iterations per solve, mean warm shift (t - last_solve of the solves
that started warm), delivered fraction of the requested energy and peak kW.  The decision, shift and warm flag of every
solve are read back between the timed steps.  Prints one JSON document (and writes it to OUT.json)."""
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

CONFIGS = {"1": 1, "3": 3, "12": 12, "None": None}


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def make(n_sites, mr):
    from adacharge_b200.generators import caltech_acn_infrastructure
    from adacharge_b200.replay_fast import DeviceFleetReplay

    return DeviceFleetReplay(caltech_acn_infrastructure(), bench.objective_components(bench.BENCH_OBJECTIVE), n_sites=n_sites, steps_per_day=288,
                             days=1, seed0=1000, Tp=bench.CONFIGS["c4"]["horizon"], max_recompute=mr)


def one_round(n_sites):
    rps = {k: make(n_sites, mr) for k, mr in CONFIGS.items()}
    ms = {k: 0.0 for k in CONFIGS}
    shifts = {k: [] for k in CONFIGS}
    for t in range(288):
        for k, rp in rps.items():
            had = rp._d["had"].clone()  # (whether each site's last solve had sessions: solver bookkeeping, not simulator state)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            rp.step(t, want_first=False)
            b.record()
            torch.cuda.synchronize()
            ms[k] += a.elapsed_time(b)
            # (the warm shifts are solver inputs, not simulator state; at max_recompute 1 every solve starts from the step before)
            sh = rp._d["shift"].cpu().numpy() if rp._event_driven else np.ones(rp.n_sites, dtype=np.int32)
            warm = rp.state()["recompute"] & (had.cpu().numpy() != 0) & (rp._ch.packed["n_sessions"].cpu().numpy() > 0)
            shifts[k] += sh[warm].tolist()
    out = {}
    for k, rp in rps.items():
        s, x = rp.summary(), rp.state()
        req = float(rp.ev_req.sum())
        req_site = np.maximum(np.bincount(rp.ev_site, weights=rp.ev_req, minlength=n_sites), 1e-9)
        frac_site = np.bincount(rp.ev_site, weights=x["ev_dlv"], minlength=n_sites) / req_site
        peak_kw = x["prev_peak"] * rp.volt[0] / 1000
        out[k] = dict(solves=s["solves"], solves_per_site_day=s["solves"] / n_sites, unsolved=s["unsolved"], device_ms_per_day=ms[k],
                      iters_mean=s["iters_mean"], warm_shift_mean=float(np.mean(shifts[k])) if shifts[k] else 0.0,
                      warm_solves=len(shifts[k]), delivered_frac=float(x["ev_dlv"].sum() / req),
                      delivered_frac_min_site=float(frac_site.min()), peak_kw_mean=float(peak_kw.mean()), peak_kw_max=float(peak_kw.max()))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?", default=None)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--sites", type=int, default=bench.CONFIGS["c4"]["batch"])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    for mr in CONFIGS.values():  # warm-up: module loads, the stream-ordered pool
        rp = make(a.sites, mr)
        for t in range(96, 99):
            rp.step(t, want_first=False)
        del rp
    torch.cuda.synchronize()
    rounds = [one_round(a.sites) for _ in range(a.rounds)]
    res = dict(card=card(), workload=f"C4 shape: DeviceFleetReplay of {a.sites} CaltechACN-shaped sites, one day (288 5-minute steps), Tp "
                                     f"{bench.CONFIGS['c4']['horizon']}, seed0 1000, configurations alternated step by step",
               rounds=rounds)
    ms = {k: [r[k]["device_ms_per_day"] for r in rounds] for k in CONFIGS}
    res["device_ms_per_day"] = {k: dict(mean=float(np.mean(v)), min=float(np.min(v)), max=float(np.max(v))) for k, v in ms.items()}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
