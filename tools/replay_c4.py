"""BASELINE config 4 at scale: closed-loop warm-started replay of many Caltech-shaped sites.
  python tools/replay_c4.py [n_sites] [t0] [t1] [days] [Tp] [host|device] [groups]   (one GPU; default: device simulator, 8 groups)
  torchrun --nproc-per-node N tools/replay_c4.py ...                                  (sites sharded over ranks)
Sites are independent closed loops: with the device simulator a rank's sites are cut into `groups` fleets that advance on
their own streams (each in lockstep internally), so one fleet's step does not wait for the slowest site of another.
Prints one JSON line: control steps per second for the whole fleet, site-steps per second, iteration statistics."""
import json
import os
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

import adacharge_b200 as ab
from adacharge_b200.generators import caltech_acn_infrastructure
from adacharge_b200.replay_fast import DeviceFleetReplay, FleetReplay
from adacharge_b200 import sharding

n_sites = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
t0 = int(sys.argv[2]) if len(sys.argv) > 2 else 0
t1 = int(sys.argv[3]) if len(sys.argv) > 3 else 288
days = int(sys.argv[4]) if len(sys.argv) > 4 else 1
Tp = int(sys.argv[5]) if len(sys.argv) > 5 else 160
on_device = (sys.argv[6] if len(sys.argv) > 6 else "device") == "device"
groups = int(sys.argv[7]) if len(sys.argv) > 7 else 8
rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
local = int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
if world > 1:
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
_r = sharding.shard_range(n_sites, rank, world)
obj = [ab.ObjectiveComponent(ab.tou_energy_cost), ab.ObjectiveComponent(ab.total_energy, 0.3), ab.ObjectiveComponent(ab.demand_charge, 1 / 30)]
opts = json.loads(os.environ.get("ACB_REPLAY_OPTS", "{}"))
infra = caltech_acn_infrastructure()
if on_device:
    g = max(1, min(groups, len(_r) // 8))
    cuts = [_r.start + round(k * len(_r) / g) for k in range(g + 1)]
    rps = [DeviceFleetReplay(infra, obj, n_sites=b - a, steps_per_day=288, days=days, seed0=1000, Tp=Tp, site_offset=a, solver_options=opts)
           for a, b in zip(cuts[:-1], cuts[1:])]
else:
    rps = [FleetReplay(infra, obj, n_sites=len(_r), steps_per_day=288, days=days, seed0=1000, Tp=Tp, site_offset=_r.start, solver_options=opts)]
streams = [torch.cuda.Stream() for _ in rps]


def run(a, b):
    for t in range(a, b):
        for rp, st in zip(rps, streams):
            with torch.cuda.stream(st):
                rp.step(t, want_first=False)


def summary():
    ss = [rp.summary() for rp in rps]
    return dict(site_steps=sum(x["site_steps"] for x in ss), unsolved=sum(x["unsolved"] for x in ss), iters=sum(x["iters_mean"] * x["site_steps"] for x in ss))


run(t0, min(t0 + 3, t1))  # warm-up steps (library load, allocator), not timed
torch.cuda.synchronize()
s0 = summary()
if world > 1:
    torch.distributed.barrier()
torch.cuda.synchronize()
w0 = time.perf_counter()
run(t0 + 3, t1)
torch.cuda.synchronize()
wall = time.perf_counter() - w0
s1 = summary()
frac = 0.0  # sum over the sites of the delivered fraction of the requested energy
for rp in rps:
    req = np.bincount(rp.ev_site, weights=rp.ev_req, minlength=rp.n_sites)
    frac += float(np.sum(np.bincount(rp.ev_site, weights=rp.state()["ev_dlv"], minlength=rp.n_sites) / np.maximum(req, 1e-9)))
vals = torch.tensor([s1["site_steps"] - s0["site_steps"], s1["unsolved"] - s0["unsolved"], s1["iters"] - s0["iters"], frac], device="cuda", dtype=torch.float64)
wt = torch.tensor([wall], device="cuda", dtype=torch.float64)
if world > 1:
    torch.distributed.all_reduce(vals, op=torch.distributed.ReduceOp.SUM)
    torch.distributed.all_reduce(wt, op=torch.distributed.ReduceOp.MAX)
site_steps, unsolved, iters, full = vals.tolist()
wall = wt.item()
if rank == 0:
    steps = t1 - t0 - 3
    print(json.dumps(dict(workload="C4 replay", simulator="device" if on_device else "host", groups_per_gpu=len(rps), n_sites=n_sites, n_gpus=world,
                          steps=steps, Tp=Tp, days=days, control_steps_per_s=round(steps / wall, 2), site_steps_per_s=round(site_steps / wall, 1),
                          wall_s=round(wall, 2), ms_per_step=round(wall * 1e3 / max(steps, 1), 3), iters_mean=round(iters / max(site_steps, 1), 1),
                          unsolved=unsolved, mean_delivered_fraction=round(full / n_sites, 4))))
if world > 1:
    torch.distributed.destroy_process_group()
