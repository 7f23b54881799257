"""DEV: per-phase cycle counts of the solve kernel (library built with -DACB_TIMING)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import common
from adacharge_b200 import _cabi, engine
site, insts, _ = common.build_instances(148, 0)
pb = engine.PackedBatch(site, insts, want_warm_out=True).upload()
pb.warm_out = dict(pb.warm_out, mu=torch.zeros((148, 256), dtype=torch.float32, device=pb.rates.device))
opt = _cabi.default_options(max_iter=300)
pb.solve(opt); torch.cuda.synchronize()
m = pb.warm_out["mu"][0, :160].cpu().numpy().reshape(32, 5)
n = m[0, 4]
print("sessions of instance 0:", int(pb.host["n_sessions"][0]), "non-check iterations timed:", n)
print("warp: col_work col_wait row_work row_wait (cycles per iteration)")
for w in (0, 1, 5, 13, 20, 26, 27, 28, 30, 31):
    print(w, (m[w, :4] / max(n, 1)).round(0))
print("mean over warps", (m[:, :4].mean(axis=0) / n).round(0), "sum", (m[:, :4].sum(axis=1) / n).mean().round(0))
