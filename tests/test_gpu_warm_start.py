"""Warm start of acb_solve_batch on both solve paths, at the C ABI (acb_batch.warm_* / out_*):

- the state a solve writes (out_v1, out_vc, out_mu, out_scal), fed to the next control step with warm_shift = 1, gives
  bit for bit what the same state shifted one column on the host gives with warm_shift = 0;
- warm_had = 0 is a cold solve, bit for bit, whatever the warm arrays hold, also with positive minimum rates (v then
  starts at clamp(0, lb, ub), not at 0) and with the second stagnation rescue allowed (it is for warm-started solves);
- the device fleet replay equals the host fleet replay, and warm-started replay steps match a cold oracle solve, on the
  general path too (tests/test_gpu_replay.py runs both on the default path).
"""
import numpy as np
import pytest
import torch

import adacharge_b200 as ab
from adacharge_b200 import _cabi, engine
from adacharge_b200.generators import session_generator, three_phase_balanced_network
from tests.replay_checks import device_vs_host_fleet_replay, warm_steps_vs_cold_oracle

pytestmark = pytest.mark.gpu
BENCH = [ab.ObjectiveComponent(ab.tou_energy_cost), ab.ObjectiveComponent(ab.total_energy, 0.3), ab.ObjectiveComponent(ab.demand_charge, 1 / 30)]

# (padded horizon, first step's horizon, minimum rate of every other session)
CASES = {"Tp64": (64, 64, 0.0), "Tp64_minrate": (64, 64, 6.0), "Tp288_minrate": (288, 200, 6.0), "Tp416": (416, 400, 0.0)}


def _pair(T0, mins, seed=3):
    """Two consecutive control steps of one site: step 1 is step 0 one period later (every window one period shorter
    at its start, same sessions in the same slots)."""
    infra = three_phase_balanced_network(4, 70.0)
    rng = np.random.default_rng(seed)
    n = 10
    st = [str(s) for s in rng.permutation(12)[:n]]
    arr = rng.integers(0, T0 // 2, n)
    dep = np.minimum(arr + rng.integers(6, T0 // 2, n), T0)
    dep[0] = T0
    mn = [mins if k % 2 == 0 else 0.0 for k in range(n)]
    e = np.maximum(rng.uniform(0.3, 0.8, n) * (dep - arr) * 32, 1.2 * np.array(mn) * (dep - arr)) * 208 * 5 / 60e3
    prices = 0.05 + 0.25 * rng.random(T0 + 2)
    out = []
    for k in (0, 1):
        sess = session_generator(n, np.maximum(arr - k, 0).tolist(), (dep - k).tolist(), e.tolist(), e.tolist(), [32] * n,
                                 min_rates=mn, station_ids=st)
        iface = ab.TestingInterface({"active_sessions": sess, "infrastructure_info": infra, "current_time": 0, "period": 5,
                                     "prices": prices[k:].tolist(), "demand_charge": 15.51, "prev_peak": 20.0})
        aco = ab.AdaptiveChargingOptimization(BENCH, iface)
        S, I = iface.active_sessions(), iface.infrastructure_info()
        out.append(aco.build_instance(S, I, prev_peak=iface.get_prev_peak()))
    return aco, aco._site_for(I, out[0]), out


def _run(aco, site, inst, Tp, path, warm=None, shift=0, had=None, want_out=False, **opt):
    pb = engine.PackedBatch(site, [inst], Tp=Tp, S_max=16, want_warm_out=want_out)
    pb.warm = warm
    pb.struct.warm_shift = shift
    pb.struct.warm_had = None if had is None else engine._ptr(had)
    pb.upload().solve(_cabi.copy_options(aco._options(inst), path=path, **opt))
    torch.cuda.synchronize()
    r = dict(rates=pb.rates.cpu().numpy(), status=pb.status.cpu().numpy(), iters=pb.iters.cpu().numpy(), stats=pb.stats.cpu().numpy())
    if want_out:
        r.update({"out_" + k: v.cpu().numpy() for k, v in pb.warm_out.items()})
    return r


def _same(a, b, what):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), f"{what}: {k} differs"


def _paths(Tp):
    return (1, 2) if Tp in engine.SUPPORTED_HORIZONS else (2,)


@pytest.mark.parametrize("case", list(CASES))
def test_warm_shift_equals_host_shifted_state(require_gpu, case):
    Tp, T0, mins = CASES[case]
    aco, site, (x0, x1) = _pair(T0, mins)
    for path in _paths(Tp):
        prev = _run(aco, site, x0, Tp, path, want_out=True)
        assert prev["status"][0] == 0
        dev = {k: torch.from_numpy(prev["out_" + k]).cuda() for k in ("v1", "vc", "mu", "scal")}

        def shift(x):  # column t of the new problem is column t + 1 of the old one
            y = torch.zeros_like(x)
            y[:, :, :-1] = x[:, :, 1:]
            return y

        a = _run(aco, site, x1, Tp, path, warm=dev, shift=1, want_out=True)
        b = _run(aco, site, x1, Tp, path, warm=dict(v1=shift(dev["v1"]), vc=shift(dev["vc"]), mu=dev["mu"], scal=dev["scal"]), want_out=True)
        # (the warm-started general-path solve at Tp = 416 stops at the iteration limit: a finding of the same kind as
        # GENERAL_STALLS in test_gpu_solver_sweep.py; equality of the two feeds is what is pinned here)
        assert a["status"][0] == (_cabi.ACB_MAX_ITER if (case, path) == ("Tp416", 2) else _cabi.ACB_SOLVED), (path, a["status"], a["stats"])
        _same(a, b, f"path {path}")
        cold = _run(aco, site, x1, Tp, path)
        assert not np.array_equal(cold["rates"], a["rates"]) or cold["iters"][0] != a["iters"][0], f"path {path}: warm start had no effect"


@pytest.mark.parametrize("opts", [{}, {"max_rescues": 2}], ids=["defaults", "two_rescues"])
@pytest.mark.parametrize("case", list(CASES))
def test_warm_had_zero_is_a_cold_solve(require_gpu, case, opts):
    Tp, T0, mins = CASES[case]
    aco, site, (_, x1) = _pair(T0, mins)
    rng = np.random.default_rng(11)
    R = max(site.R, 1)
    garbage = dict(v1=torch.from_numpy(rng.uniform(-5, 40, (1, site.N, Tp)).astype(np.float32)).cuda(),
                   vc=torch.from_numpy(rng.uniform(-50, 50, (1, R, Tp)).astype(np.float32)).cuda(),
                   mu=torch.from_numpy(rng.uniform(-3, 3, (1, 16)).astype(np.float32)).cuda(),
                   scal=torch.tensor([[3.7, 99.0]], dtype=torch.float32).cuda())
    had = torch.zeros(1, dtype=torch.int32).cuda()
    for path in _paths(Tp):
        cold = _run(aco, site, x1, Tp, path, want_out=True, **opts)
        for shift in (0, 1):
            w = _run(aco, site, x1, Tp, path, warm=garbage, shift=shift, had=had, want_out=True, **opts)
            _same(w, cold, f"path {path}, warm_shift {shift}")
        assert cold["status"][0] == 0


def test_device_fleet_replay_equals_host_fleet_replay_general_path(require_gpu):
    device_vs_host_fleet_replay(list(range(80, 110)) + list(range(288 + 90, 288 + 100)), solver_options=dict(path=2))


def test_warm_started_steps_match_a_cold_oracle_solve_general_path(require_gpu):
    warm_steps_vs_cold_oracle(solver_options=dict(path=2))
