"""The checks every fleet replay feature runs, shared by the GPU tests: the device replay against its host twin, and
warm-started replay solves against a cold float64 oracle solve."""
import numpy as np

import adacharge_b200 as ab
from adacharge_b200.generators import caltech_acn_infrastructure, three_phase_balanced_network
from adacharge_b200.replay import SiteReplay
from adacharge_b200.replay_fast import DeviceFleetReplay, FleetReplay

BENCH = [ab.ObjectiveComponent(ab.tou_energy_cost), ab.ObjectiveComponent(ab.total_energy, 0.3), ab.ObjectiveComponent(ab.demand_charge, 1 / 30)]
BENCH_SPEC = [("tou_energy_cost", 1, {}), ("total_energy", 0.3, {}), ("demand_charge", 1 / 30, {})]  # the same, as the oracle takes it


def device_equals_host(infra, objective, steps, on_step=None, **replay_kw):
    """FleetReplay and DeviceFleetReplay built alike and stepped through `steps`: at every step the applied pilots and
    every state() entry that is not None are equal bit for bit; at the end the device summary's solves and unsolved
    equal the host's statistics.  `on_step(t, host, dev, first)` runs a test's own checks after each step."""
    host, dev = FleetReplay(infra, objective, **replay_kw), DeviceFleetReplay(infra, objective, **replay_kw)
    for t in steps:
        first = host.step(t)
        np.testing.assert_array_equal(first, dev.step(t), err_msg=f"applied pilots at step {t}")
        a, b = host.state(), dev.state()
        assert a.keys() == b.keys()
        for k in a:
            assert (a[k] is None) == (b[k] is None), (t, k)
            if a[k] is not None:
                np.testing.assert_array_equal(a[k], b[k], err_msg=f"{k} at step {t}")
        if on_step is not None:
            on_step(t, host, dev, first)
    s = dev.summary()
    assert s["solves"] == sum(host.stats.solved_sites) and s["unsolved"] == sum(host.stats.unsolved), (s, host.summary())
    return host, dev


def assert_as_good_as_cold_oracle(cases, spec, infra, period, prices, demand_charge, lb_tol=0.0, ub_tol=0.0):
    """Every case (t, site, sessions, prev_peak, R, status) is a warm-started replay solve, an ordinary MPC instance:
    status 0 and a schedule R as good as a cold float64 oracle solve of the same sessions -- objective within 1e-4 of the
    terms' magnitude (the sunk demand charge can cancel the revenue), network within 1e-5 relative, energy within 1e-4,
    bounds within lb_tol / ub_tol (ub_tol may be a function of the sessions).  The oracle's interior point occasionally
    breaks down on a step with a nearly served session: looser tolerances, else the case is skipped.
    Returns (compared, skipped, worst objective error of the term scale)."""
    from oracle import mpc

    worst, compared, skipped = 0.0, 0, 0
    for t, site, sess, prev_peak, R, status in cases:
        assert status == 0, (t, site, status)
        iface = ab.TestingInterface({"active_sessions": [], "infrastructure_info": infra, "current_time": t, "period": period,
                                     "prices": prices, "demand_charge": demand_charge, "prev_peak": prev_peak})
        I = iface.infrastructure_info()
        Ro = None
        for ts in (1.0, 100.0):
            try:
                Ro = mpc.solve_mpc(spec, sess, I, iface, "SOC", False, None, prev_peak, tol_scale=ts)
                break
            except mpc.OracleInfeasible:
                pass
        if Ro is None:
            skipped += 1
            continue
        compared += 1
        f, fo = (mpc.evaluate_objective(X, spec, I, iface, sess, prev_peak) for X in (R, Ro))
        mag = sum(abs(mpc.evaluate_objective(Ro, [o], I, iface, sess, prev_peak)) for o in spec)
        assert abs(f - fo) <= 1e-4 * max(abs(fo), mag) + 1e-7, (t, site, f, fo, mag)
        worst = max(worst, abs(f - fo) / max(abs(fo), mag))
        v = mpc.violations(R, sess, I, iface)
        ub = ub_tol(sess) if callable(ub_tol) else ub_tol
        assert v["infrastructure_rel"] <= 1e-5 and v["lb"] <= lb_tol and v["ub"] <= ub and v["energy"] <= 1e-4, (t, site, v, ub)
    return compared, skipped, worst


# ---------------------------------------------------------------------------------------------------- the default replay
# (test_gpu_replay.py on the default solve path, test_gpu_warm_start.py on the general path)
def device_vs_host_fleet_replay(steps, solver_options=None):
    host, _ = device_equals_host(caltech_acn_infrastructure(), BENCH, steps, n_sites=7, steps_per_day=288, days=2, seed0=40, mean_sessions=12,
                                 Tp=160, solver_options=solver_options)
    assert min(host.stats.active_sites) < 7 < sum(host.stats.active_sites)  # idle sites occurred


def warm_steps_vs_cold_oracle(solver_options=None):
    obj = [ab.ObjectiveComponent(getattr(ab, n), c, k) for n, c, k in BENCH_SPEC]
    infra = three_phase_balanced_network(3, 30)
    rp = SiteReplay(infra, obj, n_sites=3, steps=96, period=15, seed0=5, warm_start=True, mean_sessions=7, solver_options=solver_options)
    rp.keep_problems = True
    rp.run(28, 52)
    warm = [p[:6] for p in rp.problems if p[0] > 28]  # (t, site, sessions, prev_peak, R, status)
    assert len(warm) >= 20
    compared, skipped, worst = assert_as_good_as_cold_oracle(warm, BENCH_SPEC, infra, 15, rp.prices, rp.demand_charge)
    assert compared >= 20 and skipped <= 3, (compared, skipped)
    print(f"{compared} warm-started steps compared, worst objective error {worst:.1e} of the term scale")
