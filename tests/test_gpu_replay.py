"""Closed-loop replay with warm starts (BASELINE config 4 shape, small): every step solves,
warm starts cut the iteration count, and the EVs get their energy."""
import numpy as np
import pytest

import adacharge_b200 as ab
from adacharge_b200.generators import caltech_acn_infrastructure
from adacharge_b200.replay import SiteReplay

pytestmark = pytest.mark.gpu


def _run(warm, objective):
    rp = SiteReplay(caltech_acn_infrastructure(), objective, n_sites=6, steps=288, seed0=100, warm_start=warm)
    stats = rp.run(96, 136)
    return rp, stats


def test_replay_warm_start_reduces_iterations(require_gpu):
    obj = [ab.ObjectiveComponent(ab.tou_energy_cost), ab.ObjectiveComponent(ab.total_energy, 0.3), ab.ObjectiveComponent(ab.demand_charge, 1 / 30)]
    _, cold = _run(False, obj)
    _, warm = _run(True, obj)
    for st in cold.status + warm.status:
        assert (st == 0).all()
    ic = np.concatenate(cold.iters).mean()
    iw = np.concatenate(warm.iters).mean()
    print(f"mean iterations per step: cold {ic:.0f}, warm {iw:.0f}")
    assert iw < 0.8 * ic


def test_replay_quick_charge_delivers_energy(require_gpu):
    obj = [ab.ObjectiveComponent(ab.quick_charge), ab.ObjectiveComponent(ab.equal_share, 1e-6)]
    rp = SiteReplay(caltech_acn_infrastructure(), obj, n_sites=4, steps=288, seed0=7, warm_start=True)
    stats = rp.run(60, 288)
    for st in stats.status:
        assert (st == 0).all()
    assert (stats.delivered_frac >= 0.9999).all(), stats.delivered_frac  # t_int.py:37-39 asserts >= 99.99 %


def test_fleet_replay_matches_site_replay(require_gpu):
    """The array-based replay packs the same problems as the object-based one (constant rate
    limits passed as one pair per session): same pilots, same energy, same iteration counts."""
    from adacharge_b200.replay_fast import FleetReplay

    obj = [ab.ObjectiveComponent(ab.tou_energy_cost), ab.ObjectiveComponent(ab.total_energy, 0.3), ab.ObjectiveComponent(ab.demand_charge, 1 / 30)]
    infra = caltech_acn_infrastructure()
    slow = SiteReplay(infra, obj, n_sites=5, steps=288, seed0=300, warm_start=True)
    s_stats = slow.run(30, 70)
    fast = FleetReplay(infra, obj, n_sites=5, steps_per_day=288, seed0=300, warm_start=True)
    f_stats = fast.run(30, 70)
    assert sum(f_stats.unsolved) == 0
    dl_slow = np.array([sum(ev.delivered for ev in day) for day in slow.evs])
    dl_fast = np.bincount(fast.ev_site, weights=fast.ev_dlv, minlength=5)
    np.testing.assert_allclose(dl_fast, dl_slow, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(fast.prev_peak, slow.prev_peak, rtol=1e-6, atol=1e-6)
    it_slow = np.array([it.mean() for it in s_stats.iters])
    it_fast = np.array([m for m, a in zip(f_stats.iters_mean, f_stats.active_sites) if a > 0])
    np.testing.assert_allclose(it_fast[-len(it_slow):], it_slow, rtol=1e-6)


def test_fleet_replay_idle_sites_and_multi_day(require_gpu):
    """Steps where some sites have no EV at all (zero sessions in the batch) and a two-day EV table."""
    from adacharge_b200.replay_fast import FleetReplay

    obj = [ab.ObjectiveComponent(ab.quick_charge), ab.ObjectiveComponent(ab.equal_share, 1e-6)]
    fast = FleetReplay(caltech_acn_infrastructure(), obj, n_sites=6, steps_per_day=288, days=2, seed0=11, mean_sessions=6, Tp=160)
    stats = fast.run(40, 2 * 288)
    assert sum(stats.unsolved) == 0
    assert min(stats.active_sites) < 6  # some steps had idle sites
    assert (stats.delivered_frac >= 0.9999).all(), stats.delivered_frac


def test_device_fleet_replay_equals_host_fleet_replay(require_gpu):
    """SURVEY.md 8(f) N1: the simulator side of the step on the device (active sessions, energy delivered, previous
    peak, per-EV multipliers, warm start read one column ahead inside the solve) gives the same pilots, bit for bit,
    as the host-side replay, at every step, including idle sites and a second day."""
    device_vs_host_fleet_replay(list(range(80, 125)) + list(range(288 + 90, 288 + 110)))


def device_vs_host_fleet_replay(steps, solver_options=None):
    from adacharge_b200.replay_fast import DeviceFleetReplay, FleetReplay

    obj = [ab.ObjectiveComponent(ab.tou_energy_cost), ab.ObjectiveComponent(ab.total_energy, 0.3), ab.ObjectiveComponent(ab.demand_charge, 1 / 30)]
    infra = caltech_acn_infrastructure()
    kw = dict(n_sites=7, steps_per_day=288, days=2, seed0=40, mean_sessions=12, Tp=160, solver_options=solver_options)
    host, dev = FleetReplay(infra, obj, **kw), DeviceFleetReplay(infra, obj, **kw)
    for t in steps:
        a = host.step(t)
        b = dev.step(t, want_first=True)
        np.testing.assert_array_equal(a, b, err_msg=f"first-period pilots at step {t}")
    dev.run(0, 0)  # reads the device state back
    np.testing.assert_array_equal(dev.ev_dlv, host.ev_dlv)
    np.testing.assert_array_equal(dev.prev_peak, host.prev_peak)
    s = dev.summary()
    assert s["site_steps"] == sum(host.stats.active_sites) and s["unsolved"] == sum(host.stats.unsolved)
    assert min(host.stats.active_sites) < 7 < sum(host.stats.active_sites)  # idle sites occurred


def test_warm_started_steps_match_a_cold_oracle_solve(require_gpu):
    """Every warm-started closed-loop step is an ordinary MPC instance: its schedule must be as good as a cold float64
    oracle solve of the same step (objective within 1e-4, constraints satisfied).  Small three-phase site, 15-minute
    periods, so that the oracle takes a fraction of a second per step."""
    warm_steps_vs_cold_oracle()


def warm_steps_vs_cold_oracle(solver_options=None):
    from adacharge_b200.generators import three_phase_balanced_network
    from oracle import mpc

    spec = [("tou_energy_cost", 1, {}), ("total_energy", 0.3, {}), ("demand_charge", 1 / 30, {})]
    obj = [ab.ObjectiveComponent(getattr(ab, n), c, k) for n, c, k in spec]
    infra = three_phase_balanced_network(3, 30)
    rp = SiteReplay(infra, obj, n_sites=3, steps=96, period=15, seed0=5, warm_start=True, mean_sessions=7, solver_options=solver_options)
    rp.keep_problems = True
    rp.run(28, 52)
    warm = [p for p in rp.problems if p[0] > 28]
    assert len(warm) >= 20
    worst, compared, skipped = 0.0, 0, 0
    for t, s, sess, prev_peak, R, status, iters in warm:
        assert status == 0, (t, s, status)
        iface = ab.TestingInterface({"active_sessions": [], "infrastructure_info": infra, "current_time": t, "period": 15,
                                     "prices": rp.prices, "demand_charge": rp.demand_charge, "prev_peak": prev_peak})
        I = iface.infrastructure_info()
        Ro = None
        for ts in (1.0, 100.0):  # (the float64 interior point occasionally breaks down on a step with a nearly served session: looser tolerances, else skip)
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
        # the replay's tolerance is relative to the objective's terms (the sunk demand charge can cancel the revenue)
        assert abs(f - fo) <= 1e-4 * max(abs(fo), mag) + 1e-7, (t, s, f, fo, mag)
        worst = max(worst, abs(f - fo) / max(abs(fo), mag))
        v = mpc.violations(R, sess, I, iface)
        assert v["infrastructure_rel"] <= 1e-5 and v["lb"] <= 0 and v["ub"] <= 0 and v["energy"] <= 1e-4, (t, s, v)
    assert compared >= 20 and skipped <= 3, (compared, skipped)
    print(f"{compared} warm-started steps compared, worst objective error {worst:.1e} of the term scale")
