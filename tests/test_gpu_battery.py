"""Two-stage batteries and the rampdown max-rate estimate in the fleet replays, on the GPU.

- The device replay equals the host replay bit for bit at every step (applied pilots, per-EVSE currents, recompute
  mask) and in the final state (delivered energy, battery charge, estimates, peaks), with and without the estimate, at
  max_recompute 1 and None, with quantised reallocated pilots and with uninterrupted charging.
- Batteries too large to ever limit an EV (and the estimate without batteries) give the default replay bit for bit.
- On a hand-built site the estimate caps the next solve's maximum rate at a + up_increment.
- Warm-started solves whose bounds were lowered since the site's last solve against a cold float64 oracle solve.
"""
import numpy as np
import pytest

import adacharge_b200 as ab
from adacharge_b200 import replay_fast
from adacharge_b200.generators import caltech_acn_infrastructure, three_phase_balanced_network
from adacharge_b200.interface import SessionInfo
from adacharge_b200.replay import EV
from adacharge_b200.replay_fast import DeviceFleetReplay, FleetReplay
from tests.replay_checks import BENCH, assert_as_good_as_cold_oracle, device_equals_host

pytestmark = pytest.mark.gpu
STEPS = list(range(60, 150)) + list(range(288 + 80, 288 + 110))


def _fleet(**kw):
    """Two days of a congested C4-shaped fleet (CaltechACN site, 40 mean sessions), 7 sites."""
    return dict(n_sites=7, steps_per_day=288, days=2, seed0=40, mean_sessions=40, Tp=160, **kw)


def _dev_vs_host(steps, **kw):
    """device_equals_host on the fleet, counting the EVSE-steps where a battery took less than its pilot and the
    EV-steps where the estimate moved."""
    n, last = dict(taper=0, fired=0), {}

    def on_step(t, host, dev, first):
        s = host.state()
        n["taper"] += int((s["rates"] < first).sum())
        if s["ev_ub"] is not None:
            before = last.get("ub", np.asarray(host.info.max_pilot, dtype=np.float64)[host.ev_station])  # (the estimates start at max_pilot)
            n["fired"] += int((s["ev_ub"] != before).sum())
            last["ub"] = s["ev_ub"]

    host, _ = device_equals_host(caltech_acn_infrastructure(), BENCH, steps, on_step, **_fleet(**kw))
    return host, n["taper"], n["fired"]


@pytest.mark.parametrize("max_recompute", [1, None])
@pytest.mark.parametrize("estimate", [False, True])
def test_device_replay_equals_host_replay(require_gpu, estimate, max_recompute):
    host, taper, fired = _dev_vs_host(STEPS, battery=True, estimate_max_rate=estimate, max_recompute=max_recompute)
    assert taper > 0, "no battery took less than its pilot"
    assert (fired > 0) == estimate
    assert (host.ev_charge <= host.ev_cap).all() and (host.ev_dlv <= host.ev_req + 1e-9).all()


@pytest.mark.parametrize("kw", [dict(quantize=True, reallocate=True), dict(uninterrupted_charging=True, max_recompute=None)],
                         ids=["reallocate", "uninterrupted"])
def test_device_replay_equals_host_replay_with_flags(require_gpu, kw):
    _, taper, fired = _dev_vs_host(STEPS, battery=True, estimate_max_rate=True, **kw)
    assert taper > 0 and fired > 0


def _same_as_default(cls, steps, **kw):
    """The replay with kw against the default one; returns it and its final state."""
    infra = caltech_acn_infrastructure()
    a, b = cls(infra, BENCH, **_fleet()), cls(infra, BENCH, **_fleet(**kw))
    for t in steps:
        first = b.step(t)
        np.testing.assert_array_equal(a.step(t), first, err_msg=f"step {t}")
        rates = b.state()["rates"]
        np.testing.assert_array_equal(rates, np.where(rates > 0, first, 0.0), err_msg=f"currents at step {t}")
    sa, sb = a.state(), b.state()
    for k in ("ev_dlv", "prev_peak"):
        np.testing.assert_array_equal(sa[k], sb[k], err_msg=k)
    return b, sb


@pytest.mark.parametrize("cls", [FleetReplay, DeviceFleetReplay])
def test_huge_batteries_are_the_default_replay(require_gpu, monkeypatch, cls):
    """Batteries that never reach their transition (a == p, stated in amperes) and an estimate that therefore never fires:
    the default replay bit for bit."""
    monkeypatch.setattr(replay_fast, "synthetic_batteries", lambda seed, req: (np.full(len(req), 1e9), np.zeros(len(req))))
    b, s = _same_as_default(cls, STEPS[:60], battery=True, estimate_max_rate=True)
    np.testing.assert_array_equal(s["ev_ub"], np.asarray(b.info.max_pilot)[b.ev_station])
    assert (s["ev_charge"] == s["ev_dlv"]).all()


@pytest.mark.parametrize("cls", [FleetReplay, DeviceFleetReplay])
def test_estimate_without_batteries_is_a_no_op(require_gpu, cls):
    b, s = _same_as_default(cls, STEPS[:40], estimate_max_rate=True)
    np.testing.assert_array_equal(s["ev_ub"], np.asarray(b.info.max_pilot)[b.ev_station])


# ---------------------------------------------------------------------------------------------------- semantics
def _one_ev(monkeypatch, estimate):
    monkeypatch.setattr(replay_fast, "synthetic_day", lambda *a, **k: [EV(station=5, session_id="a", arrival=10, departure=100, requested=10.0)])
    monkeypatch.setattr(replay_fast, "synthetic_batteries", lambda seed, req: (np.array([20.0]), np.array([19.0])))  # soc 0.95
    obj = [ab.ObjectiveComponent(ab.quick_charge), ab.ObjectiveComponent(ab.equal_share, 1e-6)]
    kw = dict(n_sites=1, steps_per_day=288, days=1, seed0=0, Tp=160, battery=True, estimate_max_rate=estimate)
    infra = caltech_acn_infrastructure()
    return DeviceFleetReplay(infra, obj, **kw), FleetReplay(infra, obj, **kw)


def test_estimate_caps_the_next_solve(require_gpu, monkeypatch):
    dev, host = _one_ev(monkeypatch, True)
    bound, lowered = float(dev.info.max_pilot[5]), False  # the estimate starts at the EVSE's max_pilot
    for t in range(10, 30):
        p = dev.step(t)[0, 5]
        np.testing.assert_array_equal(host.step(t)[0, 5], p)
        mx = dev._ch.dev_raw["max_rate"].cpu().numpy()[0, 0]  # the session's maximum rate after the preprocessing
        assert mx == min(32.0, bound), (t, mx, bound)
        if lowered:  # (the solve takes the bound rounded to float32)
            assert p <= np.float32(bound), (t, bound, p)
        s = dev.state()
        a = s["rates"][0, 5]
        assert a == host.rates[0, 5]
        if p - a > 1.0:
            bound, lowered = a + 1.0, True
        assert s["ev_ub"][0] == bound == host.ev_ub[0]
    assert bound < 9.0  # deep in the taper: the EV takes at most (1 - 0.95) / 0.2 * 32 = 8 A


def test_without_the_estimate_the_pilot_stays_above_the_current(require_gpu, monkeypatch):
    dev, host = _one_ev(monkeypatch, False)
    for t in range(10, 30):
        p = dev.step(t)[0, 5]
        np.testing.assert_array_equal(host.step(t)[0, 5], p)
        assert dev._ch.dev_raw["max_rate"].cpu().numpy()[0, 0] == 32.0
        a = dev.state()["rates"][0, 5]
        assert p > a + 1.0, (t, p, a)


# ---------------------------------------------------------------------------------------------------- warm starts
def test_lowered_bounds_match_a_cold_oracle_solve(require_gpu):
    """Warm-started solves where the estimate lowered some session's maximum rate since the site's previous solve are
    ordinary MPC instances: the schedule is as good as a cold float64 oracle solve of the same step."""
    spec = [("tou_energy_cost", 1, {}), ("total_energy", 0.3, {}), ("demand_charge", 1 / 30, {})]
    obj = [ab.ObjectiveComponent(getattr(ab, n), c, k) for n, c, k in spec]
    infra = three_phase_balanced_network(3, 30)
    rp = FleetReplay(infra, obj, n_sites=6, steps_per_day=96, days=1, period=15, seed0=5, mean_sessions=7, Tp=128, battery=True,
                     estimate_max_rate=True)
    last_mx = np.full(len(rp.ev_req), np.inf)  # each EV's maximum rate at its site's previous solve
    cases = []
    for t in range(96):
        _, idx, s, _, n_sess = rp._pack(t)
        mx = rp._max_rate(idx)
        had, peak = rp.had.copy(), rp.prev_peak.copy()
        sess = {b: [SessionInfo(infra["station_ids"][rp.ev_station[e]], str(e), rp.ev_req[e], rp.ev_dlv[e], int(rp.ev_arr[e]),
                                int(rp.ev_dep[e]), current_time=t, max_rates=m) for e, m in zip(idx[s == b], mx[s == b])] for b in range(rp.n_sites)}
        lowered = np.bincount(s[mx < last_mx[idx]], minlength=rp.n_sites) > 0
        rp.step(t)
        last_mx[idx] = mx
        R = rp._pb.rates.cpu().numpy().astype(np.float64)
        st = rp.state()["status"]
        for b in range(rp.n_sites):
            if lowered[b] and had[b] and n_sess[b] > 0 and len(cases) < 40:
                T = max(x.arrival_offset + x.remaining_time for x in sess[b])
                cases.append((t, b, sess[b], float(peak[b]), R[b][:, :T], int(st[b])))

    def f32_up(sess):  # a lowered bound (a + up_increment) reaches the solve rounded to float32: the rates keep that bound exactly
        return max(max(float(np.float32(x.max_rates[0])) - float(x.max_rates[0]), 0.0) for x in sess)

    compared, skipped, worst = assert_as_good_as_cold_oracle(cases, spec, infra, 15, rp.prices, rp.demand_charge, ub_tol=f32_up)
    assert compared >= 20 and skipped <= 3, (len(cases), compared, skipped)
    print(f"{compared} warm-started solves with lowered bounds compared, worst objective error {worst:.1e} of the term scale")
