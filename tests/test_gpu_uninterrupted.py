"""Uninterrupted charging in the batched API and the fleet replays (acb_admit_sessions): AdaptiveSchedulingAlgorithm's
uninterrupted_charging (reference adacharge/adacharge.py:149-150 -> acnportal's apply_minimum_charging_rate with
override = period), per instance, bit for bit what the drop-in class does with the same flags."""
import ctypes as C
from copy import deepcopy

import numpy as np
import pytest
import torch

import adacharge_b200 as ab
from adacharge_b200 import _cabi, engine
from adacharge_b200.algorithms_shim import apply_minimum_charging_rate, apply_upper_bound_estimate, enforce_pilot_limit
from adacharge_b200.batched import BatchedAdaptiveCharging, sessions_to_arrays
from adacharge_b200.generators import caltech_acn_infrastructure, config_c2, session_generator, three_phase_balanced_network
from oracle import mpc
from tests.replay_checks import assert_as_good_as_cold_oracle, device_equals_host

pytestmark = pytest.mark.gpu

BENCH_OBJ = [("tou_energy_cost", 1.0, {}), ("total_energy", 0.3, {}), ("demand_charge", 1.0 / 30.0, {})]
SPEC = [("quick_charge", 1, {}), ("equal_share", 1e-3, {})]


def _components(spec):
    return [ab.ObjectiveComponent(getattr(ab, n), c, k) for n, c, k in spec]


def _numpy_feasible(rates, infra):
    """infrastructure_constraints_feasible in plain numpy (reference adacharge/utils.py:5-12): no device code."""
    ph = np.deg2rad(np.asarray(infra.phases, dtype=float))
    for j, v in enumerate(np.asarray(infra.constraint_matrix, dtype=float)):
        a = np.stack([v * np.cos(ph), v * np.sin(ph)])
        if not np.all(np.linalg.norm(a @ rates, axis=0) <= infra.constraint_limits[j] + 1e-7):
            return False
    return True


def _reference_min_rate_loop(sessions, infra, override):
    """The per-session loop as acnportal writes it, one feasibility call per session, in pure numpy."""
    queue = deepcopy(sorted(sessions, key=lambda x: x.arrival))
    rates = np.zeros(len(infra.station_ids))
    flags = []
    for s in queue:
        i = infra.get_station_index(s.station_id)
        rates[i] = min(infra.min_pilot[i], override)
        ok = _numpy_feasible(rates, infra)
        if not ok:
            rates[i] = 0
        flags.append(ok)
    return flags


def _c2_dicts(n, seed0, infra):
    """C2 instances in shuffled slot order (arrival order != slot order) with every third session arriving now (ties)."""
    rng = np.random.default_rng(seed0)
    out = []
    for i in range(n):
        d = config_c2(seed0 + i, infra=infra, price_noise=0.2)
        ss = [d["active_sessions"][k] for k in rng.permutation(len(d["active_sessions"]))]
        for j, s in enumerate(ss):
            if j % 3 == 0:
                s["arrival"] = 0
        d["active_sessions"] = ss
        out.append(d)
    return out


class _Est:
    """max_rate_estimator with fixed per-session upper bounds."""

    def __init__(self, ub):
        self.ub = ub

    def register_interface(self, interface):
        pass

    def get_maximum_rates(self, sessions):
        return self.ub


def _raw_after_admission(bac, sess, **kw):
    """Upload, preprocess and admit one chunk; the raw tables and first-period limits as the admission left them."""
    ch = bac.chunks[0]
    bac.upload_raw(sess, **kw)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _cabi.check(_cabi.lib().acb_preprocess_sessions(bac.site.handle, C.byref(ch.sessions), 1, engine._ptr(ch.dev_raw.get("upper_bound")), st), "pre")
    bac.admit(ch, st)
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in ch.dev_raw.items()}
    out.update({k: v.cpu().numpy() for k, v in ch.limits0.items()})
    return out


@pytest.mark.parametrize("cap", [150, 20, 12, 6])
def test_admission_matches_the_sequential_loop(require_gpu, cap):
    """acb_admit_sessions against the pure-numpy loop and the drop-in's host helper: the order of the permuted tables,
    the admitted flags and the first-period limits, from slack to heavily congested transformers."""
    infra = caltech_acn_infrastructure(transformer_cap=cap)
    ds = _c2_dicts(4, 200 + cap, infra)
    ifaces = [ab.TestingInterface(d) for d in ds]
    I = ifaces[0].infrastructure_info()
    sess = sessions_to_arrays([f.active_sessions() for f in ifaces], I, S_max=54)
    bac = BatchedAdaptiveCharging(_components(SPEC), I, 5, batch=4, max_sessions=54, horizon=288, chunks=1, uninterrupted_charging=True)
    got = _raw_after_admission(bac, sess)
    refused = admitted = 0
    for b, iface in enumerate(ifaces):
        S = enforce_pilot_limit(iface.active_sessions(), I)
        want = _reference_min_rate_loop(S, I, 5)
        queue = sorted(S, key=lambda x: x.arrival)
        assert [s.arrival for s in S] != [s.arrival for s in queue]  # slot order is not arrival order
        assert len({s.arrival for s in S}) < len(S)  # ties
        n = len(S)
        np.testing.assert_array_equal(got["station"][b, :n], [I.get_station_index(s.station_id) for s in queue])
        np.testing.assert_array_equal(got["arrival"][b, :n], [s.arrival for s in queue])
        np.testing.assert_array_equal(got["remaining_demand"][b, :n], [s.remaining_demand for s in queue])
        assert (got["station"][b, n:] == -1).all()
        np.testing.assert_array_equal(got["min_rate0"][b, :n] > 0, want)
        host = apply_minimum_charging_rate(S, I, 5)
        np.testing.assert_array_equal(got["min_rate0"][b, :n], [s.min_rates[0] for s in host])
        np.testing.assert_array_equal(got["max_rate0"][b, :n], [s.max_rates[0] for s in host])
        refused += n - sum(want)
        admitted += sum(want)
    assert admitted > 0
    if cap <= 12:
        assert refused > 0


def _dropin(spec, iface, quantize, reallocate, est=None):
    alg = ab.AdaptiveSchedulingAlgorithm(_components(spec), estimate_max_rate=est is not None, max_rate_estimator=est, uninterrupted_charging=True,
                                         quantize=quantize, reallocate=reallocate, solver_options=dict(eps_rel=1e-4))
    alg.register_interface(iface)
    sched = alg.schedule(iface.active_sessions())
    I = iface.infrastructure_info()
    return None if not sched else np.stack([sched[s] for s in I.station_ids])


MODES = [(False, False), (True, False), (True, True)]
MODE_IDS = ["continuous", "quantize", "reallocate"]


@pytest.mark.parametrize("quantize,reallocate", MODES, ids=MODE_IDS)
def test_batched_equals_dropin(require_gpu, quantize, reallocate):
    """Congested transformer (some sessions refused), sessions with a positive minimum rate of their own, the estimator's
    upper bounds, an empty instance and three chunks: the pilots of every instance equal the drop-in class's."""
    infra = caltech_acn_infrastructure(transformer_cap=40)
    ds = _c2_dicts(8, 70, infra)
    ds.insert(3, dict(ds[0], active_sessions=[]))
    for d in ds[1::2]:  # a small minimum rate of their own on a few sessions that can absorb it
        for s in d["active_sessions"][1::4]:
            if s["requested_energy"] > 4 * 208 / 1000 * 5 / 60 * (s["departure"] - s["arrival"]):
                s["min_rates"] = 3.0
    ifaces = [ab.TestingInterface(d) for d in ds]
    I = ifaces[0].infrastructure_info()
    lists = [f.active_sessions() for f in ifaces]
    assert any(s.min_rates[0] > 0 for ss in lists for s in ss)
    sess = sessions_to_arrays(lists, I, S_max=54)
    rng = np.random.default_rng(1)
    upper = rng.uniform(4.0, 40.0, size=sess["max_rate"].shape)
    prices = np.stack([np.asarray(f.get_prices(288), dtype=float) for f in ifaces])
    prev = np.array([f.get_prev_peak() for f in ifaces])
    bac = BatchedAdaptiveCharging(_components(BENCH_OBJ), I, 5, batch=len(ifaces), max_sessions=54, horizon=288, demand_charge=15.51, chunks=3,
                                  estimate_max_rate=True, quantize=quantize, reallocate=reallocate, uninterrupted_charging=True)
    res = bac.schedule(sess, prices=prices, prev_peak=prev, upper_bound=upper)
    refused = 0
    for b, iface in enumerate(ifaces):
        S = lists[b]
        if not S:
            assert not res.pilots[b].any()
            continue
        est = _Est({s.session_id: upper[b, j] for j, s in enumerate(S)})
        pre = apply_minimum_charging_rate(apply_upper_bound_estimate(est, enforce_pilot_limit(S, I)), I, 5)
        assert any(s.min_rates[0] > 0 for s in pre)  # both sides take the same kernel variant
        refused += sum(s.max_rates[0] == 0 for s in pre)
        want = _dropin(BENCH_OBJ, iface, quantize, reallocate, est)
        T = want.shape[1]
        assert res.status[b] == 0 and res.T[b] == T
        np.testing.assert_array_equal(res.pilots[b, :, :T], want, err_msg=f"instance {b}")
        assert not res.pilots[b, :, T:].any()
    assert refused > 0


def _multi_and_long_cases(infra, long):
    """Instances in which one EVSE holds two sessions (the second arrives after the first leaves), or (long) a horizon
    beyond the on-chip kernel's 288 periods; shuffled arrivals with ties."""
    ids = infra["station_ids"]
    rng = np.random.default_rng(11 if long else 12)
    out = []
    for k in range(3):
        n = 30
        arr = rng.integers(0, 40, n)
        arr[::4] = 0
        dep = arr + rng.integers(40, 150, n)
        st = rng.permutation(54)[:n].tolist()
        if long:
            dep[0] = 300 + k
        else:  # EVSE st[1] gets a second session after the first one leaves
            st.append(st[1])
            arr = np.append(arr, dep[1] + 2)
            dep = np.append(dep, dep[1] + 60)
            n += 1
        dem = np.minimum(rng.uniform(2, 15, n), 0.8 * (dep - arr) * 32 * 208 / 1000 * 5 / 60)
        ss = session_generator(n, arr.tolist(), dep.tolist(), dem.tolist(), dem.tolist(), [32] * n, station_ids=[ids[i] for i in st])
        out.append({"active_sessions": ss, "infrastructure_info": infra, "current_time": 0, "period": 5, "prices": np.full(320, 0.1),
                    "demand_charge": 15.51, "prev_peak": 10.0})
    return out


@pytest.mark.parametrize("quantize,reallocate", [MODES[0], MODES[2]], ids=[MODE_IDS[0], MODE_IDS[2]])
@pytest.mark.parametrize("case", ["multi_session", "long_horizon"])
def test_batched_equals_dropin_multi_session_and_general_path(require_gpu, case, quantize, reallocate):
    """Two sessions on one EVSE (the packer's (EVSE, slot) sort then ranks by the arrival-sorted slot, as the drop-in's
    host packer does), and T > 288 (the general solve path)."""
    long = case == "long_horizon"
    infra = caltech_acn_infrastructure(transformer_cap=30)
    ifaces = [ab.TestingInterface(d) for d in _multi_and_long_cases(infra, long)]
    I = ifaces[0].infrastructure_info()
    lists = [f.active_sessions() for f in ifaces]
    sess = sessions_to_arrays(lists, I, S_max=64)
    horizon = 320 if long else 288
    prices = np.stack([np.asarray(f.get_prices(horizon), dtype=float) for f in ifaces])
    bac = BatchedAdaptiveCharging(_components(SPEC), I, 5, batch=3, max_sessions=64, horizon=horizon, multi_session=not long, chunks=1,
                                  quantize=quantize, reallocate=reallocate, uninterrupted_charging=True)
    res = bac.schedule(sess, prices=prices)
    for b, iface in enumerate(ifaces):
        pre = apply_minimum_charging_rate(enforce_pilot_limit(lists[b], I), I, 5)
        assert any(s.min_rates[0] > 0 for s in pre)
        want = _dropin(SPEC, iface, quantize, reallocate)
        T = want.shape[1]
        assert (T > 288) == long and res.status[b] == 0 and res.T[b] == T
        np.testing.assert_array_equal(res.pilots[b, :, :T], want, err_msg=f"{case}, instance {b}")


def test_small_remainder(require_gpu):
    """An arrived session that cannot absorb one period at its try rate: without skip_unabsorbable the instance is
    ACB_INFEASIBLE where the drop-in raises; with it the session keeps its own bounds and the rest is the oracle's."""
    infra = caltech_acn_infrastructure(transformer_cap=40)
    d = config_c2(17, infra=infra)
    d["active_sessions"][0]["arrival"] = 0
    d["active_sessions"][0]["requested_energy"] = d["active_sessions"][0]["energy_delivered"] + 0.05  # < 5 A for 5 minutes at 208 V
    iface = ab.TestingInterface(d)
    I = iface.infrastructure_info()
    S = iface.active_sessions()
    sess = sessions_to_arrays([S, S], I, S_max=54)
    with pytest.raises(ab.InfeasibilityException):
        _dropin(SPEC, iface, False, False)
    for skip in (False, True):
        bac = BatchedAdaptiveCharging(_components(SPEC), I, 5, batch=2, max_sessions=54, horizon=288, chunks=1, uninterrupted_charging=True,
                                      skip_unabsorbable=skip)
        res = bac.schedule(sess)
        if not skip:
            assert (res.status == _cabi.ACB_INFEASIBLE).all()
            continue
        assert (res.status == 0).all()
        np.testing.assert_array_equal(res.pilots[0], res.pilots[1])
        small = S[0]
        pre = apply_minimum_charging_rate(enforce_pilot_limit(S[1:], I), I, 5) + enforce_pilot_limit([small], I)
        assert any(s.min_rates[0] > 0 for s in pre)
        T = mpc.horizon(pre)
        R = res.pilots[0, :, :T]
        v = mpc.violations(R, pre, I, iface, "SOC", None)
        assert v["lb"] <= 1e-4 and v["ub"] <= 1e-4 and v["infrastructure_rel"] <= 1e-5 and v["energy"] <= 2e-4, v
        Ro = mpc.solve_mpc(SPEC, pre, I, iface, "SOC", False, None, iface.get_prev_peak())
        f, fo = (mpc.evaluate_objective(X, SPEC, I, iface, pre, iface.get_prev_peak()) for X in (R, Ro))
        assert abs(f - fo) <= 1e-4 * abs(fo), (f, fo)


@pytest.mark.parametrize("quantize,reallocate", [MODES[0], MODES[2]], ids=[MODE_IDS[0], MODE_IDS[2]])
def test_device_fleet_replay_equals_host(require_gpu, quantize, reallocate):
    """Two days of a congested fleet: first-period pilots, statuses, delivered energy and peaks of the device replay equal
    the host replay's, bit for bit; no site-step is infeasible; with continuous pilots every admitted EV gets at least
    its minimum."""
    n = dict(adm=0, ref=0)

    def on_step(t, host, dev, first):
        h = {k: v.numpy() for k, v in host._pb.host.items()}
        act = h["n_sessions"] > 0
        assert not (host.state()["status"][act] == _cabi.ACB_INFEASIBLE).any(), t
        for s in np.nonzero(act)[0]:
            k = h["n_sessions"][s]
            mn0, rows = h["sess_min0"][s, :k], h["sess_row"][s, :k]
            n["adm"] += int((mn0 > 0).sum())
            n["ref"] += int((h["sess_max0"][s, :k] == 0).sum())
            if not quantize:
                assert (first[s, rows] >= mn0 - 1e-4).all(), (t, s, first[s, rows], mn0)

    _, dev = device_equals_host(caltech_acn_infrastructure(transformer_cap=10), _components(BENCH_OBJ),
                                list(range(80, 130)) + list(range(288 + 90, 288 + 115)), on_step, n_sites=7, steps_per_day=288, days=2,
                                seed0=40, mean_sessions=14, Tp=160, quantize=quantize, reallocate=reallocate, uninterrupted_charging=True)
    assert not dev._ch.lb_zero
    assert n["adm"] > 0 and n["ref"] > 0, n


def test_warm_started_uninterrupted_steps_match_a_cold_oracle_solve(require_gpu):
    """Every warm-started step of the replay with uninterrupted charging is an MPC instance with first-period limits:
    its schedule is as good as a cold float64 oracle solve of the same preprocessed sessions."""
    from adacharge_b200.interface import SessionInfo
    from adacharge_b200.replay_fast import FleetReplay

    spec = [("tou_energy_cost", 1, {}), ("total_energy", 0.3, {}), ("demand_charge", 1 / 30, {})]
    infra = three_phase_balanced_network(3, 30)
    rp = FleetReplay(infra, _components(spec), n_sites=3, steps_per_day=96, days=1, period=15, seed0=5, mean_sessions=7, Tp=64,
                     uninterrupted_charging=True)
    I = rp.info
    cases, with_min = [], 0
    for t in range(28, 56):
        _, idx, s_of, pos, n_sess = rp._pack(t)
        prev_peak, owed = rp.prev_peak.copy(), rp.ev_req - rp.ev_dlv  # the state the step starts from
        rp.step(t)
        if t == 28:
            continue  # cold start
        mn0, mx0 = rp._limits0
        R_all = rp._pb.rates.cpu().numpy().astype(np.float64)
        st_all = rp.state()["status"]
        for site in np.nonzero(n_sess > 0)[0]:
            sess = []
            for j in np.nonzero(s_of == site)[0]:
                e = idx[j]
                rem = rp.ev_dep[e] - t
                sess.append(SessionInfo(I.station_ids[rp.ev_station[e]], f"ev{e}", owed[e], 0.0, t, int(rp.ev_dep[e]),
                                        current_time=t, min_rates=np.concatenate(([mn0[j]], np.zeros(rem - 1))),
                                        max_rates=np.concatenate(([mx0[j]], np.full(rem - 1, rp.ev_max[e])))))
            with_min += sum(s.min_rates[0] > 0 for s in sess)
            cases.append((t, site, sess, prev_peak[site], R_all[site, :, :mpc.horizon(sess)], st_all[site]))
    compared, skipped, worst = assert_as_good_as_cold_oracle(cases, spec, infra, 15, rp.prices, rp.demand_charge, lb_tol=1e-4, ub_tol=1e-4)
    assert compared >= 20 and skipped <= 3 and with_min > 0, (compared, skipped, with_min)
    print(f"{compared} warm-started steps compared, worst objective error {worst:.1e} of the term scale")
