"""Host-side rules of two-stage batteries and the rampdown estimate in the fleet replays (no GPU): the vectorised battery
and estimator update against a scalar loop written from the stated rules, the replay options, the battery data, the
estimate's cut of the session tables, and the C ABI of acb_fleet_ev."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import adacharge_b200 as ab
from adacharge_b200 import _cabi, replay_fast
from adacharge_b200.generators import caltech_acn_infrastructure
from adacharge_b200.replay import synthetic_batteries, synthetic_day
from adacharge_b200.replay_fast import FleetReplay, battery_current, rampdown_update

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = open(os.path.join(ROOT, "include", "adacharge_b200.h")).read()
OBJ = [ab.ObjectiveComponent(ab.total_energy)]


def _replay(**kw):
    return FleetReplay(caltech_acn_infrastructure(), OBJ, **{**dict(n_sites=3, steps_per_day=288, days=2, seed0=4, mean_sessions=20), **kw})


# ---------------------------------------------------------------------------------------------------- the model
def _literal(p, w, amax, cap, charge, owed, theta):
    """The battery rule, one EV, as DESIGN.md §8 states it."""
    if p == 0:
        a = 0.0
    else:
        soc = charge / cap
        if soc < theta:
            a = min(p, amax)
        else:
            a = min(p, ((1 - soc) / (1 - theta)) * amax)
        if charge + a * w > cap:
            a = (cap - charge) / w
        a = max(a, 0.0)
    de = max(min(a * w, owed), 0.0)
    return a, de


def _literal_ub(ub, p, a, up, down):
    return a + up if p - a > down else ub


W = 208 * 5 / 1e3 / 60  # kWh per A-period at 208 V, 5-minute periods
# (p, amax, cap, charge, owed, what the case covers)
CASES = [
    (0.0, 32.0, 50.0, 10.0, 5.0, "pilot 0"),
    (0.0, 32.0, 50.0, 45.0, 5.0, "pilot 0 in the taper"),
    (16.0, 32.0, 50.0, 10.0, 5.0, "below the transition: the pilot"),
    (40.0, 32.0, 50.0, 10.0, 5.0, "below the transition: the EV's maximum"),
    (32.0, 32.0, 50.0, 45.0, 5.0, "in the taper"),
    (4.0, 32.0, 50.0, 45.0, 5.0, "in the taper, below the taper's limit"),
    (32.0, 32.0, 50.0, 40.0, 5.0, "at the transition"),
    (32.0, 32.0, 2.0, 1.9, 5.0, "the capacity clamp"),  # (a battery small enough that the taper alone would overfill it)
    (32.0, 32.0, 50.0, 50.0, 5.0, "full"),
    (32.0, 32.0, 50.0, 10.0, 0.05, "the owed cap"),
    (32.0, 32.0, 50.0, 10.0, 0.0, "nothing owed"),
    (32.0, 32.0, 50.0, 10.0, -1e-12, "owed below 0"),
]


def test_battery_equals_the_literal_rule():
    cases = list(CASES)
    rng = np.random.default_rng(0)
    for _ in range(3000):  # random states across both stages, the clamp and the owed cap
        cap = rng.uniform(5, 80)
        cases.append((float(rng.choice([0.0, rng.uniform(0, 48), 32.0, 6.0])), float(rng.choice([32.0, 16.0, rng.uniform(6, 80)])), cap,
                      float(cap * rng.choice([rng.uniform(0, 1), rng.uniform(0.95, 1.0), 1.0])), float(rng.choice([rng.uniform(0, 3), 1e-3, 20.0])), "random"))
    p, amax, cap, charge, owed = (np.array([c[k] for c in cases]) for k in range(5))
    for theta in (0.8, 0.5, 0.95):
        a, de = battery_current(p, W, amax, cap, charge, owed, theta)
        want = np.array([_literal(*c[:1], W, *c[1:5], theta) for c in cases])
        for j, c in enumerate(cases):
            assert (a[j], de[j]) == tuple(want[j]), (c, theta, (a[j], de[j]), tuple(want[j]))
        np.testing.assert_array_equal(a.view(np.uint64) >> 63, 0)  # no negative current, not even -0
    a, _ = battery_current(p, W, amax, cap, charge, owed, 0.8)
    kinds = {c[-1]: (p[j], a[j]) for j, c in enumerate(cases)}
    assert kinds["pilot 0 in the taper"][1] == 0.0
    assert kinds["below the transition: the pilot"] == (16.0, 16.0) and kinds["below the transition: the EV's maximum"][1] == 32.0
    assert 0 < kinds["in the taper"][1] < 32.0 and kinds["in the taper, below the taper's limit"][1] == 4.0
    assert kinds["the capacity clamp"][1] == pytest.approx(0.1 / W) and kinds["full"][1] == 0.0
    # the whole charge of one EV under a constant pilot: the taper, then the clamp, then nothing
    cap, charge, owed, seen = 40.0, 20.0, 30.0, []
    while owed > 0 and len(seen) < 2000:
        a, de = battery_current(np.array([32.0]), W, np.array([32.0]), np.array([cap]), np.array([charge]), np.array([owed]), 0.8)
        want = _literal(32.0, W, 32.0, cap, charge, owed, 0.8)
        assert (a[0], de[0]) == want
        charge, owed = charge + de[0], owed - de[0]
        seen.append(a[0])
        if a[0] == 0.0:
            break
    assert seen[0] == 32.0 and min(seen) < 1.0 and charge <= cap


def test_rampdown_equals_the_literal_rule():
    rng = np.random.default_rng(1)
    n = 2000
    p = rng.choice([0.0, 8.0, 32.0], n) + rng.choice([0.0, 1.0, 0.5], n)
    a = np.maximum(p - rng.choice([0.0, 0.5, 1.0, 1.0 + 1e-9, 3.0, 20.0], n), 0.0)
    ub = rng.uniform(0, 32, n)
    for up, down in ((1.0, 1.0), (2.5, 0.0), (0.25, 4.0)):
        got, fire = rampdown_update(ub, p, a, up, down)
        want = np.array([_literal_ub(*x, up, down) for x in zip(ub, p, a)])
        np.testing.assert_array_equal(got, want)
        assert fire.any() and not fire.all()
        np.testing.assert_array_equal(got[~fire], ub[~fire])  # no min with the old value, no change where it does not fire
    got, fire = rampdown_update(np.array([5.0, 5.0, 5.0]), np.array([32.0, 10.0, 10.0]), np.array([8.0, 9.0, 8.5]), 1.0, 1.0)
    assert list(got) == [9.0, 5.0, 9.5] and list(fire) == [True, False, True]  # 9 > 5 as well: the bound can rise


# ---------------------------------------------------------------------------------------------------- options and data
@pytest.mark.parametrize("kw,what", [(dict(transition_soc=0.0), "transition_soc"), (dict(transition_soc=1.0), "transition_soc"),
                                     (dict(transition_soc=1.5), "transition_soc"), (dict(transition_soc=float("nan")), "transition_soc"),
                                     (dict(up_increment=0.0), "up_increment"), (dict(up_increment=-1.0), "up_increment"),
                                     (dict(down_threshold=-0.5), "down_threshold")])
def test_refused_options(kw, what):
    with pytest.raises(ValueError, match=what):
        _replay(battery=True, estimate_max_rate=True, **kw)


def test_battery_columns_leave_the_ev_table_alone():
    base, bat = _replay(), _replay(battery=True, estimate_max_rate=True)
    for k in ("ev_site", "ev_station", "ev_arr", "ev_dep", "ev_req", "ev_max"):
        np.testing.assert_array_equal(getattr(base, k), getattr(bat, k), err_msg=k)
    assert base.ev_cap is None and base.ev_charge is None and base.ev_ub is None
    assert _replay(estimate_max_rate=True).ev_cap is None and _replay(battery=True).ev_ub is None
    # per site-day, in the table's sorted order: each EV gets synthetic_batteries(seed of its site-day)[its index in the day]
    infra = caltech_acn_infrastructure()
    for s in range(bat.n_sites):
        for d in range(bat.days):
            evs = synthetic_day(infra, 4 + s * 2 + d, 288, 5, 20)
            cap, charge = synthetic_batteries(4 + s * 2 + d, [ev.requested for ev in evs])
            for ev, c, q in zip(evs, cap, charge):
                j = np.nonzero((bat.ev_site == s) & (bat.ev_station == ev.station) & (bat.ev_arr == ev.arrival + 288 * d))[0]
                assert len(j) == 1 and bat.ev_cap[j[0]] == c and bat.ev_charge[j[0]] == q
    np.testing.assert_array_equal(bat.ev_ub, np.asarray(bat.info.max_pilot)[bat.ev_station])


def test_synthetic_batteries():
    req = np.array([r.requested for r in synthetic_day(caltech_acn_infrastructure(), 9, 288, 5, 40)])
    day = synthetic_day(caltech_acn_infrastructure(), 9, 288, 5, 40)
    cap, charge = synthetic_batteries(9, req)
    assert [ev.requested for ev in day] == list(req)  # its own generator: the day's EVs do not move
    soc_f = (charge + req) / cap
    assert (cap >= 30).all() and (cap <= 80).all() and (soc_f >= 0.75 - 1e-12).all() and (soc_f <= 1 + 1e-12).all()
    assert (soc_f > 0.8).mean() > 0.6  # most requests end in the taper
    big = synthetic_batteries(3, [70.0, 5.0])
    assert big[0][0] >= 70.0 and big[1][0] >= -1e-9  # raised to requested / soc_f
    for a, b in zip(synthetic_batteries(9, req), synthetic_batteries(9, req)):
        np.testing.assert_array_equal(a, b)


def test_estimate_caps_the_session_tables(monkeypatch):
    """What acb_preprocess_sessions does with the estimates (min with the EV's maximum, then the minimum rate 0 wins) is
    what the host replay packs, admits with and reallocates with."""
    rp = _replay(battery=True, estimate_max_rate=True)
    t = 130
    h, idx, *_ = rp._pack(t)
    np.testing.assert_array_equal(h["max_rates"][: len(idx)], rp.ev_max[idx].astype(np.float32))  # max_pilot 32 = ev_max: no cut yet
    rp.ev_ub[idx] = np.linspace(-2.0, 40.0, len(idx))
    h, idx, *_ = rp._pack(t)
    want = np.maximum(np.minimum(rp.ev_max[idx], rp.ev_ub[idx]), 0.0)
    np.testing.assert_array_equal(rp._max_rate(idx), want)
    np.testing.assert_array_equal(h["max_rates"][: len(idx)], want.astype(np.float32))
    assert (want == 0).any() and (want == 32).any() and ((want > 0) & (want < 32)).any()
    np.testing.assert_array_equal(_replay()._max_rate(idx), rp.ev_max[idx])


# ---------------------------------------------------------------------------------------------------- the C ABI
def test_fleet_ev_abi():
    """acb_fleet_ev is mirrored field for field; acb_fleet, acb_sessions and acb_batch keep their layouts."""
    body = HDR[HDR.index("typedef struct acb_fleet_ev {"):HDR.index("} acb_fleet_ev;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in re.findall(r"(?:const\s+)?(?:int32_t|float|double)\s*\*?\s*([^;]+);", body):
        names += [re.sub(r"\[.*\]", "", x.strip().lstrip("*").split()[-1].lstrip("*")) for x in decl.split(",")]
    assert names == [n for n, _ in _cabi.FleetEV._fields_], names
    assert C.sizeof(_cabi.FleetEV) == 8 * len(names)
    assert [n for n, _ in _cabi.Fleet._fields_][-1] == "shift" and C.sizeof(_cabi.Fleet) == _cabi.Fleet.shift.offset + C.sizeof(C.c_void_p)
    assert [n for n, _ in _cabi.Sessions._fields_][-1] == "max_rate0"
    assert [n for n, _ in _cabi.Batch._fields_][-1] == "sess_max0"
    for name, params in (("acb_fleet_sessions_ev", ["site", "fleet", "ev", "t", "sessions", "sess_ev", "warm_mu", "stream"]),
                         ("acb_fleet_apply_ev", ["site", "fleet", "ev", "t", "period", "batch", "sess_ev", "first_pilots", "stats", "stream"])):
        assert name in _cabi.EXPORTS
        m = re.search(r"int %s\(([^)]*)\);" % name, HDR)
        assert m, f"{name} is declared"
        assert [p.strip().split()[-1].lstrip("*") for p in m.group(1).split(",")] == params
        assert len(getattr(_cabi.lib(), name).argtypes) == len(params)


def test_monkeypatched_batteries_reach_the_replay(monkeypatch):
    monkeypatch.setattr(replay_fast, "synthetic_batteries", lambda seed, req: (np.full(len(req), 1e9), np.zeros(len(req))))
    rp = _replay(battery=True)
    assert (rp.ev_cap == 1e9).all() and (rp.ev_charge == 0).all()
