"""Host-side rules of event-driven recompute (no GPU): the max_recompute flag of the fleet replays, the appended C ABI
fields, and the replays' numpy re-solve rule against a literal per-step loop over generator days."""
import ctypes as C
import os
import re
import warnings

import numpy as np
import pytest

import adacharge_b200 as ab
from adacharge_b200 import _cabi
from adacharge_b200.generators import caltech_acn_infrastructure
from adacharge_b200.replay import synthetic_day
from adacharge_b200.replay_fast import FleetReplay

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = open(os.path.join(ROOT, "include", "adacharge_b200.h")).read()
OBJ = [ab.ObjectiveComponent(ab.total_energy)]


def _replay(**kw):
    return FleetReplay(caltech_acn_infrastructure(), OBJ, **{**dict(n_sites=2, steps_per_day=288, days=1, seed0=1, mean_sessions=5), **kw})


@pytest.mark.parametrize("value", [None, 1, 3, np.int64(12)])
def test_accepted_values(value):
    assert _replay(max_recompute=value).max_recompute == value
    assert _replay().max_recompute == 1  # the default stays 1 (every step), not the reference's None


@pytest.mark.parametrize("value", [0, -1, 2.5, True, "3"])
def test_refused_values(value):
    with pytest.raises(ValueError, match="max_recompute"):
        _replay(max_recompute=value)


def test_quantize_overrides_to_1():
    with pytest.warns(UserWarning, match="Overriding max_recompute to 1 since quantization is on."):
        assert _replay(quantize=True, max_recompute=None).max_recompute == 1
    with pytest.warns(UserWarning, match="Overriding max_recompute to 1"):
        assert _replay(quantize=True, reallocate=True, max_recompute=5).max_recompute == 1
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        assert _replay(quantize=True).max_recompute == 1  # the default asks for nothing else: no warning
    # the drop-in class keeps the reference's rule (its default is None): any value given warns
    with pytest.warns(UserWarning, match="Overriding max_recompute"):
        assert ab.AdaptiveSchedulingAlgorithm(OBJ, quantize=True, max_recompute=1).max_recompute == 1
    assert ab.AdaptiveSchedulingAlgorithm(OBJ, max_recompute=7).max_recompute == 7


def test_abi_additions():
    """acb_batch keeps its layout: the solve mask and the per-instance warm shifts are arguments of the new entry points.
    The recompute fields are appended to acb_fleet, so the offsets of every older field stay."""
    assert [n for n, _ in _cabi.Batch._fields_][-2:] == ["sess_min0", "sess_max0"]
    assert C.sizeof(_cabi.Batch) == _cabi.Batch.sess_max0.offset + C.sizeof(C.c_void_p)
    assert [n for n, _ in _cabi.Fleet._fields_][-5:] == ["had", "max_recompute", "last_solve", "recompute", "shift"]
    assert _cabi.Fleet.had.offset < _cabi.Fleet.max_recompute.offset < _cabi.Fleet.last_solve.offset
    assert C.sizeof(_cabi.Fleet) == _cabi.Fleet.shift.offset + C.sizeof(C.c_void_p)
    for name, params in (("acb_solve_batch_masked", ["site", "batch", "solve_mask", "warm_shifts", "opt", "stream"]),
                         ("acb_quantize_pilots_masked", ["site", "mode", "sessions", "period", "batch", "solve_mask", "pilots", "stream"])):
        assert name in _cabi.EXPORTS
        m = re.search(r"int %s\(([^)]*)\);" % name, HDR)
        assert m, f"{name} is declared"
        assert [p.strip().split()[-1].lstrip("*") for p in m.group(1).split(",")] == params
        assert len(getattr(_cabi.lib(), name).argtypes) == len(params)


def _literal(evs_by_site, steps, mr):
    """The re-solve rule written out per site and step: no solve yet, an EV plugs in or unplugs now, or mr steps since
    the last solve.  Returns the decisions [steps, sites]."""
    out = np.zeros((steps, len(evs_by_site)), dtype=bool)
    for b, evs in enumerate(evs_by_site):
        last = -1
        for t in range(steps):
            event = any(a == t or d == t for a, d in evs)
            if last < 0 or event or (mr is not None and t - last >= mr):
                out[t, b] = True
                last = t
    return out


@pytest.mark.parametrize("mr", [None, 1, 3, 12])
def test_numpy_rule_equals_literal_loop(mr):
    """Two days of generator EVs per site (day d shifted by d * steps_per_day, so unplugs at midnight belong to the day
    before): FleetReplay._recompute, driven as the replay drives it, against the literal loop."""
    rp = _replay(n_sites=6, days=2, seed0=21, mean_sessions=30, max_recompute=mr)
    evs = [[(int(a), int(d)) for a, d, s in zip(rp.ev_arr, rp.ev_dep, rp.ev_site) if s == b] for b in range(rp.n_sites)]
    want = _literal(evs, rp.steps, mr)
    for t in range(rp.steps):
        rec, since = rp._recompute(t)
        np.testing.assert_array_equal(rec, want[t], err_msg=f"step {t}")
        np.testing.assert_array_equal(since, t - rp.last_solve)
        rp.last_solve[rec] = t


def test_midnight_unplug_is_an_event():
    """An EV of day 0 unplugging at t = steps_per_day is in day 0's slice of the EV table, not day 1's."""
    rp = _replay(n_sites=1, days=2, max_recompute=None)
    day0 = np.nonzero(rp.ev_arr < 288)[0]
    assert len(day0) and not (rp.ev_arr == 288).any()
    rp.last_solve[:] = 200
    rp.ev_dep[day0] = 287
    assert not rp._recompute(288)[0][0]
    rp.ev_dep[day0[-1]] = 288
    assert rp._recompute(288)[0][0]


def test_solves_per_site_day():
    """The C4 generator (Caltech site, 40 mean sessions, seeds 0-255, one site-day each), every plugged-in EV treated as
    still owing energy: solves of a site with EVs per site-day under each rule."""
    infra = caltech_acn_infrastructure()
    days = [synthetic_day(infra, s, 288, 5, 40) for s in range(256)]
    rp = _replay(n_sites=256, seed0=0, mean_sessions=40)
    got = {}
    for mr in (1, 3, 12, None):
        rp.max_recompute = mr
        rp.last_solve[:] = -1
        n = 0
        for t in range(288):
            rec, _ = rp._recompute(t)
            plugged = np.bincount(rp.ev_site[(rp.ev_arr <= t) & (t < rp.ev_dep)], minlength=256) > 0
            n += int((rec & plugged).sum())
            rp.last_solve[rec] = t
        got[mr] = n / 256
    assert len(rp.ev_arr) == sum(len(d) for d in days)
    assert {k: round(v) for k, v in got.items()} == {1: 166, 3: 83, 12: 62, None: 61}, got
