"""Host-side rules of uninterrupted charging (no GPU): the C ABI fields and entry point, the flag rules of the batched
API and the fleet replay, and the arrival column of sessions_to_arrays."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import adacharge_b200 as ab
from adacharge_b200 import _cabi
from adacharge_b200.batched import BatchedAdaptiveCharging, pilot_mode, sessions_to_arrays
from adacharge_b200.generators import caltech_acn_infrastructure, config_c2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = open(os.path.join(ROOT, "include", "adacharge_b200.h")).read()


def test_new_struct_fields_are_appended():
    """The first-period fields come last in acb_sessions and acb_batch, so the offsets of every older field stay."""
    assert [n for n, _ in _cabi.Sessions._fields_][-3:] == ["arrival", "min_rate0", "max_rate0"]
    assert [n for n, _ in _cabi.Batch._fields_][-2:] == ["sess_min0", "sess_max0"]
    assert _cabi.Batch.stats.offset < _cabi.Batch.sess_min0.offset < _cabi.Batch.sess_max0.offset
    assert _cabi.Sessions.max_rate.offset < _cabi.Sessions.arrival.offset
    assert C.sizeof(_cabi.Batch) == _cabi.Batch.sess_max0.offset + C.sizeof(C.c_void_p)


def test_admit_sessions_entry_point_matches_the_header():
    assert "acb_admit_sessions" in _cabi.EXPORTS
    m = re.search(r"int acb_admit_sessions\(([^)]*)\);", HDR)
    assert m, "acb_admit_sessions is declared"
    params = [p.strip() for p in m.group(1).split(",")]
    assert [p.split()[-1].lstrip("*") for p in params] == ["site", "sessions", "min_pilot", "override", "period", "skip_unabsorbable", "stream"]


def test_sessions_to_arrays_fills_arrival():
    d = config_c2(3)
    iface = ab.TestingInterface(d)
    S = iface.active_sessions()
    out = sessions_to_arrays([S, S[:4]], iface.infrastructure_info(), S_max=54)
    assert out["arrival"].dtype == np.int32 and out["arrival"].shape == (2, 54)
    np.testing.assert_array_equal(out["arrival"][0, : len(S)], [s.arrival for s in S])
    np.testing.assert_array_equal(out["arrival"][1, :4], [s.arrival for s in S[:4]])
    assert not out["arrival"][1, 4:].any()


def test_missing_arrival_is_refused():
    """With uninterrupted_charging, schedule() needs the absolute arrivals (the admission's order)."""
    bac = BatchedAdaptiveCharging.__new__(BatchedAdaptiveCharging)
    bac.uninterrupted_charging = True
    sess = sessions_to_arrays([ab.TestingInterface(config_c2(4)).active_sessions()],
                              ab.TestingInterface(config_c2(4)).infrastructure_info())
    bac._check_arrays(sess)
    del sess["arrival"]
    with pytest.raises(ValueError, match="arrival"):
        bac._check_arrays(sess)
    bac.uninterrupted_charging = False
    bac._check_arrays(sess)


@pytest.mark.parametrize("quantize,reallocate,ok", [(False, False, True), (True, False, True), (True, True, True), (False, True, False)])
def test_flag_combinations(quantize, reallocate, ok):
    """uninterrupted_charging combines with every pilot mode the reference allows (reallocate needs quantize)."""
    I = ab.TestingInterface(config_c2(1)).infrastructure_info()
    if ok:
        assert pilot_mode(quantize, reallocate, I) in (0, _cabi.ACB_PILOTS_DISCRETE, _cabi.ACB_PILOTS_REALLOCATE)
    else:
        with pytest.raises(ValueError):
            pilot_mode(quantize, reallocate, I)
    if ok:
        assert ab.AdaptiveSchedulingAlgorithm([ab.ObjectiveComponent(ab.quick_charge)], uninterrupted_charging=True, quantize=quantize,
                                              reallocate=reallocate).uninterrupted_charging


def test_fleet_replay_try_rates_and_kernel_variant():
    """The fleet replay offers min(min_pilot, period) and, when any try rate is positive, does not declare lb_zero."""
    from adacharge_b200.replay_fast import FleetReplay

    infra = caltech_acn_infrastructure()
    obj = [ab.ObjectiveComponent(ab.total_energy)]
    on = FleetReplay(infra, obj, n_sites=2, steps_per_day=288, days=1, seed0=1, mean_sessions=5, uninterrupted_charging=True)
    off = FleetReplay(infra, obj, n_sites=2, steps_per_day=288, days=1, seed0=1, mean_sessions=5)
    np.testing.assert_array_equal(on.try_rate, np.minimum(np.asarray(infra["min_pilot"], dtype=float), 5.0))
    assert (on.try_rate > 0).all() and not on.lb_zero and off.lb_zero
    no_min = dict(infra, min_pilot=np.zeros(len(infra["station_ids"])))
    assert FleetReplay(no_min, obj, n_sites=1, steps_per_day=288, seed0=1, mean_sessions=3, uninterrupted_charging=True).lb_zero
