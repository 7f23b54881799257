"""CPU-only: the quantize / reallocate rules of the batched API and the fleet replay, which are checked before any device
work (reference adacharge/adacharge.py:101-105)."""
import numpy as np
import pytest

import adacharge_b200 as ab
from adacharge_b200 import _cabi
from adacharge_b200.batched import BatchedAdaptiveCharging, pilot_mode
from adacharge_b200.generators import caltech_acn_infrastructure
from adacharge_b200.replay_fast import FleetReplay

OBJ = [ab.ObjectiveComponent(ab.quick_charge)]


def _info(infra):
    return ab.TestingInterface({"active_sessions": [], "infrastructure_info": infra, "current_time": 0, "period": 5}).infrastructure_info()


def test_pilot_mode_follows_the_reference_flags():
    I = _info(caltech_acn_infrastructure())
    assert pilot_mode(False, False, I) == 0
    assert pilot_mode(True, False, I) == _cabi.ACB_PILOTS_DISCRETE
    assert pilot_mode(True, True, I) == _cabi.ACB_PILOTS_REALLOCATE


@pytest.mark.parametrize("make", ["batched", "fleet"])
def test_reallocate_without_quantize_raises(make):
    infra = caltech_acn_infrastructure()
    with pytest.raises(ValueError, match="reallocate cannot be true without quantize"):
        if make == "batched":
            BatchedAdaptiveCharging(OBJ, infra, 5, batch=2, max_sessions=54, horizon=288, reallocate=True)
        else:
            FleetReplay(infra, OBJ, n_sites=2, reallocate=True)


@pytest.mark.parametrize("make", ["batched", "fleet"])
def test_quantize_needs_allowable_pilots(make):
    infra = caltech_acn_infrastructure()
    ap = list(infra["allowable_pilots"])
    ap[3] = None
    for bad in (dict(infra, allowable_pilots=None), dict(infra, allowable_pilots=ap)):
        with pytest.raises(ValueError, match="allowable_pilots"):
            if make == "batched":
                BatchedAdaptiveCharging(OBJ, bad, 5, batch=2, max_sessions=54, horizon=288, quantize=True)
            else:
                FleetReplay(bad, OBJ, n_sites=2, quantize=True)
