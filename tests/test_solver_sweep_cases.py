"""CPU checks of the stratified solver cases (tests/sweep_cases.py) and their golden file: the generator is
deterministic, every case lands in the stratum the golden file lists, the oracle reproduces the stored optima, and the
padded horizon stops at the general path's limit."""
import json
import os
import sys

import numpy as np
import pytest

from adacharge_b200 import engine
from oracle import mpc
from tests import sweep_cases as sw
from tests.scenarios import make_interface

GOLDEN_DIR = os.path.join(os.path.dirname(__file__), "golden")
with open(os.path.join(GOLDEN_DIR, "solver_sweep_golden.json")) as _f:
    GOLDEN = json.load(_f)["cases"]


def test_padded_horizon_limit():
    assert engine.padded_horizon(3616) == 3616 == engine.MAX_HORIZON
    assert engine.padded_horizon(3585) == 3616
    with pytest.raises(ValueError):
        engine.padded_horizon(3617)


def test_golden_file_lists_every_case():
    assert sorted(GOLDEN) == sorted(sw.CASES)
    assert 40 <= len(sw.CASES) <= 60


def test_generator_is_deterministic_and_matches_the_golden_hashes():
    sys.path.insert(0, GOLDEN_DIR)
    from make_solver_sweep_golden import check

    assert check() == []
    name = sw.CASES[0]
    assert sw.instance_hash(sw.build(name)) == sw.instance_hash(sw.build(name))


@pytest.mark.parametrize("name", sw.CASES)
def test_strata_assignment(name):
    """Padded horizon, staged-row warps and FAST eligibility (lb_zero, one session per EVSE, ceil(N / 3) <= 18)."""
    st, g = sw.strata(name), GOLDEN[name]["strata"]
    assert st == g
    T = sw.STRATA[name.rsplit("-s", 1)[0]]["T"]
    assert st["Tp"] == engine.padded_horizon(T)
    if st["Tp"] in engine.SUPPORTED_HORIZONS:
        assert st["staged_nw"] == 0
    else:
        assert st["staged_nw"] == min(8, 232448 // (16 * st["Tp"]))
    assert st["fast"] == (st["lb_zero"] and not st["multi"] and -(-st["N"] // 3) <= 18)


def test_strata_cover_the_plan():
    """Staged warps 8, 7 and 4 (Tp 320, 1024, 2016, 3616); every on-chip horizon with FAST, register-state and MULTI
    cases; sites of 55 .. 66 EVSEs; every row variant."""
    st = [GOLDEN[n]["strata"] for n in sw.CASES]
    assert {s["staged_nw"] for s in st} == {0, 8, 7, 4}
    assert {s["Tp"] for s in st} == {64, 128, 160, 288, 320, 1024, 2016, 3616}
    for Tp in engine.SUPPORTED_HORIZONS:
        on = [s for s in st if s["Tp"] == Tp]
        assert any(s["fast"] for s in on) and any(s["multi"] for s in on) and any(not s["lb_zero"] for s in on), Tp
    assert any(55 <= s["N"] <= 66 and s["Tp"] == Tp for s in st for Tp in (64, 160, 288))
    assert {s["variant"] for s in st} == {"fast", "minrate", "multi", "ratearr", "equality", "soft"}


def _cheapest(k):
    return sorted(sw.CASES, key=lambda n: GOLDEN[n]["seconds"])[:k]


@pytest.mark.parametrize("name", _cheapest(3))
def test_oracle_reproduces_the_stored_objective(name):
    g = GOLDEN[name]
    sc = sw.build(name)
    iface = make_interface(sc)
    S, I = iface.active_sessions(), iface.infrastructure_info()
    ct, eq, pl, pp = sc["constraint_type"], sc["equality"], sc.get("peak_limit"), iface.get_prev_peak()
    if g["method"] == "highs":
        _, f = mpc.solve_lp_highs(sc["objective"], S, I, iface, ct, eq, pl, pp)
    else:
        R = mpc.solve_mpc(sc["objective"], S, I, iface, ct, eq, pl, pp, tol_scale=1e-4 if sw.strictly_convex(name) else 1.0)
        f = mpc.evaluate_objective(R, sc["objective"], I, iface, S, pp)
    assert abs(f - g["objective"]) <= 1e-9 * max(abs(g["objective"]), 1e-12) + 1e-12, (f, g["objective"])
