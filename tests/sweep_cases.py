"""Stratified solver cases: a covering design over what selects a kernel variant of `acb_solve_batch` -- the padded
horizon Tp (on-chip instantiations 64 / 128 / 160 / 288, general path with rows in registers or staged in shared memory
with 8, 7 or 4 warps per block), the site (row warps, electrical groups, column-pass threads per period), the EVSE-row
variant (FAST: lb = 0 and one session per EVSE; register state: positive minimum rates; MULTI: two sessions on one
EVSE; per-period rate limits; energy equality; soft energy rows) -- and the coupling rows / objective terms.

A case is named `<stratum>-s<seed>` and is rebuilt from its name alone (`build(name)`).  Long horizons keep the oracle
affordable with short session windows grouped in a few bursts spread over the horizon: periods outside every window
have zero bounds, so the oracle sees a small problem while the kernels still stride over all of Tp.
tests/golden/make_solver_sweep_golden.py stores the oracle optimum of every case in tests/golden/solver_sweep_golden.json.
"""
import hashlib
import math

import numpy as np

from adacharge_b200.generators import (caltech_acn_infrastructure, hierarchical_three_phase_network, session_generator,
                                       single_phase_single_constraint, three_phase_balanced_network)

PERIOD = 5
KWH_PER_AP = 208 * PERIOD / 1e3 / 60  # kWh per A-period at 208 V

# objective mixes; QUADRATIC: those with a quadratic term (never LP-representable)
OBJECTIVES = {
    "qc": [("quick_charge", 1.0, {})],
    "qc_es": [("quick_charge", 1.0, {}), ("equal_share", 1e-3, {})],
    "bench": [("tou_energy_cost", 1.0, {}), ("total_energy", 0.3, {}), ("demand_charge", 1.0 / 30.0, {})],
    "lf": [("quick_charge", 1.0, {}), ("load_flattening", 1e-3, {})],
    "ncp2": [("tou_energy_cost", 1.0, {}), ("non_completion_penalty", 0.2, {"norm": 2})],
}
QUADRATIC = {"qc_es", "lf", "ncp2"}

# stratum -> (T, site, variant, objective, constraint type, peak limit)
# site: "single<k>" single-phase k EVSEs; "three<p>" three-phase balanced, p EVSEs per phase; "caltech" (54 EVSEs,
# NG + R = 17: two column-pass threads per period); "hier120" (hierarchical, only the general path takes it)
# variant: fast | minrate | multi | ratearr (per-period max_rates) | equality | soft (non_completion_penalty norm 2)
STRATA = {}


def _add(name, T, site, variant, obj, ct="SOC", peak=None):
    STRATA[name] = dict(T=T, site=site, variant=variant, obj=obj, ct=ct, peak=peak)


for _T in (64, 65, 128, 129, 160, 161, 288):
    _add(f"T{_T}_single_fast", _T, "single7", "fast", "qc" if _T % 2 == 0 else "bench", "LINEAR" if _T % 32 else "SOC",
         "scalar" if _T in (64, 129, 161) else ("vector" if _T in (65, 160) else None))
    _add(f"T{_T}_three_minrate", _T, "three4", "minrate", "qc_es")
    _add(f"T{_T}_caltech_{'multi' if _T % 2 == 0 else 'ratearr'}", _T, "caltech", "multi" if _T % 2 == 0 else "ratearr", "bench")
for _T in (64, 160, 288):
    _add(f"T{_T}_three20_lf", _T, "three20", "fast", "lf")   # 60 EVSEs: on chip, 20 row warps, never FAST
    _add(f"T{_T}_hier120", _T, "hier120", "fast", "bench")   # general path only
for _T in (64, 288):
    _add(f"T{_T}_three5_equality", _T, "three5", "equality", "qc")  # groups of 5 rows: partial rows across warps
for _T in (128, 288):
    _add(f"T{_T}_single_soft", _T, "single6", "soft", "ncp2")
_add("T288_three20_minrate", 288, "three20", "minrate", "bench")   # 20 row warps, register state, Tp = 288
_add("T288_caltech_ratearr_es", 288, "caltech", "ratearr", "qc_es")  # time-varying limits (ROWHI = -1) at Tp = 288
# general path only: rows staged in shared memory
_add("T289_single_fast", 289, "single8", "fast", "qc", "LINEAR", "vector")
_add("T300_single300", 300, "single300", "fast", "qc", "LINEAR")    # Tp 320, nw = 8: one group of 300 > 256 rows
_add("T1000_three3_bench", 1000, "three3", "fast", "bench", "LINEAR")  # Tp 1024, nw = 8
_add("T1000_three3_minrate", 1000, "three3", "minrate", "qc_es")
_add("T2000_single6_multi", 2000, "single6", "multi", "bench", "SOC", "scalar")  # Tp 2016, nw = 7
_add("T3616_single140", 3616, "single140", "fast", "qc", "LINEAR")  # Tp 3616 (the limit), nw = 4: one group of 140 > 128 rows
_add("T3616_three2_es", 3616, "three2", "minrate", "qc_es")
# dispatch boundary: three-phase balanced sites with N = 54 .. 72 EVSEs at Tp = 64 and 288
BOUNDARY_N = (54, 57, 60, 63, 66, 69, 72)
for _T in (64, 288):
    for _n in BOUNDARY_N:
        _add(f"boundary_T{_T}_N{_n}", _T, f"three{_n // 3}", "fast", "qc")

SEEDS = {name: (1 if name.startswith("boundary") else 0,) for name in STRATA}
CASES = [f"{s}-s{seed}" for s, seeds in SEEDS.items() for seed in seeds]


def _site(site, concurrent):
    """Infrastructure with limits that bind for about `concurrent` sessions charging at once."""
    if site == "caltech":
        return caltech_acn_infrastructure(transformer_cap=45)
    if site == "hier120":
        return hierarchical_three_phase_network(120, evses_per_pod=10, pods_per_panel=4)
    if site.startswith("single"):
        n = int(site[6:])
        return single_phase_single_constraint(n, 0.6 * 32 * min(n, concurrent))
    p = int(site[5:])
    return three_phase_balanced_network(p, 0.6 * 32 * min(3 * p, concurrent) / 3 * math.sqrt(3))


def n_evses(site):
    if site == "caltech":
        return 54
    if site == "hier120":
        return 120
    return int(site[6:]) if site.startswith("single") else 3 * int(site[5:])


def build(name):
    """The scenario dict of case `name` (the shape tests/scenarios.py uses: data=(sessions, infra), objective,
    constraint_type, equality, peak_limit, iface_extra)."""
    stratum, seed = name.rsplit("-s", 1)
    st = STRATA[stratum]
    T, variant = st["T"], st["variant"]
    rng = np.random.default_rng(_stable_seed(stratum) + int(seed))
    N = n_evses(st["site"])
    # sessions: bursts of overlapping short windows spread over the horizon, the last one ending at T
    n_burst = 1 if T <= 160 else (2 if T <= 300 else 3)
    per_burst = min(N, 12 if N <= 60 else 40) if not stratum.startswith("boundary") else N
    if st["site"] in ("single300", "single140"):
        per_burst = N // n_burst + 1
    wmax = min(T, 24 if T <= 288 else 16)
    stations, arr, dep = [], [], []
    for k in range(n_burst):
        centre = T - wmax if k == n_burst - 1 else int(rng.integers(0, T - 2 * wmax))
        pick = rng.permutation(N)[: min(per_burst, N)]
        for i in pick:
            a = centre + int(rng.integers(0, wmax // 3))
            d = min(T, a + int(rng.integers(wmax // 3, wmax - wmax // 3 + 1)))
            stations.append(int(i)); arr.append(a); dep.append(d)
    dep[-1] = T
    # one session per EVSE unless the variant asks for two: drop later duplicates (bursts may reuse an EVSE)
    seen, keep = {}, []
    for j, (i, a, d) in enumerate(zip(stations, arr, dep)):
        if i in seen and (a < dep[seen[i]] or variant != "multi"):
            if j == len(stations) - 1:  # keep the session that ends at T
                keep = [k for k in keep if stations[k] != i]
            else:
                continue
        seen[i] = j
        keep.append(j)
    stations, arr, dep = [stations[j] for j in keep], [arr[j] for j in keep], [dep[j] for j in keep]
    if variant == "multi" and len(set(stations)) == len(stations):  # make sure some EVSE holds two sessions
        j = int(np.argmin(dep[:-1]))
        if dep[j] + 3 <= T:
            stations.append(stations[j]); arr.append(dep[j]); dep.append(min(T, dep[j] + wmax // 2))
    m = len(stations)
    length = np.array(dep) - np.array(arr)
    deliverable = length * 32 * KWH_PER_AP
    frac = rng.uniform(0.05, 0.3, m) if variant == "equality" else rng.uniform(0.3, 0.9, m)
    energy = frac * deliverable
    mins = None
    maxs = [32.0] * m
    if variant == "minrate":
        mins = [6.0 if rng.random() < 0.6 else 0.0 for _ in range(m)]
        mins[0] = 6.0
        energy = np.maximum(energy, 1.05 * np.array(mins) * length * KWH_PER_AP)
    if variant == "ratearr":
        maxs = [np.where(rng.random(int(ln)) < 0.3, 16.0, 32.0) for ln in length]
    if variant == "soft":
        energy = rng.uniform(0.6, 1.4, m) * deliverable  # some requests exceed what the window can deliver
    ids = [str(s) if st["site"] != "caltech" and st["site"] != "hier120" else None for s in stations]
    infra = _site(st["site"], per_burst)
    if ids[0] is None:
        ids = [infra["station_ids"][s] for s in stations]
    sessions = session_generator(m, [int(a) for a in arr], [int(d) for d in dep], energy.tolist(), energy.tolist(), maxs,
                                 min_rates=mins, station_ids=ids)
    obj = [(n, c, dict(k)) for n, c, k in OBJECTIVES[st["obj"]]]
    if st["obj"] == "lf":
        obj[1][2]["external_signal"] = (20 + 10 * np.sin(np.arange(T) / 5.0)).tolist()
    sc = dict(data=(sessions, infra), objective=obj, constraint_type=st["ct"], equality=variant == "equality",
              iface_extra=dict(prices=(0.05 + 0.25 * rng.random(T + 4)).tolist(), demand_charge=15.51,
                               prev_peak=float(rng.choice([0.25, 0.5]) * 32 * per_burst)))  # A: a demand charge partly sunk
    if st["peak"] is not None:
        cap = 0.5 * 32 * per_burst
        sc["peak_limit"] = float(cap) if st["peak"] == "scalar" else np.linspace(cap, 0.7 * cap, T)
    return sc


def _stable_seed(s):
    return int(hashlib.sha256(s.encode()).hexdigest()[:8], 16)


def lp_representable(name):
    st = STRATA[name.rsplit("-s", 1)[0]]
    return st["obj"] not in QUADRATIC and (st["ct"] == "LINEAR" or st["site"].startswith("single"))


def strictly_convex(name):
    return STRATA[name.rsplit("-s", 1)[0]]["obj"] == "qc_es"


def strata(name):
    """What the case is meant to exercise: padded horizon, staged-row warps of the general path (0 = rows in registers),
    whether the on-chip FAST variant applies (lb_zero, one session per EVSE, ceil(N / 3) <= 18 row warps), the variant."""
    from adacharge_b200.engine import SUPPORTED_HORIZONS, padded_horizon

    sc = build(name)
    st = STRATA[name.rsplit("-s", 1)[0]]
    sessions, infra = sc["data"]
    Tp = padded_horizon(max(s["departure"] for s in sessions))
    N = len(infra["station_ids"])
    lb_zero = all(np.all(np.asarray(s["min_rates"]) == 0) for s in sessions)
    multi = len({s["station_id"] for s in sessions}) < len(sessions)
    nw = 0 if Tp in SUPPORTED_HORIZONS else min(8, 232448 // (16 * Tp))
    return dict(Tp=Tp, staged_nw=nw, fast=bool(lb_zero and not multi and -(-N // 3) <= 18), lb_zero=bool(lb_zero),
                multi=bool(multi), N=N, variant=st["variant"])


def instance_hash(sc):
    """sha256 over every array the oracle and the packer read (sessions, infrastructure, objective, prices, limits)."""
    h = hashlib.sha256()
    sessions, infra = sc["data"]

    def put(x):
        h.update(np.ascontiguousarray(np.asarray(x, dtype=np.float64)).tobytes())

    for s in sessions:
        h.update(str(s["station_id"]).encode())
        put([s["arrival"], s["departure"], s["requested_energy"], s["energy_delivered"]])
        put(np.atleast_1d(s["min_rates"])); put(np.atleast_1d(s["max_rates"]))
    for k in ("constraint_matrix", "constraint_limits", "phases", "voltages"):
        put(infra[k])
    h.update(repr([(n, c) for n, c, _ in sc["objective"]]).encode())
    for _, _, kw in sc["objective"]:
        for k in sorted(kw):
            put(kw[k])
    put(sc["iface_extra"]["prices"]); put([sc["iface_extra"]["prev_peak"], sc["iface_extra"]["demand_charge"]])
    h.update(f"{sc['constraint_type']}|{sc['equality']}".encode())
    if "peak_limit" in sc:
        put(np.atleast_1d(sc["peak_limit"]))
    return h.hexdigest()
