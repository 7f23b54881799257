"""Oracle optima of the stratified solver cases (tests/sweep_cases.py).

    python tests/golden/make_solver_sweep_golden.py [--procs 6]      # writes tests/golden/solver_sweep_golden.json
    python tests/golden/make_solver_sweep_golden.py --check          # re-derives the instance hashes and strata only

Every case is solved on the CPU: LP-representable cases (no quadratic term; LINEAR rows or single-phase SOC rows) by
HiGHS (oracle/mpc.py:solve_lp_highs), the others by the float64 interior point (oracle/mpc.py:solve_mpc).  Strictly
convex cases (quick_charge + 1e-3 equal_share: unique optimum) are solved at tol_scale = 1e-4 and also store their
rates, as make_golden.py does.  Per case: the oracle objective, the sum of the magnitudes of its terms (for the
cancelling-terms rule), a sha256 of the generated instance's arrays and what the case is meant to exercise (padded
horizon, staged-row warps, FAST eligibility).  The GPU test (tests/test_gpu_solver_sweep.py) then compares with these
numbers and pays no oracle solve.  Wall time: 9 s with 6 processes on an 8-core x86 host (no case takes more than
about a second: the windows are short).
"""
import argparse
import json
import multiprocessing as mp
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden", "solver_sweep_golden.json")


def one(name):
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"
    import numpy as np

    from oracle import mpc
    from tests import sweep_cases as sw
    from tests.scenarios import make_interface

    t0 = time.perf_counter()
    sc = sw.build(name)
    iface = make_interface(sc)
    S, I = iface.active_sessions(), iface.infrastructure_info()
    st = sw.strata(name)
    assert mpc.horizon(S) == sw.STRATA[name.rsplit("-s", 1)[0]]["T"], name
    ct, eq, pl, pp = sc["constraint_type"], sc["equality"], sc.get("peak_limit"), iface.get_prev_peak()
    rates = None
    if sw.lp_representable(name):
        R, f = mpc.solve_lp_highs(sc["objective"], S, I, iface, ct, eq, pl, pp)
        method = "highs"
    else:
        strict = sw.strictly_convex(name)
        R = mpc.solve_mpc(sc["objective"], S, I, iface, ct, eq, pl, pp, tol_scale=1e-4 if strict else 1.0)
        f = mpc.evaluate_objective(R, sc["objective"], I, iface, S, pp)
        method = "ipm"
        if strict and st["Tp"] <= 288:
            rates = np.round(R, 9).tolist()
    mag = sum(abs(mpc.evaluate_objective(R, [o], I, iface, S, pp)) for o in sc["objective"])
    v = mpc.violations(R, S, I, iface, ct, pl, eq)
    return dict(name=name, hash=sw.instance_hash(sc), strata=st, method=method, objective=float(f), term_magnitude=float(mag),
                n_sessions=len(S), oracle_violation=float(max(v["infrastructure_rel"], v.get("peak_rel", 0.0), 0.0)),
                rates=rates, seconds=round(time.perf_counter() - t0, 2))


def check(path=OUT):
    """Hashes and strata of the generator against the golden file: a list of mismatching case names."""
    from tests import sweep_cases as sw

    with open(path) as f:
        g = json.load(f)
    bad = [n for n in sw.CASES if n not in g["cases"]]
    for n, e in g["cases"].items():
        if n not in sw.CASES or e["hash"] != sw.instance_hash(sw.build(n)) or e["strata"] != sw.strata(n):
            bad.append(n)
    return bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--procs", type=int, default=max(1, (os.cpu_count() or 2)))
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--out", default=OUT)
    a = ap.parse_args()
    if a.check:
        bad = check(a.out)
        print("ok" if not bad else f"mismatch: {bad}")
        sys.exit(1 if bad else 0)
    from tests import sweep_cases as sw

    t = time.perf_counter()
    with mp.get_context("spawn").Pool(a.procs) as pool:
        rows = pool.map(one, sorted(sw.CASES, key=lambda n: -sw.STRATA[n.rsplit("-s", 1)[0]]["T"]), chunksize=1)
    out = dict(generator="tests/sweep_cases.py", wall_seconds=round(time.perf_counter() - t, 1), procs=a.procs,
               cases={r["name"]: r for r in sorted(rows, key=lambda r: sw.CASES.index(r["name"]))})
    with open(a.out, "w") as f:
        json.dump(out, f, indent=0)
    print(f"{len(rows)} cases in {out['wall_seconds']:.0f} s -> {a.out}")
    for r in sorted(rows, key=lambda r: -r["seconds"])[:5]:
        print(f"  {r['name']}: {r['seconds']} s ({r['method']})")


if __name__ == "__main__":
    main()
