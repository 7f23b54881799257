"""Event-driven recompute (max_recompute) on the GPU.

- The solver ABI (acb_solve_batch_masked's solve_mask / warm_shifts) on both solve paths: masked-in instances are bit-identical to the
  batch solved without a mask, masked-out instances keep every output and carry their warm state forward unshifted,
  and per-instance warm shifts equal the scalar warm_shift instance by instance.
- The fleet replays: the device replay equals the host replay bit for bit with max_recompute None and 3, and
  max_recompute = 1 forced onto the event-driven path equals the default every-step path.
- The semantics on a hand-built site: the solve steps, and the applied pilot as column t - t_last of the last schedule.
- Warm starts from states several columns old against a cold float64 oracle solve.
"""
import numpy as np
import pytest
import torch

import adacharge_b200 as ab
from adacharge_b200 import _cabi, engine, replay_fast
from adacharge_b200.generators import caltech_acn_infrastructure, three_phase_balanced_network
from adacharge_b200.interface import SessionInfo
from adacharge_b200.replay import EV
from adacharge_b200.replay_fast import DeviceFleetReplay, FleetReplay
from tests.replay_checks import BENCH, assert_as_good_as_cold_oracle, device_equals_host

pytestmark = pytest.mark.gpu
SENT_F, SENT_I = -7.25, 77


# ---------------------------------------------------------------------------------------------------- the solver ABI
def _batch(B, t=110, quadratic=False):
    """A fleet step of B Caltech sites (t) and the state of the step before it (t - 1) to warm-start from."""
    obj = BENCH + ([ab.ObjectiveComponent(ab.equal_share, 1e-3)] if quadratic else [])
    rp = FleetReplay(caltech_acn_infrastructure(), obj, n_sites=B, steps_per_day=288, days=1, seed0=3, mean_sessions=20, Tp=288)
    h0, h1 = rp._pack(t - 1)[0], rp._pack(t)[0]
    site = engine.get_site(rp.info, "SOC", False, True, None)
    pb = engine.PackedBatch.from_arrays(site, h0, 288, rp.N)
    db = engine.DeviceBatch(site, pb.packed, 288, rp.N, lb_zero=pb.lb_zero, pilots=True, rate_est=True)
    warm = db.new_warm_state()
    pb.upload()
    db.set_warm(None, warm)
    db.solve(rp.options)
    pb.refill(h1).upload()
    torch.cuda.synchronize()
    return rp, db, warm


def _solve(db, opts, warm, shift=1, shifts=None, mask=None):
    """Solve with every output (out_* included) filled with a sentinel first; returns the outputs as numpy."""
    out = db.new_warm_state()
    for t in [db.rates, db.pilots, db.rate_est, db.stats] + list(out.values()):
        t.fill_(SENT_F)
    db.status.fill_(SENT_I)
    db.iters.fill_(SENT_I)
    dev = db.device
    i32 = lambda a: None if a is None else torch.as_tensor(np.asarray(a, dtype=np.int32), device=dev)  # noqa: E731
    db.set_warm(warm, out, shift=shift, shifts=i32(shifts), mask=i32(mask))
    db.solve(opts)
    torch.cuda.synchronize()
    r = dict(rates=db.rates, pilots=db.pilots, rate_est=db.rate_est, status=db.status, iters=db.iters, stats=db.stats)
    r.update({"out_" + k: v for k, v in out.items()})
    return {k: v.cpu().numpy().copy() for k, v in r.items()}


def _variants():
    # (B, lb_zero, path, quadratic): on-chip FAST and non-FAST, a phased launch (B > 148 SMs), the general path
    return {"fast": (24, True, 1, True), "nonfast": (24, False, 1, False), "phased": (300, True, 1, False), "general": (24, True, 2, False)}


@pytest.mark.parametrize("variant", list(_variants()))
def test_solve_mask(require_gpu, variant):
    B, lbz, path, quad = _variants()[variant]
    rp, db, warm = _batch(B, quadratic=quad)
    db.lb_zero = lbz and db.lb_zero
    opts = _cabi.copy_options(rp.options, path=path, phase_iters=100)  # (a phased launch when B > 148 SMs)
    ref = _solve(db, opts, warm)
    assert (ref["status"] == 0).sum() >= B // 2, np.bincount(ref["status"])
    mask = np.random.default_rng(B).integers(0, 2, B)
    mask[:2] = (1, 0)
    got = _solve(db, opts, warm, mask=mask)
    w = {k: v.cpu().numpy() for k, v in warm.items()}
    on, off = mask == 1, mask == 0
    for k in ref:
        assert np.array_equal(got[k][on], ref[k][on]), f"{variant}: masked-in {k} differs at {np.nonzero(on)[0][[not np.array_equal(x, y) for x, y in zip(got[k][on], ref[k][on])]]}"
        if k.startswith("out_"):
            assert np.array_equal(got[k][off], w[k[4:]][off]), f"{variant}: masked-out {k} is not its warm state"
        else:
            assert (got[k][off] == (SENT_I if k in ("status", "iters") else SENT_F)).all(), f"{variant}: masked-out {k} was written"
    none = _solve(db, opts, warm, mask=np.zeros(B))
    for k in none:
        if k.startswith("out_"):
            assert np.array_equal(none[k], w[k[4:]])
        else:
            assert (none[k] == (SENT_I if k in ("status", "iters") else SENT_F)).all(), f"{variant}: an all-zero mask wrote {k}"


@pytest.mark.parametrize("path", [1, 2])
def test_per_instance_warm_shifts(require_gpu, path):
    shifts_of = [0, 1, 2, 5, 287, 288, 295]  # 0, 1, 2, 5, Tp - 1, Tp, Tp + 7
    rp, db, warm = _batch(21)
    opts = _cabi.copy_options(rp.options, path=path)
    shifts = np.array([shifts_of[b % len(shifts_of)] for b in range(21)])
    got = _solve(db, opts, warm, shift=1, shifts=shifts)
    for k_shift in shifts_of:
        ref = _solve(db, opts, warm, shift=k_shift)
        sel = shifts == k_shift
        for k in ref:
            assert np.array_equal(got[k][sel], ref[k][sel]), f"path {path}, shift {k_shift}: {k} differs"


# ---------------------------------------------------------------------------------------------------- the replays
@pytest.mark.parametrize("max_recompute", [None, 3])
@pytest.mark.parametrize("uninterrupted", [False, True])
def test_device_replay_equals_host_replay(require_gpu, max_recompute, uninterrupted):
    host, _ = device_equals_host(caltech_acn_infrastructure(), BENCH, list(range(60, 150)) + list(range(288 + 80, 288 + 110)), n_sites=7,
                                 steps_per_day=288, days=2, seed0=40, mean_sessions=12, Tp=160, max_recompute=max_recompute,
                                 uninterrupted_charging=uninterrupted)
    st = host.stats
    assert min(st.active_sites) < 7  # idle sites occurred
    assert sum(st.solved_sites) < sum(st.active_sites)  # sites skipped steps


@pytest.mark.parametrize("cls", [FleetReplay, DeviceFleetReplay])
def test_max_recompute_1_on_the_event_path_equals_the_default(require_gpu, cls):
    """At max_recompute = 1 (the default) every site re-solves every step and the replays leave last_solve, solve_mask and
    warm_shifts unbound.  The event-driven path forced at 1 (the re-solve decision made every step, the mask and the
    per-site shifts bound, column t - last_solve applied) gives the same pilots, energy and peaks bit for bit."""
    infra = caltech_acn_infrastructure()
    kw = dict(n_sites=5, steps_per_day=288, days=1, seed0=7, mean_sessions=10, Tp=160)
    a, b = cls(infra, BENCH, **kw), cls(infra, BENCH, max_recompute=1, **kw)
    b._event_driven = True
    if cls is DeviceFleetReplay:
        f, d = b._fleet, b._d
        f.last_solve, f.recompute, f.shift = (engine._ptr(d[k]) for k in ("last_solve", "recompute", "shift"))
    for t in range(90, 130):
        np.testing.assert_array_equal(a.step(t), b.step(t), err_msg=f"step {t}")
        assert b.state()["recompute"].all()
        if cls is DeviceFleetReplay:  # (each site's warm shift is not part of the state)
            assert (b._d["shift"].cpu().numpy() == (91 if t == 90 else 1)).all()
    sa, sb = a.state(), b.state()
    for k in ("ev_dlv", "prev_peak"):
        np.testing.assert_array_equal(sa[k], sb[k], err_msg=k)


# ---------------------------------------------------------------------------------------------------- semantics
def _site_of(evs, monkeypatch, **kw):
    monkeypatch.setattr(replay_fast, "synthetic_day", lambda *a, **k: [EV(**e) for e in evs])
    infra = caltech_acn_infrastructure()
    base = dict(n_sites=1, steps_per_day=288, days=1, seed0=0, Tp=160)
    return infra, {**base, **kw}


EVS = [dict(station=3, session_id="a", arrival=10, departure=30, requested=4.0),
       dict(station=7, session_id="b", arrival=20, departure=70, requested=9.0),
       dict(station=11, session_id="c", arrival=250, departure=280, requested=2.0)]


@pytest.mark.parametrize("max_recompute,expect", [
    (None, [0, 10, 20, 30, 70, 250, 280]),
    (4, [0, 4, 8, 10, 14, 18, 20, 24, 28, 30, 34, 38, 42, 46, 50, 54, 58, 62, 66, 70] + list(range(74, 250, 4)) + [250, 254, 258, 262,
                                                                                                               266, 270, 274, 278, 280, 284]),
])
def test_solve_steps_and_applied_columns(require_gpu, monkeypatch, max_recompute, expect):
    infra, kw = _site_of(EVS, monkeypatch, max_recompute=max_recompute)
    dev, host = DeviceFleetReplay(infra, BENCH, **kw), FleetReplay(infra, BENCH, **kw)
    solved, sched, t_last, long_idle = [], None, None, False
    for t in range(288):
        first = dev.step(t)
        np.testing.assert_array_equal(first, host.step(t), err_msg=f"step {t}")
        if dev.state()["recompute"][0]:
            solved.append(t)
            sched, t_last = dev._ch.pilots[0].cpu().numpy().copy(), t
        c = t - t_last
        want = sched[:, c] if c < dev.Tp else np.zeros(dev.N)
        np.testing.assert_array_equal(first[0], want, err_msg=f"step {t}: column {c} of the schedule solved at {t_last}")
        long_idle |= c >= dev.Tp
    assert solved == expect
    assert long_idle == (max_recompute is None)  # 30 -> 70 -> 250: more than Tp = 160 steps without a solve
    dlv = dev.state()["ev_dlv"]
    np.testing.assert_array_equal(dlv, host.state()["ev_dlv"])
    assert dlv[:2].min() > 0


# ---------------------------------------------------------------------------------------------------- warm starts
def test_old_warm_starts_match_a_cold_oracle_solve(require_gpu):
    """Solves warm-started from a state two or more columns old (max_recompute None) are ordinary MPC instances: the
    schedule is as good as a cold float64 oracle solve of the same step."""
    spec = [("tou_energy_cost", 1, {}), ("total_energy", 0.3, {}), ("demand_charge", 1 / 30, {})]
    obj = [ab.ObjectiveComponent(getattr(ab, n), c, k) for n, c, k in spec]
    infra = three_phase_balanced_network(3, 30)
    rp = FleetReplay(infra, obj, n_sites=4, steps_per_day=96, days=1, period=15, seed0=5, mean_sessions=7, Tp=128, max_recompute=None)
    cases = []
    for t in range(96):
        rec, since = rp._recompute(t)
        _, idx, s, _, n_sess = rp._pack(t)
        had, peak = rp.had.copy(), rp.prev_peak.copy()
        sess = {b: [SessionInfo(infra["station_ids"][rp.ev_station[e]], str(e), rp.ev_req[e], rp.ev_dlv[e], int(rp.ev_arr[e]),
                                   int(rp.ev_dep[e]), current_time=t, max_rates=rp.ev_max[e]) for e in idx[s == b]] for b in range(rp.n_sites)}
        rp.step(t)
        R = rp._pb.rates.cpu().numpy().astype(np.float64)
        st = rp.state()["status"]
        for b in range(rp.n_sites):
            if rec[b] and since[b] >= 2 and had[b] and n_sess[b] > 0:
                T = max(x.arrival_offset + x.remaining_time for x in sess[b])
                cases.append((t, b, sess[b], float(peak[b]), R[b][:, :T], int(st[b])))
    compared, skipped, worst = assert_as_good_as_cold_oracle(cases, spec, infra, 15, rp.prices, rp.demand_charge)
    assert compared >= 20 and skipped <= 3, (len(cases), compared, skipped)
    print(f"{compared} solves warm-started from states >= 2 columns old compared, worst objective error {worst:.1e} of the term scale")
