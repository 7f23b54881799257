"""Quantised pilots in the batched API and the device fleet replay (acb_quantize_pilots): per instance, bit for bit, what
the drop-in class does with quantize=True [, reallocate=True] (reference adacharge/adacharge.py:177-190): the solve's
float32 schedule in float64, then project_into_discrete_feasible_pilots or diff_based_reallocation, then max(., 0)."""
import ctypes as C

import numpy as np
import pytest
import torch

import adacharge_b200 as ab
from adacharge_b200 import _cabi, engine
from adacharge_b200.batched import BatchedAdaptiveCharging, sessions_to_arrays
from adacharge_b200.generators import caltech_acn_infrastructure, config_c2, config_c5, hierarchical_three_phase_network, session_generator
from oracle import postprocessing as opp
from tests.replay_checks import device_equals_host

pytestmark = pytest.mark.gpu

BENCH_OBJ = [("tou_energy_cost", 1.0, {}), ("total_energy", 0.3, {}), ("demand_charge", 1.0 / 30.0, {})]


def _components(spec):
    return [ab.ObjectiveComponent(getattr(ab, n), c, k) for n, c, k in spec]


def _dropin_post(R, S, I, iface, reallocate, post=ab):
    R = np.asarray(R, dtype=np.float64)
    out = post.diff_based_reallocation(R, S, I, iface) if reallocate else post.project_into_discrete_feasible_pilots(R, I)
    return np.maximum(out, 0)


def _assert_members(pilots, I):
    for i, a in enumerate(I.allowable_pilots):
        assert np.isin(pilots[i], a).all(), (i, np.setdiff1d(pilots[i], a))


def _chunk_rates(bac, b):
    """The float32 schedule of instance b as the batch's solve left it on the device."""
    for ch in bac.chunks:
        if ch.lo <= b < ch.hi:
            return ch.rates[b - ch.lo].cpu().numpy()
    raise IndexError(b)


def _c2_ifaces(n, seed0, infra):
    """C2 instances with every other session arriving now, so that the first-period greedy has work to do."""
    out = []
    for i in range(n):
        d = config_c2(seed0 + i, infra=infra, price_noise=0.2)
        for j, s in enumerate(d["active_sessions"]):
            if j % 2 == 0:
                s["arrival"] = 0
        out.append(ab.TestingInterface(d))
    return out


@pytest.mark.parametrize("reallocate", [False, True], ids=["discrete", "reallocate"])
def test_batched_quantized_equals_dropin(require_gpu, reallocate):
    infra = caltech_acn_infrastructure()
    ifaces = _c2_ifaces(9, 50, infra)
    obj = _components(BENCH_OBJ)
    I = ifaces[0].infrastructure_info()
    sess = sessions_to_arrays([f.active_sessions() for f in ifaces], I, S_max=54)
    prices = np.stack([np.asarray(f.get_prices(288), dtype=float) for f in ifaces])
    prev = np.array([f.get_prev_peak() for f in ifaces])
    bac = BatchedAdaptiveCharging(obj, I, 5, batch=9, max_sessions=54, horizon=288, demand_charge=15.51, chunks=3, quantize=True,
                                  reallocate=reallocate)
    res = bac.schedule(sess, prices=prices, prev_peak=prev)
    assert (res.status == 0).all()
    for b, iface in enumerate(ifaces):
        S = iface.active_sessions()
        aco = ab.AdaptiveChargingOptimization(obj, iface, solver_options=dict(eps_rel=1e-4))
        R = aco.solve(S, I, prev_peak=iface.get_prev_peak())
        T = R.shape[1]
        assert res.T[b] == T
        np.testing.assert_array_equal(res.pilots[b, :, :T], _dropin_post(R, S, I, iface, reallocate), err_msg=f"instance {b}")
        np.testing.assert_array_equal(res.pilots[b, :, :T], _dropin_post(R, S, I, iface, reallocate, post=opp), err_msg=f"oracle, instance {b}")
        assert not res.pilots[b, :, T:].any()
        _assert_members(res.pilots[b, :, :T], I)


def _ragged_infra():
    infra = caltech_acn_infrastructure()
    ap = [np.asarray(a, dtype=float) for a in infra["allowable_pilots"]]
    ap[0] = np.array([6.0, 12.0, 20.0, 32.0])  # no 0: padded zeros must stay zeros
    ap[1] = np.array([0.0, 32.0])
    ap[2] = np.array([0.0, 10.0, 13.0, 16.0, 30.0])
    return dict(infra, allowable_pilots=ap)


def test_batched_reallocation_order_and_edge_cases(require_gpu):
    """Sessions in shuffled slot order (against the drop-in with the same shuffled list); a second, later session on one
    EVSE; an instance without sessions (all-zero pilots); ragged allowable sets, one without 0."""
    infra = _ragged_infra()
    ids = infra["station_ids"]
    rng = np.random.default_rng(5)
    n = 40
    dem = rng.uniform(3, 25, n).tolist()
    base = session_generator(n, [0] * n, rng.integers(30, 150, n).tolist(), dem, dem, [32] * n, station_ids=[ids[i] for i in range(n)])
    perm = rng.permutation(n)
    shuffled = [base[k] for k in perm]
    multi = session_generator(3, [0, 60, 0], [50, 140, 100], [6.0, 8.0, 10.0], [6.0, 8.0, 10.0], [32] * 3, station_ids=[ids[5], ids[5], ids[9]])
    lists = [shuffled, multi, [], base[:25]]
    mk = lambda ss: ab.TestingInterface({"active_sessions": ss, "infrastructure_info": infra, "current_time": 0, "period": 5,  # noqa: E731
                                         "prices": np.full(288, 0.1), "demand_charge": 15.51, "prev_peak": 0.0})
    ifaces = [mk(ss) for ss in lists]
    I = ifaces[0].infrastructure_info()
    sess = sessions_to_arrays([f.active_sessions() for f in ifaces], I, S_max=54)
    obj = _components([("quick_charge", 1.0, {}), ("equal_share", 1e-3, {})])
    bac = BatchedAdaptiveCharging(obj, I, 5, batch=4, max_sessions=54, horizon=288, multi_session=True, chunks=2, quantize=True, reallocate=True)
    res = bac.schedule(sess)
    order_mattered = False
    for b, iface in enumerate(ifaces):
        S = iface.active_sessions()
        T = int(res.T[b])
        assert not res.pilots[b, :, T:].any()
        if not S:
            assert not res.pilots[b].any()
            continue
        R = _chunk_rates(bac, b)[:, :T]
        exp = _dropin_post(R, S, I, iface, True)
        np.testing.assert_array_equal(res.pilots[b, :, :T], exp, err_msg=f"instance {b}")
        np.testing.assert_array_equal(res.pilots[b, :, :T], _dropin_post(R, S, I, iface, True, post=opp), err_msg=f"oracle, instance {b}")
        _assert_members(res.pilots[b, :, :T], I)
        assert (res.pilots[b, 0, :T] >= 6).all()  # the set without 0
        if b == 0:
            unshuffled = mk(base).active_sessions()
            order_mattered = not np.array_equal(exp, _dropin_post(R, unshuffled, I, iface, True))
    print(f"shuffling the sessions changed the reallocated pilots: {order_mattered}")


def test_batched_reallocation_config_c5(require_gpu):
    """1000-EVSE hierarchical site (general solve path): N > 128 in the pairwise sum, several rows per EVSE."""
    infra = hierarchical_three_phase_network(1000)
    ds = [config_c5(seed, infra=infra) for seed in (3, 4, 5)]
    for d in ds:
        for j, s in enumerate(d["active_sessions"]):
            if j % 3 == 0:
                s["arrival"] = 0
    ifaces = [ab.TestingInterface(d) for d in ds]
    I = ifaces[0].infrastructure_info()
    sess = sessions_to_arrays([f.active_sessions() for f in ifaces], I, S_max=1000)
    ext = np.stack([np.asarray(d["external_signal"], dtype=float) for d in ds])
    obj = _components([("load_flattening", 1.0, {}), ("non_completion_penalty", 100.0, {})])
    bac = BatchedAdaptiveCharging(obj, I, 5, batch=3, max_sessions=1000, horizon=288, chunks=1, quantize=True, reallocate=True)
    res = bac.schedule(sess, external_signal=ext)
    for b, iface in enumerate(ifaces):
        S = iface.active_sessions()
        T = int(res.T[b])
        R = _chunk_rates(bac, b)[:, :T]
        np.testing.assert_array_equal(res.pilots[b, :, :T], _dropin_post(R, S, I, iface, True), err_msg=f"instance {b}")
        assert not res.pilots[b, :, T:].any()
        _assert_members(res.pilots[b, :, :T], I)


def test_device_fleet_replay_quantized_equals_host(require_gpu):
    infra = caltech_acn_infrastructure()
    sets = [np.asarray(a, dtype=float) for a in infra["allowable_pilots"]]
    n = dict(infeasible=0)

    def on_step(t, host, dev, first):
        for i, s in enumerate(sets):
            assert np.isin(first[:, i], s).all(), (t, i)
        n["infeasible"] += int((engine.constraints_feasible(host.site, first[:, :, None], 0).cpu().numpy() == 0).sum())

    host, _ = device_equals_host(infra, _components(BENCH_OBJ), list(range(80, 125)) + list(range(288 + 90, 288 + 110)), on_step, n_sites=7,
                                 steps_per_day=288, days=2, seed0=40, mean_sessions=12, Tp=160, quantize=True, reallocate=True)
    assert min(host.stats.active_sites) < 7 < sum(host.stats.active_sites)  # idle sites occurred
    # floor_to_set rounds up to a member within 0.05 A, so the reference's quantised pilots can exceed a limit by that much
    print(f"first columns over a network limit (within floor_to_set's 0.05 A): {n['infeasible']} of {65 * 7}")


def test_quantized_quick_charge_day_delivers_energy(require_gpu):
    from adacharge_b200.replay_fast import DeviceFleetReplay

    obj = _components([("quick_charge", 1.0, {}), ("equal_share", 1e-6, {})])
    rp = DeviceFleetReplay(caltech_acn_infrastructure(), obj, n_sites=4, steps_per_day=288, days=1, seed0=7, mean_sessions=20,
                           quantize=True, reallocate=True)
    stats = rp.run(0, 288)
    assert (stats.delivered_frac >= 0.99).all(), stats.delivered_frac  # t_int.py:162-165


def test_quantize_pilots_rejects_bad_arguments(require_gpu):
    infra = caltech_acn_infrastructure()
    I = ab.TestingInterface({"active_sessions": [], "infrastructure_info": infra, "current_time": 0, "period": 5}).infrastructure_info()
    bac = BatchedAdaptiveCharging(_components(BENCH_OBJ), I, 5, batch=2, max_sessions=54, horizon=288, demand_charge=15.51, chunks=1,
                                  quantize=True, reallocate=True)
    L, ch = _cabi.lib(), bac.chunks[0]
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    pil = engine._ptr(ch.pilots)

    def rc(site=bac.site.handle, mode=_cabi.ACB_PILOTS_REALLOCATE, sessions=ch.sessions, period=5.0, batch=ch.batch, pilots=pil):
        return L.acb_quantize_pilots(site, mode, None if sessions is None else C.byref(sessions), period,
                                     None if batch is None else C.byref(batch), pilots, st)

    other = _cabi.Sessions.from_buffer_copy(ch.sessions)
    other.B = 3
    no_pilots = dict(infra, allowable_pilots=None)
    Ino = ab.TestingInterface({"active_sessions": [], "infrastructure_info": no_pilots, "current_time": 0, "period": 5}).infrastructure_info()
    plain = engine.Site(Ino)
    for bad in (dict(mode=0), dict(mode=3), dict(sessions=other), dict(sessions=None), dict(batch=None), dict(pilots=None),
                dict(period=0.0), dict(site=plain.handle)):
        assert rc(**bad) == -1, bad  # ACB_E_INVALID
    torch.cuda.synchronize()


def test_reallocation_ties_follow_slot_order(require_gpu):
    """Two ClipperCreek EVSEs at 12 A round down to 8 A with the same loss; the peak (24 A) leaves room for one 8 A step,
    which goes to the session in the earlier slot (Python's sorted() is stable).  acb_quantize_pilots is run on this
    hand-made schedule with the two sessions in both orders."""
    infra = caltech_acn_infrastructure()
    ids = infra["station_ids"]
    a, b = ids.index("CA-322"), ids.index("CA-493")  # CC pod: allowable pilots 0, 8, 16, 24, 32
    mk = lambda rows: ab.TestingInterface({  # noqa: E731
        "active_sessions": session_generator(2, [0, 0], [50, 50], [30.0, 30.0], [30.0, 30.0], [32, 32], station_ids=[ids[r] for r in rows]),
        "infrastructure_info": infra, "current_time": 0, "period": 5, "prices": np.full(288, 0.1), "demand_charge": 15.51, "prev_peak": 0.0})
    ifaces = [mk([a, b]), mk([b, a])]
    I = ifaces[0].infrastructure_info()
    sess = sessions_to_arrays([f.active_sessions() for f in ifaces], I, S_max=54)
    bac = BatchedAdaptiveCharging(_components(BENCH_OBJ), I, 5, batch=2, max_sessions=54, horizon=288, demand_charge=15.51, chunks=1,
                                  quantize=True, reallocate=True)
    res = bac.schedule(sess, prices=np.full(288, 0.1))
    ch = bac.chunks[0]
    T = int(res.T[0])
    assert T == 50 and int(res.T[1]) == 50
    R = np.zeros((I.num_stations, T))
    R[[a, b], :] = 12.0
    ch.rates.zero_()
    ch.rates[:, :, :T] = torch.from_numpy(R.astype(np.float32)).to(ch.rates.device)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _cabi.check(_cabi.lib().acb_quantize_pilots(bac.site.handle, _cabi.ACB_PILOTS_REALLOCATE, C.byref(ch.sessions), 5.0, C.byref(ch.batch),
                                                engine._ptr(ch.pilots), st), "acb_quantize_pilots")
    pil = ch.pilots.cpu().numpy()
    first = {0: a, 1: b}
    for k, iface in enumerate(ifaces):
        S = iface.active_sessions()
        np.testing.assert_array_equal(pil[k, :, :T], _dropin_post(R, S, I, iface, True), err_msg=f"instance {k}")
        np.testing.assert_array_equal(pil[k, :, :T], _dropin_post(R, S, I, iface, True, post=opp), err_msg=f"oracle, instance {k}")
        assert pil[k, first[k], 0] == 16.0 and pil[k, a + b - first[k], 0] == 8.0, pil[k, [a, b], 0]
        assert not pil[k, :, T:].any()
