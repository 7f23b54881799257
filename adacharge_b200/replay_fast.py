"""Array-based closed-loop replay of many sites (BASELINE config 4 at scale; SURVEY.md
§8(f) row N1).  Same control step as replay.SiteReplay — the loop body of
AdaptiveSchedulingAlgorithm.schedule (reference adacharge/adacharge.py:135-193) for every
site at once — but the EVs of all sites live in flat numpy arrays and the acb_batch is
packed with array operations, so the host cost per step is O(milliseconds) for a thousand
sites instead of one Python object per session.  The batch always holds every site (idle
sites carry zero sessions), so the warm-start state of step t lines up with step t+1 by
construction; session multipliers follow their EV through a per-EV table on the device.

Sharding: sites are independent, so a rank replays `sharding.shard_range(n_sites, ...)`
of them with no data-path collective; `summary()` returns what `gather_summaries` reduces.
"""
from __future__ import annotations

import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _cabi, engine
from .adaptive_charging_optimization import ObjectiveComponent, pack_objective
from .interface import TestingInterface, infrastructure_from_dict
from .replay import REPLAY_SOLVER_DEFAULTS, synthetic_day


@dataclass
class FleetStats:
    iters_mean: List[float] = field(default_factory=list)
    iters_max: List[int] = field(default_factory=list)
    unsolved: List[int] = field(default_factory=list)      # instances per step whose status != ACB_SOLVED
    active_sites: List[int] = field(default_factory=list)
    host_ms: List[float] = field(default_factory=list)     # packing + bookkeeping on the host
    device_ms: List[float] = field(default_factory=list)   # upload + solve + projection + read-back of the pilots
    delivered_frac: Optional[np.ndarray] = None
    peak_kw: Optional[np.ndarray] = None


class FleetReplay:
    """`n_sites` copies of one site, `days` seeded days of EVs each (day d of site s is
    `synthetic_day(seed0 + s * days + d)` shifted by d * steps_per_day periods).  `quantize` / `reallocate` are
    AdaptiveSchedulingAlgorithm's flags: the EVs are charged with pilots from each EVSE's allowable set."""

    def __init__(self, infra: Dict, objective: List[ObjectiveComponent], n_sites: int, steps_per_day: int = 288, days: int = 1,
                 period: float = 5, prices: Optional[np.ndarray] = None, demand_charge: float = 15.51, seed0: int = 0,
                 warm_start: bool = True, solver_options: Optional[dict] = None, device=None, mean_sessions: int = 40,
                 Tp: int = 288, site_offset: int = 0, quantize: bool = False, reallocate: bool = False):
        self.infra, self.objective, self.n_sites, self.period = infra, objective, n_sites, period
        self.steps_per_day, self.days, self.steps = steps_per_day, days, steps_per_day * days
        self.warm_start, self.device, self.Tp = warm_start, device, Tp
        # closed loop: the sunk demand charge w * prev_peak is a constant of every step's objective and can cancel the
        # energy term, so the gap is taken relative to the terms' magnitude; a stalled instance stops after 40 checks
        self.options = _cabi.default_options(**{**REPLAY_SOLVER_DEFAULTS, **(solver_options or {})})
        from .generators import sce_tou_prices

        day_prices = sce_tou_prices(steps_per_day, period) if prices is None else np.asarray(prices, dtype=float)
        self.prices = np.tile(day_prices[:steps_per_day], days + 1)
        self.demand_charge = demand_charge
        self.volt = np.asarray(infra["voltages"], dtype=float)
        self.N = len(infra["station_ids"])
        self.info = infrastructure_from_dict(infra)
        from .batched import pilot_mode

        self.pilot_mode = pilot_mode(quantize, reallocate, self.info)
        cols = {k: [] for k in ("site", "station", "arr", "dep", "req", "maxrate")}
        for s in range(n_sites):
            for d in range(days):
                seed = seed0 + (site_offset + s) * days + d if days > 1 else seed0 + site_offset + s
                for ev in synthetic_day(infra, seed, steps_per_day, period, mean_sessions):
                    cols["site"].append(s)
                    cols["station"].append(ev.station)
                    cols["arr"].append(ev.arrival + d * steps_per_day)
                    cols["dep"].append(ev.departure + d * steps_per_day)
                    cols["req"].append(ev.requested)
                    cols["maxrate"].append(ev.max_rate)
        # EV table sorted by (day, site, station): a day is a contiguous slice (sessions never span midnight, so step t
        # only looks at its own day) and any active subset of it is grouped by site and ordered by EVSE row
        arr_all = np.array(cols["arr"], dtype=np.int64)
        order = np.lexsort((np.array(cols["station"]), np.array(cols["site"]), arr_all // steps_per_day))
        self.ev_site = np.array(cols["site"], dtype=np.int64)[order]
        self.ev_station = np.array(cols["station"], dtype=np.int64)[order]
        self.ev_arr = arr_all[order]
        self.ev_dep = np.array(cols["dep"], dtype=np.int64)[order]
        self.ev_req = np.array(cols["req"], dtype=np.float64)[order]
        self.ev_max = np.array(cols["maxrate"], dtype=np.float64)[order]
        self.ev_dlv = np.zeros_like(self.ev_req)
        day = self.ev_arr // steps_per_day
        edges = np.searchsorted(day, np.arange(days + 1))
        self._day_slice = [slice(int(edges[d]), int(edges[d + 1])) for d in range(days)]
        self._w_ev = self.volt[self.ev_station] * period / 1e3 / 60  # kWh per A-period of each EV's EVSE
        self.prev_peak = np.zeros(n_sites)  # A
        self.site: Optional[engine.Site] = None
        self._prev = None  # (EV index / site / position of the previous step's sessions, had-sessions mask)
        self._pb: Optional[engine.PackedBatch] = None  # one batch object for the whole replay (refilled every step)
        self._state = None  # two sets of warm-state tensors: a step reads the previous step's set and writes the other
        self.stats = FleetStats()

    # ------------------------------------------------------------------ packing
    def _objective_arrays(self, t: int, T: np.ndarray) -> Dict[str, np.ndarray]:
        """pack_objective once per distinct horizon (quick_charge depends on T), gathered per site.
        The peak baseline follows each site's own previous peak (aco.py:386-400)."""
        Tp, B = self.Tp, self.n_sites
        iface = TestingInterface({"active_sessions": [], "infrastructure_info": self.infra, "current_time": t, "period": self.period,
                                  "prices": self.prices, "demand_charge": self.demand_charge, "prev_peak": 0.0})
        uT, inv = np.unique(T, return_inverse=True)
        tab = {k: np.zeros((len(uT), Tp)) for k in ("alpha", "beta", "ext")}
        sc = {k: np.zeros(len(uT)) for k in ("qd", "gamma", "peak_w", "peak_p0")}
        has_ext = False
        # Most components give the same per-period coefficients whatever the horizon (prices, energy, peak terms);
        # quick_charge does not ((T - t) / T).  Probe the shortest and the longest horizon: if the short one is a
        # prefix of the long one, one evaluation serves every site (cut at its own T); else evaluate per horizon.
        ob_hi = pack_objective(self.objective, self.info, iface, int(uT[-1]))
        ob_lo = pack_objective(self.objective, self.info, iface, int(uT[0])) if len(uT) > 1 else ob_hi
        n0 = int(uT[0])
        prefix_ok = all(np.array_equal(ob_lo[k], ob_hi[k][:n0]) for k in ("alpha", "beta")) and \
            all(ob_lo[k] == ob_hi[k] for k in sc) and \
            ((ob_lo["ext"] is None and ob_hi["ext"] is None) or (ob_lo["ext"] is not None and ob_hi["ext"] is not None and np.array_equal(ob_lo["ext"][:n0], ob_hi["ext"][:n0])))
        if prefix_ok:
            # one coefficient vector for everybody, cut at each site's own horizon
            f32 = np.float32
            live = (np.arange(Tp)[None, :] < T[:, None])
            pad = lambda v: np.pad(np.asarray(v, dtype=f32)[:Tp], (0, max(0, Tp - len(v))))  # noqa: E731
            out = {k: pad(ob_hi[k])[None, :] * live for k in ("alpha", "beta")}
            if ob_hi["ext"] is not None:
                out["ext"] = pad(ob_hi["ext"])[None, :] * live
            for k in ("qd", "gamma", "peak_w"):
                out[k] = np.full(B, ob_hi[k], dtype=f32)
            out["peak_p0"] = np.maximum(self.prev_peak * self.volt[0] / 1000, ob_hi["peak_p0"]).astype(f32)
            return out
        for j, Tj in enumerate(uT):
            ob = ob_hi if j == len(uT) - 1 else (ob_lo if j == 0 else pack_objective(self.objective, self.info, iface, int(Tj)))
            tab["alpha"][j, :Tj], tab["beta"][j, :Tj] = ob["alpha"][:Tj], ob["beta"][:Tj]
            if ob["ext"] is not None:
                tab["ext"][j, :Tj], has_ext = ob["ext"][:Tj], True
            for k in sc:
                sc[k][j] = ob[k]
        f32 = np.float32
        out = {k: tab[k][inv].astype(f32) for k in ("alpha", "beta")}
        if has_ext:
            out["ext"] = tab["ext"][inv].astype(f32)
        for k in ("qd", "gamma", "peak_w"):
            out[k] = sc[k][inv].astype(f32)
        out["peak_p0"] = np.maximum(self.prev_peak * self.volt[0] / 1000, sc["peak_p0"][inv]).astype(f32)
        return out

    def _pack(self, t: int):
        B, S_, i32, f32 = self.n_sites, self.N, np.int32, np.float32
        sl = self._day_slice[min(t // self.steps_per_day, self.days - 1)]
        rem_c = self.ev_req[sl] - self.ev_dlv[sl]
        keep = np.nonzero((self.ev_arr[sl] <= t) & (t < self.ev_dep[sl]) & (rem_c > 1e-6))[0]
        idx, rem = keep + sl.start, rem_c[keep]
        s = self.ev_site[idx]
        n_sess = np.bincount(s, minlength=B)
        offs = np.concatenate(([0], np.cumsum(n_sess)[:-1]))
        pos = np.arange(len(idx)) - offs[s]
        st = self.ev_station[idx]
        ln = self.ev_dep[idx] - t
        T = np.ones(B, dtype=np.int64)  # idle sites: a one-period problem with no sessions
        np.maximum.at(T, s, ln)
        if T.max() > self.Tp:
            raise ValueError(f"a session needs a horizon of {T.max()} periods > Tp = {self.Tp}")
        h = dict(T=T.astype(i32), n_sessions=n_sess.astype(i32))
        flat = s * S_ + pos  # 1-D scatter index into the padded [B, S_max] tables
        for name, vals, dt in (("sess_row", st, i32), ("sess_len", ln, i32),
                               ("sess_energy", rem / self._w_ev[idx], f32),
                               ("sess_rate_off", -(np.arange(len(idx)) + 1), i32)):
            a = np.zeros(B * S_, dtype=dt)
            a[flat] = vals
            h[name] = a.reshape(B, S_)
        h["sess_start"] = np.zeros((B, S_), dtype=i32)
        h["min_rates"] = np.zeros(B * S_, dtype=f32)  # fixed length (one slot per possible session): the staging buffers are reused
        h["max_rates"] = np.zeros(B * S_, dtype=f32)
        h["max_rates"][: len(idx)] = self.ev_max[idx]
        h.update(self._objective_arrays(t, T))
        return h, idx, s, pos, n_sess

    # ------------------------------------------------------------------ one control step
    def step(self, t: int):
        t0 = time.perf_counter()
        h, idx, s, pos, n_sess = self._pack(t)
        if self.site is None:
            use_u = bool((h["gamma"] > 0).any() or (h["peak_w"] > 0).any())
            self.site = engine.get_site(self.info, "SOC", False, use_u, self.device)
        if self._pb is None:
            self._pb = engine.PackedBatch.from_arrays(self.site, h, self.Tp, self.N, multi_session=False)
            self._state = [self._pb.new_warm_state(), self._pb.new_warm_state()]
        else:
            self._pb.refill(h)  # same shapes every step: reuse the pinned staging and the device buffers
        pb = self._pb
        prev, out = self._state
        dev = pb.device
        t1 = time.perf_counter()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        idx_d = torch.from_numpy(idx).to(dev)
        s_d, pos_d = torch.from_numpy(s).to(dev), torch.from_numpy(pos).to(dev)
        if self.warm_start and self._prev is not None:
            pb.set_warm(self._warm(prev, idx_d, s_d, pos_d), out, shift=1, had=self._prev[-1])
        else:
            pb.set_warm(None, out)
        pb.upload().solve(self.options)
        pilots = self._project(pb.rates.to(torch.float64), h, idx, s, pos)
        first = pilots[:, :, 0].contiguous().cpu().numpy()
        it, stt = pb.iters.cpu().numpy(), pb.status.cpu().numpy()
        ev1.record()
        ev1.synchronize()
        t2 = time.perf_counter()
        # the simulator side: first-period pilots charge the EVs that are plugged in
        sl = self._day_slice[min(t // self.steps_per_day, self.days - 1)]
        present = np.nonzero((self.ev_arr[sl] <= t) & (t < self.ev_dep[sl]))[0] + sl.start
        e = np.minimum(first[self.ev_site[present], self.ev_station[present]] * self._w_ev[present], self.ev_req[present] - self.ev_dlv[present])
        self.ev_dlv[present] += np.maximum(e, 0.0)
        self.prev_peak = np.maximum(self.prev_peak, first.sum(axis=1))
        self._prev = (idx_d, s_d, pos_d, torch.from_numpy((n_sess > 0).astype(np.int32)).to(dev))
        self._state.reverse()
        act = n_sess > 0
        st_ = self.stats
        st_.iters_mean.append(float(it[act].mean()) if act.any() else 0.0)
        st_.iters_max.append(int(it[act].max()) if act.any() else 0)
        st_.unsolved.append(int((stt[act] != _cabi.ACB_SOLVED).sum()))
        st_.active_sites.append(int(act.sum()))
        st_.device_ms.append(ev0.elapsed_time(ev1))
        st_.host_ms.append((t1 - t0 + time.perf_counter() - t2) * 1e3)
        return first

    def _project(self, rates, h, idx, s, pos):
        """The pilots of the step's schedule (pp.py:77-118, 189-258 on the device)."""
        if self.pilot_mode:
            pilots = self._project_quantized(rates, h, idx, s, pos)
            pilots[torch.from_numpy(h["n_sessions"] == 0).to(pilots.device)] = 0.0  # idle sites: no pilots (as acb_quantize_pilots)
            return pilots
        return engine.project_continuous(self.site, rates)

    def _project_quantized(self, rates, h, idx, s, pos):
        if self.pilot_mode == _cabi.ACB_PILOTS_REALLOCATE:
            # sessions in slot order (the EV table's), all starting now; ramp = interface.remaining_amp_periods
            B, S_ = h["sess_row"].shape
            ramp, max0 = np.zeros((B, S_)), np.zeros((B, S_))
            rem = self.ev_req[idx] - self.ev_dlv[idx]
            ramp[s, pos] = rem * 1000 / self.volt[self.ev_station[idx]] * (60 / self.period)
            max0[s, pos] = self.ev_max[idx]
            return engine.reallocate(self.site, 1, rates, h["n_sessions"], h["sess_row"], h["sess_start"], ramp, max0)
        return engine.project_discrete(self.site, rates)

    def _warm(self, prev, idx_d, s_d, pos_d):
        """The previous step's state for this step's solve, which reads it one period ahead (sites idle before start
        cold through warm_had); the session multipliers follow their EV."""
        pidx, ps, ppos, _ = self._prev
        mu_ev = torch.zeros(len(self.ev_req), dtype=torch.float32, device=prev["mu"].device)
        mu_ev[pidx] = prev["mu"][ps, ppos]
        mu = torch.zeros_like(prev["mu"])
        mu[s_d, pos_d] = mu_ev[idx_d]
        return dict(prev, mu=mu)

    def run(self, t0: int = 0, t1: Optional[int] = None) -> FleetStats:
        for t in range(t0, self.steps if t1 is None else t1):
            self.step(t)
        req = np.bincount(self.ev_site, weights=self.ev_req, minlength=self.n_sites)
        dlv = np.bincount(self.ev_site, weights=self.ev_dlv, minlength=self.n_sites)
        self.stats.delivered_frac = dlv / np.maximum(req, 1e-9)
        self.stats.peak_kw = self.prev_peak * self.volt[0] / 1000
        return self.stats

    def summary(self) -> Dict[str, float]:
        s = self.stats
        n = max(len(s.device_ms), 1)
        return dict(site_steps=float(sum(s.active_sites)), steps=float(len(s.device_ms)), unsolved=float(sum(s.unsolved)),
                    device_ms=float(sum(s.device_ms)), host_ms=float(sum(s.host_ms)),
                    iters_mean=float(np.average(s.iters_mean, weights=np.maximum(s.active_sites, 1e-9))) if n else 0.0,
                    iters_max=float(max(s.iters_max, default=0)))


class DeviceFleetReplay(FleetReplay):
    """FleetReplay with the simulator side of the control step on the device as well (SURVEY.md §8(f) N1): the EV table,
    the energy delivered, the previous peaks and the per-EV warm-start multipliers stay in device arrays; a step is four
    launches on one stream -- active sessions (acb_fleet_sessions), packing (acb_pack_sessions), the warm-started solve
    whose prologue reads the previous state one column ahead (acb_batch.warm_shift) and whose epilogue projects the
    pilots, and the simulator update (acb_fleet_apply) -- with no host synchronisation between steps.  Quantised pilots
    take a fifth launch (acb_quantize_pilots) between the solve and the update.  Same schedules,
    bit for bit, as FleetReplay (tests/test_gpu_replay.py)."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        import ctypes as C

        from .batched import BatchedAdaptiveCharging

        dev = torch.device("cuda", engine._dev_index(self.device))
        opts = {**REPLAY_SOLVER_DEFAULTS, **(kw.get("solver_options") or {})}
        self._bac = BatchedAdaptiveCharging(self.objective, self.info, self.period, batch=self.n_sites, max_sessions=self.N, horizon=self.Tp,
                                            demand_charge=self.demand_charge, solver_options=opts, device=self.device, chunks=1,
                                            enforce_pilot_limit=False, quantize=self.pilot_mode != 0,
                                            reallocate=self.pilot_mode == _cabi.ACB_PILOTS_REALLOCATE)
        if self._bac.Tp != self.Tp:
            raise ValueError(f"Tp = {self.Tp} is not a padded horizon of the solve path")
        self.site = self._bac.site
        ch = self._bac.chunks[0]
        self._ch = ch
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a.astype(dt))).to(dev)  # noqa: E731
        n_ev = len(self.ev_req)
        self._d = dict(
            station=up(self.ev_station, np.int32), arr=up(self.ev_arr, np.int32), dep=up(self.ev_dep, np.int32), req=up(self.ev_req, np.float64),
            mx=up(self.ev_max, np.float64), dlv=torch.zeros(n_ev, dtype=torch.float64, device=dev), mu=torch.zeros(n_ev, dtype=torch.float32, device=dev),
            prev_peak=torch.zeros(self.n_sites, dtype=torch.float64, device=dev), had=torch.zeros(self.n_sites, dtype=torch.int32, device=dev),
            prices=up(np.concatenate([self.prices, np.zeros(self.Tp)]), np.float64),
            sess_ev=torch.full((self.n_sites, self.N), -1, dtype=torch.int32, device=dev),
            warm_mu=torch.zeros((self.n_sites, self.N), dtype=torch.float32, device=dev),
            first=torch.zeros((self.n_sites, self.N), dtype=torch.float64, device=dev), stats=torch.zeros(3, dtype=torch.float64, device=dev),
        )
        # first EV of every (day, site): the table is sorted by (day, site, station)
        key = (self.ev_arr // self.steps_per_day) * self.n_sites + self.ev_site
        off = np.searchsorted(key, np.arange(self.days * self.n_sites + 1)).astype(np.int32)
        self._d["off"] = torch.from_numpy(off).to(dev)
        f = _cabi.Fleet()
        f.n_sites, f.n_ev, f.days, f.steps_per_day = self.n_sites, n_ev, self.days, self.steps_per_day
        p = engine._ptr
        d = self._d
        f.ev_station, f.ev_arr, f.ev_dep, f.ev_req, f.ev_max = p(d["station"]), p(d["arr"]), p(d["dep"]), p(d["req"]), p(d["mx"])
        f.ev_dlv, f.ev_mu, f.day_site_off, f.prev_peak, f.had = p(d["dlv"]), p(d["mu"]), p(d["off"]), p(d["prev_peak"]), p(d["had"])
        self._fleet = f
        self._state = [ch.new_warm_state(), ch.new_warm_state()]
        ch.lb_zero = True  # the synthetic EVs have no minimum rate
        o = ch.objective
        o.prev_peak = p(d["prev_peak"])
        o.prices_stride = 0  # one price vector for the whole fleet, read from the current period on
        self._started = False
        self._C = C

    def step(self, t: int, want_first: bool = True):
        C, L, ch, d, p = self._C, _cabi.lib(), self._ch, self._d, engine._ptr
        st = C.c_void_p(torch.cuda.current_stream(self._bac.device).cuda_stream)
        o = ch.objective
        prev, out = self._state
        ch.set_warm(dict(prev, mu=d["warm_mu"]) if self.warm_start and self._started else None, out, shift=1, had=d["had"])
        o.prices = C.c_void_p(d["prices"].data_ptr() + 8 * t) if self._bac.need_prices else None
        _cabi.check(L.acb_fleet_sessions(self.site.handle, C.byref(self._fleet), t, C.byref(ch.sessions), p(d["sess_ev"]), p(d["warm_mu"]), st), "acb_fleet_sessions")
        _cabi.check(L.acb_pack_sessions(self.site.handle, C.byref(ch.sessions), C.byref(o), C.byref(ch.struct), p(ch.flags), st), "acb_pack_sessions")
        ch.solve(self._bac.options, st)
        if self.pilot_mode:  # the solve skipped the continuous projection (batch.pilots NULL); acb_fleet_apply reads batch.pilots
            _cabi.check(L.acb_quantize_pilots(self.site.handle, self.pilot_mode, C.byref(ch.sessions), float(self.period), C.byref(ch.struct), p(ch.pilots), st),
                        "acb_quantize_pilots")
            ch.bind_pilots(True)
        _cabi.check(L.acb_fleet_apply(self.site.handle, C.byref(self._fleet), t, float(self.period), C.byref(ch.struct), p(d["sess_ev"]),
                                      p(d["first"]) if want_first else None, p(d["stats"]), st), "acb_fleet_apply")
        if self.pilot_mode:
            ch.bind_pilots(False)
        self._state.reverse()
        self._started = True
        return d["first"].cpu().numpy() if want_first else None

    def run(self, t0: int = 0, t1: Optional[int] = None) -> FleetStats:
        for t in range(t0, self.steps if t1 is None else t1):
            self.step(t, want_first=False)
        torch.cuda.synchronize(self._bac.device)
        if int(self._ch.flags.cpu()[0]) != 0:
            raise ValueError("the device packer flagged the fleet's sessions (two sessions on one EVSE, or a session beyond the padded horizon)")
        self.ev_dlv = self._d["dlv"].cpu().numpy()
        self.prev_peak = self._d["prev_peak"].cpu().numpy()
        req = np.bincount(self.ev_site, weights=self.ev_req, minlength=self.n_sites)
        dlv = np.bincount(self.ev_site, weights=self.ev_dlv, minlength=self.n_sites)
        self.stats.delivered_frac = dlv / np.maximum(req, 1e-9)
        self.stats.peak_kw = self.prev_peak * self.volt[0] / 1000
        return self.stats

    def summary(self) -> Dict[str, float]:
        s = self._d["stats"].cpu().numpy()
        return dict(site_steps=float(s[0]), unsolved=float(s[2]), iters_mean=float(s[1] / max(s[0], 1.0)))
