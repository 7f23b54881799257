"""Array-based closed-loop replay of many sites (BASELINE config 4 at scale; SURVEY.md
§8(f) row N1).  Same control step as replay.SiteReplay — the loop body of
AdaptiveSchedulingAlgorithm.schedule (reference adacharge/adacharge.py:135-193) for every
site at once — but the EVs of all sites live in flat numpy arrays and the acb_batch is
packed with array operations, so the host cost per step is O(milliseconds) for a thousand
sites instead of one Python object per session.  The batch always holds every site (idle
sites carry zero sessions), so the warm-start state of a site lines up with its next solve by
construction; session multipliers follow their EV through a per-EV table on the device.

`max_recompute` is the Simulator's re-solve rule (DESIGN.md §8): a site re-solves at a plug-in or
unplug there and after `max_recompute` steps without one (None: at events only; 1, the default:
every step); in between each EVSE gets the next column of the site's last schedule.  The solve
(acb_solve_batch_masked) skips the other sites (solve_mask) and warm-starts each site from its own
last solve (warm_shifts).

`battery` gives every EV a two-stage battery (`battery_current`: acnportal's Linear2StageBattery without noise, in
amperes) that takes less than its pilot near full charge; `estimate_max_rate` is AdaptiveSchedulingAlgorithm's flag with
acnportal's SimpleRampdown estimator (`rampdown_update`), whose per-EV bound caps the session's maximum rate at every
solve (DESIGN.md §8 states both rules).

Sharding: sites are independent, so a rank replays `sharding.shard_range(n_sites, ...)`
of them with no data-path collective; `summary()` returns what `gather_summaries` reduces.
"""
from __future__ import annotations

import ctypes as C
import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _cabi, engine
from .adacharge import quantized_max_recompute
from .adaptive_charging_optimization import ObjectiveComponent, pack_objective
from .interface import TestingInterface, infrastructure_from_dict
from .replay import REPLAY_SOLVER_DEFAULTS, synthetic_batteries, synthetic_day


def battery_current(p, w, amax, cap, charge, owed, transition_soc):
    """One step of two-stage batteries, element-wise (what acb_fleet_apply_ev computes, bit for bit): the current a (A)
    each battery takes under pilot p on an EVSE of w kWh per A-period, and the energy de (kWh) it receives.
      a = 0 if p == 0; else min(p, amax) below transition_soc and min(p, (1 - soc) / (1 - transition_soc) * amax) from it
      on (soc = charge / cap), cut to (cap - charge) / w where charge + a * w would pass cap, and at least 0;
      de = max(min(a * w, owed), 0)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        soc = charge / cap
        lim = np.where(soc < transition_soc, amax, ((1.0 - soc) / (1.0 - transition_soc)) * amax)
        a = np.where(lim < p, lim, p)
        a = np.where(charge + a * w > cap, (cap - charge) / w, a)
    a = np.where(p == 0.0, 0.0, np.where(a > 0.0, a, 0.0))
    de = a * w
    de = np.where(owed < de, owed, de)
    return a, np.where(de > 0.0, de, 0.0)


def rampdown_update(ub, p, a, up_increment, down_threshold):
    """acnportal's SimpleRampdown after one applied step, element-wise: where the EV took more than down_threshold below
    its pilot its bound becomes a + up_increment, elsewhere it stays.  Returns (new bounds, where it fired)."""
    fire = (p - a) > down_threshold
    return np.where(fire, a + up_increment, ub), fire


@dataclass
class FleetStats:
    iters_mean: List[float] = field(default_factory=list)
    iters_max: List[int] = field(default_factory=list)
    unsolved: List[int] = field(default_factory=list)      # solves per step whose status != ACB_SOLVED
    active_sites: List[int] = field(default_factory=list)  # sites per step with sessions
    solved_sites: List[int] = field(default_factory=list)  # ... of which re-solved this step (the others applied their last schedule)
    host_ms: List[float] = field(default_factory=list)     # packing + bookkeeping on the host
    device_ms: List[float] = field(default_factory=list)   # upload + solve + projection + read-back of the pilots
    delivered_frac: Optional[np.ndarray] = None
    peak_kw: Optional[np.ndarray] = None


class _FleetReplayBase:
    """`n_sites` copies of one site, `days` seeded days of EVs each (day d of site s is
    `synthetic_day(seed0 + s * days + d)` shifted by d * steps_per_day periods).  `quantize` / `reallocate` are
    AdaptiveSchedulingAlgorithm's flags: the EVs are charged with pilots from each EVSE's allowable set.
    `uninterrupted_charging` is its flag too (acnportal's apply_minimum_charging_rate with override = period): each step
    the EVs of a site are offered min(min_pilot, period) as their first-period minimum in arrival order while the network
    stays feasible.  An EV whose remaining energy is less than one period at that rate is not offered it (the
    reference would make the whole site's problem infeasible until that EV leaves).
    `max_recompute` is AdaptiveSchedulingAlgorithm's kwarg as acnportal's Simulator reads it: a site re-solves when an EV
    plugs in or unplugs there or `max_recompute` steps after its last solve (None: at events only); in between its EVSEs
    get the next column of its last schedule.  The default 1 re-solves every site every step (the reference's default is
    None); with `quantize` it is 1, with the reference's warning if anything else was asked for.
    `battery`: every EV has a two-stage battery (`synthetic_batteries` of its site-day: `ev_cap`, `ev_charge`) that takes
    the current `battery_current` gives under its pilot, tapering from `transition_soc` on; the site's peak is the sum of
    those currents.  `rates` holds each EVSE's current of the last step.  `estimate_max_rate`: each EV keeps acnportal's
    SimpleRampdown estimate `ev_ub` (from its EVSE's max_pilot; `rampdown_update` with `up_increment` and
    `down_threshold`), and every solve caps the session's maximum rate at it (apply_upper_bound_estimate).  Without
    `battery` every EV takes its pilot and the estimate never moves.  Both replays take `step(t, want_first=True)` (it
    returns the applied first-period pilots [n_sites, N]) and `state()`.  FleetReplay advances `ev_dlv`, `prev_peak`,
    `ev_charge`, `ev_ub` and `rates` in place; DeviceFleetReplay copies them back at `state()` (`rates`: at want_first)."""

    def __init__(self, infra: Dict, objective: List[ObjectiveComponent], n_sites: int, steps_per_day: int = 288, days: int = 1,
                 period: float = 5, prices: Optional[np.ndarray] = None, demand_charge: float = 15.51, seed0: int = 0,
                 warm_start: bool = True, solver_options: Optional[dict] = None, device=None, mean_sessions: int = 40,
                 Tp: int = 288, site_offset: int = 0, quantize: bool = False, reallocate: bool = False,
                 uninterrupted_charging: bool = False, max_recompute: Optional[int] = 1, battery: bool = False,
                 transition_soc: float = 0.8, estimate_max_rate: bool = False, up_increment: float = 1.0, down_threshold: float = 1.0):
        if not 0.0 < transition_soc < 1.0:
            raise ValueError(f"transition_soc must be in (0, 1), not {transition_soc!r}")
        if not up_increment > 0.0:
            raise ValueError(f"up_increment must be > 0, not {up_increment!r}")
        if not down_threshold >= 0.0:
            raise ValueError(f"down_threshold must be >= 0, not {down_threshold!r}")
        self.battery, self.transition_soc = bool(battery), float(transition_soc)
        self.estimate_max_rate, self.up_increment, self.down_threshold = bool(estimate_max_rate), float(up_increment), float(down_threshold)
        if max_recompute is not None and not (isinstance(max_recompute, (int, np.integer)) and not isinstance(max_recompute, bool)
                                              and max_recompute >= 1):
            raise ValueError(f"max_recompute must be None or an integer >= 1, not {max_recompute!r}")
        self.max_recompute = quantized_max_recompute(max_recompute, quantize, default=1)
        # at 1 every site re-solves every step: the solve then needs neither the mask nor per-site warm shifts
        self._event_driven = self.max_recompute != 1
        self.infra, self.objective, self.n_sites, self.period = infra, objective, n_sites, period
        self.steps_per_day, self.days, self.steps = steps_per_day, days, steps_per_day * days
        self.warm_start, self.device, self.Tp = warm_start, device, Tp
        # closed loop: the sunk demand charge w * prev_peak is a constant of every step's objective and can cancel the
        # energy term, so the gap is taken relative to the terms' magnitude; a stalled instance stops after 40 checks
        self.solver_options = {**REPLAY_SOLVER_DEFAULTS, **(solver_options or {})}
        from .generators import sce_tou_prices

        day_prices = sce_tou_prices(steps_per_day, period) if prices is None else np.asarray(prices, dtype=float)
        self.prices = np.tile(day_prices[:steps_per_day], days + 1)
        self.demand_charge = demand_charge
        self.volt = np.asarray(infra["voltages"], dtype=float)
        self.N = len(infra["station_ids"])
        self.info = infrastructure_from_dict(infra)
        from .batched import pilot_mode

        self.pilot_mode = pilot_mode(quantize, reallocate, self.info)
        self.uninterrupted_charging = bool(uninterrupted_charging)
        self.try_rate = np.array([min(self.info.min_pilot[i], period) for i in range(self.N)], dtype=np.float64)
        # an admitted EV's first-period minimum is its EVSE's try rate: the lb_zero promise holds only if every try is 0
        self.lb_zero = not (self.uninterrupted_charging and bool(np.any(self.try_rate > 0)))
        cols = {k: [] for k in ("site", "station", "arr", "dep", "req", "maxrate", "cap", "charge")}
        for s in range(n_sites):
            for d in range(days):
                seed = seed0 + (site_offset + s) * days + d if days > 1 else seed0 + site_offset + s
                evs = synthetic_day(infra, seed, steps_per_day, period, mean_sessions)
                for ev in evs:
                    cols["site"].append(s)
                    cols["station"].append(ev.station)
                    cols["arr"].append(ev.arrival + d * steps_per_day)
                    cols["dep"].append(ev.departure + d * steps_per_day)
                    cols["req"].append(ev.requested)
                    cols["maxrate"].append(ev.max_rate)
                if self.battery:
                    cap, charge = synthetic_batteries(seed, [ev.requested for ev in evs])
                    cols["cap"] += list(cap)
                    cols["charge"] += list(charge)
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
        # batteries (kWh) and the rampdown estimate (A) per EV, None without
        self.ev_cap = np.array(cols["cap"], dtype=np.float64)[order] if self.battery else None
        self.ev_charge = np.array(cols["charge"], dtype=np.float64)[order] if self.battery else None
        self.ev_ub = np.asarray(self.info.max_pilot, dtype=np.float64)[self.ev_station] if self.estimate_max_rate else None
        self.ev_dlv = np.zeros_like(self.ev_req)
        self.prev_peak = np.zeros(n_sites)  # A
        self.rates: Optional[np.ndarray] = None  # each EVSE's current at the last step [n_sites, N] (the pilots without batteries)
        day = self.ev_arr // steps_per_day
        edges = np.searchsorted(day, np.arange(days + 1))
        self._day_slice = [slice(int(edges[d]), int(edges[d + 1])) for d in range(days)]
        self._w_ev = self.volt[self.ev_station] * period / 1e3 / 60  # kWh per A-period of each EV's EVSE
        self.stats = FleetStats()

    def run(self, t0: int = 0, t1: Optional[int] = None) -> FleetStats:
        for t in range(t0, self.steps if t1 is None else t1):
            self.step(t, want_first=False)
        s = self.state()
        req = np.bincount(self.ev_site, weights=self.ev_req, minlength=self.n_sites)
        dlv = np.bincount(self.ev_site, weights=s["ev_dlv"], minlength=self.n_sites)
        self.stats.delivered_frac = dlv / np.maximum(req, 1e-9)
        self.stats.peak_kw = s["prev_peak"] * self.volt[0] / 1000
        return self.stats


class FleetReplay(_FleetReplayBase):
    """The simulator side of the step on the host, in numpy: the reference DeviceFleetReplay is checked against."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        B = self.n_sites
        self.options = _cabi.default_options(**self.solver_options)
        self.last_solve = np.full(B, -1, dtype=np.int64)  # step of each site's last solve
        self.had = np.zeros(B, dtype=np.int32)  # 1 if the site had sessions at its last solve
        self.recompute = np.zeros(B, dtype=bool)  # the last step's re-solve decision per site
        self.site: Optional[engine.Site] = None
        self._prev = None  # EV index / site / position of the previous step's sessions
        self._sched: Optional[torch.Tensor] = None  # each site's pilots from its last solve [B, N, Tp]
        self._pb: Optional[engine.PackedBatch] = None  # one batch object for the whole replay (refilled every step)
        self._state = None  # two sets of warm-state tensors: a step reads the previous step's set and writes the other

    def state(self) -> Dict[str, Optional[np.ndarray]]:
        """The simulator state as numpy copies, the same keys on both replays: `ev_dlv` (kWh per EV), `prev_peak` (A per
        site), `recompute` (bool per site: re-solved at the last step), `status` (per site, of its last solve; None
        before the first step), `ev_charge` (with battery), `ev_ub` (with estimate_max_rate), `rates` (with either)."""
        live = dict(ev_dlv=self.ev_dlv, prev_peak=self.prev_peak, recompute=self.recompute, ev_charge=self.ev_charge, ev_ub=self.ev_ub,
                    rates=self.rates if self.battery or self.estimate_max_rate else None)
        return dict({k: None if v is None else v.copy() for k, v in live.items()}, status=None if self._pb is None else self._pb.status.cpu().numpy())

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
        h["max_rates"][: len(idx)] = self._max_rate(idx)
        h.update(self._objective_arrays(t, T))
        return h, idx, s, pos, n_sess

    def _max_rate(self, idx):
        """The maximum rate of the EVs idx as the solve sees it: their own, with estimate_max_rate cut to the estimate and
        then raised to the minimum rate 0 where it fell below (what acb_preprocess_sessions does with the upper bounds)."""
        if self.ev_ub is None:
            return self.ev_max[idx]
        ub, mx = self.ev_ub[idx], self.ev_max[idx]
        m = np.where(ub < mx, ub, mx)
        return np.where(m < 0.0, 0.0, m)

    def _admit(self, h, idx, s, pos):
        """apply_minimum_charging_rate of every site (what acb_admit_sessions does on the device): the greedy over the
        sessions in (arrival, slot) order, minus those that cannot absorb one period at their try rate, and the
        resulting first-period limits in the packed tables (sess_min0 / sess_max0)."""
        B, S_ = self.n_sites, self.N
        order = np.lexsort((pos, self.ev_arr[idx], s))  # by site, then arrival, then slot
        st, rem, flat = self.ev_station[idx], self.ev_req[idx] - self.ev_dlv[idx], s * S_ + pos
        tr = self.try_rate[st]
        ramp = rem * 1000 / self.volt[st] * (60 / self.period)  # interface.remaining_amp_periods
        cand = order[ramp[order] >= tr[order]]
        n_c = np.bincount(s[cand], minlength=B)
        c_pos = np.arange(len(cand)) - np.concatenate(([0], np.cumsum(n_c)[:-1]))[s[cand]]
        rows, tries = np.zeros((B, S_), dtype=np.int32), np.zeros((B, S_))
        rows[s[cand], c_pos], tries[s[cand], c_pos] = st[cand], tr[cand]
        adm = engine.min_rate_admission(self.site, n_c, rows, tries)[s[cand], c_pos]
        mn0, mx0 = np.zeros(len(idx)), self._max_rate(idx).copy()  # sessions left out keep their own limits (0, max rate)
        lo = np.where(0.0 < tr[cand], tr[cand], 0.0)  # max(try, min_rates[0])
        mn0[cand] = np.where(adm, lo, 0.0)
        mx0[cand] = np.where(adm, np.where(mx0[cand] < lo, lo, mx0[cand]), 0.0)
        for name, v in (("sess_min0", mn0), ("sess_max0", np.minimum(mx0, 3.0e38))):
            a = np.zeros(B * S_, dtype=np.float32)
            a[flat] = v
            h[name] = a.reshape(B, S_)
        # position of each session in its site's arrival-ordered list, as the device admission leaves the raw tables
        # (the reallocation's tie order), and its max_rates[0]
        n_s = np.bincount(s, minlength=B)
        self._arr_order = np.empty_like(pos)
        self._arr_order[order] = np.arange(len(order)) - np.concatenate(([0], np.cumsum(n_s)[:-1]))[s[order]]
        self._max0, self._limits0 = mx0, (mn0, mx0)

    def _recompute(self, t: int):
        """Which sites re-solve at step t (what acb_fleet_sessions decides on the device), and each site's t - last_solve:
        no solve yet, an EV plugs in or unplugs there now, or max_recompute steps since the last solve."""
        spd, ev = self.steps_per_day, np.zeros(self.n_sites, dtype=bool)
        d = t // spd
        slices = [self._day_slice[min(d, self.days - 1)]]
        if t % spd == 0 and 1 <= d <= self.days:
            slices.append(self._day_slice[d - 1])  # a previous-day EV unplugging at midnight
        for sl in slices:
            ev[self.ev_site[sl][(self.ev_arr[sl] == t) | (self.ev_dep[sl] == t)]] = True
        since = t - self.last_solve
        mr = self.max_recompute or 0
        return (self.last_solve < 0) | ev | ((mr > 0) & (since >= mr)), since

    # ------------------------------------------------------------------ one control step
    def step(self, t: int, want_first: bool = True):
        t0 = time.perf_counter()
        rec, since = self._recompute(t)
        h, idx, s, pos, n_sess = self._pack(t)
        if self.site is None:
            use_u = bool((h["gamma"] > 0).any() or (h["peak_w"] > 0).any())
            self.site = engine.get_site(self.info, "SOC", False, use_u, self.device)
        self._arr_order = None
        if self.uninterrupted_charging:
            self._admit(h, idx, s, pos)
        if self._pb is None:
            self._pb = engine.PackedBatch.from_arrays(self.site, h, self.Tp, self.N, multi_session=False)
            self._state = [self._pb.new_warm_state(), self._pb.new_warm_state()]
        else:
            self._pb.refill(h)  # same shapes every step: reuse the pinned staging and the device buffers
        pb = self._pb
        pb.lb_zero = pb.lb_zero and self.lb_zero
        prev, out = self._state
        dev = pb.device
        t1 = time.perf_counter()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        idx_d = torch.from_numpy(idx).to(dev)
        s_d, pos_d = torch.from_numpy(s).to(dev), torch.from_numpy(pos).to(dev)
        i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)  # noqa: E731
        rec_d, shift_d = i32(rec), i32(since)
        ev = self._event_driven
        if self.warm_start and self._prev is not None:
            pb.set_warm(self._warm(prev, idx_d, s_d, pos_d), out, shift=1, had=i32(self.had), shifts=shift_d if ev else None,
                        mask=rec_d if ev else None)
        else:
            pb.set_warm(None, out, mask=rec_d if ev else None)
        pb.upload().solve(self.options)
        pilots = self._project(pb.rates.to(torch.float64), h, idx, s, pos)
        # the sites that re-solved take their new schedule's column 0, the others column t - last_solve of their last one
        # (0 from Tp on)
        if self._sched is None:
            self._sched = pilots.clone()
        else:
            self._sched[rec_d.bool()] = pilots[rec_d.bool()]
        self.last_solve[rec] = t
        self.had[rec] = n_sess[rec] > 0
        col = t - self.last_solve
        B = self.n_sites
        first_d = self._sched.gather(2, i32(np.minimum(col, self.Tp - 1)).long().view(B, 1, 1).expand(B, self.N, 1)).squeeze(2)
        first_d[torch.from_numpy(col >= self.Tp).to(dev)] = 0.0
        first = first_d.cpu().numpy()
        it, stt = pb.iters.cpu().numpy(), pb.status.cpu().numpy()
        ev1.record()
        ev1.synchronize()
        t2 = time.perf_counter()
        # the simulator side: first-period pilots charge the EVs that are plugged in
        sl = self._day_slice[min(t // self.steps_per_day, self.days - 1)]
        present = np.nonzero((self.ev_arr[sl] <= t) & (t < self.ev_dep[sl]))[0] + sl.start
        if self.battery or self.estimate_max_rate:
            at = (self.ev_site[present], self.ev_station[present])
            p, w, owed = first[at], self._w_ev[present], self.ev_req[present] - self.ev_dlv[present]
            if self.battery:
                a, e = battery_current(p, w, self.ev_max[present], self.ev_cap[present], self.ev_charge[present], owed, self.transition_soc)
                self.ev_charge[present] += e
            else:
                a, e = p, np.maximum(np.minimum(p * w, owed), 0.0)
            self.ev_dlv[present] += e
            if self.estimate_max_rate:
                self.ev_ub[present] = rampdown_update(self.ev_ub[present], p, a, self.up_increment, self.down_threshold)[0]
            self.rates = np.zeros_like(first)
            self.rates[at] = a
        else:
            e = np.minimum(first[self.ev_site[present], self.ev_station[present]] * self._w_ev[present], self.ev_req[present] - self.ev_dlv[present])
            self.ev_dlv[present] += np.maximum(e, 0.0)
            self.rates = first
        # the site's peak: of the currents the batteries took (acb_fleet_apply_ev sums `rates` with ev_cap), else of the pilots
        self.prev_peak = np.maximum(self.prev_peak, (self.rates if self.battery else first).sum(axis=1))
        self._prev = (idx_d, s_d, pos_d)
        self._state.reverse()
        self.recompute = rec
        act = n_sess > 0
        sol = act & rec
        st_ = self.stats
        st_.iters_mean.append(float(it[sol].mean()) if sol.any() else 0.0)
        st_.iters_max.append(int(it[sol].max()) if sol.any() else 0)
        st_.unsolved.append(int((stt[sol] != _cabi.ACB_SOLVED).sum()))
        st_.active_sites.append(int(act.sum()))
        st_.solved_sites.append(int(sol.sum()))
        st_.device_ms.append(ev0.elapsed_time(ev1))
        st_.host_ms.append((t1 - t0 + time.perf_counter() - t2) * 1e3)
        return first if want_first else None

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
            rows = h["sess_row"]
            if self._arr_order is not None:  # uninterrupted charging: arrival order and max_rates[0] from the admission
                pos, mx = self._arr_order, self._max0
                rows = np.zeros((B, S_), dtype=np.int32)
                rows[s, pos] = self.ev_station[idx]
            else:
                mx = self._max_rate(idx)
            ramp[s, pos] = rem * 1000 / self.volt[self.ev_station[idx]] * (60 / self.period)
            max0[s, pos] = mx
            return engine.reallocate(self.site, 1, rates, h["n_sessions"], rows, h["sess_start"], ramp, max0)
        return engine.project_discrete(self.site, rates)

    def _warm(self, prev, idx_d, s_d, pos_d):
        """The state each site's last solve left (a step that skips a site copies it forward) for this step's solve,
        which reads it t - last_solve periods ahead (sites idle at their last solve start cold through warm_had); the
        session multipliers follow their EV."""
        pidx, ps, ppos = self._prev
        mu_ev = torch.zeros(len(self.ev_req), dtype=torch.float32, device=prev["mu"].device)
        mu_ev[pidx] = prev["mu"][ps, ppos]
        mu = torch.zeros_like(prev["mu"])
        mu[s_d, pos_d] = mu_ev[idx_d]
        return dict(prev, mu=mu)

    def summary(self) -> Dict[str, float]:
        s = self.stats
        n = max(len(s.device_ms), 1)
        return dict(site_steps=float(sum(s.active_sites)), solves=float(sum(s.solved_sites)), steps=float(len(s.device_ms)),
                    unsolved=float(sum(s.unsolved)), device_ms=float(sum(s.device_ms)), host_ms=float(sum(s.host_ms)),
                    iters_mean=float(np.average(s.iters_mean, weights=np.maximum(s.solved_sites, 1e-9))) if n else 0.0,
                    iters_max=float(max(s.iters_max, default=0)))


class DeviceFleetReplay(_FleetReplayBase):
    """The simulator side of the control step on the device as well (SURVEY.md §8(f) N1): the EV table, the energy
    delivered, the previous peaks and the per-EV warm-start multipliers stay in device arrays.  A step is, on the current
    stream with no host synchronisation: the active sessions and the re-solve decision (acb_fleet_sessions), the launch
    sequence of BatchedAdaptiveCharging (`_launch`: preprocessing, admission, packing, the solve -- masked by the
    decision, each site warm-started from its own last state t - last_solve columns ahead -- and quantised pilots, as
    configured), and the simulator update (acb_fleet_apply).  Same pilots and `state()`, bit for bit, as FleetReplay.

    The admission puts the raw tables in arrival order but leaves `sess_ev` / `warm_mu` in the EV table's (station)
    order: they are indexed like the packed batch (warm_mu, out_mu), whose (EVSE, slot) order of a single-session site
    is the station order whatever the slot order.  With `battery` or `estimate_max_rate` the fleet kernels are the _ev
    entry points (acb_fleet_ev: batteries, estimates, the per-EVSE currents in `rates`); with the estimate the
    preprocessing caps each session's maximum rate at its EV's bound."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        from .batched import BatchedAdaptiveCharging

        dev = torch.device("cuda", engine._dev_index(self.device))
        self._bac = BatchedAdaptiveCharging(self.objective, self.info, self.period, batch=self.n_sites, max_sessions=self.N, horizon=self.Tp,
                                            demand_charge=self.demand_charge, solver_options=self.solver_options, device=self.device, chunks=1,
                                            enforce_pilot_limit=False, quantize=self.pilot_mode != 0,
                                            reallocate=self.pilot_mode == _cabi.ACB_PILOTS_REALLOCATE,
                                            uninterrupted_charging=self.uninterrupted_charging, skip_unabsorbable=True,
                                            estimate_max_rate=self.estimate_max_rate)
        if self._bac.Tp != self.Tp:
            raise ValueError(f"Tp = {self.Tp} is not a padded horizon of the solve path")
        self.site = self._bac.site
        self._ch = ch = self._bac.chunks[0]
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
            last_solve=torch.full((self.n_sites,), -1, dtype=torch.int32, device=dev),
            recompute=torch.zeros(self.n_sites, dtype=torch.int32, device=dev), shift=torch.zeros(self.n_sites, dtype=torch.int32, device=dev),
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
        f.max_recompute = self.max_recompute or 0
        if self._event_driven:  # (NULL last_solve: every site solves every step, column 0 applies)
            f.last_solve, f.recompute, f.shift = p(d["last_solve"]), p(d["recompute"]), p(d["shift"])
        self._fleet = f
        self._fev = None  # batteries / estimates (acb_fleet_ev); None = the plain fleet kernels
        if self.battery or self.estimate_max_rate:
            e = _cabi.FleetEV()
            d["rates"] = torch.zeros((self.n_sites, self.N), dtype=torch.float64, device=dev)
            e.rates = p(d["rates"])
            if self.battery:
                d["cap"], d["charge"] = up(self.ev_cap, np.float64), up(self.ev_charge, np.float64)
                e.ev_cap, e.ev_charge, e.transition_soc = p(d["cap"]), p(d["charge"]), self.transition_soc
            if self.estimate_max_rate:
                d["ub"] = up(self.ev_ub, np.float64)
                e.ev_ub, e.up_increment, e.down_threshold = p(d["ub"]), self.up_increment, self.down_threshold
                e.upper_bound = p(ch.dev_raw["upper_bound"])
            self._fev = e
        self._state = [ch.new_warm_state(), ch.new_warm_state()]
        ch.lb_zero = self.lb_zero  # the synthetic EVs have no minimum rate of their own
        o = ch.objective
        o.prev_peak = p(d["prev_peak"])
        o.prices_stride = 0  # one price vector for the whole fleet, read from the current period on
        self._started = False

    def step(self, t: int, want_first: bool = True):
        L, ch, d, p = _cabi.lib(), self._ch, self._d, engine._ptr
        stream = torch.cuda.current_stream(self._bac.device)
        st = C.c_void_p(stream.cuda_stream)
        prev, out = self._state
        ev = self._event_driven
        ch.set_warm(dict(prev, mu=d["warm_mu"]) if self.warm_start and self._started else None, out, shift=1, had=d["had"],
                    shifts=d["shift"] if ev else None, mask=d["recompute"] if ev else None)
        ch.objective.prices = C.c_void_p(d["prices"].data_ptr() + 8 * t) if self._bac.need_prices else None
        fev = C.byref(self._fev) if self._fev is not None else None
        _cabi.check(L.acb_fleet_sessions_ev(self.site.handle, C.byref(self._fleet), fev, t, C.byref(ch.sessions), p(d["sess_ev"]), p(d["warm_mu"]), st),
                    "acb_fleet_sessions_ev")
        self._bac._launch(ch, stream)
        if self.pilot_mode:  # the solve skipped the continuous projection (batch.pilots NULL); acb_fleet_apply reads batch.pilots
            ch.bind_pilots(True)
        _cabi.check(L.acb_fleet_apply_ev(self.site.handle, C.byref(self._fleet), fev, t, float(self.period), C.byref(ch.struct), p(d["sess_ev"]),
                                         p(d["first"]) if want_first else None, p(d["stats"]), st), "acb_fleet_apply_ev")
        if self.pilot_mode:
            ch.bind_pilots(False)
        self._state.reverse()
        self._started = True
        if not want_first:
            return None
        first = d["first"].cpu().numpy()
        self.rates = d["rates"].cpu().numpy() if "rates" in d else first
        return first

    def state(self) -> Dict[str, Optional[np.ndarray]]:
        """FleetReplay.state, copied back (into the attributes too) once the steps enqueued so far, on any stream, have
        finished.  Raises if the device packer flagged a step's sessions (two on one EVSE, or one beyond the padded horizon)."""
        torch.cuda.synchronize(self._bac.device)
        if int(self._ch.flags.cpu()[0]) != 0:
            raise ValueError("the device packer flagged the fleet's sessions (two sessions on one EVSE, or a session beyond the padded horizon)")
        d = self._d
        get = lambda k: d[k].cpu().numpy() if k in d else None  # noqa: E731
        self.ev_dlv, self.prev_peak, self.ev_charge, self.ev_ub = get("dlv"), get("prev_peak"), get("charge"), get("ub")
        rec = d["recompute"].cpu().numpy() != 0 if self._event_driven else np.ones(self.n_sites, dtype=bool)  # (else it is not bound)
        return dict(ev_dlv=self.ev_dlv, prev_peak=self.prev_peak, recompute=rec, status=self._ch.status.cpu().numpy() if self._started else None,
                    ev_charge=self.ev_charge, ev_ub=self.ev_ub, rates=get("rates"))

    def summary(self) -> Dict[str, float]:
        s = self._d["stats"].cpu().numpy()
        # (site_steps counts the solves of sites with sessions: with max_recompute != 1 the steps in between are not in it)
        return dict(site_steps=float(s[0]), solves=float(s[0]), unsolved=float(s[2]), iters_mean=float(s[1] / max(s[0], 1.0)))
