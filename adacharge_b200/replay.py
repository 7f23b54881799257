"""Closed-loop MPC replay over many independent sites with warm starts (BASELINE config 4;
SURVEY.md §8(f) row N1).  The per-step control flow is that of
AdaptiveSchedulingAlgorithm.schedule (reference adacharge/adacharge.py:135-193) for every
site at once: active sessions -> one batched solve -> continuous-pilot projection ->
first-period pilots applied to the EVs.  The simulator side (arrivals, energy bookkeeping)
is a minimal host stand-in for acnportal's Simulator; the solve and projection run on the
GPU, warm-started from the previous step's solver state shifted by one period.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _cabi, engine
from .adaptive_charging_optimization import AdaptiveChargingOptimization, ObjectiveComponent
from .interface import SessionInfo, TestingInterface, infrastructure_from_dict


REPLAY_SOLVER_DEFAULTS = dict(term_floor=1.0, stall_exit=40, alpha=1.7, stall_checks=3)  # warm-started steps: 57 vs 61 mean iterations at the library's 1.8 / 2


@dataclass
class EV:
    station: int
    session_id: str
    arrival: int
    departure: int
    requested: float  # kWh
    delivered: float = 0.0
    max_rate: float = 32.0


def synthetic_day(infra: Dict, seed: int, steps: int = 288, period: float = 5, mean_sessions: int = 40) -> List[EV]:
    """Seeded arrival process for one site-day: workplace-like arrivals (mean 9h), 2-9 h stays."""
    rng = np.random.default_rng(seed)
    n = len(infra["station_ids"])
    k = min(n, int(rng.poisson(mean_sessions)))
    stations = rng.permutation(n)[:k]
    arr = np.clip(rng.normal(9 * 60 / period, 1.5 * 60 / period, k).astype(int), 0, steps - 13)
    dur = rng.integers(int(2 * 60 / period), int(9 * 60 / period), k)
    dep = np.minimum(arr + dur, steps)
    req = np.minimum(rng.uniform(3, 25, k), 0.9 * (dep - arr) * 32 * 208 / 1000 * period / 60)
    return [EV(int(s), f"s{seed}-{j}", int(a), int(d), float(r)) for j, (s, a, d, r) in enumerate(zip(stations, arr, dep, req))]


class _SiteIface(TestingInterface):
    """TestingInterface whose price vector is indexed by absolute time."""


@dataclass
class ReplayStats:
    iters: List[np.ndarray] = field(default_factory=list)
    status: List[np.ndarray] = field(default_factory=list)
    delivered_frac: Optional[np.ndarray] = None
    peak_kw: Optional[np.ndarray] = None


class SiteReplay:
    """`n_sites` independent copies of one site, each with its own seeded day of EVs."""

    def __init__(self, infra: Dict, objective: List[ObjectiveComponent], n_sites: int, steps: int = 288, period: float = 5,
                 prices: Optional[np.ndarray] = None, demand_charge: float = 15.51, seed0: int = 0, warm_start: bool = True,
                 solver_options: Optional[dict] = None, device=None, mean_sessions: int = 40):
        self.infra, self.objective, self.n_sites, self.steps, self.period = infra, objective, n_sites, steps, period
        self.warm_start, self.device = warm_start, device
        # closed loop: the sunk demand charge w * prev_peak is a constant of every step's objective and can cancel the
        # energy term, so the gap is taken relative to the terms' magnitude; a stalled instance stops after 40 checks
        self.options = _cabi.default_options(**{**REPLAY_SOLVER_DEFAULTS, **(solver_options or {})})
        from .generators import sce_tou_prices

        self.prices = sce_tou_prices(2 * steps, period) if prices is None else np.asarray(prices, dtype=float)
        self.demand_charge = demand_charge
        self.evs = [synthetic_day(infra, seed0 + s, steps, period, mean_sessions) for s in range(n_sites)]
        self.prev_peak = np.zeros(n_sites)  # A
        self.volt = np.asarray(infra["voltages"], dtype=float)
        self.info = infrastructure_from_dict(infra)
        self.site: Optional[engine.Site] = None
        self._warm = None  # (device tensors, per-instance {session_id: mu}, site index of each batch row)
        self.keep_problems = False  # tests: record (t, site, sessions, prev_peak, schedule, status) of every solved step
        self.problems: List[tuple] = []

    # ------------------------------------------------------------------ one control step
    def _active(self, s: int, t: int) -> List[SessionInfo]:
        out = []
        for ev in self.evs[s]:
            if ev.arrival <= t < ev.departure and ev.requested - ev.delivered > 1e-6:
                out.append(SessionInfo(self.infra["station_ids"][ev.station], ev.session_id, ev.requested, ev.delivered,
                                       ev.arrival, ev.departure, current_time=t, max_rates=ev.max_rate))
        return out

    def step(self, t: int, stats: ReplayStats):
        insts, rows, sessions_of = [], [], []
        for s in range(self.n_sites):
            sess = self._active(s, t)
            if not sess:
                continue
            iface = _SiteIface({"active_sessions": [], "infrastructure_info": self.infra, "current_time": t, "period": self.period,
                                "prices": self.prices, "demand_charge": self.demand_charge, "prev_peak": float(self.prev_peak[s])})
            aco = AdaptiveChargingOptimization(self.objective, iface, device=self.device)
            inst = aco.build_instance(sess, self.info, None, float(self.prev_peak[s]))
            if self.site is None:
                self.site = aco._site_for(self.info, inst)
            insts.append(inst)
            rows.append(s)
            sessions_of.append([sess[j].session_id for j in inst.sess_order])
        if not insts:
            self._warm = None
            return
        pb = engine.PackedBatch(self.site, insts, Tp=engine.SUPPORTED_HORIZONS[-1], S_max=len(self.infra["station_ids"]), want_warm_out=True)
        if self.warm_start and self._warm is not None:
            warm, had = self._previous_rows(rows, sessions_of, pb)
            pb.set_warm(warm, pb.warm_out, shift=1, had=had)
        pb.upload().solve(self.options)
        pilots = engine.project_continuous(self.site, pb.rates.to(torch.float64))  # pp.py:77-94 on device
        first = pilots[:, :, 0].cpu().numpy()
        it, st = pb.iters.cpu().numpy(), pb.status.cpu().numpy()
        self.last_stats = pb.stats.cpu().numpy()  # rows: r_prim, r_dual, gap, violation, rho, cost scale, restarts, averaged
        if self.keep_problems:
            R = pb.rates.cpu().numpy().astype(np.float64)
            for b, s in enumerate(rows):
                self.problems.append((t, s, self._active(s, t), float(self.prev_peak[s]), R[b][:, : insts[b].T].copy(), int(st[b]), int(it[b])))
        stats.iters.append(it)
        stats.status.append(st)
        # apply the first-period pilots (the simulator side)
        w = self.volt * self.period / 1e3 / 60
        for b, s in enumerate(rows):
            for ev in self.evs[s]:
                if ev.arrival <= t < ev.departure:
                    e = min(first[b, ev.station] * w[ev.station], ev.requested - ev.delivered)
                    ev.delivered += max(e, 0.0)
            self.prev_peak[s] = max(self.prev_peak[s], float(first[b].sum()))
        mu = pb.warm_out["mu"].cpu().numpy()
        self._warm = (pb.warm_out, [dict(zip(ids, mu[b, : len(ids)])) for b, ids in enumerate(sessions_of)], rows)

    def _previous_rows(self, rows, sessions_of, pb):
        """The previous step's state, row by row of this batch (which holds the active sites only): multipliers follow
        their session; the solve reads it one period ahead.  Sites without a row in the previous batch start cold.
        Returns (warm state, had-row mask)."""
        old, old_mu, old_rows = self._warm
        pos = {s: b for b, s in enumerate(old_rows)}
        idx = [pos.get(s, -1) for s in rows]
        dev = old["v1"].device
        had = torch.tensor([i >= 0 for i in idx], dtype=torch.int32, device=dev)
        gather = torch.tensor([max(i, 0) for i in idx], device=dev)
        mu = np.zeros((len(rows), pb.S_max), dtype=np.float32)
        for b, (i, ids) in enumerate(zip(idx, sessions_of)):
            if i >= 0:
                m = old_mu[i]
                mu[b, : len(ids)] = [m.get(sid, 0.0) for sid in ids]
        warm = dict(v1=old["v1"][gather], vc=old["vc"][gather], mu=torch.from_numpy(mu).to(dev), scal=old["scal"][gather])
        return warm, had

    def run(self, t0: int = 0, t1: Optional[int] = None) -> ReplayStats:
        stats = ReplayStats()
        for t in range(t0, self.steps if t1 is None else t1):
            self.step(t, stats)
        req = np.array([sum(ev.requested for ev in day) for day in self.evs])
        dlv = np.array([sum(ev.delivered for ev in day) for day in self.evs])
        stats.delivered_frac = dlv / np.maximum(req, 1e-9)
        stats.peak_kw = self.prev_peak * self.volt[0] / 1000
        return stats
