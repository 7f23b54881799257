"""Batched form of the per-step MPC path: many independent instances of ONE site per call.

``BatchedAdaptiveCharging.schedule(sessions, ...)`` is what ``AdaptiveSchedulingAlgorithm.schedule``
(reference adacharge/adacharge.py:135-193: build -> solve -> project the pilots -> max(., 0))
does for one site and one control step, for B instances at once (sites, scenarios, sweep points): the caller hands
over the raw session tables and the interface quantities as host arrays; this class stages them in pinned memory,
copies them to the device, packs them there (``acb_pack_sessions``: horizon, energy rows, the ObjectiveComponent
list -> cost vectors, reference aco.py:200-284, 363-408), solves (``acb_solve_batch``, whose epilogue also does the
continuous pilot projection, postprocessing.py:77-94) and copies the float64 pilots back.  With ``quantize`` (and
``reallocate``) the solve skips that projection and one more launch (``acb_quantize_pilots``) writes the discrete pilots
of project_into_discrete_feasible_pilots (postprocessing.py:97-118) or diff_based_reallocation (:189-258) instead.  The batch is cut into
chunks on their own streams so that the copies of one chunk overlap the solve of another.

Only the built-in objective functions are packed on the device (by identity, as the drop-in class recognises them);
sessions carry constant min/max rates.  Anything else goes through ``AdaptiveChargingOptimization`` per instance.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _cabi, engine
from . import adaptive_charging_optimization as aco
from .interface import infrastructure_from_dict

_KIND_OF = {
    aco.quick_charge: "quick_charge", aco.equal_share: "equal_share", aco.tou_energy_cost: "tou_energy_cost",
    aco.total_energy: "total_energy", aco.peak: "peak", aco.demand_charge: "demand_charge",
    aco.load_flattening: "load_flattening", aco.non_completion_penalty: "non_completion_penalty",
}
SESSION_FIELDS = (("station", np.int32), ("arrival_offset", np.int32), ("remaining_time", np.int32),
                  ("remaining_demand", np.float64), ("min_rate", np.float64), ("max_rate", np.float64))


def pilot_mode(quantize, reallocate, infrastructure) -> int:
    """The acb_quantize_pilots mode for AdaptiveSchedulingAlgorithm's `quantize` / `reallocate` flags (0 = continuous
    pilots), with the reference's rule (ada.py:101-105) and a check that every EVSE has its allowable pilots."""
    if reallocate and not quantize:
        raise ValueError("reallocate cannot be true without quantize. Otherwise there is nothing to reallocate :).")
    if not quantize:
        return 0
    ap = getattr(infrastructure, "allowable_pilots", None)
    n = len(infrastructure.station_ids)
    if ap is None or len(ap) != n or any(a is None or len(a) == 0 for a in ap):
        raise ValueError("quantize=True needs allowable_pilots for every EVSE of the infrastructure")
    return _cabi.ACB_PILOTS_REALLOCATE if reallocate else _cabi.ACB_PILOTS_DISCRETE


def objective_components(objective: Sequence[aco.ObjectiveComponent]):
    """ObjectiveComponent list -> (kind, coefficient, param) triples of ``acb_objective``; component kwargs win over
    caller kwargs as in build_objective (aco.py:203-217): only ``baseline_peak`` and ``norm`` matter here."""
    out = []
    for comp in objective:
        name = _KIND_OF.get(comp.function)
        if name is None:
            raise TypeError(f"objective component {getattr(comp.function, '__name__', comp.function)!r} cannot be packed on the device; "
                            f"built-ins are {sorted(_KIND_OF.values())} (use AdaptiveChargingOptimization for custom components)")
        kw = comp.kwargs or {}
        if name == "non_completion_penalty" and kw.get("norm", 1) == 2:
            name = "non_completion_penalty_l2"
        if name == "load_flattening" and kw.get("external_signal") is not None:
            raise ValueError("pass external_signal to schedule() (one row per instance), not as a component kwarg")
        out.append((_cabi.OBJ_KIND[name], float(comp.coefficient), float(kw.get("baseline_peak", 0.0))))
    baselines = {prm for k, _, prm in out if k in (_cabi.OBJ_KIND["peak"], _cabi.OBJ_KIND["demand_charge"])}
    if len(baselines) > 1:
        raise NotImplementedError("peak terms with different baselines are not supported on the device path")
    if len(out) > _cabi.ACB_MAX_COMPONENTS:
        raise ValueError(f"at most {_cabi.ACB_MAX_COMPONENTS} objective components")
    return out


@dataclass
class BatchResult:
    pilots: np.ndarray   # [B, N, Tp] float64, the pilots schedule() returns per EVSE (continuous or quantised); columns >= T[b] are zero
    status: np.ndarray   # [B] acb status
    iters: np.ndarray    # [B]
    T: np.ndarray        # [B] horizon of each instance (aco.py:243-245)
    stats: np.ndarray    # [B, ACB_NSTATS]


class _Chunk(engine.DeviceBatch):
    """One slice of the batch: pinned staging and device copies of the raw arrays, the device packer's two C structs
    (acb_sessions, acb_objective) and, as a DeviceBatch, the packed inputs that packer writes and the results."""

    def __init__(self, owner: "BatchedAdaptiveCharging", lo: int, hi: int):
        self.lo, self.hi = lo, hi
        B, S, Tp = hi - lo, owner.S_max, owner.Tp
        dev = owner.device
        self.stream = torch.cuda.Stream(device=dev)
        raw = {n: ((B, S), dt) for n, dt in SESSION_FIELDS}
        raw.update(prev_peak=((B,), np.float64))
        if owner.need_prices:
            raw["prices"] = ((B, Tp), np.float64)
        if owner.need_dc_array:
            raw["demand_charge"] = ((B,), np.float64)
        if owner.need_ext:
            raw["external_signal"] = ((B, Tp), np.float64)
        if owner.site.use_peak_row:
            raw["peak_limit"] = ((B, Tp), np.float64)
        if owner.estimate_max_rate:
            raw["upper_bound"] = ((B, S), np.float64)
        self.host = {k: torch.empty(shape, dtype=torch.from_numpy(np.empty(0, dt)).dtype).pin_memory() for k, (shape, dt) in raw.items()}
        self.dev_raw = {k: torch.empty_like(v, device=dev) for k, v in self.host.items()}
        self.h2d_bytes = sum(v.numel() * v.element_size() for v in self.host.values())
        f32, i32 = torch.float32, torch.int32
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)  # noqa: E731
        d = dict(T=mk((B,), i32), n_sessions=mk((B,), i32), sess_row=mk((B, S), i32), sess_start=mk((B, S), i32), sess_len=mk((B, S), i32),
                 sess_energy=mk((B, S), f32), sess_rate_off=mk((B, S), i32), min_rates=mk((B * S,), f32), max_rates=mk((B * S,), f32),
                 alpha=mk((B, Tp), f32), beta=mk((B, Tp), f32), qd=mk((B,), f32), gamma=mk((B,), f32), peak_w=mk((B,), f32), peak_p0=mk((B,), f32))
        if owner.need_ext:
            d["ext"] = mk((B, Tp), f32)
        if owner.site.use_peak_row:
            d["peak_limit"] = mk((B, Tp), f32)
        if owner.need_sess_quad:
            d["sess_quad"] = mk((B, S), f32)
        # pilots: continuous from the solve's epilogue; quantised from acb_quantize_pilots, without that projection first
        super().__init__(owner.site, d, Tp, S, multi_session=owner.multi_session, pilots=True)
        self.bind_pilots(not owner.pilot_mode)
        self.flags = torch.zeros((1,), dtype=i32, device=dev)
        self.flags_host = torch.zeros((1,), dtype=i32).pin_memory()
        p = engine._ptr
        s = _cabi.Sessions()
        s.B, s.S_max = B, S
        for n, _ in SESSION_FIELDS:
            setattr(s, n, p(self.dev_raw[n]))
        self.sessions = s
        o = _cabi.Objective()
        o.n = len(owner.components)
        for i, (k, c, prm) in enumerate(owner.components):
            o.kind[i], o.coef[i], o.param[i] = k, c, prm
        o.period = float(owner.period)
        o.prices, o.prices_stride = p(self.dev_raw.get("prices")), Tp
        o.prev_peak = p(self.dev_raw["prev_peak"])
        o.demand_charge, o.demand_charge_scalar = p(self.dev_raw.get("demand_charge")), float(owner.demand_charge_scalar)
        o.external_signal, o.ext_stride = p(self.dev_raw.get("external_signal")), Tp
        o.peak_limit, o.pl_stride = p(self.dev_raw.get("peak_limit")), Tp
        self.objective = o

    @property
    def batch(self) -> _cabi.Batch:
        """The chunk's acb_batch (DeviceBatch.struct), as the entry points after the packer take it."""
        return self.struct


class BatchedAdaptiveCharging:
    """B instances of one site per call.

    Args:
        objective: list of ObjectiveComponent over the built-in functions.
        infrastructure: InfrastructureInfo (or the dict form the generators produce).
        period: minutes per period (interface.period).
        batch: number of instances per call (fixed: staging and device buffers are allocated once).
        max_sessions: S_max, slots of the per-instance session table.
        horizon: largest arrival_offset + remaining_time that can occur.
        multi_session: an EVSE may hold more than one session within the horizon.
        demand_charge: $/kW (interface.get_demand_charge) when it is the same for every instance; per-instance values
            are passed to ``schedule``.
        quantize, reallocate: as AdaptiveSchedulingAlgorithm's (ada.py:101-113, 177-190): pilots rounded down into each
            EVSE's allowable set (every EVSE needs one), and with ``reallocate`` the first period's rounding loss given
            back greedily.  Bit-identical to the drop-in class with the same flags.
    """

    def __init__(self, objective: List[aco.ObjectiveComponent], infrastructure, period, batch: int, max_sessions: int, horizon: int,
                 constraint_type="SOC", enforce_energy_equality=False, peak_limit=False, multi_session=False, demand_charge=0.0,
                 per_instance_demand_charge=False, solver_options: Optional[dict] = None, device=None, chunks: int = 4,
                 enforce_pilot_limit=True, estimate_max_rate=False, quantize=False, reallocate=False):
        if isinstance(infrastructure, dict):
            infrastructure = infrastructure_from_dict(infrastructure)
        self.pilot_mode = pilot_mode(quantize, reallocate, infrastructure)
        self.components = objective_components(objective)
        kinds = {k for k, _, _ in self.components}
        K = _cabi.OBJ_KIND
        use_u = bool(kinds & {K["peak"], K["demand_charge"], K["load_flattening"]})
        self.site = engine.get_site(infrastructure, constraint_type, bool(peak_limit), use_u, device)
        self.device = torch.device("cuda", self.site.device)
        self.period, self.B, self.S_max = period, int(batch), int(max_sessions)
        self.Tp = engine.padded_horizon(int(horizon))
        self.multi_session = bool(multi_session)
        self.need_prices = K["tou_energy_cost"] in kinds
        self.need_ext = K["load_flattening"] in kinds
        self.need_dc_array = bool(per_instance_demand_charge)
        self.need_sess_quad = K["non_completion_penalty_l2"] in kinds
        # preprocessing of schedule() (ada.py:141-146) on the device: max_rate <- min(max_rate, max_pilot) and, with
        # estimate_max_rate, the estimator's per-session upper bounds (passed to schedule() as `upper_bound`)
        self.enforce_pilot_limit, self.estimate_max_rate = bool(enforce_pilot_limit), bool(estimate_max_rate)
        self.demand_charge_scalar = float(demand_charge)
        opts = dict(solver_options or {})
        if K["equal_share"] not in kinds:
            opts.setdefault("rate_tol", 0.0)  # no strictly convex term: nothing for the rate polish to do
        self.options = _cabi.default_options(equality=int(bool(enforce_energy_equality)), **opts)
        chunks = max(1, min(int(chunks), self.B))
        cuts = [round(k * self.B / chunks) for k in range(chunks + 1)]
        with torch.cuda.device(self.device):
            self.chunks = [_Chunk(self, a, b) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]
        N = self.site.N
        self.host_pilots = torch.empty((self.B, N, self.Tp), dtype=torch.float64).pin_memory()
        self.host_status = torch.empty((self.B,), dtype=torch.int32).pin_memory()
        self.host_iters = torch.empty((self.B,), dtype=torch.int32).pin_memory()
        self.host_T = torch.empty((self.B,), dtype=torch.int32).pin_memory()
        self.host_stats = torch.empty((self.B, _cabi.ACB_NSTATS), dtype=torch.float32).pin_memory()
        self.h2d_bytes = sum(c.h2d_bytes for c in self.chunks)
        self.d2h_bytes = sum(t.numel() * t.element_size() for t in (self.host_pilots, self.host_status, self.host_iters, self.host_T, self.host_stats))
        # own kernels per call and chunk: the packer + the solve (three launches when phased: solve, relaunch list, solve;
        # the general path launches per phase and is not counted here) + the preprocessing + the quantised pilots
        phased = self.options.phase_iters > 0 and self.options.phase_iters < self.options.max_iter
        self.kernel_launches_per_call = len(self.chunks) * (1 + (3 if phased else 1) + int(self.enforce_pilot_limit or self.estimate_max_rate)
                                                            + int(self.pilot_mode != 0))

    # ------------------------------------------------------------------------------------------------
    def _stage(self, ch: _Chunk, arrays: Dict[str, np.ndarray]):
        """host arrays -> the chunk's pinned staging (a plain memcpy per field)."""
        # every minimum rate 0 (the usual case) is declared to the library: fastest on-chip variant
        ch.lb_zero = not np.any(np.asarray(arrays["min_rate"])[ch.lo:ch.hi] != 0)
        for k, dst in ch.host.items():
            src = arrays.get(k)
            if src is None:
                if k == "prev_peak":
                    dst.zero_()
                    continue
                raise ValueError(f"schedule() needs `{k}` for this objective / site")
            a = np.asarray(src)
            d = dst.numpy()
            if k in ("prices", "external_signal", "peak_limit"):
                if a.ndim == 1:  # one vector for every instance
                    d[...] = a[None, : d.shape[1]]
                else:
                    d[...] = a[ch.lo:ch.hi, : d.shape[1]]
            elif a.ndim == 0:
                d[...] = a
            else:
                d[...] = a[ch.lo:ch.hi]

    def enqueue(self, ch: _Chunk, from_device_raw=False, events=None):
        """H2D of the raw arrays (unless they are already on the device), pack, solve, quantise (if asked), D2H — on the chunk's stream.
        `events`: a list that receives a (start, end) pair of CUDA events around the solve launch(es)."""
        L = _cabi.lib()
        st = C.c_void_p(ch.stream.cuda_stream)
        with torch.cuda.stream(ch.stream):
            if not from_device_raw:
                for k, t in ch.host.items():
                    ch.dev_raw[k].copy_(t, non_blocking=True)
            ch.flags.zero_()
            if self.enforce_pilot_limit or self.estimate_max_rate:
                _cabi.check(L.acb_preprocess_sessions(self.site.handle, C.byref(ch.sessions), int(self.enforce_pilot_limit),
                                                      engine._ptr(ch.dev_raw.get("upper_bound")), st), "acb_preprocess_sessions")
            _cabi.check(L.acb_pack_sessions(self.site.handle, C.byref(ch.sessions), C.byref(ch.objective), C.byref(ch.struct), engine._ptr(ch.flags), st), "acb_pack_sessions")
            if events is not None:
                ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                ev[0].record(ch.stream)
            ch.solve(self.options, st)
            if events is not None:
                ev[1].record(ch.stream)
                events.append(ev)
            if self.pilot_mode:
                _cabi.check(L.acb_quantize_pilots(self.site.handle, self.pilot_mode, C.byref(ch.sessions), float(self.period), C.byref(ch.struct),
                                                  engine._ptr(ch.pilots), st), "acb_quantize_pilots")
            if not from_device_raw:
                self.host_pilots[ch.lo:ch.hi].copy_(ch.pilots, non_blocking=True)
                self.host_status[ch.lo:ch.hi].copy_(ch.status, non_blocking=True)
                self.host_iters[ch.lo:ch.hi].copy_(ch.iters, non_blocking=True)
                self.host_T[ch.lo:ch.hi].copy_(ch.packed["T"], non_blocking=True)
                self.host_stats[ch.lo:ch.hi].copy_(ch.stats, non_blocking=True)
                ch.flags_host.copy_(ch.flags, non_blocking=True)

    def schedule_async(self, sessions: Dict[str, np.ndarray], prices=None, prev_peak=None, demand_charge=None, external_signal=None, peak_limit=None,
                       upper_bound=None, independent=False, start_event=None):
        """Stage, copy, pack, solve and copy back, chunk by chunk; returns after everything is enqueued.  By default the
        chunk streams start after the current stream's earlier work and the current stream waits for all chunks, so a
        synchronize of the current stream makes ``result()`` valid.  ``independent=True`` leaves the current stream out
        (the chunks start after ``start_event`` if given): calls on different objects then overlap on the device
        (double buffering); use ``wait()`` / ``join()`` before reading the result."""
        self.wait()  # the pinned staging and the result buffers of the previous call on this object are reused
        arrays = dict(sessions)
        arrays.update(prices=prices, prev_peak=prev_peak, demand_charge=demand_charge, external_signal=external_signal, peak_limit=peak_limit,
                      upper_bound=upper_bound)
        cur = torch.cuda.current_stream(self.device)
        for ch in self.chunks:
            self._stage(ch, arrays)
            if start_event is not None:
                ch.stream.wait_event(start_event)
            elif not independent:
                ch.stream.wait_stream(cur)
            self.enqueue(ch)
        self._finish(cur, independent)
        return self

    def _finish(self, cur, independent):
        self._done = []
        for ch in self.chunks:
            ev = torch.cuda.Event()
            ev.record(ch.stream)
            self._done.append(ev)
            if not independent:
                cur.wait_stream(ch.stream)

    def wait(self):
        """Block the host until the last call on this object has delivered its results."""
        for ev in getattr(self, "_done", ()):
            ev.synchronize()
        return self

    def join(self, stream=None):
        """Make `stream` (default: the current one) wait for the last call on this object."""
        st = stream or torch.cuda.current_stream(self.device)
        for ev in getattr(self, "_done", ()):
            st.wait_event(ev)
        return self

    def result(self, check=True) -> BatchResult:
        if check:
            fl = 0
            for ch in self.chunks:
                fl |= int(ch.flags_host[0])
            if fl & 1:
                raise ValueError("an EVSE holds more than one session in some instance: construct BatchedAdaptiveCharging(multi_session=True)")
            if fl & 2:
                raise ValueError(f"a session ends beyond the padded horizon {self.Tp}: construct with a larger `horizon`")
        return BatchResult(self.host_pilots.numpy(), self.host_status.numpy(), self.host_iters.numpy(), self.host_T.numpy(), self.host_stats.numpy())

    def schedule(self, sessions: Dict[str, np.ndarray], **kw) -> BatchResult:
        """Host arrays in, host pilots out (synchronous)."""
        self.schedule_async(sessions, **kw)
        torch.cuda.current_stream(self.device).synchronize()
        return self.result()

    # resident form (bench `value`): raw arrays already on the device, results stay there
    def upload_raw(self, sessions: Dict[str, np.ndarray], **kw):
        arrays = dict(sessions)
        arrays.update(kw)
        for ch in self.chunks:
            self._stage(ch, arrays)
            for k, t in ch.host.items():
                ch.dev_raw[k].copy_(t)
        torch.cuda.synchronize(self.device)
        return self

    def solve_resident(self, events=None, independent=False, start_event=None):
        cur = torch.cuda.current_stream(self.device)
        for ch in self.chunks:
            if start_event is not None:
                ch.stream.wait_event(start_event)
            elif not independent:
                ch.stream.wait_stream(cur)
            self.enqueue(ch, from_device_raw=True, events=events)
        self._finish(cur, independent)
        return self


def sessions_to_arrays(session_lists, infrastructure, S_max: Optional[int] = None) -> Dict[str, np.ndarray]:
    """Lists of SessionInfo (one list per instance) -> the [B, S_max] tables ``schedule`` takes.  Convenience for
    callers that hold reference-style objects; sessions must carry constant min/max rates."""
    B = len(session_lists)
    S = S_max or max(1, max(len(s) for s in session_lists))
    out = {n: np.zeros((B, S), dtype=dt) for n, dt in SESSION_FIELDS}
    out["station"][...] = -1
    for b, ss in enumerate(session_lists):
        for j, s in enumerate(ss):
            mn, mx = np.asarray(s.min_rates, dtype=float), np.asarray(s.max_rates, dtype=float)
            if mn.size and (mn.min() != mn.max() or mx.min() != mx.max()):
                raise ValueError("sessions_to_arrays: time-varying rate limits need the per-instance packer (AdaptiveChargingOptimization)")
            out["station"][b, j] = infrastructure.get_station_index(s.station_id)
            out["arrival_offset"][b, j] = s.arrival_offset
            out["remaining_time"][b, j] = s.remaining_time
            out["remaining_demand"][b, j] = s.remaining_demand
            out["min_rate"][b, j] = mn.flat[0] if mn.size else 0.0
            out["max_rate"][b, j] = mx.flat[0] if mx.size else 0.0
    return out


__all__ = ["BatchedAdaptiveCharging", "BatchResult", "sessions_to_arrays", "objective_components", "pilot_mode"]
