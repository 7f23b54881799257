"""Host side of the device path: site handles, packing of sessions / objectives into
staging tensors, and the batched solve / postprocess calls through the C ABI.

PyTorch is used only for device memory, pinned staging buffers and streams.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _cabi
from ._cabi import Batch, Options


def _dev_index(device) -> int:
    if device is None:
        return torch.cuda.current_device()
    d = torch.device(device)
    return d.index if d.index is not None else torch.cuda.current_device()


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("adacharge_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream_ptr(device_index: int):
    return C.c_void_p(torch.cuda.current_stream(device_index).cuda_stream)


class Site:
    """Device-resident constants of one charging site for one problem shape
    (constraint type, whether a peak-limit row / an aggregate-power row is present)."""

    def __init__(self, infrastructure, constraint_type="SOC", use_peak_row=False, use_agg_row=False, device=None):
        _require_cuda()
        L = _cabi.lib()
        if constraint_type not in ("SOC", "LINEAR"):
            raise ValueError(
                "Invalid infrastructure constraint type: {0}. Valid options are SOC or AFFINE.".format(constraint_type)
            )
        self.device = _dev_index(device)
        cm = infrastructure.constraint_matrix
        has_infra = not (cm is None or np.asarray(cm).shape == (0, 0))  # aco.py:146-150
        N = len(infrastructure.station_ids)
        self.N = N
        if has_infra:
            cm = np.ascontiguousarray(np.asarray(cm, dtype=np.float64))
            M = cm.shape[0]
            limits = np.ascontiguousarray(np.asarray(infrastructure.constraint_limits, dtype=np.float64))
            if constraint_type == "SOC" and infrastructure.phases is None:
                raise ValueError("phases is required when using SOC infrastructure constraints.")
            phases = None if infrastructure.phases is None else np.ascontiguousarray(np.asarray(infrastructure.phases, dtype=np.float64))
        else:
            M, cm, limits, phases = 0, None, None, None
        volt = np.ascontiguousarray(np.asarray(infrastructure.voltages, dtype=np.float64))
        mp = getattr(infrastructure, "max_pilot", None)
        mp = None if mp is None else np.ascontiguousarray(np.asarray(mp, dtype=np.float64))
        ap = getattr(infrastructure, "allowable_pilots", None)
        off = vals = None
        if ap is not None and all(a is not None for a in ap) and len(ap) == N:
            off = np.zeros(N + 1, dtype=np.int32)
            off[1:] = np.cumsum([len(a) for a in ap])
            vals = np.ascontiguousarray(np.concatenate([np.asarray(a, dtype=np.float64) for a in ap]))
        self.M = M
        self._keep = (cm, limits, phases, volt, mp, off, vals)
        h = C.c_void_p()

        def p(a):
            return None if a is None else a.ctypes.data_as(C.c_void_p)

        _cabi.check(
            L.acb_site_create(C.byref(h), self.device, N, M, p(cm), p(phases), p(limits), p(volt),
                              _cabi.ACB_SOC if constraint_type == "SOC" else _cabi.ACB_LINEAR,
                              int(use_peak_row), int(use_agg_row), p(mp), p(off), p(vals)),
            "acb_site_create",
        )
        self.handle = h
        dims = [C.c_int() for _ in range(5)]
        L.acb_site_dims(h, *[C.byref(d) for d in dims])
        _, _, self.R, self.NG, self.NP = [d.value for d in dims]
        self.constraint_type = constraint_type
        self.use_peak_row, self.use_agg_row = bool(use_peak_row), bool(use_agg_row)
        self.voltages = volt
        self.has_pilots = off is not None

    def max_horizon(self) -> int:
        return _cabi.lib().acb_site_max_horizon(self.handle)

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            _cabi.lib().acb_site_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


# Sites are cached per (infrastructure content, problem shape, device).  The cache is a small LRU: an evicted site is
# only dropped from the table -- batches that still hold it keep it alive, and Site.__del__ frees the device memory
# once the last reference is gone -- so a long simulation over changing networks does not accumulate device allocations.
SITE_CACHE_SIZE = 16
_site_cache: "OrderedDict" = None  # created lazily (keeps `import adacharge_b200` free of side effects)


def _cache():
    global _site_cache
    if _site_cache is None:
        from collections import OrderedDict

        _site_cache = OrderedDict()
    return _site_cache


def _infra_key(infra):
    cm = infra.constraint_matrix
    cmb = b"" if cm is None else np.ascontiguousarray(np.asarray(cm, dtype=np.float64)).tobytes()
    ph = b"" if infra.phases is None else np.asarray(infra.phases, dtype=np.float64).tobytes()
    ap = getattr(infra, "allowable_pilots", None)
    apb = b"" if ap is None or any(a is None for a in ap) else b"|".join(np.asarray(a, dtype=np.float64).tobytes() for a in ap)
    mp = getattr(infra, "max_pilot", None)
    lim = getattr(infra, "constraint_limits", None)
    return hash((
        cmb, ph, b"" if lim is None else np.asarray(lim, dtype=np.float64).tobytes(),
        np.asarray(infra.voltages, dtype=np.float64).tobytes(), apb,
        b"" if mp is None else np.asarray(mp, dtype=np.float64).tobytes(), tuple(infra.station_ids),
    ))


def _cache_put(key, site):
    c = _cache()
    c[key] = site
    c.move_to_end(key)
    while len(c) > SITE_CACHE_SIZE:
        c.popitem(last=False)
    return site


def get_site(infra, constraint_type="SOC", use_peak_row=False, use_agg_row=False, device=None) -> Site:
    key = (_infra_key(infra), constraint_type, bool(use_peak_row), bool(use_agg_row), _dev_index(device) if torch.cuda.is_available() else -1)
    c = _cache()
    s = c.get(key)
    if s is None:
        return _cache_put(key, Site(infra, constraint_type, use_peak_row, use_agg_row, device))
    c.move_to_end(key)
    return s


class _PilotsOnly:
    """View of an infrastructure without its network rows: what the pilot projections read (postprocessing.py:92, 114)."""

    def __init__(self, infra):
        self.constraint_matrix, self.constraint_limits, self.phases = None, None, None
        self.station_ids, self.voltages = infra.station_ids, infra.voltages
        self.max_pilot, self.allowable_pilots = getattr(infra, "max_pilot", None), getattr(infra, "allowable_pilots", None)


def get_post_site(infra, network=True, device=None) -> Site:
    """Site for the postprocessing kernels: any cached site of this infrastructure carries the float64 constants they
    need; otherwise a SOC site (network=True) or a pilots-only site (network=False, no phases required) is built."""
    ik, dv = _infra_key(infra), _dev_index(device) if torch.cuda.is_available() else -1
    c = _cache()
    for key, s in reversed(c.items()):
        if key[0] == ik and key[-1] == dv and (not network or (key[1] == "SOC" and s.M == (0 if infra.constraint_matrix is None else np.asarray(infra.constraint_matrix).shape[0]))):
            return s
    if network or infra.phases is not None:
        return get_site(infra, "SOC", False, False, device)
    return _cache_put((ik, "PILOTS", False, False, dv), Site(_PilotsOnly(infra), "SOC", False, False, device))


# ----------------------------------------------------------------------------- packing
@dataclass
class Instance:
    """One MPC instance in host form (what build_problem derives from the reference's
    arguments): sessions as (row, start, len, energy[A*periods], min_rates, max_rates),
    objective pieces in minimisation form."""

    T: int
    sess_row: np.ndarray
    sess_start: np.ndarray
    sess_len: np.ndarray
    sess_energy: np.ndarray
    min_rates: List[np.ndarray]
    max_rates: List[np.ndarray]
    alpha: np.ndarray
    beta: np.ndarray
    qd: float = 0.0
    gamma: float = 0.0
    ext: Optional[np.ndarray] = None
    peak_w: float = 0.0
    peak_p0: float = 0.0
    peak_limit: Optional[np.ndarray] = None
    sess_order: Optional[np.ndarray] = None  # packed position -> index in the caller's session list
    sess_quad: Optional[np.ndarray] = None   # per-session weight of (energy - planned)^2 in (A*periods)^2 (non_completion_penalty, norm 2)
    peak_terms: Optional[list] = None        # [(baseline kW, weight)] ascending when peak components differ in baseline (host walks the pieces)


def pack_sessions(sessions, infra, period) -> dict:
    """Session table sorted by EVSE row (the kernel wants each row's sessions
    contiguous).  Energy in A*periods: remaining_demand / (V_i * period / 1e3 / 60)
    (aco.py:114-122)."""
    rows = np.array([infra.get_station_index(s.station_id) for s in sessions], dtype=np.int64)
    order = np.argsort(rows, kind="stable")
    volt = np.asarray(infra.voltages, dtype=np.float64)
    out = dict(sess_row=[], sess_start=[], sess_len=[], sess_energy=[], min_rates=[], max_rates=[], order=order)
    for j in order:
        s = sessions[j]
        i = int(rows[j])
        rt = int(s.remaining_time)
        w = volt[i] * period / 1e3 / 60
        out["sess_row"].append(i)
        out["sess_start"].append(int(s.arrival_offset))
        out["sess_len"].append(rt)
        out["sess_energy"].append(float(s.remaining_demand) / w)
        mn = np.broadcast_to(np.asarray(s.min_rates, dtype=np.float64), (rt,)) if np.ndim(s.min_rates) == 0 else np.asarray(s.min_rates, dtype=np.float64)[:rt]
        mx = np.broadcast_to(np.asarray(s.max_rates, dtype=np.float64), (rt,)) if np.ndim(s.max_rates) == 0 else np.asarray(s.max_rates, dtype=np.float64)[:rt]
        out["min_rates"].append(mn)
        out["max_rates"].append(mx)
    return out


SUPPORTED_HORIZONS = (64, 128, 160, 288)  # padded horizons the on-chip solve kernel is instantiated for
MAX_HORIZON = 3616  # longest padded horizon of the general (streaming) path: rows are staged in shared memory


def padded_horizon(T: int) -> int:
    """Smallest padded horizon that can hold T periods: one of the on-chip kernel's, else the next multiple of 32
    (solved by the general path; reference aco.py:243-245 puts no limit on T)."""
    for t in SUPPORTED_HORIZONS:
        if t >= T:
            return t
    Tp = ((int(T) + 31) // 32) * 32
    if Tp > MAX_HORIZON:
        raise ValueError(f"horizon {T} exceeds the longest supported horizon {MAX_HORIZON} periods")
    return Tp


class DeviceBatch:
    """Device side of one acb_batch (include/adacharge_b200.h): the packed inputs, the result and scratch tensors, and
    the struct that points at them.  The struct is filled once, here; afterwards only the warm-start and pilots
    pointers and the two declared flags change (set_warm, or warm / warm_out alone; bind_pilots; lb_zero,
    multi_session), so a batch that is solved every step is not rebuilt.  Entry points that take an acb_batch get
    ``C.byref(self.struct)``.

    `packed` holds the input tensors by acb_batch field name (`T`, `n_sessions`, `sess_*`, `min_rates`, `max_rates`,
    `alpha`, `beta`, `qd`, `gamma`, `peak_w`, `peak_p0`; `ext`, `peak_limit`, `sess_quad` optional).  `pilots`
    allocates the float64 [B, N, Tp] pilots the solve's epilogue writes; `rate_est` the rate polish's estimate."""

    def __init__(self, site: Site, packed: Dict[str, torch.Tensor], Tp: int, S_max: int, multi_session=False, lb_zero=False,
                 pilots=False, rate_est=False):
        B, N, R = int(packed["T"].shape[0]), site.N, site.R
        dev = torch.device("cuda", site.device)
        self.site, self.device, self.B, self.Tp, self.S_max, self.packed = site, dev, B, Tp, S_max, packed
        self.rates = torch.empty((B, N, Tp), dtype=torch.float32, device=dev)
        self.status = torch.empty((B,), dtype=torch.int32, device=dev)
        self.iters = torch.empty((B,), dtype=torch.int32, device=dev)
        self.stats = torch.empty((B, _cabi.ACB_NSTATS), dtype=torch.float32, device=dev)
        self.work = torch.empty((B, N + max(R, 1), Tp), dtype=torch.float32, device=dev)
        self.pilots = torch.empty((B, N, Tp), dtype=torch.float64, device=dev) if pilots else None
        self.rate_est = torch.full((B,), -1.0, dtype=torch.float32, device=dev) if rate_est else None
        s = self.struct = Batch()
        s.B, s.Tp, s.S_max = B, Tp, S_max
        for name, t in packed.items():
            setattr(s, name, _ptr(t))
        s.work, s.rates, s.status, s.iters, s.stats = _ptr(self.work), _ptr(self.rates), _ptr(self.status), _ptr(self.iters), _ptr(self.stats)
        s.pilots, s.rate_est = _ptr(self.pilots), _ptr(self.rate_est)
        self.multi_session, self.lb_zero = multi_session, lb_zero
        self.set_warm()

    @property
    def multi_session(self) -> bool:
        """Declared to the library: an EVSE may hold more than one session."""
        return bool(self.struct.multi_session)

    @multi_session.setter
    def multi_session(self, v):
        self.struct.multi_session = int(bool(v))

    @property
    def lb_zero(self) -> bool:
        """Declared to the library: every minimum rate of the batch is 0 (the usual case; its fastest on-chip variant)."""
        return bool(self.struct.lb_zero)

    @lb_zero.setter
    def lb_zero(self, v):
        self.struct.lb_zero = int(bool(v))

    def new_warm_state(self) -> Dict[str, torch.Tensor]:
        """One zeroed set of warm-start tensors of this batch's shape: v1 [B, N, Tp], vc [B, max(R, 1), Tp], mu [B, S_max],
        scal [B, 2] (rho, peak level)."""
        B, Tp = self.B, self.Tp
        mk = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=self.device)  # noqa: E731
        return dict(v1=mk(B, self.site.N, Tp), vc=mk(B, max(self.site.R, 1), Tp), mu=mk(B, self.S_max), scal=mk(B, 2))

    def set_warm(self, warm: Optional[Dict[str, torch.Tensor]] = None, out: Optional[Dict[str, torch.Tensor]] = None, shift: int = 0,
                 had: Optional[torch.Tensor] = None):
        """Where the following solves start from and where they leave their final state (see `warm`, `warm_out`).
        `warm` is read `shift` columns ahead (1: the previous control step's state), and an instance whose `had` [B]
        int32 entry is 0 starts cold (its site was idle before)."""
        self.warm, self.warm_out = warm, out
        self.struct.warm_shift, self.struct.warm_had = shift, _ptr(had)
        self._had = had  # the struct holds a raw pointer: keep the tensor alive

    @property
    def warm(self) -> Optional[Dict[str, torch.Tensor]]:
        """Warm-start inputs of the following solves: a new_warm_state() set (None: a cold start)."""
        return self._warm

    @warm.setter
    def warm(self, w: Optional[Dict[str, torch.Tensor]]):
        s, d = self.struct, w or {}
        s.warm_v1, s.warm_vc, s.warm_mu, s.warm_scal = _ptr(d.get("v1")), _ptr(d.get("vc")), _ptr(d.get("mu")), _ptr(d.get("scal"))
        self._warm = w

    @property
    def warm_out(self) -> Optional[Dict[str, torch.Tensor]]:
        """Where the following solves write their final state: a new_warm_state() set (None: not written)."""
        return self._warm_out

    @warm_out.setter
    def warm_out(self, o: Optional[Dict[str, torch.Tensor]]):
        s, d = self.struct, o or {}
        s.out_v1, s.out_vc, s.out_mu, s.out_scal = _ptr(d.get("v1")), _ptr(d.get("vc")), _ptr(d.get("mu")), _ptr(d.get("scal"))
        self._warm_out = o

    def bind_pilots(self, on: bool):
        """Point acb_batch.pilots at `self.pilots` (on) or at nothing: the solve's epilogue writes the continuous pilots
        there, and acb_fleet_apply reads the pilots from there."""
        self.struct.pilots = _ptr(self.pilots) if on else None

    def solve(self, options: Options, stream=None):
        """Enqueue acb_solve_batch on `stream` (a cudaStream_t; default: the current stream)."""
        st = _stream_ptr(self.site.device) if stream is None else stream
        _cabi.check(_cabi.lib().acb_solve_batch(self.site.handle, C.byref(self.struct), C.byref(options), st), "acb_solve_batch")
        return self


class PackedBatch(DeviceBatch):
    """A batch packed on the host: pinned staging of the acb_batch inputs (`host`), copied into the device inputs by
    upload()."""

    def __init__(self, site: Site, instances: Sequence[Instance], Tp: Optional[int] = None, S_max: Optional[int] = None,
                 want_warm_out=False):
        B = len(instances)
        Tmax = max(i.T for i in instances)
        if Tp is None:
            Tp = padded_horizon(Tmax)
        Tp_, S_ = Tp, S_max or max(4, max(len(i.sess_row) for i in instances))
        f32, i32 = np.float32, np.int32
        h = {}
        multi_session = any(len(set(i.sess_row.tolist())) < len(i.sess_row) for i in instances)
        h["T"] = np.array([i.T for i in instances], dtype=i32)
        h["n_sessions"] = np.array([len(i.sess_row) for i in instances], dtype=i32)
        for name in ("sess_row", "sess_start", "sess_len"):
            a = np.zeros((B, S_), dtype=i32)
            for b, inst in enumerate(instances):
                v = getattr(inst, name)
                a[b, : len(v)] = v
            h[name] = a
        a = np.zeros((B, S_), dtype=f32)
        offs = np.zeros((B, S_), dtype=i32)
        mins, maxs, o = [], [], 0
        for b, inst in enumerate(instances):
            a[b, : len(inst.sess_energy)] = inst.sess_energy
            for s, (mn, mx) in enumerate(zip(inst.min_rates, inst.max_rates)):
                if len(mn) and mn.min() == mn.max() and mx.min() == mx.max():
                    # constant limits (the usual case): one (min, max) pair, offset -(p + 1)
                    offs[b, s] = -(o + 1)
                    mn, mx = mn[:1], mx[:1]
                else:
                    offs[b, s] = o
                mins.append(mn)
                maxs.append(mx)
                o += len(mn)
        h["sess_energy"], h["sess_rate_off"] = a, offs
        h["min_rates"] = np.concatenate(mins).astype(f32) if mins else np.zeros(1, f32)
        h["max_rates"] = np.minimum(np.concatenate(maxs), 3.0e38).astype(f32) if maxs else np.zeros(1, f32)
        for name in ("alpha", "beta"):
            a = np.zeros((B, Tp_), dtype=f32)
            for b, inst in enumerate(instances):
                a[b, : inst.T] = getattr(inst, name)[: inst.T]
            h[name] = a
        for name in ("qd", "gamma", "peak_w", "peak_p0"):
            h[name] = np.array([getattr(i, name) for i in instances], dtype=f32)
        if any(i.ext is not None for i in instances):
            a = np.zeros((B, Tp_), dtype=f32)
            for b, inst in enumerate(instances):
                if inst.ext is not None:
                    a[b, : inst.T] = inst.ext[: inst.T]
            h["ext"] = a
        if any(i.sess_quad is not None for i in instances):
            a = np.zeros((B, S_), dtype=f32)
            for b, inst in enumerate(instances):
                if inst.sess_quad is not None:
                    a[b, : len(inst.sess_quad)] = inst.sess_quad
            h["sess_quad"] = a
        if site.use_peak_row:
            a = np.full((B, Tp_), 3.0e38, dtype=f32)
            for b, inst in enumerate(instances):
                if inst.peak_limit is None:
                    raise ValueError("site was built with a peak-limit row but an instance has no peak_limit")
                a[b, : inst.T] = np.broadcast_to(np.asarray(inst.peak_limit, dtype=np.float64), (inst.T,))
            h["peak_limit"] = a
        self._stage(site, h, Tp_, S_, multi_session, want_warm_out)

    @classmethod
    def from_arrays(cls, site: Site, host: Dict[str, np.ndarray], Tp: int, S_max: int, multi_session=False, want_warm_out=False):
        """Batch from already-packed host arrays (the acb_batch fields of include/adacharge_b200.h
        by name; `T`, `n_sessions`, `sess_*`, `min_rates`, `max_rates`, `alpha`, `beta`, `qd`,
        `gamma`, `peak_w`, `peak_p0` required, `ext` / `peak_limit` optional).  Used by callers
        that keep their sessions in arrays (replay_fast) instead of SessionInfo objects."""
        if Tp % 32 != 0 or Tp <= 0 or Tp > MAX_HORIZON:
            raise ValueError(f"Tp must be a positive multiple of 32, at most {MAX_HORIZON}")
        if site.use_peak_row and "peak_limit" not in host:
            raise ValueError("site was built with a peak-limit row but the batch has no peak_limit")
        self = cls.__new__(cls)
        self._stage(site, host, Tp, S_max, multi_session, want_warm_out)
        return self

    def _stage(self, site: Site, h: Dict[str, np.ndarray], Tp: int, S_max: int, multi_session: bool, want_warm_out: bool):
        self.host = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in h.items()}
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.host.values())
        dev = torch.device("cuda", site.device)
        packed = {k: torch.empty_like(t, device=dev) for k, t in self.host.items()}
        # the rate polish needs a strictly convex objective: without a quadratic term the library is told not to
        # allocate its previous-schedule scratch
        self.any_quadratic = bool(np.any(np.asarray(h["qd"]) > 0))
        super().__init__(site, packed, Tp, S_max, multi_session=multi_session, lb_zero=_all_zero(h["min_rates"]), rate_est=self.any_quadratic)
        if want_warm_out:
            self.warm_out = self.new_warm_state()
        self._uploaded = False

    def refill(self, h: Dict[str, np.ndarray]):
        """Overwrite the pinned staging buffers in place with a new batch of the same shape (same field names, shapes
        and dtypes as at construction): callers that solve a fresh batch every step (the replay) keep one PackedBatch
        instead of pinning new host memory each time.  Follow with upload() / solve()."""
        if set(h) != set(self.host):
            raise ValueError(f"refill needs exactly the fields of the original batch: {sorted(self.host)}")
        for k, v in h.items():
            dst = self.host[k].numpy()
            if dst.shape != v.shape or dst.dtype != v.dtype:
                raise ValueError(f"refill: field {k} changed shape or dtype ({dst.shape} {dst.dtype} -> {v.shape} {v.dtype})")
            dst[...] = v
        self.any_quadratic = bool(np.any(np.asarray(h["qd"]) > 0))
        self.lb_zero = _all_zero(h["min_rates"])
        return self

    def upload(self):
        for k, t in self.host.items():
            self.packed[k].copy_(t, non_blocking=True)
        self._uploaded = True
        return self

    def solve(self, options: Optional[Options] = None):
        """Enqueue the batched solve on the current stream (asynchronous)."""
        if not self._uploaded:
            self.upload()
        opt = options or _cabi.default_options()
        if not self.any_quadratic and opt.rate_tol > 0:
            opt = _cabi.copy_options(opt, rate_tol=0.0)
        return super().solve(opt)

    def bounds(self):
        """charging_rate_bounds on device -> (lb, ub) tensors [B, N, Tp]."""
        if not self._uploaded:
            self.upload()
        lb = torch.empty_like(self.rates)
        ub = torch.empty_like(self.rates)
        _cabi.check(
            _cabi.lib().acb_charging_rate_bounds(self.site.handle, C.byref(self.struct), _ptr(lb), _ptr(ub), _stream_ptr(self.site.device)),
            "acb_charging_rate_bounds",
        )
        return lb, ub


def _all_zero(min_rates) -> bool:
    return not bool(np.any(np.asarray(min_rates) != 0))


# ------------------------------------------------------------------------ postprocessing
def _as_dev_f64(site: Site, rates) -> torch.Tensor:
    if isinstance(rates, torch.Tensor):
        return rates.to(device=torch.device("cuda", site.device), dtype=torch.float64).contiguous()
    return torch.from_numpy(np.ascontiguousarray(np.asarray(rates, dtype=np.float64))).to(torch.device("cuda", site.device))


def project_continuous(site: Site, rates) -> torch.Tensor:
    r = _as_dev_f64(site, rates)
    r3 = r if r.dim() == 3 else r.unsqueeze(0)
    out = torch.empty_like(r3)
    _cabi.check(_cabi.lib().acb_project_continuous(site.handle, _ptr(r3), _ptr(out), r3.shape[0], r3.shape[2], _stream_ptr(site.device)), "acb_project_continuous")
    return out if r.dim() == 3 else out[0]


def project_discrete(site: Site, rates) -> torch.Tensor:
    r = _as_dev_f64(site, rates)
    r3 = r if r.dim() == 3 else r.unsqueeze(0)
    out = torch.empty_like(r3)
    _cabi.check(_cabi.lib().acb_project_discrete(site.handle, _ptr(r3), _ptr(out), r3.shape[0], r3.shape[2], _stream_ptr(site.device)), "acb_project_discrete")
    return out if r.dim() == 3 else out[0]


def reallocate(site: Site, mode: int, rates, n_sessions, sess_row, sess_start, sess_ramp, sess_max0, order=None, peak_limit=None) -> torch.Tensor:
    """rates [B,N,T] float64; per-session arrays [B,S_max] (numpy).  Returns the device tensor."""
    dev = torch.device("cuda", site.device)
    r3 = _as_dev_f64(site, rates)
    B, _, T = r3.shape
    out = torch.empty_like(r3)

    def up(a, dt):
        return None if a is None else torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=dt))).to(dev)

    S_max = int(np.asarray(sess_row).shape[1])
    t = dict(ns=up(n_sessions, np.int32), row=up(sess_row, np.int32), st=up(sess_start, np.int32), ramp=up(sess_ramp, np.float64),
             mx=up(sess_max0, np.float64), order=up(order, np.int32), pk=up(peak_limit, np.float64))
    _cabi.check(
        _cabi.lib().acb_reallocate(site.handle, mode, _ptr(r3), _ptr(out), B, T, S_max, _ptr(t["ns"]), _ptr(t["row"]), _ptr(t["st"]),
                                   _ptr(t["ramp"]), _ptr(t["mx"]), _ptr(t["order"]), _ptr(t["pk"]), _stream_ptr(site.device)),
        "acb_reallocate",
    )
    return out


def constraints_feasible(site: Site, rates, col=0) -> torch.Tensor:
    r = _as_dev_f64(site, rates)
    r3 = r if r.dim() == 3 else r.unsqueeze(0)
    out = torch.empty((r3.shape[0],), dtype=torch.int32, device=r3.device)
    _cabi.check(_cabi.lib().acb_constraints_feasible(site.handle, _ptr(r3), r3.shape[0], r3.shape[2], col, _ptr(out), _stream_ptr(site.device)), "acb_constraints_feasible")
    return out


def min_rate_admission(site: Site, n_sessions, sess_row, try_rate) -> np.ndarray:
    """Batched greedy of apply_minimum_charging_rate: [B, S_max] arrays in offer order -> admitted flags (numpy bool)."""
    dev = torch.device("cuda", site.device)
    rows = np.ascontiguousarray(np.asarray(sess_row, dtype=np.int32))
    B, S_max = rows.shape
    t = dict(ns=torch.from_numpy(np.ascontiguousarray(np.asarray(n_sessions, dtype=np.int32))).to(dev), row=torch.from_numpy(rows).to(dev),
             tr=torch.from_numpy(np.ascontiguousarray(np.asarray(try_rate, dtype=np.float64))).to(dev))
    out = torch.zeros((B, S_max), dtype=torch.int32, device=dev)
    _cabi.check(_cabi.lib().acb_min_rate_admission(site.handle, B, S_max, _ptr(t["ns"]), _ptr(t["row"]), _ptr(t["tr"]), _ptr(out),
                                                   _stream_ptr(site.device)), "acb_min_rate_admission")
    return out.cpu().numpy().astype(bool)
