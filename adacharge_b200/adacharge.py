"""AdaptiveSchedulingAlgorithm / AdaptiveChargingAlgorithmOffline — the adapter of
reference adacharge/adacharge.py ("ada.py") re-hosted over the device path.  Control
flow, kwargs and error rules are the reference's; the arithmetic happens in
AdaptiveChargingOptimization.solve and the postprocessing kernels."""
from __future__ import annotations

import warnings
from copy import deepcopy

import numpy as np

from .algorithms_shim import BaseAlgorithm, apply_upper_bound_estimate, apply_minimum_charging_rate, enforce_pilot_limit
from .adaptive_charging_optimization import AdaptiveChargingOptimization
from .interface import SessionInfo
from .postprocessing import (
    project_into_continuous_feasible_pilots, project_into_discrete_feasible_pilots, diff_based_reallocation,
)


def get_active_sessions(active_evs, current_time):
    """List of SessionInfo for the currently charging EVs (ada.py:18-39)."""
    return [
        SessionInfo(ev.station_id, ev.session_id, ev.requested_energy, ev.energy_delivered, ev.arrival, ev.departure,
                    current_time=current_time)
        for ev in active_evs
    ]


def quantized_max_recompute(max_recompute, quantize, default=None):
    """The re-solve period that goes with `quantize` (ada.py:106-113): quantised pilots are recomputed every period, so
    with `quantize` it is 1, with the reference's warning when the caller asked for anything but `default`."""
    if not quantize:
        return max_recompute
    if max_recompute != default:
        warnings.warn("Overriding max_recompute to 1 since quantization is on.")
    return 1


class AdaptiveSchedulingAlgorithm(BaseAlgorithm):
    """MPC based adaptive scheduling algorithm (ada.py:42-193); same kwargs.
    ``solver`` is accepted and ignored; ``solver_options`` goes to the device solver."""

    def __init__(self, objective, constraint_type="SOC", enforce_energy_equality=False, solver=None, peak_limit=None,
                 estimate_max_rate=False, max_rate_estimator=None, uninterrupted_charging=False, quantize=False,
                 reallocate=False, max_recompute=None, allow_overcharging=False, verbose=False, solver_options=None):
        super().__init__()
        self.objective = objective
        self.constraint_type = constraint_type
        self.enforce_energy_equality = enforce_energy_equality
        self.solver = solver
        self.peak_limit = peak_limit
        self.estimate_max_rate = estimate_max_rate
        self.max_rate_estimator = max_rate_estimator
        self.uninterrupted_charging = uninterrupted_charging
        self.quantize = quantize
        self.reallocate = reallocate
        self.verbose = verbose
        self.solver_options = solver_options
        if not self.quantize and self.reallocate:  # ada.py:101-105
            raise ValueError("reallocate cannot be true without quantize. Otherwise there is nothing to reallocate :).")
        self.max_recompute = quantized_max_recompute(max_recompute, self.quantize)
        self.allow_overcharging = allow_overcharging

    def register_interface(self, interface):
        self._interface = interface
        if self.max_rate_estimator is not None:
            self.max_rate_estimator.register_interface(interface)

    def schedule(self, active_sessions):
        """See BaseAlgorithm (ada.py:135-193)."""
        if len(active_sessions) == 0:
            return {}
        infrastructure = self.interface.infrastructure_info()
        active_sessions = enforce_pilot_limit(active_sessions, infrastructure)
        if self.estimate_max_rate:
            active_sessions = apply_upper_bound_estimate(self.max_rate_estimator, active_sessions)
        if self.uninterrupted_charging:
            active_sessions = apply_minimum_charging_rate(active_sessions, infrastructure, self.interface.period)
        optimizer = AdaptiveChargingOptimization(
            self.objective, self.interface, self.constraint_type, self.enforce_energy_equality, solver=self.solver,
            solver_options=self.solver_options,
        )
        if self.peak_limit is None or np.isscalar(self.peak_limit):
            trimmed_peak = self.peak_limit
        else:
            t = self.interface.current_time
            horizon = max(s.arrival_offset + s.remaining_time for s in active_sessions)
            trimmed_peak = self.peak_limit[t : t + horizon]
        rates_matrix = optimizer.solve(
            active_sessions, infrastructure, peak_limit=trimmed_peak, prev_peak=self.interface.get_prev_peak(), verbose=self.verbose,
        )
        if self.quantize:
            if self.reallocate:
                rates_matrix = diff_based_reallocation(rates_matrix, active_sessions, infrastructure, self.interface)
            else:
                rates_matrix = project_into_discrete_feasible_pilots(rates_matrix, infrastructure)
        else:
            rates_matrix = project_into_continuous_feasible_pilots(rates_matrix, infrastructure)
        rates_matrix = np.maximum(rates_matrix, 0)
        return {station_id: rates_matrix[i, :] for i, station_id in enumerate(infrastructure.station_ids)}


class AdaptiveChargingAlgorithmOffline(BaseAlgorithm):
    """Offline optimisation with perfect future information (ada.py:196-294)."""

    def __init__(self, objective, constraint_type="SOC", enforce_energy_equality=False, solver=None, peak_limit=None,
                 verbose=False, solver_options=None):
        super().__init__()
        self.max_recompute = 1
        self.objective = objective
        self.constraint_type = constraint_type
        self.enforce_energy_equality = enforce_energy_equality
        self.solver = solver
        self.peak_limit = peak_limit
        self.verbose = verbose
        self.solver_options = solver_options
        self.sessions = None
        self.session_ids = None
        self.internal_schedule = None

    def register_events(self, events):
        """Only Plugin events are considered (ada.py:234-247)."""
        active_evs = [deepcopy(event[1].ev) for event in events.queue if event[1].event_type == "Plugin"]
        self.sessions = get_active_sessions(active_evs, 0)
        self.session_ids = set(s.session_id for s in self.sessions)

    def solve(self):
        if self._interface is None:
            raise ValueError("Error: self.interface is None. Please register interface before calling solve.")
        if self.sessions is None:
            raise ValueError("No events registered. Please register an event queue before calling solve.")
        infrastructure = self.interface.infrastructure_info()
        self.sessions = enforce_pilot_limit(self.sessions, infrastructure)
        optimizer = AdaptiveChargingOptimization(
            self.objective, self.interface, self.constraint_type, self.enforce_energy_equality, solver=self.solver,
            solver_options=self.solver_options,
        )
        rates_matrix = optimizer.solve(self.sessions, infrastructure, self.peak_limit, verbose=self.verbose)
        rates_matrix = project_into_continuous_feasible_pilots(rates_matrix, infrastructure)
        self.internal_schedule = {station_id: rates_matrix[i, :] for i, station_id in enumerate(infrastructure.station_ids)}

    def schedule(self, active_evs):
        if self.internal_schedule is None:
            raise ValueError("No internal schedule found. Make sure to call solve before calling schedule or running a simulation.")
        for ev in active_evs:
            if ev.session_id not in self.session_ids:
                raise ValueError(f"Error: Session {ev.session_id} not included in offline solve.")
        current_time = self.interface.current_time
        return {ev.station_id: [self.internal_schedule[ev.station_id][current_time]] for ev in active_evs}


__all__ = ["get_active_sessions", "AdaptiveSchedulingAlgorithm", "AdaptiveChargingAlgorithmOffline"]
