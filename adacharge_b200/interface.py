"""Data carriers the MPC path reads: SessionInfo / InfrastructureInfo / Interface.

The reference takes these from acnportal (``from acnportal.acnsim.interface import
Interface, SessionInfo, InfrastructureInfo`` — reference
adacharge/adaptive_charging_optimization.py:5).  acnportal is not vendored in the
reference and is not installed in this image, so this module provides stand-ins with
exactly the attributes the hot path reads (SURVEY.md §8(b) "fields read").  When
acnportal *is* importable its own classes are used unchanged, and everything in
adacharge_b200 works on them by duck typing.

Behaviour recalled from public acnportal 0.3.x ("[acnportal, recalled]"); the way
the reference *uses* each field is cited per attribute.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np

try:  # pragma: no cover - acnportal is absent in this image
    from acnportal.acnsim.interface import (  # type: ignore
        Interface,
        SessionInfo,
        InfrastructureInfo,
    )

    HAVE_ACNPORTAL = True
except Exception:  # noqa: BLE001
    HAVE_ACNPORTAL = False

    class SessionInfo:
        """One active charging session.

        Constructed by the reference as ``SessionInfo(station_id, session_id,
        requested_energy, energy_delivered, arrival, departure, current_time=...)``
        (reference adacharge/adacharge.py:29-37).  Fields read on the path:
        station_id/session_id (aco.py:63,115), arrival_offset, remaining_time,
        min_rates, max_rates (aco.py:62-73), remaining_demand (aco.py:118-122).
        """

        def __init__(
            self,
            station_id: str,
            session_id: str,
            requested_energy: float,
            energy_delivered: float,
            arrival: int,
            departure: int,
            estimated_departure: Optional[int] = None,
            current_time: int = 0,
            min_rates=0,
            max_rates=float("inf"),
        ):
            self.station_id = station_id
            self.session_id = session_id
            self.requested_energy = requested_energy
            self.energy_delivered = energy_delivered
            self.arrival = arrival
            self.departure = departure
            self.estimated_departure = (
                estimated_departure if estimated_departure is not None else departure
            )
            self.current_time = current_time
            rt = self.remaining_time
            self.min_rates = (
                np.full(rt, float(min_rates))
                if np.isscalar(min_rates)
                else np.array(min_rates, dtype=float)
            )
            self.max_rates = (
                np.full(rt, float(max_rates))
                if np.isscalar(max_rates)
                else np.array(max_rates, dtype=float)
            )

        @property
        def remaining_demand(self) -> float:
            return self.requested_energy - self.energy_delivered

        @property
        def arrival_offset(self) -> int:
            return int(max(self.arrival - self.current_time, 0))

        @property
        def remaining_time(self) -> int:
            return int(
                max(
                    min(
                        self.departure - self.arrival,
                        self.departure - self.current_time,
                    ),
                    0,
                )
            )

    class InfrastructureInfo:
        """Electrical description of a site.

        Fields read on the path: station_ids (aco.py:246,253), num_stations
        (aco.py:311, pp.py:91), get_station_index (aco.py:106, pp.py:148), voltages
        (aco.py:114,338,390), constraint_matrix M x N (aco.py:146-157), phases in
        degrees (aco.py:152-156), constraint_limits (aco.py:163), constraint_ids
        (aco.py:160), max_pilot (pp.py:92,162), allowable_pilots ragged (pp.py:114,176).
        """

        def __init__(
            self,
            constraint_matrix,
            constraint_limits,
            phases,
            voltages,
            constraint_ids: List[str],
            station_ids: List[str],
            max_pilot,
            min_pilot,
            allowable_pilots=None,
            is_continuous=None,
        ):
            self.constraint_matrix = (
                None if constraint_matrix is None else np.asarray(constraint_matrix)
            )
            self.constraint_limits = np.asarray(constraint_limits)
            self.phases = None if phases is None else np.asarray(phases)
            self.voltages = np.asarray(voltages)
            self.constraint_ids = list(constraint_ids)
            self.station_ids = list(station_ids)
            self._station_ids_dict = {sid: i for i, sid in enumerate(self.station_ids)}
            self.max_pilot = np.asarray(max_pilot)
            self.min_pilot = np.asarray(min_pilot)
            if allowable_pilots is None:
                allowable_pilots = [None] * self.num_stations
            self.allowable_pilots = allowable_pilots
            if is_continuous is None:
                is_continuous = np.ones(self.num_stations, dtype=bool)
            self.is_continuous = np.asarray(is_continuous)

        @property
        def num_stations(self) -> int:
            return len(self.station_ids)

        def get_station_index(self, station_id: str) -> int:
            return self._station_ids_dict[station_id]

    class Interface:
        """Minimal base: what the algorithm may ask of its environment."""

        period: float = 5
        current_time: int = 0

        def active_sessions(self) -> List[SessionInfo]:
            raise NotImplementedError

        def infrastructure_info(self) -> InfrastructureInfo:
            raise NotImplementedError

        def get_prices(self, length: int, start: Optional[int] = None):
            raise NotImplementedError

        def get_demand_charge(self, start: Optional[int] = None) -> float:
            raise NotImplementedError

        def get_prev_peak(self) -> float:
            raise NotImplementedError

        def remaining_amp_periods(self, session: SessionInfo) -> float:
            raise NotImplementedError


def infrastructure_from_dict(d: Dict) -> InfrastructureInfo:
    """InfrastructureInfo from its dict form (what the generators produce and TestingInterface holds)."""
    return InfrastructureInfo(
        np.array(d["constraint_matrix"]),
        np.array(d["constraint_limits"]),
        np.array(d["phases"]),
        np.array(d["voltages"]),
        d["constraint_ids"],
        d["station_ids"],
        np.array(d["max_pilot"]),
        np.array(d["min_pilot"]),
        d.get("allowable_pilots"),
        d.get("is_continuous"),
    )


class TestingInterface(Interface):
    """Dict-backed Interface used by the reference tests
    (``TestingInterface({...})`` — reference tests/test_adaptive_charging_optimization.py:31-39,
    tests/test_postprocessing.py:179-186).  [acnportal, recalled]

    Extra keys understood here (all optional): ``prices`` (vector indexed from
    ``current_time``), ``demand_charge``, ``prev_peak``.
    """

    __test__ = False  # not a pytest class

    def __init__(self, data: Dict):
        self.data = data

    @property
    def current_time(self) -> int:
        return self.data.get("current_time", 0)

    @property
    def period(self) -> float:
        return self.data["period"]

    def active_sessions(self) -> List[SessionInfo]:
        return [
            SessionInfo(current_time=self.current_time, **s)
            for s in self.data["active_sessions"]
        ]

    def infrastructure_info(self) -> InfrastructureInfo:
        return infrastructure_from_dict(self.data["infrastructure_info"])

    def get_prices(self, length: int, start: Optional[int] = None):
        if start is None:
            start = self.current_time
        p = np.asarray(self.data["prices"], dtype=float)
        return p[start : start + length]

    def get_demand_charge(self, start: Optional[int] = None) -> float:
        return self.data["demand_charge"]

    def get_prev_peak(self) -> float:
        return self.data.get("prev_peak", 0)

    def remaining_amp_periods(self, session: SessionInfo) -> float:
        """kWh -> A*periods at the session's EVSE voltage. [acnportal, recalled]"""
        infra = self.data["infrastructure_info"]
        i = list(infra["station_ids"]).index(session.station_id)
        voltage = np.asarray(infra["voltages"])[i]
        return session.remaining_demand * 1000 / voltage * (60 / self.period)


def earliest_deadline_first(sessions: List[SessionInfo], iface: Interface):
    """Sort key used by the reference's reallocation KATs
    (tests/test_postprocessing.py:14,190). [acnportal, recalled]"""
    return sorted(sessions, key=lambda s: s.estimated_departure)


__all__ = [
    "Interface",
    "SessionInfo",
    "InfrastructureInfo",
    "TestingInterface",
    "infrastructure_from_dict",
    "earliest_deadline_first",
    "HAVE_ACNPORTAL",
]
