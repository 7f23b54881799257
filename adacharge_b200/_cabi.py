"""ctypes binding of libadacharge_b200.so (include/adacharge_b200.h).

There is no CPU fallback: if the shared library is missing every entry point raises
``NativeLibraryMissing`` with the build command.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libadacharge_b200.so")

ACB_SOC, ACB_LINEAR = 0, 1
ACB_SOLVED, ACB_MAX_ITER, ACB_INFEASIBLE, ACB_NUMERICAL, ACB_INVALID = 0, 1, 2, 3, 4
ACB_NSTATS = 8
ACB_PILOTS_DISCRETE, ACB_PILOTS_REALLOCATE = 1, 2  # acb_quantize_pilots modes
EXPORTS = [
    "acb_site_create", "acb_site_destroy", "acb_site_dims", "acb_site_max_horizon", "acb_default_options",
    "acb_solve_batch", "acb_charging_rate_bounds", "acb_project_continuous", "acb_project_discrete",
    "acb_reallocate", "acb_quantize_pilots", "acb_constraints_feasible", "acb_min_rate_admission", "acb_pack_sessions", "acb_preprocess_sessions", "acb_fleet_sessions", "acb_fleet_apply", "acb_last_error", "acb_version",
]
ACB_MAX_COMPONENTS = 16
# acb_objective.kind values (include/adacharge_b200.h)
OBJ_KIND = {"quick_charge": 0, "equal_share": 1, "tou_energy_cost": 2, "total_energy": 3, "peak": 4, "demand_charge": 5,
            "load_flattening": 6, "non_completion_penalty": 7, "non_completion_penalty_l2": 8}


class NativeLibraryMissing(RuntimeError):
    pass


class Options(C.Structure):
    _fields_ = [
        ("eps_abs", C.c_float), ("eps_rel", C.c_float), ("viol_tol", C.c_float), ("viol_abs", C.c_float), ("rho0", C.c_float),
        ("kappa", C.c_float), ("alpha", C.c_float), ("max_iter", C.c_int32), ("check_every", C.c_int32),
        ("equality", C.c_int32), ("adapt_rho", C.c_int32), ("restart", C.c_int32), ("avg_every", C.c_int32), ("stall_checks", C.c_int32), ("max_rescues", C.c_int32), ("path", C.c_int32), ("stall_exit", C.c_int32), ("dual_refine", C.c_int32), ("term_floor", C.c_float), ("rho_curv", C.c_float),
        ("rate_tol", C.c_float), ("polish_min_qd", C.c_float), ("newton_rel", C.c_float), ("phase_iters", C.c_int32),
    ]


_P = C.c_void_p


class Batch(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("Tp", C.c_int32), ("S_max", C.c_int32), ("multi_session", C.c_int32), ("lb_zero", C.c_int32),
        ("T", _P), ("n_sessions", _P), ("sess_row", _P), ("sess_start", _P), ("sess_len", _P),
        ("sess_energy", _P), ("sess_rate_off", _P), ("min_rates", _P), ("max_rates", _P),
        ("alpha", _P), ("beta", _P), ("qd", _P), ("gamma", _P), ("ext", _P), ("peak_w", _P), ("peak_p0", _P),
        ("peak_limit", _P), ("sess_quad", _P), ("work", _P),
        ("warm_v1", _P), ("warm_vc", _P), ("warm_mu", _P), ("warm_scal", _P), ("warm_shift", C.c_int32), ("warm_had", _P),
        ("out_v1", _P), ("out_vc", _P), ("out_mu", _P), ("out_scal", _P),
        ("rates", _P), ("pilots", _P), ("rate_est", _P), ("status", _P), ("iters", _P), ("stats", _P),
    ]


class Sessions(C.Structure):
    _fields_ = [("B", C.c_int32), ("S_max", C.c_int32), ("station", _P), ("arrival_offset", _P), ("remaining_time", _P),
                ("remaining_demand", _P), ("min_rate", _P), ("max_rate", _P)]


class Objective(C.Structure):
    _fields_ = [("n", C.c_int32), ("kind", C.c_int32 * ACB_MAX_COMPONENTS), ("coef", C.c_double * ACB_MAX_COMPONENTS),
                ("param", C.c_double * ACB_MAX_COMPONENTS), ("period", C.c_double), ("prices", _P), ("prices_stride", C.c_int32),
                ("prev_peak", _P), ("demand_charge", _P), ("demand_charge_scalar", C.c_double), ("external_signal", _P),
                ("ext_stride", C.c_int32), ("peak_limit", _P), ("pl_stride", C.c_int32)]


class Fleet(C.Structure):
    _fields_ = [("n_sites", C.c_int32), ("n_ev", C.c_int32), ("days", C.c_int32), ("steps_per_day", C.c_int32), ("ev_station", _P), ("ev_arr", _P),
                ("ev_dep", _P), ("ev_req", _P), ("ev_max", _P), ("ev_dlv", _P), ("ev_mu", _P), ("day_site_off", _P), ("prev_peak", _P), ("had", _P)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryMissing(
            f"{LIB_PATH} not found: build it with `make -C {os.path.join(_HERE, 'csrc')}` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback."
        )
    L = C.CDLL(LIB_PATH)
    L.acb_last_error.restype = C.c_char_p
    L.acb_site_create.argtypes = [C.POINTER(_P), C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P]
    L.acb_site_destroy.argtypes = [_P]
    L.acb_site_destroy.restype = None
    L.acb_site_dims.argtypes = [_P] + [C.POINTER(C.c_int)] * 5
    L.acb_site_max_horizon.argtypes = [_P]
    L.acb_default_options.argtypes = [C.POINTER(Options)]
    L.acb_default_options.restype = None
    L.acb_solve_batch.argtypes = [_P, C.POINTER(Batch), C.POINTER(Options), _P]
    L.acb_charging_rate_bounds.argtypes = [_P, C.POINTER(Batch), _P, _P, _P]
    L.acb_project_continuous.argtypes = [_P, _P, _P, C.c_int, C.c_int, _P]
    L.acb_project_discrete.argtypes = [_P, _P, _P, C.c_int, C.c_int, _P]
    L.acb_reallocate.argtypes = [_P, C.c_int, _P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P]
    L.acb_quantize_pilots.argtypes = [_P, C.c_int, C.POINTER(Sessions), C.c_double, C.POINTER(Batch), _P, _P]
    L.acb_constraints_feasible.argtypes = [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P]
    L.acb_min_rate_admission.argtypes = [_P, C.c_int, C.c_int, _P, _P, _P, _P, _P]
    L.acb_preprocess_sessions.argtypes = [_P, C.POINTER(Sessions), C.c_int, _P, _P]
    L.acb_fleet_sessions.argtypes = [_P, C.POINTER(Fleet), C.c_int, C.POINTER(Sessions), _P, _P, _P]
    L.acb_fleet_apply.argtypes = [_P, C.POINTER(Fleet), C.c_int, C.c_double, C.POINTER(Batch), _P, _P, _P, _P]
    L.acb_pack_sessions.argtypes = [_P, C.POINTER(Sessions), C.POINTER(Objective), C.POINTER(Batch), _P, _P]
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().acb_last_error().decode()
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise RuntimeError(f"{what} failed ({rc}): {msg}")


def copy_options(o: Options, **over) -> Options:
    c = Options.from_buffer_copy(o)
    for k, v in over.items():
        setattr(c, k, v)
    return c


def default_options(**over) -> Options:
    o = Options()
    lib().acb_default_options(C.byref(o))
    for k, v in over.items():
        if not hasattr(o, k):
            raise TypeError(f"unknown solver option {k!r}")
        setattr(o, k, v)
    return o
