"""ctypes binding of the C ABI in ``include/gfr_b200.h`` (``libgfr_b200.so``).

The library is the product path: there is no Python / CPU fallback.  ``load_library`` raises if
the shared object has not been built (``python -m grid_fed_rl_b200.build`` or
``__graft_entry__.build()``), and every entry point returns ``GFR_E_CUDA`` without a device.
"""

from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Tuple

import numpy as np

from .topology import FeederSoA

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgfr_b200.so")

GFR_OK, GFR_E_ARG, GFR_E_CUDA, GFR_E_LIMIT = 0, -1, -2, -3
SOLVER_SWEEP, SOLVER_NEWTON = 0, 1
SOLVERS = {"sweep": SOLVER_SWEEP, "newton": SOLVER_NEWTON, "newton_raphson": SOLVER_NEWTON}
BUS_SLACK, BUS_PV, BUS_PQ = 0, 1, 2
OBS_F64, OBS_F32 = 0, 1

_i32p, _f64p, _u8p, _u64p = C.POINTER(C.c_int32), C.POINTER(C.c_double), C.POINTER(C.c_uint8), C.POINTER(C.c_uint64)


class FeederDesc(C.Structure):
    _fields_ = [
        ("n_bus", C.c_int32), ("n_levels", C.c_int32), ("n_load", C.c_int32), ("n_gen", C.c_int32),
        ("n_bat", C.c_int32), ("n_pool", C.c_int32), ("lanes_hint", C.c_int32), ("n_tie", C.c_int32),
        ("s_base", C.c_double),
        ("order", _i32p), ("parent", _i32p), ("level_ptr", _i32p), ("child_ptr", _i32p),
        ("child_idx", _i32p), ("lane_of", _i32p),
        ("bus_type", _i32p), ("vm_set", _f64p), ("g", _f64p), ("b", _f64p), ("gdiag", _f64p),
        ("bdiag", _f64p), ("r", _f64p), ("x", _f64p), ("line_of", _i32p), ("from_is_parent", _i32p),
        ("rating", _f64p), ("load_bus", _i32p), ("load_base", _f64p), ("load_p", _f64p),
        ("load_q", _f64p), ("gen_type", _i32p), ("gen_bus", _i32p), ("gen_cap", _f64p),
        ("gen_p0", _f64p), ("gen_p1", _f64p), ("gen_p2", _f64p), ("bat_bus", _i32p),
        ("bat_cap", _f64p), ("bat_rating", _f64p), ("bat_eff", _f64p), ("bat_soc0", _f64p),
        ("load_profile", _f64p),
        ("tie_line", _i32p), ("tie_from", _i32p), ("tie_to", _i32p), ("tie_r", _f64p), ("tie_x", _f64p),
        ("tie_rating", _f64p), ("tie_zinv", _f64p),
    ]


class NetworkDesc(C.Structure):
    _fields_ = [("n_bus", C.c_int32), ("n_line", C.c_int32), ("s_base", C.c_double),
                ("bus_type", _i32p), ("vm_set", _f64p), ("line_from", _i32p), ("line_to", _i32p),
                ("line_r", _f64p), ("line_x", _f64p), ("line_rating", _f64p)]


class SolverCfg(C.Structure):
    _fields_ = [("solver", C.c_int32), ("max_iterations", C.c_int32), ("tolerance", C.c_double),
                ("acceleration", C.c_double), ("lanes", C.c_int32), ("reserved", C.c_int32)]


class EnvCfg(C.Structure):
    _fields_ = [("timestep", C.c_double), ("episode_length", C.c_int32),
                ("stochastic_loads", C.c_int32), ("weather_variation", C.c_int32),
                ("reserved", C.c_int32), ("v_min", C.c_double), ("v_max", C.c_double),
                ("f_min", C.c_double), ("f_max", C.c_double), ("safety_penalty", C.c_double),
                ("load_noise", C.c_double), ("solver", SolverCfg), ("env_id_offset", C.c_int64)]


class StepOut(C.Structure):
    _fields_ = [("reward", C.c_void_p), ("terminated", C.c_void_p), ("truncated", C.c_void_p),
                ("error", C.c_void_p), ("converged", C.c_void_p), ("iterations", C.c_void_p),
                ("max_voltage", C.c_void_p), ("min_voltage", C.c_void_p), ("losses", C.c_void_p),
                ("max_mismatch", C.c_void_p), ("violations", C.c_void_p),
                ("violation_count", C.c_void_p), ("current_step", C.c_void_p),
                ("episode_reward", C.c_void_p), ("noise_used", C.c_void_p)]


class SolOut(C.Structure):
    _fields_ = [("converged", C.c_void_p), ("iterations", C.c_void_p), ("bus_voltages", C.c_void_p),
                ("bus_angles", C.c_void_p), ("line_flows", C.c_void_p), ("line_loadings", C.c_void_p),
                ("losses", C.c_void_p), ("max_mismatch", C.c_void_p)]


# every exported symbol with its signature (tests check the library exports all of them)
SIGNATURES: Dict[str, Tuple[object, List[object]]] = {
    "gfr_abi_version": (C.c_int, []),
    "gfr_last_error": (C.c_char_p, []),
    "gfr_feeder_create": (C.c_int, [C.POINTER(FeederDesc), C.c_int, C.POINTER(C.c_void_p)]),
    "gfr_feeder_destroy": (None, [C.c_void_p]),
    "gfr_env_create": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(EnvCfg), C.POINTER(C.c_void_p)]),
    "gfr_env_destroy": (None, [C.c_void_p]),
    "gfr_env_num_envs": (C.c_int64, [C.c_void_p]),
    "gfr_env_obs_dim": (C.c_int, [C.c_void_p]),
    "gfr_env_act_dim": (C.c_int, [C.c_void_p]),
    "gfr_env_noise_dim": (C.c_int, [C.c_void_p]),
    "gfr_env_obs": (C.c_void_p, [C.c_void_p]),
    "gfr_env_bind_obs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gfr_env_bind_obs_buffers": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "gfr_env_obs_current": (C.c_void_p, [C.c_void_p]),
    "gfr_env_obs_to_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "gfr_env_launch_info": (C.c_int, [C.c_void_p, _i32p, _i32p, _i32p, C.POINTER(C.c_int64)]),
    "gfr_env_state_bytes": (C.c_int64, [C.c_void_p]),
    "gfr_env_state_get": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gfr_env_state_set": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gfr_env_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]),
    "gfr_env_reset_outputs": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(StepOut), C.c_void_p]),
    "gfr_env_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(StepOut), C.c_void_p]),
    "gfr_solve": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(SolverCfg), C.POINTER(SolOut), C.c_void_p]),
    "gfr_solve_pq": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.POINTER(SolverCfg), C.POINTER(SolOut),
                               C.c_void_p]),
    "gfr_network_create": (C.c_int, [C.POINTER(NetworkDesc), C.c_int, C.POINTER(C.c_void_p)]),
    "gfr_network_destroy": (None, [C.c_void_p]),
    "gfr_network_unknowns": (C.c_int, [C.c_void_p]),
    "gfr_network_solve": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(SolverCfg), C.POINTER(SolOut), C.c_void_p]),
    "gfr_network_solve_pq": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.POINTER(SolverCfg),
                                       C.POINTER(SolOut), C.c_void_p]),
    "gfr_noise_fill": (C.c_int, [C.c_int, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gfr_fp64_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    "gfr_launch_count": (C.c_int64, []),
    "gfr_auto_lanes": (C.c_int, [C.c_int, C.c_int, C.c_int]),
}

_LIB = None


class NativeLibraryMissing(RuntimeError):
    pass


def load_library(path: str = LIB_PATH) -> C.CDLL:
    """Load ``libgfr_b200.so`` (once).  torch is imported first so that both share one CUDA runtime."""
    global _LIB
    if _LIB is not None and path == LIB_PATH:
        return _LIB
    if not os.path.exists(path):
        raise NativeLibraryMissing(
            f"{path} is missing: build it with `python -m grid_fed_rl_b200.build` "
            "(nvcc, sm_100a).  grid_fed_rl_b200 has no CPU fallback.")
    import torch  # noqa: F401  (loads libcudart / libc10_cuda before ours)
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.gfr_abi_version() != 1:
        raise RuntimeError("libgfr_b200.so has an unexpected ABI version")
    if path == LIB_PATH:
        _LIB = lib
    return lib


def check(lib: C.CDLL, rc: int) -> None:
    if rc != GFR_OK:
        msg = lib.gfr_last_error().decode("utf-8", "replace")
        from .errors import GridLimitError, InvalidConfigurationError, NativeRuntimeError
        exc = {GFR_E_ARG: InvalidConfigurationError, GFR_E_LIMIT: GridLimitError}.get(rc, NativeRuntimeError)
        raise exc(f"libgfr_b200 ({rc}): {msg}")


def _ptr(arr: np.ndarray, ctype):
    return arr.ctypes.data_as(C.POINTER(ctype))


def make_network_desc(buses, lines, s_base: float):
    """``gfr_network_desc`` from the reference's ``List[Bus]`` / ``List[Line]`` (their order is kept)
    + the numpy arrays that must outlive it.  No radiality requirement."""
    index = {b.id: i for i, b in enumerate(buses)}
    tmap = {"slack": BUS_SLACK, "pv": BUS_PV}
    keep = dict(
        bus_type=np.array([tmap.get(b.bus_type, BUS_PQ) for b in buses], dtype=np.int32),
        vm_set=np.array([float(b.voltage_magnitude) for b in buses], dtype=np.float64),
        line_from=np.array([index[l.from_bus] for l in lines], dtype=np.int32),
        line_to=np.array([index[l.to_bus] for l in lines], dtype=np.int32),
        line_r=np.array([float(l.resistance) for l in lines], dtype=np.float64),
        line_x=np.array([float(l.reactance) for l in lines], dtype=np.float64),
        line_rating=np.array([float(l.rating) for l in lines], dtype=np.float64))
    d = NetworkDesc()
    d.n_bus, d.n_line, d.s_base = len(buses), len(lines), float(s_base)
    for k, a in keep.items():
        setattr(d, k, _ptr(a, C.c_int32 if a.dtype == np.int32 else C.c_double))
    return d, keep


def make_feeder_desc(soa: FeederSoA):
    """``gfr_feeder_desc`` for a compiled feeder + the numpy arrays that must outlive it."""
    keep: Dict[str, np.ndarray] = {}

    def i32(name):
        a = np.ascontiguousarray(getattr(soa, name), dtype=np.int32)
        if a.size == 0:
            a = np.zeros(1, dtype=np.int32)
        keep[name] = a
        return _ptr(a, C.c_int32)

    def f64(name):
        a = np.ascontiguousarray(getattr(soa, name), dtype=np.float64)
        if a.size == 0:
            a = np.zeros(1, dtype=np.float64)
        keep[name] = a
        return _ptr(a, C.c_double)

    d = FeederDesc()
    d.n_bus, d.n_levels, d.n_load, d.n_gen, d.n_bat = (soa.n_bus, soa.n_levels, soa.n_load,
                                                      soa.n_gen, soa.n_bat)
    d.n_pool = int(soa.n_pool)
    d.lanes_hint = int(getattr(soa, "lanes_hint", 0) or 0)
    d.s_base = float(soa.s_base)
    for name in ("order", "parent", "level_ptr", "child_ptr", "child_idx", "bus_type", "line_of", "from_is_parent",
                 "load_bus", "gen_type", "gen_bus", "bat_bus"):
        setattr(d, name, i32(name))
    if getattr(soa, "lane_of", None) is not None:        # optional: NULL = position inside the level
        d.lane_of = i32("lane_of")
    d.n_tie = int(getattr(soa, "n_tie", 0))
    if d.n_tie:
        for name in ("tie_line", "tie_from", "tie_to"):
            setattr(d, name, i32(name))
        for name in ("tie_r", "tie_x", "tie_rating", "tie_zinv"):
            setattr(d, name, f64(name))
    for name in ("vm_set", "g", "b", "gdiag", "bdiag", "r", "x", "rating", "load_base", "load_p",
                 "load_q", "gen_cap", "gen_p0", "gen_p1", "gen_p2", "bat_cap", "bat_rating",
                 "bat_eff", "bat_soc0", "load_profile"):
        setattr(d, name, f64(name))
    return d, keep


def make_solver_cfg(solver: str = "newton", tolerance: float = 1e-6, max_iterations: int = 50,
                    acceleration: float = 1.0, lanes: int = 0) -> SolverCfg:
    if solver not in SOLVERS:
        from .errors import InvalidConfigurationError
        raise InvalidConfigurationError(f"solver must be one of {sorted(SOLVERS)}, got {solver!r}")
    return SolverCfg(SOLVERS[solver], int(max_iterations), float(tolerance), float(acceleration),
                     int(lanes), 0)


def make_env_cfg(*, timestep=1.0, episode_length=86400, stochastic_loads=True,
                 weather_variation=True, voltage_limits=(0.95, 1.05), frequency_limits=(59.5, 60.5),
                 safety_penalty=100.0, load_noise=0.1, solver_cfg: SolverCfg,
                 env_id_offset: int = 0) -> EnvCfg:
    return EnvCfg(float(timestep), int(episode_length), int(bool(stochastic_loads)),
                  int(bool(weather_variation)), 0, float(voltage_limits[0]), float(voltage_limits[1]),
                  float(frequency_limits[0]), float(frequency_limits[1]), float(safety_penalty),
                  float(load_noise), solver_cfg, int(env_id_offset))
