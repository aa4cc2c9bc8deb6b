"""TEST INFRASTRUCTURE: ctypes wrapper of the host emulation of the device functions (a group of
1 - 16 lanes = as many host threads meeting at barriers).  Lets the CPU-only test tier exercise the
very same arithmetic, schedules and hand-offs the kernels run."""
import ctypes as C

import numpy as np

from grid_fed_rl_b200 import _native as nat
from grid_fed_rl_b200.topology import compile_feeder, compile_for_solver

from .build import build

_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.emu_create.restype = C.c_void_p
        L.emu_create.argtypes = [C.POINTER(nat.FeederDesc), C.c_longlong, C.POINTER(nat.EnvCfg)]
        L.emu_destroy.argtypes = [C.c_void_p]
        L.emu_obs.restype = C.POINTER(C.c_double)
        L.emu_obs.argtypes = [C.c_void_p]
        L.emu_obs_dim.argtypes = [C.c_void_p]
        L.emu_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double]
        L.emu_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(nat.StepOut)]
        L.emu_solve.argtypes = [C.POINTER(nat.FeederDesc), C.c_longlong, C.c_void_p,
                                C.POINTER(nat.SolverCfg), C.POINTER(nat.SolOut)]
        L.emu_noise_fill.argtypes = [C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.emu_schedule_info.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        _LIB = L
    return _LIB


EMU_LANES = (1, 2, 4, 8, 16)

STEP_FIELDS = dict(reward=np.float64, terminated=np.uint8, truncated=np.uint8, error=np.uint8,
                   converged=np.uint8, iterations=np.int32, max_voltage=np.float64,
                   min_voltage=np.float64, losses=np.float64, max_mismatch=np.float64,
                   violations=np.uint8, violation_count=np.int32, current_step=np.int32,
                   episode_reward=np.float64, noise_used=np.float64)


class EmuEnv:
    def __init__(self, feeder, num_envs=1, solver="newton", tolerance=1e-6, max_iterations=50,
                 renewable_sources=None, lanes=0, emu_lanes=None, **kw):
        """``lanes``: the lane count the feeder is compiled (scheduled) for, 0 = the auto rule.
        ``emu_lanes``: the lane count emulated (1, 2, 4, 8, 16); default = ``lanes`` when it is one of
        those, else 1 (the library then re-cuts the schedule for one lane)."""
        self.soa, used = compile_for_solver(feeder, solver, lanes, renewable_sources=renewable_sources)
        if emu_lanes is None:
            emu_lanes = used if used in EMU_LANES else 1
        self.emu_lanes = emu_lanes
        self.desc, self._keep = nat.make_feeder_desc(self.soa)
        scfg = nat.make_solver_cfg(solver, tolerance, max_iterations, lanes=emu_lanes)
        self.cfg = nat.make_env_cfg(solver_cfg=scfg, **kw)
        self.B = num_envs
        self.h = lib().emu_create(C.byref(self.desc), num_envs, C.byref(self.cfg))
        assert self.h, "emu_create failed"
        self.D = lib().emu_obs_dim(self.h)
        self.L = self.soa.n_load
        info = (C.c_int * 4)()
        lib().emu_schedule_info(self.h, info)
        self.schedule = dict(rows=info[0], positions=info[1], pool_slots=info[2], register_edges=info[3])

    def __del__(self):
        if getattr(self, "h", None):
            lib().emu_destroy(self.h)
            self.h = None

    def obs(self):
        return np.ctypeslib.as_array(lib().emu_obs(self.h), shape=(self.B, self.D)).copy()

    def reset(self, noise=None, seeds=None, mask=None, start_time=0.0):
        nz = None if noise is None else np.ascontiguousarray(noise, dtype=np.float64)[:, :4].copy()
        sd = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        mk = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        p = lambda a: None if a is None else a.ctypes.data
        lib().emu_reset(self.h, p(sd), p(mk), p(nz), float(start_time))
        return self.obs()

    def step(self, actions, noise=None):
        act = np.ascontiguousarray(actions, dtype=np.float64).reshape(self.B, -1)
        nz = None if noise is None else np.ascontiguousarray(noise, dtype=np.float64).reshape(self.B, 4 + self.L)
        out = {k: np.zeros((self.B, 4) if k == "violations" else ((self.B, 4 + self.L) if k == "noise_used" else self.B), dtype=t)
               for k, t in STEP_FIELDS.items()}
        so = nat.StepOut(*[out[k].ctypes.data for k, _ in nat.StepOut._fields_])
        lib().emu_step(self.h, act.ctypes.data, None if nz is None else nz.ctypes.data, C.byref(so))
        out["obs"] = self.obs()
        out["viol_count"] = out["violation_count"]
        return out


def emu_solve(feeder, p_inj, solver="newton", tolerance=1e-6, max_iterations=50, lanes=0, emu_lanes=None,
              acceleration=1.0):
    soa, used = compile_for_solver(feeder, solver, lanes, with_components=False)
    if emu_lanes is None:
        emu_lanes = used if used in EMU_LANES else 1
    desc, keep = nat.make_feeder_desc(soa)
    p = np.ascontiguousarray(np.atleast_2d(p_inj), dtype=np.float64)
    B, n, m = p.shape[0], soa.n_bus, soa.n_line
    out = dict(converged=np.zeros(B, np.uint8), iterations=np.zeros(B, np.int32),
               bus_voltages=np.zeros((B, n)), bus_angles=np.zeros((B, n)), line_flows=np.zeros((B, m)),
               line_loadings=np.zeros((B, m)), losses=np.zeros(B), max_mismatch=np.zeros(B))
    so = nat.SolOut(*[out[k].ctypes.data for k, _ in nat.SolOut._fields_])
    cfg = nat.make_solver_cfg(solver, tolerance, max_iterations, acceleration, lanes=emu_lanes)
    rc = lib().emu_solve(C.byref(desc), B, p.ctypes.data, C.byref(cfg), C.byref(so))
    assert rc == 0
    return out


def emu_noise(seeds, draws, n_slots):
    s = np.ascontiguousarray(seeds, dtype=np.uint64)
    d = np.ascontiguousarray(draws, dtype=np.uint64)
    out = np.zeros((s.size, n_slots))
    lib().emu_noise_fill(s.size, n_slots, s.ctypes.data, d.ctypes.data, out.ctypes.data)
    return out
