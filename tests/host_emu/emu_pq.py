"""TEST INFRASTRUCTURE: the host emulation of the solve with specified reactive power (gfr_emu_pq.cpp: the SPEC_Q
variants of the tree Newton and of the sweep on 1 - 16 emulated lanes), built with the flags of
tests/host_emu/build.py into tests/host_emu/_build/libgfr_emu_pq.so."""
import ctypes as C
import os
import subprocess

import numpy as np

from grid_fed_rl_b200 import _native as nat
from grid_fed_rl_b200.topology import compile_for_solver

from . import build as emu_build
from .emu import EMU_LANES

SRC = os.path.join(emu_build.HERE, "gfr_emu_pq.cpp")
OUT = os.path.join(emu_build.OUT_DIR, "libgfr_emu_pq.so")
_LIB = None


def build() -> str:
    os.makedirs(emu_build.OUT_DIR, exist_ok=True)
    deps = [SRC] + emu_build.DEPENDS[1:]
    if os.path.exists(OUT) and all(os.path.getmtime(d) <= os.path.getmtime(OUT) for d in deps):
        return OUT
    cmd = ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=fast", "-pthread",
           "-fvisibility-inlines-hidden", "-Wl,-Bsymbolic", "-DGFR_WIDE_GROUP_MIN_LANES=8", "-o", OUT, SRC, "-lm"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("g++ failed:\n" + res.stdout + res.stderr)
    return OUT


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.emu_solve_pq.argtypes = [C.POINTER(nat.FeederDesc), C.c_longlong, C.c_void_p, C.c_void_p,
                                   C.POINTER(nat.SolverCfg), C.POINTER(nat.SolOut)]
        _LIB = L
    return _LIB


def emu_solve_pq(feeder, p_inj, q_inj, solver="newton", tolerance=1e-6, max_iterations=50, lanes=0, emu_lanes=None,
                 acceleration=1.0):
    """The Q kernels' solve of ``p_inj`` / ``q_inj`` [B, n] (pu, ``feeder.buses`` order) on the host; same arguments
    and result dict as ``emu.emu_solve``, and the acceleration factor of the Newton update."""
    soa, used = compile_for_solver(feeder, solver, lanes, with_components=False)
    if emu_lanes is None:
        emu_lanes = used if used in EMU_LANES else 1
    desc, keep = nat.make_feeder_desc(soa)
    p = np.ascontiguousarray(np.atleast_2d(p_inj), dtype=np.float64)
    q = np.ascontiguousarray(np.broadcast_to(np.atleast_2d(q_inj), p.shape), dtype=np.float64)
    B, n, m = p.shape[0], soa.n_bus, soa.n_line
    out = dict(converged=np.zeros(B, np.uint8), iterations=np.zeros(B, np.int32),
               bus_voltages=np.zeros((B, n)), bus_angles=np.zeros((B, n)), line_flows=np.zeros((B, m)),
               line_loadings=np.zeros((B, m)), losses=np.zeros(B), max_mismatch=np.zeros(B))
    so = nat.SolOut(*[out[k].ctypes.data for k, _ in nat.SolOut._fields_])
    cfg = nat.make_solver_cfg(solver, tolerance, max_iterations, acceleration, lanes=emu_lanes)
    rc = lib().emu_solve_pq(C.byref(desc), B, p.ctypes.data, q.ctypes.data, C.byref(cfg), C.byref(so))
    assert rc == 0
    return out
