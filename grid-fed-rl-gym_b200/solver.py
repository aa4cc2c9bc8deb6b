"""``B200PowerFlowSolver`` - the reference's solver plugin surface on the CUDA path.

Reference (paths under /root/reference/grid_fed_rl/):
  * ``PowerFlowSolver.__init__(tolerance, max_iterations)`` + abstract
    ``solve(buses, lines, loads, generation) -> PowerFlowSolution``   environments/power_flow.py:28-46
  * ``NewtonRaphsonSolver`` defaults 1e-6 / 50, ``acceleration_factor``  environments/power_flow.py:79-87
  * the documented two-argument form ``solver.solve(feeder, loading_conditions)``
    (README.md:200, API_REFERENCE.md:407,429; never implemented upstream)

Both call shapes are accepted.  Quantities are taken in the units the caller uses, exactly
like the reference solver (which never converts): pass per-unit injections with per-unit
impedances.  The two-argument form with a ``{'loads': {bus: W}, 'generation': {bus: W}}`` dict
divides by the feeder's base power first (deviation D1, DESIGN.md).

Specified reactive power (the reference's ``Q_spec`` row, which it leaves at 0) goes in as ``q_inj``
[B, n] pu next to ``p_inj``, as a ``(p, q)`` tuple in place of ``p_inj``, or as ``'reactive_loads'`` /
``'reactive_generation'`` ({bus: var}) in the two-argument form's dict.  Q entries of the slack and of PV
buses are ignored.  The reference's four-argument form stays active power only, as its signature is.
"""

from __future__ import annotations

import ctypes as C
from typing import Any, Dict, Optional

import numpy as np
import torch

from . import _native as nat
from .components import FeederParameters, PowerFlowSolution
from .env import NativeFeeder, _cuda_device
from .errors import GridLimitError, InvalidConfigurationError, NetworkTopologyError
from .topology import FeederSoA, TopologyError, auto_lanes, compile_for_solver


class _Topology:
    """Just enough of a feeder for ``compile_feeder`` when only buses + lines are given."""

    def __init__(self, buses, lines, base_power_mva: float) -> None:
        self.name = "adhoc"
        self.buses, self.lines, self.loads, self.generators = list(buses), list(lines), [], {}
        self.parameters = FeederParameters(base_voltage=1.0, base_power=base_power_mva, frequency=60.0)


def _signature(buses, lines):
    return (tuple((b.id, b.bus_type, float(b.voltage_magnitude)) for b in buses),
            tuple((l.id, l.from_bus, l.to_bus, float(l.resistance), float(l.reactance), float(l.rating))
                  for l in lines))


class NativeNetwork:
    """A (possibly meshed) network resident on one device (``gfr_network``): buses and lines in the
    caller's order, solved by the dense Newton-Raphson kernel."""

    def __init__(self, buses, lines, s_base: float, device: torch.device) -> None:
        self.lib = nat.load_library()
        self.device = device
        self.n_bus, self.n_line = len(buses), len(lines)
        desc, self._keep = nat.make_network_desc(buses, lines, s_base)
        h = C.c_void_p()
        nat.check(self.lib, self.lib.gfr_network_create(C.byref(desc), device.index, C.byref(h)))
        self.handle = h
        self.unknowns = int(self.lib.gfr_network_unknowns(h))

    def close(self) -> None:
        if getattr(self, "handle", None):
            self.lib.gfr_network_destroy(self.handle)
            self.handle = None

    def __del__(self) -> None:
        try:
            self.close()
        except Exception:
            pass


def _injections(p_inj, q_inj, n: int, dev):
    """(p, q) as [B, n] float64 tensors on ``dev`` (q None when no reactive power is given); ``p_inj`` may be a
    ``(p, q)`` pair."""
    if q_inj is None and isinstance(p_inj, tuple) and len(p_inj) == 2:
        p_inj, q_inj = p_inj

    def one(x, name):
        t = torch.as_tensor(x)
        if t.dim() == 1:
            t = t[None, :]
        if t.dim() != 2 or t.shape[1] != n:
            raise InvalidConfigurationError(f"{name} must be [B, {n}], got {tuple(t.shape)}")
        return t.to(device=dev, dtype=torch.float64).contiguous()
    p = one(p_inj, "p_inj")
    if q_inj is None:
        return p, None
    q = one(q_inj, "q_inj")
    if q.shape != p.shape:
        raise InvalidConfigurationError(f"q_inj must have the shape of p_inj {tuple(p.shape)}, got {tuple(q.shape)}")
    return p, q


def is_radial(buses, lines) -> bool:
    """True when the lines form a spanning tree of the buses (what the tree-ordered kernels need)."""
    if len(lines) != len(buses) - 1:
        return False
    index = {b.id: i for i, b in enumerate(buses)}
    root = list(range(len(buses)))

    def find(a):
        while root[a] != a:
            root[a] = root[root[a]]
            a = root[a]
        return a
    for ln in lines:
        a, b = find(index[ln.from_bus]), find(index[ln.to_bus])
        if a == b:
            return False
        root[a] = b
    return True


class B200PowerFlowSolver:
    """Batched load flow on one GPU.  ``method`` is "newton" (the reference's polar Newton-Raphson
    iterates, solved by tree-ordered block elimination; radial feeders of any size), "sweep"
    (backward / forward sweep; radial, or weakly meshed with the loops restored by the compensation
    method: one current per loop-closing line, corrected every iteration), "dense" (the same Newton-Raphson on the dense Jacobian,
    eliminated with partial pivoting by one CTA per instance: any connected network, cycles
    included, up to ~80 buses; ``dense_kernel`` = "auto" | "shared" | "registers" picks where the
    system lives during the elimination) or "auto" ("newton" on a radial network, "dense" on a
    meshed one that fits, the compensation sweep - run tight - on one that does not)."""

    METHODS = tuple(sorted(set(nat.SOLVERS) | {"dense", "auto"}))
    DENSE_KERNELS = {"auto": 0, "shared": 1, "registers": 2}

    def __init__(self, tolerance: float = 1e-6, max_iterations: int = 50, method: str = "newton",
                 acceleration_factor: float = 1.0, device="cuda", lanes: int = 0,
                 dense_kernel: str = "auto", **kwargs) -> None:
        if method not in self.METHODS:
            raise InvalidConfigurationError(f"method must be one of {list(self.METHODS)}")
        if dense_kernel not in self.DENSE_KERNELS:
            raise InvalidConfigurationError(f"dense_kernel must be one of {list(self.DENSE_KERNELS)}")
        self.dense_kernel = self.DENSE_KERNELS[dense_kernel]
        self.tolerance, self.max_iterations = float(tolerance), int(max_iterations)
        self.method, self.acceleration_factor = method, float(acceleration_factor)
        self.lanes = int(lanes)
        self._device_arg = device
        self._cache: Dict[Any, NativeFeeder] = {}
        self.last: Optional[PowerFlowSolution] = None

    # -- compiled topologies ------------------------------------------------------
    def _compile(self, feeder, method: Optional[str] = None) -> FeederSoA:
        method = method or ("newton" if self.method in ("auto", "dense") else self.method)
        soa, self._lanes_used = compile_for_solver(feeder, method, self.lanes, with_components=False)
        return soa

    def _native(self, key, make_soa) -> NativeFeeder:
        nf = self._cache.get(key)
        if nf is None:
            try:
                soa = make_soa()
            except TopologyError as exc:
                raise NetworkTopologyError(str(exc)) from exc
            nf = NativeFeeder(soa, _cuda_device(self._device_arg))
            if len(self._cache) >= 8:
                self._cache.pop(next(iter(self._cache))).close()
            self._cache[key] = nf
        return nf

    def _use_dense(self, buses, lines) -> bool:
        return self.method == "dense" or (self.method == "auto" and not is_radial(buses, lines))

    def _network(self, buses, lines, s_base: float) -> NativeNetwork:
        key = ("net", _signature(buses, lines), float(s_base))
        net = self._cache.get(key)
        if net is None:
            net = NativeNetwork(buses, lines, s_base, _cuda_device(self._device_arg))
            if len(self._cache) >= 8:
                self._cache.pop(next(iter(self._cache))).close()
            self._cache[key] = net
        return net

    def solve_network_batch(self, net: NativeNetwork, p_inj, q_inj=None) -> PowerFlowSolution:
        """The dense path: ``p_inj`` (and ``q_inj``, or None for Q_spec = 0) [B, n] per-unit injections in the
        network's bus order."""
        dev, lib = net.device, net.lib
        p, q = _injections(p_inj, q_inj, net.n_bus, dev)
        B, n, m = p.shape[0], net.n_bus, net.n_line
        f64 = dict(dtype=torch.float64, device=dev)
        out = dict(converged=torch.zeros(B, dtype=torch.uint8, device=dev),
                   iterations=torch.zeros(B, dtype=torch.int32, device=dev),
                   bus_voltages=torch.empty(B, n, **f64), bus_angles=torch.empty(B, n, **f64),
                   line_flows=torch.empty(B, m, **f64), line_loadings=torch.empty(B, m, **f64),
                   losses=torch.empty(B, **f64), max_mismatch=torch.empty(B, **f64))
        so = nat.SolOut(*[out[k].data_ptr() for k, _ in nat.SolOut._fields_])
        cfg = nat.make_solver_cfg("newton", self.tolerance, self.max_iterations, self.acceleration_factor,
                                  self.dense_kernel)
        nat.check(lib, lib.gfr_network_solve_pq(net.handle, B, p.data_ptr(), None if q is None else q.data_ptr(),
                                                C.byref(cfg), C.byref(so), torch.cuda.current_stream(dev).cuda_stream))
        out["converged"] = out["converged"].view(torch.bool)
        return PowerFlowSolution(**out)

    def solve_batch(self, feeder, p_inj, q_inj=None) -> PowerFlowSolution:
        """``p_inj`` [B, n] per-unit injections (generation minus load) in ``feeder.buses`` order, and
        ``q_inj`` [B, n] their reactive parts (None: Q_spec = 0; ``p_inj`` may also be a ``(p, q)`` pair);
        returns a ``PowerFlowSolution`` of tensors with a leading B axis."""
        if q_inj is None and isinstance(p_inj, tuple) and len(p_inj) == 2:
            p_inj, q_inj = p_inj
        if isinstance(feeder, NativeNetwork):
            return self.solve_network_batch(feeder, p_inj, q_inj)
        sweep_ties = False
        if not isinstance(feeder, (NativeFeeder, FeederSoA)) and self._use_dense(feeder.buses, feeder.lines):
            s_base = float(feeder.parameters.base_power) * 1e6
            try:
                return self.solve_network_batch(self._network(feeder.buses, feeder.lines, s_base), p_inj, q_inj)
            except GridLimitError:
                # the dense Jacobian does not fit an SM (e.g. IEEE-123 with its 26 tie lines: 244 unknowns):
                # "auto" falls back to the sweep on the spanning tree with the loops restored by compensation
                if self.method != "auto":
                    raise
                sweep_ties = True
        if isinstance(feeder, NativeFeeder):
            nf = feeder
        elif isinstance(feeder, FeederSoA):
            nf = self._native(("soa", id(feeder)), lambda: feeder)
        elif sweep_ties:
            nf = self._native(("feeder-sweep", id(feeder), _signature(feeder.buses, feeder.lines)),
                              lambda: self._compile(feeder, "sweep"))
        else:
            nf = self._native(("feeder", id(feeder), _signature(feeder.buses, feeder.lines)),
                              lambda: self._compile(feeder))
        dev, soa, lib = nf.device, nf.soa, nf.lib
        p, q = _injections(p_inj, q_inj, soa.n_bus, dev)
        B, n, m = p.shape[0], soa.n_bus, soa.n_line
        f64 = dict(dtype=torch.float64, device=dev)
        out = dict(converged=torch.zeros(B, dtype=torch.uint8, device=dev),
                   iterations=torch.zeros(B, dtype=torch.int32, device=dev),
                   bus_voltages=torch.empty(B, n, **f64), bus_angles=torch.empty(B, n, **f64),
                   line_flows=torch.empty(B, m, **f64), line_loadings=torch.empty(B, m, **f64),
                   losses=torch.empty(B, **f64), max_mismatch=torch.empty(B, **f64))
        so = nat.SolOut(*[out[k].data_ptr() for k, _ in nat.SolOut._fields_])
        method = "newton" if self.method in ("auto", "dense") else self.method
        if soa.n_tie:
            method = "sweep"                 # a tree with ties compiled for the compensation sweep
        cfg = nat.make_solver_cfg(method, self.tolerance if not sweep_ties else min(self.tolerance, 1e-9), self.max_iterations if not sweep_ties else max(self.max_iterations, 200),
                                  self.acceleration_factor,
                                  self.lanes or getattr(soa, "lanes_hint", 0) or auto_lanes(soa.n_bus, method))
        nat.check(lib, lib.gfr_solve_pq(nf.handle, B, p.data_ptr(), None if q is None else q.data_ptr(), C.byref(cfg),
                                        C.byref(so), torch.cuda.current_stream(dev).cuda_stream))
        out["converged"] = out["converged"].view(torch.bool)
        return PowerFlowSolution(**out)

    # -- the reference's two call shapes ----------------------------------------------
    def solve(self, *args):
        if len(args) == 4:
            return self._solve_reference_form(*args)
        if len(args) == 2:
            return self._solve_feeder_form(*args)
        raise TypeError("solve(buses, lines, loads, generation) or solve(feeder, loading_conditions)")

    def _solve_reference_form(self, buses, lines, loads: Dict[Any, float],
                              generation: Dict[Any, float]) -> PowerFlowSolution:
        # power_flow.py:105-121: P_spec = generation - load at each bus id; Q_spec = 0
        if self._use_dense(buses, lines):
            nf = self._network(buses, lines, 1.0)
        else:
            nf = self._native(("lists", _signature(buses, lines)),
                              lambda: self._compile(_Topology(buses, lines, 1e-6)))
        index = {b.id: i for i, b in enumerate(buses)}
        p = np.zeros((1, len(buses)))
        for bus, v in loads.items():
            if bus in index:
                p[0, index[bus]] -= v
        for bus, v in generation.items():
            if bus in index:
                p[0, index[bus]] += v
        return self._unwrap(self.solve_batch(nf, p))

    def _solve_feeder_form(self, feeder, loading_conditions):
        if isinstance(loading_conditions, dict):
            s_base = float(feeder.parameters.base_power) * 1e6
            index = {b.id: i for i, b in enumerate(feeder.buses)}
            p = np.zeros((1, len(feeder.buses)))
            for bus, v in loading_conditions.get("loads", {}).items():
                p[0, index[bus]] -= v / s_base
            for bus, v in loading_conditions.get("generation", {}).items():
                p[0, index[bus]] += v / s_base
            q = None
            if "reactive_loads" in loading_conditions or "reactive_generation" in loading_conditions:
                q = np.zeros((1, len(feeder.buses)))
                for bus, v in loading_conditions.get("reactive_loads", {}).items():
                    q[0, index[bus]] -= v / s_base
                for bus, v in loading_conditions.get("reactive_generation", {}).items():
                    q[0, index[bus]] += v / s_base
            return self._unwrap(self.solve_batch(feeder, p, q))
        return self.solve_batch(feeder, loading_conditions)

    def _unwrap(self, sol: PowerFlowSolution) -> PowerFlowSolution:
        one = PowerFlowSolution(
            converged=bool(sol.converged[0].item()), iterations=int(sol.iterations[0].item()),
            bus_voltages=sol.bus_voltages[0].cpu().numpy(), bus_angles=sol.bus_angles[0].cpu().numpy(),
            line_flows=sol.line_flows[0].cpu().numpy(), line_loadings=sol.line_loadings[0].cpu().numpy(),
            losses=float(sol.losses[0].item()), max_mismatch=float(sol.max_mismatch[0].item()))
        self.last = one
        return one

    def close(self) -> None:
        for nf in self._cache.values():
            nf.close()
        self._cache.clear()
