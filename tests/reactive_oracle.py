"""TEST INFRASTRUCTURE: the oracle's polar Newton-Raphson (``oracle.port.newton_raphson``) with the reference's
``Q_spec`` row filled in - the checker of the solve entry points that take specified reactive power.

``newton_raphson_pq(net, p_spec, q_spec)`` is ``port.newton_raphson`` term by term, except that the Q mismatch of a
PQ bus is ``q_spec - Q_calc`` instead of ``0 - Q_calc``.  ``q_spec=None`` returns ``port.newton_raphson`` itself,
and the tests check that ``q_spec = 0`` reproduces it bit for bit, so the two cannot drift apart unnoticed.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np

from oracle import port


def newton_raphson_pq(net: port.DenseNetwork, p_spec: np.ndarray, q_spec: Optional[np.ndarray] = None,
                      tolerance: float = 1e-6, max_iterations: int = 50, acceleration: float = 1.0,
                      j11_fix: bool = True) -> Dict[str, np.ndarray]:
    """Batched polar NR.  ``p_spec`` / ``q_spec`` [B, n] pu, generation minus load; Q entries of the slack and of
    PV buses are ignored (no Q equation there)."""
    if q_spec is None:
        return port.newton_raphson(net, p_spec, tolerance, max_iterations, acceleration, j11_fix)
    p_spec = np.atleast_2d(np.asarray(p_spec, dtype=float))
    q_spec = np.broadcast_to(np.atleast_2d(np.asarray(q_spec, dtype=float)), p_spec.shape)
    B, n = p_spec.shape
    Y, G, Bm = net.Y, net.Y.real, net.Y.imag
    ns, pq = net.non_slack, net.pq
    V = np.ones((B, n), dtype=complex)
    fixed = np.concatenate([[net.slack], net.pv]).astype(np.int64)
    V[:, fixed] = net.vm_set[fixed]
    converged = np.zeros(B, dtype=bool)
    iterations = np.full(B, max_iterations, dtype=np.int32)
    max_mismatch = np.full(B, np.inf)
    active = np.ones(B, dtype=bool)
    is_ns = np.zeros(n, dtype=bool); is_ns[ns] = True
    is_pq = np.zeros(n, dtype=bool); is_pq[pq] = True
    gd, bd = np.diag(G), np.diag(Bm)

    for it in range(max_iterations):
        idx = np.flatnonzero(active)
        if idx.size == 0:
            break
        Va_ = V[idx]
        S = Va_ * np.conj(Va_ @ Y.T)
        dP = np.where(is_ns, p_spec[idx] - S.real, 0.0)
        dQ = np.where(is_pq, q_spec[idx] - S.imag, 0.0)
        mm = np.maximum(np.max(np.abs(dP), axis=1), np.max(np.abs(dQ), axis=1))
        max_mismatch[idx] = mm
        done = mm < tolerance
        converged[idx[done]] = True
        iterations[idx[done]] = it + 1
        active[idx[done]] = False
        keep = ~done
        idx = idx[keep]
        if idx.size == 0:
            break
        Vc, dP, dQ = V[idx], dP[keep], dQ[keep]
        Vm, Va = np.abs(Vc), np.angle(Vc)
        dth = Va[:, :, None] - Va[:, None, :]
        cs, sn = np.cos(dth), np.sin(dth)
        A = G * sn - Bm * cs
        C = G * cs + Bm * sn
        VV = Vm[:, :, None] * Vm[:, None, :]
        J11 = VV * A
        d11 = -np.sum(VV * A, axis=2) + Vm * Vm * bd
        if j11_fix:
            d11 = d11 - 2.0 * Vm * Vm * bd
        J12 = Vm[:, :, None] * C
        d12 = np.sum(Vm[:, None, :] * C, axis=2) + Vm * gd
        J21 = -VV * C
        d21 = np.sum(VV * C, axis=2) - Vm * Vm * gd
        J22 = Vm[:, :, None] * A
        d22 = np.sum(Vm[:, None, :] * A, axis=2) - Vm * bd
        ar = np.arange(n)
        for Jb, db in ((J11, d11), (J12, d12), (J21, d21), (J22, d22)):
            Jb[:, ar, ar] = db
        J = np.block([[J11[:, ns][:, :, ns], J12[:, ns][:, :, pq]],
                      [J21[:, pq][:, :, ns], J22[:, pq][:, :, pq]]])
        rhs = np.concatenate([dP[:, ns], dQ[:, pq]], axis=1)
        try:
            dx = np.linalg.solve(J, rhs[:, :, None])[:, :, 0]
            singular = np.zeros(idx.size, dtype=bool)
        except np.linalg.LinAlgError:
            dx = np.zeros_like(rhs)
            singular = np.zeros(idx.size, dtype=bool)
            for q in range(idx.size):
                try:
                    dx[q] = np.linalg.solve(J[q], rhs[q])
                except np.linalg.LinAlgError:
                    singular[q] = True
        iterations[idx[singular]] = it + 1
        active[idx[singular]] = False
        ok = ~singular
        dVa, dVm = dx[:, :ns.size], dx[:, ns.size:]
        Vn = Vc.copy()
        Vn[:, ns] = np.abs(Vn[:, ns]) * np.exp(1j * (np.angle(Vn[:, ns]) + acceleration * dVa))
        Vn[:, pq] = (np.abs(Vn[:, pq]) + acceleration * dVm) * np.exp(1j * np.angle(Vn[:, pq]))
        V[idx[ok]] = Vn[ok]

    I = net.y * (V[:, net.fr] - V[:, net.to])
    Sij = V[:, net.fr] * np.conj(I)
    with np.errstate(divide="ignore", invalid="ignore"):
        loadings = np.where(net.rating > 0, np.abs(Sij) / net.rating, 0.0)
    losses = np.sum(V * np.conj(V @ Y.T), axis=1).real
    return dict(converged=converged, iterations=iterations, bus_voltages=np.abs(V),
                bus_angles=np.angle(V), line_flows=Sij.real, line_loadings=loadings,
                losses=losses, max_mismatch=max_mismatch, line_s_abs=np.abs(Sij))


def load_pq(feeder, s_base: Optional[float] = None):
    """(p, q) [n] pu in ``feeder.buses`` order: every load at its compiled power factor, generation minus load
    (``Load.active_power`` / ``Load.reactive_power`` over the base power)."""
    if s_base is None:
        s_base = float(feeder.parameters.base_power) * 1e6
    index = {b.id: i for i, b in enumerate(feeder.buses)}
    p, q = np.zeros(len(feeder.buses)), np.zeros(len(feeder.buses))
    for ld in feeder.loads:
        p[index[ld.bus]] -= float(ld.active_power) / s_base
        q[index[ld.bus]] -= float(ld.reactive_power) / s_base
    return p, q
