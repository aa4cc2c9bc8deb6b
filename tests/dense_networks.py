"""TEST INFRASTRUCTURE: meshed networks with an exact number of Newton unknowns, for the dense kernels
(csrc/gfr_dense.cuh).

The dense kernels pick their code by N = (#non-slack buses) + (#PQ buses): the register kernel has one instantiation
per R = ceil(N / 8), with and without specified Q, and odd N (which needs PV buses) takes other branches of both
kernels' column handling than even N.  ``mesh_with_unknowns(N, seed)`` builds a network with exactly N unknowns, so
that a test can reach every one of them:

* n buses in a permuted order, a random spanning tree plus about n / 5 chords, lines in random orientation;
* the slack at a random position other than 0 (so the column maps are not the identity shifted by one);
* k PV buses at set magnitudes in 0.98 - 1.03, k in {0, 1} (n = ceil(N / 2) + 1), or with ``pv_heavy`` at least a
  third of the non-slack buses;
* r in 0.002 - 0.02 pu, x in 0.004 - 0.04 pu.

Across N the set holds parallel line pairs, zero-impedance chords (open lines: |z| <= 1e-12) and zero ratings
(loading 0): the first chord is a parallel copy of a tree line when N % 3 == 0 and has zero impedance when
N % 3 == 1, and the first line has rating 0 when N % 4 == 0.

``injections(buses, lines, B, seed)`` draws P uniform in [-0.6, 0.2] / n and Q uniform in [-0.3, 0.15] / n per bus,
and scales row 0 up until the oracle's first correction turns some bus by more than 0.25 rad (the range where
``sincos_small`` halves its argument); that row need not converge.
"""
from __future__ import annotations

import math
from types import SimpleNamespace

import numpy as np

from grid_fed_rl_b200.components import Bus, FeederParameters, Line
from oracle import port
from tests.reactive_oracle import newton_raphson_pq

S_BASE_MVA = 10.0
BIG_ANGLE = 0.25


def _sizes(N: int, pv_heavy: bool):
    """(n, k): bus count and PV count with 2 (n - 1) - k = N."""
    if not pv_heavy:
        k = N % 2
        return (N + k) // 2 + 1, k
    m = max(1, math.ceil(3 * N / 5))                      # non-slack buses
    while not (3 * (2 * m - N) >= m and 2 * m - N <= m):
        m += 1
    return m + 1, 2 * m - N


def mesh_with_unknowns(N: int, seed: int, pv_heavy: bool = False):
    """(buses, lines) with exactly N = (#non-slack) + (#PQ) unknowns."""
    assert N >= 1
    n, k = _sizes(N, pv_heavy)
    rs = np.random.RandomState(seed * 7919 + N * 2 + int(pv_heavy))
    order = rs.permutation(n)                             # tree node t is bus order[t] in the bus list
    ids = 100 + 3 * np.arange(n)                          # ids unrelated to positions
    slack = int(rs.randint(1, n))
    others = [i for i in range(n) if i != slack]
    pv = set(int(i) for i in rs.choice(others, size=k, replace=False)) if k else set()
    buses = []
    for i in range(n):
        kind = "slack" if i == slack else ("pv" if i in pv else "pq")
        b = Bus(int(ids[i]), 1.0, kind)
        if kind == "pv":
            b.voltage_magnitude = float(rs.uniform(0.98, 1.03))
        elif kind == "slack":
            b.voltage_magnitude = float(rs.uniform(1.0, 1.03))
        buses.append(b)

    def line(a, b):
        if rs.rand() < 0.5:
            a, b = b, a
        return Line(len(lines), int(ids[a]), int(ids[b]), float(rs.uniform(0.002, 0.02)),
                    float(rs.uniform(0.004, 0.04)), float(rs.uniform(0.5, 4.0)) * 1e6)

    lines, tree = [], []
    for t in range(1, n):
        a, b = int(order[int(rs.randint(0, t))]), int(order[t])
        tree.append((a, b))
        lines.append(line(a, b))
    chords = n // 5
    have = set(frozenset(e) for e in tree)
    for c in range(chords):
        if c == 0 and N % 3 == 0:                         # a parallel pair
            a, b = tree[int(rs.randint(0, len(tree)))]
            lines.append(line(a, b))
            continue
        for _ in range(100):
            a, b = (int(x) for x in rs.choice(n, size=2, replace=False))
            if frozenset((a, b)) not in have:
                break
        have.add(frozenset((a, b)))
        ln = line(a, b)
        if c == 0 and N % 3 == 1:                         # zero impedance: an open line
            ln.resistance = ln.reactance = 0.0
        lines.append(ln)
    if N % 4 == 0:
        lines[0].rating = 0.0
    return buses, lines


def dense_smem_bytes(n: int, N: int, registers: bool) -> int:
    """Shared memory of one dense-kernel CTA (``dense_smem_bytes`` / ``dense_reg_smem_bytes`` in gfr_dense.cuh)."""
    b = (N | 1) * N * 8 + N * 8 + n * 32 + 64 * 8
    return b + 3 * 128 * 8 + 128 * 4 + 64 if registers else b


def fits(N: int, smem_optin: int, pv_heavy: bool = False) -> bool:
    """Whether gfr_network_create takes the generated network with N unknowns (it sizes the register kernel's
    shared memory up to 127 unknowns and the shared-memory kernel's above)."""
    n, _ = _sizes(N, pv_heavy)
    return dense_smem_bytes(n, N, N <= 127) <= smem_optin


def n_max(smem_optin: int) -> int:
    """The largest N of the (non pv-heavy) family that fits ``smem_optin`` bytes of shared memory per block."""
    N = 1
    while fits(N + 1, smem_optin):
        N += 1
    return N


def as_feeder(buses, lines):
    """What B200PowerFlowSolver.solve_batch takes: buses, lines and the base power."""
    return SimpleNamespace(name="mesh", buses=buses, lines=lines, loads=[], generators={},
                           parameters=FeederParameters(base_voltage=1.0, base_power=S_BASE_MVA, frequency=60.0))


def unknowns(buses) -> int:
    net_ns = sum(b.bus_type != "slack" for b in buses)
    return net_ns + sum(b.bus_type == "pq" for b in buses)


def injections(buses, lines, B: int, seed: int):
    """(p, q) [B, n] pu; row 0 is scaled up until the oracle's first correction exceeds BIG_ANGLE rad."""
    n = len(buses)
    rs = np.random.RandomState(seed)
    p = rs.uniform(-0.6, 0.2, size=(B, n)) / n
    q = rs.uniform(-0.3, 0.15, size=(B, n)) / n
    net = port.DenseNetwork(buses, lines)
    p[:, net.slack] = 0.0
    q[:, net.slack] = 0.0
    for _ in range(40):
        first = newton_raphson_pq(net, p[:1], q[:1], 0.0, 1)
        if np.max(np.abs(first["bus_angles"])) > BIG_ANGLE:
            break
        p[0] *= 1.5
        q[0] *= 1.5
    return p, q
