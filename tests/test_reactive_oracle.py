"""Specified reactive power on the CPU tier: the oracle with the Q_spec row filled in (tests/reactive_oracle.py), and
the specified-Q variants of the tree Newton and of the sweep (csrc/gfr_device.cuh, SPEC_Q) on the host emulation
at 1 - 16 lanes against it."""
import numpy as np
import pytest

from oracle import port
from oracle.ref_harness import make_feeder
from tests.golden_util import TOL_PU, feeder_for, golden_names, load_golden
from tests.host_emu import emu, emu_pq
from tests.reactive_oracle import load_pq, newton_raphson_pq

RADIAL = ("ieee13", "ieee34", "ieee123", "synthetic60:7")


def _pf_batch(f, B, seed, lo=0.3, hi=1.0):
    """B load-only injection rows at the loads' compiled power factor, each instance scaled by its own factor."""
    p0, q0 = load_pq(f)
    s = np.random.RandomState(seed).uniform(lo, hi, size=(B, 1))
    return s * p0, s * q0


def _pv_feeder():
    import grid_fed_rl_b200 as m
    f = m.SimpleRadialFeeder(9)
    f.buses[4].bus_type = "pv"; f.buses[4].voltage_magnitude = 1.01
    f.buses[7].bus_type = "pv"; f.buses[7].voltage_magnitude = 0.99
    return f


def _random_pq(n, B, seed, slack=0):
    """Random P and Q of both signs (generation and load, inductive and capacitive)."""
    rs = np.random.RandomState(seed)
    p = rs.uniform(-0.06, 0.02, size=(B, n)); q = rs.uniform(-0.04, 0.04, size=(B, n))
    p[:, slack] = 0.0; q[:, slack] = 0.0
    return p, q


def _check(sol, ref, iterations=True):
    ok = ref["converged"]
    assert ok.any()
    assert np.array_equal(sol["converged"].astype(bool)[ok], ok[ok])
    if iterations:
        assert np.array_equal(sol["converged"].astype(bool), ok)
        assert np.all(np.abs(sol["iterations"].astype(int) - ref["iterations"]) <= 1)
    for k in ("bus_voltages", "bus_angles", "line_flows"):
        assert np.max(np.abs(sol[k][ok] - ref[k][ok])) <= TOL_PU, k


# ----------------------------------------------------------------------------- the oracle

@pytest.mark.parametrize("name", golden_names("solve_"))
def test_oracle_q_zero_is_the_p_only_oracle(name):
    g = load_golden(name)
    f = feeder_for(g)
    net = port.DenseNetwork(f.buses, f.lines)
    tol, it = float(g["meta"][0]), int(g["meta"][1])
    a = port.newton_raphson(net, g["p_spec"], tol, it)
    b = newton_raphson_pq(net, g["p_spec"], None, tol, it)
    c = newton_raphson_pq(net, g["p_spec"], np.zeros_like(g["p_spec"]), tol, it)
    for k in a:
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], c[k]), k


@pytest.mark.parametrize("spec", RADIAL)
def test_oracle_solution_satisfies_the_specified_power(spec):
    """V conj(YV) = P + jQ at every PQ bus of a converged solution, computed here from Ybus alone."""
    f = make_feeder(None, spec, use_reference_classes=False)
    net = port.DenseNetwork(f.buses, f.lines)
    p, q = _pf_batch(f, 4, seed=1)
    assert np.abs(q).max() > 0
    ref = newton_raphson_pq(net, p, q, 1e-11, 50)
    assert ref["converged"].all()
    V = ref["bus_voltages"] * np.exp(1j * ref["bus_angles"])
    S = V * np.conj(V @ net.Y.T)
    assert np.max(np.abs(S[:, net.pq] - (p + 1j * q)[:, net.pq])) <= 1e-9
    assert np.max(np.abs(S.real[:, net.non_slack] - p[:, net.non_slack])) <= 1e-9


@pytest.mark.parametrize("spec", RADIAL)
def test_oracle_inductive_load_lowers_every_pq_voltage(spec):
    f = make_feeder(None, spec, use_reference_classes=False)
    net = port.DenseNetwork(f.buses, f.lines)
    p, q = _pf_batch(f, 3, seed=2)
    with_q = newton_raphson_pq(net, p, q, 1e-10, 50)
    no_q = newton_raphson_pq(net, p, np.zeros_like(q), 1e-10, 50)
    assert with_q["converged"].all() and no_q["converged"].all()
    dv = with_q["bus_voltages"][:, net.pq] - no_q["bus_voltages"][:, net.pq]
    assert np.all(dv < 0.0), (spec, dv.max())


# ----------------------------------------------------------------------------- host emulation of the SPEC_Q kernels

@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16])
@pytest.mark.parametrize("spec", RADIAL)
def test_emu_newton_with_q_matches_oracle(spec, lanes):
    f = make_feeder(None, spec, use_reference_classes=False)
    net = port.DenseNetwork(f.buses, f.lines)
    p, q = _pf_batch(f, 3, seed=10 + lanes)
    ref = newton_raphson_pq(net, p, q, 1e-10, 50)
    assert ref["converged"].all()
    sol = emu_pq.emu_solve_pq(f, p, q, "newton", 1e-10, 50, lanes=lanes, emu_lanes=lanes)
    _check(sol, ref)


@pytest.mark.parametrize("lanes", [1, 4, 16])
def test_emu_newton_with_q_pv_buses_and_both_signs(lanes):
    """PV buses hold |V| and have no Q equation: their Q entries (and the slack's) change nothing."""
    f = _pv_feeder()
    net = port.DenseNetwork(f.buses, f.lines)
    p, q = _random_pq(9, 6, seed=3)
    ref = newton_raphson_pq(net, p, q, 1e-10, 50)
    assert ref["converged"].all()
    sol = emu_pq.emu_solve_pq(f, p, q, "newton", 1e-10, 50, lanes=lanes, emu_lanes=lanes)
    _check(sol, ref)
    q2 = q.copy(); q2[:, [0, 4, 7]] = np.random.RandomState(4).uniform(-1, 1, size=(6, 3))
    sol2 = emu_pq.emu_solve_pq(f, p, q2, "newton", 1e-10, 50, lanes=lanes, emu_lanes=lanes)
    for k in ("bus_voltages", "bus_angles", "line_flows", "iterations"):
        assert np.array_equal(sol[k], sol2[k]), k


@pytest.mark.parametrize("spec", ["ieee34", "synthetic60:7"])
def test_emu_newton_random_q_both_signs(spec):
    f = make_feeder(None, spec, use_reference_classes=False)
    net = port.DenseNetwork(f.buses, f.lines)
    p0, _ = load_pq(f)
    rs = np.random.RandomState(6)
    p = p0 * rs.uniform(0.2, 0.8, size=(4, 1))
    q = np.abs(p0).max() * rs.uniform(-0.5, 0.5, size=p.shape)
    q[:, net.slack] = 0.0
    ref = newton_raphson_pq(net, p, q, 1e-10, 50)
    assert ref["converged"].all()
    for lanes in (1, 8):
        _check(emu_pq.emu_solve_pq(f, p, q, "newton", 1e-10, 50, lanes=lanes, emu_lanes=lanes), ref)


@pytest.mark.parametrize("lanes", [1, 2, 8, 16])
@pytest.mark.parametrize("spec", RADIAL)
def test_emu_sweep_with_q_matches_oracle(spec, lanes):
    f = make_feeder(None, spec, use_reference_classes=False)
    net = port.DenseNetwork(f.buses, f.lines)
    p, q = _pf_batch(f, 3, seed=20 + lanes)
    ref = newton_raphson_pq(net, p, q, 1e-10, 50)
    sol = emu_pq.emu_solve_pq(f, p, q, "sweep", 1e-11, 200, lanes=lanes, emu_lanes=lanes)
    _check(sol, ref, iterations=False)


@pytest.mark.parametrize("lanes", [1, 4, 8])
@pytest.mark.parametrize("spec", ["meshieee34", "mesh40:3:0.05", "meshieee123"])
def test_emu_sweep_with_q_on_meshed_feeders(spec, lanes):
    """Ties kept: the compensation sweep with specified Q against the oracle's dense Newton-Raphson."""
    f = make_feeder(None, spec, use_reference_classes=False)
    net = port.DenseNetwork(f.buses, f.lines)
    p, q = _pf_batch(f, 2, seed=30 + lanes, lo=0.3, hi=0.7)
    ref = newton_raphson_pq(net, p, q, 1e-10, 50)
    sol = emu_pq.emu_solve_pq(f, p, q, "sweep", 1e-11, 300, lanes=lanes, emu_lanes=lanes)
    _check(sol, ref, iterations=False)


@pytest.mark.parametrize("solver", ["newton", "sweep"])
def test_emu_q_zero_matches_p_only_path(solver):
    """q_inj = 0 through the SPEC_Q variants agrees with the P-only path to rounding, with equal iterations."""
    for name in ("solve_ieee13", "solve_ieee34", "solve_ieee123", "solve_synthetic60"):
        g = load_golden(name)
        f = feeder_for(g)
        tol, it = (float(g["meta"][0]), int(g["meta"][1])) if solver == "newton" else (1e-11, 200)
        for lanes in (1, 8):
            a = emu.emu_solve(f, g["p_spec"], solver, tol, it, lanes=lanes, emu_lanes=lanes)
            b = emu_pq.emu_solve_pq(f, g["p_spec"], np.zeros_like(g["p_spec"]), solver, tol, it, lanes=lanes,
                                    emu_lanes=lanes)
            assert np.array_equal(a["iterations"], b["iterations"]) and np.array_equal(a["converged"], b["converged"])
            for k in ("bus_voltages", "bus_angles", "line_flows", "losses"):
                assert np.max(np.abs(a[k] - b[k])) <= 1e-12, (name, lanes, k)
