"""CPU tier, Newton iterate by iterate: the exact-N meshed network generator of the dense-kernel tests
(tests/dense_networks.py), and the tree Newton on the host emulation (P only and with specified Q, 1 / 8 / 16 lanes)
stopped after 1, 2 and 3 updates and run to convergence, at acceleration 1.0, 0.7 and 1.2, against the oracle run
with the same settings (tests/newton_checks.py)."""
import numpy as np
import pytest

from oracle import port
from oracle.ref_harness import make_feeder
from tests import dense_networks as dn
from tests.host_emu import emu, emu_pq
from tests.newton_checks import as_numpy, borderline_rows, check_converged, check_truncated
from tests.reactive_oracle import load_pq, newton_raphson_pq

# B200's opt-in shared memory per block: N_max of the generated networks follows from it (tests/dense_networks.py)
B200_SMEM_OPTIN = 227 * 1024


# ----------------------------------------------------------------------------- the generator

def test_generator_gives_exact_unknowns_and_oracle_converges():
    n_max = dn.n_max(B200_SMEM_OPTIN)
    assert 160 <= n_max < 200
    for N in range(1, n_max + 1):
        for pv_heavy in (False, True) if N % 8 == 1 else (False,):
            buses, lines = dn.mesh_with_unknowns(N, seed=0, pv_heavy=pv_heavy)
            assert dn.unknowns(buses) == N
            net = port.DenseNetwork(buses, lines)
            assert net.slack != 0 and net.non_slack.size + net.pq.size == N
            k = net.pv.size
            if pv_heavy:
                assert 3 * k >= net.non_slack.size
            else:
                assert k == N % 2 and len(buses) == (N + 1) // 2 + 1
            p, q = dn.injections(buses, lines, 6, seed=N)
            ref = newton_raphson_pq(net, p[1:], q[1:], 1e-10, 30)
            assert ref["converged"].all() and ref["iterations"].max() <= 8, (N, pv_heavy)


def test_generator_covers_the_special_lines_and_the_large_first_correction():
    parallel = open_z = zero_rating = 0
    for N in range(8, 40):
        buses, lines = dn.mesh_with_unknowns(N, seed=0)
        ends = [frozenset((ln.from_bus, ln.to_bus)) for ln in lines]
        parallel += len(ends) != len(set(ends))
        open_z += any(abs(complex(ln.resistance, ln.reactance)) <= port.OPEN_Z for ln in lines)
        zero_rating += any(ln.rating == 0 for ln in lines)
        assert len(lines) > len(buses) - 1                    # meshed
    assert parallel and open_z and zero_rating
    buses, lines = dn.mesh_with_unknowns(40, seed=0)          # N % 4 == 0: a zero rating, loading 0
    net = port.DenseNetwork(buses, lines)
    p, q = dn.injections(buses, lines, 4, seed=1)
    ref = newton_raphson_pq(net, p, q, 1e-10, 30)
    assert np.all(ref["line_loadings"][:, net.rating == 0] == 0.0)
    first = newton_raphson_pq(net, p, q, 0.0, 1)
    big = np.max(np.abs(first["bus_angles"]), axis=1)
    assert big[0] > dn.BIG_ANGLE and np.all(big[1:] < dn.BIG_ANGLE)


# ----------------------------------------------------------------------------- tree Newton on the host emulation

def _pv_feeder():
    import grid_fed_rl_b200 as m
    f = m.SimpleRadialFeeder(9)
    f.buses[4].bus_type = "pv"; f.buses[4].voltage_magnitude = 1.01
    f.buses[7].bus_type = "pv"; f.buses[7].voltage_magnitude = 0.99
    return f


def feeder_and_batch(spec, B, seed):
    """A feeder and B injection rows (p, q): power-factor loads, each row scaled by its own factor; the 9-bus PV
    feeder takes random P and Q of both signs."""
    if spec == "pv9":
        f = _pv_feeder()
        rs = np.random.RandomState(seed)
        p = rs.uniform(-0.06, 0.02, size=(B, 9)); q = rs.uniform(-0.04, 0.04, size=(B, 9))
        p[:, 0] = q[:, 0] = 0.0
        return f, p, q
    f = make_feeder(None, spec, use_reference_classes=False)
    p0, q0 = load_pq(f)
    s = np.random.RandomState(seed).uniform(0.3, 1.0, size=(B, 1))
    return f, s * p0, s * q0


ACCELERATIONS = (1.0, 0.7, 1.2)
TRUNCATED = (1, 2, 3)
TOL = 1e-10
EMU_BOUND = 1e-12      # the emulation is the kernels' arithmetic on the host: measured <= 8e-13 pu (IEEE-13)


@pytest.mark.parametrize("with_q", [False, True], ids=["p", "pq"])
@pytest.mark.parametrize("lanes", [1, 8, 16])
@pytest.mark.parametrize("spec", ["ieee34", "ieee123", "pv9"])
def test_emulated_tree_newton_iterates_match_oracle(spec, lanes, with_q):
    f, p, q = feeder_and_batch(spec, 4, seed=lanes)
    q = q if with_q else None
    net = port.DenseNetwork(f.buses, f.lines)
    s_base = float(f.parameters.base_power) * 1e6

    def run(max_it, accel):
        kw = dict(lanes=lanes, emu_lanes=lanes, acceleration=accel)
        if q is None:
            return as_numpy(emu.emu_solve(f, p, "newton", TOL, max_it, **kw))
        return as_numpy(emu_pq.emu_solve_pq(f, p, q, "newton", TOL, max_it, **kw))

    for accel in ACCELERATIONS:
        for k in TRUNCATED:
            ref = newton_raphson_pq(net, p, q, TOL, k, accel)
            assert not ref["converged"].any()
            check_truncated(run(k, accel), ref, s_base, EMU_BOUND, ctx=(spec, accel, k))
        ref = newton_raphson_pq(net, p, q, TOL, 60, accel)
        assert ref["converged"].all()
        near = borderline_rows(net, p, q, ref, TOL, accel)
        check_converged(run(60, accel), ref, s_base, near, TOL, ctx=(spec, accel))
