"""GPU tier, Newton iterate by iterate: every Newton path stopped after 1, 2 and 3 updates and run to convergence, at
acceleration 1.0, 0.7 and 1.2, against the oracle run with the same settings (tests/newton_checks.py):

* the tree Newton through the solve surface, P only and with specified Q, on 1 - 256 lanes (warp-sized groups up to
  32, CTA-wide groups with the image in global memory above);
* both dense kernels at every N from 1 to the largest that fits the device's shared memory (tests/dense_networks.py):
  every register tile shape R = ceil(N / 8), odd and even N, P only and with Q, the slack away from bus 0;
* instances independent of their neighbours and of the batch size, NaN / Inf rows included;
* the environment step on steps that stop at max_iterations, all rows against the oracle environment.

The largest differences measured on each path are printed at the end of the module (pytest -s)."""
from functools import lru_cache

import numpy as np
import pytest
import torch

from oracle import port
from oracle.ref_harness import make_feeder
from tests import dense_networks as dn
from tests.golden_util import obs_layout
from tests.newton_checks import as_numpy, borderline_rows, check_converged, check_truncated
from tests.reactive_oracle import newton_raphson_pq
from tests.test_newton_iterates import ACCELERATIONS, TRUNCATED, feeder_and_batch

pytestmark = pytest.mark.gpu

BOUND = 1e-10          # truncated runs: the kernels against the oracle, pu
TOL = 1e-10
MAXDIFF = {}


def _record(path, d):
    MAXDIFF[path] = max(MAXDIFF.get(path, 0.0), d)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k in sorted(MAXDIFF):
        print(f"\n[newton iterates] largest difference {k}: {MAXDIFF[k]:.2e} pu", end="")


def _m():
    import grid_fed_rl_b200 as m
    return m


# ----------------------------------------------------------------------------- tree Newton, solve surface

TREE_FEEDERS = ("ieee13", "ieee34", "ieee123", "synthetic60:7", "pv9")


@lru_cache(maxsize=None)
def _tree_case(spec):
    f, p, q = feeder_and_batch(spec, 16, seed=17)
    return f, p, q, port.DenseNetwork(f.buses, f.lines)


@lru_cache(maxsize=None)
def _tree_ref(spec, with_q, max_it, accel):
    f, p, q, net = _tree_case(spec)
    q = q if with_q else None
    ref = newton_raphson_pq(net, p, q, TOL, max_it, accel)
    near = borderline_rows(net, p, q, ref, TOL, accel) if ref["converged"].all() else None
    return ref, near


@pytest.mark.parametrize("with_q", [False, True], ids=["p", "pq"])
@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32, 64, 128, 256])
@pytest.mark.parametrize("spec", TREE_FEEDERS)
def test_tree_newton_iterates_match_oracle(spec, lanes, with_q):
    m = _m()
    f, p, q, net = _tree_case(spec)
    s_base = float(f.parameters.base_power) * 1e6
    solver = m.B200PowerFlowSolver(tolerance=TOL, lanes=lanes)
    path = f"tree lanes {'<= 32' if lanes <= 32 else '>= 64'}"
    for accel in ACCELERATIONS:
        solver.acceleration_factor = accel
        for k in TRUNCATED + (60,):
            solver.max_iterations = k
            try:
                sol = as_numpy(solver.solve_batch(f, p, q if with_q else None))
            except m.GridLimitError as exc:          # one thread per instance on a 123-bus feeder
                pytest.skip(str(exc))
            ref, near = _tree_ref(spec, with_q, k, accel)
            ctx = (spec, lanes, with_q, accel, k)
            if k in TRUNCATED:
                assert not ref["converged"].any()
                _record(path + " truncated", check_truncated(sol, ref, s_base, BOUND, ctx))
            else:
                assert ref["converged"].all()
                _record(path + " converged", check_converged(sol, ref, s_base, near, TOL, ctx))
    solver.close()


# ----------------------------------------------------------------------------- dense kernels, every N

def _smem_optin():
    return int(torch.cuda.get_device_properties(torch.cuda.current_device()).shared_memory_per_block_optin)


def _n_max():
    return dn.n_max(_smem_optin())


# N_max depends on the device; the collection covers the B200's (168 with 227 KB per block) and each test past the
# device's own limit checks that the network is refused
N_RANGE = range(1, dn.n_max(227 * 1024) + 1)


def _dense_solver(kernel, **kw):
    return _m().B200PowerFlowSolver(method="dense", dense_kernel=kernel, tolerance=TOL, **kw)


def _dense_runs(kernels, f, net, p, q, accel, N, pv_heavy):
    """Truncated at 1 and 2 updates and converged, on each kernel, against the oracle."""
    s_base = dn.S_BASE_MVA * 1e6
    sols = {}
    for kernel in kernels:
        solver = _dense_solver(kernel, acceleration_factor=accel)
        for k in (1, 2, 30):
            solver.max_iterations = k
            sol = as_numpy(solver.solve_batch(f, p, q))
            sols[kernel, k] = sol
            ref = newton_raphson_pq(net, p, q, TOL, k, accel)
            ctx = (N, kernel, q is not None, pv_heavy, accel, k)
            if k < 30:
                _record(f"dense {kernel} truncated", check_truncated(sol, ref, s_base, BOUND, ctx))
            else:
                assert ref["converged"][1:].all(), ctx
                near = borderline_rows(net, p, q, ref, TOL, accel)
                _record(f"dense {kernel} converged", check_converged(sol, ref, s_base, near, TOL, ctx))
        solver.close()
    return sols


@pytest.mark.parametrize("N", N_RANGE)
def test_dense_kernels_every_unknown_count(N):
    m = _m()
    if N > _n_max():
        pytest.skip("beyond this device's shared memory")
    buses, lines = dn.mesh_with_unknowns(N, seed=0)
    f = dn.as_feeder(buses, lines)
    net = port.DenseNetwork(buses, lines)
    assert net.non_slack.size + net.pq.size == N and net.slack != 0
    p, q = dn.injections(buses, lines, 12, seed=N)
    kernels = ("registers", "shared") if N <= 127 else ("shared",)
    for qq in (None, q):
        sols = _dense_runs(kernels, f, net, p, qq, 1.0, N, False)
        auto = as_numpy(_dense_solver("auto", max_iterations=30).solve_batch(f, p, qq))
        same = sols["registers" if N <= 127 else "shared", 30]
        for k in auto:
            assert np.array_equal(auto[k], same[k], equal_nan=True), (N, k)
        if N % 8 == 4:                                         # one N per R at acceleration 0.7
            _dense_runs(kernels, f, net, p, qq, 0.7, N, False)
    if N % 8 == 1 and dn.fits(N, _smem_optin(), pv_heavy=True):   # the pv-heavy family, once per R
        pb, pl = dn.mesh_with_unknowns(N, seed=1, pv_heavy=True)
        pnet = port.DenseNetwork(pb, pl)
        assert pnet.non_slack.size + pnet.pq.size == N and 3 * pnet.pv.size >= pnet.non_slack.size
        pp, pq_ = dn.injections(pb, pl, 12, seed=1000 + N)
        for qq in (None, pq_):
            _dense_runs(kernels, dn.as_feeder(pb, pl), pnet, pp, qq, 1.0, N, True)
    if N == 128:
        with pytest.raises(m.GridLimitError):
            _dense_solver("registers").solve_batch(f, p)


def test_dense_limits_follow_the_shared_memory_formula():
    """N_max from dense_smem_bytes / dense_reg_smem_bytes and the device's opt-in shared memory per block: N_max
    solves on "shared" and "auto", N_max + 1 is refused by both."""
    m = _m()
    N = _n_max()
    for n_try, ok in ((N, True), (N + 1, False)):
        buses, lines = dn.mesh_with_unknowns(n_try, seed=0)
        f = dn.as_feeder(buses, lines)
        p, q = dn.injections(buses, lines, 2, seed=3)
        for kernel in ("shared", "auto"):
            if ok:
                sol = _dense_solver(kernel, max_iterations=30).solve_batch(f, p, q)
                assert bool(sol.converged[1])
            else:
                with pytest.raises(m.GridLimitError):
                    _dense_solver(kernel).solve_batch(f, p, q)


# ----------------------------------------------------------------------------- instances are independent

def _bad_rows(p, q, rows, pq_cols):
    """NaN / +Inf / -Inf in the P or the Q injection of a PQ bus (both have an equation there)."""
    p, q = p.copy(), q.copy()
    for j, (r, v) in enumerate(zip(rows, (np.nan, np.inf, -np.inf, np.nan))):
        (p if j % 2 == 0 else q)[r, pq_cols[(7 * j) % len(pq_cols)]] = v
    return p, q


def _independence(solve, p, q, pq_cols, distinct, B, max_it):
    """``distinct`` rows tiled into B: every copy equals the solve of its row alone; rows with NaN / Inf among them
    fail cleanly and leave their neighbours as they were."""
    tile = np.arange(B) % distinct
    pb, qb = p[tile], q[tile]
    big = solve(pb, qb)
    for r in range(distinct):
        one = solve(p[r:r + 1], q[r:r + 1])
        for k, v in big.items():
            assert np.array_equal(v[tile == r], np.broadcast_to(one[k], v[tile == r].shape)), (r, k)
    bad = np.array([3, B // 2 + 1, B // 2 + 2, B - 1])
    pn, qn = _bad_rows(pb, qb, bad, pq_cols)
    assert not np.isfinite(pn[bad] + qn[bad]).all(axis=1).any()
    dirty = solve(pn, qn)
    assert not dirty["converged"][bad].any()
    assert np.all(dirty["iterations"][bad] == max_it)
    assert np.all(np.isnan(dirty["max_mismatch"][bad]))
    keep = np.setdiff1d(np.arange(B), bad)
    for k, v in dirty.items():
        assert np.array_equal(v[keep], big[k][keep]), k


@pytest.mark.parametrize("kernel", ["registers", "shared"])
def test_dense_instances_are_independent(kernel):
    buses, lines = dn.mesh_with_unknowns(45, seed=2)
    f = dn.as_feeder(buses, lines)
    p, q = dn.injections(buses, lines, 6, seed=5)
    p, q = p[1:], q[1:]
    pq_cols = port.DenseNetwork(buses, lines).pq
    solver = _dense_solver(kernel, max_iterations=12)
    B = 148 * 24 * 3 + 7                                     # more than one resident wave of the smallest tiles

    def solve(a, b):
        return as_numpy(solver.solve_batch(f, a, b))
    _independence(solve, p, q, pq_cols, 5, B, 12)


@pytest.mark.parametrize("lanes", [8, 64])
def test_tree_instances_are_independent(lanes):
    f, p, q = feeder_and_batch("ieee123", 5, seed=9)
    pq_cols = port.DenseNetwork(f.buses, f.lines).pq
    solver = _m().B200PowerFlowSolver(tolerance=TOL, max_iterations=12, lanes=lanes)
    B = 40000                                                # several resident waves at 8 and 64 lanes

    def solve(a, b):
        return as_numpy(solver.solve_batch(f, a, b))
    _independence(solve, p, q, pq_cols, 5, B, 12)


# ----------------------------------------------------------------------------- the environment step, not converged

@pytest.mark.parametrize("spec,lanes,accel", [("ieee13", 2, 1.0), ("ieee34", 4, 1.0), ("ieee123", 8, 1.0),
                                              ("ieee123", 64, 1.0), ("ieee123", 8, 0.7)])
@pytest.mark.parametrize("max_it", [1, 2])
def test_step_stopped_at_max_iterations_matches_oracle(spec, lanes, accel, max_it):
    """The environment builds the observation, reward and flags of a non-converged step from the last iterate
    (reference grid_env.py:724-731): every row against the oracle environment with the same settings."""
    m = _m()
    f = make_feeder(None, spec, use_reference_classes=False)
    B, steps = 48, 4
    kw = dict(timestep=60.0, episode_length=100, renewable_sources=["solar", "wind"])
    env = m.BatchedGridEnvironment(f, B, solver="newton", lanes=lanes, tolerance=1e-8, max_iterations=max_it,
                                   acceleration=accel, repair=False, **kw)
    ref = port.PortEnv(f, B, tolerance=1e-8, max_iterations=max_it, acceleration=accel, **kw)
    rs = np.random.RandomState(max_it * 10 + lanes)
    start = 11.5 * 3600.0
    nz0 = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3))], axis=1)
    env.reset(noise=nz0, options={"start_time": start})
    ref.reset(nz0, start_time=start)
    lay = obs_layout(ref.n, ref.m, ref.L, ref.G, ref.Bt)
    s_base = ref.s_base
    for t in range(steps):
        act = rs.uniform(-1, 1, size=(B, ref.A))
        nz = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3 + ref.L))], axis=1)
        obs, reward, term, trunc, info = env.step(act, nz)
        r = ref.step(act, nz)
        o = obs.cpu().numpy()
        assert not r["converged"].all()
        assert np.array_equal(info["power_flow_converged"].cpu().numpy(), r["converged"])
        assert np.array_equal(info["iterations"].cpu().numpy(), r["iterations"])
        d = max(np.max(np.abs(o[:, lay["vm"]] - r["obs"][:, lay["vm"]])),
                np.max(np.abs(o[:, lay["va"]] - r["obs"][:, lay["va"]])),
                np.max(np.abs(o[:, lay["p"]] - r["obs"][:, lay["p"]])) / s_base,
                np.max(np.abs(info["total_losses"].cpu().numpy() - r["losses"])) / s_base)
        assert d <= BOUND, (t, d)
        _record("environment step truncated", d)
        assert np.max(np.abs(o[:, lay["freq"]] - r["obs"][:, lay["freq"]])) <= 1e-9
        assert np.allclose(reward.cpu().numpy(), r["reward"], rtol=1e-9, atol=1e-6)
        assert np.array_equal(term.cpu().numpy(), r["terminated"])
        assert np.array_equal(info["current_step"].cpu().numpy(), r["current_step"])
        vm, fr = r["obs"][:, lay["vm"]], r["obs"][:, lay["freq"]]
        margin = np.minimum(np.min(np.abs(vm - 0.95), axis=1), np.min(np.abs(vm - 1.05), axis=1))
        margin = np.minimum(margin, np.minimum(np.abs(fr - 59.5), np.abs(fr - 60.5)))
        clear = margin > 1e-9
        assert clear.mean() > 0.9
        assert np.array_equal(info["constraint_violations"].cpu().numpy()[clear], r["violations"][clear])
        assert np.array_equal(info["constraint_violation_count"].cpu().numpy()[clear], r["viol_count"][clear])
        assert np.array_equal(trunc.cpu().numpy()[clear], r["truncated"][clear])
    env.close()
