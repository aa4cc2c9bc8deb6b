"""GPU tier, specified reactive power: the solve entry points with q_inj (gfr_solve_pq / gfr_network_solve_pq through
B200PowerFlowSolver) against the oracle with the Q_spec row filled in (tests/reactive_oracle.py), on every solver
path - tree Newton, sweep with and without ties, both dense kernels, "auto" - and the P-only path left as it was."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import port
from oracle.ref_harness import make_feeder
from tests.golden_util import TOL_PU, feeder_for, golden_names, load_golden
from tests.reactive_oracle import load_pq, newton_raphson_pq

pytestmark = pytest.mark.gpu

RADIAL = ("ieee13", "ieee34", "ieee123", "synthetic60:7")
MESHED = ("meshieee34", "mesh40:3:0.05", "mesh72:5:0.02", "meshieee123")


def _pf_batch(f, B, seed, lo=0.3, hi=1.0):
    p0, q0 = load_pq(f)
    s = np.random.RandomState(seed).uniform(lo, hi, size=(B, 1))
    return s * p0, s * q0


def _check(sol, ref, f, tol, iterations=True, rows=slice(None)):
    """Converged rows: the state and losses within TOL_PU; line loadings (|S| s_base / rating on the solve surface,
    |S| / rating in the oracle) within what a TOL_PU error of |S| allows; the mismatch below the tolerance ``tol``."""
    ok = ref["converged"]
    assert ok.any()
    conv = sol.converged.cpu().numpy()[rows]
    assert np.all(conv[ok])
    if iterations:
        assert np.array_equal(conv, ok)
        assert np.all(np.abs(sol.iterations.cpu().numpy()[rows].astype(int) - ref["iterations"]) <= 1)
    for k in ("bus_voltages", "bus_angles", "line_flows", "losses"):
        assert np.max(np.abs(getattr(sol, k).cpu().numpy()[rows][ok] - ref[k][ok])) <= TOL_PU, k
    s_base = float(f.parameters.base_power) * 1e6
    got, want = sol.line_loadings.cpu().numpy()[rows][ok], ref["line_loadings"][ok] * s_base
    with np.errstate(divide="ignore", invalid="ignore"):
        per_pu = np.where(ref["line_s_abs"][ok] > 0, want / ref["line_s_abs"][ok], 0.0)   # s_base / rating
    assert np.all(np.abs(got - want) <= TOL_PU * per_pu + 1e-12), "line_loadings"
    assert np.all(sol.max_mismatch.cpu().numpy()[rows][ok] < tol), "max_mismatch"


def _solver(**kw):
    import grid_fed_rl_b200 as m
    return m.B200PowerFlowSolver(**kw)


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32, 64, 128, 256])
@pytest.mark.parametrize("spec", RADIAL)
def test_newton_with_q_matches_oracle(spec, lanes):
    import grid_fed_rl_b200 as m
    f = make_feeder(None, spec, use_reference_classes=False)
    p, q = _pf_batch(f, 24, seed=lanes)
    ref = newton_raphson_pq(port.DenseNetwork(f.buses, f.lines), p, q, 1e-10, 50)
    assert ref["converged"].all()
    try:
        sol = _solver(tolerance=1e-10, lanes=lanes).solve_batch(f, p, q)
    except m.GridLimitError as exc:            # one thread per instance on a 123-bus feeder
        pytest.skip(str(exc))
    _check(sol, ref, f, 1e-10)


@pytest.mark.parametrize("lanes", [1, 8, 32, 64])
@pytest.mark.parametrize("spec", RADIAL + MESHED)
def test_sweep_with_q_matches_oracle(spec, lanes):
    import grid_fed_rl_b200 as m
    f = make_feeder(None, spec, use_reference_classes=False)
    p, q = _pf_batch(f, 16, seed=100 + lanes, hi=0.7)
    ref = newton_raphson_pq(port.DenseNetwork(f.buses, f.lines), p, q, 1e-10, 50)
    try:
        sol = _solver(method="sweep", tolerance=1e-11, max_iterations=300, lanes=lanes).solve_batch(f, p, q)
    except m.GridLimitError as exc:
        pytest.skip(str(exc))
    _check(sol, ref, f, 1e-11, iterations=False)


@pytest.mark.parametrize("where", ["shared", "registers"])
@pytest.mark.parametrize("name", [n for n in golden_names("meshsolve_") if "ieee123" not in n])
def test_dense_with_q_matches_oracle(name, where):
    f = feeder_for(load_golden(name))
    net = port.DenseNetwork(f.buses, f.lines)
    if where == "registers" and net.non_slack.size + net.pq.size > 127:
        pytest.skip("more unknowns than the register kernel takes")
    p, q = _pf_batch(f, 12, seed=7, hi=0.7)
    ref = newton_raphson_pq(net, p, q, 1e-10, 30)
    sol = _solver(method="dense", dense_kernel=where, tolerance=1e-10, max_iterations=30).solve_batch(f, p, q)
    _check(sol, ref, f, 1e-10)


@pytest.mark.parametrize("spec", ["ieee34", "meshieee34", "mesh40:3:0.05", "meshieee123"])
def test_auto_with_q_matches_oracle(spec):
    """"auto": Newton on a radial feeder, the dense kernels on a meshed one, and the tight compensation sweep on
    IEEE-123 with its 26 ties (beyond the dense kernels) - Q reaches each of them."""
    f = make_feeder(None, spec, use_reference_classes=False)
    p, q = _pf_batch(f, 8, seed=3, hi=0.7)
    ref = newton_raphson_pq(port.DenseNetwork(f.buses, f.lines), p, q, 1e-10, 50)
    sol = _solver(method="auto", tolerance=1e-10).solve_batch(f, p, q)
    _check(sol, ref, f, 1e-10, iterations=spec != "meshieee123")


def test_full_size_ieee123_newton_8_lanes():
    """131 072 IEEE-123 instances at power-factor loads, each scaled by its own factor; 64 sampled rows replayed."""
    f = make_feeder(None, "ieee123", use_reference_classes=False)
    B = 131072
    p, q = _pf_batch(f, B, seed=11)
    sol = _solver(tolerance=1e-8, lanes=8).solve_batch(f, torch.from_numpy(p), torch.from_numpy(q))
    assert bool(sol.converged.all())
    rows = np.sort(np.random.RandomState(12).choice(B, 64, replace=False))
    ref = newton_raphson_pq(port.DenseNetwork(f.buses, f.lines), p[rows], q[rows], 1e-8, 50)
    _check(sol, ref, f, 1e-8, rows=rows)


# ----------------------------------------------------------------------------- P-only callers

def _native_and_cfg(solver, f, p):
    from grid_fed_rl_b200 import _native as nat
    solver.solve_batch(f, p)
    nf = next(iter(solver._cache.values()))
    cfg = nat.make_solver_cfg(solver.method, solver.tolerance, solver.max_iterations, solver.acceleration_factor,
                              solver.lanes)
    return nat, nf, cfg


def _raw_solve(nat, fn, handle, p, cfg, n, m):
    B = p.shape[0]
    out = dict(converged=torch.zeros(B, dtype=torch.uint8, device="cuda"),
               iterations=torch.zeros(B, dtype=torch.int32, device="cuda"),
               bus_voltages=torch.empty(B, n, dtype=torch.float64, device="cuda"),
               bus_angles=torch.empty(B, n, dtype=torch.float64, device="cuda"),
               line_flows=torch.empty(B, m, dtype=torch.float64, device="cuda"),
               line_loadings=torch.empty(B, m, dtype=torch.float64, device="cuda"),
               losses=torch.empty(B, dtype=torch.float64, device="cuda"),
               max_mismatch=torch.empty(B, dtype=torch.float64, device="cuda"))
    so = nat.SolOut(*[out[k].data_ptr() for k, _ in nat.SolOut._fields_])
    rc = fn(handle, B, p.data_ptr(), C.byref(cfg), C.byref(so), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, out


@pytest.mark.parametrize("method,lanes", [("newton", 1), ("newton", 8), ("newton", 64), ("sweep", 1), ("sweep", 8)])
@pytest.mark.parametrize("name", ["solve_ieee13", "solve_ieee34", "solve_ieee123", "solve_synthetic60"])
def test_p_only_path_unchanged(name, method, lanes):
    """q_inj=None returns exactly what gfr_solve returns; q_inj = 0 through the Q kernels agrees to 1e-12."""
    import grid_fed_rl_b200 as m
    g = load_golden(name)
    f = feeder_for(g)
    tol, it = (float(g["meta"][0]), int(g["meta"][1])) if method == "newton" else (1e-11, 200)
    s = _solver(method=method, tolerance=tol, max_iterations=it, lanes=lanes)
    try:
        nat, nf, cfg = _native_and_cfg(s, f, g["p_spec"])
    except m.GridLimitError as exc:
        pytest.skip(str(exc))
    p = torch.as_tensor(g["p_spec"], device="cuda").contiguous()
    n, mm = nf.soa.n_bus, nf.soa.n_line
    rc, direct = _raw_solve(nat, nf.lib.gfr_solve, nf.handle, p, cfg, n, mm)
    assert rc == 0
    a = s.solve_batch(f, g["p_spec"])
    b = s.solve_batch(f, g["p_spec"], np.zeros_like(g["p_spec"]))
    for k, v in direct.items():
        got = getattr(a, k)
        assert torch.equal(got.view(torch.uint8) if k == "converged" else got, v), k
    assert torch.equal(a.iterations, b.iterations) and torch.equal(a.converged, b.converged)
    for k in ("bus_voltages", "bus_angles", "line_flows", "losses"):
        assert float((getattr(a, k) - getattr(b, k)).abs().max()) <= 1e-12, k


# ----------------------------------------------------------------------------- call shapes and errors

def test_call_shapes_agree():
    import grid_fed_rl_b200 as m
    f = make_feeder(None, "ieee13", use_reference_classes=False)
    s_base = float(f.parameters.base_power) * 1e6
    s = _solver(tolerance=1e-10)
    loads = {ld.bus: 0.0 for ld in f.loads}
    qloads = {ld.bus: 0.0 for ld in f.loads}
    for ld in f.loads:
        loads[ld.bus] += float(ld.active_power)
        qloads[ld.bus] += float(ld.reactive_power)
    one = s.solve(f, {"loads": loads, "reactive_loads": qloads})
    p, q = load_pq(f)
    batch = s.solve_batch(f, p[None], q[None])
    pair = s.solve_batch(f, (p, q))
    two_arg_pair = s.solve(f, (p[None], q[None]))
    assert one.converged and bool(batch.converged[0])
    for k in ("bus_voltages", "bus_angles", "line_flows", "line_loadings"):
        assert np.max(np.abs(getattr(one, k) - getattr(batch, k)[0].cpu().numpy())) <= 1e-13, k
        assert torch.equal(getattr(batch, k), getattr(pair, k)) and torch.equal(getattr(batch, k), getattr(two_arg_pair, k)), k
    gen_form = s.solve(f, {"loads": loads, "reactive_generation": {b: -v for b, v in qloads.items()}})
    assert np.array_equal(gen_form.bus_voltages, one.bus_voltages)
    # no reactive keys: the P-only path
    p_only = s.solve(f, {"loads": loads})
    assert np.array_equal(p_only.bus_voltages, s.solve_batch(f, p[None]).bus_voltages[0].cpu().numpy())
    pq = port.DenseNetwork(f.buses, f.lines).pq
    assert np.all(one.bus_voltages[pq] < p_only.bus_voltages[pq])
    for bad in (np.zeros((1, len(f.buses) + 1)), np.zeros((2, len(f.buses))), np.zeros((1, 1, len(f.buses)))):
        with pytest.raises(m.InvalidConfigurationError):
            s.solve_batch(f, p[None], bad)
    with pytest.raises(m.InvalidConfigurationError):
        _solver(method="dense").solve_batch(f, p[None], np.zeros((1, 3)))


def test_null_p_inj_is_an_argument_error():
    f = make_feeder(None, "ieee13", use_reference_classes=False)
    p, q = load_pq(f)
    s = _solver()
    nat, nf, cfg = _native_and_cfg(s, f, p[None])
    qt = torch.as_tensor(q[None], device="cuda").contiguous()
    so = nat.SolOut()
    rc = nf.lib.gfr_solve_pq(nf.handle, 1, None, qt.data_ptr(), C.byref(cfg), C.byref(so), None)
    assert rc == nat.GFR_E_ARG
    net = s._network(f.buses, f.lines, 1.0)
    rc = net.lib.gfr_network_solve_pq(net.handle, 1, None, qt.data_ptr(), C.byref(cfg), C.byref(so), None)
    assert rc == nat.GFR_E_ARG


@pytest.mark.parametrize("method,kw", [("newton", dict(lanes=1)), ("newton", dict(lanes=4)), ("newton", dict(lanes=64)),
                                       ("dense", dict(dense_kernel="shared")), ("dense", dict(dense_kernel="registers"))])
def test_pv_and_slack_q_entries_change_nothing(method, kw):
    import grid_fed_rl_b200 as m
    f = m.SimpleRadialFeeder(9)
    f.buses[4].bus_type = "pv"; f.buses[4].voltage_magnitude = 1.01
    f.buses[7].bus_type = "pv"; f.buses[7].voltage_magnitude = 0.99
    rs = np.random.RandomState(5)
    p = rs.uniform(-0.06, 0.02, size=(32, 9)); p[:, 0] = 0
    q = rs.uniform(-0.04, 0.04, size=(32, 9)); q[:, 0] = 0; q[:, [4, 7]] = 0
    ref = newton_raphson_pq(port.DenseNetwork(f.buses, f.lines), p, q, 1e-10, 50)
    s = _solver(method=method, tolerance=1e-10, **kw)
    a = s.solve_batch(f, p, q)
    _check(a, ref, f, 1e-10)
    q2 = q.copy(); q2[:, [0, 4, 7]] = rs.uniform(-1, 1, size=(32, 3))
    b = s.solve_batch(f, p, q2)
    for k in ("bus_voltages", "bus_angles", "line_flows", "iterations", "converged"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k
