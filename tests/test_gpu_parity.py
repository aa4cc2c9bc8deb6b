"""GPU tier: the CUDA path, called through the C ABI (ctypes) exactly as a user would, against
 (a) the frozen outputs of the reference itself (tests/golden, written by oracle/ref_harness.py),
 (b) the numpy oracle (oracle/port.py) on seeded batches,
 (c) size-independent properties at BASELINE.json's full sizes.
Tolerances (BASELINE.json north_star): |V|, angle, line flow, losses within 1e-8 pu in fp64;
flags and counters bit-exact; Newton iteration counts within +-1."""
import numpy as np
import pytest
import torch

from oracle import port
from tests.golden_util import (TOL_PU, feeder_for, golden_names, load_golden, obs_layout, port_trace,
                               replay_trace)

pytestmark = pytest.mark.gpu

LANES = (1, 2, 4, 8, 16, 32)
REPL = 3      # replicas of the golden instance per batch: all must agree bit for bit


def _factory(solver, lanes, tol_override=None):
    import grid_fed_rl_b200 as m

    class _One:
        def __init__(self, feeder, kw):
            kw = dict(kw)
            tol = kw.pop("tolerance")
            try:
                self.env = m.BatchedGridEnvironment(feeder, REPL, solver=solver, lanes=lanes,
                                                    tolerance=tol_override or tol, repair=False, **kw)
            except m.GridLimitError as exc:     # e.g. one thread per instance on a 123-bus feeder
                pytest.skip(str(exc))

        def reset(self, noise4, start_time):
            nz = np.tile(np.asarray(noise4)[None, :4], (REPL, 1))
            obs, _ = self.env.reset(noise=nz, options={"start_time": start_time})
            obs = obs.cpu().numpy()
            assert np.array_equal(obs[0], obs[1]) and np.array_equal(obs[0], obs[2])
            return obs[0]

        def step(self, action, noise):
            obs, reward, term, trunc, info = self.env.step(np.tile(action[None, :], (REPL, 1)),
                                                           np.tile(noise[None, :], (REPL, 1)))
            out = dict(obs=obs, reward=reward, terminated=term, truncated=trunc,
                       error=info["error"], converged=info["power_flow_converged"],
                       iterations=info["iterations"], losses=info["total_losses"],
                       violations=info["constraint_violations"],
                       viol_count=info["constraint_violation_count"],
                       current_step=info["current_step"], episode_reward=info["episode_reward"])
            out = {k: v.cpu().numpy() for k, v in out.items()}
            for k, v in out.items():
                assert np.array_equal(v[0], v[1], equal_nan=True) and np.array_equal(v[0], v[2], equal_nan=True), k
            return {k: v[0] for k, v in out.items()}
    return _One


@pytest.mark.parametrize("lanes", LANES)
@pytest.mark.parametrize("name", golden_names("trace_"))
def test_newton_step_matches_reference_trace(name, lanes):
    if "_long_" in name and lanes not in (4, 16):
        pytest.skip("long traces run at two lane counts")
    g = load_golden(name)
    exact = replay_trace(_factory("newton", lanes), g, ctx=f"{name}/lanes{lanes}")
    assert exact >= 0.9 * g["obs"].shape[0]


@pytest.mark.parametrize("lanes", (64, 256))
@pytest.mark.parametrize("name", ("trace_ieee13_s0", "trace_ieee34_s0", "trace_ieee123_s0", "trace_fixture3_s0"))
def test_cta_per_instance_matches_reference_trace(name, lanes):
    """LANES > 32: one CTA per instance, CTA barriers, feeder image read from global memory."""
    g = load_golden(name)
    exact = replay_trace(_factory("newton", lanes), g, ctx=f"{name}/cta{lanes}")
    assert exact >= 0.9 * g["obs"].shape[0]
    gs = port_trace(g, tolerance=1e-10)
    exact = replay_trace(_factory("sweep", lanes, 1e-11), gs, ctx=f"{name}/sweep/cta{lanes}", check_iterations=False)
    assert exact >= 0.9 * g["obs"].shape[0]


@pytest.mark.parametrize("lanes", (1, 8, 32))
@pytest.mark.parametrize("name", [n for n in golden_names("trace_") if "_long_" not in n])
def test_sweep_step_matches_oracle_trace(name, lanes):
    g = port_trace(load_golden(name), tolerance=1e-10)
    exact = replay_trace(_factory("sweep", lanes, 1e-11), g, ctx=f"{name}/sweep/lanes{lanes}",
                         check_iterations=False)
    assert exact >= 0.9 * g["obs"].shape[0]


@pytest.mark.parametrize("lanes", LANES)
@pytest.mark.parametrize("name", golden_names("solve_"))
def test_solver_matches_reference(name, lanes):
    import grid_fed_rl_b200 as m
    g = load_golden(name)
    f = feeder_for(g)
    tol, max_it = float(g["meta"][0]), int(g["meta"][1])
    s = m.B200PowerFlowSolver(tolerance=tol, max_iterations=max_it, method="newton", lanes=lanes)
    try:
        sol = s.solve_batch(f, g["p_spec"])
    except m.GridLimitError as exc:
        pytest.skip(str(exc))
    conv = g["converged"]
    assert np.array_equal(sol.converged.cpu().numpy(), conv)
    assert np.all(np.abs(sol.iterations.cpu().numpy().astype(int) - g["iterations"]) <= 1)
    for k in ("bus_voltages", "bus_angles", "line_flows", "losses"):
        if conv.any():
            assert np.max(np.abs(getattr(sol, k).cpu().numpy()[conv] - g[k][conv])) <= TOL_PU, k
    # |S| s_base / rating against the reference's |S| / rating
    s_base = f.parameters.base_power * 1e6
    if conv.any():
        assert np.allclose(sol.line_loadings.cpu().numpy()[conv], g["line_loadings"][conv] * s_base,
                           rtol=1e-7, atol=1e-12)
    # sweep, both sides tight
    net = port.DenseNetwork(f.buses, f.lines)
    ref = port.newton_raphson(net, g["p_spec"], 1e-10, 50)
    sw = m.B200PowerFlowSolver(tolerance=1e-11, max_iterations=200, method="sweep", lanes=lanes)
    try:
        sol = sw.solve_batch(f, g["p_spec"])
    except m.GridLimitError as exc:               # a 1 000-bus feeder on one thread per instance
        pytest.skip(str(exc))
    ok = ref["converged"]
    assert np.all(sol.converged.cpu().numpy()[ok])
    for k in ("bus_voltages", "bus_angles", "line_flows", "losses"):
        if ok.any():
            assert np.max(np.abs(getattr(sol, k).cpu().numpy()[ok] - ref[k][ok])) <= TOL_PU, k


def test_reference_call_shapes_appendix_a():
    """SURVEY Appendix A through solve(buses, lines, loads, generation) and solve(feeder, dict)."""
    import grid_fed_rl_b200 as m
    from oracle.ref_harness import make_feeder
    f = make_feeder(None, "fixture3", use_reference_classes=False)
    s = m.B200PowerFlowSolver(tolerance=1e-10, max_iterations=50)
    sol = s.solve(f.buses, f.lines, {2: 0.1, 3: 0.05}, {})
    assert sol.converged and sol.iterations == 4
    assert np.allclose(sol.bus_voltages, [1, 0.998491585126075, 0.997739099627788], atol=1e-11)
    assert np.allclose(sol.bus_angles, [0, -0.003004662358732, -0.004259387863609], atol=1e-11)
    assert np.allclose(sol.line_flows, [0.15026346387586, 0.05003767014433], atol=1e-11)
    assert abs(sol.losses - 2.6346387586110437e-04) < 1e-12
    s6 = m.B200PowerFlowSolver(tolerance=1e-6, max_iterations=50)
    assert s6.solve(f.buses, f.lines, {2: 0.1, 3: 0.05}, {}).iterations == 3
    sol2 = s.solve(f, {"loads": {2: 0.1 * 1e7, 3: 0.05 * 1e7}, "generation": {}})
    assert np.allclose(sol2.bus_voltages, sol.bus_voltages, atol=1e-13)


def _batch_against_port(spec, B, steps, solver, lanes, seed, tol=1e-8, **kw):
    import grid_fed_rl_b200 as m
    from oracle.ref_harness import make_feeder
    f = make_feeder(None, spec, use_reference_classes=False)
    kw = dict(dict(timestep=60.0, episode_length=steps - 3, renewable_sources=["solar", "wind"]), **kw)
    start = 11.5 * 3600.0
    env = m.BatchedGridEnvironment(f, B, solver=solver, lanes=lanes, tolerance=tol, repair=False, **kw)
    ptol = 1e-10 if solver == "sweep" else tol
    ref = port.PortEnv(f, B, tolerance=ptol, **kw)
    rs = np.random.RandomState(seed)
    L, A = ref.L, ref.A
    nz0 = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3))], axis=1)
    obs, _ = env.reset(noise=nz0, options={"start_time": start})
    robs = ref.reset(nz0, start_time=start)
    assert np.max(np.abs(obs.cpu().numpy() - robs)) < 1e-9
    lay = obs_layout(ref.n, ref.m, L, ref.G, ref.Bt)
    s_base = ref.s_base
    for t in range(steps):
        act = rs.uniform(-1, 1, size=(B, A))
        if t == 2 and A > 1:
            act[1, 0] = np.nan
        nz = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3 + L))], axis=1)
        obs, reward, term, trunc, info = env.step(act, nz)
        r = ref.step(act, nz)
        o = obs.cpu().numpy()
        ok = r["converged"] | r["error"]
        assert np.array_equal(info["power_flow_converged"].cpu().numpy(), r["converged"])
        assert np.array_equal(info["error"].cpu().numpy(), r["error"])
        assert np.max(np.abs(o[ok][:, lay["vm"]] - r["obs"][ok][:, lay["vm"]])) <= TOL_PU
        assert np.max(np.abs(o[ok][:, lay["va"]] - r["obs"][ok][:, lay["va"]])) <= TOL_PU
        assert np.max(np.abs(o[ok][:, lay["p"]] - r["obs"][ok][:, lay["p"]])) / s_base <= TOL_PU
        assert np.max(np.abs(info["total_losses"].cpu().numpy()[ok] - r["losses"][ok])) / s_base <= TOL_PU
        assert np.max(np.abs(o[ok][:, lay["freq"]] - r["obs"][ok][:, lay["freq"]])) <= 1e-9
        assert np.max(np.abs(o[ok][:, lay["soc"]] - r["obs"][ok][:, lay["soc"]])) <= 1e-12
        assert np.allclose(o[ok][:, lay["gen"]], r["obs"][ok][:, lay["gen"]], rtol=1e-12, atol=1e-6)
        assert np.allclose(reward.cpu().numpy()[ok], r["reward"][ok], rtol=1e-9, atol=1e-6)
        assert np.array_equal(term.cpu().numpy(), r["terminated"])
        assert np.array_equal(info["current_step"].cpu().numpy(), r["current_step"])
        if solver == "newton":
            assert np.all(np.abs(info["iterations"].cpu().numpy().astype(int) - r["iterations"]) <= 1)
        # flags: exact wherever no voltage / frequency sits within 1e-9 of a limit
        vm, fr = r["obs"][:, lay["vm"]], r["obs"][:, lay["freq"]]
        margin = np.minimum(np.min(np.abs(vm - 0.95), axis=1), np.min(np.abs(vm - 1.05), axis=1))
        margin = np.minimum(margin, np.minimum(np.abs(fr - 59.5), np.abs(fr - 60.5)))
        clear = ok & (margin > 1e-9)
        assert clear.mean() > 0.9
        assert np.array_equal(info["constraint_violations"].cpu().numpy()[clear], r["violations"][clear])
        assert np.array_equal(info["constraint_violation_count"].cpu().numpy()[clear], r["viol_count"][clear])
        assert np.array_equal(trunc.cpu().numpy()[clear], r["truncated"][clear])
        done = r["terminated"] | r["truncated"]
        if done.any():
            nzr = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3))], axis=1)
            env.reset(noise=nzr, mask=done, options={"start_time": start})
            ref.reset(nzr, mask=done, start_time=start)
    env.close()


@pytest.mark.parametrize("lanes", LANES)
def test_batch_ieee13_newton_vs_oracle(lanes):
    _batch_against_port("ieee13", 333, 16, "newton", lanes, seed=lanes)


@pytest.mark.parametrize("lanes", (1, 4, 32))
def test_batch_ieee13_sweep_vs_oracle(lanes):
    _batch_against_port("ieee13", 257, 14, "sweep", lanes, seed=10 + lanes, tol=1e-11)


@pytest.mark.parametrize("lanes", (4, 8, 32))
def test_batch_ieee34_vs_oracle(lanes):
    _batch_against_port("ieee34", 130, 10, "newton", lanes, seed=20 + lanes, renewable_sources=["solar"])
    _batch_against_port("ieee34", 130, 10, "sweep", lanes, seed=30 + lanes, tol=1e-11, renewable_sources=["solar"])


@pytest.mark.parametrize("lanes", (8, 16, 32))
def test_batch_ieee123_newton_vs_oracle(lanes):
    _batch_against_port("ieee123", 40, 5, "newton", lanes, seed=40 + lanes, tol=1e-6)


def test_pv_bus_feeder_vs_oracle():
    """PV buses (none in the shipped feeders): |V| held, no Q equation - against the oracle port."""
    import grid_fed_rl_b200 as m
    f = m.SimpleRadialFeeder(9)
    f.buses[4].bus_type = "pv"; f.buses[4].voltage_magnitude = 1.01
    f.buses[7].bus_type = "pv"; f.buses[7].voltage_magnitude = 0.99
    rs = np.random.RandomState(5)
    p = rs.uniform(-0.08, 0.02, size=(64, 9)); p[:, 0] = 0
    net = port.DenseNetwork(f.buses, f.lines)
    ref = port.newton_raphson(net, p, 1e-10, 50)
    for lanes in (1, 4, 32):
        sol = m.B200PowerFlowSolver(tolerance=1e-10, lanes=lanes).solve_batch(f, p)
        assert np.array_equal(sol.converged.cpu().numpy(), ref["converged"]) and ref["converged"].all()
        assert np.max(np.abs(sol.bus_voltages.cpu().numpy() - ref["bus_voltages"])) <= TOL_PU
        assert np.max(np.abs(sol.bus_angles.cpu().numpy() - ref["bus_angles"])) <= TOL_PU
        assert np.max(np.abs(sol.line_flows.cpu().numpy() - ref["line_flows"])) <= TOL_PU
        assert np.all(np.abs(sol.iterations.cpu().numpy().astype(int) - ref["iterations"]) <= 1)
    with pytest.raises(m.InvalidConfigurationError):
        m.B200PowerFlowSolver(method="sweep").solve_batch(f, p)


@pytest.mark.parametrize("lanes", [8, 64, 128])
def test_hub_with_more_pool_children_than_a_packed_record_holds(lanes):
    """A hub with 13 children on CTA-wide groups (64 / 128 lanes): 12 pool children, the packed pool-child record of
    the hub's position holds 8, so that position walks the child list instead; the others take the record.  Both
    solvers and one environment step against the oracle."""
    import grid_fed_rl_b200 as m
    f = m.SimpleRadialFeeder(18)
    for ln in f.lines[3:16]:
        ln.from_bus = 4
    for ld in f.loads:
        ld.base_power *= 0.2; ld.active_power *= 0.2; ld.reactive_power *= 0.2
    f = m.repair_topology(f)
    n = len(f.buses)
    rs = np.random.RandomState(5)
    p = -np.abs(rs.uniform(0.002, 0.01, size=(37, n))); p[:, 0] = 0.0
    ref = port.newton_raphson(port.DenseNetwork(f.buses, f.lines), p, 1e-10, 50)
    assert ref["converged"].all()
    for method, tol, it in (("newton", 1e-10, 50), ("sweep", 1e-11, 200)):
        sol = m.B200PowerFlowSolver(tolerance=tol, max_iterations=it, method=method, lanes=lanes).solve_batch(f, p)
        assert bool(sol.converged.all()), method
        assert np.max(np.abs(sol.bus_voltages.cpu().numpy() - ref["bus_voltages"])) <= TOL_PU
        assert np.max(np.abs(sol.bus_angles.cpu().numpy() - ref["bus_angles"])) <= TOL_PU
        assert np.max(np.abs(sol.line_flows.cpu().numpy() - ref["line_flows"])) <= TOL_PU
    # one step of the environment on the same lanes: the batched loops around the solve (injections, flat start,
    # observation) against a one-lane run
    kw = dict(timestep=60.0, repair=False, tolerance=1e-10, start_time=12 * 3600.0)
    a = m.BatchedGridEnvironment(f, 33, lanes=1, **kw); a.reset(seed=2)
    b = m.BatchedGridEnvironment(f, 33, lanes=lanes, **kw); b.reset(seed=2)
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    for _ in range(3):
        act = a.sample_actions(g)
        oa, ra, _, _, ia = a.step(act)
        ob, rb, _, _, ib = b.step(act)
        assert torch.allclose(oa, ob, rtol=1e-11, atol=1e-6) and torch.allclose(ra, rb, rtol=1e-11, atol=1e-9)
        assert torch.equal(ia["iterations"], ib["iterations"])
    a.close(); b.close()


def test_philox_noise_matches_oracle_and_replays():
    import ctypes as C
    import grid_fed_rl_b200 as m
    from grid_fed_rl_b200 import _native as nat
    lib = nat.load_library()
    rs = np.random.RandomState(0)
    seeds = rs.randint(0, 2**63 - 1, size=300, dtype=np.int64)
    draws = rs.randint(0, 2**40, size=300, dtype=np.int64)
    d_seeds, d_draws = torch.as_tensor(seeds).cuda(), torch.as_tensor(draws).cuda()
    for n_slots in (4, 5, 12, 99):
        out = torch.empty(300, n_slots, dtype=torch.float64, device="cuda")
        nat.check(lib, lib.gfr_noise_fill(0, 300, n_slots, d_seeds.data_ptr(), d_draws.data_ptr(),
                                          out.data_ptr(), None))
        torch.cuda.synchronize()
        ref = port.philox_noise(seeds.astype(np.uint64), draws.astype(np.uint64), n_slots)
        assert np.max(np.abs(out.cpu().numpy() - ref)) < 1e-12
    # throughput mode: the env's own stream == the oracle's Philox row, and replaying the recorded
    # row through the oracle reproduces the step
    from oracle.ref_harness import make_feeder
    f = make_feeder(None, "ieee13", use_reference_classes=False)
    kw = dict(timestep=30.0, renewable_sources=["solar", "wind"])
    B = 100
    env = m.BatchedGridEnvironment(f, B, solver="newton", tolerance=1e-8, repair=False, record_noise=True,
                                   env_id_offset=1000, **kw)
    ref = port.PortEnv(f, B, tolerance=1e-8, **kw)
    env.reset(seed=7, options={"start_time": 12 * 3600.0})
    sd = np.arange(B, dtype=np.uint64) + np.uint64(1007)
    nz0 = port.philox_noise(sd, np.zeros(B, dtype=np.uint64), 4)
    ref.reset(nz0, start_time=12 * 3600.0)
    lay = obs_layout(ref.n, ref.m, ref.L, ref.G, ref.Bt)
    for t in range(6):
        act = rs.uniform(-1, 1, size=(B, ref.A))
        obs, reward, _, _, info = env.step(act)
        used = env.noise_used.cpu().numpy()
        expect = port.philox_noise(sd, np.full(B, t + 1, dtype=np.uint64), 4 + ref.L)
        assert np.max(np.abs(used - expect)) < 1e-12
        r = ref.step(act, used)
        assert np.max(np.abs(obs.cpu().numpy()[:, lay["vm"]] - r["obs"][:, lay["vm"]])) <= TOL_PU
        assert np.allclose(reward.cpu().numpy(), r["reward"], rtol=1e-9, atol=1e-6)


def test_reset_mask_autoreset_and_checkpoint():
    import grid_fed_rl_b200 as m
    f = m.repair_topology(m.IEEE13Bus())
    kw = dict(renewable_sources=["solar", "wind"], episode_length=5, timestep=60.0, repair=False)
    a = m.BatchedGridEnvironment(f, 64, **kw)
    a.reset(seed=3)
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    for _ in range(3):
        a.step(a.sample_actions(g))
    sd = a.state_dict()
    b = m.BatchedGridEnvironment(f, 64, **kw)
    b.load_state_dict(sd)
    act = a.sample_actions(g)
    oa, ra, ta, _, ia = a.step(act)
    ob, rb, tb, _, ib = b.step(act)
    assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(ia["current_step"], ib["current_step"])
    # masked reset touches only the selected instances
    before = a.get_observation().clone()
    info_before = {k: v.clone() for k, v in ia.items() if isinstance(v, torch.Tensor)}
    r_before = ra.clone()                      # (the step's return values are the live output buffers)
    mask = torch.zeros(64, dtype=torch.bool, device="cuda"); mask[::4] = True
    obs, info = a.reset(mask=mask)
    assert torch.equal(obs[~mask], before[~mask])
    assert torch.all(obs[mask][:, 0] == 1.0) and torch.all(info["current_step"][mask] == 0)
    assert torch.all(info["current_step"][~mask] == 4)
    # ... and so do the info arrays (one launch, gfr_env_reset_outputs): zeros / 1.0 pu where reset, untouched elsewhere
    for k, v in info_before.items():
        assert torch.equal(info[k][~mask], v[~mask]), k
        want = 1.0 if k in ("max_voltage", "min_voltage") else 0
        assert torch.all(info[k][mask] == want), k
    assert torch.all(a._out["reward"][mask] == 0) and torch.equal(a._out["reward"][~mask], r_before[~mask])
    # an unmasked reset clears every row
    _, info = a.reset()
    assert all(torch.all(info[k] == (1.0 if k in ("max_voltage", "min_voltage") else 0))
               for k in info_before)
    # auto-reset: instances that terminate come back at step 0 with the initial observation
    c = m.BatchedGridEnvironment(f, 32, auto_reset=True, **kw)
    c.reset(seed=5)
    for t in range(5):
        obs, rew, term, trunc, info = c.step(c.sample_actions(g))
    assert bool(term.all())
    assert torch.all(obs[:, 0] == 1.0) and "final_observation" in info
    obs, rew, term, trunc, info = c.step(c.sample_actions(g))
    assert torch.all(info["current_step"] == 1) and not bool(term.any())


def test_full_size_properties_ieee123():
    """BASELINE config 4 per-GPU size: 131,072 IEEE-123 instances, Newton, Philox noise."""
    import grid_fed_rl_b200 as m
    f = m.repair_topology(m.IEEE123Bus(seed=0))
    B = 131072
    kw = dict(renewable_sources=["solar", "wind"], solver="newton", tolerance=1e-6, repair=False)
    env = m.BatchedGridEnvironment(f, B, start_time=12 * 3600.0, **kw)
    env.reset(seed=11)
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    act = env.sample_actions(g)
    obs, reward, term, trunc, info = env.step(act)
    assert bool(info["power_flow_converged"].all())
    assert int(info["iterations"].min()) >= 2 and int(info["iterations"].max()) <= 6
    assert torch.isfinite(obs).all() and torch.isfinite(reward).all()
    n, mlines = env.soa.n_bus, env.soa.n_line
    lay = obs_layout(n, mlines, env.soa.n_load, env.soa.n_gen, env.soa.n_bat)
    vm = obs[:, lay["vm"]]
    assert torch.all(vm[:, 0] == 1.0)                                  # slack magnitude
    assert torch.equal(info["max_voltage"], vm.max(dim=1).values)
    assert torch.equal(info["min_voltage"], vm.min(dim=1).values)
    assert torch.equal(info["constraint_violations"][:, 1], (vm < 0.95).any(dim=1))
    # power balance: the slack line flow(s) carry load - generation + losses; losses > 0 and small
    assert torch.all(info["total_losses"] > 0) and torch.all(info["total_losses"] < 0.05 * env.soa.s_base)
    # determinism + independence from the thread mapping
    first = obs.clone(); r1 = reward.clone()
    for lanes in (8, 32):
        e2 = m.BatchedGridEnvironment(f, 4096, start_time=12 * 3600.0, lanes=lanes, **kw)
        e2.reset(seed=11)
        o2, r2, _, _, i2 = e2.step(act[:4096])
        assert torch.max(torch.abs(o2[:, lay["vm"]] - first[:4096, lay["vm"]])) < 1e-12
        assert torch.allclose(r2, r1[:4096], rtol=1e-12, atol=1e-9)
        e2.close()
    env2 = m.BatchedGridEnvironment(f, B, start_time=12 * 3600.0, **kw)
    env2.reset(seed=11)
    o3, r3, _, _, _ = env2.step(act)
    assert torch.equal(o3, first) and torch.equal(r3, r1)


@pytest.mark.parametrize("spec,B", [("ieee13", 65536), ("ieee34", 262144)])
def test_full_size_properties_sweep_configs(spec, B):
    """BASELINE configs 2 and 3 at their full sizes (IEEE-13 x 65,536 and IEEE-34 x 262,144, backward /
    forward sweep, in-kernel noise): every instance converges, the observation is consistent with the
    reported extremes and flags, a re-run is bit-identical, a different thread mapping and a smaller
    batch (another launch plan: the wave-balanced one) give the same state, and the Newton kernel fed the
    same noise rows lands on the same voltages (two algorithms, one fixed point)."""
    import grid_fed_rl_b200 as m
    from oracle.ref_harness import make_feeder
    f = make_feeder(None, spec, use_reference_classes=False)
    srcs = ["solar", "wind"] if spec == "ieee13" else ["solar"]
    kw = dict(renewable_sources=srcs, repair=False, start_time=12 * 3600.0)
    env = m.BatchedGridEnvironment(f, B, solver="sweep", tolerance=1e-10, record_noise=True, **kw)
    env.reset(seed=21)
    g = torch.Generator(device="cuda"); g.manual_seed(4)
    act = env.sample_actions(g)
    obs, reward, term, trunc, info = env.step(act)
    assert bool(info["power_flow_converged"].all())
    assert torch.isfinite(obs).all() and torch.isfinite(reward).all()
    n, mlines = env.soa.n_bus, env.soa.n_line
    lay = obs_layout(n, mlines, env.soa.n_load, env.soa.n_gen, env.soa.n_bat)
    vm = obs[:, lay["vm"]]
    assert torch.equal(info["max_voltage"], vm.max(dim=1).values)
    assert torch.equal(info["min_voltage"], vm.min(dim=1).values)
    assert torch.equal(info["constraint_violations"][:, 1], (vm < 0.95).any(dim=1))
    assert torch.all(info["total_losses"] > 0)
    first, r1 = obs.clone(), reward.clone()
    noise = env.noise_used.clone()
    # bit-identical re-run
    env2 = m.BatchedGridEnvironment(f, B, solver="sweep", tolerance=1e-10, **kw)
    env2.reset(seed=21)
    o2, r2, _, _, _ = env2.step(act)
    assert torch.equal(o2, first) and torch.equal(r2, r1)
    env2.close()
    # another thread mapping, another launch plan (a batch below one wave is spread over all SMs)
    sub = 3000
    for lanes in (1, 4):
        e3 = m.BatchedGridEnvironment(f, sub, solver="sweep", tolerance=1e-10, lanes=lanes, **kw)
        e3.reset(seed=21)
        o3, r3, _, _, _ = e3.step(act[:sub])
        assert torch.max(torch.abs(o3[:, lay["vm"]] - first[:sub, lay["vm"]])) < 1e-10
        assert torch.allclose(r3, r1[:sub], rtol=1e-9, atol=1e-7)
        e3.close()
    # Newton on the same noise rows: same fixed point
    e4 = m.BatchedGridEnvironment(f, sub, solver="newton", tolerance=1e-10, **kw)
    e4.reset(seed=21)
    o4, r4, _, _, i4 = e4.step(act[:sub], noise=noise[:sub])
    assert bool(i4["power_flow_converged"].all())
    assert torch.max(torch.abs(o4[:, lay["vm"]] - first[:sub, lay["vm"]])) < 1e-8
    assert torch.max(torch.abs(o4[:, lay["va"]] - first[:sub, lay["va"]])) < 1e-8
    e4.close()
    env.close()


def test_sharding_is_seed_stable():
    """Results do not depend on how instances are split over ranks (SURVEY 8e)."""
    import grid_fed_rl_b200 as m
    f = m.repair_topology(m.IEEE13Bus())
    kw = dict(renewable_sources=["solar", "wind"], solver="sweep", tolerance=1e-10, repair=False,
              start_time=9 * 3600.0)
    whole = m.BatchedGridEnvironment(f, 1000, **kw)
    whole.reset(seed=42)
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    act = whole.sample_actions(g)
    ow = whole.step(act)[0].clone()
    for rank in range(3):
        lo, hi = m.shard_range(1000, rank, 3)
        part = m.BatchedGridEnvironment(f, hi - lo, env_id_offset=lo, **kw)
        part.reset(seed=42)
        op = part.step(act[lo:hi])[0]
        assert torch.equal(op, ow[lo:hi])


def _synthetic(n, seed, scale):
    import grid_fed_rl_b200 as m
    cfg = m.NetworkConfig(num_buses=n, connectivity=0.0, load_probability=0.9, dg_probability=0.4,
                          min_load_kw=20, max_load_kw=300, line_length_range=(0.05, 1.5))
    f = m.repair_topology(m.SyntheticFeeder(cfg, seed=seed))
    for ld in f.loads:                       # as generated the feeder is far beyond its loadability
        ld.base_power *= scale; ld.active_power *= scale; ld.reactive_power *= scale
    return f


@pytest.mark.parametrize("lanes", (8, 32, 128))
def test_synthetic_300_bus_feeder_vs_oracle(lanes):
    """A larger radial feeder with hundreds of loads / generators / batteries (BASELINE config 5's
    generator at a size the dense oracle still solves quickly)."""
    import grid_fed_rl_b200 as m
    f = _synthetic(300, 300, 0.1)
    kw = dict(timestep=60.0, renewable_sources=["solar", "wind"], tolerance=1e-8)
    B = 6
    env = m.BatchedGridEnvironment(f, B, lanes=lanes, repair=False, **kw)
    ref = port.PortEnv(f, B, **kw)
    rs = np.random.RandomState(lanes)
    nz0 = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3))], axis=1)
    env.reset(noise=nz0, options={"start_time": 13 * 3600.0}); ref.reset(nz0, start_time=13 * 3600.0)
    lay = obs_layout(ref.n, ref.m, ref.L, ref.G, ref.Bt)
    for t in range(3):
        act = rs.uniform(-1, 1, size=(B, ref.A))
        nz = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3 + ref.L))], axis=1)
        obs, reward, term, trunc, info = env.step(act, nz)
        r = ref.step(act, nz)
        o = obs.cpu().numpy()
        assert r["converged"].all() and bool(info["power_flow_converged"].all())
        assert np.max(np.abs(o[:, lay["vm"]] - r["obs"][:, lay["vm"]])) <= TOL_PU
        assert np.max(np.abs(o[:, lay["va"]] - r["obs"][:, lay["va"]])) <= TOL_PU
        assert np.max(np.abs(o[:, lay["p"]] - r["obs"][:, lay["p"]])) / ref.s_base <= TOL_PU
        assert np.allclose(o[:, lay["gen"]], r["obs"][:, lay["gen"]], rtol=1e-12, atol=1e-6)
        assert np.allclose(o[:, lay["soc"]], r["obs"][:, lay["soc"]], atol=1e-12)
        assert np.allclose(reward.cpu().numpy(), r["reward"], rtol=1e-9, atol=1e-6)
        assert np.all(np.abs(info["iterations"].cpu().numpy().astype(int) - r["iterations"]) <= 1)


def test_synthetic_1000_bus_feeder_runs():
    """BASELINE config 5's feeder: n = 1000, D = 6320, 403 actions.  Functional check: both solvers
    converge to the same state (the dense oracle is too slow at this size)."""
    import grid_fed_rl_b200 as m
    f = _synthetic(1000, 1000, 0.03)
    kw = dict(timestep=60.0, renewable_sources=["solar", "wind"], repair=False, start_time=12 * 3600.0)
    a = m.BatchedGridEnvironment(f, 64, solver="newton", tolerance=1e-9, **kw)          # auto: one CTA per instance
    assert a.launch_info()["lanes"] in (64, 128)
    b = m.BatchedGridEnvironment(f, 64, solver="sweep", tolerance=1e-11, lanes=32, **kw)
    assert a.obs_dim == 6320 and a.act_dim == 403
    a.reset(seed=1); b.reset(seed=1)
    g = torch.Generator(device="cuda"); g.manual_seed(0)
    for _ in range(2):
        act = a.sample_actions(g)
        oa, ra, _, _, ia = a.step(act)
        ob, rb, _, _, ib = b.step(act)
        assert bool(ia["power_flow_converged"].all()) and bool(ib["power_flow_converged"].all())
        assert torch.max(torch.abs(oa[:, :2000] - ob[:, :2000])) <= TOL_PU
        assert torch.allclose(ra, rb, rtol=1e-9, atol=1e-5)


def test_edge_case_feeders_vs_oracle():
    """Smallest feeders, no loads, a single instance, out-of-range actions, loads driven to zero."""
    import grid_fed_rl_b200 as m
    cases = []
    two = m.SimpleRadialFeeder(2)
    cases.append(("two buses", two, {}))
    bare = m.SimpleRadialFeeder(4)
    bare.loads.clear()                                  # no loads at all: only the template battery
    cases.append(("no loads", bare, {}))
    cases.append(("radial 7, no renewables, deterministic", m.SimpleRadialFeeder(7),
                  dict(stochastic_loads=False, weather_variation=False)))
    for name, f, extra in cases:
        for B in (1, 5):
            for solver, tol, ptol in (("newton", 1e-9, 1e-9), ("sweep", 1e-12, 1e-10)):
                kw = dict(timestep=900.0, renewable_sources=["solar", "wind"], **extra)
                env = m.BatchedGridEnvironment(f, B, solver=solver, tolerance=tol, repair=False, **kw)
                ref = port.PortEnv(f, B, tolerance=ptol, **kw)
                rs = np.random.RandomState(B)
                nz0 = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3))], axis=1)
                o0, _ = env.reset(noise=nz0, options={"start_time": 6 * 3600.0})
                r0 = ref.reset(nz0, start_time=6 * 3600.0)
                assert np.max(np.abs(o0.cpu().numpy() - r0)) < 1e-9, name
                for t in range(6):
                    act = rs.uniform(-3, 3, size=(B, ref.A))          # out of range: never clipped upstream
                    nz = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3 + ref.L))], axis=1)
                    if ref.L:
                        nz[:, 4] = -15.0                                  # 1 + 0.1 z < 0: the load clamps at zero
                    obs, reward, term, trunc, info = env.step(act, nz)
                    r = ref.step(act, nz)
                    assert np.array_equal(info["power_flow_converged"].cpu().numpy(), r["converged"]), name
                    assert r["converged"].all(), name
                    assert np.max(np.abs(obs.cpu().numpy()[:, :2 * ref.n] - r["obs"][:, :2 * ref.n])) <= TOL_PU, name
                    assert np.allclose(obs.cpu().numpy(), r["obs"], rtol=1e-9, atol=1e-6), name
                    assert np.allclose(reward.cpu().numpy(), r["reward"], rtol=1e-9, atol=1e-6), name
                    assert np.array_equal(info["constraint_violation_count"].cpu().numpy(), r["viol_count"]), name
                    assert np.array_equal(trunc.cpu().numpy(), r["truncated"]), name
                env.close()


def test_bad_arguments_raise():
    import grid_fed_rl_b200 as m
    f = m.repair_topology(m.IEEE13Bus())
    with pytest.raises(m.InvalidConfigurationError):
        m.BatchedGridEnvironment(f, 4, solver="gauss")
    with pytest.raises(m.InvalidConfigurationError):
        m.BatchedGridEnvironment(f, 0)
    with pytest.raises(m.InvalidConfigurationError):
        m.BatchedGridEnvironment(f, 4, lanes=3)
    with pytest.raises(m.InvalidConfigurationError):
        m.BatchedGridEnvironment(f, 4, device="cpu")
    with pytest.raises(m.NetworkTopologyError):
        m.BatchedGridEnvironment(m.IEEE34Bus(seed=0), 4, repair=False)      # meshed / disconnected as shipped
    env = m.BatchedGridEnvironment(f, 4, renewable_sources=["solar"])
    with pytest.raises(m.InvalidActionError):
        env.step(np.zeros((4, env.act_dim + 1)))
    with pytest.raises(m.InvalidActionError):
        env.step(np.zeros((3, env.act_dim)))


def test_diverging_instances_are_data_not_errors():
    """An overloaded feeder: the reference runs Newton to max_iterations and reports
    converged=False; the env keeps stepping (grid_env.py:724-731).  Flags and iteration counts must
    agree with the oracle; the (chaotic) voltages are not compared."""
    import grid_fed_rl_b200 as m
    f = m.repair_topology(m.IEEE13Bus())
    for ld in f.loads:
        ld.base_power *= 9.0; ld.active_power *= 9.0; ld.reactive_power *= 9.0
    kw = dict(timestep=60.0, renewable_sources=["solar", "wind"], tolerance=1e-6, max_iterations=12)
    B = 48
    for lanes in (4, 16):
        env = m.BatchedGridEnvironment(f, B, lanes=lanes, repair=False, **kw)
        ref = port.PortEnv(f, B, **kw)
        rs = np.random.RandomState(3)
        nz0 = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3))], axis=1)
        env.reset(noise=nz0, options={"start_time": 18 * 3600.0}); ref.reset(nz0, start_time=18 * 3600.0)
        act = rs.uniform(-1, 1, size=(B, ref.A))
        nz = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3 + ref.L))], axis=1)
        with np.errstate(all="ignore"):
            r = ref.step(act, nz)
        obs, reward, term, trunc, info = env.step(act, nz)
        conv = info["power_flow_converged"].cpu().numpy()
        assert not r["converged"].all(), "the case is meant to diverge"
        assert np.array_equal(conv, r["converged"])
        its = info["iterations"].cpu().numpy().astype(int)
        assert np.all(np.abs(its - r["iterations"])[r["converged"]] <= 1)
        assert np.all(its[~r["converged"]] == 12)
        env.step(act, nz)                                   # and the environment keeps going
        assert int(info["current_step"].min()) == 2
        env.close()


@pytest.mark.parametrize("spec,lanes", (("ieee34", 4), ("ieee34", 8), ("ieee123", 8), ("ieee123", 16)))
def test_schedule_variants_agree(spec, lanes):
    """WHERE a hand-off travels - registers along a lane's path, a shared-memory slot between lanes - never
    changes what is computed: a padded pool gives the same bits; another lane assignment (no lane table:
    fewer register hand-offs), the level schedule without path following, and a description cut for another
    lane count (re-cut by the library) give the same values to rounding and the same iteration counts."""
    import dataclasses
    import grid_fed_rl_b200 as m
    from grid_fed_rl_b200.topology import compile_feeder
    f = m.repair_topology({"ieee34": lambda: m.IEEE34Bus(seed=0), "ieee123": lambda: m.IEEE123Bus(seed=0)}[spec]())
    kw = dict(renewable_sources=["solar", "wind"], root="center")
    default = compile_feeder(f, width=lanes, paths=True, **kw)
    assert default.lane_of is not None
    n = default.n_bus
    plans = {
        "default": default,
        "padded": dataclasses.replace(default, n_pool=min(n, 40)),
        "no_lane_table": dataclasses.replace(default, lane_of=None),
        "level_schedule": compile_feeder(f, width=lanes, paths=False, **kw),
        "other_width": compile_feeder(f, width=2 * lanes, paths=True, **kw),
    }
    B = 96
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    ref = None
    for name, soa in plans.items():
        env = m.BatchedGridEnvironment(soa, B, solver="newton", tolerance=1e-6, lanes=lanes, repair=False,
                                       start_time=12 * 3600.0)
        assert env.launch_info()["lanes"] == lanes
        env.reset(seed=3)
        if ref is None:
            acts = [env.sample_actions(g) for _ in range(3)]
        outs = []
        for a in acts:
            obs, reward, term, trunc, info = env.step(a)
            outs.append((obs.clone(), reward.clone(), info["iterations"].clone(), info["max_mismatch"].clone()))
        assert bool(info["power_flow_converged"].all()), name
        if ref is None:
            ref = outs
        else:
            for (o, r, it, mm), (o0, r0, it0, mm0) in zip(outs, ref):
                if name == "padded":
                    assert torch.equal(o, o0) and torch.equal(r, r0) and torch.equal(it, it0) and torch.equal(mm, mm0), name
                else:
                    # another schedule sums a bus's children in another order: same values to rounding
                    # (line flows are in W: rounding noise of 1e-16 x 1e7 VA; voltages and angles in pu / rad)
                    assert torch.allclose(o, o0, rtol=1e-11, atol=1e-6) and torch.equal(it, it0), name
                    assert torch.allclose(o[:, :2 * n], o0[:, :2 * n], rtol=0, atol=1e-11), name
        env.close()


# ----------------------------------------------------------------------------- meshed networks (dense path)

@pytest.mark.parametrize("name", golden_names("meshsolve_"))
def test_dense_solver_matches_reference_on_meshed_networks(name):
    """Networks with cycles (loop-closing lines kept): the dense Newton-Raphson kernel against the
    frozen outputs of the reference's own solver, through solve(buses, lines, loads, generation)
    and through the batched form."""
    import grid_fed_rl_b200 as m
    from grid_fed_rl_b200.solver import is_radial
    g = load_golden(name)
    f = feeder_for(g)
    assert not is_radial(f.buses, f.lines)
    tol, max_it = float(g["meta"][0]), int(g["meta"][1])
    unknowns = 2 * (len(f.buses) - 1)
    if unknowns > 165:
        pytest.skip("too large for the dense kernels: see test_sweep_takes_meshed_networks")
    for method, where in (("dense", "auto"), ("auto", "auto"), ("dense", "shared"), ("dense", "registers")):
        if where == "registers" and unknowns > 127:
            continue
        solver = m.B200PowerFlowSolver(tolerance=tol, max_iterations=max_it, method=method, dense_kernel=where)
        sol = solver.solve_batch(f, g["p_spec"])
        conv = g["converged"]
        assert np.array_equal(sol.converged.cpu().numpy(), conv)
        assert np.all(np.abs(sol.iterations.cpu().numpy().astype(int) - g["iterations"]) <= 1)
        if conv.any():
            for k in ("bus_voltages", "bus_angles", "line_flows", "losses"):
                got = getattr(sol, k).cpu().numpy()
                assert np.max(np.abs(got[conv] - g[k][conv])) <= TOL_PU, k
            s_base = f.parameters.base_power * 1e6
            got = sol.line_loadings.cpu().numpy()     # D1: |S| s_base / rating; the frozen reference has |S| / rating
            assert np.allclose(got[conv], g["line_loadings"][conv] * s_base, rtol=1e-7, atol=1e-12)
        # the reference's 4-argument call shape, one case
        p = g["p_spec"][0]
        loads = {b.id: -p[i] for i, b in enumerate(f.buses) if p[i] < 0}
        gen = {b.id: p[i] for i, b in enumerate(f.buses) if p[i] > 0}
        one = solver.solve(f.buses, f.lines, loads, gen)
        assert one.converged == bool(conv[0]) and abs(one.iterations - int(g["iterations"][0])) <= 1
        if conv[0]:
            assert np.max(np.abs(one.bus_voltages - g["bus_voltages"][0])) <= TOL_PU
            assert np.max(np.abs(one.line_flows - g["line_flows"][0])) <= TOL_PU
        solver.close()


def test_dense_and_tree_solvers_agree_on_radial_feeders():
    """On a radial feeder both paths run the same Newton iterates: same iteration counts, same state."""
    import grid_fed_rl_b200 as m
    f = m.repair_topology(m.IEEE34Bus(seed=0))
    rs = np.random.RandomState(3)
    n = len(f.buses)
    base = np.zeros(n)
    idx = {b.id: i for i, b in enumerate(f.buses)}
    for ld in f.loads:
        base[idx[ld.bus]] += ld.base_power / (f.parameters.base_power * 1e6)
    p = -base[None, :] * rs.uniform(0.2, 1.5, size=(300, n))
    tree = m.B200PowerFlowSolver(tolerance=1e-8, method="newton").solve_batch(f, p)
    dense = m.B200PowerFlowSolver(tolerance=1e-8, method="dense").solve_batch(f, p)
    assert bool(tree.converged.all()) and bool(dense.converged.all())
    assert torch.equal(tree.iterations, dense.iterations)
    for k in ("bus_voltages", "bus_angles", "line_flows", "losses"):
        assert torch.max(torch.abs(getattr(tree, k) - getattr(dense, k))) < 1e-10, k
    assert torch.allclose(tree.line_loadings, dense.line_loadings, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("num_buses,conn,seed", [(9, 0.3, 1), (14, 0.2, 2), (28, 0.08, 3), (33, 0.06, 4),
                                                 (47, 0.04, 5), (49, 0.04, 6), (60, 0.03, 7), (70, 0.03, 8)])
def test_dense_register_and_shared_memory_kernels_agree(num_buses, conn, seed):
    """The register-resident Gauss-Jordan elimination against the shared-memory LU on eight meshes with 16, 26, 54,
    64, 92, 96, 118 and 138 unknowns (register tiles R = 2, 4, 7, 8, 12, 12, 15: both sides of the switches from 8 to
    16 to 32 thread columns at 56 and 96 unknowns, and one network beyond the register kernel's 127): same pivots,
    so the same convergence flags and iteration counts and the same state to rounding; above 127 unknowns "auto" is
    the shared-memory kernel and "registers" is refused.  Every R, odd and even N, against the oracle:
    tests/test_gpu_newton_iterates.py."""
    import grid_fed_rl_b200 as m
    f = m.repair_topology(m.SyntheticFeeder(m.NetworkConfig(num_buses=num_buses, connectivity=conn,
                                                            load_probability=0.9, dg_probability=0.3), seed=seed),
                          keep_cycles=True)
    n = len(f.buses)
    rs = np.random.RandomState(seed)
    base = np.zeros(n)
    idx = {b.id: i for i, b in enumerate(f.buses)}
    for ld in f.loads:
        base[idx[ld.bus]] += ld.base_power / (f.parameters.base_power * 1e6)
    p = -base[None, :] * (0.3 / max(base.sum(), 1e-9)) * rs.uniform(0.0, 2.0, size=(517, n))
    p[5] *= 3000.0                                            # one instance far beyond the nose: must not converge
    shared = m.B200PowerFlowSolver(tolerance=1e-8, max_iterations=15, method="dense", dense_kernel="shared")
    a = shared.solve_batch(f, p)
    unknowns = 2 * (n - 1)
    if unknowns > 127:
        with pytest.raises(m.GridLimitError):
            m.B200PowerFlowSolver(method="dense", dense_kernel="registers").solve_batch(f, p)
        b = m.B200PowerFlowSolver(tolerance=1e-8, max_iterations=15, method="dense").solve_batch(f, p)
        for k in ("bus_voltages", "bus_angles", "line_flows", "losses", "iterations", "converged"):
            assert torch.equal(getattr(a, k), getattr(b, k)), k
        return
    b = m.B200PowerFlowSolver(tolerance=1e-8, max_iterations=15, method="dense", dense_kernel="registers").solve_batch(f, p)
    assert torch.equal(a.converged, b.converged)
    assert int(a.converged.sum()) >= 500 and not bool(a.converged[5])
    c = a.converged
    assert torch.equal(a.iterations[c], b.iterations[c])
    for k in ("bus_voltages", "bus_angles", "line_flows", "losses"):
        assert torch.max(torch.abs(getattr(a, k)[c] - getattr(b, k)[c])) < 1e-10, k


def test_dense_solver_limits_and_singular_network():
    import grid_fed_rl_b200 as m
    f = m.repair_topology(m.IEEE123Bus(seed=0))          # 244 unknowns: does not fit an SM's shared memory
    with pytest.raises(m.GridLimitError):
        m.B200PowerFlowSolver(method="dense").solve_batch(f, np.zeros((1, len(f.buses))))
    # a bus hanging on an open line (|z| <= 1e-12 -> y = 0, power_flow.py:61-64): singular Jacobian,
    # the reference warns and stops; converged = False after one iteration
    g = m.SimpleRadialFeeder(4)
    g.lines[-1].resistance = g.lines[-1].reactance = 0.0
    p = np.array([[0.0, -0.01, -0.01, -0.01]])
    for where in ("shared", "registers"):
        sol = m.B200PowerFlowSolver(method="dense", dense_kernel=where).solve_batch(g, p)
        assert not bool(sol.converged[0]) and int(sol.iterations[0]) == 1


# ----------------------------------------------------------------------------- weakly meshed feeders (sweep + compensation)

@pytest.mark.parametrize("lanes", (1, 8, 32, 64))
@pytest.mark.parametrize("name", golden_names("meshtrace_"))
def test_sweep_steps_meshed_feeders(name, lanes):
    """Environments on feeders with their loop-closing lines kept (the shipped IEEE-34 loop, IEEE-123's 26 ties, a
    synthetic mesh with 37): the reference steps them with its dense Newton-Raphson (frozen traces, pinned to the
    oracle at their own tolerance by test_oracle_golden); the kernels walk the spanning tree and restore the loops
    by compensation - one current per tie, corrected every iteration through the inverse loop-impedance matrix."""
    g = port_trace(load_golden(name), tolerance=1e-10)
    exact = replay_trace(_factory("sweep", lanes, 1e-11), g, ctx=f"{name}/sweep/lanes{lanes}", check_iterations=False)
    assert exact >= 0.9 * g["obs"].shape[0]


@pytest.mark.parametrize("name", [n for n in golden_names("meshsolve_") if "overload" not in n])
def test_sweep_takes_meshed_networks(name):
    """The solver surface on meshed networks through the sweep (any size the tree kernels take - IEEE-123 with its 26
    ties is beyond the dense kernels; method="auto" falls back to this path there), against the frozen reference."""
    import grid_fed_rl_b200 as m
    g = load_golden(name)
    f = feeder_for(g)
    conv = g["converged"]
    net = port.DenseNetwork(f.buses, f.lines)
    ref = port.newton_raphson(net, g["p_spec"], 1e-10, 50)
    methods = [("sweep", 1e-11, 300)]
    if 2 * (len(f.buses) - 1) > 165:
        methods.append(("auto", 1e-8, 50))
        with pytest.raises(m.GridLimitError):
            m.B200PowerFlowSolver(method="dense").solve_batch(f, g["p_spec"])
    for method, tol, max_it in methods:
        for lanes in (0, 8, 32):
            sol = m.B200PowerFlowSolver(tolerance=tol, max_iterations=max_it, method=method, lanes=lanes).solve_batch(f, g["p_spec"])
            assert bool(sol.converged.all()) and conv.all()
            for k in ("bus_voltages", "bus_angles", "line_flows", "losses"):
                assert np.max(np.abs(getattr(sol, k).cpu().numpy() - ref[k])) <= TOL_PU, (method, k)
            # and against the frozen reference run itself (its own tolerance: 1e-8 or looser)
            assert np.max(np.abs(sol.bus_voltages.cpu().numpy() - g["bus_voltages"])) <= 1e-6
    with pytest.raises(m.NetworkTopologyError):
        m.B200PowerFlowSolver(method="newton").solve_batch(f, g["p_spec"])


def test_meshed_environment_options():
    """keep_cycles=True: a repair keeps the loop-closing lines (sweep only); the default repair drops them (D4-iii)."""
    import grid_fed_rl_b200 as m
    raw = m.IEEE123Bus(seed=0)
    a = m.BatchedGridEnvironment(raw, 8, solver="sweep", tolerance=1e-10, renewable_sources=["solar", "wind"])
    b = m.BatchedGridEnvironment(raw, 8, solver="sweep", tolerance=1e-10, renewable_sources=["solar", "wind"], keep_cycles=True)
    assert a.soa.n_tie == 0 and a.soa.n_line == 122 and b.soa.n_tie == 26 and b.soa.n_line == 148
    assert b.obs_dim == a.obs_dim + 2 * 26
    with pytest.raises(m.InvalidConfigurationError):
        m.BatchedGridEnvironment(raw, 8, solver="newton", keep_cycles=True)
    b.reset(seed=1)
    g = torch.Generator(device="cuda"); g.manual_seed(0)
    obs, reward, term, trunc, info = b.step(b.sample_actions(g))
    assert bool(info["power_flow_converged"].all()) and torch.isfinite(obs).all()
