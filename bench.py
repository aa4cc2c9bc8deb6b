#!/usr/bin/env python
"""bench.py - env-steps/s of the fused batched GridEnvironment.step on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload ieee123|ieee13|ieee34|...] [--lanes L]
                  [--scaling weak|strong] [--no-configs] [--no-cpu] [--dump-outputs DIR]
  python bench.py --impl reference ...      # the CPU oracle (port of the reference path) on host cores

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over one batch of
instances: load / weather / battery update, Newton-Raphson (or sweep) load flow, constraints,
reward, observation - one kernel launch.  Inputs (actions) are resident in HBM for `value`;
`e2e` repeats the measurement through the public API with pinned HOST action buffers and a
device->host read of reward + done flags every step.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# workload name -> (feeder spec, per-GPU instances, solver, tolerance, max_iterations)
WORKLOADS = {
    # BASELINE.json configs[3]: the configuration the metric is quoted on; 131,072 per GPU
    # (x8 = 1,048,576 instances), weak scaling
    "ieee123": ("ieee123", 131072, "newton", 1e-6, 50),
    "ieee13": ("ieee13", 65536, "sweep", 1e-8, 50),       # configs[1]
    "ieee34": ("ieee34", 262144, "sweep", 1e-8, 50),      # configs[2]
    "ieee13_newton": ("ieee13", 65536, "newton", 1e-6, 50),
    "ieee34_newton": ("ieee34", 262144, "newton", 1e-6, 50),
    "ieee123_sweep": ("ieee123", 131072, "sweep", 1e-8, 50),
    # IEEE-123 with its 26 loop-closing tie lines KEPT (148 lines): sweep on the spanning tree + compensation
    "ieee123_mesh": ("ieee123mesh", 131072, "sweep", 1e-8, 100),
    # configs[4]: synthetic 1,000-bus radial feeder, 16,384 instances over 8 GPUs
    "synthetic1000": ("synthetic1000", 2048, "newton", 1e-6, 50),
}
ENV_KW = dict(timestep=1.0, renewable_sources=["solar", "wind"], stochastic_loads=True,
              weather_variation=True)
START_TIME = 12 * 3600.0     # daylight, so the solar branch is exercised (SURVEY 8d)


def make_feeder(spec):
    import grid_fed_rl_b200 as m
    if spec == "synthetic1000":
        # ScalableFeeder(1000)'s parameters (synthetic.py:236-252) but radial; loads scaled by 0.03 so that
        # the feeder is inside its loadability (sum P = 0.43 pu; SURVEY 8d config 5)
        cfg = m.NetworkConfig(num_buses=1000, connectivity=0.0, load_probability=0.9, dg_probability=0.4,
                              min_load_kw=20, max_load_kw=300, line_length_range=(0.05, 1.5))
        f = m.repair_topology(m.SyntheticFeeder(cfg, seed=1000))
        for ld in f.loads:
            ld.base_power *= 0.03; ld.active_power *= 0.03; ld.reactive_power *= 0.03
        return f
    if spec == "ieee123mesh":
        return m.repair_topology(m.IEEE123Bus(seed=0), keep_cycles=True)
    f = {"ieee13": m.IEEE13Bus, "ieee34": lambda: m.IEEE34Bus(seed=0),
         "ieee123": lambda: m.IEEE123Bus(seed=0)}[spec]()
    return m.repair_topology(f)


def algorithmic_bytes(soa):
    """SURVEY 8(d): reads actions + state, writes state + observation + outputs, per env-step."""
    return 8 * soa.obs_dim + 8 * soa.act_dim + 32 * soa.n_bat + 199


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop_evt.wait(0.004)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def physical_gpu_index(local_index):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_index])
        except Exception:
            return local_index
    return local_index


# ----------------------------------------------------------------------------- CPU oracle legs

def _cpu_worker(args):
    spec, B, steps, solver_tol, seed, threads = args
    import numpy as np
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=threads)
    except Exception:
        import contextlib
        ctx = contextlib.nullcontext()
    from oracle import port
    f = make_feeder(spec)
    with ctx:
        env = port.PortEnv(f, B, tolerance=solver_tol, **ENV_KW)
        rs = np.random.RandomState(seed)
        nz0 = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3))], axis=1)
        env.reset(nz0, start_time=START_TIME)
        acts = [rs.uniform(-1, 1, size=(B, env.A)) for _ in range(steps + 1)]
        nzs = [np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3 + env.L))], axis=1)
               for _ in range(steps + 1)]
        env.step(acts[0], nzs[0])                       # warm-up (allocations, BLAS threads)
        t0 = time.perf_counter()
        conv = 0
        for t in range(steps):
            conv += int(env.step(acts[t + 1], nzs[t + 1])["converged"].sum())
        dt = time.perf_counter() - t0
    return B * steps, dt, conv


def cpu_baseline(spec, tol, B=32, steps=2):
    """The oracle (numpy port of the reference's step + dense Newton-Raphson) on ONE host thread."""
    n, dt, conv = _cpu_worker((spec, B, steps, tol, 0, 1))
    return {"value": n / dt, "unit": "env-steps/s", "cores": 1, "kind": "port",
            "sample": f"oracle/port.py PortEnv, {spec}, {B} instances x {steps} steps, dense NR tol {tol:g}, "
                      f"1 thread, {dt:.1f} s", "converged_frac": conv / n}


def _ref_server(conn, spec, B, tol, seed):
    """A warm oracle worker: one PortEnv over its own shard, one step per 'go'."""
    import numpy as np
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=1)
    except Exception:
        pass
    from oracle import port
    env = port.PortEnv(make_feeder(spec), B, tolerance=tol, **ENV_KW)
    rs = np.random.RandomState(seed)
    env.reset(np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3))], axis=1),
              start_time=START_TIME)
    conn.send("ready")
    while True:
        msg = conn.recv()
        if msg == "stop":
            break
        act = rs.uniform(-1, 1, size=(B, env.A))
        nz = np.concatenate([rs.random_sample((B, 1)), rs.standard_normal((B, 3 + env.L))], axis=1)
        out = env.step(act, nz)
        conn.send(int(out["converged"].sum()))


def run_reference(args):
    """--impl reference: the CPU oracle (numpy port of the reference's step with its dense
    Newton-Raphson; the reference itself is Python and does not travel to the GPU box) on every
    host core: one single-threaded process per core, each stepping its own shard of instances."""
    import multiprocessing as mp
    spec, B_gpu, solver, tol, max_it = WORKLOADS[args.workload]
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = os.cpu_count() or 1
    per_proc = {"ieee123": 48, "ieee123mesh": 48, "ieee34": 384, "ieee13": 2048, "synthetic1000": 1}[spec]
    ptol = tol if solver == "newton" else 1e-8
    steps, warm = max(1, args.steps), max(0, args.warmup)
    ctx = mp.get_context("spawn")
    procs = []
    for i in range(cores):
        parent, child = ctx.Pipe()
        pr = ctx.Process(target=_ref_server, args=(child, spec, per_proc, ptol, 100 + i), daemon=True)
        pr.start()
        procs.append((pr, parent))
    for _, c in procs:
        assert c.recv() == "ready"

    def one_step():
        for _, c in procs:
            c.send("go")
        return sum(c.recv() for _, c in procs)

    for _ in range(warm):
        one_step()
    t0 = time.perf_counter()
    conv = 0
    for _ in range(steps):
        conv += one_step()
    wall = time.perf_counter() - t0
    for pr, c in procs:
        c.send("stop")
    for pr, _ in procs:
        pr.join(timeout=5)
    total = per_proc * cores * steps
    value = total / wall
    line = {"metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": 1e3 * wall / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": f"{spec} GridEnvironment.step, CPU oracle (oracle/port.py: dense "
                                   f"Newton-Raphson tol {ptol:g}), bounded sample of {per_proc * cores} "
                                   f"instances per step", "instances_per_step": per_proc * cores},
            "converged_frac": conv / total,
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                             "sample": f"{cores} single-threaded processes x {per_proc} instances x {steps} steps"},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm

L2_BYTES = 126e6          # B200: 2 x 63 MB


def load_profile_facts():
    """Per-workload facts measured with ncu and kept under profiles/ (written by profiles/summarize_ncu.py
    --json from the committed captures): DRAM bytes per launch, FP64 lane operations per env-step."""
    facts = {}
    pdir = os.path.join(ROOT, "profiles")
    try:
        names = sorted(n for n in os.listdir(pdir) if n.startswith("r02_ncu_") and n.endswith(".json"))
    except OSError:
        names = []
    for n in names:
        try:
            with open(os.path.join(pdir, n)) as fh:
                j = json.load(fh)
            facts[(j["workload"], int(j["instances"]))] = dict(j, source="profiles/" + n)
        except Exception:
            pass
    return facts


def reference_cpu_rates():
    try:
        with open(os.path.join(ROOT, "profiles", "r02_reference_cpu_rates.json")) as fh:
            return json.load(fh)
    except Exception:
        return None


def bind_to_gpu_numa_node(index):
    """Pin this rank to the CPUs next to its GPU before any pinned buffer is allocated (NUMA-local staging
    buffers: with 8 ranks sharing one host the observation copies otherwise cross sockets)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, mk in enumerate(mask) for b in range(64) if (mk >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def device_timed(dev, world, step_fn, k, max_over_ranks):
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(k):
        step_fn(i)
    ev1.record()
    barrier()
    return max_over_ranks(ev0.elapsed_time(ev1), dev)     # a timed region counts as its slowest rank


def make_envs(m, name, B, dev, rank, lanes, seed, obs_dtype=None, min_bytes=2 * L2_BYTES, obs_buffers=0):
    """The environment(s) of one workload: when one step's working set would sit in the 126 MB L2, several
    environments are stepped round-robin so that every step streams from / to HBM."""
    spec, _, solver, tol, max_it = WORKLOADS[name]
    feeder = make_feeder(spec)
    kw = dict(ENV_KW)
    if obs_dtype is not None:
        kw["obs_dtype"] = obs_dtype
    if obs_buffers:
        kw["obs_buffers"] = obs_buffers
    envs = []
    while True:
        env = m.BatchedGridEnvironment(feeder, B, device=dev, solver=solver, tolerance=tol, max_iterations=max_it,
                                       lanes=lanes, repair=False, start_time=START_TIME,
                                       env_id_offset=(rank * 16 + len(envs)) * B, **kw)
        env.reset(seed=seed)
        envs.append(env)
        if len(envs) * B * algorithmic_bytes(env.soa) >= min_bytes or len(envs) >= 8:
            return envs


def measure_device(m, lib, name, B, dev, world, rank, lanes, seed, K, W, max_over_ranks, peak, facts):
    """Device-resident arm of one workload: actions in HBM, one kernel launch per step, CUDA events."""
    import torch
    import torch.distributed as dist
    envs = make_envs(m, name, B, dev, rank, lanes, seed)
    env = envs[0]
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    R = 4
    actions = [env.sample_actions(gen) for _ in range(R)]
    E = len(envs)
    last = [None]

    def dev_step(i):
        last[0] = envs[i % E].step(actions[i % R])

    for i in range(max(W, E)):
        dev_step(i)
    l0 = lib.gfr_launch_count()
    ms = device_timed(dev, world, dev_step, K, max_over_ranks)
    launches = lib.gfr_launch_count() - l0
    info = env._info()
    conv = float(info["power_flow_converged"].double().mean().item())
    its = float(info["iterations"].double().mean().item())
    if world > 1:
        t = torch.tensor([conv, its], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        conv, its = (t / world).tolist()
    soa, li = env.soa, env.launch_info()
    abytes = algorithmic_bytes(soa)
    solver = WORKLOADS[name][2]
    value = B * world * K / (ms * 1e-3)
    achieved = abytes * B / (ms / K * 1e-3) / 1e9          # GB/s of the one kernel a step launches
    ws = B * abytes
    fact = facts.get((name, B))
    res = {
        "value": value, "ms_per_step": ms / K, "steps": K, "converged_frac": conv, "mean_iterations": its,
        "workload": f"{WORKLOADS[name][0]} fused GridEnvironment.step, {solver} load flow tol {WORKLOADS[name][3]:g}, "
                    f"{B} instances per GPU, in-kernel Philox noise, random U(-1,1) policy",
        "instances_per_gpu": B, "n_bus": soa.n_bus, "obs_dim": soa.obs_dim, "act_dim": soa.act_dim, "solver": solver,
        "launch": li,
        "l2": (f"per-step working set {ws / 1e6:.0f} MB > 2 x 126 MB L2: no flush needed" if E == 1 else
               f"per-step working set {ws / 1e6:.0f} MB would sit in the 126 MB L2: {E} environments stepped "
               f"round-robin ({E * ws / 1e6:.0f} MB between two visits of the same buffers)"),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak[0], "unit": "GB/s", "frac": achieved / peak[0],
                     "traffic": fact.get("dram_bytes_per_launch") if fact else None,
                     "traffic_source": fact.get("source") if fact else None,
                     "peak_source": peak[1], "algorithmic_bytes_per_env_step": abytes,
                     "kernel": f"step_kernel<{li['lanes']},{solver}>", "kernel_ms": ms / K},
        "gpu_launches": int(launches),
    }
    return res, envs, actions, last[0]


DUMP_BYTES = 60_000_000      # array data of one --dump-outputs directory (64 MB with the .npy headers, with room)


def dump_outputs(out_dir, outputs, limit=DUMP_BYTES):
    """Writes one step's outputs - what ``BatchedGridEnvironment.step`` returns: observation, reward, the two done
    flags and every tensor of ``info`` - as ``<out_dir>/<name>.npy``, so that two builds can be compared output for
    output.  Every array keeps the same instances (rows): all of them when they fit in ``limit`` bytes, else a sorted
    sample drawn with a fixed seed; ``rows.npy`` lists them.  fp32 / fp64 arrays keep their type, flags and counters
    become fp64 (exactly)."""
    import numpy as np
    import torch
    obs, reward, terminated, truncated, info = outputs
    arrays = {"obs": obs, "reward": reward, "terminated": terminated, "truncated": truncated}
    arrays.update((k, v) for k, v in info.items() if isinstance(v, torch.Tensor))
    arrays = {k: v if v.dtype in (torch.float32, torch.float64) else v.to(torch.float64) for k, v in arrays.items()}
    B = obs.shape[0]
    row_bytes = 8 + sum(v[0].numel() * v.element_size() for v in arrays.values())
    n = min(B, limit // row_bytes)
    rows = np.arange(B) if n == B else np.sort(np.random.default_rng(0).choice(B, size=n, replace=False))
    idx = torch.as_tensor(rows, device=obs.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.index_select(0, idx).cpu().numpy())


def run_gpu(args):
    import torch
    import torch.distributed as dist
    import grid_fed_rl_b200 as m
    from grid_fed_rl_b200 import _native
    from grid_fed_rl_b200.distributed import max_over_ranks

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU oracle")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = bind_to_gpu_numa_node(physical_gpu_index(local))
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    spec, B, solver, tol, max_it = WORKLOADS[args.workload]
    if args.scaling == "strong":
        # SURVEY 8(d) config 4: 1,048,576 instances in total, split evenly over the GPUs
        total = args.total_envs or 1_048_576
        B = total // world
    if args.envs:
        B = args.envs
    lib = _native.load_library()
    K, W = args.steps, max(args.warmup, 3)
    peak = hbm_peak()
    facts = load_profile_facts()

    sampler = ClockSampler(physical_gpu_index(local))
    sampler.start()
    main, envs, actions, last = measure_device(m, lib, args.workload, B, dev, world, rank, args.lanes, args.seed, K, W,
                                               max_over_ranks, peak, facts)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)       # before the end-to-end arms step the environment again
    env = envs[0]
    value, ms = main["value"], main["ms_per_step"] * K
    if args.kernel_only:                 # tuning aid (tools/): the device-resident arm only
        sampler.stop()
        if rank == 0:
            print(json.dumps({"value": value, "ms_per_step": ms / K, "mean_iterations": main["mean_iterations"],
                              "converged_frac": main["converged_frac"],
                              "config": {"launch": main["launch"], "instances_per_gpu": B}}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- end-to-end arm: every step copies ITS actions from pinned host memory (H2D) and its result back (D2H),
    #      and the host reads each step's result.  Through the public API (HostStepper over
    #      BatchedGridEnvironment.step): serial (copy, step, copy, synchronise), as a depth-2 pipeline (the next
    #      step's action copy overlaps the running kernel on a second stream), and with every step's OBSERVATION
    #      brought to the host too - what a host-side policy sees (fp64, and fp32 as the reference declares its
    #      observation space, written by the kernel into alternating buffers so that the copy of step t overlaps
    #      the kernel of step t + 1).
    from grid_fed_rl_b200.pipeline import HostStepper
    R = len(actions)
    host_act = [a.cpu().pin_memory() for a in actions]

    def e2e_run(e, depth, observations=False, k_steps=None):
        stepper = HostStepper(e, depth=depth, observations=observations)
        checksum = [0.0]
        k_run = k_steps or K

        def run(k):
            for i in range(k):
                stepper.submit(host_act[i % R])
                if i + 1 >= depth:
                    checksum[0] += float(stepper.result()["reward"][0])      # the host consumes the result
            while stepper._pending:
                checksum[0] += float(stepper.result()["reward"][0])

        run(3)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        run(k_run)
        ev1.record()
        barrier()
        return max_over_ranks(ev0.elapsed_time(ev1), dev), stepper

    K_obs = max(2, min(K, 20))
    ms_obs, st_obs = e2e_run(env, 2, observations=True, k_steps=K_obs)
    obs64 = {"value": B * world * K_obs / (ms_obs * 1e-3), "d2h_bytes_per_step": st_obs.d2h_bytes_per_step, "steps": K_obs,
             "gb_per_s_d2h": st_obs.d2h_bytes_per_step / (ms_obs / K_obs * 1e-3) / 1e9, "dtype": "f64"}
    del st_obs
    ms_serial, stepper = e2e_run(env, 1)
    ms_e2e, stepper = e2e_run(env, 2)
    e2e_value = B * world * K / (ms_e2e * 1e-3)
    e2e_serial = B * world * K / (ms_serial * 1e-3)
    h2d, d2h = stepper.h2d_bytes_per_step, stepper.d2h_bytes_per_step
    del stepper
    for e in envs:
        e.close()
    envs = []
    # fp32 observations, alternating device buffers (a second environment: the option is fixed at construction)
    env32 = make_envs(m, args.workload, B, dev, rank, args.lanes, args.seed, obs_dtype="float32", min_bytes=0)[0]
    ms32, st32 = e2e_run(env32, 2, observations=True, k_steps=K_obs)
    obs32 = {"value": B * world * K_obs / (ms32 * 1e-3), "d2h_bytes_per_step": st32.d2h_bytes_per_step, "steps": K_obs,
             "gb_per_s_d2h": st32.d2h_bytes_per_step / (ms32 / K_obs * 1e-3) / 1e9, "dtype": "f32",
             "note": "observation written as fp32 by the kernel (the reference declares float32, grid_env.py:346) into "
                     "two alternating device buffers; the copy of step t runs on the copy stream under the kernel of "
                     "step t + 1"}
    del st32
    env32.close()

    # ---- the other BASELINE configurations, device-resident arm only, in the same JSON line
    others = {}
    if not args.no_configs and args.scaling == "weak":
        for name in ("ieee13", "ieee34", "synthetic1000", "ieee13_newton", "ieee34_newton", "ieee123_mesh"):
            if name == args.workload:
                continue
            Bn = WORKLOADS[name][1]
            Kn = max(20, min(K, 200))
            res, es, _, _ = measure_device(m, lib, name, Bn, dev, world, rank, 0, args.seed, Kn, W, max_over_ranks, peak, facts)
            for e in es:
                e.close()
            others[name] = res
        others["synthetic1000_rollout"] = measure_rollout(m, dev, world, rank, max_over_ranks, args)
    clocks = sampler.stop()          # sampled across the timed regions

    fp64_peak = ctypes.c_double(0.0)
    if rank == 0:
        _native.check(lib, lib.gfr_fp64_peak(local, ctypes.byref(fp64_peak)))
        fact = facts.get((args.workload, B))
        lane_ops = fact.get("fp64_lane_ops_per_env_step") if fact else None
        line = {
            "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": main["workload"], "instances_per_gpu": B, "total_instances": B * world,
                       "n_bus": main["n_bus"], "obs_dim": main["obs_dim"], "act_dim": main["act_dim"], "solver": solver,
                       "parallelism": f"shard{world}", "l2": main["l2"], "launch": main["launch"],
                       "numa_bound_cpus": numa_cpus},
            "converged_frac": main["converged_frac"], "converged_solves_per_s": value * main["converged_frac"],
            "mean_iterations": main["mean_iterations"],
            "roofline": dict(main["roofline"],
                             note="not HBM bound: ncu shows issue slots and the L1 / shared-memory data pipe as the busiest "
                                  "units (DESIGN.md section 5, profiles/r02_*); see also `fp64`"),
            # FP64 side (the contract's roofline bounds are hbm | tensor; this kernel is neither): FP64 lane operations
            # per env-step (ncu: executed DFMA / DMUL / DADD thread instructions / instances, profiles/) x env-steps/s,
            # against the DFMA issue rate measured on this device just now (gfr_fp64_peak)
            "fp64": {"lane_ops_per_env_step": lane_ops,
                     "achieved_gops": (lane_ops * value / world / 1e9) if lane_ops else None,
                     "peak_gops": fp64_peak.value * 1e3 / 2.0, "peak_dfma_tflops": fp64_peak.value,
                     "frac": (lane_ops * value / world / 1e9 / (fp64_peak.value * 1e3 / 2.0))
                             if fp64_peak.value and lane_ops else None,
                     "source": fact.get("source") if fact else None},
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / K,
                    "serial_value": e2e_serial, "serial_ms_per_step": ms_serial / K,
                    "with_observations": obs64, "with_observations_f32": obs32,
                    "note": "HostStepper (public API): pinned host actions in, reward + terminated + truncated out, every "
                            "step, each result read by the host; `value` = depth-2 pipeline, `serial_value` = "
                            "copy-step-copy-sync.  `value` is what a DEVICE-side policy sees (the observation stays in "
                            "HBM); a HOST-side policy sees `with_observations_f32` (or `with_observations` in fp64): "
                            "every observation row crosses PCIe"},
            "gpu_launches": main["gpu_launches"], "clocks": clocks,
            "configs": others,
        }
        ref = reference_cpu_rates()
        if ref:
            line["reference_cpu_measured_in_build_container"] = ref
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(spec, tol if solver == "newton" else 1e-8,
                                                *{"ieee123": (256, 12), "ieee123mesh": (256, 12), "ieee34": (2048, 12), "ieee13": (16384, 12), "synthetic1000": (2, 2)}[spec])
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_rollout(m, dev, world, rank, max_over_ranks, args):
    """BASELINE configs[4]: synthetic 1,000-bus feeder, 2,048 instances per GPU (16,384 over 8), generating offline
    rollout data: GraphedCollector replays chunks of steps (action sampling, fused step, copies into the
    {observations, actions, rewards, next_observations, terminals} block, masked reset) as one CUDA graph."""
    import torch
    from grid_fed_rl_b200.compat import GraphedCollector
    name = "synthetic1000"
    B, chunk, chunks = WORKLOADS[name][1], 4, 6
    # the block is fp32 like the reference's GridDataset arrays: the kernel writes its observation in fp32 too (one
    # buffer: a captured graph replays fixed pointers), so the copies into the block are plain copies
    env = make_envs(m, name, B, dev, rank, 0, args.seed, obs_dtype="float32", min_bytes=0, obs_buffers=1)[0]
    col = GraphedCollector(env, chunk=chunk, dtype=torch.float32)
    col.run_chunk(); col.run_chunk()                       # eager + capture, then one replay
    ms = device_timed(dev, world, lambda i: col.run_chunk(), chunks, max_over_ranks)
    steps = chunks * chunk
    bytes_per_step = B * 4 * (2 * env.obs_dim + env.act_dim + 2)
    out = {"value": B * world * steps / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms / steps,
           "instances_per_gpu": B, "steps": steps, "chunk": chunk,
           "rollout_bytes_per_step": bytes_per_step, "rollout_gb_per_s_per_gpu": bytes_per_step / (ms / steps * 1e-3) / 1e9,
           "obs_dtype": "f32",
           "note": "transitions land in a device-resident fp32 block with the reference's GridDataset field names "
                   "(algorithms/base.py:180-298); nothing leaves the GPU"}
    env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed steps of the headline workload (its device-resident and end-to-end arms); the other "
                         "configurations and the observation arms report their own step counts")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="ieee123", choices=sorted(WORKLOADS))
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--envs", type=int, default=0, help="instances per GPU (default: the workload's)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--kernel-only", action="store_true", help="tuning aid: time the device-resident arm only")
    ap.add_argument("--no-configs", action="store_true", help="skip the sub-results of the other BASELINE configurations")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the workload's per-GPU size on every GPU; strong: --total-envs (1,048,576) split over the GPUs")
    ap.add_argument("--total-envs", type=int, default=0, help="instances in total for --scaling strong")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the headline workload's last timed step to DIR/<name>.npy (rank 0's "
                         "instances; a fixed sample of them when they exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
