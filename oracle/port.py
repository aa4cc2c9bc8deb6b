"""CPU oracle for the batched GridEnvironment.step path - TEST INFRASTRUCTURE ONLY.

This file is a numpy restatement of the reference's algorithm for the hot path.
It is the *checker*: only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it.  The
product (``grid_fed_rl_b200``) never does, and has no CPU fallback.

Parity status: **pinned against the reference itself** - ``oracle/ref_harness.py``
imports the unmodified reference from ``/root/reference``, runs it with the four
documented deviations D1-D4 (DESIGN.md) and freezes its outputs under
``tests/golden/``; ``tests/test_oracle_golden.py`` replays those traces through
this file.  The reference's own tests hold no numerical golden vectors for this
path (SURVEY section 4), so the frozen reference outputs are the pin.

What is restated (reference file:line, relative to /root/reference/grid_fed_rl):
  * Ybus                         environments/power_flow.py:48-73
  * Newton-Raphson loop          environments/power_flow.py:89-211
  * polar Jacobian               environments/power_flow.py:213-295  (+ D2: J11 diagonal sign)
  * polar update                 environments/power_flow.py:297-327
  * line flows / losses          environments/power_flow.py:329-358, :199-200
  * env step orchestration       environments/grid_env.py:410-619
  * actions / batteries          environments/grid_env.py:621-651, environments/dynamics.py:189-220,304-324
  * weather                      environments/grid_env.py:653-681
  * loads / solar / wind         environments/dynamics.py:54-75,120-142,158-170
  * injections                   environments/grid_env.py:683-720 (+ D3: battery at its own bus)
  * state update / frequency     environments/grid_env.py:722-751, environments/dynamics.py:260-273
  * observation / reward         environments/grid_env.py:753-826
  * constraints / done           environments/base.py:140-167, environments/grid_env.py:563-608
  * reset                        environments/grid_env.py:360-408

Everything is vectorised over a leading env axis B; the linear solve is the
same LAPACK ``dgesv`` (``np.linalg.solve``) the reference calls at
power_flow.py:187, on the same dense (2(n-1))^2 Jacobian.
"""

from __future__ import annotations

from typing import Any, Dict, Optional, Sequence

import numpy as np

OPEN_Z = 1e-12
DEFAULT_PROFILE = np.array([0.5, 0.4, 0.4, 0.4, 0.4, 0.5, 0.7, 0.9, 0.8, 0.7, 0.6, 0.6,
                            0.7, 0.7, 0.6, 0.6, 0.7, 0.9, 1.0, 0.9, 0.8, 0.7, 0.6, 0.5])


# --------------------------------------------------------------------------- solver

class DenseNetwork:
    """Dense Ybus and index sets of one feeder, in ``feeder.buses`` / ``feeder.lines`` order."""

    def __init__(self, buses: Sequence[Any], lines: Sequence[Any]) -> None:
        n = len(buses)
        self.n, self.m = n, len(lines)
        self.index = {b.id: i for i, b in enumerate(buses)}
        Y = np.zeros((n, n), dtype=complex)
        self.y = np.zeros(self.m, dtype=complex)
        self.fr = np.zeros(self.m, dtype=np.int64)
        self.to = np.zeros(self.m, dtype=np.int64)
        self.rating = np.array([float(ln.rating) for ln in lines])
        for k, ln in enumerate(lines):
            i, j = self.index[ln.from_bus], self.index[ln.to_bus]
            z = complex(ln.resistance, ln.reactance)
            y = 1.0 / z if abs(z) > OPEN_Z else 0.0
            Y[i, j] -= y
            Y[j, i] -= y
            Y[i, i] += y
            Y[j, j] += y
            self.y[k], self.fr[k], self.to[k] = y, i, j
        self.Y = Y
        slack = [i for i, b in enumerate(buses) if b.bus_type == "slack"]
        self.slack = slack[-1] if slack else 0     # the reference's loop keeps the last one
        self.pv = np.array([i for i, b in enumerate(buses) if b.bus_type == "pv"], dtype=np.int64)
        self.pq = np.array([i for i, b in enumerate(buses)
                            if b.bus_type not in ("slack", "pv")], dtype=np.int64)
        self.non_slack = np.array([i for i in range(n) if i != self.slack], dtype=np.int64)
        self.vm_set = np.array([float(b.voltage_magnitude) for b in buses])


def newton_raphson(net: DenseNetwork, p_spec: np.ndarray, tolerance: float = 1e-6,
                   max_iterations: int = 50, acceleration: float = 1.0,
                   j11_fix: bool = True) -> Dict[str, np.ndarray]:
    """Batched polar NR.  ``p_spec`` [B,n] (pu, generation minus load), ``Q_spec`` = 0."""
    p_spec = np.atleast_2d(np.asarray(p_spec, dtype=float))
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
        dQ = np.where(is_pq, 0.0 - S.imag, 0.0)
        mm = np.maximum(np.max(np.abs(dP), axis=1), np.max(np.abs(dQ), axis=1))
        max_mismatch[idx] = mm
        done = mm < tolerance                      # NaN compares False, as in the reference
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
        A = G * sn - Bm * cs                       # [b,i,j]
        C = G * cs + Bm * sn
        VV = Vm[:, :, None] * Vm[:, None, :]
        # J11 dP/dVa  (power_flow.py:243-251) + D2
        J11 = VV * A
        d11 = -np.sum(VV * A, axis=2) + Vm * Vm * bd
        if j11_fix:
            d11 = d11 - 2.0 * Vm * Vm * bd
        # J12 dP/dVm  (power_flow.py:254-263)
        J12 = Vm[:, :, None] * C
        d12 = np.sum(Vm[:, None, :] * C, axis=2) + Vm * gd
        # J21 dQ/dVa  (power_flow.py:266-274)
        J21 = -VV * C
        d21 = np.sum(VV * C, axis=2) - Vm * Vm * gd
        # J22 dQ/dVm  (power_flow.py:277-287)
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
                    singular[q] = True            # reference: warn + break, converged stays False
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


# --------------------------------------------------------------------------- Philox (throughput-mode noise)

PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85


def philox4x32_10(counter: np.ndarray, key: np.ndarray) -> np.ndarray:
    """Philox4x32-10 (Salmon et al., SC'11).  counter [...,4] uint32, key [...,2] uint32."""
    c = [counter[..., i].astype(np.uint64) for i in range(4)]
    k0 = key[..., 0].astype(np.uint64)
    k1 = key[..., 1].astype(np.uint64)
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(PHILOX_M0) * c[0]
        p1 = np.uint64(PHILOX_M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(PHILOX_W0)) & mask
        k1 = (k1 + np.uint64(PHILOX_W1)) & mask
    return np.stack(c, axis=-1).astype(np.uint32)


def _u53(hi: np.ndarray, lo: np.ndarray) -> np.ndarray:
    """Two 32-bit words -> uniform in (0,1) on a 2^-53 grid, never 0 or 1."""
    k = (hi.astype(np.uint64) >> np.uint64(5)) * np.uint64(1 << 26) + (lo.astype(np.uint64) >> np.uint64(6))
    return (k.astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


def philox_noise(seed: np.ndarray, draw: np.ndarray, n_slots: int) -> np.ndarray:
    """The noise row the kernel generates in throughput mode.

    seed [B] uint64 (Philox key), draw [B] uint64 (per-env draw counter: one
    tick per reset / step), returns [B, n_slots]: slot 0 is a uniform, slots
    1.. are standard normals (Box-Muller, two per Philox block).
    Block q of a row uses counter (draw_lo, draw_hi, q, 0).
    """
    seed = np.asarray(seed, dtype=np.uint64)
    draw = np.asarray(draw, dtype=np.uint64)
    Bn = seed.shape[0]
    key = np.stack([seed & np.uint64(0xFFFFFFFF), seed >> np.uint64(32)], axis=-1).astype(np.uint32)
    n_norm = n_slots - 1
    n_blk = 1 + (n_norm + 1) // 2
    out = np.empty((Bn, n_slots))
    ctr = np.zeros((Bn, n_blk, 4), dtype=np.uint32)
    ctr[:, :, 0] = (draw & np.uint64(0xFFFFFFFF)).astype(np.uint32)[:, None]
    ctr[:, :, 1] = (draw >> np.uint64(32)).astype(np.uint32)[:, None]
    ctr[:, :, 2] = np.arange(n_blk, dtype=np.uint32)[None, :]
    w = philox4x32_10(ctr, key[:, None, :].repeat(n_blk, axis=1))
    u1 = _u53(w[..., 0], w[..., 1])
    u2 = _u53(w[..., 2], w[..., 3])
    out[:, 0] = u1[:, 0]
    rad = np.sqrt(-2.0 * np.log(u1[:, 1:]))
    ang = 2.0 * np.pi * u2[:, 1:]
    z = np.stack([rad * np.cos(ang), rad * np.sin(ang)], axis=-1).reshape(Bn, -1)
    out[:, 1:] = z[:, :n_norm]
    return out


# --------------------------------------------------------------------------- env

def _components(feeder, renewable_sources):
    """D3: which generators / batteries the environment holds, in dict order."""
    index = {b.id: i for i, b in enumerate(feeder.buses)}
    src = list(renewable_sources or [])
    gens, bats = [], []
    for gid, info in feeder.generators.items():
        t = info.get("type")
        if t == "battery":
            bats.append(dict(id=gid, bus=index[info["bus"]], cap=float(info["capacity_kwh"]),
                             rating=float(info["power_rating_kw"]) * 1e3,
                             eff=float(info["efficiency"])))
        elif t == "solar" and "solar" in src:
            eff = float(info.get("efficiency", 0.18))
            gens.append(dict(id=gid, type="solar", bus=index[info["bus"]],
                             cap=float(info["capacity"]), eff=eff,
                             area=float(info["capacity"]) / (eff * 1000)))
        elif t == "wind" and "wind" in src:
            gens.append(dict(id=gid, type="wind", bus=index[info["bus"]],
                             cap=float(info["capacity"]), ci=float(info.get("cut_in_speed", 3.0)),
                             vr=float(info.get("rated_speed", 12.0)),
                             co=float(info.get("cut_out_speed", 25.0))))
    if not bats:
        home = feeder.loads[0].bus if feeder.loads else feeder.buses[0].id
        bats.append(dict(id=f"battery_{home}", bus=index[home], cap=1e3, rating=0.5e6, eff=0.95))
    return gens, bats


class PortEnv:
    """Batched restatement of the reference ``GridEnvironment`` (with D1-D3) on a radial,
    repaired feeder (D4 is applied by the caller, upstream of oracle and kernel alike)."""

    def __init__(self, feeder, num_envs: int, timestep: float = 1.0, episode_length: int = 86400,
                 stochastic_loads: bool = True, renewable_sources: Optional[Sequence[str]] = None,
                 weather_variation: bool = True, voltage_limits=(0.95, 1.05),
                 frequency_limits=(59.5, 60.5), safety_penalty: float = 100.0,
                 tolerance: float = 1e-6, max_iterations: int = 50, acceleration: float = 1.0) -> None:
        """``acceleration``: the factor of the Newton update (the reference's ``acceleration_factor``)."""
        self.B = int(num_envs)
        self.net = DenseNetwork(feeder.buses, feeder.lines)
        self.s_base = float(feeder.parameters.base_power) * 1e6
        self.dt, self.episode_length = float(timestep), int(episode_length)
        self.stochastic_loads, self.weather_variation = stochastic_loads, weather_variation
        self.v_lo, self.v_hi = voltage_limits
        self.f_lo, self.f_hi = frequency_limits
        self.penalty = float(safety_penalty)
        self.tol, self.max_it, self.accel = tolerance, max_iterations, float(acceleration)
        idx = self.net.index
        self.load_bus = np.array([idx[l.bus] for l in feeder.loads], dtype=np.int64)
        self.load_base = np.array([float(l.base_power) for l in feeder.loads])
        self.load_p = np.array([float(l.active_power) for l in feeder.loads])
        self.load_q = np.array([float(l.reactive_power) for l in feeder.loads])
        self.gens, self.bats = _components(feeder, renewable_sources)
        self.n, self.m = self.net.n, self.net.m
        self.L, self.G, self.Bt = len(feeder.loads), len(self.gens), len(self.bats)
        self.A = self.Bt + self.G
        self.D = 2 * self.n + 2 * self.m + 1 + 2 * self.L + self.G + 2 * self.Bt
        self.n_noise = 4 + self.L
        self.profile = DEFAULT_PROFILE
        B = self.B
        # construction-time state (grid_env.py:212-218, dynamics.py:240)
        self.time = np.zeros(B); self.step_count = np.zeros(B, dtype=np.int32)
        self.irr = np.zeros(B); self.wind = np.full(B, 5.0)
        self.temp = np.full(B, 25.0); self.cloud = np.full(B, 0.3)
        self.freq = np.full(B, 60.0)
        self.soc = np.full((B, self.Bt), 0.5); self.bpow = np.zeros((B, self.Bt))
        self.vm = np.ones((B, self.n)); self.va = np.zeros((B, self.n))
        self.line_p = np.zeros((B, self.m)); self.line_loading = np.zeros((B, self.m))
        self.total_losses = np.zeros(B); self.episode_reward = np.zeros(B)
        self.viol_count = np.zeros(B, dtype=np.int32)
        self.curtail = np.ones((B, self.G))

    # -- pieces ---------------------------------------------------------------
    def _hour(self, t):
        return np.fmod(t / 3600, 24)          # Python float % on non-negative operands

    def _update_weather(self, sel, noise):
        if not self.weather_variation:
            return
        hour = self._hour(self.time[sel])
        day = (hour >= 6) & (hour <= 18)
        base = np.where(day, 1000 * np.sin(np.pi * (hour - 6) / 12), 0.0)
        self.irr[sel] = base * (0.8 + 0.4 * noise[:, 0])
        self.wind[sel] = np.maximum(0, np.minimum(30, self.wind[sel] + (0 + noise[:, 1] * 0.5)))
        self.temp[sel] = (25 + 10 * np.sin(2 * np.pi * (hour - 12) / 24)) + (0 + noise[:, 2] * 2)
        self.cloud[sel] = np.maximum(0, np.minimum(1, self.cloud[sel] + (0 + noise[:, 3] * 0.1)))

    def _renewable(self, sel):
        """Uncurtailed P_g [b,G] at the current time / weather."""
        out = np.zeros((sel.size, self.G))
        hour = self._hour(self.time[sel])
        for k, gdef in enumerate(self.gens):
            if gdef["type"] == "solar":
                day = (hour >= 6) & (hour <= 18)
                sun = np.where(day, np.sin(np.pi * (hour - 6) / 12), 0.0)
                actual = (1000 * sun) * (1 - 0.8 * self.cloud[sel])
                tf = 1 - 0.004 * np.maximum(0, self.temp[sel] - 25)
                out[:, k] = np.minimum(actual * gdef["area"] * gdef["eff"] * tf, gdef["cap"])
            else:
                v = self.wind[sel]
                ratio = ((v - gdef["ci"]) / (gdef["vr"] - gdef["ci"])) ** 3
                p = np.where(v <= gdef["vr"], gdef["cap"] * ratio, gdef["cap"])
                out[:, k] = np.where((v < gdef["ci"]) | (v > gdef["co"]), 0.0, p)
        return out

    def _observation(self, sel):
        b = sel.size
        obs = np.empty((b, self.D))
        o = 0
        obs[:, o:o + 2 * self.n:2] = self.vm[sel]; obs[:, o + 1:o + 2 * self.n:2] = self.va[sel]
        o += 2 * self.n
        obs[:, o:o + 2 * self.m:2] = self.line_p[sel]
        obs[:, o + 1:o + 2 * self.m:2] = self.line_loading[sel]
        o += 2 * self.m
        obs[:, o] = self.freq[sel]; o += 1
        obs[:, o:o + 2 * self.L:2] = self.load_p; obs[:, o + 1:o + 2 * self.L:2] = self.load_q
        o += 2 * self.L
        obs[:, o:o + self.G] = self._renewable(sel); o += self.G
        obs[:, o:o + 2 * self.Bt:2] = self.soc[sel]; obs[:, o + 1:o + 2 * self.Bt:2] = self.bpow[sel]
        return obs

    # -- API --------------------------------------------------------------------
    def reset(self, noise: Optional[np.ndarray] = None, mask: Optional[np.ndarray] = None,
              start_time: float = 0.0) -> np.ndarray:
        """``noise`` [B,>=4]: the 4 weather draws ``reset`` consumes (grid_env.py:402)."""
        sel = np.arange(self.B) if mask is None else np.flatnonzero(mask)
        self.time[sel] = 0.0; self.step_count[sel] = 0
        self.episode_reward[sel] = 0.0; self.viol_count[sel] = 0; self.total_losses[sel] = 0.0
        self.vm[sel] = 1.0; self.va[sel] = 0.0
        self.line_p[sel] = 0.0; self.line_loading[sel] = 0.0
        self.freq[sel] = 60.0; self.soc[sel] = 0.5; self.bpow[sel] = 0.0
        if self.weather_variation:
            self._update_weather(sel, np.asarray(noise, dtype=float)[sel])
        obs = self._observation(sel)
        self.time[sel] = start_time          # harness extension: time of day of the first step
        return obs

    def step(self, actions: np.ndarray, noise: Optional[np.ndarray] = None) -> Dict[str, np.ndarray]:
        B, Bt, G = self.B, self.Bt, self.G
        actions = np.asarray(actions, dtype=float).reshape(B, self.A).copy()
        invalid = ~np.all(np.isfinite(actions), axis=1)
        if self.A == 1:
            # a 1-element rejected action is replaced by [0.0] and the step goes on
            # (robust_validation.py:237-246 -> grid_env.py:428, 624-625)
            actions[invalid] = 0.0
            invalid[:] = False
        out = dict(
            obs=np.empty((B, self.D)), reward=np.zeros(B), terminated=np.zeros(B, dtype=bool),
            truncated=np.zeros(B, dtype=bool), error=invalid.copy(),
            converged=np.zeros(B, dtype=bool), iterations=np.zeros(B, dtype=np.int32),
            max_voltage=np.zeros(B), min_voltage=np.zeros(B), losses=np.zeros(B),
            max_mismatch=np.zeros(B), violations=np.zeros((B, 4), dtype=bool))
        bad = np.flatnonzero(invalid)
        if bad.size:
            # grid_env.py:454-467: nothing advanced, -2*penalty, terminated
            out["obs"][bad] = self._observation(bad)
            out["reward"][bad] = -self.penalty * 2
            out["terminated"][bad] = True
            out["max_voltage"][bad] = self.vm[bad].max(axis=1)
            out["min_voltage"][bad] = self.vm[bad].min(axis=1)
        sel = np.flatnonzero(~invalid)
        if sel.size:
            self._step_valid(sel, actions[sel], None if noise is None else np.asarray(noise)[sel], out)
        out.update(viol_count=self.viol_count.copy(), current_step=self.step_count.copy(),
                   episode_reward=self.episode_reward.copy())
        return out

    def _step_valid(self, sel, act, noise, out):
        dt, Bt, G = self.dt, self.Bt, self.G
        b = sel.size
        # --- actions -> batteries (grid_env.py:629-641, dynamics.py:189-220,304-324)
        for k, bat in enumerate(self.bats):
            cmd = act[:, k] * bat["rating"]
            soc, cur = self.soc[sel, k], self.bpow[sel, k]
            cap, eff, rating = bat["cap"], bat["eff"], bat["rating"]
            # discharge
            e_d = np.minimum(np.minimum(cmd, rating) * dt / 3600, soc * cap * eff)
            p_d = e_d * 3600 / dt
            soc_d = soc - e_d / (cap * eff)
            # charge
            e_c = np.minimum(np.minimum(-cmd, rating) * dt / 3600, ((1.0 - soc) * cap) / eff)
            p_c = e_c * 3600 / dt
            soc_c = soc + e_c * eff / cap
            self.soc[sel, k] = np.where(cmd > 0, soc_d, np.where(cmd < 0, soc_c, soc))
            self.bpow[sel, k] = np.where(cmd > 0, p_d, np.where(cmd < 0, -p_c, cur))
        curtail = (act[:, Bt:] + 1) / 2                                  # grid_env.py:648
        self.curtail[sel] = curtail
        # --- time, weather
        self.time[sel] += dt
        self.step_count[sel] += 1
        if self.weather_variation:
            self._update_weather(sel, noise)
        t = self.time[sel]
        # --- injections (grid_env.py:683-720)
        loads_w = np.zeros((b, self.n)); gen_w = np.zeros((b, self.n))
        if self.stochastic_loads:
            hour = self._hour(t)
            hi = hour.astype(np.int64)
            nxt = (hi + 1) % 24
            frac = hour - hi
            mult = self.profile[hi] * (1 - frac) + self.profile[nxt] * frac
            mult = mult[:, None] * (1 + (0 + 0.1 * noise[:, 4:4 + self.L]))
            p_load = np.maximum(0, self.load_base * mult * 1.0)
        else:
            p_load = np.broadcast_to(self.load_base, (b, self.L))
        for l in range(self.L):
            loads_w[:, self.load_bus[l]] += p_load[:, l]
        p_ren = self._renewable(sel)
        for k, gdef in enumerate(self.gens):
            gen_w[:, gdef["bus"]] += p_ren[:, k] * curtail[:, k]
        for k, bat in enumerate(self.bats):
            cur = self.bpow[sel, k]
            gen_w[:, bat["bus"]] += np.where(cur > 0, cur, 0.0)
            loads_w[:, bat["bus"]] += np.where(cur < 0, np.abs(cur), 0.0)
        # --- D1 + solve (power_flow.py:105-121)
        p_spec = np.zeros((b, self.n))
        p_spec -= loads_w / self.s_base
        p_spec += gen_w / self.s_base
        sol = newton_raphson(self.net, p_spec, self.tol, self.max_it, self.accel)
        flows_w = sol["line_flows"] * self.s_base
        losses_w = sol["losses"] * self.s_base
        # --- state update (grid_env.py:722-739, base.py:261-264)
        self.vm[sel] = sol["bus_voltages"]; self.va[sel] = sol["bus_angles"]
        self.line_p[sel] = flows_w
        self.line_loading[sel] = np.where(self.net.rating > 0, np.abs(flows_w) / self.net.rating, 0.0)
        self.total_losses[sel] += losses_w * dt / 3600
        # --- frequency (grid_env.py:741-751, dynamics.py:260-273)
        total_load = 0.0
        for v in self.load_p:
            total_load = total_load + v
        total_gen = np.zeros(b)
        for k in range(G):
            total_gen = total_gen + p_ren[:, k]
        imb = (total_gen - total_load - losses_w) / 1e6
        f = self.freq[sel]
        df = (imb - 1.0 * (f - 60.0)) / (2 * 5.0 * 60.0)
        f = f + df * dt
        self.freq[sel] = np.maximum(55.0, np.minimum(65.0, f))
        # --- observation, reward (grid_env.py:753-826)
        obs = self._observation(sel)
        reward = np.zeros(b)
        dev = np.zeros(b)
        for i in range(self.n):
            dev = dev + np.abs(self.vm[sel, i] - 1.0)
        reward = reward - dev * 10
        reward = reward - np.abs(self.freq[sel] - 60.0) * 20
        reward = reward - np.sum(self.line_loading[sel] > 0.8, axis=1) * 50
        reward = reward - self.total_losses[sel] * 0.1
        tot_ren = np.zeros(b); tot_cur = np.zeros(b)
        for k in range(G):
            tot_ren = tot_ren + p_ren[:, k]
            tot_cur = tot_cur + p_ren[:, k] * (1 - curtail[:, k])
        reward = reward + (tot_ren - tot_cur) * 1e-5
        for k in range(Bt):
            s = self.soc[sel, k]
            reward = reward + np.where((s >= 0.2) & (s <= 0.8), 1.0, -5.0)
        # --- done / constraints (base.py:140-167, grid_env.py:563-608)
        terminated = self.step_count[sel] >= self.episode_length
        vm = self.vm[sel]
        with np.errstate(invalid="ignore"):
            viol = np.stack([np.any(vm > self.v_hi, axis=1), np.any(vm < self.v_lo, axis=1),
                             self.freq[sel] > self.f_hi, self.freq[sel] < self.f_lo], axis=1)
        anyv = viol.any(axis=1)
        self.viol_count[sel] += anyv
        truncated = anyv & (self.viol_count[sel] > 10)
        reward = np.where(truncated, reward - self.penalty, reward)
        self.episode_reward[sel] += reward
        out["obs"][sel] = obs; out["reward"][sel] = reward
        out["terminated"][sel] = terminated; out["truncated"][sel] = truncated
        out["converged"][sel] = sol["converged"]; out["iterations"][sel] = sol["iterations"]
        out["max_voltage"][sel] = sol["bus_voltages"].max(axis=1)
        out["min_voltage"][sel] = sol["bus_voltages"].min(axis=1)
        out["losses"][sel] = losses_w; out["max_mismatch"][sel] = sol["max_mismatch"]
        out["violations"][sel] = viol
