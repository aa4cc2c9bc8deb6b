"""Feeder repair (D4) and compilation to the structure-of-arrays the kernels read.

Two host-side steps sit upstream of *both* the CPU oracle and the CUDA path, so
that they solve the same network with the same bus / line numbering:

``repair_topology(feeder)``
    Turns a shipped feeder into a connected radial tree (deviation D4 in
    DESIGN.md).  The reference's own Ybus treats ``abs(z) <= 1e-12`` as an open
    line (reference ``grid_fed_rl/environments/power_flow.py:62-63``), which
    islands three IEEE-13 buses, and its IEEE-34 / IEEE-123 generators produce
    several components plus cycles (SURVEY F5).  Buses, loads and generators
    are passed through untouched; only ``lines`` changes, kept lines preserve
    their reference order and repair lines are appended at the end.

``compile_feeder(feeder, ...)``
    Bus order = ``feeder.buses`` order, line order = ``feeder.lines`` order
    (these indices are what "topology ordering" means in the parity tests),
    plus a breadth-first (level) permutation with ``parent[]`` used by the
    leaf->root / root->leaf traversals on the device.
"""

from __future__ import annotations

from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np

# zero-length IEEE-13 entries keep their configured impedance, un-scaled, as pu
# (reference ieee_feeders.py:64,67,79-80): XFM1 and SWITCH.
IEEE13_ZERO_LENGTH_PU: Dict[str, Tuple[float, float]] = {
    "line_633_634": (0.0, 0.06),
    "line_671_692": (1e-4, 1e-4),
}

OPEN_Z = 1e-12  # reference power_flow.py:63


class TopologyError(ValueError):
    """The feeder cannot be compiled for the radial solvers."""


class RepairedFeeder:
    """Same buses / loads / generators objects as the source feeder, new ``lines``."""

    def __init__(self, source, lines: List[Any], dropped: List[Any], added: List[Any]) -> None:
        self.name = getattr(source, "name", type(source).__name__)
        self.parameters = source.parameters
        self.buses = source.buses
        self.loads = source.loads
        self.generators = source.generators
        self.lines = lines
        self.dropped_lines = dropped
        self.added_lines = added
        self.source = source


def _slack_index(buses: Sequence[Any]) -> int:
    idx = [i for i, b in enumerate(buses) if b.bus_type == "slack"]
    if len(idx) != 1:
        raise TopologyError(f"exactly one slack bus is required, found {len(idx)}")
    return idx[0]


def _new_line(proto, **kw):
    """Build a line of the same class as the feeder's own lines (so a reference
    feeder keeps reference ``Line`` objects with their ``update_state``)."""
    return type(proto)(**kw)


def repair_topology(feeder, zero_length_pu: Optional[Dict[str, Tuple[float, float]]] = None,
                    keep_cycles: bool = False):
    """Deviation D4 (ii)+(iii): see module docstring.  Returns a ``RepairedFeeder``.
    ``keep_cycles=True`` keeps the lines that close a cycle (only open lines are dropped, islands
    are still chained to their list predecessor): a meshed network for the dense solver
    (``B200PowerFlowSolver(method="dense")``); the tree-ordered kernels need the default."""
    overrides = IEEE13_ZERO_LENGTH_PU if zero_length_pu is None else zero_length_pu
    buses = list(feeder.buses)
    n = len(buses)
    index = {b.id: i for i, b in enumerate(buses)}
    slack = _slack_index(buses)

    # (ii) zero-impedance entries: configured pu value if known
    lines: List[Any] = []
    for ln in feeder.lines:
        z = complex(ln.resistance, ln.reactance)
        if abs(z) <= OPEN_Z and ln.id in overrides:
            r, x = overrides[ln.id]
            ln = _new_line(ln, id=ln.id, from_bus=ln.from_bus, to_bus=ln.to_bus,
                           resistance=r, reactance=x, rating=ln.rating)
        lines.append(ln)

    live = [ln for ln in lines if abs(complex(ln.resistance, ln.reactance)) > OPEN_Z]
    if not live:
        raise TopologyError("feeder has no line with a non-zero impedance")
    med_r = float(np.median([ln.resistance for ln in live]))
    med_x = float(np.median([ln.reactance for ln in live]))
    ratings = [ln.rating for ln in live]
    modal_rating = max(sorted(set(ratings)), key=ratings.count)

    # (iii) radialise: union-find in list order, cycle-closing (and open) lines are dropped
    root = list(range(n))

    def find(a: int) -> int:
        while root[a] != a:
            root[a] = root[root[a]]
            a = root[a]
        return a

    kept: List[Any] = []
    dropped: List[Any] = []
    for ln in lines:
        if ln.from_bus not in index or ln.to_bus not in index:
            raise TopologyError(f"line {ln.id} references an unknown bus")
        if abs(complex(ln.resistance, ln.reactance)) <= OPEN_Z:
            dropped.append(ln)
            continue
        a, b = find(index[ln.from_bus]), find(index[ln.to_bus])
        if a == b:
            (kept if keep_cycles else dropped).append(ln)
        else:
            root[a] = b
            kept.append(ln)

    added: List[Any] = []
    for i in range(n):
        if find(i) == find(slack):
            continue
        j = i - 1 if i > 0 else slack
        ln = _new_line(lines[0], id=f"repair_{buses[j].id}_{buses[i].id}", from_bus=buses[j].id,
                       to_bus=buses[i].id, resistance=med_r, reactance=med_x, rating=modal_rating)
        root[find(i)] = find(j)
        kept.append(ln)
        added.append(ln)
    # one pass can leave a component attached to a predecessor that was itself
    # not yet on the slack's side only if i-1 was unreachable; chaining in list
    # order makes that impossible for i>slack, but check anyway
    if any(find(i) != find(slack) for i in range(n)):
        raise TopologyError("repair failed to connect every bus to the slack bus")
    if len(kept) != n - 1 and not keep_cycles:
        raise TopologyError("repair did not produce a spanning tree")
    return RepairedFeeder(feeder, kept, dropped, added)


# --------------------------------------------------------------------------- SoA

GEN_SOLAR, GEN_WIND = 0, 1
BUS_SLACK, BUS_PV, BUS_PQ = 0, 1, 2

# reference dynamics.py:43-48 - the default 24-point residential load profile
DEFAULT_LOAD_PROFILE = (0.5, 0.4, 0.4, 0.4, 0.4, 0.5, 0.7, 0.9, 0.8, 0.7, 0.6, 0.6,
                        0.7, 0.7, 0.6, 0.6, 0.7, 0.9, 1.0, 0.9, 0.8, 0.7, 0.6, 0.5)


@dataclass
class FeederSoA:
    """Compiled feeder.  "ref order" = position in ``feeder.buses`` / ``feeder.lines``;
    "level order" = breadth-first position k (k=0 is the slack bus)."""
    name: str
    n_bus: int
    n_line: int
    s_base: float                      # VA
    bus_ids: list                      # ref order
    line_ids: list                     # ref order
    # level order ---------------------------------------------------------
    order: np.ndarray                  # int32[n]  level k -> ref bus index (k = 0 is the ROOT of the elimination tree)
    rank: np.ndarray                   # int32[n]  ref bus index -> level k
    parent: np.ndarray                 # int32[n]  parent level index, -1 for k=0
    level_ptr: np.ndarray              # int32[n_levels+1]  level l = [ptr[l], ptr[l+1])
    child_ptr: np.ndarray              # int32[n+1] children of k = child_idx[child_ptr[k] : child_ptr[k+1]]
    child_idx: np.ndarray              # int32[n-1] level indices of the children, parent by parent
    n_pool: int                        # Newton: shared-memory hand-off slots to provide at least (0: as few as the library's plan needs)
    lane_of: Optional[np.ndarray]      # int32[n]  lane (< width) that eliminates bus k; None: position inside the level
    bus_type: np.ndarray               # int32[n]  BUS_*
    vm_set: np.ndarray                 # f64[n]   slack / pv magnitude (bus.voltage_magnitude)
    g: np.ndarray                      # f64[n]   series conductance of the branch parent[k]-k (k>=1)
    b: np.ndarray                      # f64[n]   series susceptance of that branch
    gdiag: np.ndarray                  # f64[n]   Re Y_kk summed in line order (reference Ybus)
    bdiag: np.ndarray                  # f64[n]   Im Y_kk
    r: np.ndarray                      # f64[n]   branch resistance (pu)  - sweep
    x: np.ndarray                      # f64[n]   branch reactance (pu)   - sweep
    line_of: np.ndarray                # int32[n] ref line index of that branch (-1 for k=0)
    from_is_parent: np.ndarray         # int32[n] 1 if line.from_bus is the parent end
    rating: np.ndarray                 # f64[n]   VA
    # components (ref order of feeder.loads / generators) ------------------
    load_bus: np.ndarray               # int32[L] level index
    load_base: np.ndarray              # f64[L]   W
    load_p: np.ndarray                 # f64[L]   static active_power (obs, frequency model)
    load_q: np.ndarray                 # f64[L]   static reactive_power (obs)
    gen_ids: list
    gen_type: np.ndarray               # int32[G] GEN_*
    gen_bus: np.ndarray                # int32[G] level index
    gen_cap: np.ndarray                # f64[G]   W
    gen_p0: np.ndarray                 # f64[G]   solar: panel_area        wind: cut_in_speed
    gen_p1: np.ndarray                 # f64[G]   solar: efficiency        wind: rated_speed
    gen_p2: np.ndarray                 # f64[G]   solar: unused            wind: cut_out_speed
    bat_ids: list
    bat_bus: np.ndarray                # int32[Bt] level index
    bat_cap: np.ndarray                # f64[Bt]
    bat_rating: np.ndarray             # f64[Bt]
    bat_eff: np.ndarray                # f64[Bt]
    bat_soc0: np.ndarray               # f64[Bt]
    load_profile: np.ndarray = field(default_factory=lambda: np.array(DEFAULT_LOAD_PROFILE))
    # loop-closing lines of a weakly meshed feeder (sweep solver only; empty for a radial feeder) ------------
    tie_line: np.ndarray = field(default_factory=lambda: np.zeros(0, dtype=np.int32))    # int32[t] ref line index
    tie_from: np.ndarray = field(default_factory=lambda: np.zeros(0, dtype=np.int32))    # int32[t] level index of line.from_bus
    tie_to: np.ndarray = field(default_factory=lambda: np.zeros(0, dtype=np.int32))      # int32[t] level index of line.to_bus
    tie_r: np.ndarray = field(default_factory=lambda: np.zeros(0))                       # f64[t] pu
    tie_x: np.ndarray = field(default_factory=lambda: np.zeros(0))                       # f64[t] pu
    tie_rating: np.ndarray = field(default_factory=lambda: np.zeros(0))                  # f64[t] VA
    tie_zinv: np.ndarray = field(default_factory=lambda: np.zeros(0))                    # f64[t, t, 2] inverse loop-impedance matrix (re, im)

    @property
    def n_tie(self) -> int:
        return int(self.tie_line.size)

    @property
    def n_load(self) -> int:
        return int(self.load_bus.size)

    @property
    def n_gen(self) -> int:
        return int(self.gen_bus.size)

    @property
    def n_bat(self) -> int:
        return int(self.bat_bus.size)

    @property
    def n_levels(self) -> int:
        return int(self.level_ptr.size - 1)

    @property
    def obs_dim(self) -> int:
        # reference grid_env.py:307-314
        return (2 * self.n_bus + 2 * self.n_line + 1 + 2 * self.n_load + self.n_gen
                + 2 * self.n_bat)

    @property
    def act_dim(self) -> int:
        # reference grid_env.py:351
        return self.n_bat + self.n_gen


def _series_admittance(r: float, x: float) -> complex:
    # same expression, same Python complex division as reference power_flow.py:62-63
    z = complex(r, x)
    return 1.0 / z if abs(z) > OPEN_Z else 0.0


def _rooted_tree(n: int, root: int, adj):
    """Breadth-first walk of the tree from ``root``.  Returns (bfs, parent_ref, depth, pending):
    ``bfs`` lists ref bus indices root first, ``parent_ref[v]`` = (parent, line index) ((-1, -1) for the
    root), ``pending[v]`` = number of children of v (what must be eliminated before v)."""
    parent_ref = {root: (-1, -1)}
    depth = {root: 0}
    bfs = [root]
    for u in bfs:
        for v, k in adj[u]:
            if v not in parent_ref:
                parent_ref[v] = (u, k)
                depth[v] = depth[u] + 1
                bfs.append(v)
    if len(bfs) != n:
        raise TopologyError("feeder is not connected (run repair_topology first)")
    pending = [0] * n
    for v in bfs[1:]:
        pending[parent_ref[v][0]] += 1
    return bfs, parent_ref, depth, pending


def _schedule(n: int, root: int, adj, width: Optional[int]):
    """Order the buses for leaf -> root elimination on ``width`` lanes.

    Returns (order, parent_ref, level_of): ``order`` lists ref bus indices level by level,
    level 0 = {root}; every bus sits in a later level than its parent, and each level holds at
    most ``width`` buses when a width is given.  Levels are the time steps (reversed) of Hu's
    highest-level-first list schedule, which is optimal for unit tasks on an in-tree: with
    unbounded width it is the plain height-from-the-leaves layering.
    """
    bfs, parent_ref, depth, pending = _rooted_tree(n, root, adj)
    ready = [v for v in bfs if pending[v] == 0]
    steps = []
    while ready:
        ready.sort(key=lambda v: (-depth[v], v))
        take = ready if width is None else ready[:width]
        rest = [] if width is None else ready[width:]
        steps.append(take)
        for v in take:
            u = parent_ref[v][0]
            if u >= 0:
                pending[u] -= 1
                if pending[u] == 0:
                    rest.append(u)
        ready = rest
    steps.reverse()                      # level 0 = last eliminated = root
    assert steps[0] == [root]
    # As-late-as-possible pass: a bus that is not on a critical path is moved next to its parent's
    # level when there is room, so that its contribution to the parent stays parked only briefly
    # (fewer pool slots alive at once).  Parents are settled before their children.
    level = {}
    for l, members in enumerate(steps):
        for v in members:
            level[v] = l
    room = [None if width is None else width - len(members) for members in steps]
    for v in bfs[1:]:                    # breadth-first from the root: parents first
        target = level[parent_ref[v][0]] + 1
        cur = level[v]
        while target < cur:
            if room[target] is None or room[target] > 0:
                if room[target] is not None:
                    room[target] -= 1
                    room[cur] += 1
                level[v] = target
                break
            target += 1
    steps = [[] for _ in steps]
    for v in bfs:
        steps[level[v]].append(v)
    assert all(steps) and steps[0] == [root]
    # Inside a level the buses follow their parents' positions: consecutive lanes then gather from
    # (nearly) consecutive parent entries - distinct shared-memory banks - and the children of one
    # bus sit next to each other.
    order, level_of, pos = [], {}, {-1: -1}
    for l, members in enumerate(steps):
        for v in sorted(members, key=lambda v: (pos[parent_ref[v][0]], v)):
            level_of[v] = l
            pos[v] = len(order)
            order.append(v)
    return order, parent_ref, level_of


CHAIN_MIN_LANES = 8        # groups of this many lanes and more sum pool hand-offs along sibling chains (gfr_device.cuh)


def _schedule_paths(n: int, root: int, adj, width: int):
    """Order the buses for leaf -> root elimination on ``width`` lanes so that a lane FOLLOWS A PATH:
    list scheduling in elimination time where a lane whose last bus's parent has become ready takes
    that parent next (then Hu's rule, deepest first, for the lanes left).  A bus that is eliminated
    right after one of its children on the same lane gets that child's Schur terms in registers
    instead of through shared memory (and hands its correction back the same way on the way down);
    every non-leaf bus can have one such child at most, and this rule reaches that bound on the
    IEEE feeders (IEEE-123 on 8 lanes: 78 of 122 branches, in the same 17 steps as Hu's schedule).

    Returns (order, parent_ref, level_of, lane_of): ``order`` lists ref bus indices level by level,
    level 0 = {root}; a level is one elimination step (reversed), at most ``width`` buses."""
    bfs, parent_ref, depth, pending = _rooted_tree(n, root, adj)
    ready = set(v for v in bfs if pending[v] == 0)
    last = [None] * width                 # the bus each lane eliminated in the previous step
    steps = []                            # per step: {bus: lane}
    while ready:
        cont = {}
        for lane in range(width):
            b = last[lane]
            if b is not None:
                u = parent_ref[b][0]
                if u >= 0 and u in ready and u not in cont:
                    cont[u] = lane
        take = sorted(ready, key=lambda v: (0 if v in cont else 1, -depth[v], v))[:width]
        assign = {v: cont[v] for v in take if v in cont}
        free = [lane for lane in range(width) if lane not in assign.values()]
        for v in take:
            if v not in assign:
                assign[v] = free.pop(0)
        last = [None] * width
        for v, lane in assign.items():
            last[lane] = v
            ready.discard(v)
        for v in assign:
            u = parent_ref[v][0]
            if u >= 0:
                pending[u] -= 1
                if pending[u] == 0:
                    ready.add(u)
        steps.append(assign)
    steps.reverse()                       # level 0 = last eliminated = root
    assert list(steps[0]) == [root]
    # Placement of the leaves that hand over through shared memory: a leaf eliminated long before its parent
    # parks its contribution in a pool slot all that time, so it moves to a free lane of a row nearer the
    # parent's.  From CHAIN_MIN_LANES lanes on, not into a row that already holds more of its siblings than
    # another candidate row does: there siblings in different rows chain their hand-offs (each adds an earlier
    # one's partial sum to its own, see csrc/gfr_image.hpp) and the parent reads one sum per chain; siblings in
    # one row cannot chain.  Fewer lanes take the row nearest the parent's.
    row_of = {v: l for l, assign in enumerate(steps) for v in assign}
    has_kids = set(parent_ref[v][0] for v in bfs[1:])
    kids_of = {}
    for v in bfs[1:]:
        kids_of.setdefault(parent_ref[v][0], []).append(v)

    def is_heir(v):
        u = parent_ref[v][0]
        return row_of[v] == row_of[u] + 1 and steps[row_of[v]][v] == steps[row_of[u]].get(u)

    for v in sorted((v for v in bfs[1:] if v not in has_kids), key=lambda v: -(row_of[v] - row_of[parent_ref[v][0]])):
        u = parent_ref[v][0]
        cur = row_of[v]
        if is_heir(v):
            continue                      # the heir of its parent: nothing parked
        rows = [r for r in range(row_of[u] + 1, cur + 1) if r == cur or len(steps[r]) < width]
        if width >= CHAIN_MIN_LANES:
            sibs = [row_of[w] for w in kids_of[u] if w != v and not is_heir(w)]
            r = min(rows, key=lambda r: (sibs.count(r), r))
        else:
            r = rows[0]
        if r != cur:
            lane = min(set(range(width)) - set(steps[r].values()))
            del steps[cur][v]
            steps[r][v] = lane
            row_of[v] = r
    order, level_of, lane_of = [], {}, {}
    for l, assign in enumerate(steps):
        for v in sorted(assign, key=lambda v: assign[v]):
            level_of[v] = l
            lane_of[v] = assign[v]
            order.append(v)
    return order, parent_ref, level_of, lane_of


def tree_center(n: int, adj, fallback: int) -> int:
    """A bus of minimum eccentricity (the middle of a longest path): rooting the elimination
    there halves the number of sequential levels of a feeder whose slack bus sits at one end."""
    def far(s):
        dist = {s: 0}
        q = [s]
        for u in q:
            for v, _ in adj[u]:
                if v not in dist:
                    dist[v] = dist[u] + 1
                    q.append(v)
        t = max(dist, key=lambda v: (dist[v], -v))
        return t, dist
    if n == 1:
        return fallback
    a, _ = far(fallback)
    b, da = far(a)
    # walk back from b towards a
    path = [b]
    while path[-1] != a:
        u = path[-1]
        path.append(next(v for v, _ in adj[u] if da[v] == da[u] - 1))
    return path[len(path) // 2]


def compile_feeder(feeder, renewable_sources: Optional[Sequence[str]] = None,
                   with_components: bool = True, root: str = "slack",
                   width: Optional[int] = None, paths: bool = False) -> FeederSoA:
    """Compile a *connected* feeder (run ``repair_topology`` first if it is not): radial, or weakly
    meshed - lines that close a cycle (in list order, as ``repair_topology(keep_cycles=True)`` keeps them)
    become *ties*: the traversal tree is the rest, and the sweep solver restores the loops with the
    compensation method (one current per tie, corrected every iteration through the inverse
    loop-impedance matrix computed here).  The tree-ordered Newton kernels take radial feeders only.

    ``renewable_sources`` has the reference meaning (grid_env.py:167,273,282): a
    generator of type "solar"/"wind" becomes an environment generator only if
    its type is listed.  Generators of type "battery" always become batteries; a
    feeder without one gets the reference's template unit (grid_env.py:292-297)
    at its first load bus (deviation D3).

    ``root`` / ``width`` shape the device-side traversal only (never the bus / line numbering of
    the results): ``root="center"`` roots the elimination tree at the tree's center instead of
    the slack bus (Newton only; the sweep needs the slack at the root), ``width`` caps the buses
    per level at the number of lanes that will cooperate on one instance.  ``paths`` (needs a width)
    lets lanes follow paths of the tree (``_schedule_paths``: register hand-off between a bus and the
    child eliminated just before it on the same lane - what the Newton kernels want).  The hand-offs
    that do go through shared memory get their slots from the native library.
    """
    buses, lines = list(feeder.buses), list(feeder.lines)
    n, m = len(buses), len(lines)
    if n < 1:
        raise TopologyError("feeder has no buses")
    if m < n - 1:
        raise TopologyError(f"a connected feeder needs at least n-1 lines, this one has {n} buses and {m} lines "
                            "(run repair_topology first)")
    index = {b.id: i for i, b in enumerate(buses)}
    if len(index) != n:
        raise TopologyError("duplicate bus ids")
    slack = _slack_index(buses)

    adj: List[List[Tuple[int, int]]] = [[] for _ in range(n)]
    ydiag = np.zeros(n, dtype=complex)
    ys: List[complex] = []
    uf = list(range(n))                   # spanning tree = the lines that do not close a cycle, in list order
    ties: List[int] = []

    def _find(a: int) -> int:
        while uf[a] != a:
            uf[a] = uf[uf[a]]
            a = uf[a]
        return a

    for k, ln in enumerate(lines):
        if ln.from_bus not in index or ln.to_bus not in index:
            raise TopologyError(f"line {ln.id} references an unknown bus")
        i, j = index[ln.from_bus], index[ln.to_bus]
        if i == j:
            raise TopologyError(f"line {ln.id} is a self loop")
        y = _series_admittance(ln.resistance, ln.reactance)
        if y == 0.0:
            raise TopologyError(f"line {ln.id} has zero impedance (open in the reference Ybus)")
        ys.append(y)
        ydiag[i] += y          # accumulation order = line order, as the reference Ybus
        ydiag[j] += y
        a, b = _find(i), _find(j)
        if a == b:
            ties.append(k)     # closes a cycle: a tie, restored by the sweep's compensation step
            continue
        uf[a] = b
        adj[i].append((j, k))
        adj[j].append((i, k))
    if m - len(ties) != n - 1:
        raise TopologyError("feeder is not connected (run repair_topology first)")

    if root not in ("slack", "center"):
        raise TopologyError("root must be 'slack' or 'center'")
    if width is not None and int(width) < 1:
        raise TopologyError("width must be >= 1")
    root_ref = slack if root == "slack" else tree_center(n, adj, slack)
    lane_map = None
    if paths and width is not None:
        order, parent_ref, level_of, lane_map = _schedule_paths(n, root_ref, adj, int(width))
    else:
        order, parent_ref, level_of = _schedule(n, root_ref, adj, None if width is None else int(width))
    rank = np.empty(n, dtype=np.int32)
    rank[np.array(order)] = np.arange(n, dtype=np.int32)

    parent = np.full(n, -1, dtype=np.int32)
    line_of = np.full(n, -1, dtype=np.int32)
    from_is_parent = np.zeros(n, dtype=np.int32)
    g = np.zeros(n); b = np.zeros(n); r = np.zeros(n); x = np.zeros(n); rating = np.zeros(n)
    for k in range(1, n):
        u, li = parent_ref[order[k]]
        parent[k] = rank[u]
        line_of[k] = li
        ln = lines[li]
        from_is_parent[k] = 1 if index[ln.from_bus] == u else 0
        g[k], b[k] = ys[li].real, ys[li].imag
        r[k], x[k] = ln.resistance, ln.reactance
        rating[k] = ln.rating
    levels = np.array([level_of[v] for v in order])
    n_levels = int(levels.max()) + 1
    level_ptr = np.searchsorted(levels, np.arange(n_levels + 1)).astype(np.int32)
    child_cnt = np.bincount(parent[1:], minlength=n) if n > 1 else np.zeros(n, dtype=np.int64)
    child_ptr = np.zeros(n + 1, dtype=np.int32)
    child_ptr[1:] = np.cumsum(child_cnt)
    child_idx = np.zeros(max(n - 1, 0), dtype=np.int32)
    fill = child_ptr[:-1].copy()
    for k in range(1, n):
        child_idx[fill[parent[k]]] = k
        fill[parent[k]] += 1
    for k in range(1, n):
        assert parent[k] < k and levels[parent[k]] < levels[k]
    lane_of = None if lane_map is None else np.array([lane_map[v] for v in order], dtype=np.int32)

    # ---- ties: end points in level order and the inverse of the loop-impedance matrix
    #      Z_loop[i][j] = sum over tree branches e of z_e s_i(e) s_j(e) + [i == j] z_tie_i, where
    #      s_i(e) = [to-end of tie i below e] - [from-end of tie i below e] (non-zero on the tree path between
    #      the two ends): d(V_from - V_to - z_tie J)_i / dJ_j = -Z_loop[i][j] for tie currents J (from -> to)
    tie_soa = {}
    if ties:
        t = len(ties)
        tf = np.array([rank[index[lines[k].from_bus]] for k in ties], dtype=np.int32)
        tt = np.array([rank[index[lines[k].to_bus]] for k in ties], dtype=np.int32)
        S = np.zeros((t, n))
        for i in range(t):
            for end, sign in ((tt[i], 1.0), (tf[i], -1.0)):
                k = int(end)
                while k > 0:
                    S[i, k] += sign
                    k = int(parent[k])
        zb = r + 1j * x                                       # branch above bus k (0 for the root)
        zt = np.array([complex(lines[k].resistance, lines[k].reactance) for k in ties])
        zloop = (S * zb[None, :]) @ S.T + np.diag(zt)
        zinv = np.linalg.inv(zloop)
        tie_soa = dict(tie_line=np.array(ties, dtype=np.int32), tie_from=tf, tie_to=tt,
                       tie_r=zt.real.copy(), tie_x=zt.imag.copy(),
                       tie_rating=np.array([float(lines[k].rating) for k in ties]),
                       tie_zinv=np.stack([zinv.real, zinv.imag], axis=-1).copy())

    tmap = {"slack": BUS_SLACK, "pv": BUS_PV}
    bus_type = np.array([tmap.get(buses[i].bus_type, BUS_PQ) for i in order], dtype=np.int32)
    vm_set = np.array([float(buses[i].voltage_magnitude) for i in order])

    soa = dict(
        name=getattr(feeder, "name", type(feeder).__name__), n_bus=n, n_line=m,
        s_base=float(feeder.parameters.base_power) * 1e6,
        bus_ids=[b_.id for b_ in buses], line_ids=[l_.id for l_ in lines],
        order=np.array(order, dtype=np.int32), rank=rank, parent=parent, level_ptr=level_ptr,
        child_ptr=child_ptr, child_idx=child_idx, n_pool=0, lane_of=lane_of,
        bus_type=bus_type, vm_set=vm_set, g=g, b=b,
        gdiag=ydiag.real[order].copy(), bdiag=ydiag.imag[order].copy(), r=r, x=x,
        line_of=line_of, from_is_parent=from_is_parent, rating=rating, **tie_soa)

    # ---- components -------------------------------------------------------
    loads = list(feeder.loads) if with_components else []
    for ld in loads:
        if ld.bus not in index:
            raise TopologyError(f"load {ld.id} references an unknown bus")
    soa.update(
        load_bus=np.array([rank[index[ld.bus]] for ld in loads], dtype=np.int32),
        load_base=np.array([float(ld.base_power) for ld in loads]),
        load_p=np.array([float(ld.active_power) for ld in loads]),
        load_q=np.array([float(ld.reactive_power) for ld in loads]))

    sources = list(renewable_sources or [])
    gen_ids, gtype, gbus, gcap, p0, p1, p2 = [], [], [], [], [], [], []
    bat_ids, bbus, bcap, brat, beff = [], [], [], [], []
    gens = feeder.generators if with_components else {}
    for gid, info in gens.items():
        kind = info.get("type")
        if kind == "battery":
            bat_ids.append(gid)
            bbus.append(rank[index[info["bus"]]])
            bcap.append(float(info["capacity_kwh"]))
            brat.append(float(info["power_rating_kw"]) * 1e3)
            beff.append(float(info["efficiency"]))
        elif kind == "solar" and "solar" in sources:
            eff = float(info.get("efficiency", 0.18))
            gen_ids.append(gid); gtype.append(GEN_SOLAR); gbus.append(rank[index[info["bus"]]])
            gcap.append(float(info["capacity"]))
            p0.append(float(info["capacity"]) / (eff * 1000)); p1.append(eff); p2.append(0.0)
        elif kind == "wind" and "wind" in sources:
            gen_ids.append(gid); gtype.append(GEN_WIND); gbus.append(rank[index[info["bus"]]])
            gcap.append(float(info["capacity"]))
            p0.append(float(info.get("cut_in_speed", 3.0)))
            p1.append(float(info.get("rated_speed", 12.0)))
            p2.append(float(info.get("cut_out_speed", 25.0)))
    if with_components and not bat_ids:
        home = loads[0].bus if loads else buses[slack].id
        bat_ids.append(f"battery_{home}")
        bbus.append(rank[index[home]])
        bcap.append(1e3); brat.append(0.5e6); beff.append(0.95)
    soa.update(
        gen_ids=gen_ids, gen_type=np.array(gtype, dtype=np.int32),
        gen_bus=np.array(gbus, dtype=np.int32), gen_cap=np.array(gcap, dtype=float),
        gen_p0=np.array(p0, dtype=float), gen_p1=np.array(p1, dtype=float),
        gen_p2=np.array(p2, dtype=float),
        bat_ids=bat_ids, bat_bus=np.array(bbus, dtype=np.int32),
        bat_cap=np.array(bcap, dtype=float), bat_rating=np.array(brat, dtype=float),
        bat_eff=np.array(beff, dtype=float), bat_soc0=np.full(len(bat_ids), 0.5))
    return FeederSoA(**soa)


def auto_lanes(n_bus: int, solver: str = "newton", depth: Optional[int] = None) -> int:
    """Threads cooperating on one instance when the caller does not say.  The rule itself lives in the
    native library (``gfr_auto_lanes`` in csrc/gfr_b200.cu, with the measurements it comes from) so that a
    C-ABI caller passing ``lanes = 0`` and this module can never disagree; ``depth`` = levels of the
    center-rooted tree (decides between two and four Newton lanes on small feeders)."""
    from . import _native as nat
    code = nat.SOLVERS.get(solver, nat.SOLVER_NEWTON)
    return int(nat.load_library().gfr_auto_lanes(int(n_bus), code, int(depth or 0)))


def compile_for_solver(feeder, solver: str = "newton", lanes: int = 0,
                       renewable_sources: Optional[Sequence[str]] = None,
                       with_components: bool = True):
    """``compile_feeder`` with the traversal the kernels want: both solvers walk the tree rooted
    at its center when that shortens it (the sweep handles the slack bus wherever it sits, Newton
    always gains); levels are capped at the lane count (Hu's schedule).  Returns (FeederSoA, lanes)."""
    if not int(lanes):
        depth = None
        if len(feeder.buses) <= 45 and solver != "sweep":      # the shape decides between two and four lanes
            depth = compile_feeder(feeder, root="center", renewable_sources=renewable_sources,
                                   with_components=False).n_levels
        lanes = auto_lanes(len(feeder.buses), solver, depth)
    lanes = int(lanes)
    newton = solver != "sweep"
    kw = dict(renewable_sources=renewable_sources, with_components=with_components,
              width=lanes if (lanes > 1 or newton) else None, paths=newton)
    soa = compile_feeder(feeder, root="center", **kw)
    if solver == "sweep":
        # the sweep pays one extra bus-parallel pass per iteration when the slack is not the root:
        # only worth it if the center-rooted tree is clearly shallower
        alt = compile_feeder(feeder, root="slack", **kw)
        if soa.n_levels > 0.75 * alt.n_levels:
            soa = alt
    if soa.n_tie and solver != "sweep":
        raise TopologyError(f"the feeder has {soa.n_tie} loop-closing lines: the tree-ordered Newton-Raphson takes radial "
                            "feeders (solver='sweep' restores the loops by compensation; repair_topology() drops them)")
    soa.lanes_hint = lanes             # the lane count the level schedule was capped for
    return soa, lanes
