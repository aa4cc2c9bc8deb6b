"""CPU tier: the Newton plan of the pool hand-offs (sibling chains, slots, back-substitution slots).

The children that are not their parent's heir hand their Schur terms up through shared-memory pool slots.
They are summed along sibling chains: a child may absorb the partial sum of a sibling eliminated in an
earlier row, and the parent gathers the chain tails.  These tests replay the library's plan
(csrc/gfr_image.hpp) row by row, as the kernels run it with a group barrier after every row, for every
feeder of tests/golden and every lane count the kernels are instantiated for."""
import os
import sys
from collections import Counter

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import pool_gather_stats as pgs  # noqa: E402
from oracle.ref_harness import FEEDER_SPECS, raw_feeder  # noqa: E402

FL_C_REG, FL_P_REG, FL_VALID = pgs.FL_C_REG, pgs.FL_P_REG, pgs.FL_VALID

_FEEDERS = {}


def _soa(spec, lanes):
    import grid_fed_rl_b200 as m
    from grid_fed_rl_b200.topology import compile_for_solver
    if spec not in _FEEDERS:
        _FEEDERS[spec] = m.repair_topology(raw_feeder(None, spec, use_reference_classes=False))
    soa, used = compile_for_solver(_FEEDERS[spec], "newton", lanes, with_components=False)
    assert used == lanes
    return soa


def replay_up(pl):
    """Leaf -> root: every read of a row sees the slots as the rows before it left them; writes come after
    every read of the row (the barrier that ends a row orders them for the next).  Returns, per bus, the
    multiset of children whose hand-off reached it."""
    lanes, nrows = pl["lanes"], pl["nrows"]
    bus, parent, flags = pl["bus"], pl["parent"], pl["flags"]
    content = {}                       # slot -> (row written, writer bus, Counter of buses summed in it)
    sent = {}                          # bus -> Counter: its own hand-off (itself + what it absorbed)
    got = {}
    for r in range(nrows - 1, -1, -1):
        read_now = set()
        for p in range(r * lanes, (r + 1) * lanes):
            if not flags[p] & FL_VALID:
                continue
            k = int(bus[p])
            total = Counter()
            if flags[p] & FL_C_REG:
                h = int(bus[p + lanes])            # the heir: same lane, one row earlier
                assert flags[p + lanes] & FL_P_REG and parent[p + lanes] == k
                total += sent[h]
            for s in pl["tails"][p]:
                assert s in content, f"bus {k} gathers slot {s} that nothing wrote"
                wr, w, c = content[s]
                assert wr > r and parent[pos_of(pl, w)] == k, f"bus {k} gathers slot {s} of bus {w} (row {wr})"
                total += c
                read_now.add(s)
            got[k] = total
            own = Counter({k: 1})
            a = int(pl["absorb"][p])
            if a >= 0:
                assert a in content
                wr, w, c = content[a]
                assert wr > r, f"bus {k} absorbs slot {a} written in row {wr}, not strictly earlier than {r}"
                assert k != 0 and parent[pos_of(pl, w)] == parent[p] and w != k, f"bus {k} absorbs a non-sibling"
                own += c
                read_now.add(a)
            sent[k] = own
        written = set()
        for p in range(r * lanes, (r + 1) * lanes):
            if not flags[p] & FL_VALID or flags[p] & FL_P_REG:
                continue
            s = int(pl["slot"][p])
            assert 0 <= s < pl["n_pool"]
            assert s not in read_now, f"slot {s} written in row {r}, which also reads it"
            assert s not in written, f"slot {s} written twice in row {r}"
            written.add(s)
            content[s] = (r, int(bus[p]), sent[int(bus[p])])
    return got


def replay_down(pl):
    """Root -> leaf: a bus with children behind pool slots writes its correction once; each of them reads it."""
    lanes, nrows = pl["lanes"], pl["nrows"]
    bus, parent, flags = pl["bus"], pl["parent"], pl["flags"]
    content = {}
    for r in range(nrows):
        read_now = set()
        for p in range(r * lanes, (r + 1) * lanes):
            if flags[p] & FL_VALID and not flags[p] & FL_P_REG:
                s = int(pl["x_slot"][p])
                assert content.get(s) == int(parent[p]), f"bus {bus[p]} reads slot {s}: {content.get(s)}, not its parent"
                read_now.add(s)
        for p in range(r * lanes, (r + 1) * lanes):
            s = int(pl["kids_x_slot"][p])
            if flags[p] & FL_VALID and s >= 0:
                assert 0 <= s < pl["n_pool"] and s not in read_now, f"slot {s} written in row {r}, which also reads it"
                content[s] = int(bus[p])


def pos_of(pl, k):
    return pl["_pos"][k]


@pytest.mark.parametrize("lanes", pgs.LANE_COUNTS)
@pytest.mark.parametrize("spec", FEEDER_SPECS)
def test_pool_chain_plan(spec, lanes):
    soa = _soa(spec, lanes)
    pl = pgs.plan(soa, lanes)
    valid = (pl["flags"] & FL_VALID) != 0
    pl["_pos"] = {int(pl["bus"][p]): p for p in range(pl["P"]) if valid[p]}
    n = int(valid.sum())
    par = np.asarray(soa.parent)
    kids = {k: Counter() for k in range(n)}
    for c in range(1, n):
        kids[int(par[c])][c] += 1
    # every child's contribution reaches its parent exactly once: in registers, directly or through a chain
    got = replay_up(pl)
    for k in range(n):
        assert got[k] == kids[k], f"bus {k}: {dict(got[k])} reached it, its children are {sorted(kids[k])}"
    replay_down(pl)
    for p in range(pl["P"]):          # a correction slot exactly where there are children behind pool slots
        if valid[p]:
            k = int(pl["bus"][p])
            pool_kids = [c for c in kids[k] if not pl["flags"][pl["_pos"][c]] & FL_P_REG]
            assert (pl["kids_x_slot"][p] >= 0) == bool(pool_kids)
    # no more slots, and no more gather iterations, than when the parent gathered every pool child itself
    old = pgs.legacy(pl)
    assert pl["n_pool"] <= old["n_pool"]
    after = [len(t) for t in pl["tails"]]
    assert pgs.warp_iterations(after, lanes, pl["nrows"]) <= pgs.warp_iterations(old["gather"], lanes, pl["nrows"])


def test_ieee123_on_8_lanes():
    """The headline schedule: 17 rows, 78 hand-offs in registers, at most 17 pool slots, and the 44 pool
    children of its 11 hub buses gathered in at most 12 warp-level iterations per pass (35 without chains)."""
    soa = _soa("ieee123", 8)
    pl = pgs.plan(soa, 8)
    assert pl["nrows"] == 17
    assert int(((pl["flags"] & FL_P_REG) != 0).sum()) - 1 == 78          # the root carries P_REG too
    assert pl["n_pool"] <= 17
    s = pgs.stats(soa, 8)
    assert s["pool_children"] == 44 and s["gather_before"] == 35 and s["gather_after"] <= 12
