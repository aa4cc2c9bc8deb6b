"""Counts what the Newton row passes do with the children handed over through shared-memory pool slots.

For every Newton workload of bench.py (and its lane count) it prints the schedule's rows, positions and pool
slots, the absorb reads of the sibling chains, and the warp-level iterations of the pool gather loop per
leaf -> root pass (elimination, mismatch-only and first-iteration passes run the same loop): before the chains
(the parent summed every pool child itself) and with them (the parent sums the chain tails).  A warp-level
iteration count is, summed over the rows, the largest count among the lanes of a warp (32 lanes at most).

    python tools/pool_gather_stats.py [--lanes 8 16 ...]

The plan is the library's own (csrc/gfr_image.hpp, compiled for the host from tools/pool_plan.cpp with g++
into a temporary directory); the "before" figures are recomputed from the same schedule.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SRC = os.path.join(ROOT, "tools", "pool_plan.cpp")
DEPENDS = [SRC] + [os.path.join(ROOT, "grid-fed-rl-gym_b200", "csrc", f) for f in ("gfr_image.hpp", "gfr_device.cuh")] + \
          [os.path.join(ROOT, "include", "gfr_b200.h")]
# record bits (csrc/gfr_device.cuh)
FL_C_REG, FL_P_REG, FL_VALID = 32, 64, 128
LANE_COUNTS = (1, 2, 4, 8, 16, 32, 64, 128, 256)     # the lane counts the kernels are instantiated for

_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha1()
        for p in DEPENDS:
            with open(p, "rb") as fh:
                h.update(fh.read())
        out = os.path.join(tempfile.gettempdir(), f"gfr_pool_plan_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = out + f".{os.getpid()}"
            res = subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-fvisibility-inlines-hidden",
                                  "-o", tmp, SRC], capture_output=True, text=True)
            if res.returncode != 0:
                raise RuntimeError("g++ failed:\n" + res.stdout + res.stderr)
            os.replace(tmp, out)
        _LIB = C.CDLL(out)
    return _LIB


def plan(soa, lanes: int) -> dict:
    """The library's Newton plan of a compiled feeder on `lanes` lanes, decoded per position."""
    from grid_fed_rl_b200 import _native as nat
    desc, keep = nat.make_feeder_desc(soa)
    info = (C.c_int * 4)()
    err = C.create_string_buffer(256)
    L = _lib()
    if L.pool_plan(C.byref(desc), lanes, info, None, 0, None, 0, err, 256) != 0:
        raise ValueError(err.value.decode())
    nrows, P, n_pool, n_list = info
    sched = np.zeros(4 * P, np.int32)
    tails = np.zeros(max(n_list, 1), np.int32)
    L.pool_plan(C.byref(desc), lanes, info, sched.ctypes.data_as(C.c_void_p), sched.size,
                tails.ctypes.data_as(C.c_void_p), tails.size, err, 256)
    del keep
    r = sched.reshape(P, 4).view(np.uint32).astype(np.int64)
    begin, ntail = r[:, 1] & 0xFFFFF, r[:, 3] & 0xFFFF
    return dict(lanes=lanes, nrows=nrows, P=P, n_pool=n_pool,
                bus=r[:, 0] & 0xFFFF, parent=r[:, 0] >> 16, flags=r[:, 2] & 0xFF,
                slot=(r[:, 2] >> 8) & 0xFFF, x_slot=r[:, 2] >> 20, kids_x_slot=(r[:, 1] >> 20) - 1,
                absorb=(r[:, 3] >> 16) - 1,
                tails=[[int(s) for s in tails[b:b + c]] for b, c in zip(begin, ntail)])


def legacy(pl: dict) -> dict:
    """What the plan was before sibling chains, on the same schedule: every pool child gathered by its parent,
    each slot held from its child's row up to the parent's (slots reused by later rows only)."""
    lanes, nrows, P = pl["lanes"], pl["nrows"], pl["P"]
    valid = (pl["flags"] & FL_VALID) != 0
    pos_of = {int(pl["bus"][p]): p for p in range(P) if valid[p]}
    pool_kids = {p: [] for p in range(P)}
    for c in range(P):
        if valid[c] and pl["bus"][c] != 0 and not pl["flags"][c] & FL_P_REG:
            pool_kids[pos_of[int(pl["parent"][c])]].append(c)
    slot, free, np_ = {}, [], 0
    for r in range(nrows - 1, -1, -1):
        released = [slot[c] for p in range(r * lanes, (r + 1) * lanes) for c in pool_kids[p]]
        for p in range(r * lanes, (r + 1) * lanes):
            if valid[p] and not pl["flags"][p] & FL_P_REG:
                if free:
                    s = min(free); free.remove(s)
                else:
                    s, np_ = np_, np_ + 1
                slot[p] = s
        free += released
    return dict(gather=np.array([len(pool_kids[p]) for p in range(P)]), n_pool=max(np_, 1))


def warp_iterations(counts, lanes: int, nrows: int) -> int:
    """Sum over rows (and warps of a CTA-wide group) of the largest per-lane count in a warp."""
    w = min(lanes, 32)
    c = np.asarray(counts).reshape(nrows, lanes // w, w)
    return int(c.max(axis=2).sum())


def stats(soa, lanes: int) -> dict:
    pl = plan(soa, lanes)
    old = legacy(pl)
    after = np.array([len(t) for t in pl["tails"]])
    return dict(rows=pl["nrows"], positions=pl["P"], pool_slots=pl["n_pool"], pool_slots_before=old["n_pool"],
                pool_children=int(old["gather"].sum()), absorb_reads=int((pl["absorb"] >= 0).sum()),
                gather_before=warp_iterations(old["gather"], lanes, pl["nrows"]),
                gather_after=warp_iterations(after, lanes, pl["nrows"]))


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--lanes", type=int, nargs="*", default=None,
                    help="lane counts to show besides each workload's own (the auto rule's)")
    args = ap.parse_args()
    import bench
    from grid_fed_rl_b200.topology import compile_for_solver
    head = (f"{'workload':<15} {'lanes':>5} {'rows':>4} {'pos':>5} {'slots':>11} {'pool kids':>9} "
            f"{'absorbs':>7} {'gather it/pass':>15}")
    print(head)
    print("-" * len(head))
    for name, (spec, _, solver, _, _) in bench.WORKLOADS.items():
        if solver != "newton":
            continue
        f = bench.make_feeder(spec)
        _, auto = compile_for_solver(f, "newton", 0, with_components=False)
        for lanes in [auto] + [ln for ln in (args.lanes or []) if ln != auto]:
            soa, used = compile_for_solver(f, "newton", lanes, with_components=False)
            s = stats(soa, used)
            print(f"{name:<15} {used:>5} {s['rows']:>4} {s['positions']:>5} "
                  f"{s['pool_slots_before']:>4} -> {s['pool_slots']:<4} {s['pool_children']:>9} {s['absorb_reads']:>7} "
                  f"{s['gather_before']:>6} -> {s['gather_after']:<6}")


if __name__ == "__main__":
    main()
