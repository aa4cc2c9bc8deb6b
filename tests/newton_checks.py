"""TEST INFRASTRUCTURE: a Newton solve checked iterate by iterate against the oracle (tests/reactive_oracle.py).

End-state checks cannot see most kernel errors: Newton corrects them, at the cost of an iteration or two.  A solve
stopped at ``max_iterations`` = 1, 2, 3 is a deterministic function of the first iterates, so it is compared with the
oracle run with the same ``max_iterations`` and acceleration to rounding (``check_truncated``).  A converged solve
is compared to the solver bound, with exact iteration counts (``check_converged``).

Results are dicts of numpy arrays with the keys of ``PowerFlowSolution``; line loadings on the solve surface are
|S| s_base / rating, the oracle's are |S| / rating.
"""
from __future__ import annotations

import numpy as np

from tests.golden_util import TOL_PU
from tests.reactive_oracle import newton_raphson_pq

STATE = ("bus_voltages", "bus_angles", "line_flows", "losses")


def as_numpy(sol) -> dict:
    """A PowerFlowSolution of tensors (or a dict of arrays) as a dict of numpy arrays."""
    get = sol.get if isinstance(sol, dict) else (lambda k: getattr(sol, k))
    out = {}
    for k in STATE + ("converged", "iterations", "line_loadings", "max_mismatch"):
        v = get(k)
        v = v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)
        out[k] = v.astype(bool) if k == "converged" else v
    return out


def max_state_diff(sol: dict, ref: dict, rows=slice(None), scale=None) -> float:
    """The largest difference of |V|, angle, line P and losses; line P and losses over ``scale`` [B] when given."""
    d = 0.0
    for k in STATE:
        e = np.abs(sol[k][rows] - ref[k][rows])
        if scale is not None and k in ("line_flows", "losses"):
            e = e / (scale[rows][:, None] if e.ndim == 2 else scale[rows])
        d = max(d, float(np.max(e, initial=0.0)))
    return d


def _loadings_agree(sol, ref, s_base, rows, rtol):
    a, b = sol["line_loadings"][rows], ref["line_loadings"][rows] * s_base
    return np.all(np.abs(a - b) <= rtol * np.abs(b) + 1e-12)


def check_truncated(sol: dict, ref: dict, s_base: float, bound: float = 1e-10, ctx="") -> float:
    """A solve stopped at ``max_iterations``: flags, counts and NaN-ness exact, the state within ``bound`` pu,
    loadings within a relative 1e-9, the mismatch within 1e-10 + 1e-7 |mm|.  Returns the largest state difference.

    Line P and losses are compared relative to max(1, sum of |S| over the lines) of the row: 1 pu for an iterate
    near the operating point, but a diverging iterate (|V| of 10 - 40 pu after the second update of a row whose
    first correction is > 0.25 rad) carries line flows of 1e4 pu, and the oracle's losses, Re sum V conj(Y V), are
    a difference of injections that size: rounding alone moves them by more than 1e-10 there, while |V| and the
    angles still agree with a 40-digit Newton to 1e-12."""
    assert np.array_equal(sol["converged"], ref["converged"]), ctx
    assert np.array_equal(sol["iterations"].astype(int), ref["iterations"].astype(int)), ctx
    for k in STATE + ("line_loadings", "max_mismatch"):
        assert np.array_equal(np.isnan(sol[k]), np.isnan(ref[k])), (ctx, k)
    fin = ~np.isnan(ref["bus_voltages"]).any(axis=1)
    scale = np.maximum(1.0, np.sum(ref["line_s_abs"], axis=1))
    d = max_state_diff(sol, ref, fin, scale)
    assert d <= bound, (ctx, d)
    assert _loadings_agree(sol, ref, s_base, fin, 1e-9), ctx
    mm, rm = sol["max_mismatch"][fin], ref["max_mismatch"][fin]
    assert np.all(np.abs(mm - rm) <= 1e-10 + 1e-7 * np.abs(rm)), (ctx, np.max(np.abs(mm - rm)))
    return d


def borderline_rows(net, p, q, ref, tolerance, acceleration):
    """Rows whose oracle mismatch at the deciding check is within a factor 10 of the tolerance: at the converging
    check above tolerance / 10, or at the one before below 10 tolerance.  Rounding may move those by one iteration."""
    it = ref["iterations"].astype(int)
    near = ref["converged"] & (ref["max_mismatch"] > 0.1 * tolerance)
    for k in np.unique(it[ref["converged"] & (it > 1)]):
        rows = np.flatnonzero(ref["converged"] & (it == k))
        prev = newton_raphson_pq(net, p[rows], None if q is None else q[rows], tolerance, int(k) - 1, acceleration)
        near[rows] |= prev["max_mismatch"] < 10.0 * tolerance
    return near


def check_converged(sol: dict, ref: dict, s_base: float, near, tolerance: float, ctx="") -> float:
    """A solve run to convergence: flags exact, iteration counts exact except on borderline rows (``near``), which
    may differ by one and must be under 5 % of the rows; the state within the solver bound (1e-8 pu) and the
    mismatch below the tolerance on converged rows.  Returns the largest state difference on converged rows.  (A
    row that diverges is chaotic after a few updates: only its flag is compared.)"""
    assert np.array_equal(sol["converged"], ref["converged"]), ctx
    ok = ref["converged"]
    di = np.abs(sol["iterations"].astype(int) - ref["iterations"].astype(int))[ok]
    off = di != 0
    assert np.all(di <= 1) and np.all(near[ok][off]), (ctx, np.flatnonzero(off))
    assert off.sum() <= 0.05 * off.size, (ctx, int(off.sum()))
    d = max_state_diff(sol, ref, ok)
    assert d <= TOL_PU, (ctx, d)
    assert _loadings_agree(sol, ref, s_base, ok, 1e-7), ctx
    assert np.all(sol["max_mismatch"][ok] < tolerance), ctx
    return d
