#!/usr/bin/env python
"""Price loops with the "max" tolerance type (price_solver.py:121-128) on the route it had before the parametric loop
served it - the thread-per-EV loop (mode 3) at N = 12, 24, the phase-split loop (mode 1) at N = 48, 96 - and on the
parametric loop (automatic mode), next to the parametric loop with "avg".  1,024 groups x 32 EVs per EV type, seeded,
capped at 60 iterations; one untimed run of each path first.  The two "max" paths must give the same iteration counts.
    python tools/time_max_tol_loops.py"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "incentive-design-mpc_b200")):
    sys.path.insert(0, p)
from chargingstation import settings  # noqa: E402
from chargingstation.lompc import LoMPCConstants  # noqa: E402
from chargingstation.price_solver import PriceSolver  # noqa: E402

settings.PRINT_LEVEL = 0
EV = {"small": (0.05, 10.0, 0.9, 0.25), "large": (0.025, 50.0, 0.9, 0.15)}
G, n = 1024, 32
for N in (12, 24, 48, 96):
    for ev, (delta, theta, y_max, w_max) in EV.items():
        rng = np.random.default_rng(N)
        off = (np.arange(G + 1) * n).astype(np.int32)
        y0 = np.sort(0.3 + 0.2 * rng.random(G * n)).reshape(G, n)[rng.permutation(G)].ravel()
        w_ref = w_max * rng.random((G, N)) * 0.6
        args = (off, y0, w_ref, np.zeros(G), np.zeros((G, 3 * N)))
        res = {}
        for name, mode, tol_type in (("max_old_route", 3 if N <= 24 else 1, "max"), ("max_parametric", 0, "max"),
                                     ("avg_parametric", 0, "avg")):
            ps = PriceSolver(N, LoMPCConstants(delta, theta, y_max, w_max, ev), "linear-convex")
            ps.set_loop_mode(mode)
            ps.compute_optimal_prices_batch(*args, max_iter=60, tol_type=tol_type)
            t0 = time.perf_counter()
            prices, st = ps.compute_optimal_prices_batch(*args, max_iter=60, tol_type=tol_type)
            ms = (time.perf_counter() - t0) * 1e3
            res[name] = (ms, prices, st["iter"].copy(), int(ps._lib.price_last_qp_solves(ps._h)))
        old, new = res["max_old_route"], res["max_parametric"]
        assert np.array_equal(old[2], new[2]), "the two max paths disagree on iteration counts"
        small = np.abs(old[1]) <= 1e3
        print(json.dumps({
            "N": N, "ev": ev, "groups": G, "evs": G * n,
            "max_old_route": "thread-per-EV" if N <= 24 else "phase-split",
            "max_old_route_ms": round(old[0], 3), "max_parametric_ms": round(new[0], 3),
            "avg_parametric_ms": round(res["avg_parametric"][0], 3),
            "max_iters_mean": float(new[2].mean()), "avg_iters_mean": float(res["avg_parametric"][2].mean()),
            # (the phase-split loop does not count its solves: every EV and the virtual EV per iteration)
            "max_old_route_qp_solves": old[3] if N <= 24 else int(np.sum((n + 1) * (old[2] + 1))),
            "max_parametric_qp_solves": new[3], "avg_parametric_qp_solves": res["avg_parametric"][3],
            "max_price_diff": float(np.max(np.abs(old[1] - new[1])[small]))}), flush=True)
