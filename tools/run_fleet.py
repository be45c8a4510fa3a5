#!/usr/bin/env python
"""BASELINE.json configs[3]: closed loop over S stations, device-resident (chargingstation.fleet).
Prints one JSON line: per-step latency (CUDA events), p50/p95, price-loop iterations.

    python tools/run_fleet.py --stations 4096 --steps 96 --chain reference
    python tools/run_fleet.py --stations 4096 --steps 16 --evs-min 100 --evs-max 900 --profile   # mixed sizes
    python tools/run_fleet.py --stations 4096 --steps 16 --station-mix --profile   # per-station BiMPC constants
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "incentive-design-mpc_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def fleet_consts(steps, N_lo, N_bi, M, P):
    from chargingstation import settings
    from chargingstation.bimpc import BiMPCChargingCostType, BiMPCConstants
    from chargingstation.charging_station import ChargingStationConstants
    from chargingstation.demand_data import medium_term_demand_forecast
    from chargingstation.lompc import LoMPCConstants
    settings.PRINT_LEVEL = 0
    dem = medium_term_demand_forecast(steps + N_bi + 1 + 24, 0.25) * (M / 500)
    cb = BiMPCConstants(1e3, 1, 1, 0.3, 0.3, BiMPCChargingCostType.EXP_UNWEIGHTED, 5)
    cs = LoMPCConstants(0.05, 10, 0.9, 0.25, "small")
    cl = LoMPCConstants(0.025, 50, 0.9, 0.15, "large")
    return ChargingStationConstants(steps, N_bi, N_lo, M, P, dem, cb, cs, cl, "linear-convex")


def fleet_demand(consts, S, steps, N_bi, seed=4):
    """SURVEY.md 8d config 4: per-station demand = the bundled profile circularly shifted by U{0..23}
    hours and scaled by U(0.22, 0.26)/0.25.  (SURVEY proposed U(0.22, 0.28); above 0.26 a station that starts
    at the evening peak with its battery empty has NO feasible BiMPC plan - demand + robustness margin
    exceed u_g_max - which the reference would report as an infeasible cvxpy problem.)"""
    rng = np.random.default_rng(seed)
    L = steps + N_bi + 1
    out = np.empty((S, L))
    for s in range(S):
        sh = int(rng.integers(24))
        out[s] = consts.demand[sh:sh + L] * (rng.uniform(0.22, 0.26) / 0.25)
    return out


def station_sizes(S, lo, hi, seed=5):
    """EVs per type of every station, uniform on {lo..hi} from a fixed seed."""
    return np.random.default_rng(seed).integers(lo, hi + 1, S)


def station_mix(base, S, seed=6):
    """Per-station BiMPC constants from a fixed seed: the base station's battery capacity x_max and rate u_b_max
    scaled by U(1, 2), its grid limit u_g_max by U(1, 1.5) and its generation cost c_g by U(0.5, 2); the cost type
    is WEIGHTED, UNWEIGHTED or EXP_UNWEIGHTED (exp_rate 5) with equal probability.  No limit is scaled below the base
    station's: with the demand of fleet_demand, batteries scaled by 0.80-0.87 left the first step's program too
    tight for the interior point (status 2)."""
    import dataclasses

    from chargingstation.bimpc import BiMPCChargingCostType
    rng = np.random.default_rng(seed)
    types = list(BiMPCChargingCostType)
    out = []
    for _ in range(S):
        bat = rng.uniform(1.0, 2.0)
        out.append(dataclasses.replace(base, x_max=base.x_max * bat, u_b_max=base.u_b_max * bat,
                                       u_g_max=base.u_g_max * rng.uniform(1.0, 1.5),
                                       c_g=base.c_g * rng.uniform(0.5, 2.0),
                                       charging_cost_type=types[int(rng.integers(len(types)))]))
    return out


def card():
    """Name and power limit of cuda:0 (the power limit is read, never set)."""
    import subprocess

    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit"] = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        out["power_limit"] = "unknown"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--stations", type=int, default=64)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--evs", type=int, default=500)
    ap.add_argument("--evs-min", type=int, default=None,
                    help="with --evs-max: station sizes uniform on {min..max}, demand scaled by size / 500")
    ap.add_argument("--evs-max", type=int, default=None)
    ap.add_argument("--station-mix", action="store_true",
                    help="per-station BiMPC constants (battery, grid limit, generation cost, cost type), fixed seed")
    ap.add_argument("--partitions", type=int, default=12)
    ap.add_argument("--n-lo", type=int, default=24)
    ap.add_argument("--n-bi", type=int, default=24)
    ap.add_argument("--chain", default="reference")
    ap.add_argument("--max-price-iter", type=int, default=1000)
    ap.add_argument("--profile", action="store_true", help="CUDA-event timing of the phases of every step")
    ap.add_argument("--loop-mode", type=int, default=0, help="price_set_loop_mode: 0 auto, 2 parametric, 3 thread-per-EV")
    args = ap.parse_args()
    import torch
    from chargingstation.fleet import ChargingStationFleet
    nevs = None
    if args.evs_min is not None or args.evs_max is not None:
        assert args.evs_min is not None and args.evs_max is not None and 1 <= args.evs_min <= args.evs_max
        nevs = station_sizes(args.stations, args.evs_min, args.evs_max)
        consts = fleet_consts(args.steps, args.n_lo, args.n_bi, 500, args.partitions)
        demand = fleet_demand(consts, args.stations, args.steps, args.n_bi) * (nevs[:, None] / 500)
    else:
        consts = fleet_consts(args.steps, args.n_lo, args.n_bi, args.evs, args.partitions)
        demand = fleet_demand(consts, args.stations, args.steps, args.n_bi)
    bimpc_consts = station_mix(consts.bimpc_consts, args.stations) if args.station_mix else None
    fleet = ChargingStationFleet(consts, args.stations, demand=demand, seed=4, rng="device", chain=args.chain,
                                 max_price_iter=args.max_price_iter, nevs=nevs, bimpc_consts=bimpc_consts)
    fleet.profile = args.profile
    for k in ("s", "l"):
        fleet.solver[k].set_loop_mode(args.loop_mode)
    fleet.sort_stations = not os.environ.get("FLEET_NO_ORDER")
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    wall = []
    for t in range(args.steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev0[t].record()
        fleet.step()
        ev1[t].record()
        torch.cuda.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3)
    ms = np.array([a.elapsed_time(b) for a, b in zip(ev0, ev1)])
    log = fleet.log
    sizes = (f"{args.evs}+{args.evs}" if nevs is None else f"U{{{args.evs_min}..{args.evs_max}}} per type")
    out = {**card(), "loop_mode": args.loop_mode,
           "pivot_overflows": [fleet.solver[k].last_pivot_overflows() for k in ("s", "l")],
           "config": f"{args.stations} stations x ({sizes}) EVs, P={args.partitions}, N_lo={args.n_lo}, "
                     f"N_bi={args.n_bi}, {args.steps} closed-loop steps, chain={args.chain}"
                     f"{', per-station BiMPC constants' if args.station_mix else ''}",
           "step_ms_p50": float(np.median(ms)), "step_ms_p95": float(np.percentile(ms, 95)),
           "step_ms_first": float(ms[0]), "step_ms_mean": float(ms.mean()), "wall_ms_p50": float(np.median(wall)),
           "price_loop_iters_per_step": fleet.price_loop_iters,
           "bimpc_iters_mean": float(log["bimpc_iters"].double().mean()),
           "bimpc_failed": int((log["bimpc_status"] != 0).sum()),
           "price_loop_qp_solves": int(fleet.qp_solves), "qp_solves_per_s": fleet.qp_solves / (ms.sum() * 1e-3),
           "cycles_lompc_passes": fleet.cycles[0], "cycles_price_steps": fleet.cycles[1],
           "k1_iters_per_solve": fleet.cycles[2] / max(1, fleet.qp_solves), "warp_passes_without_k1_iteration": fleet.cycles[3] / max(1, fleet.cycles[4])}
    out["evs_per_type"] = {"total": int(fleet.B), "mean": float(fleet.nevs.mean()), "min": int(fleet.nevs.min()),
                           "p50": float(np.median(fleet.nevs)), "p95": float(np.percentile(fleet.nevs, 95)),
                           "max": int(fleet.nevs.max())}
    st = log["bimpc_status"].cpu().numpy()
    out["bimpc_status_counts"] = {str(v): int((st == v).sum()) for v in np.unique(st)}
    bc = fleet.bimpc_consts
    q = lambda v: {"min": float(np.min(v)), "p50": float(np.median(v)), "max": float(np.max(v))}  # noqa: E731
    out["bimpc_consts"] = {f: q([getattr(c, f) for c in bc]) for f in ("x_max", "u_b_max", "u_g_max", "c_g", "delta")}
    out["bimpc_consts"]["cost_types"] = {t: sum(c.charging_cost_type.name == t for c in bc)
                                         for t in sorted({c.charging_cost_type.name for c in bc})}
    it = log["bimpc_iters"].cpu().numpy()
    out["bimpc_iters_by_cost_type"] = {t: float(it[:, [c.charging_cost_type.name == t for c in bc]].mean())
                                       for t in out["bimpc_consts"]["cost_types"]}
    if args.profile:
        out["phase_ms_median"] = {k: float(np.median([d[k] for d in fleet.phase_ms])) for k in fleet.phase_ms[0]}
        out["phase_ms_p95"] = {k: float(np.percentile([d[k] for d in fleet.phase_ms], 95)) for k in fleet.phase_ms[0]}
    for k in ("s", "l"):
        ni = log[f"niter_{k}"].cpu().numpy()
        mp = log[f"Mp_{k}"].cpu().numpy()
        v = ni[mp > 0]
        out[f"niter_{k}"] = {"mean": float(v.mean()), "p50": float(np.median(v)), "p95": float(np.percentile(v, 95)),
                             "max": int(v.max()), "capped": int((v >= args.max_price_iter - 1).sum()),
                             "groups": int(v.size)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
