#!/usr/bin/env python
"""Forward + backward time and peak memory of one loss over G groups of EVs that share their group's prices: the
A_bar-metric tracking error of every group's mean (price_solver.py:205-209), summed over the groups.

  grouped: LoMPC.solve_lompc_groups_diff (lompc_group_solve_dev, then one lompc_group_vjp_dev call in backward);
  gather:  lmbd[group_of], lmbd_r[group_of] -> LoMPC.solve_lompc_diff -> group means by index_add
           (autograd scatter-adds the [B, 3N] gradient back to [G, 3N]).

Shapes: G = 1,024 groups of 32 EVs (configs[2]); the closed loop's 49,152 groups (4,096 stations x 12 partitions of
500 EVs, B = 2,048,000) at N = 24 and N = 96; both EV types.  Closed-loop-scale prices (0.05 theta U).  Wall clock
around `reps` forward + backward passes, each ending in a device synchronise (both forwards also make one host sync
to check the status), after `warm` untimed ones; the two paths alternate.  Peak memory: torch.cuda.max_memory_allocated
during one pass, minus what was allocated before it (inputs and upstream data).  The grouped path also keeps device
workspace outside the torch allocator (the handle's price-loop workspace): z[B,N] and z'w[B] of the backward pass,
which outlives the forward's group index; `grouped_workspace_MB` is that size and `grouped_total_MB` the sum of both.
Checks that both paths give the same gradients (1e-9 relative; the row records the difference) before timing.
Records the card's name and power limit with the numbers.
    python tools/time_group_vjp.py [--out profiles/r4c_time_group_vjp.jsonl]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "incentive-design-mpc_b200")):
    sys.path.insert(0, p)
from chargingstation.lompc import LoMPC, LoMPCConstants  # noqa: E402

EV = {"small": (0.05, 10.0, 0.9, 0.25), "large": (0.025, 50.0, 0.9, 0.15)}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = (x.strip() for x in q.split(","))
    except Exception:
        name, limit = torch.cuda.get_device_name(0), "unknown"
    return name, limit


def fleet_sizes(stations, evs=500, parts=12):
    return [len(x) for x in np.array_split(np.arange(evs), parts)] * stations


def tracking(w_avg, w_ref, lr, delta):
    v = w_avg - w_ref
    return ((torch.cumsum(v, 1) ** 2).sum() + (lr / delta * (v * v).sum(1)).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4c_time_group_vjp.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the B200 kernels and has nothing to run here")
    name, limit = card()
    dev = torch.device("cuda:0")
    rows = []
    shapes = [("configs[2]", 24, [32] * 1024), ("closed loop", 24, fleet_sizes(4096)),
              ("closed loop", 96, fleet_sizes(4096))]
    for label, N, sizes in shapes:
        for ev, (delta, theta, y_max, w_max) in EV.items():
            s = LoMPC(N, LoMPCConstants(delta, theta, y_max, w_max, ev))
            G, B = len(sizes), int(np.sum(sizes))
            g = torch.Generator(device=dev).manual_seed(N * 7 + G)
            lm = 0.05 * theta * torch.rand((G, 3 * N), generator=g, dtype=torch.float64, device=dev)
            lr = 3 * N * delta * torch.rand(G, generator=g, dtype=torch.float64, device=dev)
            gam = y_max * torch.rand(B, generator=g, dtype=torch.float64, device=dev)
            w_ref = 0.4 * w_max * torch.rand((G, N), generator=g, dtype=torch.float64, device=dev)
            off = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32), device=dev)
            go = torch.repeat_interleave(torch.arange(G, device=dev), torch.as_tensor(sizes, device=dev))
            cnt = torch.as_tensor(sizes, dtype=torch.float64, device=dev)

            def grouped():
                lm_t, lr_t = lm.clone().requires_grad_(), lr.clone().requires_grad_()
                _, w_avg = s.solve_lompc_groups_diff(off, lm_t, lr_t, gam)
                tracking(w_avg, w_ref, lr_t, delta).backward()
                torch.cuda.synchronize()
                return lm_t.grad, lr_t.grad

            def gather():
                lm_t, lr_t = lm.clone().requires_grad_(), lr.clone().requires_grad_()
                w, _ = s.solve_lompc_diff(lm_t[go], lr_t[go], gam)
                w_avg = torch.zeros((G, N), dtype=torch.float64, device=dev).index_add(0, go, w) / cnt[:, None]
                tracking(w_avg, w_ref, lr_t, delta).backward()
                torch.cuda.synchronize()
                return lm_t.grad, lr_t.grad

            a, b = grouped(), gather()
            rel = max(float((x - y).abs().max()) / max(1.0, float(y.abs().max())) for x, y in zip(a, b))
            assert rel <= 1e-9, rel
            del a, b
            peak = {}
            for nm, fn in (("grouped", grouped), ("gather", gather)):
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                fn()
                peak[nm] = torch.cuda.max_memory_allocated() - base
            # lompc_group_vjp_dev's workspace (256-byte aligned pieces); larger than the forward's group_of + 3 [G]
            ws = ((B * N * 8 + 255) // 256 + (B * 8 + 255) // 256) * 256
            reps = 20 if B <= 100000 else 5
            t = {"grouped": [], "gather": []}
            for _ in range(2):  # warm-up
                grouped()
                gather()
            for _ in range(reps):
                for nm, fn in (("grouped", grouped), ("gather", gather)):
                    t0 = time.perf_counter()
                    fn()
                    t[nm].append(time.perf_counter() - t0)
            r = {"card": name, "power_limit": limit, "shape": label, "N": N, "ev": ev, "G": G, "B": B,
                 "grouped_ms": round(1e3 * float(np.median(t["grouped"])), 3),
                 "gather_ms": round(1e3 * float(np.median(t["gather"])), 3),
                 "grouped_ms_min": round(1e3 * min(t["grouped"]), 3), "gather_ms_min": round(1e3 * min(t["gather"]), 3),
                 "grouped_peak_MB": round(peak["grouped"] / 1e6, 1), "gather_peak_MB": round(peak["gather"] / 1e6, 1),
                 "grouped_workspace_MB": round(ws / 1e6, 1), "grouped_total_MB": round((peak["grouped"] + ws) / 1e6, 1),
                 "max_rel_grad_diff": rel, "reps": reps}
            r["speedup"] = round(r["gather_ms"] / r["grouped_ms"], 2)
            rows.append(r)
            print(json.dumps(r), flush=True)
            del lm, lr, gam, w_ref, off, go, cnt
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
