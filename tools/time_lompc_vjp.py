#!/usr/bin/env python
"""Time of one lompc_vjp_dev launch (the backward pass of LoMPC.solve_lompc_diff: grad_w and grad_cost given, every
output written) next to the forward solve (lompc_solve_batch_dev, automatic kernel choice) on the same batch.
N in {12, 24, 96, 168}, B in {1,024; 16,384; 524,288}, both EV types, prices drawn like tests/test_lompc_gpu.py.
CUDA events around `reps` back-to-back launches after `warm` untimed ones; at B = 524,288 every input is larger than
the 126 MB L2 (N = 12: lmbd alone is 151 MB), so the timed launches stream from HBM; the smaller batches run from L2.
Records the card's name and power limit with the numbers.
    python tools/time_lompc_vjp.py [--out profiles/r4b_time_lompc_vjp.jsonl]"""
import argparse
import json
import os
import subprocess
import sys

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


def time_us(fn, warm, reps):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4b_time_lompc_vjp.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the B200 kernels and has nothing to run here")
    name, limit = card()
    dev = torch.device("cuda:0")
    rows = []
    for N in (12, 24, 96, 168):
        for ev, (delta, theta, y_max, w_max) in EV.items():
            s = LoMPC(N, LoMPCConstants(delta, theta, y_max, w_max, ev))
            for B in (1024, 16384, 524288):
                g = torch.Generator(device=dev).manual_seed(N * 7 + B)
                lm = theta * torch.rand((B, 3 * N), generator=g, dtype=torch.float64, device=dev)
                lr = 3 * N * delta * torch.rand(B, generator=g, dtype=torch.float64, device=dev)
                gam = y_max * torch.rand(B, generator=g, dtype=torch.float64, device=dev)
                gw = torch.randn((B, N), generator=g, dtype=torch.float64, device=dev)
                gc = torch.randn(B, generator=g, dtype=torch.float64, device=dev)
                w, cost = s.solve_lompc_batch(lm, lr, gam)
                out = (torch.empty_like(lm), torch.empty_like(lr), torch.empty_like(gam))
                h, lib = s._h, s._lib
                stream = torch.cuda.current_stream(dev).cuda_stream
                ptrs = [x.data_ptr() for x in (lm, lr, gam, w, cost, gw, gc) + out]

                def fwd():
                    lib.lompc_solve_batch_dev(h, B, ptrs[0], 3 * N, ptrs[1], 1, ptrs[2], ptrs[3], ptrs[4],
                                              None, None, None, stream)

                def vjp():
                    lib.lompc_vjp_dev(h, B, ptrs[0], 3 * N, ptrs[1], 1, ptrs[2], ptrs[3], ptrs[5], ptrs[6],
                                      ptrs[7], ptrs[8], ptrs[9], None, stream)

                reps = 200 if B <= 16384 else (40 if N <= 24 else 10)
                t_f = time_us(fwd, 3, reps)
                t_v = time_us(vjp, 3, reps)
                # bytes the VJP must move: lmbd, w, grad_w, grad_lmbd rows + lmbd_r, gamma, grad_cost, 2 outputs
                vjp_bytes = B * 8 * (3 * N + N + N + 3 * N + 5)
                r = {"card": name, "power_limit": limit, "N": N, "ev": ev, "B": B, "forward_us": round(t_f, 2),
                     "vjp_us": round(t_v, 2), "vjp_over_forward": round(t_v / t_f, 3),
                     "vjp_GB_per_s": round(vjp_bytes / t_v / 1e3, 1), "reps": reps}
                rows.append(r)
                print(json.dumps(r), flush=True)
                del lm, lr, gam, gw, gc, w, cost, out
                torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
