#!/usr/bin/env python
"""Benchmark of the LoMPC hot path (BASELINE.json: "LL-MPC QP solves/sec").

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # reference CPU path (restated)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results to DIR/*.npy

Workload at N=1 = BASELINE.json configs[1]: 1,024 independent horizon-24
lower-level MPC QPs (512 small-EV + 512 large-EV), inputs drawn as the
reference's own timing script does (test/test_lompc.py:34-36), seed 2.  Under
torchrun every rank runs its own 1,024 QPs (weak scaling, no data-path
collective: the QPs are independent).  One "step" = one pass of the hot path
over that batch = ONE kernel launch: both EV types go through a solve set
(chargingstation.lompc.LoMPCSet -> lompc_set_solve_*), whose warp-cooperative
kernel serves every segment.

`value`  : QP solves/s, inputs resident in HBM, CUDA events around each step,
           L2 flushed between steps, max over ranks.
`e2e`    : the same metric through the public API (LoMPCSet.solve ->
           lompc_set_solve_host) with the inputs in pinned HOST memory: one H2D
           copy, the launch, one D2H copy and the synchronisation are inside the
           timed region (wall clock).
`roofline`: reported against the BINDING roof: the arithmetic intensity of the
           exact method (2.6-4.3 flop/B) is below the machine balance (measured
           DFMA peak / measured HBM bandwidth = 5.2 flop/B), so that is HBM;
           the FP64 figures (peak = DFMA chain measured in this run) are next to it.
`cpu_baseline`: oracle/lompc_oracle.c (a C restatement of the cvxpy->CLARABEL
           interior-point solve; cvxpy itself is not installable here) on all
           host threads, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "incentive-design-mpc_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

N_HORIZON = 24
METRIC = "lompc_qp_solves_per_sec"
UNIT = "QP/s"

# (delta, theta, y_max, w_max, type): example/real_time_price_control.py:26-39
EV_CONSTS = {"small": (0.05, 10.0, 0.9, 0.25), "large": (0.025, 50.0, 0.9, 0.15)}


def draw_workload(batch: int, N: int, seed: int):
    """configs[1]: half small, half large EVs; test/test_lompc.py:34-36 distributions."""
    rng = np.random.default_rng(seed)
    out = {}
    for ev in ("small", "large"):
        delta, theta, y_max, w_max = EV_CONSTS[ev]
        B = batch // 2
        out[ev] = (theta * rng.random((B, 3 * N)), 3 * N * delta * rng.random(B), y_max * rng.random(B))
    return out


def flops_per_qp(ev: str, N: int, iters_mean: float, optimistic: bool = True) -> float:
    """Algorithmic FP64 flops of one solve (FMA = 2, comparisons / selects not counted; DESIGN.md section 4):
    setup + final cost 16N (25N large), backward sweep 19N (20N), forward sweep 14N (31N) with the objective
    of the rollout, 3N (17N) without it -- the optimistic phase of K1, which is the one that runs on strictly
    convex stage costs such as this workload's (every price > 0).  A solve that stops after `it` iterations
    ran it+1 backward and it forward sweeps."""
    if ev == "small":
        return N * (16 + 19 * (iters_mean + 1) + (3 if optimistic else 14) * iters_mean)
    return N * (25 + 20 * (iters_mean + 1) + (17 if optimistic else 31) * iters_mean)


def bytes_per_qp(N: int) -> int:
    return 8 * (4 * N + 3)  # SURVEY.md 8d: 8(3N+2) in + 8(N+1) out


class ClockSampler:
    """Samples SM clocks / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            if os.environ.get("BENCH_NO_NVML"):
                raise RuntimeError("disabled")
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.01)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# --------------------------------------------------------------------------- CPU arm
def cpu_pass(work, N, nthreads=0):
    """One pass of the restated reference CPU path over the workload; returns threads used."""
    from oracle import c_oracle, lompc_oracle as orc
    used = 1
    for ev, (lm, lr, gam) in work.items():
        o = orc.small_ev_consts() if ev == "small" else orc.large_ev_consts()
        _, _, _, used = c_oracle.solve_lompc_batch(N, o, lm, lr, gam, nthreads=nthreads)
    return used


def run_reference(args, rank: int, world: int) -> None:
    if rank != 0:
        return
    work = draw_workload(args.batch, N_HORIZON, 2)
    for _ in range(max(args.warmup, 1)):
        used = cpu_pass(work, N_HORIZON)
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_pass(work, N_HORIZON)
    dt = (time.perf_counter() - t0) / steps
    value = args.batch / dt
    sample = (f"{args.batch} QPs/step ({args.batch // 2} small + {args.batch // 2} large, N={N_HORIZON}), "
              f"{steps} steps, oracle/lompc_oracle.c IPM tol 1e-8")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "cvxpy/CLARABEL are not installable in this image; this arm times the C restatement "
                "of the reference's interior-point solve on all host threads",
    }
    print(json.dumps(line), flush=True)


def workload_config(args):
    return {"workload": f"BASELINE.json configs[1]: {args.batch} independent horizon-{N_HORIZON} LoMPC QPs per GPU "
                        f"({args.batch // 2} small-EV + {args.batch // 2} large-EV), inputs as test_lompc.py:34-36, seed 2",
            "batch_per_gpu": args.batch, "horizon": N_HORIZON,
            "l2": "inputs larger than L2: every timed step solves its OWN resident batch, and right before the timed "
                  "region the kernel runs over other resident batches of together 1.25x the L2 size (they are the "
                  "warm-up steps), so no timed batch is cached; `step_latency` keeps the flushed single-step number",
            "launch": "one launch per step (the warp-cooperative kernel serves both EV types, lompc_set_solve_dev_at); "
                      "the K timed steps are one CUDA graph between two events"}


# --------------------------------------------------------------------------- GPU arm
def run_ours(args, rank: int, local_rank: int, world: int) -> None:
    import torch
    import torch.distributed as dist
    from chargingstation import _native
    from chargingstation.lompc import LoMPC, LoMPCConstants, LoMPCSet

    lib = _native.load()
    if lib.lompc_device_count() <= local_rank:
        raise RuntimeError("bench.py needs a CUDA device: this path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    N = N_HORIZON
    work = draw_workload(args.batch, N, 2 + rank)
    solvers, dev_in = {}, {}
    for ev, (lm, lr, gam) in work.items():
        delta, theta, y_max, w_max = EV_CONSTS[ev]
        solvers[ev] = LoMPC(N, LoMPCConstants(delta, theta, y_max, w_max, ev), device=local_rank)
        dev_in[ev] = tuple(torch.from_numpy(x).to(dev) for x in (lm, lr, gam))
    # Both EV types in one solve set: the workload is written ONCE into the set's pinned input views (the host
    # buffers of the e2e leg) and uploaded once into its device block (the HBM-resident inputs of `value`).
    evs_order = ("large", "small")  # the slower EV type first: its warps are scheduled (and fed over PCIe) first
    sset = LoMPCSet([solvers[ev] for ev in evs_order], [work[ev][2].shape[0] for ev in evs_order])
    for i, ev in enumerate(evs_order):
        lm, lr, gam = work[ev]
        sset.lmbd[i][:], sset.lmbd_r[i][:], sset.gamma[i][:] = lm, lr, gam
    sset.upload(torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step_device():
        sset.solve_dev(torch.cuda.current_stream(dev).cuda_stream)  # one launch, device block -> device block

    def step_host():
        sset.solve()  # one H2D copy, one launch, one D2H copy, synchronise; raises on a failed QP

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # iteration statistics (for the flop model) + a correctness spot check before timing
    iters_mean = {}
    for ev in ("small", "large"):
        _, _, info = solvers[ev].solve_lompc_batch(*dev_in[ev], return_info=True)
        torch.cuda.synchronize()
        assert int(info["status"].max()) == 0, "solver reported a non-converged QP"
        assert float(info["kkt_res"].max()) <= 1e-10
        iters_mean[ev] = float(info["iters"].double().mean())

    # FP64 peak of this device, measured now
    tf = _native.C.c_double()
    ms = _native.C.c_double()
    _native.raise_for(lib.lompc_measure_fp64_peak(local_rank, 4096, _native.C.byref(tf), _native.C.byref(ms)))
    fp64_peak = tf.value

    # ---- device-timed leg.  K + E batches of the workload's shape are RESIDENT in HBM, each in its own packed
    # block (batch 0 = the seeded workload, the others drawn from the same distributions): E "other" batches of
    # together more than the L2 are solved right before the timed region (they are the warm-up AND they evict the
    # timed batches from the cache), then EXACTLY K steps - one launch each, every step on its own batch - are timed
    # as one region between two events.  Both passes are CUDA graphs, so no host call sits inside the region.
    K, W = args.steps, max(args.warmup, 3)
    in_bytes, out_bytes = sset.h2d_bytes, sset.d2h_bytes
    l2_bytes = torch.cuda.get_device_properties(dev).L2_cache_size
    E = max(W, int(1.25 * l2_bytes / (in_bytes + out_bytes)) + 1)
    R = K + E
    in_blocks = torch.zeros((R, in_bytes), dtype=torch.uint8, device=dev)
    out_blocks = torch.zeros((R, out_bytes), dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    in_f64 = in_blocks.view(torch.float64)
    for i, ev in enumerate(evs_order):
        delta, theta, y_max, w_max = EV_CONSTS[ev]
        B = work[ev][2].shape[0]
        o_lm, o_lr, o_ga, _, _ = sset.offsets(i)
        in_f64[:, o_lm // 8: o_lm // 8 + B * 3 * N] = theta * torch.rand((R, B * 3 * N), dtype=torch.float64, device=dev, generator=gen)
        in_f64[:, o_lr // 8: o_lr // 8 + B] = 3 * N * delta * torch.rand((R, B), dtype=torch.float64, device=dev, generator=gen)
        in_f64[:, o_ga // 8: o_ga // 8 + B] = y_max * torch.rand((R, B), dtype=torch.float64, device=dev, generator=gen)
        for x, o in zip(dev_in[ev], (o_lm, o_lr, o_ga)):  # batch 0 = the seeded workload
            in_f64[0, o // 8: o // 8 + x.numel()] = x.reshape(-1)
    torch.cuda.synchronize()

    def launch_on(r):
        sset.solve_dev_at(in_blocks[r].data_ptr(), out_blocks[r].data_ptr(), torch.cuda.current_stream(dev).cuda_stream)

    launch_on(0)
    torch.cuda.synchronize()
    # batch 0 solved in its block == the seeded workload solved through the per-object API
    o_w = {ev: sset.offsets(i)[3] for i, ev in enumerate(evs_order)}
    for ev in evs_order:
        w_chk, _ = solvers[ev].solve_lompc_batch(*dev_in[ev])
        got = out_blocks.view(torch.float64)[0, o_w[ev] // 8: o_w[ev] // 8 + w_chk.numel()].reshape(w_chk.shape)
        assert torch.equal(got, w_chk), "solve set on a resident block differs from the per-object solve"
    assert int(out_blocks[:1].view(torch.int64)[0, 0]) % 4 == 0, "a QP of the seeded batch failed"
    graph_evict, graph_timed = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph_evict):
        for r in range(K, R):
            launch_on(r)
    l0 = lib.lompc_launch_count()
    with torch.cuda.graph(graph_timed):
        for r in range(K):
            launch_on(r)
    per_replay = lib.lompc_launch_count() - l0
    graph_evict.replay()
    graph_timed.replay()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    graph_evict.replay()  # warm-up steps on the other batches; leaves none of the timed batches in L2
    barrier()
    sampler.start()
    e_start, e_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_start.record()
    graph_timed.replay()  # exactly K steps
    e_stop.record()
    barrier()
    launches = per_replay
    dev_ms = e_start.elapsed_time(e_stop)
    assert int(out_blocks[:K].view(torch.int64)[:, 0].remainder(4).max()) == 0, "a QP inside the timed region failed"
    last_block = out_blocks[K - 1].cpu().numpy() if args.dump_outputs else None  # the last timed step's out block

    # ---- the same K steps with independent steps allowed to OVERLAP: the batches of different steps have nothing to
    # do with each other, and one 1,024-QP launch (256 single-warp CTAs) leaves most of the GPU idle, so a caller with
    # several sets in flight gets more than 1 / latency.  Reported next to `value`, which stays the one-stream number.
    overlapped = {}
    for S in (2, 4, 8):
        side = [torch.cuda.Stream(dev) for _ in range(S)]
        g_ov = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_ov):
            main = torch.cuda.current_stream(dev)
            fork = torch.cuda.Event()
            fork.record(main)
            for st_ in side:
                st_.wait_event(fork)
            for r in range(K):
                with torch.cuda.stream(side[r % S]):
                    launch_on(r)
            for st_ in side:
                join = torch.cuda.Event()
                join.record(st_)
                main.wait_event(join)
        out_blocks[:K].zero_()
        graph_evict.replay()
        barrier()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record()
        g_ov.replay()
        o1.record()
        barrier()
        assert int(out_blocks[:K].view(torch.int64)[:, 0].remainder(4).max()) == 0, "a QP of an overlapped step failed"
        w0_ = o_w[evs_order[0]] // 8  # (the blocks were zeroed above: every step must have written its results)
        assert float(out_blocks[:K].view(torch.float64)[:, w0_: w0_ + 64 * N].abs().sum(dim=1).min()) > 0.0, \
            "an overlapped step did not run"
        ov_ms = o0.elapsed_time(o1)
        if world > 1:
            t_ov = torch.tensor([ov_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t_ov, op=dist.ReduceOp.MAX)
            ov_ms = float(t_ov.item())
        overlapped[str(S)] = {"ms_per_step": ov_ms / K, "value": world * args.batch * K / (ov_ms * 1e-3)}
        del g_ov

    # ---- single-step latency with the L2 flushed before every step (round 1's methodology, kept for comparison):
    # one graph replay between two events, 256 MiB memset in between
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step_device()
    lat_steps = min(K, 20)
    for _ in range(3):
        flush.zero_()
        graph.replay()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(lat_steps)]
    for e0, e1 in evs:
        flush.zero_()  # L2 flush, outside the timed events
        e0.record()
        graph.replay()
        e1.record()
    barrier()
    step_ms = [e0.elapsed_time(e1) for e0, e1 in evs]

    # end-to-end through the public API with pinned host buffers (wall clock, copies inside)
    for _ in range(max(args.warmup, 3)):
        step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    e2e_last = [(w.copy(), c.copy()) for w, c in zip(sset.w, sset.cost)] if args.dump_outputs else None

    # saturating batch (explains `value`: 1,024 QPs cannot fill 148 SMs)
    sat = None
    if not args.no_saturated:
        sat = saturated_run(solvers, dev, rank, fp64_peak)
    clocks = sampler.stop()
    closed = None
    if args.closed_loop_stations > 0:
        closed = closed_loop_leg(args, rank, world, dev)
    sharded = None
    if args.sharded_iters > 0:
        sharded = sharded_leg(args, rank, world, dev)

    t = torch.tensor([dev_ms, e2e_s], dtype=torch.float64, device=dev)
    per_rank = None
    if world > 1:
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = {"ms_per_step": [float(x[0]) / args.steps for x in allt],
                    "e2e_ms_per_step": [float(x[1]) / args.steps * 1e3 for x in allt],
                    }
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_s = float(t[0]), float(t[1])

    if rank == 0:
        total_qps = args.batch * world
        ms_per_step = dev_ms / args.steps
        value = total_qps / (ms_per_step * 1e-3)
        flops_step = sum(flops_per_qp(ev, N, iters_mean[ev]) * (args.batch // 2) for ev in ("small", "large"))
        achieved_tf = flops_step / (ms_per_step * 1e-3) / 1e12
        bytes_step = bytes_per_qp(N) * args.batch
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic, traffic_src = None, None
        try:  # DRAM bytes of the dominant kernel from the committed ncu --set full capture, per launch
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["set_1024"]
            if args.batch == tj["qps"]:
                traffic = tj["bytes_per_launch"]
                traffic_src = (f"dram__bytes_read + dram__bytes_write of one launch, {tj['source']}; algorithmic "
                               f"{bytes_per_qp(N) * args.batch} B per launch ({tj['note']})")
        except Exception:
            pass
        h2d, d2h = sset.h2d_bytes, sset.d2h_bytes  # the packed blocks actually copied (segments 256-byte aligned)
        step_s = ms_per_step * 1e-3
        hbm_gbs = bytes_step / step_s / 1e9
        t_hbm, t_fp64 = bytes_step / (hbm_peak * 1e9), flops_step / (fp64_peak * 1e12)
        binding = "hbm" if t_hbm >= t_fp64 else "fp64"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "roofline": {
                # the binding roof of this workload: max(bytes / HBM peak, flops / FP64 peak) is the HBM term
                # (arithmetic intensity flops_step / bytes_step below the machine balance)
                "bound": "hbm" if binding == "hbm" else "tensor", "binding_roof": binding,
                "achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback",
                "arithmetic_intensity_flop_per_byte": flops_step / bytes_step,
                "machine_balance_flop_per_byte": fp64_peak * 1e12 / (hbm_peak * 1e9),
                "roof_time_us": max(t_hbm, t_fp64) * 1e6,
                "mean_iters": iters_mean, "flops_per_step": flops_step, "bytes_per_step": bytes_step,
                "fp64": {"achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved_tf / fp64_peak,
                         "peak_source": "DFMA chain microbenchmark measured in this run "
                                        "(MEASURED_PEAKS.json has no FP64 figure)"},
                "note": "1,024 QPs (256 warps of the warp-cooperative kernel) cannot fill 148 SMs: this configuration is "
                        "bound by launch + dependent-issue latency (an empty launch between the two events costs "
                        "~5 us of the step); see `saturated` for the throughput regime (one QP per thread)",
            },
            "e2e": {"value": total_qps * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s / args.steps * 1e3,
                    "api": "LoMPCSet.solve() -> lompc_set_solve_host: the caller's inputs live in the set's pinned host "
                           "views; ONE launch (a CUDA graph) + stream synchronise per step",
                    "transfer": "zero-copy: the kernel loads the step's inputs from the pinned host block and stores w / "
                                "cost / status into the pinned host output block over PCIe (h2d / d2h bytes = those "
                                "blocks); LOMPC_SET_MAPPED=0 selects the staged variant (1 H2D copy + launch + 1 D2H copy)"
                                if os.environ.get("LOMPC_SET_MAPPED", "1") != "0" else
                                "staged: 1 cudaMemcpyAsync H2D + launch + 1 cudaMemcpyAsync D2H, status reduced on the device"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "saturated": sat,
            "closed_loop": closed,
            "sharded": sharded,
            "per_rank": per_rank,
            "overlapped_steps": {"by_streams": overlapped, "unit": UNIT,
                                 "note": "the same K steps on the same resident batches, issued round-robin on 2 / 4 / 8 "
                                         "streams inside one CUDA graph (independent steps may overlap); `value` "
                                         "above is the one-stream figure"},
            "step_latency": {"ms_per_step_l2_flushed": float(np.median(step_ms)), "steps": len(step_ms),
                             "min_ms": float(np.min(step_ms)), "max_ms": float(np.max(step_ms)),
                             "note": "ONE step between two events after a 256 MiB memset (round 1's methodology): "
                                     "includes the ~5 us an empty launch costs between two events"},
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_leg(args)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, sset, evs_order, last_block, e2e_last)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(path, sset, evs_order, last_block, e2e_last):
    """Writes what the timed steps returned in their last step as float64 DIR/<name>.npy, so that two builds can be
    compared output for output (the inputs are seeded): `step_*` is the out block of the device-timed leg's last
    step (w [B, N] and cost [B] of every EV type, and the worst QP status of the launch), `e2e_*` the w / cost views
    of the set after the last end-to-end step (the seeded workload)."""
    os.makedirs(path, exist_ok=True)
    out = {"step_worst_status": np.array([last_block[:8].view(np.int64)[0] % 4])}
    f64 = last_block.view(np.float64)
    for i, ev in enumerate(evs_order):
        B, N = sset.batch_sizes[i], sset.N
        o_w, o_cost = sset.offsets(i)[3:]
        out[f"step_w_{ev}"] = f64[o_w // 8: o_w // 8 + B * N].reshape(B, N)
        out[f"step_cost_{ev}"] = f64[o_cost // 8: o_cost // 8 + B]
        out[f"e2e_w_{ev}"], out[f"e2e_cost_{ev}"] = e2e_last[i]
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def saturated_run(solvers, dev, rank, fp64_peak):
    """Same kernel, same distributions, at a batch that fills the GPU (2 x 2^19 QPs)."""
    import torch
    N = N_HORIZON
    Bs = 1 << 19
    rng = np.random.default_rng(1000 + rank)
    res = {"batch": 2 * Bs, "per_type": {}}
    tot_ms, tot_flops = 0.0, 0.0
    for ev in ("small", "large"):
        delta, theta, y_max, w_max = EV_CONSTS[ev]
        lm = torch.from_numpy(theta * rng.random((Bs, 3 * N))).to(dev)
        lr = torch.from_numpy(3 * N * delta * rng.random(Bs)).to(dev)
        gam = torch.from_numpy(y_max * rng.random(Bs)).to(dev)
        out = (torch.empty((Bs, N), dtype=torch.float64, device=dev), torch.empty((Bs,), dtype=torch.float64, device=dev))
        _, _, info = solvers[ev].solve_lompc_batch(lm, lr, gam, return_info=True)
        it_mean = float(info["iters"].double().mean())
        for _ in range(3):
            solvers[ev].solve_lompc_batch(lm, lr, gam, out=out)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            solvers[ev].solve_lompc_batch(lm, lr, gam, out=out)  # 2^19 x 792 B = 415 MB > L2
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        fl = flops_per_qp(ev, N, it_mean) * Bs
        res["per_type"][ev] = {"qp_per_s": Bs / (ms * 1e-3), "ms": ms, "mean_iters": it_mean,
                               "fp64_tflops": fl / (ms * 1e-3) / 1e12,
                               "fp64_frac": fl / (ms * 1e-3) / 1e12 / fp64_peak,
                               "hbm_gbs": bytes_per_qp(N) * Bs / (ms * 1e-3) / 1e9}
        tot_ms += ms
        tot_flops += fl
        del lm, lr, gam, out
    res["value"] = 2 * Bs / (tot_ms * 1e-3)
    res["unit"] = UNIT
    res["fp64_tflops"] = tot_flops / (tot_ms * 1e-3) / 1e12
    res["fp64_frac"] = res["fp64_tflops"] / fp64_peak
    res["note"] = "inputs larger than L2 (415 MB per type); CUDA events around 5 back-to-back launches"
    return res


def closed_loop_leg(args, rank, world, dev):
    """BASELINE.json's second metric, "closed-loop price-step p50 latency", on configs[3]'s shape: S stations
    per GPU (500 + 500 EVs, 12 partitions, N_lo = N_bi = 24), device-resident closed loop
    (chargingstation.fleet), CUDA events around every step.  Stations are independent, so ranks hold whole
    stations (no data-path collective inside the price loop); the one exchange per step is the fleet's
    aggregate planned grid load, an all-reduce of N_bi doubles over NCCL."""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from run_fleet import fleet_consts, fleet_demand
    from chargingstation.fleet import ChargingStationFleet
    S, T = args.closed_loop_stations, args.closed_loop_steps
    consts = fleet_consts(T, 24, 24, 500, 12)
    demand = fleet_demand(consts, S, T, 24, seed=4 + rank)
    fleet = ChargingStationFleet(consts, S, demand=demand, seed=4 + rank, rng="device", chain=args.closed_loop_chain,
                                 device=dev.index)
    ms, agg_ms = [], []
    agg = torch.zeros(24, dtype=torch.float64, device=dev)
    for t in range(T):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        fleet.step()
        e1.record()
        agg.copy_(fleet.bi["u_g"].sum(dim=0))  # aggregate planned generation of this rank's stations
        if world > 1:
            dist.all_reduce(agg)
        e2.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e2))
        agg_ms.append(e1.elapsed_time(e2))
    t = torch.tensor(ms, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # a step ends when the slowest rank has finished it
    ms = t.cpu().numpy()
    solves = torch.tensor([float(fleet.qp_solves)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(solves)
    niter = torch.cat([fleet.log["niter_s"].flatten(), fleet.log["niter_l"].flatten()]).double()
    niter = niter[niter >= 0]
    steady = ms[min(8, T // 2):]  # the first steps start from the all-EVs-in-4-partitions initial condition
    return {"metric": "closed_loop_price_step_latency_ms", "p50_ms": float(np.median(ms)),
            "p95_ms": float(np.percentile(ms, 95)), "p50_ms_after_warmup": float(np.median(steady)),
            "stations_per_gpu": S, "stations_total": S * world, "steps": T, "chain": args.closed_loop_chain,
            "evs_total": 1000 * S * world, "qp_solves_in_price_loops": int(solves.item()),
            "qp_solves_per_s": float(solves.item() / (ms.sum() * 1e-3)),
            "price_iters_mean": float(niter.mean()), "price_iters_p95": float(np.percentile(niter.cpu().numpy(), 95)),
            "bimpc_not_converged": int((fleet.log["bimpc_status"] != 0).sum()),
            "aggregate_allreduce_wait_ms_p50": float(np.median(agg_ms)),  # includes waiting for the slowest rank
            "config": "BASELINE.json configs[3] shape (SURVEY.md 8d config 4): stations of 500+500 EVs, P=12, "
                      "N_lo=N_bi=24, demand profile shifted U{0..23} h and scaled U(0.22,0.26)/0.25 per station, "
                      "device RNG; the full size of configs[3] is 4096 stations x 96 steps (the default of this leg)"}


def sharded_leg(args, rank, world, dev):
    """BASELINE.json configs[2]: the 65,536-EV batch (2,048 groups x 32 EVs, half small-EV and half large-EV groups,
    N = 24, "linear-convex" prices, inputs as SURVEY.md 8d config 3, seed 3) sharded by EV index over the ranks, with
    the aggregate-load all-reduce (the [G, N] fp64 partial sums of price_solver.py:199-210) inside the price loop.
    STRONG scaling: the batch is fixed, every rank solves B / world EVs per iteration and all ranks run the
    replicated group phase.  The loop is pipelined (chargingstation/sharded.py): no host synchronisation inside."""
    import torch
    import torch.distributed as dist
    from chargingstation.lompc import LoMPCConstants
    from chargingstation.price_solver import PriceSolver
    from chargingstation.sharded import compute_optimal_prices_sharded, shard_groups
    N, G, EVS, MAX_IT = 24, 1024, 32, args.sharded_iters
    rng = np.random.default_rng(3)
    out = {"metric": "sharded_price_loop_ms", "n_gpus": world, "groups": 2 * G, "evs": 2 * G * EVS, "max_iter": MAX_IT,
           "allreduce_bytes_per_iter": G * N * 8, "per_type": {}}
    tot_ms, tot_qp, tot_ar_ms = 0.0, 0, 0.0
    for ev in ("small", "large"):
        delta, theta, y_max, w_max = EV_CONSTS[ev]
        off = (np.arange(G + 1) * EVS).astype(np.int64)
        y0 = 0.3 + 0.2 * rng.random(off[-1])               # charging_station.py:95-100, settings.py:27-28
        # groups = SoC partitions (charging_station.py:111-116 puts EVs of similar SoC together): sorted, so that
        # the tolerance sqrt(N) y0_rng + eps_tol (price_solver.py:184) is tight and the groups stay active -
        # with unsorted SoCs every group converges within 6 iterations and the leg would time its set-up
        y0.sort()
        w_ref = w_max * rng.random((G, N))                  # test_price_solver.py:34
        ps = PriceSolver(N, LoMPCConstants(delta, theta, y_max, w_max, ev), "linear-convex", device=dev.index)
        loc_off, loc_y0, (lo, hi) = shard_groups(off, y0, rank, world)
        call = lambda it: compute_optimal_prices_sharded(ps, loc_off, loc_y0, w_ref, np.zeros(G),  # noqa: E731
                                                         np.zeros((G, 3 * N)), max_iter=it)
        call(3)  # warm-up: allocations, NCCL channels
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        prices, stats = call(MAX_IT)
        e1.record()
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3
        ms = e0.elapsed_time(e1)
        # the collective alone: the same [G, N] buffer all-reduced back to back
        ar_ms = 0.0
        if world > 1:
            buf = torch.zeros((G, N), dtype=torch.float64, device=dev)
            for _ in range(5):
                dist.all_reduce(buf)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(50):
                dist.all_reduce(buf)
            a1.record()
            torch.cuda.synchronize()
            ar_ms = a0.elapsed_time(a1) / 50
        t = torch.tensor([ms, wall_ms, ar_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall_ms, ar_ms = (float(v) for v in t)
        it = np.asarray(stats["iter"])
        ran = int(stats["total_iters"])
        loops = min(ran + 1, MAX_IT)  # ev-phases executed
        qps = int(np.sum((np.minimum(it, MAX_IT - 1) + 1) * (EVS + 2)))
        out["exchange"] = ("NVLink peer memory (CUDA IPC regions, flags, rank-ordered sums inside the group phase)"
                           if getattr(ps, "_peer_state", None) is not None and world > 1 else
                           ("dist.all_reduce (NCCL)" if world > 1 else "none (one rank)"))
        out["per_type"][ev] = {"ms": ms, "wall_ms": wall_ms, "iterations": loops, "us_per_iteration": ms * 1e3 / loops,
                               # (a stand-alone dist.all_reduce of the same [G, N] buffer, for comparison: with the
                               # peer exchange the loop itself makes no NCCL call)
                               "allreduce_us": ar_ms * 1e3, "allreduce_share": ar_ms * loops / ms if ms > 0 else 0.0,
                               "converged_groups": int(np.sum(it < MAX_IT - 1)), "iters_mean": float(it.mean()),
                               "qp_solves": qps, "price_checksum": float(np.sum(prices)),
                               "local_evs": int(hi - lo)}
        if world == 1:
            # the same 1,024 groups through the device-resident loop a one-GPU caller gets from
            # PriceSolver.compute_optimal_prices_batch (one launch: a warp per group, parametric in gamma, DESIGN 4);
            # reported beside the phase-split loop above, which is the code every N runs and the leg's `ms`
            y0_all, zG = y0, np.zeros(G)
            ps.compute_optimal_prices_batch(off, y0_all, w_ref, zG, np.zeros((G, 3 * N)), max_iter=3)
            torch.cuda.synchronize()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            prices_r, stats_r = ps.compute_optimal_prices_batch(off, y0_all, w_ref, zG, np.zeros((G, 3 * N)),
                                                                max_iter=MAX_IT)
            r1.record()
            torch.cuda.synchronize()
            out["per_type"][ev]["resident_loop"] = {
                "ms": r0.elapsed_time(r1), "iters_equal": bool(np.array_equal(np.asarray(stats_r["iter"]), it)),
                "max_price_diff": float(np.max(np.abs(prices_r - prices))),
                "note": "price_solve_dev through the class API with host arrays (its small copies are inside)"}
        tot_ms += ms
        tot_qp += qps
        tot_ar_ms += ar_ms * loops
    if world > 1:
        out["allreduce_note"] = ("allreduce_us / allreduce_share: a stand-alone dist.all_reduce of the same [G, N] buffer "
                                 "timed after the loop, for comparison - with the peer-memory exchange the loop itself "
                                 "makes no NCCL call")
    out["ms"] = tot_ms
    out["qp_solves"] = tot_qp
    out["qp_per_s"] = tot_qp / (tot_ms * 1e-3)
    out["allreduce_share"] = tot_ar_ms / tot_ms if tot_ms > 0 else 0.0
    out["scaling"] = "strong (fixed 65,536-EV batch)"
    out["config"] = ("BASELINE.json configs[2] (SURVEY.md 8d config 3) as a price loop: 1,024 small-EV + 1,024 large-EV "
                     "groups x 32 EVs, N=24, w_ref = w_max U(0,1), y0 = U(0.3,0.5) sorted into SoC partitions, seed 3, EVs "
                     "block-sharded by index (groups straddle ranks), one all-reduce of [G,N] fp64 per price iteration, "
                     "loop capped at max_iter")
    return out


def cpu_baseline_leg(args):
    work = draw_workload(args.batch, N_HORIZON, 2)
    used = cpu_pass(work, N_HORIZON)  # warm-up
    t0 = time.perf_counter()
    cpu_pass(work, N_HORIZON)
    one = time.perf_counter() - t0
    reps = max(1, min(200, int(3.0 / max(one, 1e-9))))
    t0 = time.perf_counter()
    for _ in range(reps):
        cpu_pass(work, N_HORIZON)
    dt = (time.perf_counter() - t0) / reps
    return {"value": args.batch / dt, "unit": UNIT, "cores": used, "kind": "port",
            "sample": f"{reps} passes over the same {args.batch}-QP workload (oracle/lompc_oracle.c, "
                      f"Clarabel-style IPM, tol 1e-8, OpenMP on {used} threads, {reps * dt:.1f} s wall)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="QPs per GPU per step (configs[1]: 1024)")
    ap.add_argument("--no-saturated", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--closed-loop-stations", type=int, default=4096,
                    help="stations per GPU of the closed-loop latency leg (0 = skip; configs[3]: 4096)")
    ap.add_argument("--closed-loop-steps", type=int, default=96, help="closed-loop steps (configs[3]: 96)")
    ap.add_argument("--closed-loop-chain", default="reference", choices=["reference", "partition"])
    ap.add_argument("--sharded-iters", type=int, default=200,
                    help="price iterations of the configs[2] leg (65,536 EVs sharded over the ranks; 0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the CUDA path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
