"""Device-resident closed loop over S charging stations (BASELINE.json configs[3]: "full
bilevel price loop over 4,096 stations, closed-loop 96 steps").  Not in the reference, which
simulates ONE station with Python loops over partitions and EVs
(charging_station.py:156-370); every station here follows exactly that loop:

    partition the EVs by SoC      charging_station.py:111-116   fleet_partition_dev
    group statistics              price_solver.py:66-77          price_group_stats_dev
    BiMPC parameters + solve      charging_station.py:187-227    fleet_bimpc_params_dev, bimpc_solve_batch_dev
    price loop per partition      charging_station.py:265-305    price_solve_chain_dev / price_solve_dev
    EV responses                  charging_station.py:307-327    price_w0_price0_dev
    plant update                  charging_station.py:329-365    fleet_apply_charge_dev, fleet_battery_dev

State (SoCs, partition indices, battery, warm-start prices) stays in HBM between steps; the
host only sequences kernel launches and reads P+1 slice sizes per EV type and step.

``chain="reference"`` keeps the reference's warm-start chain: the PriceSolver of an EV type
is shared by its P partitions, so partition p starts from the prices of the last non-empty
partition solved before it (``prev_prices``, price_solver.py:56,104,166) - here
``price_solve_chain_dev``: one CTA per station walks its P partitions in that order, stations
never wait for each other.
``chain="partition"`` solves all P*S groups of a type in ONE device loop, each group
warm-started from its own prices of the previous step (different iterates, same fixed-point
conditions; P times fewer sequential loops).

``rng="numpy"`` draws arrivals on the host from ``np.random.RandomState(seed + s)`` in the
reference's order (parity with ``ChargingStation`` after ``np.random.seed(seed + s)``);
``rng="device"`` uses the counter-based generator of ``fleet_apply_charge_dev``."""
from __future__ import annotations

import ctypes as C

import numpy as np

from chargingstation import _native
from chargingstation.bimpc import BiMPC
from chargingstation.charging_station import ChargingStationConstants, partition_edges
from chargingstation.price_solver import PriceSolver, tol_type_max
from chargingstation.settings import (MAX_INITIAL_SOC, MAX_PRICE_SOLVER_ITERATIONS, MIN_FULL_CHARGE_FRACTION,
                                      MIN_INITIAL_SOC, PRICE_SOLVER_TOL_TYPE)


class ChargingStationFleet:
    def __init__(self, consts: ChargingStationConstants, nstations: int, demand: np.ndarray | None = None,
                 seed: int = 0, rng: str = "device", chain: str = "reference", device: int = 0,
                 max_price_iter: int = MAX_PRICE_SOLVER_ITERATIONS, tol_type: str | None = None) -> None:
        """
        consts:     the station's constants (every station shares them); ``consts.demand`` is
                    used for all stations unless ``demand`` [S, >= Tf + N_bi + 1] is given.
        tol_type:   convergence test of the price loops, "avg" or "max" (price_solver.py:121-128);
                    None = PRICE_SOLVER_TOL_TYPE.
        """
        import torch
        assert rng in ("device", "numpy") and chain in ("reference", "partition")
        assert consts.simulation_length >= 1
        assert (consts.horizon_bimpc >= consts.horizon_lompc) and (consts.horizon_lompc >= 1)
        assert consts.nEVs_per_EV_type >= 1 and consts.npartitions >= 1 and nstations >= 1
        self.torch = torch
        self.dev = torch.device("cuda", device)
        self.device = int(device)
        self.consts = consts
        self.S, self.M, self.P = int(nstations), consts.nEVs_per_EV_type, consts.npartitions
        self.Tf, self.N_bi, self.N_lo = consts.simulation_length, consts.horizon_bimpc, consts.horizon_lompc
        self.r = 2 * self.N_lo if consts.price_type == "linear" else 3 * self.N_lo
        self.rng_mode, self.chain, self.seed = rng, chain, int(seed)
        self.max_price_iter = int(max_price_iter)
        self.tol_type = tol_type
        tol_type_max(tol_type, PRICE_SOLVER_TOL_TYPE)  # rejects anything but "avg", "max" and None here
        S, M, P, N_lo, N_bi = self.S, self.M, self.P, self.N_lo, self.N_bi
        if demand is None:
            demand = np.broadcast_to(consts.demand, (S, consts.demand.shape[0]))
        demand = np.ascontiguousarray(demand, dtype=np.float64)
        assert demand.shape[0] == S and demand.shape[1] >= self.Tf + N_bi + 1
        self.profile_len = demand.shape[1]
        self._lib = _native.load()
        self.bimpc = BiMPC(N_bi, P, consts.bimpc_consts, consts.small_EV_consts, consts.large_EV_consts, device=device)
        self.ev = {"s": consts.small_EV_consts, "l": consts.large_EV_consts}
        self.solver = {k: PriceSolver(N_lo, self.ev[k], consts.price_type, device=device) for k in ("s", "l")}
        self.Bcap = (self.ev["s"].theta + self.ev["l"].theta) * M
        f64, i32 = torch.float64, torch.int32
        z = lambda *shape, dtype=f64: torch.zeros(shape, dtype=dtype, device=self.dev)  # noqa: E731
        # ---- state
        if rng == "numpy":
            self._rs = [np.random.RandomState(self.seed + s) for s in range(S)]
            y0 = {"s": np.empty((S, M)), "l": np.empty((S, M))}
            for s in range(S):  # charging_station.py:95-100: small first, then large
                for k in ("s", "l"):
                    y0[k][s] = MIN_INITIAL_SOC + (MAX_INITIAL_SOC - MIN_INITIAL_SOC) * self._rs[s].random_sample((M,))
        else:
            g = np.random.default_rng(self.seed)
            y0 = {k: MIN_INITIAL_SOC + (MAX_INITIAL_SOC - MIN_INITIAL_SOC) * g.random((S, M)) for k in ("s", "l")}
        self.y = {k: torch.from_numpy(y0[k]).to(self.dev) for k in ("s", "l")}
        self.idx = {k: z(S, M, dtype=i32) for k in ("s", "l")}
        self.x = z(S)
        self.ncharged = {k: z(S, dtype=i32) for k in ("s", "l")}
        self.prev = {k: z(S, 3 * N_lo) for k in ("s", "l")}          # reference chain: one warm start per station
        self.prices = {k: z(P * S, 3 * N_lo) for k in ("s", "l")}    # prices of every group (partition-major)
        self.t = 0
        self.demand = torch.from_numpy(demand).to(self.dev)
        self.edges = {k: torch.from_numpy(partition_edges(MIN_INITIAL_SOC, self.ev[k].y_max, P)).to(self.dev)
                      for k in ("s", "l")}
        # ---- per-step work buffers
        G, B = P * S, S * M
        self.w = {}
        for k in ("s", "l"):
            self.w[k] = dict(counts=z(G, dtype=i32), off=z(G + 1, dtype=i32), reb=z(P, S + 1, dtype=i32),
                             ysort=z(B), perm=z(B, dtype=i32), gamma=z(B), y0_rng=z(G), gamma_sc=z(G), gamma_sm=z(G),
                             w_ref=z(G, N_lo), iters=z(G, dtype=i32), pre=z(G), post=z(G), red=z(G), w0=z(B),
                             price0=z(G), w_sum=z(S), w_mean=z(G), mask=z(S, M, dtype=i32))
        self.bi = dict(Mp_s=z(S, P), Mp_l=z(S, P), beta_s=z(S, P), beta_l=z(S, P), gamma_s=z(S, P), gamma_l=z(S, P),
                       x0=z(S), demand=z(S, N_bi), w_hat_s=z(S, P, N_bi), w_hat_l=z(S, P, N_bi), u_g=z(S, N_bi),
                       status=z(S, dtype=i32), iters=z(S, dtype=i32), obj=z(S))
        self.lmbd_r0 = z(G)
        # ---- logs (reference schema, one leading station axis; filled step by step on the device)
        Tf = self.Tf
        self.inexact_steps = 0  # steps that raised the warning below
        self.log = {"u_g": z(Tf, S), "x": z(Tf, S), "bimpc_iters": z(Tf, S, dtype=i32), "bimpc_status": z(Tf, S, dtype=i32)}
        for k in ("s", "l"):
            for name in ("w", "w_hat", "beta", "gamma_m", "avg_price", "price_red"):
                self.log[f"{name}_{k}"] = z(Tf, P, S)
            self.log[f"niter_{k}"] = z(Tf, P, S, dtype=i32)
            self.log[f"Mp_{k}"] = z(Tf, P, S, dtype=i32)
        self.ncharged_logged = {k: z(S, dtype=i32) for k in ("s", "l")}
        self.sort_stations = True
        self.order = {"s": None, "l": None}  # launch order of the chain kernel (longest chains of the last step first)
        self.price_loop_iters = []  # per step: total device-loop iterations of the price loops
        self.qp_solves = 0   # LoMPC QPs solved inside the price loops so far
        self.cycles = [0, 0, 0, 0, 0]  # SM cycles (summed over groups) in the LoMPC passes / the price steps; K1
        # iterations summed over the solves; warp passes without a K1 iteration; warp passes
        from concurrent.futures import ThreadPoolExecutor
        self._pool = ThreadPoolExecutor(max_workers=2)
        self.streams = {k: torch.cuda.Stream(self.dev) for k in ("s", "l")}
        self._lock = __import__("threading").Lock()
        self.profile = False  # True: record CUDA events at the phase boundaries of every step
        self.phase_ms = []    # per step: {phase: ms}

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return self.torch.cuda.current_stream(self.dev).cuda_stream

    def _ck(self, rc):
        _native.raise_for(rc)

    def _account(self, h) -> None:
        with self._lock:
            self.qp_solves += self._lib.price_last_qp_solves(h)
            self.cycles[0] += self._lib.price_last_cycles(h, 0)
            self.cycles[1] += self._lib.price_last_cycles(h, 1)
            for i in (2, 3, 4):
                self.cycles[i] += self._lib.price_last_cycles(h, i)

    # ------------------------------------------------------------------ one closed-loop step
    def step(self) -> None:
        torch, lib, st = self.torch, self._lib, self._stream()
        S, M, P, N_lo, N_bi, t = self.S, self.M, self.P, self.N_lo, self.N_bi, self.t
        G, B = P * S, S * M
        lmbd_r = 0.0  # charging_station.py:162
        tol_max = tol_type_max(self.tol_type, PRICE_SOLVER_TOL_TYPE)
        marks = []

        def mark(name):
            if self.profile:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((name, e))

        mark("start")
        # ---- partitions, group statistics
        for k in ("s", "l"):
            w, h = self.w[k], self.solver[k]._h
            self._ck(lib.fleet_partition_dev(self.device, S, M, P, self.edges[k].data_ptr(), self.y[k].data_ptr(),
                                             self.idx[k].data_ptr(), w["counts"].data_ptr(), w["off"].data_ptr(),
                                             w["reb"].data_ptr(), w["ysort"].data_ptr(), w["perm"].data_ptr(), st))
            self._ck(lib.price_group_stats_dev(h, G, B, w["off"].data_ptr(), w["ysort"].data_ptr(),
                                               w["gamma"].data_ptr(), w["y0_rng"].data_ptr(),
                                               w["gamma_sc"].data_ptr(), w["gamma_sm"].data_ptr(), st))
        mark("partition+stats")
        # ---- upper level
        ws, wl, bi = self.w["s"], self.w["l"], self.bi
        self._ck(lib.fleet_bimpc_params_dev(
            self.device, S, P, N_bi, N_lo, float(self.Bcap), float(self.solver["s"].eps_tol), lmbd_r,
            float(self.ev["s"].delta), float(self.ev["l"].delta), ws["counts"].data_ptr(), wl["counts"].data_ptr(),
            ws["y0_rng"].data_ptr(), wl["y0_rng"].data_ptr(), ws["gamma_sm"].data_ptr(), wl["gamma_sm"].data_ptr(),
            self.x.data_ptr(), self.demand.data_ptr(), self.profile_len, t, bi["Mp_s"].data_ptr(),
            bi["Mp_l"].data_ptr(), bi["beta_s"].data_ptr(), bi["beta_l"].data_ptr(), bi["gamma_s"].data_ptr(),
            bi["gamma_l"].data_ptr(), bi["x0"].data_ptr(), bi["demand"].data_ptr(), st))
        self._ck(lib.bimpc_solve_batch_dev(
            self.bimpc._h, S, bi["Mp_s"].data_ptr(), bi["Mp_l"].data_ptr(), bi["beta_s"].data_ptr(),
            bi["beta_l"].data_ptr(), bi["gamma_s"].data_ptr(), bi["gamma_l"].data_ptr(), bi["x0"].data_ptr(),
            bi["demand"].data_ptr(), bi["w_hat_s"].data_ptr(), bi["w_hat_l"].data_ptr(), bi["u_g"].data_ptr(),
            bi["status"].data_ptr(), bi["iters"].data_ptr(), bi["obj"].data_ptr(), st))
        for k in ("s", "l"):
            self._ck(lib.fleet_wref_dev(self.device, S, P, N_bi, N_lo, bi["w_hat_" + k].data_ptr(),
                                        self.w[k]["w_ref"].data_ptr(), st))
        mark("bimpc")
        # ---- price loops: the two EV types are independent chains (separate PriceSolver objects in the
        # reference, charging_station.py:58-59) -> one host thread and one CUDA stream per type
        main = torch.cuda.current_stream(self.dev)
        ready = torch.cuda.Event()
        ready.record(main)

        def run_type(k):
            w, h = self.w[k], self.solver[k]._h
            stream = self.streams[k]
            stream.wait_event(ready)
            sp = stream.cuda_stream
            total = C.c_int32(0)
            iters_sum = 0
            with torch.cuda.stream(stream):
                if self.chain == "reference":
                    # one CTA per station walks its P partitions in order (price_station_chain_kernel)
                    self._ck(lib.price_solve_chain_dev(
                        h, S, P, B, w["off"].data_ptr(), w["ysort"].data_ptr(), w["w_ref"].data_ptr(),
                        self.lmbd_r0.data_ptr(), self.r, self.max_price_iter, tol_max, float(self.solver[k].eps_reg),
                        float(self.solver[k].eps_tol), self.prev[k].data_ptr(), self.prices[k].data_ptr(),
                        w["iters"].data_ptr(), w["pre"].data_ptr(), w["post"].data_ptr(),
                        self.order[k].data_ptr() if self.order[k] is not None else None, C.byref(total), sp))
                    # next step's launch order: stations with the longest chains first
                    if self.sort_stations:
                        self.order[k] = torch.argsort(w["iters"].view(P, S).clamp(min=0).sum(dim=0), descending=True,
                                                      stable=True).to(torch.int32)
                    iters_sum += total.value
                    self._account(h)
                    self._ck(lib.fleet_keep_prices_dev(
                        self.device, G, 3 * N_lo, w["counts"].data_ptr(), self.prices[k].data_ptr(),
                        self.prices[k].data_ptr(), w["pre"].data_ptr(), w["post"].data_ptr(), w["red"].data_ptr(), sp))
                else:
                    self._ck(lib.price_solve_dev(
                        h, G, B, w["off"].data_ptr(), w["ysort"].data_ptr(), w["w_ref"].data_ptr(),
                        self.lmbd_r0.data_ptr(), self.r, self.max_price_iter, tol_max, float(self.solver[k].eps_reg),
                        float(self.solver[k].eps_tol), self.prices[k].data_ptr(), w["iters"].data_ptr(),
                        w["pre"].data_ptr(), w["post"].data_ptr(), None, None, None, 0, C.byref(total), sp))
                    iters_sum += total.value
                    self._account(h)
                    # price reduction / NaN for empty groups
                    self._ck(lib.fleet_keep_prices_dev(
                        self.device, G, 3 * N_lo, w["counts"].data_ptr(), self.prices[k].data_ptr(),
                        self.prices[k].data_ptr(), w["pre"].data_ptr(), w["post"].data_ptr(), w["red"].data_ptr(), sp))
            done = torch.cuda.Event()
            done.record(stream)
            return iters_sum, done

        results = list(self._pool.map(run_type, ("s", "l")))
        loop_iters = 0
        for iters_sum, done in results:
            loop_iters += iters_sum
            main.wait_event(done)
        self.price_loop_iters.append(loop_iters)
        mark("price_loops")
        # the price loops above already synchronised with the host, so these reads cost one small copy each
        n_bad = int(torch.count_nonzero(bi["status"]))
        n_cap = sum(int(lib.price_last_cycles(self.solver[k]._h, w)) for k in ("s", "l") for w in (6, 7))
        if n_bad or n_cap:
            import warnings
            warnings.warn(f"fleet step {t}: {n_bad} station(s) with an unsolved BiMPC (status in logs()['bimpc_status']), "
                          f"{n_cap} price step(s) / LoMPC solve(s) stopped at their iteration cap", RuntimeWarning,
                          stacklevel=2)
        self.inexact_steps += bool(n_bad or n_cap)
        # ---- EV responses at the final prices
        for k in ("s", "l"):
            w, h = self.w[k], self.solver[k]._h
            self._ck(lib.price_w0_price0_dev(h, G, B, w["off"].data_ptr(), w["gamma"].data_ptr(),
                                             self.prices[k].data_ptr(), self.lmbd_r0.data_ptr(), w["w0"].data_ptr(),
                                             w["price0"].data_ptr(), st))
        mark("ev_response")
        # ---- logs of this step (charging_station.py:371-433; x is logged before the update)
        L = self.log
        L["u_g"][t].copy_(bi["u_g"][:, 0])
        L["x"][t].copy_(self.x)
        L["bimpc_iters"][t].copy_(bi["iters"])
        L["bimpc_status"][t].copy_(bi["status"])
        # the reference logs the departure counters BEFORE this step's plant update (:399-400)
        self.ncharged_logged = {k: self.ncharged[k].clone() for k in ("s", "l")}
        # ---- plant
        for ti, k in enumerate(("s", "l")):
            w = self.w[k]
            seed = self.seed if self.rng_mode == "device" else -1
            self._ck(lib.fleet_apply_charge_dev(
                self.device, S, M, P, float(MIN_FULL_CHARGE_FRACTION * self.ev[k].y_max), float(MIN_INITIAL_SOC),
                float(MAX_INITIAL_SOC), seed, ti, t, w["off"].data_ptr(), w["perm"].data_ptr(), w["w0"].data_ptr(),
                self.y[k].data_ptr(), w["mask"].data_ptr(), w["w_sum"].data_ptr(), w["w_mean"].data_ptr(),
                self.ncharged[k].data_ptr(), st))
        if self.rng_mode == "numpy":
            self._host_arrivals()
        self._ck(lib.fleet_battery_dev(self.device, S, N_bi, float(self.ev["s"].theta), float(self.ev["l"].theta),
                                       float(self.Bcap), bi["u_g"].data_ptr(), ws["w_sum"].data_ptr(),
                                       wl["w_sum"].data_ptr(), self.demand.data_ptr(), self.profile_len, t,
                                       self.x.data_ptr(), st))
        for k in ("s", "l"):
            w = self.w[k]
            L[f"w_{k}"][t].copy_(w["w_mean"].view(P, S))
            L[f"w_hat_{k}"][t].copy_(bi["w_hat_" + k][:, :, 0].t())
            L[f"beta_{k}"][t].copy_(bi["beta_" + k].t())
            L[f"gamma_m_{k}"][t].copy_(bi["gamma_" + k].t())
            L[f"avg_price_{k}"][t].copy_(w["price0"].view(P, S))
            L[f"price_red_{k}"][t].copy_(w["red"].view(P, S))
            L[f"niter_{k}"][t].copy_(w["iters"].view(P, S))
            L[f"Mp_{k}"][t].copy_(w["counts"].view(P, S))
        mark("plant+logs")
        if self.profile:
            torch.cuda.synchronize(self.dev)
            self.phase_ms.append({n1: e0.elapsed_time(e1) for (_, e0), (n1, e1) in zip(marks[:-1], marks[1:])})
        self.t += 1

    def _host_arrivals(self) -> None:
        """Replacement SoCs from the per-station np.random streams, small EVs first
        (charging_station.py:333-346)."""
        torch = self.torch
        masks = {k: self.w[k]["mask"].cpu().numpy().astype(bool) for k in ("s", "l")}
        ys = {k: self.y[k].cpu().numpy() for k in ("s", "l")}
        for s in range(self.S):
            for k in ("s", "l"):
                n = int(masks[k][s].sum())
                ys[k][s, masks[k][s]] = MIN_INITIAL_SOC + (MAX_INITIAL_SOC - MIN_INITIAL_SOC) * \
                    self._rs[s].random_sample((n,))
        for k in ("s", "l"):
            self.y[k].copy_(torch.from_numpy(ys[k]))

    def simulate(self, steps: int | None = None) -> dict:
        for _ in range(self.Tf - self.t if steps is None else steps):
            self.step()
        return self.log

    # ------------------------------------------------------------------ logs in the reference schema
    def station_logs(self, s: int) -> dict:
        """``ChargingStation.logs`` of station s (charging_station.py:118-149)."""
        L = {k: v[:, ..., s].cpu().numpy() if v.dim() == 3 else v[:, s].cpu().numpy() for k, v in self.log.items()}
        T = lambda a: np.ascontiguousarray(a.T)  # noqa: E731  [Tf, P] -> [P, Tf]
        return {
            "constants": self.consts,
            "inputs": {"w_s": T(L["w_s"]), "w_l": T(L["w_l"]), "w_hat_s": T(L["w_hat_s"]), "w_hat_l": T(L["w_hat_l"]),
                       "u_g": L["u_g"]},
            "states": {"x": L["x"]},
            "bounds": {"beta_s": T(L["beta_s"]), "beta_l": T(L["beta_l"])},
            "statistics": {"ncharged_s": int(self.ncharged_logged["s"][s]),
                           "ncharged_l": int(self.ncharged_logged["l"][s]),
                           "gamma_sm": T(L["gamma_m_s"]), "gamma_lm": T(L["gamma_m_l"]),
                           "niter_s": T(L["niter_s"]).astype(int), "niter_l": T(L["niter_l"]).astype(int),
                           "Mp_s": T(L["Mp_s"]).astype(int), "Mp_l": T(L["Mp_l"]).astype(int)},
            "prices": {"lmbd_r": np.zeros(self.Tf), "avg_price_s": T(L["avg_price_s"]),
                       "avg_price_l": T(L["avg_price_l"]), "price_red_s": T(L["price_red_s"]),
                       "price_red_l": T(L["price_red_l"])},
        }
