"""The "max" tolerance type of the price loop (settings.PRICE_SOLVER_TOL_TYPE, price_solver.py:121-128: the loop stops
when the largest error of a single EV is within the tolerance) on every loop that serves it: the parametric
one-warp-per-group loop (loop modes 0 and 2), the thread-per-EV loop (mode 3, N = 12 and 24) and the phase-split loop
(mode 1), against oracle/price_oracle.py run with the same tolerance type.

The parametric loop solves only some EVs of a group and interpolates the others, so its w_err_max is the maximum over
the EVs it solved and over the first and last EV of every interpolated stretch (the error is convex in gamma where the
solution is affine).  The first test checks that maximum directly, through the price_debug_record_errors hook, at
given prices; the others check whole loops."""
import ctypes as C

import numpy as np
import pytest

from oracle import lompc_oracle as orc
from oracle import price_oracle as po

pytestmark = pytest.mark.gpu


def _consts(ev):
    from chargingstation.lompc import LoMPCConstants
    o = orc.small_ev_consts() if ev == "small" else orc.large_ev_consts()
    return o, LoMPCConstants(o.delta, o.theta, o.y_max, o.w_max, o.ev_type)


@pytest.fixture
def oracle_max(monkeypatch):
    """The oracle loop with the "max" tolerance type (it reads its module constant at every test)."""
    monkeypatch.setattr(po, "PRICE_SOLVER_TOL_TYPE", "max")


def _close(a, b):
    """Prices within the bars of the other loop tests: 1e-6 relative where |price| <= 1e3; above, where the
    closed-form regulariser divides by a response of rounding-error size, 1e-3 of the price."""
    small = np.abs(b) <= 1e3
    err = np.abs(a - b)
    return (np.max(err[small], initial=0.0) <= 1e-6 * max(1.0, np.max(np.abs(b[small]), initial=0.0))
            and np.all(err[~small] <= 1e-3 * np.abs(b[~small])))


def _groups(rng, G):
    counts = np.array([1, 2, 3, 9, 33, 70] + list(rng.integers(4, 60, G - 6)))
    spans = np.concatenate([[0.0, 0.02, 0.45, 0.1, 0.3, 0.45], rng.uniform(0.0, 0.45, G - 6)])
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    y0 = np.concatenate([0.3 + sp * rng.random(n) for n, sp in zip(counts, spans)])
    return off, y0


@pytest.mark.parametrize("N", [12, 24, 48, 96])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_parametric_max_error_at_given_prices(ev, N):
    """Teacher-forced: with max_iter = 1 and a group's prices as its warm start, the w_err_max the parametric loop
    tests (price_solver.py:196-214) equals the oracle's maximum over every EV, to 1e-9 relative; also with a pivot pool
    of 4 slots, where many EVs are solved one by one.  About 40 groups per case, prices drawn per group from theta * U
    (many critical regions per group) and 0.05 theta * U (the closed loop's scale).  Three kinds of w_ref: random; the
    chord midpoint c of the extreme EVs' solutions; and c moved away from the solution w_j of the EV nearest gamma_sc,
    along the part of w_j - c that is A-bar-orthogonal to the chord.  The last one puts the largest error inside the
    group, next to the virtual EV, wherever the solution path bends there - the EVs whose error only the interpolated
    ends of an interval (not the solved pivots) can report."""
    import torch
    from chargingstation import _native
    from chargingstation.price_solver import PriceSolver
    o, c = _consts(ev)
    lib = _native.load()
    rng = np.random.default_rng(4000 + N + (ev == "large"))
    G = 40
    off, y0 = _groups(rng, G)
    lr = np.where(np.arange(G) % 4 == 3, float(N), 0.0)
    rec = [torch.zeros(G, dtype=torch.float64, device="cuda:0") for _ in range(2)]
    inside, near_sc, checked = 0, 0, 0
    assert lib.price_debug_record_errors(rec[0].data_ptr(), None) != 0  # both arrays or neither
    for price_type in ("linear-convex", "linear"):
        ps = PriceSolver(N, c, price_type)
        ora = po.PriceOracle(N, o, price_type, fast=True)
        for scale in (1.0, 0.05):
            lam = np.zeros((G, 3 * N))
            lam[:, : ps.r] = scale * o.theta * rng.random((G, ps.r))
            for kind in ("random", "chord", "bend"):
                w_ref = o.w_max * 0.6 * rng.random((G, N))
                o_max, o_avg = np.zeros(G), np.zeros(G)
                for g in range(G):
                    yg = y0[off[g]: off[g + 1]]
                    ora.set_charge_levels(yg)
                    gam = np.sort(o.y_max - yg)
                    w_all = ora._solve_evs(lam[g], lr[g], gam)  # EVs by ascending gamma
                    A_bar, _ = ora._metric(lr[g])
                    if kind != "random":
                        w_ref[g] = _chord_ref(w_all, gam, ora.gamma_sc, A_bar, bend=kind == "bend")
                    o_max[g], _, o_avg[g], _ = ora.get_w_err(lam[g], lr[g], w_ref[g], A_bar)
                    d = w_all - w_ref[g]
                    err = np.sqrt(np.einsum("ij,jk,ik->i", d, A_bar, d))
                    j = int(np.argmax(err))
                    if len(yg) > 2 and err[j] > max(err[0], err[-1]) * (1 + 1e-9) + 1e-12:
                        inside += 1
                        vpos = int(np.searchsorted(gam, ora.gamma_sc, side="right"))
                        near_sc += j in (vpos - 1, vpos)
                for pool in (32, 4):
                    assert lib.price_debug_pivot_pool(pool) == 0
                    assert lib.price_debug_record_errors(rec[0].data_ptr(), rec[1].data_ptr()) == 0
                    try:
                        for r in rec:
                            r.fill_(-1.0)
                        _, st = ps.compute_optimal_prices_batch(off, y0, w_ref, lr, lam, max_iter=1, tol_type="max")
                    finally:
                        assert lib.price_debug_record_errors(None, None) == 0
                        assert lib.price_debug_pivot_pool(32) == 0
                    d_max, d_avg = rec[0].cpu().numpy(), rec[1].cpu().numpy()
                    case = (price_type, scale, kind, pool)
                    bad = np.abs(d_max - o_max) > 1e-9 * np.maximum(1.0, o_max)
                    assert not bad.any(), (case, np.flatnonzero(bad), d_max[bad], o_max[bad])
                    assert np.all(np.abs(d_avg - o_avg) <= 1e-9 * np.maximum(1.0, o_avg)), case
                    checked += G
    print(f"[N = {N}, {ev}] {checked} group errors checked; oracle argmax strictly inside the group in {inside} of "
          f"{checked // 2} group instances, {near_sc} of them next to gamma_sc")
    assert inside > 0 and near_sc > 0


def _chord_ref(w_all, gam, gamma_sc, A_bar, bend):
    """The chord midpoint c of the extreme EVs' solutions; with ``bend``, c - t u, where u is the part of w_j - c
    (w_j: the EV nearest gamma_sc) A-bar-orthogonal to the chord and t = 2 |h|^2 / |u|^2 (h: the half chord), capped at
    1e3: then |w_j - w_ref| exceeds the extreme EVs' errors whenever u is not of rounding size."""
    c = 0.5 * (w_all[0] + w_all[-1])
    if not bend:
        return c
    h = 0.5 * (w_all[-1] - w_all[0])
    d = w_all[int(np.argmin(np.abs(gam - gamma_sc)))] - c
    hh = h @ A_bar @ h
    u = d - (d @ A_bar @ h) / hh * h if hh > 0 else d
    uu = u @ A_bar @ u
    return c - (min(1e3, 2 * hh / uu) if uu > 0 else 0.0) * u


def _loop_groups(N, ev):
    rng = np.random.default_rng(500 + N + (ev == "large"))
    counts = np.array([1, 2, 9, 33, 47, 70])
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    spans = [0.0, 0.02, 0.05, 0.3, 0.04, 0.45]
    y0 = np.concatenate([0.3 + sp * rng.random(n) for n, sp in zip(counts, spans)])
    return rng, off, y0


@pytest.mark.parametrize("N", [12, 24, 48, 96])
@pytest.mark.parametrize("ev", ["small", "large"])
@pytest.mark.parametrize("price_type,lmbd_r", [("linear-convex", 0.0), ("linear", 0.0), ("linear-convex", 1.0)],
                         ids=["linear-convex", "linear", "linear-convex-lr"])
def test_max_tolerance_loops_against_oracle(ev, N, price_type, lmbd_r, oracle_max):
    """Whole loops (price_solver.py:79-174) with tol_type="max": the parametric loop (automatic mode and mode 2), the
    thread-per-EV loop (mode 3, N = 12 and 24) and the phase-split loop (mode 1).  Iteration counts equal to each
    other and to the oracle's, prices and price_after_reg within the bars of the "avg" tests."""
    from chargingstation import settings
    from chargingstation.price_solver import PriceSolver
    settings.PRINT_LEVEL = 0
    o, c = _consts(ev)
    rng, off, y0 = _loop_groups(N, ev)
    G = len(off) - 1
    w_ref = o.w_max * rng.random((G, N)) * 0.6
    lr = np.full(G, lmbd_r * N)
    modes = (0, 2, 3, 1) if N <= 24 else (0, 2, 1)
    out = {}
    for mode in modes:
        ps = PriceSolver(N, c, price_type)
        ps.set_loop_mode(mode)
        prices, st = ps.compute_optimal_prices_batch(off, y0, w_ref, lr, np.zeros((G, 3 * N)), max_iter=60,
                                                     tol_type="max")
        out[mode] = (prices, st["iter"].copy(), st["price_after_reg"].copy())
        if mode == 2:
            assert ps.last_nnqp_cap_hits() == 0
            assert int(ps._lib.price_last_qp_solves(ps._h)) < int(np.sum((np.diff(off) + 1) * (st["iter"] + 1)))
    for mode in modes:
        assert np.array_equal(out[mode][1], out[2][1]), (mode, out[mode][1], out[2][1])
    for g in range(G):
        ora = po.PriceOracle(N, o, price_type, fast=True)
        ora.set_charge_levels(y0[off[g]: off[g + 1]])
        lam_o, st_o = ora.compute_optimal_prices(w_ref[g], lr[g], max_iter=60)
        assert out[2][1][g] == st_o["iter"], (g, out[2][1][g], st_o["iter"])
        for mode in modes:
            assert _close(out[mode][0][g], lam_o), (mode, g)
            assert abs(out[mode][2][g] - st_o["price_after_reg"]) <= 1e-6 * max(1.0, abs(st_o["price_after_reg"])), (mode, g)
    # "avg" and "max" are different tests: with these inputs they stop at different iterations somewhere
    ps = PriceSolver(N, c, price_type)
    _, st_avg = ps.compute_optimal_prices_batch(off, y0, w_ref, lr, np.zeros((G, 3 * N)), max_iter=60, tol_type="avg")
    assert not np.array_equal(st_avg["iter"], out[2][1])


def test_tol_type_is_validated():
    from chargingstation.price_solver import PriceSolver
    o, c = _consts("small")
    ps = PriceSolver(12, c, "linear-convex")
    off = np.array([0, 3], dtype=np.int32)
    args = (off, np.array([0.3, 0.4, 0.5]), np.zeros((1, 12)), np.zeros(1), np.zeros((1, 36)))
    for bad in ("Max", "mean", ""):
        with pytest.raises(ValueError):
            ps.compute_optimal_prices_batch(*args, tol_type=bad)
    ps.compute_optimal_prices_batch(*args, tol_type="avg", max_iter=2)


@pytest.mark.parametrize("ev", ["small", "large"])
def test_parametric_max_loop_degenerate_groups(ev, oracle_max):
    """The six groups of test_parametric_loop_degenerate_groups under "max": SoCs equal to the last bit (gamma_sc
    rounds onto the largest gamma), identical SoCs, two values, one EV, two EVs, a wide group.  Same iteration counts as
    the thread-per-EV loop and the oracle, prices within the bars."""
    from chargingstation.price_solver import PriceSolver
    o, c = _consts(ev)
    N = 12
    rng = np.random.default_rng(78)
    base = 0.7627601805992867
    cases = {
        "equal_to_the_last_bit": np.array([base, np.nextafter(base, 1.0), np.nextafter(np.nextafter(base, 1.0), 1.0)] * 4),
        "identical": np.full(9, 0.41),
        "two_values": np.array([0.35] * 5 + [0.39] * 4),
        "one_ev": np.array([0.52]),
        "two_evs": np.array([0.31, 0.33]),
        "wide": 0.3 + 0.3 * rng.random(37),
    }
    for name, y0 in cases.items():
        w_ref = o.w_max * rng.random(N) * 0.6
        ora = po.PriceOracle(N, o, "linear-convex", fast=True)
        ora.set_charge_levels(y0)
        lam_o, st_o = ora.compute_optimal_prices(w_ref, 0.0, max_iter=300)
        out = {}
        for mode in (3, 2):
            ps = PriceSolver(N, c, "linear-convex")
            ps.set_loop_mode(mode)
            off = np.array([0, len(y0)], dtype=np.int32)
            prices, st = ps.compute_optimal_prices_batch(off, y0, w_ref[None], np.zeros(1), np.zeros((1, 3 * N)),
                                                         max_iter=300, tol_type="max")
            out[mode] = (prices[0], int(st["iter"][0]))
            assert ps.last_pivot_overflows() == 0
        assert out[2][1] == out[3][1] == st_o["iter"], (name, out[2][1], out[3][1], st_o["iter"])
        assert _close(out[2][0], lam_o) and _close(out[3][0], lam_o), name


@pytest.mark.parametrize("N", [12, 24, 48])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_max_tolerance_station_chain(ev, N):
    """price_solve_chain_dev (one warp per station walking its partitions in the reference's warm-start order) with
    the "max" tolerance type: the parametric chain against the thread-per-EV chain at N = 12 and 24 and against the
    chain of phase-split loops at N = 48.  Per-group iteration counts equal, prices within the bars."""
    import torch
    from chargingstation import _native
    from chargingstation.price_solver import PriceSolver
    o, c = _consts(ev)
    lib = _native.load()
    rng = np.random.default_rng(600 + N + (ev == "large"))
    S, P = 6, 4
    counts = rng.integers(0, 40, P * S)
    counts[[1, 7]] = 0, 1  # an empty and a single-EV partition
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    y0 = np.concatenate([0.3 + 0.1 * (g // S) + 0.1 * rng.random(n) for g, n in enumerate(counts)])
    w_ref = o.w_max * 0.6 * rng.random((P * S, N))
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    out = {}
    for mode in (2, 3 if N <= 24 else 1):
        ps = PriceSolver(N, c, "linear-convex")
        ps.set_loop_mode(mode)
        d_off, d_y0, d_wref = t(off), t(y0), t(w_ref)
        d_prev = torch.zeros((S, 3 * N), dtype=torch.float64, device=dev)
        d_lr = torch.zeros(P * S, dtype=torch.float64, device=dev)
        d_prices = torch.zeros((P * S, 3 * N), dtype=torch.float64, device=dev)
        d_iters = torch.zeros(P * S, dtype=torch.int32, device=dev)
        d_pre, d_post = torch.zeros(P * S, dtype=torch.float64, device=dev), torch.zeros(P * S, dtype=torch.float64, device=dev)
        mx = C.c_int32(0)
        _native.raise_for(lib.price_solve_chain_dev(
            ps._h, S, P, int(off[-1]), d_off.data_ptr(), d_y0.data_ptr(), d_wref.data_ptr(), d_lr.data_ptr(), 3 * N,
            200, 1, 0.01, 0.01, d_prev.data_ptr(), d_prices.data_ptr(), d_iters.data_ptr(), d_pre.data_ptr(),
            d_post.data_ptr(), None, C.byref(mx), torch.cuda.current_stream().cuda_stream))
        out[mode] = (d_iters.cpu().numpy(), d_prices.cpu().numpy(), d_prev.cpu().numpy())
    a, b = out[2], out[3 if N <= 24 else 1]
    assert np.array_equal(a[0], b[0]), (a[0], b[0])
    assert a[0][1] == -1 and np.max(a[0]) > 0
    for g in range(P * S):
        assert _close(a[1][g], b[1][g]), g
    for s in range(S):
        assert _close(a[2][s], b[2][s]), s


def test_fleet_with_max_tolerance():
    """ChargingStationFleet(tol_type="max"), 3 stations, 3 closed-loop steps: the default (parametric) price loops
    against the thread-per-EV loops on both solvers - partition sizes and price-loop iteration counts equal, every other
    log within 1e-8."""
    from chargingstation import settings
    from chargingstation.bimpc import BiMPCChargingCostType, BiMPCConstants
    from chargingstation.charging_station import ChargingStationConstants
    from chargingstation.demand_data import medium_term_demand_forecast
    from chargingstation.fleet import ChargingStationFleet
    from chargingstation.lompc import LoMPCConstants
    settings.PRINT_LEVEL = 0
    Tf, N_bi, N_lo, M, P, S = 3, 16, 12, 120, 12, 3
    dem = medium_term_demand_forecast(Tf + N_bi + 1, 0.25) * (M / 500)
    cb = BiMPCConstants(1e3, 1, 1, 0.3, 0.3, BiMPCChargingCostType(1), 5)
    consts = ChargingStationConstants(Tf, N_bi, N_lo, M, P, dem, cb, LoMPCConstants(0.05, 10, 0.9, 0.25, "small"),
                                      LoMPCConstants(0.025, 50, 0.9, 0.15, "large"), "linear-convex")
    with pytest.raises(ValueError):
        ChargingStationFleet(consts, S, seed=3, tol_type="maximum")
    logs = {}
    for mode in (0, 3):
        fleet = ChargingStationFleet(consts, S, seed=3, rng="device", chain="reference", tol_type="max")
        for k in ("s", "l"):
            fleet.solver[k].set_loop_mode(mode)
        fleet.simulate()
        logs[mode] = {k: v.cpu().numpy() for k, v in fleet.log.items()}
    a, b = logs[0], logs[3]
    assert np.max(a["niter_s"]) > 0
    for key in a:
        if key.startswith(("niter_", "Mp_", "bimpc_")):
            assert np.array_equal(a[key], b[key]), key
        else:
            assert np.array_equal(np.isnan(a[key]), np.isnan(b[key])), key
            d = np.abs(a[key] - b[key]) / np.maximum(1.0, np.abs(b[key]))
            assert np.nanmax(d, initial=0.0) <= 1e-8, key
