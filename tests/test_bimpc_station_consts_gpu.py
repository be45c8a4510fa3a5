"""The batched BiMPC kernel with one set of constants per station (bimpc_solve_kernel<true>, reached through
`BiMPC.solve_bimpc_batch(consts=...)` and `bimpc_solve_batch_consts_dev`).

Station s of a mixed batch must come out with the bits a handle created with its constants gives it alone: both
paths run the same kernel body on the same values.  Shared constants must give the bits of the uniform entry point,
the kernel must agree with its per-station host twin, and a station with an infeasible program or invalid constants
must not disturb its neighbours."""
import ctypes as C
import warnings

import numpy as np
import pytest

from bimpc_cases import draw_station, stack
from oracle import bimpc_oracle as bo
from test_bimpc_envelope_gpu import (check_against_twin, consts, mirror, mixed_batch, p_max, sweep_actives,
                                     with_active)
from test_bimpc_station_consts_cpu import degenerate, mixed_consts, public_consts

W, U, E = bo.WEIGHTED, bo.UNWEIGHTED, bo.EXP_UNWEIGHTED
B200_OPTIN = 232448


def solve_mixed(base, cs, stations):
    """The per-station solve of `stations` (station s with constants cs[s]) on a handle created with `base`."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return mirror(base).solve_bimpc_batch(*stack(stations), consts=[public_consts(c) for c in cs])


def solve_alone(c, par):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return mirror(c).solve_bimpc_batch(*stack([par]))


def assert_station_bits(got, s, ref, r=0, label=None):
    for x, y in zip(got[:3], ref[:3]):
        assert np.array_equal(x[s], y[r]), (label, s)
    for key in ("status", "iters", "objective"):
        assert got[3][key][s] == ref[3][key][r] or (np.isnan(got[3][key][s]) and np.isnan(ref[3][key][r])), \
            (label, s, key)


# (N, P): N = 1, 24, 48; nb on both sides of 32 and 64; P_max(N) of a B200
SHAPES = [(1, 1), (1, p_max(1, B200_OPTIN)), (12, 32), (24, 16), (24, p_max(24, B200_OPTIN)), (48, 1),
          (48, p_max(48, B200_OPTIN))]


def shape_batch(N, P):
    """Stations of every active count of the envelope sweep, each with its own constants from MIX (cycled), and at
    P = 32 the nb = 32, 33, 64, 65 stations."""
    cs_all = mixed_consts(N, P)
    rng = np.random.default_rng(31 * N + P)
    actives = sweep_actives(P) + ([31, 32, 63, 64] if P == 32 else [])
    cs, stations = [], []
    for i, a in enumerate(actives * 2):
        c = cs_all[i % len(cs_all)]
        cs.append(c)
        stations.append(with_active(rng, c, a))
    return cs, stations


@pytest.mark.gpu
@pytest.mark.parametrize("N,P", SHAPES, ids=[f"N{n}-P{p}" for n, p in SHAPES])
def test_mixed_batch_station_is_its_own_handle_alone(N, P):
    base = consts(N, P, E)
    cs, stations = shape_batch(N, P)
    got = solve_mixed(base, cs, stations)
    for s, (c, par) in enumerate(zip(cs, stations)):
        assert_station_bits(got, s, solve_alone(c, par), label=(N, P))
    assert np.mean(got[3]["status"] == 0) >= 0.8, got[3]["status"]


@pytest.mark.gpu
def test_large_mixed_batch_switches_constants_between_stations():
    """1,536 stations at P_max(24) = 37 (one CTA per SM, about ten stations each), of random kinds and with constants
    drawn at random from MIX: each persistent CTA changes constants from station to station.  Every station has the
    bits of its constants' handle solving the stations of those constants as a uniform batch, and a sample has the
    bits of that handle solving it alone."""
    import torch
    N, P, S = 24, 37, 1536
    assert S > 2 * torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(77)
    cs_all = mixed_consts(N, P)
    kinds, stations = mixed_batch(cs_all[0], S, rng)
    pick = rng.integers(len(cs_all), size=S)
    cs = [cs_all[i] for i in pick]
    got = solve_mixed(consts(N, P, W), cs, stations)
    for i, c in enumerate(cs_all):
        idx = np.nonzero(pick == i)[0]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            ref = mirror(c).solve_bimpc_batch(*stack([stations[s] for s in idx]))
        for r, s in enumerate(idx):
            assert_station_bits(got, s, ref, r, label=(i, kinds[s]))
    for s in rng.choice(S, 48, replace=False):
        assert_station_bits(got, s, solve_alone(cs[s], stations[s]), label=kinds[s])
    ok = np.array(kinds) != "infeasible"
    assert np.mean(got[3]["status"][ok] == 0) >= 0.95


def _dev_buffers(b, stations, consts_list):
    import torch
    dev = torch.device("cuda", b.device)
    S, P, N = len(stations), b.P, b.N
    ins = [torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device=dev) for a in stack(stations)]
    out = {"ws": torch.full((S, P, N), -1.0, dtype=torch.float64, device=dev),
           "wl": torch.full((S, P, N), -1.0, dtype=torch.float64, device=dev),
           "ug": torch.full((S, N), -1.0, dtype=torch.float64, device=dev),
           "st": torch.full((S,), -1, dtype=torch.int32, device=dev),
           "it": torch.full((S,), -1, dtype=torch.int32, device=dev),
           "obj": torch.full((S,), -1.0, dtype=torch.float64, device=dev)}
    from chargingstation.bimpc import stage_weights, station_constants
    sc = station_constants(consts_list, S)
    cst = {f: torch.from_numpy(sc[f]).to(dev) for f in ("delta", "c_g", "u_g_max", "u_b_max", "x_max", "cost_type")}
    cst["omega"] = torch.from_numpy(np.stack([stage_weights(b._lib, N, ct, er)
                                              for ct, er in zip(sc["cost_type"], sc["exp_rate"])])).to(dev)
    return ins, out, cst


CONST_ORDER = ("delta", "c_g", "u_g_max", "u_b_max", "x_max", "cost_type", "omega")


def _dev_consts_solve(b, ins, out, cst, ptrs=None):
    import torch
    stream = torch.cuda.Stream(b.device)
    torch.cuda.synchronize(b.device)
    ptrs = ptrs if ptrs is not None else [cst[k].data_ptr() for k in CONST_ORDER]
    with torch.cuda.stream(stream):
        rc = b._lib.bimpc_solve_batch_consts_dev(b._h, len(ins[0]), *ptrs, *[t.data_ptr() for t in ins],
                                                 *[out[k].data_ptr() for k in ("ws", "wl", "ug", "st", "it", "obj")],
                                                 C.c_void_p(stream.cuda_stream))
    stream.synchronize()
    return rc, {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("cost", [W, U, E])
def test_shared_constants_give_the_bits_of_the_uniform_entry_point(cost):
    """Per-station arrays that all hold the handle's constants, through the device entry point on a non-default
    stream: the bits of bimpc_solve_batch_dev."""
    from test_bimpc_envelope_gpu import _dev_solve
    c = consts(24, 37, cost)
    rng = np.random.default_rng(40 + cost)
    _, stations = mixed_batch(c, 600, rng)
    b = mirror(c)
    ref = _dev_solve(b, stations, True)
    ins, out, cst = _dev_buffers(b, stations, [public_consts(c)] * len(stations))
    rc, got = _dev_consts_solve(b, ins, out, cst)
    assert rc == 0
    for k in ref:
        assert np.array_equal(got[k], ref[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("N,P", [(16, 12), (24, 16), (48, 12), (12, 32)])
def test_per_station_kernel_against_per_station_twin(N, P):
    """Equal statuses, iteration counts within the envelope tests' allowance, and their twin bars (objective and
    feasibility only for the stations whose delta or c_g is 0)."""
    from test_bimpc_envelope_gpu import ITER_OFF_FRACTION
    from test_bimpc_station_consts_cpu import twin_consts
    cs_all = mixed_consts(N, P)
    rng = np.random.default_rng(5 * N + P)
    cs, stations = [], []
    for i in range(3 * len(cs_all)):
        c = cs_all[i % len(cs_all)]
        cs.append(c)
        stations.append(draw_station(rng, c) if i % 3 else with_active(rng, c, P))
    got = solve_mixed(consts(N, P, U), cs, stations)
    ref = twin_consts(cs, stations)
    assert np.array_equal(got[3]["status"], ref[3]["status"]) and (ref[3]["status"] == 0).all()
    d = np.abs(got[3]["iters"].astype(int) - ref[3]["iters"].astype(int))
    assert d.max() <= 1 and np.count_nonzero(d) <= max(1, int(ITER_OFF_FRACTION * len(d))), d
    for s, (c, par) in enumerate(zip(cs, stations)):
        def one(r):
            return r[0][s:s + 1], r[1][s:s + 1], r[2][s:s + 1], {k: v[s:s + 1] for k, v in r[3].items()}
        if degenerate(c):
            k = bo.kkt_certificate(c, par, got[0][s], got[1][s], got[2][s], multipliers=False)
            assert k["max_violation"] <= 1e-8
            assert abs(k["objective"] - ref[3]["objective"][s]) <= 1e-8 * max(1.0, abs(k["objective"]))
            assert abs(k["objective"] - got[3]["objective"][s]) <= 1e-9 * max(1.0, abs(k["objective"]))
        else:
            check_against_twin(c, [par], one(got), one(ref))


@pytest.mark.gpu
def test_infeasible_and_invalid_stations_leave_their_neighbours_alone():
    """An infeasible station (status 1) and stations with invalid constants (negative, NaN or inf field, unknown
    cost type, exp_rate < 1 through the host entry point, a non-finite omega row through the device entry point)
    get their status; every other station keeps the bits it has in a clean batch."""
    N, P = 16, 12
    cs_all = mixed_consts(N, P)
    rng = np.random.default_rng(12)
    cs = [cs_all[i % len(cs_all)] for i in range(12)]
    stations = [draw_station(rng, c) for c in cs]
    base = consts(N, P, U)
    b = mirror(base)
    clean = b.solve_bimpc_batch(*stack(stations), consts=[public_consts(c) for c in cs])
    assert (clean[3]["status"] == 0).all()
    from chargingstation.bimpc import station_constants
    bad = [public_consts(c) for c in cs]
    # the host checks of solve_bimpc_batch would refuse these: go through the C host entry point directly
    sc = station_constants(bad, len(cs))
    sc["delta"][2] = -1.0
    sc["c_g"][4] = np.nan
    sc["x_max"][5] = np.inf
    sc["cost_type"][7] = 3
    sc["exp_rate"][9] = 0.5
    st2 = list(stations)
    st2[1] = stations[1][:7] + (stations[1][7] * 10.0,)  # infeasible demand
    arrs = [np.ascontiguousarray(a) for a in stack(st2)]
    S = len(cs)
    ws, wl, ug = np.empty((S, P, N)), np.empty((S, P, N)), np.empty((S, N))
    st, it, obj = np.empty(S, np.int32), np.empty(S, np.int32), np.empty(S)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = b._lib.bimpc_solve_batch_consts_host(
        b._h, S, *[p(sc[f]) for f in ("delta", "c_g", "u_g_max", "u_b_max", "x_max", "cost_type", "exp_rate")],
        *[p(a) for a in arrs], p(ws), p(wl), p(ug), p(st), p(it), p(obj))
    from chargingstation import _native
    assert rc == _native.ERR_NOT_CONVERGED
    assert st[1] != 0 and all(st[i] == 2 for i in (2, 4, 5, 7, 9)), st
    keep = [i for i in range(S) if i not in (1, 2, 4, 5, 7, 9)]
    got = (ws, wl, ug, {"status": st, "iters": it, "objective": obj})
    for s in keep:
        assert_station_bits(got, s, clean, s)
    # a non-finite omega row on the device path
    ins, out, cst = _dev_buffers(b, stations, [public_consts(c) for c in cs])
    cst["omega"][3, 5] = float("nan")
    cst["omega"][6, 0] = float("inf")
    rc, d = _dev_consts_solve(b, ins, out, cst)
    assert rc == 0 and d["st"][3] == 2 and d["st"][6] == 2
    for s in set(range(S)) - {3, 6}:
        assert_station_bits((d["ws"], d["wl"], d["ug"], {"status": d["st"], "iters": d["it"], "objective": d["obj"]}),
                            s, clean, s)


@pytest.mark.gpu
def test_null_constants_launch_nothing():
    import torch
    from chargingstation import _native
    c = consts(16, 12, U)
    stations = [draw_station(np.random.default_rng(2), c) for _ in range(3)]
    b = mirror(c)
    ins, out, cst = _dev_buffers(b, stations, [public_consts(c)] * 3)
    lib = b._lib
    for i in range(len(CONST_ORDER)):
        ptrs = [cst[k].data_ptr() for k in CONST_ORDER]
        ptrs[i] = None
        n0 = lib.lompc_launch_count()
        rc, d = _dev_consts_solve(b, ins, out, cst, ptrs)
        assert rc == _native.ERR_ARG and lib.lompc_launch_count() == n0, CONST_ORDER[i]
        assert np.all(d["st"] == -1) and np.all(d["ws"] == -1.0)
    # the host entry point likewise
    S, P, N = 3, c.P, c.N
    arrs = [np.ascontiguousarray(a) for a in stack(stations)]
    outs = [np.empty((S, P, N)), np.empty((S, P, N)), np.empty((S, N)), np.empty(S, np.int32), np.empty(S, np.int32),
            np.empty(S)]
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    one = np.ones(S)
    ct = np.ones(S, np.int32)
    for i in range(7):
        cargs = [p(one)] * 5 + [p(ct), p(one * 5)]
        cargs[i] = None
        n0 = lib.lompc_launch_count()
        rc = lib.bimpc_solve_batch_consts_host(b._h, S, *cargs, *[p(a) for a in arrs], *[p(o) for o in outs])
        assert rc == _native.ERR_ARG and lib.lompc_launch_count() == n0, i
    torch.cuda.synchronize()
