"""Fleets whose stations have their own BiMPC constants (``ChargingStationFleet(bimpc_consts=...)``): against
single-station runs with those constants, against the default fleet when every station holds the shared constants,
and at fleet scale against a small fleet of its first stations."""
import copy
import dataclasses

import numpy as np
import pytest

import test_fleet_gpu as closed_loop_tests
import test_fleet_kernels_gpu as kt
from test_fleet_sizes_gpu import MIRROR_SIZES, _assert_same_state, _ragged_demand, _state
from chargingstation.settings import MIN_INITIAL_SOC


def station_mix(base):
    """Six BiMPC constant sets around `base` (normalised units): every cost type, exp_rate 1, 2, 5 and inf, battery
    capacity and rate, grid limit, generation cost and charging-cost weight scaled."""
    from chargingstation.bimpc import BiMPCChargingCostType as T
    r = dataclasses.replace
    return [r(base, delta=2e3, c_g=1.3, u_g_max=1.1, charging_cost_type=T.UNWEIGHTED),
            r(base, x_max=0.45, u_b_max=0.36, u_g_max=1.2, c_g=0.7, charging_cost_type=T.WEIGHTED),
            r(base, x_max=0.6, u_b_max=0.45, charging_cost_type=T.EXP_UNWEIGHTED, exp_rate=5),
            r(base, u_g_max=1.5, c_g=2.0, charging_cost_type=T.EXP_UNWEIGHTED, exp_rate=2),
            r(base, delta=5e2, x_max=0.36, charging_cost_type=T.EXP_UNWEIGHTED, exp_rate=1),
            r(base, x_max=0.4, c_g=0.8, charging_cost_type=T.EXP_UNWEIGHTED, exp_rate=np.inf)]


def mirror_mix(base):
    """Five sets for the comparison with the single-station mirror: every cost type, with exp_rate 1 for
    EXP_UNWEIGHTED.  With exp_rate > 1 (sets 2, 3 and 5 of station_mix) the mirror's price loop and the fleet's chain
    kernel end up to 1e-7 apart at N_lo = 24 in avg_price_l, and the gap then reaches the reduced prices and the SoCs.
    A uniform fleet given such a set through consts.bimpc_consts, without per-station constants, shows the same
    gap (9.6e-8 and 4.6e-8 in avg_price_l for sets 3 and 2 on a B200).  That is a property of the price loops under
    those weights, beyond the 1e-8 bars of this comparison.  test_mixed_constants_station_is_its_own_fleet checks
    every set of station_mix bit for bit."""
    from chargingstation.bimpc import BiMPCChargingCostType as T
    r = dataclasses.replace
    mix = station_mix(base)
    return [mix[0], mix[1], r(mix[2], charging_cost_type=T.UNWEIGHTED),
            r(mix[3], charging_cost_type=T.WEIGHTED), mix[4]]


@pytest.mark.gpu
@pytest.mark.parametrize("price_type", ["linear-convex", "linear"])
@pytest.mark.parametrize("N_bi,N_lo", [(16, 12), (24, 24)], ids=["Nlo12", "Nlo24"])
def test_mixed_constants_ragged_fleet_equals_single_station_runs(price_type, N_bi, N_lo):
    """Stations of sizes {1, 9, 40, 120, 300}, each with its own constants, against ChargingStation with that
    nEVs_per_EV_type, those constants, its demand and seed + s (reference chain; the bars of
    test_fleet_sizes_gpu.py::test_ragged_fleet_equals_single_station_runs)."""
    from chargingstation.charging_station import ChargingStation
    from chargingstation.fleet import ChargingStationFleet
    Tf, P = 4, 12
    S = len(MIRROR_SIZES)
    consts = closed_loop_tests._consts(Tf, N_bi, N_lo, 500, P, 1, price_type)
    mix = mirror_mix(consts.bimpc_consts)
    demand = np.array([1.0, 0.97, 1.04, 0.99, 1.02])[:, None] * _ragged_demand(consts, MIRROR_SIZES)
    fleet = ChargingStationFleet(consts, S, demand=demand, seed=100, rng="numpy", chain="reference",
                                 nevs=MIRROR_SIZES, bimpc_consts=mix)
    assert fleet.bimpc_consts == mix
    fleet.simulate()
    assert np.all(fleet.log["bimpc_status"].cpu().numpy() == 0)
    for s, n in enumerate(MIRROR_SIZES):
        c = copy.copy(consts)
        c.nEVs_per_EV_type = int(n)
        c.demand = demand[s]
        c.bimpc_consts = mix[s]
        np.random.seed(100 + s)
        one = ChargingStation(c)
        ref = one.simulate()
        got = fleet.station_logs(s)
        assert got["constants"].nEVs_per_EV_type == n and got["constants"].bimpc_consts == mix[s]
        for key in ("Mp_s", "Mp_l", "niter_s", "niter_l"):
            assert np.array_equal(got["statistics"][key], ref["statistics"][key]), (s, key)
        assert got["statistics"]["ncharged_s"] == ref["statistics"]["ncharged_s"]
        assert got["statistics"]["ncharged_l"] == ref["statistics"]["ncharged_l"]
        for grp, key in (("inputs", "u_g"), ("states", "x"), ("inputs", "w_hat_s"), ("inputs", "w_hat_l"),
                         ("inputs", "w_s"), ("inputs", "w_l"), ("bounds", "beta_s"), ("bounds", "beta_l"),
                         ("statistics", "gamma_sm"), ("statistics", "gamma_lm"), ("prices", "avg_price_s"),
                         ("prices", "avg_price_l")):
            err = np.max(np.abs(got[grp][key] - ref[grp][key]) / np.maximum(1.0, np.abs(ref[grp][key])))
            assert err <= 1e-8, (s, grp, key)
        for key in ("price_red_s", "price_red_l"):
            a, b = got["prices"][key], ref["prices"][key]
            assert np.array_equal(np.isnan(a), np.isnan(b))
            assert np.nanmax(np.abs(a - b) / np.maximum(1.0, np.abs(b))) <= 1e-8
        assert np.max(np.abs(fleet.y["s"][s, :n].cpu().numpy() - one.y_s)) <= 1e-9
        assert np.max(np.abs(fleet.y["l"][s, :n].cpu().numpy() - one.y_l)) <= 1e-9
        assert abs(float(fleet.x[s]) - one.x) <= 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("chain", ["reference", "partition"])
@pytest.mark.parametrize("price_type", ["linear-convex", "linear"])
@pytest.mark.parametrize("N_bi,N_lo", [(16, 12), (24, 24)], ids=["Nlo12", "Nlo24"])
def test_mixed_constants_station_is_its_own_fleet(chain, price_type, N_bi, N_lo):
    """Station s of the mixed, ragged fleet has the bits of a one-station fleet of its size, constants (through
    consts.bimpc_consts, the uniform kernel), demand and seed + s, in every log, its state and its prices."""
    from chargingstation.fleet import ChargingStationFleet
    Tf, P = 4, 12
    sizes = np.append(MIRROR_SIZES, 75)
    S = len(sizes)
    consts = closed_loop_tests._consts(Tf, N_bi, N_lo, 500, P, 1, price_type)
    mix = station_mix(consts.bimpc_consts)
    demand = _ragged_demand(consts, sizes, np.random.default_rng(9))
    fleet = ChargingStationFleet(consts, S, demand=demand, seed=100, rng="numpy", chain=chain,
                                 nevs=sizes, bimpc_consts=mix)
    fleet.simulate()
    assert np.all(fleet.log["bimpc_status"].cpu().numpy() == 0)
    big = _state(fleet)
    for s, n in enumerate(sizes):
        one = ChargingStationFleet(dataclasses.replace(consts, nEVs_per_EV_type=int(n), bimpc_consts=mix[s]), 1,
                                   demand=demand[s:s + 1], seed=100 + s, rng="numpy", chain=chain)
        one.simulate()
        for k, v in _state(one).items():
            if k.startswith("log_"):
                mine = big[k][..., s:s + 1]
            elif k[:-2] in ("y", "idx"):
                mine = big[k][s:s + 1, :n]
            elif k[:-2] == "prices":
                mine = big[k].reshape(P, S, -1)[:, s]
            else:
                mine = big[k][s:s + 1]
            kt.assert_same(mine.view(np.uint8), v.view(np.uint8), (s, k))


@pytest.mark.gpu
@pytest.mark.parametrize("chain", ["reference", "partition"])
def test_shared_constants_per_station_is_the_default_fleet(chain):
    """bimpc_consts = S copies of consts.bimpc_consts runs the per-station kernel and gives the bits of the default
    fleet (the uniform kernel): logs, SoCs, prices and battery states."""
    from chargingstation.fleet import ChargingStationFleet
    Tf, S, M, P = 3, 6, 40, 6
    consts = closed_loop_tests._consts(Tf, 16, 12, M, P, 2)
    demand = np.array([1.0, 0.97, 1.04, 1.01, 0.99, 1.02])[:, None] * consts.demand[None, :]
    y0 = np.random.default_rng(2).uniform(MIN_INITIAL_SOC, 0.84, (2, S, M))  # EVs leave within the three steps
    runs = []
    for bc in (None, [copy.copy(consts.bimpc_consts) for _ in range(S)]):
        f = ChargingStationFleet(consts, S, demand=demand, seed=11, rng="device", chain=chain, bimpc_consts=bc)
        assert (f._bi_consts is None) == (bc is None)
        for i, k in enumerate(("s", "l")):
            f.y[k].copy_(f.torch.from_numpy(y0[i]))
        f.simulate()
        assert f.station_logs(2)["constants"].bimpc_consts == consts.bimpc_consts
        runs.append(_state(f))
    _assert_same_state(*runs)
    assert int(runs[0]["ncharged_s"].sum() + runs[0]["ncharged_l"].sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("chain", ["reference", "partition"])
def test_mixed_stations_do_not_depend_on_fleet_size(chain):
    """Stations 0..7 of a 1,200-station fleet of mixed constants and sizes and an 8-station fleet with the same
    SoCs, sizes, constants and demand give the same bits."""
    from chargingstation.fleet import ChargingStationFleet
    Tf, P, S_big, S_small = 3, 12, 1200, 8
    rng = np.random.default_rng(41)
    nevs = rng.integers(1, 301, S_big)
    nevs[:S_small] = (300, 1, 129, 257, 40, 256, 9, 128)
    consts = closed_loop_tests._consts(Tf, 16, 12, 500, P, 2)
    mix = station_mix(consts.bimpc_consts)
    bc = [mix[i] for i in rng.integers(len(mix), size=S_big)]
    bc[:S_small] = [mix[i % len(mix)] for i in range(S_small)]
    demand = _ragged_demand(consts, nevs, rng)
    big = ChargingStationFleet(consts, S_big, demand=demand, seed=13, rng="device", chain=chain, nevs=nevs,
                               bimpc_consts=bc)
    small = ChargingStationFleet(consts, S_small, demand=demand[:S_small], seed=13, rng="device", chain=chain,
                                 nevs=nevs[:S_small], bimpc_consts=bc[:S_small])
    pad = np.arange(300)[None, :] >= nevs[:S_small, None]
    for k in ("s", "l"):
        y0 = rng.uniform(MIN_INITIAL_SOC, 0.84, (S_small, 300))
        y0[pad] = np.nan
        y0 = big.torch.from_numpy(y0).to(big.dev)
        big.y[k][:S_small].copy_(y0)
        small.y[k].copy_(y0)
    big_log, small_log = big.simulate(), small.simulate()
    for key in big_log:
        kt.assert_same(big_log[key][..., :S_small].cpu().numpy(), small_log[key].cpu().numpy(), key)
    for k in ("s", "l"):
        kt.assert_same(big.y[k][:S_small].cpu().numpy(), small.y[k].cpu().numpy(), "y_" + k)
        kt.assert_same(big.idx[k][:S_small].cpu().numpy(), small.idx[k].cpu().numpy(), "idx_" + k)
    kt.assert_same(big.x[:S_small].cpu().numpy(), small.x.cpu().numpy(), "x")
    assert np.mean(big_log["bimpc_status"].cpu().numpy() == 0) >= 0.99
    assert len({(c.charging_cost_type, c.x_max) for c in bc[:S_small]}) == len(mix)
