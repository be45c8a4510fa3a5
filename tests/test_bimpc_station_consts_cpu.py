"""Per-station BiMPC constants without a GPU: the per-station mode of the kernel body (host twin) against the dense
oracle and against the uniform mode, the stage weights every per-station row is built from, the host-side checks of
`BiMPC.solve_bimpc_batch(consts=...)` and `ChargingStationFleet(bimpc_consts=...)`, and the compiled kernels' SASS."""
import copy
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import hostsim
from hostsim import bimpc_consts as hostsim_consts
from bimpc_cases import draw_station, stack
from oracle import bimpc_oracle as bo

W, U, E = bo.WEIGHTED, bo.UNWEIGHTED, bo.EXP_UNWEIGHTED
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "incentive-design-mpc_b200", "csrc", "liblompc_b200.so")
UNIFORM_KERNEL = "_ZN5bimpc18bimpc_solve_kernelILb0EEEvNS_8BiConstsENS_6BiArgsE"
PER_STATION_KERNEL = "_ZN5bimpc18bimpc_solve_kernelILb1EEEvNS_8BiConstsENS_6BiArgsE"

# (cost type, changes to example_consts): every cost type, exp_rate 1, 5 and inf, delta = 0, c_g = 0 and battery /
# grid limits and generation cost scaled up and down.  Every station of these shapes has a feasible program.
MIX = [(W, dict(x_max=0.45, u_b_max=0.36, u_g_max=1.2, c_g=0.7)),
       (U, dict(c_g=0.0)),
       (E, dict(exp_rate=5.0, delta=0.0)),
       (E, dict(exp_rate=1.0)),
       (E, dict(exp_rate=np.inf)),
       (U, dict(x_max=0.27, u_b_max=0.27, u_g_max=0.9, c_g=1.5))]
MIX_SHAPES = [(16, 12), (24, 16), (48, 12)]


def mixed_consts(N, P, mix=MIX):
    """One oracle BiConsts per entry of `mix`, at (N, P)."""
    out = []
    for cost, kw in mix:
        c = bo.example_consts(N, P)
        c.cost_type = cost
        for k, v in kw.items():
            setattr(c, k, v)
        out.append(c)
    return out


def degenerate(c):
    """delta = 0 or c_g = 0: the optimum is not unique in w or in u_g."""
    return c.delta == 0.0 or c.c_g == 0.0


def mixed_batch(N, P, mix=MIX, seed=0):
    cs = mixed_consts(N, P, mix)
    rng = np.random.default_rng(seed + 7 * N + P)
    return cs, [draw_station(rng, c) for c in cs]


def twin_consts(cs, stations, **kw):
    return hostsim_consts.bimpc_solve_consts(cs, *stack(stations), np.stack([bo.stage_weights(c) for c in cs]), **kw)


def public_consts(c):
    """The mirror's BiMPCConstants of an oracle BiConsts."""
    from chargingstation.bimpc import BiMPCChargingCostType, BiMPCConstants
    return BiMPCConstants(c.delta, c.c_g, c.u_g_max, c.u_b_max, c.x_max, BiMPCChargingCostType(c.cost_type),
                          c.exp_rate)


# ----------------------------------------------------------------------------------------- twin against the oracle
@pytest.mark.parametrize("N,P", MIX_SHAPES, ids=[f"N{n}-P{p}" for n, p in MIX_SHAPES])
def test_twin_per_station_against_oracle(N, P):
    """Each station of a mixed batch, solved by the per-station twin with its own constants, against the dense
    oracle with the same constants: the bars of test_bimpc_envelope_gpu.py (u_g 1e-4 at exp_rate = inf; objective
    and feasibility only where delta = 0 or c_g = 0 leave the optimum non-unique)."""
    from test_bimpc_envelope_gpu import EXP_INF_UG_BAR, check_against_oracle
    cs, stations = mixed_batch(N, P)
    ws, wl, ug, info = twin_consts(cs, stations)
    assert (info["status"] == 0).all(), info["status"]
    for s, (c, par) in enumerate(zip(cs, stations)):
        if degenerate(c):
            _, _, _, io = bo.solve_ipm(c, *par)
            assert io["status"] == 0
            k = bo.kkt_certificate(c, par, ws[s], wl[s], ug[s], multipliers=False)
            assert k["max_violation"] <= 1e-8, (s, k)
            assert abs(k["objective"] - io["objective"]) <= 1e-7 * max(1.0, abs(io["objective"])), (s, k)
        else:
            check_against_oracle(c, par, ws[s], wl[s], ug[s], ug_bar=EXP_INF_UG_BAR if np.isinf(c.exp_rate) else 2e-5)
        # the twin's objective (compact partition list, its own constants) against the certificate's
        k = bo.kkt_certificate(c, par, ws[s], wl[s], ug[s], multipliers=False)
        assert abs(info["objective"][s] - k["objective"]) <= 1e-9 * max(1.0, abs(k["objective"])), s


@pytest.mark.parametrize("N,P", MIX_SHAPES, ids=[f"N{n}-P{p}" for n, p in MIX_SHAPES])
def test_twin_per_station_is_the_uniform_twin_of_each_station(N, P):
    """Station s of a mixed batch has the bits the uniform twin gives it with its constants."""
    cs, stations = mixed_batch(N, P)
    got = twin_consts(cs, stations)
    for s, c in enumerate(cs):
        ref = hostsim.bimpc_solve(c, *stack([stations[s]]), bo.stage_weights(c))
        for x, y in zip(got[:3], ref[:3]):
            assert np.array_equal(x[s], y[0]), s
        for key in ("status", "iters", "objective"):
            assert got[3][key][s] == ref[3][key][0], (s, key)


@pytest.mark.parametrize("cost", [W, U, E])
@pytest.mark.parametrize("N,P", [(1, 3), (16, 12), (48, 12)])
def test_twin_with_shared_constants_is_the_uniform_twin(N, P, cost):
    c = mixed_consts(N, P, [(cost, {})])[0]
    rng = np.random.default_rng(N + P + cost)
    stations = [draw_station(rng, c) for _ in range(4)] + [draw_station(rng, c, active_s=[], active_l=[])]
    om = bo.stage_weights(c)
    ref = hostsim.bimpc_solve(c, *stack(stations), om)
    got = hostsim_consts.bimpc_solve_consts([c] * len(stations), *stack(stations), np.tile(om, (len(stations), 1)))
    for x, y in zip(got[:3], ref[:3]):
        assert np.array_equal(x, y)
    for key in ("status", "iters", "objective"):
        assert np.array_equal(got[3][key], ref[3][key]), key
    assert (ref[3]["status"] == 0).all()


def test_twin_flags_invalid_constants_and_leaves_neighbours_alone():
    """A negative, NaN or inf constant, an unknown cost type or a non-finite stage weight gives status 2; the
    stations around it keep their bits."""
    N, P = 16, 12
    c = mixed_consts(N, P, [(U, {})])[0]
    rng = np.random.default_rng(3)
    good = [draw_station(rng, c) for _ in range(2)]
    om = bo.stage_weights(c)
    ref = hostsim.bimpc_solve(c, *stack(good), om)
    bad_cases = [("delta", -1.0), ("c_g", np.nan), ("u_g_max", np.inf), ("u_b_max", -0.1), ("x_max", np.nan),
                 ("cost_type", 3), ("cost_type", -1), ("omega", np.nan), ("omega", np.inf)]
    for field, v in bad_cases:
        bad = copy.copy(c)
        om_bad = om.copy()
        if field == "omega":
            om_bad[N // 2] = v
        else:
            setattr(bad, field, v)
        got = hostsim_consts.bimpc_solve_consts([c, bad, c], *stack([good[0], good[0], good[1]]),
                                                np.stack([om, om_bad, om]))
        assert got[3]["status"][1] == 2, (field, v)
        for s, r in ((0, 0), (2, 1)):
            for x, y in zip(got[:3], ref[:3]):
                assert np.array_equal(x[s], y[r]), (field, v, s)
            assert got[3]["iters"][s] == ref[3]["iters"][r] and got[3]["status"][s] == 0


# ---------------------------------------------------------------------------------------------------- stage weights
def _lib():
    from chargingstation import _native
    return _native.load()


@pytest.mark.parametrize("cost", [W, U, E])
def test_stage_weights_have_the_bits_of_the_create_loop(cost):
    lib = _lib()
    for N in (1, 2, 7, 16, 24, 47, 48):
        for rate in (1.0, 1.0000001, 1.5, 2.0, 3.7, 5.0, 10.0, 1e3, 1e300, np.inf):
            om = np.full(N, -1.0)
            assert lib.bimpc_stage_weights(N, cost, rate, om.ctypes.data_as(C.c_void_p)) == 0
            ref = hostsim_consts.stage_weights_loop(N, cost, rate)
            assert np.array_equal(om.view(np.uint64), ref.view(np.uint64)), (N, rate)
            assert np.all(np.isfinite(om))
    from chargingstation.bimpc import stage_weights
    assert stage_weights(lib, 5, E, 5.0).tolist() == [5.0 ** -4, 5.0 ** -3, 5.0 ** -2, 0.2, 1.0]


def test_stage_weights_refusals():
    from chargingstation import _native
    lib = _lib()
    om = np.full(4, -1.0)
    p = om.ctypes.data_as(C.c_void_p)
    for cost, rate in ((3, 5.0), (-1, 5.0), (E, 0.5), (U, 0.99), (E, np.nan)):
        assert lib.bimpc_stage_weights(4, cost, rate, p) == _native.ERR_CONSTS, (cost, rate)
    assert lib.bimpc_stage_weights(0, E, 5.0, p) == _native.ERR_ARG
    assert lib.bimpc_stage_weights(4, E, 5.0, None) == _native.ERR_ARG
    assert np.all(om == -1.0)


# ---------------------------------------------------------------------------------------------- host-side checks
class _DeviceWork(Exception):
    pass


class _Refuse:
    def __getattr__(self, name):
        raise _DeviceWork(name)


def _bad_consts(base, S):
    """(label, constants list, exception type) of every refusal."""
    ok = [copy.copy(base) for _ in range(S)]

    def with_(field, v):
        out = [copy.copy(c) for c in ok]
        setattr(out[1], field, v)
        return out
    return [("too few", ok[:-1], AssertionError), ("too many", ok + [base], AssertionError),
            ("one for all", base, AssertionError),
            ("negative delta", with_("delta", -1.0), AssertionError),
            ("negative c_g", with_("c_g", -0.5), AssertionError),
            ("negative u_g_max", with_("u_g_max", -1e-9), AssertionError),
            ("negative u_b_max", with_("u_b_max", -0.3), AssertionError),
            ("negative x_max", with_("x_max", -0.3), AssertionError),
            ("NaN x_max", with_("x_max", np.nan), AssertionError),
            ("exp_rate < 1", with_("exp_rate", 0.5), AssertionError),
            ("unknown cost type", with_("charging_cost_type", 2), NotImplementedError),
            ("cost type as a string", with_("charging_cost_type", "WEIGHTED"), NotImplementedError)]


def _base_public():
    from chargingstation.bimpc import BiMPCChargingCostType, BiMPCConstants
    return BiMPCConstants(1e3, 1.0, 1.0, 0.3, 0.3, BiMPCChargingCostType.EXP_UNWEIGHTED, 5)


def test_solve_bimpc_batch_checks_consts_before_device_work():
    from chargingstation.bimpc import BiMPC
    N, P, S = 8, 3, 3
    b = BiMPC.__new__(BiMPC)  # no handle: the library must not be reached
    b.N, b.P, b._h, b._lib = N, P, None, _Refuse()
    c = mixed_consts(N, P, [(U, {})])[0]
    rng = np.random.default_rng(1)
    arrs = stack([draw_station(rng, c) for _ in range(S)])
    cases = _bad_consts(_base_public(), S)
    for label, consts, exc in cases:
        with pytest.raises(exc) as ei:
            b.solve_bimpc_batch(*arrs, consts=consts)
        if label not in ("too few", "too many", "one for all"):
            assert "station 1" in str(ei.value), label
    with pytest.raises(_DeviceWork):
        b.solve_bimpc_batch(*arrs, consts=[_base_public()] * S)
    with pytest.raises(_DeviceWork):
        b.solve_bimpc_batch(*arrs)


@pytest.fixture
def no_device(monkeypatch):
    """Any step past the fleet's host-side checks raises _DeviceWork."""
    from chargingstation import fleet

    def refuse(*args, **kwargs):
        raise _DeviceWork()

    monkeypatch.setattr(fleet._native, "load", refuse)
    monkeypatch.setattr(fleet, "BiMPC", refuse)
    monkeypatch.setattr(fleet, "PriceSolver", refuse)
    return fleet.ChargingStationFleet


def test_fleet_checks_bimpc_consts_before_device_work(no_device):
    import test_fleet_gpu as closed_loop_tests
    consts = closed_loop_tests._consts(2, 8, 4, 40, 6, 1)
    cases = _bad_consts(consts.bimpc_consts, 3)
    for label, bc, exc in cases:
        with pytest.raises(exc) as ei:
            no_device(consts, 3, bimpc_consts=bc)
        if label not in ("too few", "too many", "one for all"):
            assert "station 1" in str(ei.value), label
    for bc in (None, [consts.bimpc_consts] * 3, tuple(copy.copy(consts.bimpc_consts) for _ in range(3))):
        with pytest.raises(_DeviceWork):
            no_device(consts, 3, bimpc_consts=bc)
    with pytest.raises(_DeviceWork):
        no_device(consts, 3, nevs=[1, 9, 40], bimpc_consts=[consts.bimpc_consts] * 3)


# -------------------------------------------------------------------------------------------------------------- SASS
@pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(LIB),
                    reason="needs cuobjdump and the built library")
def test_both_kernels_are_built_and_the_per_station_one_keeps_to_registers():
    """Both instantiations are in the library; the per-station one stays within the register cap of four stations
    per SM (128) with no stack and no local-memory instruction."""
    res = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True).stdout
    usage = {}
    for name in (UNIFORM_KERNEL, PER_STATION_KERNEL):
        m = re.search(re.escape(name) + r":\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", res)
        assert m, name
        usage[name] = tuple(int(g) for g in m.groups())
    reg, stack_, local = usage[PER_STATION_KERNEL]
    assert reg <= 128 and stack_ == 0 and local == 0, usage
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", PER_STATION_KERNEL, LIB], capture_output=True,
                          text=True).stdout
    ops = [m.group(1) for m in re.finditer(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", sass)]
    assert len(ops) > 5000, "kernel not found in the library"
    assert not any(o.startswith(("LDL", "STL")) for o in ops)
