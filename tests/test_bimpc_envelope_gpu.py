"""The batched BiMPC kernel (csrc/bimpc_solve.cuh) over the whole envelope bimpc_create accepts: every horizon up to
kMaxN = 48, partition counts up to what one station's scratch leaves of the shared-memory opt-in, the compaction
edges, mixed batches on the persistent grid, constants at the edge of the mirror's asserts, binding constraints,
the envelope boundary and the status paths.

Three references:
- the host twin (tests/hostsim): the same kernel body run by one thread.  A wrong chunk or tile of the parallel
  decomposition gives an inexact Newton direction; the IPM recomputes its residuals from the iterate, so such an
  error shows up as a different iteration count or status rather than as a wrong converged point;
- the dense oracle (oracle/bimpc_oracle.solve_ipm) and its NNLS certificate, where affordable;
- the primal certificate (feasibility and objective of the returned point), at every shape.

The GPU tests are marked `gpu`; the tests without the mark pin the algorithm (twin against oracle) at the same
shapes, edges and constants on a machine without a GPU."""
import ctypes as C
import warnings

import numpy as np
import pytest

import hostsim
from bimpc_cases import draw_station, stack
from oracle import bimpc_oracle as bo

W, U, E = bo.WEIGHTED, bo.UNWEIGHTED, bo.EXP_UNWEIGHTED
COST = {W: "W", U: "U", E: "E"}
K_MAX_N = 48        # bimpc::kMaxN
THREADS = 128       # bimpc::kThreads
GLOBAL_VECS = 5     # bimpc::kGlobalVecs
B200_OPTIN = 232448  # shared memory a CTA may opt into on a B200 (bytes)


def scratch_doubles(N, P, T=THREADS):
    """bimpc::scratch_doubles: doubles of shared memory one station needs."""
    Q2 = 2 * P
    QN, nb = Q2 * N, Q2 + 1
    return ((9 - GLOBAL_VECS) * QN + (QN + N) + 2 * (nb * (nb + 1) // 2) + 2 * nb * nb + 40 * N + 8 * nb + 3 * T +
            5 * Q2 + 16)


def p_max(N, optin):
    """The largest P bimpc_create accepts at horizon N."""
    P = 1
    while scratch_doubles(N, P + 1) * 8 <= optin:
        P += 1
    return P


def consts(N, P, cost=E, **kw):
    c = bo.example_consts(N, P)
    c.cost_type = cost
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def n_blocks(c, par):
    """Newton block size nb of a station: 1 + the partitions the kernel keeps (EVs, or a target with cost weight)."""
    m = np.concatenate([c.theta_s * par[0], c.theta_l * par[1]])
    g = np.concatenate([par[4], par[5]])
    a = m * m if c.cost_type == W else np.ones_like(m)
    return 1 + int(np.count_nonzero((m != 0) | ((g != 0) & (a != 0))))


def with_active(rng, c, n_active, track_empty=False):
    """A station with `n_active` of its 2P partitions populated, chosen at random (small ones are q < P)."""
    q = rng.choice(2 * c.P, n_active, replace=False)
    return draw_station(rng, c, active_s=[p for p in q if p < c.P], active_l=[p - c.P for p in q if p >= c.P],
                        track_empty=track_empty)


def twin(c, stations, **kw):
    return hostsim.bimpc_solve(c, *stack(stations), bo.stage_weights(c), **kw)


def mirror(c):
    from chargingstation.bimpc import BiMPC, BiMPCChargingCostType, BiMPCConstants
    from chargingstation.lompc import LoMPCConstants
    cb = BiMPCConstants(c.delta, c.c_g, c.u_g_max, c.u_b_max, c.x_max, BiMPCChargingCostType(c.cost_type), c.exp_rate)
    cs = LoMPCConstants(0.05, c.theta_s, 0.9, c.w_max_s, "small")
    cl = LoMPCConstants(0.025, c.theta_l, 0.9, c.w_max_l, "large")
    return BiMPC(c.N, c.P, cb, cs, cl)


def w_determined(c, par):
    """[2, P, N] mask of the w entries the program pins.  UNWEIGHTED: every kept partition has unit curvature in its
    cumulative charge.  WEIGHTED: only partitions with EVs (an empty one has zero weight, its w is arbitrary).
    EXP_UNWEIGHTED: the cumulative charge at stage k has curvature 2 delta omega_k, so w_k is pinned where omega_k and
    omega_{k-1} are >= 1e-3 (the last five stages at exp_rate 5, none but N = 1 at exp_rate = inf)."""
    N, P = c.N, c.P
    mask = np.ones((2, P, N), dtype=bool)
    if c.cost_type == W:
        mask &= np.stack([par[0] > 0, par[1] > 0])[:, :, None]
    if c.cost_type == E:
        om = bo.stage_weights(c)
        mask &= (om >= 1e-3) & (np.concatenate([[1.0], om[:-1]]) >= 1e-3)
    return mask


def inactive_slots(c, par):
    """[2, P] partitions the kernel leaves out of its system: their w must come back exactly 0.0."""
    return ~np.stack([par[0] > 0, par[1] > 0]) & ((np.stack([par[4], par[5]]) == 0) | (c.cost_type == W))


# Bars of the GPU against the twin (the same algorithm; the device differs in summation order, FMA contraction and
# the reciprocal of the elimination pivots).
OBJ_TWIN, UG_TWIN, W_TWIN = 1e-9, 1e-8, 1e-7
ITER_OFF_FRACTION = 0.1  # at most this fraction of a shape's stations (and at least one) may differ by one iteration


def check_against_twin(c, stations, gpu, ref, *, cert=True):
    """The GPU solve `gpu` = (ws, wl, ug, info) of `stations` against the twin's `ref` and the primal certificate."""
    ws, wl, ug, info = gpu
    rws, rwl, rug, rinfo = ref
    assert np.array_equal(info["status"], rinfo["status"]), (info["status"], rinfo["status"])
    d = np.abs(info["iters"].astype(int) - rinfo["iters"].astype(int))
    assert d.max() <= 1 and np.count_nonzero(d) <= max(1, int(ITER_OFF_FRACTION * len(d))), (info["iters"],
                                                                                             rinfo["iters"])
    for s, par in enumerate(stations):
        if info["status"][s] != 0:
            continue
        ob, rob = info["objective"][s], rinfo["objective"][s]
        assert abs(ob - rob) <= OBJ_TWIN * max(1.0, abs(rob)), (s, ob, rob)
        assert np.max(np.abs(ug[s] - rug[s])) <= UG_TWIN, s
        m = w_determined(c, par)
        dw = np.abs(np.stack([ws[s], wl[s]]) - np.stack([rws[s], rwl[s]]))[m]
        assert dw.size == 0 or dw.max() <= W_TWIN, (s, dw.max())
        z = inactive_slots(c, par)
        assert np.all(np.stack([ws[s], wl[s]])[z] == 0.0), s
        if cert:
            k = bo.kkt_certificate(c, par, ws[s], wl[s], ug[s], multipliers=False)
            assert k["max_violation"] <= 1e-8, (s, k)
            # the kernel's objective comes from its compact partition list, the certificate's from the returned
            # [P, N] arrays: they agree only if every partition came back in its own slot
            assert abs(ob - k["objective"]) <= 1e-9 * max(1.0, abs(ob)), (s, ob, k["objective"])


def check_against_oracle(c, par, w_s, w_l, u_g, *, ug_bar=2e-5, multipliers=False):
    wso, wlo, ugo, io = bo.solve_ipm(c, *par)
    assert io["status"] == 0
    k = bo.kkt_certificate(c, par, w_s, w_l, u_g, multipliers=multipliers)
    assert k["max_violation"] <= 1e-8
    assert abs(k["objective"] - io["objective"]) <= 1e-7 * max(1.0, abs(io["objective"])), (k, io["objective"])
    assert np.max(np.abs(u_g - ugo)) <= ug_bar
    assert k["stationarity"] <= 1e-6 and k["complementarity"] <= 1e-7, k  # (0.0 where not computed)
    return k


# ---------------------------------------------------------------------------------------------------------- 1. shapes
# (N, P, cost types).  Together: N in {1, 2, 5, 12, 24, 33, 47, 48}; P = 1, 2, 15, 16, 31, 32 (nb = 3, 5, 31, 33,
# 63, 65: both sides of 32 and 64); P_max(N) at N = 1, 24, 48 (nb = 93, 75, 61).
SWEEP = [(1, 1, (W, U, E)), (1, 46, (W, U, E)), (2, 2, (W, E)), (2, 32, (U,)), (5, 15, (U, E)), (5, 16, (W,)),
         (12, 31, (W, E)), (12, 32, (U,)), (24, 16, (W,)), (24, 37, (W, U, E)), (33, 31, (U, E)), (33, 2, (W,)),
         (47, 5, (W, U, E)), (47, 15, (U,)), (48, 30, (W, U, E)), (48, 1, (U, E))]


def sweep_actives(P):
    """Active partition counts of a shape's stations: full, one emptied, half, a third, a single one."""
    return [2 * P, max(1, 2 * P - 1), P, max(1, 2 * P // 3), 1]


def sweep_stations(N, P, cost):
    c = consts(N, P, cost)
    rng = np.random.default_rng(1000 * N + 10 * P + cost)
    return c, [with_active(rng, c, a) for a in sweep_actives(P)]


SWEEP_CASES = [pytest.param(N, P, cost, id=f"N{N}-P{P}-nb{'/'.join(str(a + 1) for a in sweep_actives(P))}-{COST[cost]}")
               for N, P, costs in SWEEP for cost in costs]


@pytest.mark.gpu
@pytest.mark.parametrize("N,P,cost", SWEEP_CASES)
def test_shape_against_twin(N, P, cost):
    c, stations = sweep_stations(N, P, cost)
    assert [n_blocks(c, s) for s in stations] == [a + 1 for a in sweep_actives(P)]
    gpu = mirror(c).solve_bimpc_batch(*stack(stations))
    ref = twin(c, stations)
    assert (ref[3]["status"] == 0).all()
    check_against_twin(c, stations, gpu, ref)


# affordable dense-oracle shapes (the oracle takes ~14 s at (24, 37)), one station each
ORACLE_SHAPES = [pytest.param(24, 16, W, id="N24-P16-nb33-W"), pytest.param(48, 12, U, id="N48-P12-nb25-U"),
                 pytest.param(24, 37, E, id="N24-P37-nb75-E")]
# cheap large-P shapes for the NNLS certificate
CERT_SHAPES = [pytest.param(2, 40, E, id="N2-P40-nb81-E"), pytest.param(8, 16, W, id="N8-P16-nb33-W")]


def _full_station(N, P, cost):
    c = consts(N, P, cost)
    return c, with_active(np.random.default_rng(N * 100 + P), c, 2 * P)


@pytest.mark.gpu
@pytest.mark.parametrize("N,P,cost", ORACLE_SHAPES + CERT_SHAPES)
def test_shape_against_oracle(N, P, cost):
    c, par = _full_station(N, P, cost)
    ws, wl, ug, info = mirror(c).solve_bimpc_batch(*stack([par]))
    assert info["status"][0] == 0
    check_against_oracle(c, par, ws[0], wl[0], ug[0], multipliers=N * P <= 128)


@pytest.mark.parametrize("N,P,cost", ORACLE_SHAPES + CERT_SHAPES + [
    pytest.param(1, 3, W, id="N1-P3-nb7-W"), pytest.param(1, 3, U, id="N1-P3-nb7-U"),
    pytest.param(2, 1, E, id="N2-P1-nb3-E"), pytest.param(2, 1, W, id="N2-P1-nb3-W"),
    pytest.param(47, 5, U, id="N47-P5-nb11-U"), pytest.param(1, 46, U, id="N1-P46-nb93-U")])
def test_twin_shape_against_oracle(N, P, cost):
    c, par = _full_station(N, P, cost)
    ws, wl, ug, info = twin(c, [par])
    assert info["status"][0] == 0
    check_against_oracle(c, par, ws[0], wl[0], ug[0], multipliers=N * P <= 128)


# ------------------------------------------------------------------------------------------------- 2. compaction edges
def edge_stations(c, rng):
    """Named stations at the compaction edges of a (16, 12)-sized shape."""
    P = c.P
    out = {"none": draw_station(rng, c, active_s=[], active_l=[]),
           "none-tracked": draw_station(rng, c, active_s=[], active_l=[], track_empty=True)}
    for where, p in (("first", 0), ("mid", P // 2), ("last", P - 1)):
        out[f"one-small-{where}"] = draw_station(rng, c, active_s=[p], active_l=[])
        out[f"one-large-{where}"] = draw_station(rng, c, active_s=[], active_l=[p])
    out["half-tracked"] = with_active(rng, c, P, track_empty=True)
    out["one-tracked"] = draw_station(rng, c, active_s=[1], active_l=[], track_empty=True)
    return out


def nb_stations(c, rng):
    """Stations whose Newton blocks are exactly 32, 33, 64 and 65 wide (needs 2P >= 64)."""
    return {f"nb{a + 1}": with_active(rng, c, a) for a in (31, 32, 63, 64)}


EDGE_SETS = [pytest.param(16, 12, cost, id=f"N16-P12-{COST[cost]}") for cost in (W, U, E)] + \
            [pytest.param(12, 32, cost, id=f"N12-P32-nb32/33/64/65-{COST[cost]}") for cost in (U, W)]


def _edge_case(N, P, cost):
    c = consts(N, P, cost)
    rng = np.random.default_rng(7 * N + P + cost)
    named = edge_stations(c, rng) if P < 32 else nb_stations(c, rng)
    return c, named


def _check_edge_blocks(c, named):
    for name, par in named.items():
        nb = n_blocks(c, par)
        if name.startswith("nb"):
            assert nb == int(name[2:]), name
        elif name.startswith("none"):
            assert nb == (2 * c.P + 1 if name == "none-tracked" and c.cost_type != W else 1), name
        elif name.startswith("one-"):
            assert nb == (2 * c.P + 1 if name == "one-tracked" and c.cost_type != W else 2), name


@pytest.mark.gpu
@pytest.mark.parametrize("N,P,cost", EDGE_SETS)
def test_compaction_edges(N, P, cost):
    """Each edge station alone and all of them in one batch: against the twin, inactive partitions exactly 0.0 in
    their own slots, and the same bits alone and in the batch."""
    c, named = _edge_case(N, P, cost)
    _check_edge_blocks(c, named)
    stations = list(named.values())
    b = mirror(c)
    batch = b.solve_bimpc_batch(*stack(stations))
    check_against_twin(c, stations, batch, twin(c, stations))
    for s, par in enumerate(stations):
        alone = b.solve_bimpc_batch(*stack([par]))
        for x, y in zip(alone[:3], batch[:3]):
            assert np.array_equal(x[0], y[s]), list(named)[s]
        for key in ("status", "iters", "objective"):
            assert alone[3][key][0] == batch[3][key][s], (list(named)[s], key)


@pytest.mark.parametrize("N,P,cost", EDGE_SETS)
def test_twin_compaction_edges_against_oracle(N, P, cost):
    c, named = _edge_case(N, P, cost)
    _check_edge_blocks(c, named)
    # the oracle on a few of them (each takes about a second at (16, 12), more at (12, 32))
    picks = ["none", "none-tracked", "one-small-first", "one-large-last", "half-tracked"] if P < 32 else ["nb33", "nb65"]
    stations = [named[k] for k in picks]
    ws, wl, ug, info = twin(c, stations)
    assert (info["status"] == 0).all()
    for s, par in enumerate(stations):
        check_against_oracle(c, par, ws[s], wl[s], ug[s])
        assert np.all(np.stack([ws[s], wl[s]])[inactive_slots(c, par)] == 0.0)


# ----------------------------------------------------------------------------------- 3. mixed persistent batch, bitwise
def mixed_batch(c, S, rng):
    """S stations whose kinds (active counts, tracked empties, an infeasible one now and then) are drawn at random,
    so that consecutive stations of one persistent CTA mostly differ in their block count."""
    P = c.P
    kinds = ["full", "draw", "half", "third", "one-small", "one-large", "none", "none-tracked", "half-tracked",
             "infeasible"]
    make = {
        "full": lambda: with_active(rng, c, 2 * P),
        "draw": lambda: draw_station(rng, c),
        "half": lambda: with_active(rng, c, P),
        "third": lambda: with_active(rng, c, 2 * P // 3),
        "one-small": lambda: draw_station(rng, c, active_s=[int(rng.integers(P))], active_l=[]),
        "one-large": lambda: draw_station(rng, c, active_s=[], active_l=[int(rng.integers(P))]),
        "none": lambda: draw_station(rng, c, active_s=[], active_l=[]),
        "none-tracked": lambda: draw_station(rng, c, active_s=[], active_l=[], track_empty=True),
        "half-tracked": lambda: with_active(rng, c, P, track_empty=True),
        "infeasible": lambda: (lambda p: p[:7] + (p[7] * 10.0,))(draw_station(rng, c)),
    }
    # the infeasible kind runs to the iteration cap: keep it rare
    prob = np.array([1.0] * 9 + [0.2])
    ks = rng.choice(len(kinds), S, p=prob / prob.sum())
    return [kinds[k] for k in ks], [make[kinds[k]]() for k in ks]


def _dev_solve(b, stations, with_objective):
    """bimpc_solve_batch_dev on torch tensors, on a non-default stream."""
    import torch
    dev = torch.device("cuda", b.device)
    arrs = stack(stations)
    S, P, N = len(stations), b.P, b.N
    ins = [torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device=dev) for a in arrs]
    out = {"ws": torch.full((S, P, N), -1.0, dtype=torch.float64, device=dev),
           "wl": torch.full((S, P, N), -1.0, dtype=torch.float64, device=dev),
           "ug": torch.full((S, N), -1.0, dtype=torch.float64, device=dev),
           "st": torch.full((S,), -1, dtype=torch.int32, device=dev),
           "it": torch.full((S,), -1, dtype=torch.int32, device=dev),
           "obj": torch.full((S,), -1.0, dtype=torch.float64, device=dev)}
    torch.cuda.synchronize(dev)
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        rc = b._lib.bimpc_solve_batch_dev(b._h, S, *[t.data_ptr() for t in ins],
                                          *[out[k].data_ptr() for k in ("ws", "wl", "ug", "st", "it")],
                                          out["obj"].data_ptr() if with_objective else None,
                                          C.c_void_p(stream.cuda_stream))
    assert rc == 0, rc
    stream.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.gpu
def test_mixed_persistent_batch_is_bitwise_station_local():
    """At P_max(24) = 37 (one CTA per SM) a batch of 1,536 stations makes every CTA solve about ten stations in the
    same scratch, of different block counts.  Every station must come out with the bits it gets alone, and the
    device entry point (caller's tensors, non-default stream, with and without the objective) with the bits of the
    host entry point."""
    import torch
    c = consts(24, 37, U)
    S = 1536
    rng = np.random.default_rng(2024)
    kinds, stations = mixed_batch(c, S, rng)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert S > 2 * sms
    b = mirror(c)
    with pytest.warns(RuntimeWarning):  # the infeasible stations
        ws, wl, ug, info = b.solve_bimpc_batch(*stack(stations))
    assert np.all((info["status"] == 0) == (np.array(kinds) != "infeasible")), info["status"]
    # solo solves: every kind, and mostly second and later stations of their CTA (index >= one per SM)
    sample = set(rng.choice(np.arange(sms, S), 200, replace=False).tolist())
    for k in set(kinds):
        sample.update([i for i, kk in enumerate(kinds) if kk == k][:2])
    for s in sorted(sample):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            a = b.solve_bimpc_batch(*stack([stations[s]]))
        assert np.array_equal(a[0][0], ws[s]) and np.array_equal(a[1][0], wl[s]) and np.array_equal(a[2][0], ug[s]), \
            (s, kinds[s])
        for key in ("status", "iters", "objective"):
            assert a[3][key][0] == info[key][s], (s, kinds[s], key)
    for with_objective in (True, False):
        d = _dev_solve(b, stations, with_objective)
        assert np.array_equal(d["ws"], ws) and np.array_equal(d["wl"], wl) and np.array_equal(d["ug"], ug)
        assert np.array_equal(d["st"], info["status"]) and np.array_equal(d["it"], info["iters"])
        if with_objective:
            assert np.array_equal(d["obj"], info["objective"])
        else:
            assert np.all(d["obj"] == -1.0)  # NULL: nothing written


# ------------------------------------------------------------------------------------ 4. constants at the asserts' edge
# exp_rate = inf (the reference's "np.Inf if only the cost at the final timestep is needed"): stage weights 0, ..., 0, 1.
# u_g bar against the oracle: 1e-4 instead of 2e-5.  At (48, 4) the kernel's algorithm stops (tol 1e-9) 5.3e-5 away
# from the oracle in u_g; both points pass the NNLS certificate, the kernel's with the larger residuals (stationarity
# 1.2e-8 against 1.7e-9, complementarity 7.9e-9 against 2.1e-10), and a tol-1e-12 run of the same algorithm ends
# within 1.2e-6 of the oracle.  The gap is the stopping tolerance in a direction the final-stage-only cost leaves
# flat, not an error of the kernel; the certificate keeps the point honest.
EXP_INF_UG_BAR = 1e-4
EXP_INF = [pytest.param(24, 12, id="N24-P12"), pytest.param(48, 4, id="N48-P4")]


def _exp_inf_stations(N, P):
    c = consts(N, P, E, exp_rate=np.inf)
    rng = np.random.default_rng(N * 100 + P)
    return c, [draw_station(rng, c) for _ in range(3)] + [with_active(rng, c, P, track_empty=True)]


@pytest.mark.gpu
@pytest.mark.parametrize("N,P", EXP_INF)
def test_exp_rate_inf(N, P):
    c, stations = _exp_inf_stations(N, P)
    assert bo.stage_weights(c).tolist() == [0.0] * (N - 1) + [1.0]
    gpu = mirror(c).solve_bimpc_batch(*stack(stations))
    check_against_twin(c, stations, gpu, twin(c, stations))
    ws, wl, ug, _ = gpu
    check_against_oracle(c, stations[0], ws[0], wl[0], ug[0], ug_bar=EXP_INF_UG_BAR, multipliers=True)


@pytest.mark.parametrize("N,P", EXP_INF)
def test_twin_exp_rate_inf_against_oracle(N, P):
    c, stations = _exp_inf_stations(N, P)
    ws, wl, ug, info = twin(c, stations[:1])
    assert info["status"][0] == 0
    check_against_oracle(c, stations[0], ws[0], wl[0], ug[0], ug_bar=EXP_INF_UG_BAR, multipliers=True)


@pytest.mark.gpu
def test_exp_rate_one_is_unweighted_bitwise():
    """exp_rate = 1 makes every EXP_UNWEIGHTED stage weight exactly 1.0, and the cost type is read nowhere else."""
    cu, ce = consts(24, 12, U), consts(24, 12, E, exp_rate=1.0)
    rng = np.random.default_rng(5)
    stations = [draw_station(rng, cu) for _ in range(3)] + [with_active(rng, cu, 12, track_empty=True),
                                                            draw_station(rng, cu, active_s=[], active_l=[],
                                                                         track_empty=True)]
    a = mirror(cu).solve_bimpc_batch(*stack(stations))
    b = mirror(ce).solve_bimpc_batch(*stack(stations))
    for x, y in zip(a[:3], b[:3]):
        assert np.array_equal(x, y)
    for key in ("status", "iters", "objective"):
        assert np.array_equal(a[3][key], b[3][key])
    assert (a[3]["status"] == 0).all()


DEGENERATE = [pytest.param({"delta": 0.0}, U, id="delta0-U"), pytest.param({"delta": 0.0}, W, id="delta0-W"),
              pytest.param({"c_g": 0.0}, U, id="c_g0-U"), pytest.param({"c_g": 0.0}, E, id="c_g0-E")]


def _degenerate(kw, cost):
    c = consts(16, 12, cost, **kw)
    rng = np.random.default_rng(17 + cost)
    return c, [draw_station(rng, c) for _ in range(3)]


@pytest.mark.gpu
@pytest.mark.parametrize("kw,cost", DEGENERATE)
def test_degenerate_costs(kw, cost):
    """delta = 0 or c_g = 0: the optimum is not unique, so only objective and feasibility are compared."""
    c, stations = _degenerate(kw, cost)
    ws, wl, ug, info = mirror(c).solve_bimpc_batch(*stack(stations))
    ref = twin(c, stations)
    assert (info["status"] == 0).all() and (ref[3]["status"] == 0).all()
    for s, par in enumerate(stations):
        k = bo.kkt_certificate(c, par, ws[s], wl[s], ug[s], multipliers=False)
        assert k["max_violation"] <= 1e-8
        assert abs(k["objective"] - ref[3]["objective"][s]) <= 1e-8 * max(1.0, abs(k["objective"]))
        assert abs(k["objective"] - info["objective"][s]) <= 1e-9 * max(1.0, abs(k["objective"]))
    _, _, _, io = bo.solve_ipm(c, *stations[0])
    assert abs(info["objective"][0] - io["objective"]) <= 1e-7 * max(1.0, abs(io["objective"]))


@pytest.mark.parametrize("kw,cost", DEGENERATE)
def test_twin_degenerate_costs_against_oracle(kw, cost):
    c, stations = _degenerate(kw, cost)
    ws, wl, ug, info = twin(c, stations[:1])
    assert info["status"][0] == 0
    _, _, _, io = bo.solve_ipm(c, *stations[0])
    k = bo.kkt_certificate(c, stations[0], ws[0], wl[0], ug[0], multipliers=False)
    assert k["max_violation"] <= 1e-8
    assert abs(k["objective"] - io["objective"]) <= 1e-7 * max(1.0, abs(io["objective"]))


# ------------------------------------------------------------------------------------------- 5. binding constraints
def slacks(c, par, w_s, w_l, u_g):
    """Smallest slack of each constraint family at a point (w at 0 and w_max over the partitions with EVs)."""
    Mp_s, Mp_l, b_s, b_l, _, _, x0, dem = par
    d = c.theta_s * Mp_s @ b_s + c.theta_l * Mp_l @ b_l
    u_b = u_g - dem - c.theta_s * Mp_s @ w_s - c.theta_l * Mp_l @ w_l
    lim = c.u_b_max - d * (np.arange(c.N) == 0)
    x = x0 + np.cumsum(u_b)
    act = np.concatenate([Mp_s > 0, Mp_l > 0])
    w = np.concatenate([w_s, w_l])[act]
    w_max = np.concatenate([np.full(c.P, c.w_max_s), np.full(c.P, c.w_max_l)])[act][:, None]
    inf = np.inf
    return {"w=0": w.min() if w.size else inf, "w=w_max": (w_max - w).min() if w.size else inf,
            "u_g=0": u_g.min(), "u_g=u_g_max": (c.u_g_max - u_g).min(), "u_b=+u_b_max": (lim - u_b).min(),
            "u_b=-u_b_max": (u_b + lim).min(), "x=d": (x - d).min(), "x=x_max-d": (c.x_max - d - x).min()}


def binding_case(name, cost):
    """(consts, station, the families that must be binding) of one scenario at (16, 12)."""
    c = consts(16, 12, cost)
    rng = np.random.default_rng(3)
    base = draw_station(rng, c)
    if name == "w-and-state":  # the drawn station: w at both bounds, the battery both empty and full
        return c, base, ["w=0", "w=w_max", "x=d", "x=x_max-d"]
    if name == "u_g-zero":  # no EVs, no demand, a charged battery: nothing to generate
        par = draw_station(rng, c, active_s=[], active_l=[])
        return c, par[:6] + (0.1, np.zeros(c.N)), ["u_g=0"]
    if name == "u_g-max":  # four times the EVs: generation runs at its limit while they charge
        return c, (base[0] * 4, base[1] * 4) + base[2:], ["u_g=u_g_max"]
    if name == "battery-rate":  # a slow battery under a demand that alternates with zero
        c.u_b_max = 0.02
        return c, base[:7] + (np.where(np.arange(c.N) % 2 == 0, base[7], 0.0),), ["u_b=+u_b_max", "u_b=-u_b_max"]
    raise KeyError(name)


BINDING = [pytest.param(n, cost, id=f"{n}-{COST[cost]}") for n, costs in
           (("w-and-state", (U, W)), ("u_g-zero", (U, E)), ("u_g-max", (U, W)), ("battery-rate", (U, E, W)))
           for cost in costs]


@pytest.mark.parametrize("name,cost", BINDING)
def test_twin_binding_scenario(name, cost):
    """Each scenario really has the families it names binding (slack <= 1e-7) at the twin's solution, which the
    dense oracle confirms."""
    c, par, fams = binding_case(name, cost)
    ws, wl, ug, info = twin(c, [par])
    assert info["status"][0] == 0
    sl = slacks(c, par, ws[0], wl[0], ug[0])
    assert all(sl[f] <= 1e-7 for f in fams), sl
    check_against_oracle(c, par, ws[0], wl[0], ug[0])


@pytest.mark.gpu
@pytest.mark.parametrize("name,cost", BINDING)
def test_binding_scenario(name, cost):
    c, par, fams = binding_case(name, cost)
    ref = twin(c, [par])
    sl = slacks(c, par, ref[0][0], ref[1][0], ref[2][0])
    assert all(sl[f] <= 1e-7 for f in fams), sl
    gpu = mirror(c).solve_bimpc_batch(*stack([par]))
    check_against_twin(c, [par], gpu, ref)
    sl = slacks(c, par, gpu[0][0], gpu[1][0], gpu[2][0])
    assert all(-1e-8 <= sl[f] <= 1e-7 for f in fams), sl


# ------------------------------------------------------------------------------- 6. envelope boundary and refusals
def test_p_max_restatement_matches_the_b200_envelope():
    assert [p_max(N, B200_OPTIN) for N in (1, 24, 48)] == [46, 37, 30]


@pytest.mark.gpu
def test_envelope_boundary_and_refusals():
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    c = consts(K_MAX_N, 2)
    assert mirror(c).solve_bimpc_batch(*stack([draw_station(np.random.default_rng(1), c)]))[3]["status"][0] == 0
    with pytest.raises(ValueError):
        mirror(consts(K_MAX_N + 1, 2))
    for N in (1, 24, 48):
        P = p_max(N, optin)
        with pytest.raises(ValueError):
            mirror(consts(N, P + 1))
        # a refused create leaves nothing behind: the next create and solve work
        c = consts(N, P, U)
        stations = [draw_station(np.random.default_rng(N), c)]
        gpu = mirror(c).solve_bimpc_batch(*stack(stations))
        check_against_twin(c, stations, gpu, twin(c, stations), cert=False)


@pytest.mark.gpu
def test_two_handles_alive_alternately():
    """A P_max handle and a small one at N = 24 share the kernel's opt-in attribute: used alternately, each gives the
    bits it gives alone."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    cb, cs = consts(24, p_max(24, optin), U), consts(24, 3, U)
    rng = np.random.default_rng(9)
    sb = [draw_station(rng, cb) for _ in range(3)]
    ss = [draw_station(rng, cs) for _ in range(3)]
    alone_b = mirror(cb).solve_bimpc_batch(*stack(sb))
    alone_s = mirror(cs).solve_bimpc_batch(*stack(ss))
    hb, hs = mirror(cb), mirror(cs)
    for _ in range(2):
        for h, st, ref in ((hs, ss, alone_s), (hb, sb, alone_b)):
            out = h.solve_bimpc_batch(*stack(st))
            for x, y in zip(out[:3], ref[:3]):
                assert np.array_equal(x, y)
            assert np.array_equal(out[3]["iters"], ref[3]["iters"]) and (out[3]["status"] == 0).all()


# ----------------------------------------------------------------------------------------------------- 7. status paths
@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 5])
def test_iteration_cap(k):
    c = consts(16, 12, E)
    rng = np.random.default_rng(k)
    stations = [draw_station(rng, c) for _ in range(3)]
    b = mirror(c)
    b.set_options(max_iter=k)
    with pytest.warns(RuntimeWarning, match="not solved"):
        ws, wl, ug, info = b.solve_bimpc_batch(*stack(stations))
    ref = twin(c, stations, max_iter=k)
    assert (info["status"] == 1).all() and (info["iters"] == k).all()
    assert np.array_equal(info["status"], ref[3]["status"]) and np.array_equal(info["iters"], ref[3]["iters"])


@pytest.mark.gpu
def test_tight_tolerance_converges():
    c = consts(16, 12)
    par = draw_station(np.random.default_rng(7), c)
    b = mirror(c)
    b.set_options(tol=1e-12)
    ws, wl, ug, info = b.solve_bimpc_batch(*stack([par]))
    assert info["status"][0] == 0 and info["iters"][0] <= 40


@pytest.mark.gpu
def test_infeasible_station_leaves_its_neighbours_alone():
    c = consts(16, 12, U)
    rng = np.random.default_rng(21)
    stations = [draw_station(rng, c) for _ in range(5)]
    bad = stations[2][:7] + (stations[2][7] * 10.0,)
    b = mirror(c)
    clean = b.solve_bimpc_batch(*stack(stations))
    with pytest.warns(RuntimeWarning):
        mixed = b.solve_bimpc_batch(*stack(stations[:2] + [bad] + stations[3:]))
    assert mixed[3]["status"][2] != 0
    keep = [0, 1, 3, 4]
    for x, y in zip(mixed[:3], clean[:3]):
        assert np.array_equal(x[keep], y[keep])
    for key in ("status", "iters", "objective"):
        assert np.array_equal(mixed[3][key][keep], clean[3][key][keep])


def nonfinite_stations(c):
    """(label, station) with one NaN or inf in demand, x0, gamma, Mp or beta - in a populated partition and in an
    empty one (which the kernel would otherwise leave out of its system unread)."""
    base = draw_station(np.random.default_rng(4), c)  # P > 3: small partition P-1 and large partition 0 are empty
    out = []
    for bad in (np.nan, np.inf):
        for label, idx, j in (("demand", 7, 3), ("x0", 6, None), ("gamma_sm", 4, 0), ("gamma_sm-empty", 4, -1),
                              ("gamma_lm-empty", 5, 0), ("Mp_s", 0, 1), ("Mp_l-empty", 1, 0), ("beta_l", 3, 2),
                              ("beta_s-empty", 2, -1)):
            par = [np.array(v, dtype=float) for v in base]
            if j is None:
                par[idx] = np.array(bad)
            else:
                par[idx][j] = bad
            out.append((f"{label}={bad}", tuple(par)))
    return out


def test_twin_rejects_nonfinite_inputs():
    for cost in (W, U, E):
        c = consts(16, 12, cost)
        for label, par in nonfinite_stations(c):
            assert twin(c, [par])[3]["status"][0] == 2, (COST[cost], label)


@pytest.mark.gpu
def test_nonfinite_inputs_never_converge():
    """fmax / fmin drop NaN in the residual maxima and the ratio test, and an empty partition is left out of the
    system: a NaN or inf input must still come back with status 2, through the mirror and the device entry point,
    without disturbing the other stations of its batch."""
    for cost in (W, U, E):
        c = consts(16, 12, cost)
        cases = nonfinite_stations(c)
        good = draw_station(np.random.default_rng(5), c)
        stations = [good] + [p for _, p in cases] + [good]
        b = mirror(c)
        with pytest.warns(RuntimeWarning):
            ws, wl, ug, info = b.solve_bimpc_batch(*stack(stations))
        assert info["status"][0] == 0 and info["status"][-1] == 0
        assert np.array_equal(ws[0], ws[-1]) and np.array_equal(ug[0], ug[-1])
        for (label, _), st in zip(cases, info["status"][1:-1]):
            assert st == 2, (COST[cost], label)
        d = _dev_solve(b, stations, True)
        assert np.array_equal(d["st"], info["status"])
