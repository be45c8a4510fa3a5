"""Fleets whose stations hold different numbers of EVs: the *_sized_dev entry points of
include/fleet_b200.h against NumPy twins, and ChargingStationFleet(nevs=...) against the
single-station mirror, against the uniform fleet, against one-station fleets and at fleet scale.

Layout under test: per EV type the state is [S, M] with M = max(nevs); station s owns the first
nevs[s] slots of its row and the padding is never read or written; the EV-sorted arrays hold
sum(nevs) EVs.  The twins below are those of tests/test_fleet_kernels_gpu.py restricted to the
first nevs[s] slots of each row, and are held to the same bars (bit for bit, except the three
quantities that may hold an FMA)."""
import copy
import dataclasses

import numpy as np
import pytest

import test_fleet_gpu as closed_loop_tests
import test_fleet_kernels_gpu as kt
from chargingstation.charging_station import assign_partitions, partition_edges
from chargingstation.settings import MAX_INITIAL_SOC, MIN_INITIAL_SOC

THETA_S, THETA_L = 10.0, 50.0  # theta of the two EV types in the closed-loop scenarios
FILL = -7                      # what every output buffer holds before a call


# ============================================================================ NumPy twins
def twin_partition_sized(edges, y, idx, nevs):
    """charging_station.py:111-116 and the group sort of charging_station.py:221-223 on the first
    nevs[s] slots of every row; padding indices keep their values."""
    S, M = y.shape
    P = len(edges) - 1
    idx = np.array(idx, dtype=np.int64)
    per_station = np.zeros((S, P), dtype=np.int64)
    for s in range(S):
        n = int(nevs[s])
        assign_partitions(y[s, :n], edges, idx[s, :n])  # idx[s, :n] is a view: updated in place
        per_station[s] = np.bincount(idx[s, :n], minlength=P)
    counts = per_station.T.reshape(P * S)
    off = np.concatenate([[0], np.cumsum(counts)])
    off_rebased = np.stack([off[p * S: p * S + S + 1] - off[p * S] for p in range(P)])
    B = int(np.sum(nevs))
    y_sorted, perm = np.empty(B), np.empty(B, dtype=np.int64)
    for s in range(S):
        n = int(nevs[s])
        order = np.argsort(idx[s, :n], kind="stable")
        local = np.concatenate([[0], np.cumsum(per_station[s])])
        for p in np.nonzero(per_station[s])[0]:
            b0, seg = off[p * S + s], order[local[p]: local[p + 1]]
            y_sorted[b0: b0 + len(seg)] = y[s, seg]
            perm[b0: b0 + len(seg)] = seg
    return dict(idx=idx, counts=counts, off=off, off_rebased=off_rebased, y_sorted=y_sorted, perm=perm)


def twin_apply_charge_sized(P, off, perm, w0_sorted, y, ncharged, full_level, rng_seed, ev_type, t, nevs):
    """twin_apply_charge with departures and arrivals on the first nevs[s] slots only; the mask
    keeps FILL on the padding."""
    S, M = y.shape
    real = np.arange(M)[None, :] < np.asarray(nevs)[:, None]
    y = y.copy()
    w_sum, w_mean = np.zeros(S), np.zeros(P * S)
    for s in range(S):
        tot = 0.0
        for p in range(P):
            g = p * S + s
            b0, b1 = int(off[g]), int(off[g + 1])
            w = w0_sorted[b0:b1]
            group = float(np.cumsum(w)[-1]) if b1 > b0 else 0.0
            y[s, perm[b0:b1]] += w
            w_mean[g] = group / (b1 - b0) if b1 > b0 else 0.0
            tot += group
        w_sum[s] = tot
    with np.errstate(invalid="ignore"):
        leave = (y > full_level) & real
    u = np.full((S, M), np.nan)
    if rng_seed >= 0:
        for s, ev in zip(*np.nonzero(leave)):
            u[s, ev] = kt.counter_uniform(rng_seed, ev_type, int(s), int(ev), t)
            y[s, ev] = MIN_INITIAL_SOC + (MAX_INITIAL_SOC - MIN_INITIAL_SOC) * u[s, ev]
    mask = np.where(real, leave, FILL).astype(np.int32)
    return dict(y=y, mask=mask, w_sum=w_sum, w_mean=w_mean, ncharged=ncharged + leave.sum(axis=1)), u


def twin_bimpc_params_sized(P, N_bi, N_lo, Bcap, eps_tol, lmbd_r, delta, counts, y0_rng, gamma_sm, x, profile, t):
    """twin_bimpc_params with each station's own capacity Bcap[s] (charging_station.py:170-171)."""
    out = kt.twin_bimpc_params(P, N_bi, N_lo, 1.0, eps_tol, lmbd_r, delta, counts, y0_rng, gamma_sm, x, profile, t)
    S = len(x)
    for k in ("s", "l"):
        out["Mp_" + k] = counts[0 if k == "s" else 1].reshape(P, S).T / Bcap[:, None]
    out["demand"] = profile[:, t: t + N_bi] / Bcap[:, None]
    return out


def twin_battery_sized(x, u_g, theta_s, theta_l, Bcap, w_sum_s, w_sum_l, profile, t):
    return x + (u_g[:, 0] + (-theta_s * w_sum_s - theta_l * w_sum_l - profile[:, t]) / Bcap)


# ============================================================================ inputs
def sizes(rng, S, M, kind):
    """EVs per station: "full" = M everywhere, "ones" = 1 everywhere, "mixed" = U{1..M} with 1 and
    M present (and 128, 129, 256, 257 where they fit: the trip boundaries of assign and departures)."""
    if kind == "full":
        return np.full(S, M, dtype=np.int64)
    if kind == "ones":
        return np.ones(S, dtype=np.int64)
    n = rng.integers(1, M + 1, S)
    special = [1, M] + [v for v in (128, 129, 256, 257) if v < M]
    k = min(S, len(special))
    n[:k] = special[:k]
    return n


def padded_socs(rng, S, M, edges, nevs):
    """kt.socs on the real slots; the padding holds SoCs inside a partition and far above the departure
    level (a kernel that read them would assign, sort or replace them)."""
    y, idx0 = kt.socs(rng, S, M, edges)
    pad = np.arange(M)[None, :] >= nevs[:, None]
    y[pad] = rng.uniform(edges[0], edges[-1], int(pad.sum()))
    return y, idx0, pad


# ============================================================================ device calls
class _SizedDev(kt._Dev):
    """kt._Dev plus the four sized entry points.  Sorted outputs get 16 guard slots past sum(nevs)."""

    GUARD = 16

    def partition_sized(self, edges, y, idx, nevs):
        torch = self.torch
        S, M = y.shape
        P = len(edges) - 1
        B = int(np.sum(nevs))
        d_edges, d_y, d_n = self.f64(edges), self.f64(y), self.i32(nevs)
        out = dict(idx=self.i32(idx), counts=self.fill((P * S,), FILL, torch.int32),
                   off=self.fill((P * S + 1,), FILL, torch.int32), off_rebased=self.fill((P, S + 1), FILL, torch.int32),
                   y_sorted=self.fill((B + self.GUARD,), float(FILL), torch.float64),
                   perm=self.fill((B + self.GUARD,), FILL, torch.int32))
        self.call("fleet_partition_sized_dev", 3, S, M, P, d_n.data_ptr(), d_edges.data_ptr(), d_y.data_ptr(),
                  out["idx"].data_ptr(), out["counts"].data_ptr(), out["off"].data_ptr(),
                  out["off_rebased"].data_ptr(), out["y_sorted"].data_ptr(), out["perm"].data_ptr())
        got = self.host(out)
        for k in ("y_sorted", "perm"):
            assert np.all(got[k][B:] == FILL), k + " written past sum(nevs)"
            got[k] = got[k][:B]
        return got

    def apply_charge_sized(self, P, off, perm, w0_sorted, y, ncharged, full_level, rng_seed, ev_type, t, nevs):
        torch = self.torch
        S, M = y.shape
        ins = dict(off=self.i32(off), perm=self.i32(perm), w0=self.f64(w0_sorted), nevs=self.i32(nevs))
        out = dict(y=self.f64(y), ncharged=self.i32(ncharged), w_sum=self.fill((S,), float(FILL), torch.float64),
                   mask=self.fill((S, M), FILL, torch.int32), w_mean=self.fill((P * S,), float(FILL), torch.float64))
        self.call("fleet_apply_charge_sized_dev", 1, S, M, P, ins["nevs"].data_ptr(), full_level, MIN_INITIAL_SOC,
                  MAX_INITIAL_SOC, rng_seed, ev_type, t, ins["off"].data_ptr(), ins["perm"].data_ptr(),
                  ins["w0"].data_ptr(), out["y"].data_ptr(), out["mask"].data_ptr(), out["w_sum"].data_ptr(),
                  out["w_mean"].data_ptr(), out["ncharged"].data_ptr())
        return self.host(out)

    def bimpc_params_sized(self, P, N_bi, N_lo, Bcap, eps_tol, lmbd_r, delta, counts, y0_rng, gamma_sm, x, profile, t):
        torch = self.torch
        S, L = profile.shape
        ins = [self.i32(counts[0]), self.i32(counts[1]), self.f64(y0_rng[0]), self.f64(y0_rng[1]),
               self.f64(gamma_sm[0]), self.f64(gamma_sm[1]), self.f64(x), self.f64(profile)]
        d_bcap = self.f64(Bcap)
        names = ("Mp_s", "Mp_l", "beta_s", "beta_l", "gamma_s", "gamma_l")
        out = {k: self.fill((S, P), float(FILL), torch.float64) for k in names}
        out["x0"] = self.fill((S,), float(FILL), torch.float64)
        out["demand"] = self.fill((S, N_bi), float(FILL), torch.float64)
        self.call("fleet_bimpc_params_sized_dev", 1, S, P, N_bi, N_lo, d_bcap.data_ptr(), eps_tol, lmbd_r, delta[0],
                  delta[1], *[a.data_ptr() for a in ins[:7]], ins[7].data_ptr(), L, t,
                  *[out[k].data_ptr() for k in names + ("x0", "demand")])
        return self.host(out)

    def battery_sized(self, x, u_g, theta_s, theta_l, Bcap, w_sum_s, w_sum_l, profile, t):
        S, N_bi = u_g.shape
        ins = [self.f64(u_g), self.f64(w_sum_s), self.f64(w_sum_l), self.f64(profile)]
        d_bcap, d_x = self.f64(Bcap), self.f64(x)
        self.call("fleet_battery_sized_dev", 1, S, N_bi, theta_s, theta_l, d_bcap.data_ptr(),
                  *[a.data_ptr() for a in ins], profile.shape[1], t, d_x.data_ptr())
        return d_x.cpu().numpy()


@pytest.fixture(scope="module")
def dev():
    import torch

    from chargingstation import _native
    return _SizedDev(torch, _native.load())


# ============================================================================ CPU: sized twins against uniform ones
@pytest.mark.parametrize("S,M,P", [(1, 1, 1), (3, 40, 6), (5, 300, 12)])
def test_sized_twins_with_every_station_full_are_the_uniform_twins(S, M, P):
    rng = np.random.default_rng(S + M + P)
    edges = partition_edges(MIN_INITIAL_SOC, kt.Y_MAX, P)
    y, idx0 = kt.socs(rng, S, M, edges)
    full = np.full(S, M)
    tw, tws = kt.twin_partition(edges, y, idx0), twin_partition_sized(edges, y, idx0, full)
    kt.check_partition(tws, tw)
    w0 = rng.uniform(0.0, 0.05, S * M)
    args = (P, tw["off"], tw["perm"], w0, y, np.zeros(S, dtype=np.int64), kt.FULL_LEVEL, 3, 1, 2)
    (a, ua), (b, ub) = kt.twin_apply_charge(*args), twin_apply_charge_sized(*args, full)
    for k in a:
        kt.assert_same(b[k], a[k], k)
    kt.assert_same(ub, ua, "u")


def test_sized_partition_twin_leaves_the_padding_alone():
    rng = np.random.default_rng(1)
    S, M, P = 6, 50, 6
    edges = partition_edges(MIN_INITIAL_SOC, kt.Y_MAX, P)
    nevs = np.array([1, 50, 7, 49, 25, 3])
    y, idx0, pad = padded_socs(rng, S, M, edges, nevs)
    tw = twin_partition_sized(edges, y, idx0, nevs)
    kt.assert_same(tw["idx"][pad], idx0[pad], "idx padding")
    assert tw["off"][-1] == nevs.sum()
    assert np.all(tw["counts"].reshape(P, S).sum(axis=0) == nevs)
    for s in range(S):
        one = kt.twin_partition(edges, y[s:s + 1, :nevs[s]], idx0[s:s + 1, :nevs[s]])
        kt.assert_same(tw["idx"][s, :nevs[s]], one["idx"][0], "idx")


# ============================================================================ GPU: sized kernels against the twins
# (S, M, P, sizes): assign trips = ceil(nevs[s] / 128), departure trips = ceil(nevs[s] / 256)
SIZED_GRID = [
    (1, 1, 1, "full"), (1, 300, 12, "ones"), (3, 40, 6, "mixed"), (7, 257, 12, "mixed"), (2, 1000, 64, "mixed"),
    (85, 500, 12, "mixed"), (86, 257, 12, "ones"), (1025, 257, 64, "mixed"), (5000, 127, 12, "mixed"),
    (4096, 900, 12, "mixed"),   # the ragged closed-loop shape: U{1..900}
    (4096, 500, 12, "full"),    # the benchmark's fleet through the sized entry points
]


def _sized_id(c):
    S, M, P, kind = c
    return f"S{S}-M{M}-P{P}-{kind}"


@pytest.mark.gpu
@pytest.mark.parametrize("S,M,P,kind", SIZED_GRID, ids=[_sized_id(c) for c in SIZED_GRID])
def test_partition_sized_matches_twin(dev, S, M, P, kind):
    rng = np.random.default_rng(S * 7 + M * 3 + P)
    edges = partition_edges(MIN_INITIAL_SOC, kt.Y_MAX, P)
    nevs = sizes(rng, S, M, kind)
    y, idx0, pad = padded_socs(rng, S, M, edges, nevs)
    got = dev.partition_sized(edges, y, idx0, nevs)
    want = twin_partition_sized(edges, y, idx0, nevs)
    kt.check_partition(got, want)
    kt.assert_same(got["idx"][pad], idx0[pad], "idx padding")
    assert got["off"][-1] == nevs.sum()


@pytest.mark.gpu
@pytest.mark.parametrize("S,M,P,kind", SIZED_GRID, ids=[_sized_id(c) for c in SIZED_GRID])
def test_apply_charge_sized_matches_twin(dev, S, M, P, kind):
    rng = np.random.default_rng(S * 11 + M * 5 + P)
    edges = partition_edges(MIN_INITIAL_SOC, kt.Y_MAX, P)
    nevs = sizes(rng, S, M, kind)
    real = np.arange(M)[None, :] < nevs[:, None]
    y = rng.uniform(MIN_INITIAL_SOC, kt.FULL_LEVEL, (S, M))
    y[-1, nevs[-1] - 1] = np.nextafter(kt.FULL_LEVEL, 1.0)  # at least one departure
    y[~real] = 0.95  # padding far above the departure level
    tw = twin_partition_sized(edges, y, rng.integers(0, P, (S, M)), nevs)
    B = int(nevs.sum())
    w0 = rng.uniform(0.0, 0.05, B)
    w0[rng.random(B) < 0.05] = 0.0
    ncharged = rng.integers(0, 1000, S)
    seed, ev_type, t = 1234 + S, int(rng.integers(2)), int(rng.integers(96))
    for rng_seed in (seed, -1):
        want, u = twin_apply_charge_sized(P, tw["off"], tw["perm"], w0, y, ncharged, kt.FULL_LEVEL, rng_seed, ev_type,
                                          t, nevs)
        got = dev.apply_charge_sized(P, tw["off"], tw["perm"], w0, y, ncharged, kt.FULL_LEVEL, rng_seed, ev_type, t,
                                     nevs)
        assert want["mask"][real].any()
        kt.check_apply_charge(got, want, u)
        kt.assert_same(got["y"][~real], y[~real], "y padding")
        assert np.all(got["mask"][~real] == FILL)


@pytest.mark.gpu
@pytest.mark.parametrize("S,M,P", [(3, 1000, 12), (1025, 257, 64), (64, 300, 12)])
def test_partition_sized_degenerate_groups(dev, S, M, P):
    """Every station has all its real EVs in one partition (a different one per station), so its
    other P - 1 groups are empty; the padding SoCs lie in yet another partition."""
    rng = np.random.default_rng(S + M + P)
    edges = partition_edges(MIN_INITIAL_SOC, kt.Y_MAX, P)
    nevs = sizes(rng, S, M, "mixed")
    q = rng.integers(0, P, S)
    y = rng.uniform(edges[q], edges[q + 1], (M, S)).T
    pad = np.arange(M)[None, :] >= nevs[:, None]
    y[pad] = ((edges[(q + 1) % P] + edges[(q + 1) % P + 1]) / 2)[:, None].repeat(M, axis=1)[pad]
    idx0 = rng.integers(0, P, (S, M))
    got = dev.partition_sized(edges, y, idx0, nevs)
    want = twin_partition_sized(edges, y, idx0, nevs)
    kt.check_partition(got, want)
    per = want["counts"].reshape(P, S)
    assert np.all(per[q, np.arange(S)] == nevs) and np.all(np.count_nonzero(per, axis=0) == 1)


PARAM_SHAPES = [(1, 1, 1, 1), (7, 12, 16, 12), (86, 64, 16, 12), (1025, 12, 48, 24), (4096, 12, 24, 24)]


@pytest.mark.gpu
@pytest.mark.parametrize("lmbd_r", [0.0, 24.0])
@pytest.mark.parametrize("S,P,N_bi,N_lo", PARAM_SHAPES, ids=[f"S{a}-P{b}-Nbi{c}-Nlo{d}" for a, b, c, d in PARAM_SHAPES])
def test_bimpc_params_sized_matches_twin(dev, S, P, N_bi, N_lo, lmbd_r):
    rng = np.random.default_rng(S + P + N_bi)
    L = N_bi + 5
    nevs = sizes(rng, S, 900, "mixed")
    Bcap = (THETA_S + THETA_L) * nevs.astype(np.float64)
    counts = [rng.integers(0, 40, P * S) * (rng.random(P * S) < 0.6) for _ in range(2)]
    y0_rng = [rng.uniform(0, 0.1, P * S) for _ in range(2)]
    gamma_sm = [rng.uniform(0.3, 0.6, P * S) for _ in range(2)]
    x, profile = rng.uniform(0, 0.3, S), rng.uniform(0, 400, (S, L)) * (nevs[:, None] / 500)
    args = (P, N_bi, N_lo, Bcap, 0.01, lmbd_r, (0.05, 0.025), counts, y0_rng, gamma_sm, x, profile, L - N_bi)
    got, want = dev.bimpc_params_sized(*args), twin_bimpc_params_sized(*args)
    for k in ("Mp_s", "Mp_l", "gamma_s", "gamma_l", "x0", "demand"):
        kt.assert_same(got[k], want[k], k)
    for k in ("beta_s", "beta_l"):
        kt.assert_within_ulps(got[k], want[k], want[k], k)
        kt.assert_same(got[k] == 0.0, want[k] == 0.0, k + " zero")


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 129, 5000])
def test_battery_sized_matches_twin(dev, S):
    rng = np.random.default_rng(S)
    N_bi, L = 16, 24
    nevs = sizes(rng, S, 900, "mixed")
    Bcap = (THETA_S + THETA_L) * nevs.astype(np.float64)
    x, u_g = rng.uniform(0, 0.3, S), rng.uniform(0, 0.2, (S, N_bi))
    ws, wl = rng.uniform(0, 0.05, S) * nevs, rng.uniform(0, 0.03, S) * nevs
    profile = rng.uniform(0, 2000, (S, L)) * (nevs[:, None] / 500)
    t = L - 1
    got = dev.battery_sized(x, u_g, THETA_S, THETA_L, Bcap, ws, wl, profile, t)
    want = twin_battery_sized(x, u_g, THETA_S, THETA_L, Bcap, ws, wl, profile, t)
    mag = np.max(np.abs([x, want, u_g[:, 0], THETA_S * ws / Bcap, THETA_L * wl / Bcap, profile[:, t] / Bcap]), axis=0)
    kt.assert_within_ulps(got, want, mag, "x")


@pytest.mark.gpu
@pytest.mark.parametrize("S,M,P", [(7, 257, 12), (4096, 500, 12)])
def test_sized_entry_points_with_uniform_sizes_give_the_bits_of_the_uniform_ones(dev, S, M, P):
    """nevs[s] = M and Bcap[s] = Bcap for every station reproduce the uniform entry points bit for bit."""
    rng = np.random.default_rng(S + M)
    edges = partition_edges(MIN_INITIAL_SOC, kt.Y_MAX, P)
    full = np.full(S, M)
    y, idx0 = kt.socs(rng, S, M, edges)
    a, b = dev.partition(edges, y, idx0), dev.partition_sized(edges, y, idx0, full)
    for k in a:
        kt.assert_same(b[k], a[k], k)
    y = rng.uniform(MIN_INITIAL_SOC, 0.84, (S, M))
    w0 = rng.uniform(0.0, 0.2, S * M)
    nc = rng.integers(0, 100, S)
    for seed in (5, -1):
        a = dev.apply_charge(P, b["off"], b["perm"], w0, y, nc, kt.FULL_LEVEL, seed, 1, 7)
        c = dev.apply_charge_sized(P, b["off"], b["perm"], w0, y, nc, kt.FULL_LEVEL, seed, 1, 7, full)
        for k in a:
            kt.assert_same(c[k].view(np.uint8), a[k].view(np.uint8), k)
    Bcap = (THETA_S + THETA_L) * M
    N_bi, N_lo, L = 24, 24, 30
    counts = [rng.integers(0, M // 4, P * S) for _ in range(2)]
    y0_rng, gamma_sm = [rng.uniform(0, 0.1, P * S)] * 2, [rng.uniform(0.3, 0.6, P * S)] * 2
    x, profile = rng.uniform(0, 0.3, S), rng.uniform(0, 400, (S, L))
    common = (0.01, 24.0, (0.05, 0.025), counts, y0_rng, gamma_sm, x, profile, 3)
    a = dev.bimpc_params(P, N_bi, N_lo, Bcap, *common)
    c = dev.bimpc_params_sized(P, N_bi, N_lo, np.full(S, Bcap), *common)
    for k in a:
        kt.assert_same(c[k].view(np.uint8), a[k].view(np.uint8), k)
    u_g, ws, wl = rng.uniform(0, 0.2, (S, N_bi)), rng.uniform(0, 25, S), rng.uniform(0, 15, S)
    a = dev.battery(x, u_g, THETA_S, THETA_L, Bcap, ws, wl, profile, 5)
    c = dev.battery_sized(x, u_g, THETA_S, THETA_L, np.full(S, Bcap), ws, wl, profile, 5)
    kt.assert_same(c.view(np.uint8), a.view(np.uint8), "x")


@pytest.mark.gpu
def test_sized_entry_points_refuse_null_sizes_and_launch_nothing(dev):
    torch, lib = dev.torch, dev.lib
    S, M, P, N_bi, L = 2, 4, 3, 4, 8
    keep = []

    def buf(dtype, n):
        t = torch.zeros(n, dtype=dtype, device="cuda")
        keep.append(t)
        return t.data_ptr()

    f, i = torch.float64, torch.int32
    g = [buf(f, 64) for _ in range(16)]
    gi = [buf(i, 64) for _ in range(6)]
    st = torch.cuda.current_stream().cuda_stream
    calls = {
        "partition": lambda n: lib.fleet_partition_sized_dev(0, S, M, P, n, *g[:2], *gi[:4], g[2], gi[4], st),
        "apply_charge": lambda n: lib.fleet_apply_charge_sized_dev(0, S, M, P, n, kt.FULL_LEVEL, 0.3, 0.5, 1, 0, 0,
                                                                   gi[0], gi[1], g[0], g[1], gi[2], g[2], g[3], gi[3],
                                                                   st),
        "bimpc_params": lambda b: lib.fleet_bimpc_params_sized_dev(0, S, P, N_bi, 4, b, 0.01, 0.0, 0.05, 0.025, gi[0],
                                                                   gi[1], *g[:6], L, 0, *g[6:14], st),
        "battery": lambda b: lib.fleet_battery_sized_dev(0, S, N_bi, 10.0, 50.0, b, *g[:4], L, 0, g[4], st),
    }
    ones_i = torch.ones(S, dtype=i, device="cuda")
    ones_f = torch.full((S,), 60.0, dtype=f, device="cuda")
    for name, call in calls.items():
        n0 = lib.lompc_launch_count()
        assert call(None) == kt.ERR_ARG, name
        assert lib.lompc_launch_count() == n0, name
        good = (ones_f if name in ("bimpc_params", "battery") else ones_i).data_ptr()
        assert call(good) == 0, name
        assert lib.lompc_launch_count() - n0 == (3 if name == "partition" else 1), name
    torch.cuda.synchronize()


# ============================================================================ GPU: the closed loop
MIRROR_SIZES = np.array([1, 9, 40, 120, 300])


def _ragged_demand(consts, nevs, rng=None):
    """consts.demand (made for 500 EVs) scaled by each station's size / 500, and when rng is given
    shifted by U{0..23} h and scaled by U(0.9, 1.1) per station as in test_fleet_gpu."""
    rows = []
    for n in nevs:
        d = consts.demand
        if rng is not None:
            d = np.roll(d, int(rng.integers(24))) * rng.uniform(0.9, 1.1)
        rows.append(d * (n / 500))
    return np.stack(rows)


@pytest.mark.gpu
@pytest.mark.parametrize("price_type", ["linear-convex", "linear"])
@pytest.mark.parametrize("N_bi,N_lo", [(16, 12), (24, 24)], ids=["Nlo12", "Nlo24"])
def test_ragged_fleet_equals_single_station_runs(price_type, N_bi, N_lo):
    """Every station of a fleet of sizes {1, 9, 40, 120, 300} against ChargingStation with that
    nEVs_per_EV_type, its demand and seed + s: the assertions and bars of
    test_fleet_gpu.py::test_fleet_reference_chain_equals_single_station_runs."""
    from chargingstation.charging_station import ChargingStation
    from chargingstation.fleet import ChargingStationFleet
    Tf, P = 4, 12
    S = len(MIRROR_SIZES)
    consts = closed_loop_tests._consts(Tf, N_bi, N_lo, 500, P, 1, price_type)
    demand = np.array([1.0, 0.97, 1.04, 0.99, 1.02])[:, None] * _ragged_demand(consts, MIRROR_SIZES)
    fleet = ChargingStationFleet(consts, S, demand=demand, seed=100, rng="numpy", chain="reference",
                                 nevs=MIRROR_SIZES)
    assert fleet.M == 300 and fleet.B == MIRROR_SIZES.sum()
    fleet.simulate()
    for s, n in enumerate(MIRROR_SIZES):
        c = copy.copy(consts)
        c.nEVs_per_EV_type = int(n)
        c.demand = demand[s]
        np.random.seed(100 + s)
        one = ChargingStation(c)
        ref = one.simulate()
        got = fleet.station_logs(s)
        assert got["constants"].nEVs_per_EV_type == n
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


def _state(fleet):
    """Everything a fleet carries from step to step, and its logs, on the host."""
    out = {"log_" + k: v.cpu().numpy() for k, v in fleet.log.items()}
    for k in ("s", "l"):
        for name in ("y", "idx", "ncharged", "prices", "prev"):
            out[f"{name}_{k}"] = getattr(fleet, name)[k].cpu().numpy()
    out["x"] = fleet.x.cpu().numpy()
    return out


def _assert_same_state(a, b):
    assert a.keys() == b.keys()
    for k in a:
        kt.assert_same(a[k].view(np.uint8), b[k].view(np.uint8), k)


@pytest.mark.gpu
@pytest.mark.parametrize("rng", ["numpy", "device"])
@pytest.mark.parametrize("chain", ["reference", "partition"])
def test_uniform_nevs_is_the_default_fleet(rng, chain):
    from chargingstation.fleet import ChargingStationFleet
    Tf, S, M, P = 3, 4, 40, 6
    consts = closed_loop_tests._consts(Tf, 16, 12, M, P, 1)
    demand = np.array([1.0, 0.97, 1.04, 1.01])[:, None] * consts.demand[None, :]
    y0 = np.random.default_rng(2).uniform(MIN_INITIAL_SOC, 0.84, (2, S, M))  # EVs leave within the three steps
    runs = []
    for nevs in (None, [M] * S):
        f = ChargingStationFleet(consts, S, demand=demand, seed=11, rng=rng, chain=chain, nevs=nevs)
        for i, k in enumerate(("s", "l")):
            f.y[k].copy_(f.torch.from_numpy(y0[i]))
        f.simulate()
        assert f.M == M and f.B == S * M and np.array_equal(f.nevs, np.full(S, M))
        assert f.station_logs(1)["constants"] is consts
        runs.append(_state(f))
    _assert_same_state(*runs)
    assert int(runs[0]["ncharged_s"].sum() + runs[0]["ncharged_l"].sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("chain", ["reference", "partition"])
def test_station_does_not_depend_on_its_neighbours(chain):
    """Station s of a ragged fleet (NumPy RNG) gives the bits of a one-station fleet of nevs[s] EVs
    with seed + s, in every log, its state and its prices; the padding of its rows stays untouched."""
    from chargingstation.fleet import ChargingStationFleet
    Tf, P = 4, 12
    nevs = np.array([120, 1, 40, 9, 300, 75])
    consts = closed_loop_tests._consts(Tf, 16, 12, 500, P, 2)
    demand = _ragged_demand(consts, nevs, np.random.default_rng(8))
    fleet = ChargingStationFleet(consts, len(nevs), demand=demand, seed=100, rng="numpy", chain=chain, nevs=nevs)
    fleet.simulate()
    big = _state(fleet)
    S, M = len(nevs), fleet.M
    for s, n in enumerate(nevs):
        one = ChargingStationFleet(dataclasses.replace(consts, nEVs_per_EV_type=int(n)), 1, demand=demand[s:s + 1],
                                   seed=100 + s, rng="numpy", chain=chain)
        one.simulate()
        small = _state(one)
        for k, v in small.items():
            if k.startswith("log_"):
                mine = big[k][..., s:s + 1]
            elif k[:-2] in ("y", "idx"):
                mine = big[k][s:s + 1, :n]
                pad = big[k][s, n:]
                assert np.all(np.isnan(pad)) if k[0] == "y" else np.all(pad == 0), (s, k)
            elif k[:-2] == "prices":
                mine = big[k].reshape(P, S, -1)[:, s]
            else:
                mine = big[k][s:s + 1]
            kt.assert_same(mine.view(np.uint8), v.view(np.uint8), (s, k))


@pytest.mark.gpu
@pytest.mark.parametrize("chain", ["reference", "partition"])
def test_ragged_fleet_device_rng_properties(chain):
    """64 stations of 1..200 EVs, device RNG: every station keeps its own population, converged groups
    meet the robustness bound, every BiMPC is solved, the padding is never written, and two runs are
    bit-identical."""
    from chargingstation.fleet import ChargingStationFleet
    Tf, S, P = 5, 64, 12
    rng = np.random.default_rng(4)
    nevs = rng.integers(1, 201, S)
    nevs[:2] = (1, 200)
    consts = closed_loop_tests._consts(Tf, 16, 12, 500, P, 2)
    demand = _ragged_demand(consts, nevs, rng)
    fleet = ChargingStationFleet(consts, S, demand=demand, seed=7, rng="device", chain=chain, nevs=nevs)
    log = fleet.simulate()
    real = np.arange(fleet.M)[None, :] < nevs[:, None]
    for k in ("s", "l"):
        Mp = log[f"Mp_{k}"].cpu().numpy()
        assert np.all(Mp.sum(axis=1) == nevs[None, :])
        niter = log[f"niter_{k}"].cpu().numpy()
        assert np.all(niter[Mp > 0] >= 0) and np.all(niter[Mp == 0] == -1)
        conv = (Mp > 0) & (niter < 999)
        assert conv.sum() >= 0.98 * (Mp > 0).sum()
        err = np.abs(log[f"w_{k}"].cpu().numpy() - log[f"w_hat_{k}"].cpu().numpy())
        assert np.all(err[conv] <= log[f"beta_{k}"].cpu().numpy()[conv] + 1e-9)
        y = fleet.y[k].cpu().numpy()
        assert y[real].min() >= 0.3 and y[real].max() <= 0.95 * 0.9 + 1e-12
        assert np.all(np.isnan(y[~real]))
        assert np.all(fleet.idx[k].cpu().numpy()[~real] == 0)
    assert np.all(log["bimpc_status"].cpu().numpy() == 0)
    x = log["x"].cpu().numpy()
    assert x.min() >= -1e-9 and x.max() <= 0.3 + 1e-9
    again = ChargingStationFleet(consts, S, demand=demand, seed=7, rng="device", chain=chain, nevs=nevs)
    again.simulate()
    _assert_same_state(_state(fleet), _state(again))


@pytest.mark.gpu
@pytest.mark.parametrize("chain", ["reference", "partition"])
def test_ragged_stations_do_not_depend_on_fleet_size(chain):
    """test_fleet_kernels_gpu.py::test_fleet_stations_do_not_depend_on_fleet_size with stations of
    1..300 EVs: stations 0..7 of a 1,200-station fleet (the compact price step) and of an 8-station
    fleet with the same SoCs, sizes and demand give the same bits."""
    from chargingstation.fleet import ChargingStationFleet
    Tf, P, S_big, S_small = 3, 12, 1200, 8
    rng = np.random.default_rng(37)
    nevs = rng.integers(1, 301, S_big)
    nevs[:S_small] = (300, 1, 129, 257, 40, 256, 9, 128)
    consts = closed_loop_tests._consts(Tf, 16, 12, 500, P, 2)
    demand = _ragged_demand(consts, nevs, rng)
    big = ChargingStationFleet(consts, S_big, demand=demand, seed=13, rng="device", chain=chain, nevs=nevs)
    small = ChargingStationFleet(consts, S_small, demand=demand[:S_small], seed=13, rng="device", chain=chain,
                                 nevs=nevs[:S_small])
    assert big.M == small.M == 300
    # the constructor's draws depend on S; SoCs up to 0.84 make EVs leave within the three steps
    pad = np.arange(300)[None, :] >= nevs[:S_small, None]
    for k in ("s", "l"):
        y0 = rng.uniform(MIN_INITIAL_SOC, 0.84, (S_small, 300))
        y0[pad] = np.nan
        y0 = big.torch.from_numpy(y0).to(big.dev)
        big.y[k][:S_small].copy_(y0)
        small.y[k].copy_(y0)
    big_log, small_log = big.simulate(), small.simulate()
    assert big_log.keys() == small_log.keys()
    for key in big_log:
        kt.assert_same(big_log[key][..., :S_small].cpu().numpy(), small_log[key].cpu().numpy(), key)
    for k in ("s", "l"):
        kt.assert_same(big.y[k][:S_small].cpu().numpy(), small.y[k].cpu().numpy(), "y_" + k)
        kt.assert_same(big.ncharged[k][:S_small].cpu().numpy(), small.ncharged[k].cpu().numpy(), "ncharged_" + k)
        kt.assert_same(big.idx[k][:S_small].cpu().numpy(), small.idx[k].cpu().numpy(), "idx_" + k)
    kt.assert_same(big.x[:S_small].cpu().numpy(), small.x.cpu().numpy(), "x")
    assert int(small.ncharged["s"].sum() + small.ncharged["l"].sum()) > 0
