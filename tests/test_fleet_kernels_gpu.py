"""The six plumbing entry points of the fleet loop (include/fleet_b200.h, csrc/fleet_api.cu)
against a NumPy float64 twin written from the reference lines each one replaces, and the
closed loop at fleet scale against the same stations in a small fleet.

Shapes are chosen for the launch geometry of fleet_api.cu: assign_kernel walks a station's
M EVs 128 at a time, apply_charge_kernel 256 at a time, scan_kernel gives each of its 1,024
threads ceil(P*S / 1024) counts, and gather_kernel runs one thread per group.  The grid below
makes each of these loops take one, two and many trips (the closed-loop benchmark runs
M = 500 and P*S = 49,152).

Bars: integer outputs, copies, plain additions in the documented order and divisions are
compared bit for bit (NaN positions included).  Three quantities hold a product that nvcc may
contract with an addition into one FMA (beta, the replacement SoC and the battery update);
they are held to 2 ulp of their operands' magnitude instead."""

import numpy as np
import pytest

import test_fleet_gpu as closed_loop_tests
from chargingstation.charging_station import assign_partitions, partition_edges
from chargingstation.settings import MAX_INITIAL_SOC, MIN_FULL_CHARGE_FRACTION, MIN_INITIAL_SOC

ERR_ARG = -2
Y_MAX = 0.9                                    # y_max of both EV types in the closed-loop scenarios
FULL_LEVEL = MIN_FULL_CHARGE_FRACTION * Y_MAX  # the departure threshold fleet.py passes
MASK64 = (1 << 64) - 1


# ============================================================================ NumPy twins
def twin_partition(edges, y, idx):
    """charging_station.py:111-116 per station on a copy of idx, then the group sort of
    charging_station.py:221-223 per station, laid out partition-major (g = p*S + s)."""
    S, M = y.shape
    P = len(edges) - 1
    idx = np.array(idx, dtype=np.int64)
    for s in range(S):
        assign_partitions(y[s], edges, idx[s])  # idx[s] is a view: updated in place
    per_station = np.stack([np.bincount(idx[s], minlength=P) for s in range(S)])  # [S, P]
    counts = per_station.T.reshape(P * S)
    off = np.concatenate([[0], np.cumsum(counts)])
    off_rebased = np.stack([off[p * S: p * S + S + 1] - off[p * S] for p in range(P)])
    y_sorted = np.empty(S * M)
    perm = np.empty(S * M, dtype=np.int64)
    for s in range(S):
        order = np.argsort(idx[s], kind="stable")
        local = np.concatenate([[0], np.cumsum(per_station[s])])
        for p in np.nonzero(per_station[s])[0]:
            b0, seg = off[p * S + s], order[local[p]: local[p + 1]]
            y_sorted[b0: b0 + len(seg)] = y[s, seg]
            perm[b0: b0 + len(seg)] = seg
    return dict(idx=idx, counts=counts, off=off, off_rebased=off_rebased, y_sorted=y_sorted, perm=perm)


def twin_bimpc_params(P, N_bi, N_lo, Bcap, eps_tol, lmbd_r, delta, counts, y0_rng, gamma_sm, x, profile, t):
    """charging_station.py:196-211 and price_solver.py:182-186 per EV type: group arrays
    partition-major [P*S] in, station-major [S, P] out.  delta, counts, y0_rng and gamma_sm are
    (small, large) pairs."""
    S = len(x)
    out = {}
    for k, d, n, rng, gsm in zip(("s", "l"), delta, counts, y0_rng, gamma_sm):
        n, rng, gsm = n.reshape(P, S).T, rng.reshape(P, S).T, gsm.reshape(P, S).T
        kappa = lmbd_r / d + 1e-5
        bound = (np.sqrt(N_lo) * rng + eps_tol) * np.min((1, 1 / np.sqrt(kappa)))
        out["Mp_" + k] = n / Bcap
        out["beta_" + k] = np.where(n > 0, bound, 0.0)
        out["gamma_" + k] = np.where(n > 0, gsm, 0.0)
    out["x0"] = x.copy()
    out["demand"] = profile[:, t: t + N_bi] / Bcap
    return out


def twin_wref(w_hat, N_lo):
    """w_ref[p*S + s, k] = w_hat[s, p, k] for k < N_lo (charging_station.py:269)."""
    S, P, _ = w_hat.shape
    return w_hat[:, :, :N_lo].transpose(1, 0, 2).reshape(P * S, N_lo)


def twin_keep_prices(counts, src, pre, post):
    """prices = 0 for an empty group (charging_station.py:270) and price_red = post - pre, or
    NaN for an empty group (charging_station.py:422-433)."""
    full = counts > 0
    return np.where(full[:, None], src, 0.0), np.where(full, post - pre, np.nan)


def counter_uniform(seed, a, b, c, d):
    """Twin of the kernel's counter-based generator on Python ints masked to 64 bits."""
    z = (seed + 0x9E3779B97F4A7C15 * (a + 1) + 0xBF58476D1CE4E5B9 * (b + 1) + 0x94D049BB133111EB * (c + 1) +
         0xD6E8FEB86659FD93 * (d + 1)) & MASK64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK64
    z = z ^ (z >> 31)
    z = ((z ^ (z >> 33)) * 0xFF51AFD7ED558CCD) & MASK64
    z = z ^ (z >> 33)
    return (z >> 11) * 2.0 ** -53


def twin_apply_charge(P, off, perm, w0_sorted, y, ncharged, full_level, rng_seed, ev_type, t,
                      y0_min=MIN_INITIAL_SOC, y0_max=MAX_INITIAL_SOC):
    """charging_station.py:329-349 with the orders fleet_b200.h documents: each group's w0 summed
    in sorted order, w_sum[s] = the group sums added in p order.  Returns the outputs and the
    uniform draw of every replaced EV (NaN elsewhere)."""
    S, M = y.shape
    y = y.copy()
    w_sum, w_mean = np.zeros(S), np.zeros(P * S)
    for s in range(S):
        tot = 0.0
        for p in range(P):
            g = p * S + s
            b0, b1 = int(off[g]), int(off[g + 1])
            w = w0_sorted[b0:b1]
            group = float(np.cumsum(w)[-1]) if b1 > b0 else 0.0  # cumsum adds left to right, as the kernel
            y[s, perm[b0:b1]] += w
            w_mean[g] = group / (b1 - b0) if b1 > b0 else 0.0
            tot += group
        w_sum[s] = tot
    leave = y > full_level
    u = np.full((S, M), np.nan)
    if rng_seed >= 0:
        for s, ev in zip(*np.nonzero(leave)):
            u[s, ev] = counter_uniform(rng_seed, ev_type, int(s), int(ev), t)
            y[s, ev] = y0_min + (y0_max - y0_min) * u[s, ev]
    return dict(y=y, mask=leave.astype(np.int32), w_sum=w_sum, w_mean=w_mean,
                ncharged=ncharged + leave.sum(axis=1)), u


def twin_battery(x, u_g, theta_s, theta_l, Bcap, w_sum_s, w_sum_l, profile, t):
    """charging_station.py:353-365 with ADD_RESIDUAL_CHARGE_TO_BATTERY = False."""
    return x + (u_g[:, 0] + (-theta_s * w_sum_s - theta_l * w_sum_l - profile[:, t]) / Bcap)


# ============================================================================ inputs
def socs(rng, S, M, edges, special=True):
    """SoCs over the partitions plus, when `special`, about 2 % of them exactly on an edge and
    about 0.5 % each below edges[0], above edges[P] and NaN; previous indices in [0, P)."""
    P = len(edges) - 1
    y = rng.uniform(edges[0], edges[-1], (S, M))
    if special:
        r = rng.random((S, M))
        on_edge = r < 0.02
        y[on_edge] = edges[rng.integers(0, P + 1, on_edge.sum())]
        y[(r >= 0.02) & (r < 0.025)] = edges[0] - 0.01
        y[(r >= 0.025) & (r < 0.03)] = edges[-1] + 0.01
        y[(r >= 0.03) & (r < 0.035)] = np.nan
    return y, rng.integers(0, P, (S, M))


def edge_socs(edges):
    """(SoC, previous index, expected index) of the edge semantics of charging_station.py:111-116."""
    P = len(edges) - 1
    prev = max(P - 1, 1) if P > 1 else 0
    rows = [(edges[0], prev, 0), (edges[P], 0, P - 1),
            (np.nextafter(edges[0], -1.0), prev, prev), (edges[0] - 0.1, prev, prev),
            (np.nextafter(edges[P], 2.0), prev, prev), (edges[P] + 0.1, prev, prev), (np.nan, prev, prev)]
    for q in range(1, P):  # on an interior edge the higher partition wins; one ulp either side decides alone
        rows += [(edges[q], 0, q), (np.nextafter(edges[q], -1.0), 0, q - 1), (np.nextafter(edges[q], 2.0), 0, q)]
    y, prev_idx, want = (np.array(c) for c in zip(*rows))
    return y, prev_idx.astype(np.int64), want.astype(np.int64)


def in_sorted_order(w, tw, S, P):
    """w[S, M] per EV -> the group-sorted order of the partition twin tw."""
    out = np.empty(w.size)
    for g in range(P * S):
        b0, b1 = tw["off"][g], tw["off"][g + 1]
        out[b0:b1] = w[g % S, tw["perm"][b0:b1]]
    return out


# ============================================================================ device calls
@pytest.fixture(scope="module")
def dev():
    import torch

    from chargingstation import _native
    return _Dev(torch, _native.load())


class _Dev:
    """Device buffers and the six entry points; each call checks its return code and the
    number of launches it adds."""

    def __init__(self, torch, lib):
        self.torch, self.lib = torch, lib
        self.stream = None  # None: torch's current stream

    def put(self, a, dtype=None):
        a = np.ascontiguousarray(a if dtype is None else np.asarray(a).astype(dtype))
        return self.torch.from_numpy(a).to("cuda")

    def i32(self, a):
        return self.put(a, np.int32)

    def f64(self, a):
        return self.put(a, np.float64)

    def fill(self, shape, value, dtype):
        return self.torch.full(shape, value, dtype=dtype, device="cuda")

    def _s(self):
        if self.stream is not None:
            return self.stream.cuda_stream
        return self.torch.cuda.current_stream().cuda_stream

    def call(self, name, launches, *args):
        if self.stream is not None:  # the inputs were written on torch's current stream
            self.stream.wait_stream(self.torch.cuda.current_stream())
        n0 = self.lib.lompc_launch_count()
        rc = getattr(self.lib, name)(0, *args, self._s())
        assert rc == 0, (name, rc)
        assert self.lib.lompc_launch_count() - n0 == launches, name
        self.torch.cuda.synchronize()

    @staticmethod
    def host(d):
        return {k: v.cpu().numpy() for k, v in d.items()}

    def partition(self, edges, y, idx):
        torch = self.torch
        S, M = y.shape
        P = len(edges) - 1
        d_edges, d_y = self.f64(edges), self.f64(y)
        out = dict(idx=self.i32(idx), counts=self.fill((P * S,), -7, torch.int32),
                   off=self.fill((P * S + 1,), -7, torch.int32), off_rebased=self.fill((P, S + 1), -7, torch.int32),
                   y_sorted=self.fill((S * M,), -7.0, torch.float64), perm=self.fill((S * M,), -7, torch.int32))
        self.call("fleet_partition_dev", 3, S, M, P, d_edges.data_ptr(), d_y.data_ptr(), out["idx"].data_ptr(),
                  out["counts"].data_ptr(), out["off"].data_ptr(), out["off_rebased"].data_ptr(),
                  out["y_sorted"].data_ptr(), out["perm"].data_ptr())
        return self.host(out)

    def apply_charge(self, P, off, perm, w0_sorted, y, ncharged, full_level, rng_seed, ev_type, t, mask=True,
                     w_mean=True):
        torch = self.torch
        S, M = y.shape
        ins = dict(off=self.i32(off), perm=self.i32(perm), w0=self.f64(w0_sorted))
        out = dict(y=self.f64(y), ncharged=self.i32(ncharged), w_sum=self.fill((S,), -7.0, torch.float64))
        if mask:
            out["mask"] = self.fill((S, M), -7, torch.int32)
        if w_mean:
            out["w_mean"] = self.fill((P * S,), -7.0, torch.float64)
        ptr = lambda k: out[k].data_ptr() if k in out else None  # noqa: E731
        self.call("fleet_apply_charge_dev", 1, S, M, P, full_level, MIN_INITIAL_SOC, MAX_INITIAL_SOC, rng_seed,
                  ev_type, t, ins["off"].data_ptr(), ins["perm"].data_ptr(), ins["w0"].data_ptr(), ptr("y"),
                  ptr("mask"), ptr("w_sum"), ptr("w_mean"), ptr("ncharged"))
        return self.host(out)

    def bimpc_params(self, P, N_bi, N_lo, Bcap, eps_tol, lmbd_r, delta, counts, y0_rng, gamma_sm, x, profile, t):
        torch = self.torch
        S, L = profile.shape
        ins = [self.i32(counts[0]), self.i32(counts[1]), self.f64(y0_rng[0]), self.f64(y0_rng[1]),
               self.f64(gamma_sm[0]), self.f64(gamma_sm[1]), self.f64(x), self.f64(profile)]
        names = ("Mp_s", "Mp_l", "beta_s", "beta_l", "gamma_s", "gamma_l")
        out = {k: self.fill((S, P), -7.0, torch.float64) for k in names}
        out["x0"] = self.fill((S,), -7.0, torch.float64)
        out["demand"] = self.fill((S, N_bi), -7.0, torch.float64)
        self.call("fleet_bimpc_params_dev", 1, S, P, N_bi, N_lo, Bcap, eps_tol, lmbd_r, delta[0], delta[1],
                  *[a.data_ptr() for a in ins[:7]], ins[7].data_ptr(), L, t,
                  *[out[k].data_ptr() for k in names + ("x0", "demand")])
        return self.host(out)

    def wref(self, w_hat, N_lo):
        S, P, N_bi = w_hat.shape
        d = self.f64(w_hat)
        out = dict(w_ref=self.fill((P * S, N_lo), -7.0, self.torch.float64))
        self.call("fleet_wref_dev", 1, S, P, N_bi, N_lo, d.data_ptr(), out["w_ref"].data_ptr())
        return self.host(out)["w_ref"]

    def keep_prices(self, counts, src, pre, post, mode):
        """mode: "in place" (src == dst, as fleet.py calls it), "out of place" or "no red"."""
        S, row = src.shape
        d_counts, d_src = self.i32(counts), self.f64(src)
        d_dst = d_src if mode == "in place" else self.fill((S, row), -7.0, self.torch.float64)
        d_pre, d_post = self.f64(pre), self.f64(post)
        d_red = self.fill((S,), -7.0, self.torch.float64)
        red = mode != "no red"
        self.call("fleet_keep_prices_dev", 1, S, row, d_counts.data_ptr(), d_src.data_ptr(), d_dst.data_ptr(),
                  d_pre.data_ptr() if red else None, d_post.data_ptr() if red else None,
                  d_red.data_ptr() if red else None)
        return d_dst.cpu().numpy(), d_red.cpu().numpy()

    def battery(self, x, u_g, theta_s, theta_l, Bcap, w_sum_s, w_sum_l, profile, t):
        S, N_bi = u_g.shape
        ins = [self.f64(u_g), self.f64(w_sum_s), self.f64(w_sum_l), self.f64(profile)]
        d_x = self.f64(x)
        self.call("fleet_battery_dev", 1, S, N_bi, theta_s, theta_l, Bcap, *[a.data_ptr() for a in ins],
                  profile.shape[1], t, d_x.data_ptr())
        return d_x.cpu().numpy()


# ============================================================================ comparisons
def assert_same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if got.dtype.kind == "f":
        bad = ~((got == want) | (np.isnan(got) & np.isnan(want)))
    else:
        bad = got != want
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:5].tolist())


def assert_within_ulps(got, want, magnitude, what, ulps=2):
    bar = ulps * np.spacing(np.abs(magnitude))
    err = np.abs(got - want)
    assert np.all(err <= bar), (what, float(np.max(err / bar)))


def check_partition(got, want):
    for k in ("idx", "counts", "off", "off_rebased", "perm", "y_sorted"):
        assert_same(got[k], want[k], k)


def check_apply_charge(got, want, u, y0_min=MIN_INITIAL_SOC, y0_max=MAX_INITIAL_SOC):
    for k in ("mask", "ncharged", "w_sum", "w_mean"):
        if k in got:
            assert_same(got[k], want[k], k)
    new = ~np.isnan(u)
    assert_same(got["y"][~new], want["y"][~new], "y")
    # y0_min + (y0_max - y0_min) * u may be one FMA on the device
    assert_within_ulps(got["y"][new], want["y"][new], np.maximum(y0_min, (y0_max - y0_min) * u[new]), "new SoC")


# ============================================================================ CPU: the twin against the mirror
@pytest.mark.parametrize("S,M,P", [(1, 1, 1), (3, 40, 6), (5, 300, 12), (2, 1000, 64)])
def test_partition_twin_matches_the_mirror_bookkeeping(S, M, P):
    """Anchors the partition twin to the reference: idx by an EV-by-EV loop of charging_station.py:111-116,
    and every group the y[idx == p] selection of charging_station.py:203, with the counts of np.bincount."""
    rng = np.random.default_rng(S * 1000 + M + P)
    edges = partition_edges(MIN_INITIAL_SOC, Y_MAX, P)
    y, idx0 = socs(rng, S, M, edges)
    ye, prev, _ = edge_socs(edges)
    n = min(len(ye), M)
    y[0, :n], idx0[0, :n] = ye[:n], prev[:n]
    tw = twin_partition(edges, y, idx0)
    for s in range(S):
        for i in range(M):
            want = idx0[s, i]
            for p in range(P):
                if edges[p] <= y[s, i] <= edges[p + 1]:
                    want = p
            assert tw["idx"][s, i] == want
        counts = np.bincount(tw["idx"][s], minlength=P)
        for p in range(P):
            g = p * S + s
            assert tw["counts"][g] == counts[p]
            sel = slice(tw["off"][g], tw["off"][g + 1])
            assert_same(tw["y_sorted"][sel], y[s][tw["idx"][s] == p], "y_sorted")
            assert_same(tw["perm"][sel], np.nonzero(tw["idx"][s] == p)[0], "perm")
            assert tw["off_rebased"][p, s] == tw["off"][g] - tw["off"][p * S]
        assert tw["off_rebased"][P - 1, S] == S * M - tw["off"][(P - 1) * S]
    assert tw["off"][-1] == S * M


def test_edge_socs_follow_the_reference_rule():
    for P in (1, 2, 12, 64):
        edges = partition_edges(MIN_INITIAL_SOC, Y_MAX, P)
        y, prev, want = edge_socs(edges)
        idx = prev.copy()
        assign_partitions(y, edges, idx)
        assert_same(idx, want, f"P={P}")


# ============================================================================ GPU: kernels against the twin
# (S, M, P): assign trips = ceil(M / 128), departure trips = ceil(M / 256), scan counts per thread =
# ceil(P*S / 1024), gather threads = P*S.
GRID = [
    (1, 1, 1), (1, 2, 2), (2, 127, 64), (7, 128, 31), (2, 129, 63), (7, 255, 12),
    (85, 256, 12),      # P*S = 1,020: one count per scan thread
    (86, 257, 12),      # P*S = 1,032: two
    (85, 500, 2), (1, 1000, 64), (7, 1000, 63),
    (1025, 1, 1), (1025, 129, 2), (1025, 257, 64),  # P*S = 1,025, 2,050, 65,600
    (4096, 2, 1),       # P*S = 4 * 1,024
    (4096, 500, 12),    # the benchmark's fleet: P*S = 48 * 1,024, four assign and two departure trips
    (5000, 127, 12),    # P*S = 60,000
    (5000, 256, 1), (86, 1000, 31),
    (1024, 1000, 64),   # P*S = 64 * 1,024, eight assign and four departure trips
]


def _grid_id(c):
    S, M, P = c
    return f"S{S}-M{M}-P{P}-PS{P * S}"


@pytest.mark.gpu
@pytest.mark.parametrize("S,M,P", GRID, ids=[_grid_id(c) for c in GRID])
def test_partition_matches_twin(dev, S, M, P):
    rng = np.random.default_rng(S * 7 + M * 3 + P)
    edges = partition_edges(MIN_INITIAL_SOC, Y_MAX, P)
    y, idx0 = socs(rng, S, M, edges)
    check_partition(dev.partition(edges, y, idx0), twin_partition(edges, y, idx0))


APPLY_GRID = GRID + [(7, 300, 100), (3, 1000, 256), (2, 257, 256)]  # beyond partition's 64: offsets from the twin


@pytest.mark.gpu
@pytest.mark.parametrize("S,M,P", APPLY_GRID, ids=[_grid_id(c) for c in APPLY_GRID])
def test_apply_charge_matches_twin(dev, S, M, P):
    rng = np.random.default_rng(S * 11 + M * 5 + P)
    edges = partition_edges(MIN_INITIAL_SOC, Y_MAX, P)
    y = rng.uniform(MIN_INITIAL_SOC, FULL_LEVEL, (S, M))
    y[-1, -1] = np.nextafter(FULL_LEVEL, 1.0)  # at least one departure
    tw = twin_partition(edges, y, rng.integers(0, P, (S, M)))
    w0 = rng.uniform(0.0, 0.05, S * M)
    w0[rng.random(S * M) < 0.05] = 0.0
    ncharged = rng.integers(0, 1000, S)
    seed, ev_type, t = 1234 + S, int(rng.integers(2)), int(rng.integers(96))
    want, u = twin_apply_charge(P, tw["off"], tw["perm"], w0, y, ncharged, FULL_LEVEL, seed, ev_type, t)
    got = dev.apply_charge(P, tw["off"], tw["perm"], w0, y, ncharged, FULL_LEVEL, seed, ev_type, t)
    assert want["mask"].any()
    check_apply_charge(got, want, u)


@pytest.mark.gpu
@pytest.mark.parametrize("embedded", [False, True], ids=["small", "embedded"])
@pytest.mark.parametrize("rng_seed", [-1, 9], ids=["mask_only", "device_rng"])
def test_apply_charge_departure_edges(dev, embedded, rng_seed):
    """y + w exactly on full_level stays (strict >, charging_station.py:335), one ulp above leaves; with
    rng_seed = -1 only the mask is written and a leaver keeps y + w."""
    S, M, P = (1, 6, 2) if not embedded else (1025, 257, 12)
    rng = np.random.default_rng(77 + embedded)
    edges = partition_edges(MIN_INITIAL_SOC, Y_MAX, P)
    y = rng.uniform(MIN_INITIAL_SOC, FULL_LEVEL, (S, M))
    w_full = np.zeros((S, M))
    above = np.nextafter(FULL_LEVEL, 1.0)
    s_at = S - 1
    cases = [(FULL_LEVEL, 0.0), (above, 0.0), (FULL_LEVEL - 0.25, 0.25), (above - 0.25, 0.25),
             (FULL_LEVEL - 0.125, 0.125), (np.nextafter(FULL_LEVEL, 0.0), 0.0)]
    cols = [0, 1, 2, M - 3, M - 2, M - 1] if embedded else list(range(6))
    for c, (yy, ww) in zip(cols, cases):
        y[s_at, c], w_full[s_at, c] = yy, ww
    lands = y[s_at, cols] + w_full[s_at, cols]
    assert list(lands) == [FULL_LEVEL, above, FULL_LEVEL, above, FULL_LEVEL, np.nextafter(FULL_LEVEL, 0.0)]
    tw = twin_partition(edges, y, np.zeros((S, M), dtype=np.int64))
    w0_sorted = in_sorted_order(w_full, tw, S, P)
    ncharged = np.full(S, 5)
    want, u = twin_apply_charge(P, tw["off"], tw["perm"], w0_sorted, y, ncharged, FULL_LEVEL, rng_seed, 1, 3)
    got = dev.apply_charge(P, tw["off"], tw["perm"], w0_sorted, y, ncharged, FULL_LEVEL, rng_seed, 1, 3)
    check_apply_charge(got, want, u)
    assert list(got["mask"][s_at, cols]) == [0, 1, 0, 1, 0, 0]
    if rng_seed < 0:
        assert got["y"][s_at, cols[1]] == above and got["y"][s_at, cols[3]] == above


@pytest.mark.gpu
@pytest.mark.parametrize("embedded", [False, True], ids=["small", "embedded"])
@pytest.mark.parametrize("P", [1, 2, 12, 64])
def test_partition_edge_socs(dev, P, embedded):
    """SoCs on edges[0], on every interior edge (the higher partition wins), on edges[P], one ulp
    either side, below edges[0], above edges[P] and NaN (each SoC outside every partition keeps its
    non-zero previous index)."""
    edges = partition_edges(MIN_INITIAL_SOC, Y_MAX, P)
    ye, prev, want = edge_socs(edges)
    n = len(ye)
    if embedded:  # the edge SoCs spread over all eight assign trips of station 1,000 of 1,025
        S, M = 1025, 1000
        rng = np.random.default_rng(P)
        y, idx0 = socs(rng, S, M, edges)
        cols = np.linspace(0, M - 1, n).astype(int)
        y[1000, cols], idx0[1000, cols] = ye, prev
        s_at = 1000
    else:
        S, M, cols, s_at = 1, n, np.arange(n), 0
        y, idx0 = ye[None, :].copy(), prev[None, :].copy()
    got = dev.partition(edges, y, idx0)
    check_partition(got, twin_partition(edges, y, idx0))
    assert_same(got["idx"][s_at, cols], want, "edge SoCs")


@pytest.mark.gpu
@pytest.mark.parametrize("S,M,P", [(3, 1000, 12), (1025, 257, 64)])
def test_partition_degenerate_groups(dev, S, M, P):
    """Station 0 has all its EVs in one partition (one group of M, the rest empty); the other
    stations use two partitions out of P."""
    rng = np.random.default_rng(S + P)
    edges = partition_edges(MIN_INITIAL_SOC, Y_MAX, P)
    y = np.empty((S, M))
    y[0] = rng.uniform(edges[P // 2], edges[P // 2 + 1], M)
    for s in range(1, S):
        q = rng.integers(0, P, 2)
        y[s] = np.where(rng.random(M) < 0.5, (edges[q[0]] + edges[q[0] + 1]) / 2, edges[q[1] + 1])
    idx0 = rng.integers(0, P, (S, M))
    got = dev.partition(edges, y, idx0)
    want = twin_partition(edges, y, idx0)
    check_partition(got, want)
    assert want["counts"][(P // 2) * S] == M
    assert np.count_nonzero(want["counts"].reshape(P, S)[:, 0]) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("S,M,P", [(2, 40, 6), (1025, 500, 12)])
def test_two_closed_loop_steps_at_kernel_level(dev, S, M, P):
    """partition -> apply_charge (device RNG) -> partition with the previous indices: EVs charge
    and leave, so they change partition between the two calls."""
    rng = np.random.default_rng(M)
    edges = partition_edges(MIN_INITIAL_SOC, Y_MAX, P)
    y, idx0 = socs(rng, S, M, edges, special=False)
    got = dev.partition(edges, y, idx0)
    want = twin_partition(edges, y, idx0)
    check_partition(got, want)
    w0 = rng.uniform(0.0, 0.2, S * M)
    ncharged = np.zeros(S, dtype=np.int64)
    a_want, u = twin_apply_charge(P, want["off"], want["perm"], w0, y, ncharged, FULL_LEVEL, 3, 0, 0)
    a_got = dev.apply_charge(P, want["off"], want["perm"], w0, y, ncharged, FULL_LEVEL, 3, 0, 0)
    check_apply_charge(a_got, a_want, u)
    y2 = a_got["y"]  # the device's SoCs; the replaced ones are within 2 ulp of the twin's
    got2 = dev.partition(edges, y2, got["idx"])
    want2 = twin_partition(edges, y2, want["idx"])
    check_partition(got2, want2)
    assert np.count_nonzero(want2["idx"] != want["idx"]) > S * M // 10


PARAM_SHAPES = [  # (S, P, N_bi, N_lo): threads = S * max(P, N_bi)
    (1, 1, 1, 1), (7, 12, 16, 12), (86, 64, 16, 12), (1025, 12, 48, 24), (5000, 12, 16, 12), (3, 2, 48, 1),
    (4096, 31, 24, 24),
]


@pytest.mark.gpu
@pytest.mark.parametrize("lmbd_r", [0.0, 24.0])
@pytest.mark.parametrize("S,P,N_bi,N_lo", PARAM_SHAPES, ids=[f"S{a}-P{b}-Nbi{c}-Nlo{d}" for a, b, c, d in PARAM_SHAPES])
def test_bimpc_params_matches_twin(dev, S, P, N_bi, N_lo, lmbd_r):
    rng = np.random.default_rng(S + P + N_bi)
    L = N_bi + 5
    counts = [rng.integers(0, 40, P * S) * (rng.random(P * S) < 0.6) for _ in range(2)]  # ~40 % empty groups
    y0_rng = [rng.uniform(0, 0.1, P * S) for _ in range(2)]
    gamma_sm = [rng.uniform(0.3, 0.6, P * S) for _ in range(2)]
    x, profile = rng.uniform(0, 0.3, S), rng.uniform(0, 400, (S, L))
    args = (P, N_bi, N_lo, 3600.0, 0.01, lmbd_r, (0.05, 0.025), counts, y0_rng, gamma_sm, x, profile, L - N_bi)
    got, want = dev.bimpc_params(*args), twin_bimpc_params(*args)
    for k in ("Mp_s", "Mp_l", "gamma_s", "gamma_l", "x0", "demand"):
        assert_same(got[k], want[k], k)
    for k in ("beta_s", "beta_l"):  # sqrt(N_lo) * y0_rng + eps_tol may be one FMA on the device
        assert_within_ulps(got[k], want[k], want[k], k)
        assert_same(got[k] == 0.0, want[k] == 0.0, k + " zero")


@pytest.mark.gpu
@pytest.mark.parametrize("lmbd_r", [0.0, 24.0])
def test_bimpc_params_beta_equals_the_price_solver_bound(dev, lmbd_r):
    """beta of one group against PriceSolver.get_robustness_bounds of the same EVs (price_solver.py:182-186)."""
    from chargingstation import settings
    from chargingstation.lompc import LoMPCConstants
    from chargingstation.price_solver import PriceSolver
    settings.PRINT_LEVEL = 0
    rng = np.random.default_rng(5)
    N_bi, N_lo, S, P = 16, 12, 3, 4
    consts = (LoMPCConstants(0.05, 10, 0.9, 0.25, "small"), LoMPCConstants(0.025, 50, 0.9, 0.15, "large"))
    counts, y0_rng, gamma_sm, want = [], [], [], []
    for c in consts:
        ps = PriceSolver(N_lo, c, "linear-convex")
        ys = rng.uniform(0.3, 0.5, 37)
        ps.set_charge_levels(ys)
        n = np.zeros(P * S, dtype=np.int64)
        n[1 * S + 2] = len(ys)  # group (p = 1, s = 2)
        rg = np.zeros(P * S)
        rg[1 * S + 2] = ps.y0_rng
        counts.append(n), y0_rng.append(rg), gamma_sm.append(np.zeros(P * S))
        want.append(ps.get_robustness_bounds(lmbd_r)[1])
    got = dev.bimpc_params(P, N_bi, N_lo, 3600.0, float(ps.eps_tol), lmbd_r, (consts[0].delta, consts[1].delta),
                           counts, y0_rng, gamma_sm, np.zeros(S), np.ones((S, N_bi)), 0)
    for k, w in zip(("beta_s", "beta_l"), want):
        assert_within_ulps(got[k][2, 1], w, w, k)
        assert np.count_nonzero(got[k]) == 1


WREF_SHAPES = [(1, 1, 1, 1), (7, 12, 16, 12), (5000, 12, 16, 16), (1025, 64, 48, 1), (4096, 12, 16, 12)]


@pytest.mark.gpu
@pytest.mark.parametrize("S,P,N_bi,N_lo", WREF_SHAPES, ids=[f"S{a}-P{b}-Nbi{c}-Nlo{d}" for a, b, c, d in WREF_SHAPES])
def test_wref_matches_twin(dev, S, P, N_bi, N_lo):
    w_hat = np.random.default_rng(S + N_lo).uniform(0, 0.25, (S, P, N_bi))
    assert_same(dev.wref(w_hat, N_lo), twin_wref(w_hat, N_lo), "w_ref")


KEEP_SHAPES = [(1, 1), (7, 36), (1025, 24), (49152, 36), (60000, 72)]  # (groups, row)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["in place", "out of place", "no red"])
@pytest.mark.parametrize("G,row", KEEP_SHAPES, ids=[f"G{a}-row{b}" for a, b in KEEP_SHAPES])
def test_keep_prices_matches_twin(dev, G, row, mode):
    rng = np.random.default_rng(G + row)
    counts = rng.integers(0, 3, G)
    counts[0] = 0
    src = rng.normal(size=(G, row))
    src.flat[:: 7] = -0.0  # copies must keep every bit
    pre, post = rng.normal(size=G), rng.normal(size=G)
    dst, red = dev.keep_prices(counts, src, pre, post, mode)
    want_dst, want_red = twin_keep_prices(counts, src, pre, post)
    assert_same(dst.view(np.int64), want_dst.view(np.int64), "dst bits")
    if mode == "no red":
        assert np.all(red == -7.0)
    else:
        assert_same(red, want_red, "price_red")
        assert np.isnan(red[0])


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 127, 128, 129, 5000])
def test_battery_matches_twin(dev, S):
    rng = np.random.default_rng(S)
    N_bi, L, M = 16, 24, 300
    Bcap = (10 + 50) * M
    x, u_g = rng.uniform(0, 0.3, S), rng.uniform(0, 0.2, (S, N_bi))
    ws, wl = rng.uniform(0, 0.05 * M, S), rng.uniform(0, 0.03 * M, S)
    profile = rng.uniform(0, 2000, (S, L))
    t = L - 1
    got = dev.battery(x, u_g, 10.0, 50.0, float(Bcap), ws, wl, profile, t)
    want = twin_battery(x, u_g, 10.0, 50.0, float(Bcap), ws, wl, profile, t)
    # -theta_s w_sum_s - theta_l w_sum_l may be one FMA on the device
    mag = np.max(np.abs([x, want, u_g[:, 0], 10.0 * ws / Bcap, 50.0 * wl / Bcap, profile[:, t] / Bcap]), axis=0)
    assert_within_ulps(got, want, mag, "x")


# ============================================================================ GPU: the C ABI contract
@pytest.mark.gpu
def test_invalid_arguments_return_err_arg_and_launch_nothing(dev):
    torch, lib = dev.torch, dev.lib
    S, M, P, N_bi, N_lo, L = 2, 4, 65, 4, 4, 8
    keep = []  # keeps the buffers alive until the end of the test

    def buf(dtype, n):  # zeros: every index buffer is valid, every offset array is empty
        t = torch.zeros(n, dtype=dtype, device="cuda")
        keep.append(t)
        return t.data_ptr()

    f, i = torch.float64, torch.int32
    edges, y, idx = buf(f, P + 2), buf(f, S * M), buf(i, S * M)
    counts, off, reb = buf(i, P * S + 1), buf(i, P * S + 2), buf(i, (P + 1) * (S + 1))
    ys, perm = buf(f, S * M), buf(i, S * M)
    g = [buf(f, 300 * S) for _ in range(14)]
    gi = [buf(i, 300 * S) for _ in range(4)]
    stream = torch.cuda.current_stream().cuda_stream

    def params(t):  # 2 count arrays, 6 more inputs (the last is the [S, L] profile), 8 outputs
        return lib.fleet_bimpc_params_dev(0, S, 4, N_bi, N_lo, 1.0, 0.01, 0.0, 0.05, 0.025, gi[0], gi[1], *g[:6], L, t,
                                          *g[6:14], stream)

    calls = {
        "partition P=0": lambda: lib.fleet_partition_dev(0, S, M, 0, edges, y, idx, counts, off, reb, ys, perm, stream),
        "partition P=65": lambda: lib.fleet_partition_dev(0, S, M, 65, edges, y, idx, counts, off, reb, ys, perm,
                                                          stream),
        "apply_charge P=257": lambda: lib.fleet_apply_charge_dev(0, S, M, 257, FULL_LEVEL, 0.3, 0.5, 1, 0, 0, gi[0],
                                                                 gi[1], g[0], g[1], gi[2], g[2], g[3], gi[3], stream),
        "apply_charge no mask": lambda: lib.fleet_apply_charge_dev(0, S, M, 4, FULL_LEVEL, 0.3, 0.5, -1, 0, 0, gi[0],
                                                                   gi[1], g[0], g[1], None, g[2], g[3], gi[3], stream),
        "params t + N_bi > L": lambda: params(L - N_bi + 1),
        "battery t = L": lambda: lib.fleet_battery_dev(0, S, N_bi, 10.0, 50.0, 1.0, *g[:4], L, L, g[4], stream),
        "wref N_bi < N_lo": lambda: lib.fleet_wref_dev(0, S, 4, 3, 4, g[0], g[1], stream),
        "keep_prices no pre": lambda: lib.fleet_keep_prices_dev(0, S, 4, gi[0], g[0], g[1], None, g[2], g[3], stream),
        "keep_prices no post": lambda: lib.fleet_keep_prices_dev(0, S, 4, gi[0], g[0], g[1], g[2], None, g[3], stream),
    }
    for name, call in calls.items():
        n0 = lib.lompc_launch_count()
        assert call() == ERR_ARG, name
        assert lib.lompc_launch_count() == n0, name
    # the same calls one step inside their limits succeed (3 launches for partition, 1 for the others)
    ok = {
        "partition P=64": (3, lambda: lib.fleet_partition_dev(0, S, M, 64, edges, y, idx, counts, off, reb, ys, perm,
                                                              stream)),
        "apply_charge P=256": (1, lambda: lib.fleet_apply_charge_dev(0, S, M, 256, FULL_LEVEL, 0.3, 0.5, 1, 0, 0,
                                                                     gi[0], gi[1], g[0], g[1], gi[2], g[2], g[3],
                                                                     gi[3], stream)),
        "params t + N_bi = L": (1, lambda: params(L - N_bi)),
        "battery t = L - 1": (1, lambda: lib.fleet_battery_dev(0, S, N_bi, 10.0, 50.0, 1.0, *g[:4], L, L - 1, g[4],
                                                               stream)),
        "wref N_bi = N_lo": (1, lambda: lib.fleet_wref_dev(0, S, 4, 4, 4, g[0], g[1], stream)),
        "keep_prices no red": (1, lambda: lib.fleet_keep_prices_dev(0, S, 4, gi[0], g[0], g[1], None, None, None,
                                                                    stream)),
    }
    for name, (n, call) in ok.items():
        n0 = lib.lompc_launch_count()
        assert call() == 0, name
        assert lib.lompc_launch_count() - n0 == n, name
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_side_stream_gives_the_same_bits(dev):
    """One kernel-level closed-loop step on torch's current stream and on a side stream."""
    torch = dev.torch
    S, M, P, N_bi, N_lo = 1025, 257, 12, 16, 12
    rng = np.random.default_rng(21)
    edges = partition_edges(MIN_INITIAL_SOC, Y_MAX, P)
    y, idx0 = socs(rng, S, M, edges)
    w0 = rng.uniform(0, 0.05, S * M)
    w_hat = rng.uniform(0, 0.25, (S, P, N_bi))
    profile = rng.uniform(0, 400, (S, N_bi + 3))
    x, u_g = rng.uniform(0, 0.3, S), rng.uniform(0, 0.2, (S, N_bi))
    src, pre, post = rng.normal(size=(P * S, 3 * N_lo)), rng.normal(size=P * S), rng.normal(size=P * S)

    def step():
        out = {}
        part = dev.partition(edges, y, idx0)
        out.update({"part_" + k: v for k, v in part.items()})
        cnt = part["counts"]
        prm = dev.bimpc_params(P, N_bi, N_lo, 3600.0, 0.01, 24.0, (0.05, 0.025), (cnt, cnt[::-1].copy()),
                               (pre, post), (post, pre), x, profile, 3)
        out.update({"prm_" + k: v for k, v in prm.items()})
        out["w_ref"] = dev.wref(w_hat, N_lo)
        out["dst"], out["red"] = dev.keep_prices(cnt, src, pre, post, "in place")
        ac = dev.apply_charge(P, part["off"], part["perm"], w0, y, np.arange(S), FULL_LEVEL, 5, 1, 2)
        out.update({"ac_" + k: v for k, v in ac.items()})
        out["x"] = dev.battery(x, u_g, 10.0, 50.0, 3600.0, ac["w_sum"], ac["w_sum"][::-1].copy(), profile, 2)
        return out

    main = step()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    dev.stream = side
    try:
        again = step()
    finally:
        dev.stream = None
    assert main.keys() == again.keys()
    for k in main:
        assert_same(main[k].view(np.uint8), again[k].view(np.uint8), k)
    check_partition({k[5:]: v for k, v in again.items() if k.startswith("part_")}, twin_partition(edges, y, idx0))


# ============================================================================ GPU: the closed loop
@pytest.mark.gpu
@pytest.mark.parametrize("chain", ["reference", "partition"])
def test_fleet_stations_do_not_depend_on_fleet_size(chain):
    """Stations 0..7 of a 1,200-station fleet and of an 8-station fleet with the same SoCs and
    demand give the same bits in every log, in y, x and ncharged.  The large fleet runs the scan at
    15 counts per thread (the small one at 1), the compact price step (from 1,184 chains or groups per
    launch) and the EV-response kernel at 360,000 QPs per EV type instead of 2,400."""
    from chargingstation.fleet import ChargingStationFleet
    Tf, M, P, S_big, S_small = 3, 300, 12, 1200, 8
    consts = closed_loop_tests._consts(Tf, 16, 12, M, P, 2)
    rng = np.random.default_rng(31)
    demand = np.stack([np.roll(consts.demand, int(rng.integers(24))) * rng.uniform(0.9, 1.1) for _ in range(S_big)])
    big = ChargingStationFleet(consts, S_big, demand=demand, seed=13, rng="device", chain=chain)
    small = ChargingStationFleet(consts, S_small, demand=demand[:S_small], seed=13, rng="device", chain=chain)
    # the constructor draws the large EVs after all S*M small ones, so it would give rows that depend on S;
    # SoCs up to 0.84 make EVs leave (and draw replacements) within the three steps
    for k in ("s", "l"):
        y0 = big.torch.from_numpy(rng.uniform(MIN_INITIAL_SOC, 0.84, (S_small, M))).to(big.dev)
        big.y[k][:S_small].copy_(y0)
        small.y[k].copy_(y0)
    big_log, small_log = big.simulate(), small.simulate()
    assert big_log.keys() == small_log.keys()
    for key in big_log:
        assert_same(big_log[key][..., :S_small].cpu().numpy(), small_log[key].cpu().numpy(), key)
    for k in ("s", "l"):
        assert_same(big.y[k][:S_small].cpu().numpy(), small.y[k].cpu().numpy(), "y_" + k)
        assert_same(big.ncharged[k][:S_small].cpu().numpy(), small.ncharged[k].cpu().numpy(), "ncharged_" + k)
        assert_same(big.idx[k][:S_small].cpu().numpy(), small.idx[k].cpu().numpy(), "idx_" + k)
    assert_same(big.x[:S_small].cpu().numpy(), small.x.cpu().numpy(), "x")
    assert int(small.ncharged["s"].sum() + small.ncharged["l"].sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("price_type", ["linear-convex", "linear"])
def test_fleet_reference_chain_equals_single_station_runs_at_multi_trip_sizes(price_type):
    """test_fleet_reference_chain_equals_single_station_runs, same assertions and bars, at M = 300:
    assign takes three trips per station and the departure loop two."""
    closed_loop_tests.test_fleet_reference_chain_equals_single_station_runs(price_type, (16, 12, 300, 12))
