"""The differentiable grouped LoMPC solve (lompc_group_solve_dev / lompc_group_vjp_dev, LoMPC.solve_lompc_groups_diff):
G groups of EVs, each group's EVs sharing its prices.  Checked against the plain batched solve on the gathered rows,
price_w_err_dev's group means, the dense reference group_vjp_dense of tests/test_group_grad_cpu.py, the EV-order sum
of per-row lompc_vjp_dev rows, finite differences of the GPU forward, torch.autograd.gradcheck, and G separate
solve_lompc_diff calls with broadcast prices (the project's use case)."""
import itertools

import numpy as np
import pytest
import torch

from chargingstation import _native
from chargingstation.autodiff import lompc_group_solve, lompc_group_vjp
from chargingstation.lompc import LoMPC, LoMPCConstants
from oracle import lompc_oracle as orc
from test_group_grad_cpu import group_vjp_dense
from test_lompc_grad_cpu import classify, margins

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
_SOLVERS = {}


def consts_of(ev):
    return orc.small_ev_consts() if ev == "small" else orc.large_ev_consts()


def solver(ev, N):
    if (ev, N) not in _SOLVERS:
        o = consts_of(ev)
        _SOLVERS[(ev, N)] = LoMPC(N, LoMPCConstants(o.delta, o.theta, o.y_max, o.w_max, o.ev_type))
    return _SOLVERS[(ev, N)]


def T(x):
    return torch.as_tensor(np.asarray(x, dtype=np.float64), device=DEV).contiguous()


def offsets(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)


def OFF(sizes):
    return torch.as_tensor(offsets(sizes), device=DEV)


def group_of(sizes):
    return np.repeat(np.arange(len(sizes)), sizes)


def draw_groups(rng, o, N, sizes, price="convex", lr_pos=True, regime="random"):
    """Group prices drawn like tests/test_lompc_grad_gpu.py (or at the closed-loop scale 0.05 theta U), gamma per EV."""
    G = len(sizes)
    lm = (o.theta if regime == "random" else 0.05 * o.theta) * rng.random((G, 3 * N))
    if price == "linear":
        lm[:, 2 * N:] = 0.0
    lr = 3 * N * o.delta * rng.random(G) if lr_pos else np.zeros(G)
    gam = o.y_max * rng.random(int(np.sum(sizes)))
    return lm, lr, gam


def run(s, sizes, lm, lr, gam, gw=None, ga=None, need=(True, True, True), w=None):
    """Device forward (unless w is given) and VJP; host arrays out."""
    off = OFF(sizes)
    if w is None:
        w, w_avg, st_f = lompc_group_solve(s, off, T(lm), T(lr), T(gam))
    st = torch.empty(len(gam), dtype=torch.int32, device=DEV)
    grads = lompc_group_vjp(s, off, T(lm), T(lr), T(gam), w, None if gw is None else T(gw),
                            None if ga is None else T(ga), need, st)
    torch.cuda.synchronize()
    return w, [None if x is None else x.cpu().numpy() for x in grads], st.cpu().numpy()


def check_dense(o, N, sizes, lm, lr, gam, w, gw, ga, got, bar=1e-9):
    ref = group_vjp_dense(N, o, offsets(sizes), lm, lr, gam, w, gw, ga)
    for name, a, r in zip(("lmbd", "lmbd_r", "gamma"), got, ref):
        r = np.atleast_2d(r.T).T if r.ndim == 1 else r
        a = np.atleast_2d(a.T).T if a.ndim == 1 else a
        for j in range(len(r)):
            err = np.max(np.abs(a[j] - r[j]))
            assert err <= bar * max(1.0, np.max(np.abs(r[j]))), (N, name, j, err)


# ------------------------------------------------------------------------------------------------------- forward
@pytest.mark.parametrize("N,B_extra", [(12, 0), (24, 0), (24, 8000), (96, 0)])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_forward_equals_the_plain_solve_and_the_group_means(ev, N, B_extra):
    """w = solve_lompc_batch on the gathered rows (same bits); w_avg = the EV-order sum / n_g (same bits), 0 for an
    empty group.  Where K1 takes the same kernel for both (N = 24, more than 6,144 EVs: the register kernel; below
    that the plain call takes the warp-cooperative kernel and price_w_err_dev's fused error epilogue the thread
    kernel), w_avg also equals price_w_err_dev's bits."""
    o, s = consts_of(ev), solver(ev, N)
    rng = np.random.default_rng(10 + N + (ev == "large"))
    sizes = [0, 1, 31, 32, 33, 0, 500] + ([B_extra] if B_extra else [])
    lm, lr, gam = draw_groups(rng, o, N, sizes)
    lm[::2] *= 0.05
    go = group_of(sizes)
    w, w_avg, st = lompc_group_solve(s, OFF(sizes), T(lm), T(lr), T(gam))
    wp, _ = s.solve_lompc_batch(T(lm[go]), T(lr[go]), T(gam))
    torch.cuda.synchronize()
    assert torch.equal(w, wp) and int(st.abs().max()) == 0
    wn, wa = w.cpu().numpy(), w_avg.cpu().numpy()
    off = offsets(sizes)
    for g in range(len(sizes)):
        acc = np.zeros(N)
        for i in range(off[g], off[g + 1]):
            acc += wn[i]
        assert np.array_equal(wa[g], acc / sizes[g] if sizes[g] else np.zeros(N)), g
    if N == 24 and B_extra:
        ref = torch.full((len(sizes), N), float("nan"), dtype=torch.float64, device=DEV)
        w_ref = torch.zeros((len(sizes), N), dtype=torch.float64, device=DEV)
        args = (OFF(sizes), T(gam), T(lm), T(lr), w_ref, ref)  # (kept alive until the launch is enqueued)
        _native.raise_for(s._lib.price_w_err_dev(s._h, len(sizes), len(gam), *[x.data_ptr() for x in args],
                                                 None, None, None, None, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        ne = np.array(sizes) > 0
        assert torch.equal(w_avg[ne], ref[ne])


# ----------------------------------------------------------------------------------------------- dense reference
@pytest.mark.parametrize("N", [1, 2, 12, 24, 48, 96, 168, 512])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_against_the_dense_reference(ev, N):
    """Both price types, lmbd_r = 0 and > 0, random and closed-loop-scale prices (lmbd_r = 0 there: free d = 0
    stages for the large EV); upstream on w only, on w_avg only and on both; one empty group."""
    o, s = consts_of(ev), solver(ev, N)
    rng = np.random.default_rng(100 * N + (ev == "large"))
    parts = [draw_groups(rng, o, N, [3], price, lr_pos and regime == "random", regime)
             for price, lr_pos, regime in itertools.product(("linear", "convex"), (False, True), ("random", "closed"))]
    lm = np.concatenate([p[0] for p in parts] + [o.theta * rng.random((1, 3 * N))])
    lr = np.concatenate([p[1] for p in parts] + [[0.5]])
    gam = np.concatenate([p[2] for p in parts])
    sizes = [3] * len(parts) + [0]
    B, G = len(gam), len(sizes)
    gw, ga = rng.standard_normal((B, N)), rng.standard_normal((G, N))
    w = None
    for up_w, up_a in ((gw, None), (None, ga), (gw, ga)):
        w, got, st = run(s, sizes, lm, lr, gam, up_w, up_a, w=w)
        assert (st == 0).all()
        check_dense(o, N, sizes, lm, lr, gam, w.cpu().numpy(), up_w, up_a, got)
        assert np.all(got[0][-1] == 0.0) and got[1][-1] == 0.0
    if ev == "large" and N >= 12:
        wn = w.cpu().numpy()
        go = group_of(sizes)
        d = 2 * (lr[go, None] * o.theta ** 2 + 3 * o.theta / (4 * o.w_max) * lm[go, 2 * N:])
        free = np.array([~classify(o, wn[b]) for b in range(B)])
        assert ((d == 0) & free).any(), "no free d = 0 stage was exercised"


# ------------------------------------------------------------------------------------------------ per-row VJP
@pytest.mark.parametrize("ev", ["small", "large"])
def test_against_the_ev_order_sum_of_per_row_vjps(ev):
    """lompc_vjp_dev on the gathered rows with upstream grad_w[i] + grad_w_avg[g] / n_g, its rows added in EV order
    on the host: within 1e-12 of the summed magnitudes."""
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(200 + (ev == "large"))
    sizes = [0, 1, 31, 32, 33, 500, 7]
    lm, lr, gam = draw_groups(rng, o, N, sizes)
    lm[1::2] *= 0.05
    B, G = len(gam), len(sizes)
    gw, ga = rng.standard_normal((B, N)), rng.standard_normal((G, N))
    w, got, st = run(s, sizes, lm, lr, gam, gw, ga)
    assert (st == 0).all()
    go = group_of(sizes)
    up = gw + ga[go] / np.array(sizes)[go][:, None]
    rows = s.solve_lompc_vjp(T(lm[go]), T(lr[go]), T(gam), w, T(up))
    rows = [x.cpu().numpy() for x in rows]
    off = offsets(sizes)
    for g in range(G):
        acc_lm, acc_lr, mag_lm, mag_lr = np.zeros(3 * N), 0.0, np.zeros(3 * N), 0.0
        for i in range(off[g], off[g + 1]):
            acc_lm += rows[0][i]
            acc_lr += rows[1][i]
            mag_lm += np.abs(rows[0][i])
            mag_lr += abs(rows[1][i])
        assert np.max(np.abs(got[0][g] - acc_lm)) <= 1e-12 * max(1.0, mag_lm.max()), g
        assert abs(got[1][g] - acc_lr) <= 1e-12 * max(1.0, mag_lr), g
    assert np.max(np.abs(got[2] - rows[2])) <= 1e-12 * max(1.0, np.abs(rows[2]).max())


# ---------------------------------------------------------------------------------- gradcheck and finite differences
def _margin_groups(s, o, N, sizes, rng, need, lr_shared=None):
    """Groups whose every EV has margin >= need at the GPU solution (gammas drawn until enough qualify)."""
    G = len(sizes)
    lm = o.theta * rng.random((G, 3 * N))
    lr = np.full(G, lr_shared) if lr_shared is not None else 3 * N * o.delta * rng.random(G)
    gam = []
    for g in range(G):
        got = []
        for _ in range(50):
            cand = o.y_max * rng.random(64)
            w, _ = s.solve_lompc_batch(np.tile(lm[g], (64, 1)), np.full(64, lr[g]), cand)
            got += [cand[b] for b in range(64) if min(margins(N, o, lm[g], lr[g], cand[b], w[b])[:2]) >= need]
            if len(got) >= sizes[g]:
                break
        assert len(got) >= sizes[g]
        gam += got[:sizes[g]]
    return lm, lr, np.array(gam)


@pytest.mark.parametrize("mode", ["per_group", "broadcast_lmbd_r"])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_gradcheck(ev, mode):
    N, o = 12, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(300 + (ev == "large") + 2 * (mode == "per_group"))
    sizes = [2, 1]
    lm, lr, gam = _margin_groups(s, o, N, sizes, rng, 1e-4, 0.3 if mode != "per_group" else None)
    off = OFF(sizes)
    lm_t, ga_t = T(lm).requires_grad_(), T(gam).requires_grad_()
    lr_t = T(lr[:1] if mode != "per_group" else lr).requires_grad_()
    assert torch.autograd.gradcheck(lambda a, b, c: s.solve_lompc_groups_diff(off, a, b, c), (lm_t, lr_t, ga_t),
                                    eps=1e-6, atol=1e-6, rtol=1e-5)


@pytest.mark.parametrize("ev", ["small", "large"])
def test_against_finite_differences_of_the_gpu_forward(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(400 + (ev == "large"))
    sizes = [5, 3, 8]
    lm, lr, gam = _margin_groups(s, o, N, sizes, rng, 1e-5)
    B, G = len(gam), len(sizes)
    gw, ga = rng.standard_normal((B, N)), rng.standard_normal((G, N))
    _, (g_lm, g_lr, g_ga), _ = run(s, sizes, lm, lr, gam, gw, ga)
    off = OFF(sizes)

    def f(lm_, lr_, gam_):
        w, w_avg, _ = lompc_group_solve(s, off, T(lm_), T(lr_), T(gam_))
        return float((w * T(gw)).sum() + (w_avg * T(ga)).sum())

    h = 1e-7
    for blk in range(5):
        v_lm, v_lr, v_ga = np.zeros_like(lm), np.zeros(G), np.zeros(B)
        if blk < 3:
            v_lm[:, blk * N:(blk + 1) * N] = rng.standard_normal((G, N)) * np.maximum(lm[:, blk * N:(blk + 1) * N], 1e-2)
        elif blk == 3:
            v_lr = rng.standard_normal(G) * lr
        else:
            v_ga = rng.standard_normal(B) * 1e-1
        fd = (f(lm + h * v_lm, lr + h * v_lr, gam + h * v_ga) - f(lm - h * v_lm, lr - h * v_lr, gam - h * v_ga)) / (2 * h)
        an = np.sum(g_lm * v_lm) + g_lr @ v_lr + g_ga @ v_ga
        scale = max(np.sum(np.abs(g_lm * v_lm)) + np.abs(g_lr) @ np.abs(v_lr) + np.abs(g_ga) @ np.abs(v_ga), 1.0)
        assert abs(an - fd) <= 1e-5 * scale, (blk, an, fd)


# ------------------------------------------------------------------------------------------- group compositions
def _fleet_sizes(stations, evs=500, parts=12):
    """The closed loop's partition sizes: each station's EVs split into `parts` nearly equal partitions."""
    one = [len(x) for x in np.array_split(np.arange(evs), parts)]
    return one * stations


@pytest.mark.parametrize("scale", ["small", "fleet"])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_each_group_has_the_same_bits_alone_in_a_batch_on_a_second_run_and_stream(ev, scale):
    """Sizes 0, 1, 31, 32, 33 and 500; at fleet scale behind them 49,152 groups of the closed loop (4,096 stations x
    12 partitions of 500 EVs, B > 2,000,000).  A group's gradient does not depend on the rest of the batch (the same w
    is passed in: K1 itself picks its kernel by batch size, and its kernels round differently)."""
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    head = [0, 1, 31, 32, 33, 500]
    sizes = head + (_fleet_sizes(4096) if scale == "fleet" else [3, 0, 2])
    G, B = len(sizes), int(np.sum(sizes))
    if scale == "fleet":
        assert G >= 49152 and B >= 2_000_000
    gen = torch.Generator(device=DEV)
    gen.manual_seed(500 + (ev == "large"))
    lm = 0.05 * o.theta * torch.rand((G, 3 * N), generator=gen, dtype=torch.float64, device=DEV)
    lr = 3 * N * o.delta * torch.rand(G, generator=gen, dtype=torch.float64, device=DEV)
    gam = o.y_max * torch.rand(B, generator=gen, dtype=torch.float64, device=DEV)
    gw = torch.randn((B, N), generator=gen, dtype=torch.float64, device=DEV)
    ga = torch.randn((G, N), generator=gen, dtype=torch.float64, device=DEV)
    off = OFF(sizes)
    w, w_avg, st = lompc_group_solve(s, off, lm, lr, gam)
    assert int(st.abs().max()) == 0

    def vjp(off_, lm_, lr_, gam_, w_, gw_, ga_):
        out = lompc_group_vjp(s, off_, lm_, lr_, gam_, w_, gw_, ga_)
        torch.cuda.synchronize()
        return out

    full = vjp(off, lm, lr, gam, w, gw, ga)
    again = vjp(off, lm, lr, gam, w, gw, ga)
    side = torch.cuda.Stream(DEV)
    with torch.cuda.stream(side):
        other = vjp(off, lm, lr, gam, w, gw, ga)
    side.synchronize()
    for a, b, c in zip(full, again, other):
        assert torch.equal(a, b) and torch.equal(a, c)
    offn = offsets(sizes)
    probe = list(range(len(head))) + [G - 1] + ([G // 2] if scale == "fleet" else [])
    for g in probe:
        b0, b1 = int(offn[g]), int(offn[g + 1])
        one_off = torch.tensor([0, b1 - b0], dtype=torch.int32, device=DEV)
        one = vjp(one_off, lm[g:g + 1], lr[g:g + 1], gam[b0:b1], w[b0:b1], gw[b0:b1], ga[g:g + 1])
        assert torch.equal(one[0], full[0][g:g + 1]) and torch.equal(one[1], full[1][g:g + 1]), g
        assert torch.equal(one[2], full[2][b0:b1]), g
        if b1 == b0:
            assert not full[0][g].any() and not full[1][g].any()


# ---------------------------------------------------------------------------------------- invalid input and NaN
@pytest.mark.parametrize("ev", ["small", "large"])
def test_invalid_groups_and_nan_isolation(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(600 + (ev == "large"))
    sizes = [4, 3, 5, 2, 6]
    lm, lr, gam = draw_groups(rng, o, N, sizes)
    B, G = len(gam), len(sizes)
    off = offsets(sizes)
    gw, ga = rng.standard_normal((B, N)), rng.standard_normal((G, N))
    w, clean, st = run(s, sizes, lm, lr, gam, gw, ga)
    assert (st == 0).all()
    # group 1: a negative price; group 3: NaN lmbd_r; one EV of group 2 with gamma > y_max, one of group 4 NaN gamma
    lm2, lr2, gam2 = lm.copy(), lr.copy(), gam.copy()
    lm2[1, 5] = -1.0
    lr2[3] = np.nan
    gam2[off[2] + 1] = o.y_max + 0.01
    gam2[off[4]] = np.nan
    _, got, st = run(s, sizes, lm2, lr2, gam2, gw, ga, w=w)
    expect = np.zeros(B, dtype=np.int32)
    expect[off[1]:off[2]] = _native.ST_NEGATIVE
    expect[off[3]:off[4]] = _native.ST_NEGATIVE
    expect[off[2] + 1] = _native.ST_BAD_GAMMA
    expect[off[4]] = _native.ST_NEGATIVE
    assert np.array_equal(st, expect)
    for g in (1, 3):
        assert np.all(got[0][g] == 0.0) and got[1][g] == 0.0 and np.all(got[2][off[g]:off[g + 1]] == 0.0)
    assert np.array_equal(got[0][0], clean[0][0]) and got[1][0] == clean[1][0]
    assert got[2][off[2] + 1] == 0.0 and got[2][off[4]] == 0.0
    # the groups with one invalid EV: the sums over the others (the same upstream, so z of the others is unchanged)
    wn = w.cpu().numpy()
    for g, bad in ((2, off[2] + 1), (4, off[4])):
        keep = [i for i in range(off[g], off[g + 1]) if i != bad]
        up = gw[keep] + ga[g] / sizes[g]
        rows = s.solve_lompc_vjp(T(np.repeat(lm[g:g + 1], len(keep), 0)), T(np.full(len(keep), lr[g])), T(gam[keep]),
                                 T(wn[keep]), T(up))
        ref = rows[0].sum(0).cpu().numpy()
        assert np.max(np.abs(got[0][g] - ref)) <= 1e-12 * max(1.0, np.abs(ref).max())
    # the forward raises: a negative price (ValueError), gamma > y_max alone (AssertionError)
    off_t = OFF(sizes)
    with pytest.raises(ValueError):
        s.solve_lompc_groups_diff(off_t, T(lm2).requires_grad_(), T(lr), T(gam))
    gam3 = gam.copy()
    gam3[off[2] + 1] = o.y_max + 0.01
    with pytest.raises(AssertionError):
        s.solve_lompc_groups_diff(off_t, T(lm).requires_grad_(), T(lr), T(gam3))
    # malformed offsets: ValueError at the same sync, nothing read out of bounds
    for bad_off in ([0, 4, 3, 12, 14, 20], [1, 4, 7, 12, 14, 20], [0, 4, 7, 12, 14, 19], [0, 4, 7, 12, 14, 99]):
        with pytest.raises(ValueError):
            s.solve_lompc_groups_diff(torch.tensor(bad_off, dtype=torch.int32, device=DEV), T(lm), T(lr), T(gam))
    # NaN upstream in one group leaves every other group's bits unchanged
    for which in ("avg", "ev"):
        ga_n, gw_n = ga.copy(), gw.copy()
        if which == "avg":
            ga_n[2, 3] = np.nan
        else:
            gw_n[off[2] + 1, 3] = np.nan
        _, nan, _ = run(s, sizes, lm, lr, gam, gw_n, ga_n, w=w)
        others = [g for g in range(G) if g != 2]
        ev_others = np.r_[0:off[2], off[3]:B]
        assert np.array_equal(nan[0][others], clean[0][others]) and np.array_equal(nan[1][others], clean[1][others])
        assert np.array_equal(nan[2][ev_others], clean[2][ev_others])
        assert np.isnan(nan[0][2]).any() and np.isnan(nan[1][2])


@pytest.mark.parametrize("ev", ["small", "large"])
def test_every_subset_of_needs_input_grad(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(700 + (ev == "large"))
    sizes = [7, 0, 12, 1]
    lm, lr, gam = draw_groups(rng, o, N, sizes)
    off = OFF(sizes)
    gw, ga = T(rng.standard_normal((len(gam), N))), T(rng.standard_normal((len(sizes), N)))
    for bc in (False, True):
        lr_in = T(lr[:1]) if bc else T(lr)

        def grads(req):
            leaves = [x.clone().requires_grad_(r) for x, r in zip((T(lm), lr_in, T(gam)), req)]
            w, w_avg = s.solve_lompc_groups_diff(off, *leaves)
            ((w * gw).sum() + (w_avg * ga).sum()).backward()
            return [x.grad for x in leaves]

        full = grads((True, True, True))
        assert full[1].shape == lr_in.shape
        for req in itertools.product((False, True), repeat=3):
            if not any(req):
                continue
            for r, g, f in zip(req, grads(req), full):
                assert (g is None) if not r else torch.equal(g, f), (bc, req)
        if bc:  # a one-element lmbd_r: the sum over the groups of the per-group gradients
            per = lompc_group_vjp(s, off, T(lm), T(np.full(len(sizes), lr[0])), T(gam),
                                  s.solve_lompc_groups_diff(off, T(lm), lr_in, T(gam))[0], gw, ga)[1]
            assert torch.equal(full[1], per.sum(0, keepdim=True))
    # empty batch and float lmbd_r: w_avg and the gradients are zeros
    e_off = torch.zeros(3, dtype=torch.int32, device=DEV)
    lm_t = T(lm[:2]).requires_grad_()
    w, w_avg = s.solve_lompc_groups_diff(e_off, lm_t, 0.5, T(gam[:0]))
    assert w.shape == (0, N) and torch.equal(w_avg, torch.zeros((2, N), dtype=torch.float64, device=DEV))
    (w_avg * ga[:2]).sum().backward()
    assert torch.equal(lm_t.grad, torch.zeros_like(lm_t))


# ------------------------------------------------------------------------------------- the project's use case
@pytest.mark.parametrize("ev", ["small", "large"])
def test_group_tracking_errors_against_separate_broadcast_solves(ev):
    """d/d(lmbd, lmbd_r) of sum_g ||w_avg_g - w_ref_g||^2 in the A_bar metric (price_solver.py:205-209:
    v'A'Av + kappa v'v, kappa = lmbd_r / delta) for G groups in one call, against G solve_lompc_diff calls with
    broadcast prices (an empty group's mean is the constant 0)."""
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(800 + (ev == "large"))
    sizes = [70, 1, 33, 0, 12]
    G = len(sizes)
    lm = 0.3 * o.theta * rng.random((G, 3 * N))
    lr = 0.5 * o.delta * rng.random(G)
    gam = o.y_max - (0.2 + 0.3 * rng.random(int(np.sum(sizes))))
    w_ref = T(o.w_max * 0.4 * rng.random((G, N)))

    def track(w_avg_g, w_ref_g, lr_g):
        v = w_avg_g - w_ref_g
        return (torch.cumsum(v, 0) ** 2).sum() + lr_g / o.delta * (v * v).sum()

    lm_t, lr_t = T(lm).requires_grad_(), T(lr).requires_grad_()
    _, w_avg = s.solve_lompc_groups_diff(OFF(sizes), lm_t, lr_t, T(gam))
    sum(track(w_avg[g], w_ref[g], lr_t[g]) for g in range(G)).backward()
    off = offsets(sizes)
    for g in range(G):
        lm_g, lr_g = T(lm[g]).requires_grad_(), T(lr[g:g + 1]).requires_grad_()
        if sizes[g]:
            w, _ = s.solve_lompc_diff(lm_g, lr_g, T(gam[off[g]:off[g + 1]]))
            mean = w.mean(0)
        else:
            mean = torch.zeros(N, dtype=torch.float64, device=DEV)
        track(mean, w_ref[g], lr_g[0]).backward()
        ref_lm = lm_g.grad if lm_g.grad is not None else torch.zeros_like(lm_g)
        assert torch.max(torch.abs(lm_t.grad[g] - ref_lm)) <= 1e-12 * max(1.0, float(ref_lm.abs().max())), g
        assert abs(float(lr_t.grad[g] - lr_g.grad[0])) <= 1e-12 * max(1.0, abs(float(lr_g.grad[0]))), g
    assert float(lm_t.grad.abs().max()) > 1e-6
