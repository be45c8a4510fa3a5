"""The device-side vector-Jacobian product of the LoMPC solve (lompc_vjp_dev) and the autograd function built on it
(LoMPC.solve_lompc_diff / solve_lompc_vjp), against the dense reference VJP of tests/test_lompc_grad_cpu.py, finite
differences of the GPU forward and torch.autograd.gradcheck."""
import itertools

import numpy as np
import pytest
import torch

from chargingstation import _native
from chargingstation.lompc import LoMPC, LoMPCConstants
from oracle import lompc_oracle as orc
from test_lompc_grad_cpu import classify, margins, vjp_dense

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


def np_(x):
    return None if x is None else x.detach().cpu().numpy()


def draw(rng, o, N, B, price="convex", lr_pos=True, regime="random"):
    """Rows drawn like tests/test_lompc_gpu.py (test_lompc.py:34-36), or at the closed-loop scale (0.05 theta U)."""
    lm = (o.theta if regime == "random" else 0.05 * o.theta) * rng.random((B, 3 * N))
    if price == "linear":
        lm[:, 2 * N:] = 0.0
    lr = 3 * N * o.delta * rng.random(B) if lr_pos else np.zeros(B)
    gam = o.y_max * rng.random(B)
    return lm, lr, gam


def solve_and_vjp(s, lm, lr, gam, gw, gc, w=None):
    if w is None:
        w, _ = s.solve_lompc_batch(T(lm), T(lr), T(gam))
    out = s.solve_lompc_vjp(T(lm), T(lr), T(gam), T(w) if not torch.is_tensor(w) else w,
                            None if gw is None else T(gw), None if gc is None else T(gc), return_info=True)
    torch.cuda.synchronize()
    return np_(w) if torch.is_tensor(w) else w, [np_(x) for x in out[:3]], np_(out[3]["status"])


def check_rows(o, N, lm, lr, gam, w, gw, gc, got, rows=None, bar=1e-9):
    """Every output of every row within bar * max(1, |ref|_inf) of vjp_dense at the kernel's own w."""
    g_lm, g_lr, g_ga = got
    for b in (range(len(gam)) if rows is None else rows):
        lmb = lm[b] if lm.ndim == 2 else lm
        lrb = lr[b] if np.ndim(lr) else float(lr)
        ref = vjp_dense(N, o, lmb, lrb, gam[b], w[b], None if gw is None else gw[b], None if gc is None else gc[b])
        for name, a, r in (("lmbd", g_lm[b], ref[0]), ("lmbd_r", g_lr[b], ref[1]), ("gamma", g_ga[b], ref[2])):
            err = np.max(np.abs(a - r))
            assert err <= bar * max(1.0, np.max(np.abs(r))), (N, b, name, err, np.max(np.abs(r)))


# ------------------------------------------------------------------------------------------------ the oracle
@pytest.mark.parametrize("N", [1, 2, 3, 12, 24, 48, 96, 168, 512])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_kernel_against_dense_oracle(ev, N):
    """Random and closed-loop-scale prices (lmbd_r = 0 there, so the large EV has d = 0 stages), both price types,
    lmbd_r = 0 and > 0.  The recursion is a backward-stable factorisation of H_FF (d + M >= c > 0 pivots, P <= cN),
    and agrees with the dense solve to ~1e-17 relative on the CPU; 1e-9 leaves room for the dense solve's own
    rounding at N = 512."""
    o, s = consts_of(ev), solver(ev, N)
    rng = np.random.default_rng(10 * N + (ev == "large"))
    parts = []
    for price, lr_pos, regime in itertools.product(("linear", "convex"), (False, True), ("random", "closed")):
        parts.append(draw(rng, o, N, 3, price, lr_pos and regime == "random", regime))
    lm, lr, gam = (np.concatenate(x) for x in zip(*parts))
    B = len(gam)
    gw, gc = rng.standard_normal((B, N)), rng.standard_normal(B)
    w, got, st = solve_and_vjp(s, lm, lr, gam, gw, gc)
    assert (st == 0).all()
    check_rows(o, N, lm, lr, gam, w, gw, gc, got)
    if ev == "large" and N >= 12:
        d = 2 * (lr[:, None] * o.theta ** 2 + 3 * o.theta / (4 * o.w_max) * lm[:, 2 * N:])
        free = np.array([~classify(o, w[b]) for b in range(B)])
        assert ((d == 0) & free).any(), "no free d = 0 stage was exercised"


# ---------------------------------------------------------------------------------------- finite differences
def _nondegenerate(o, N, lm, lr, gam, w, need=1e-5):
    return [b for b in range(len(gam)) if min(margins(N, o, lm[b], lr[b], gam[b], w[b])[:2]) >= need]


@pytest.mark.parametrize("ev", ["small", "large"])
def test_kernel_against_finite_differences_of_the_gpu_forward(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(5 + (ev == "large"))
    lm, lr, gam = draw(rng, o, N, 64)
    w, _ = s.solve_lompc_batch(lm, lr, gam)
    rows = _nondegenerate(o, N, lm, lr, gam, w)
    assert len(rows) >= 16
    lm, lr, gam, w = lm[rows], lr[rows], gam[rows], w[rows]
    B = len(rows)
    gw, gc = rng.standard_normal((B, N)), rng.standard_normal(B)
    _, (g_lm, g_lr, g_ga), _ = solve_and_vjp(s, lm, lr, gam, gw, gc, w)
    grad = np.concatenate([g_lm, g_lr[:, None], g_ga[:, None]], axis=1)
    p = np.concatenate([lm, lr[:, None], gam[:, None]], axis=1)

    def f(x):
        w, cost = s.solve_lompc_batch(np.ascontiguousarray(x[:, :3 * N]), x[:, 3 * N].copy(), x[:, 3 * N + 1].copy())
        return np.sum(gw * w, axis=1) + gc * cost

    for blk in range(5):
        v = np.zeros_like(p)
        sl = slice(blk * N, (blk + 1) * N) if blk < 3 else slice(3 * N + blk - 3, 3 * N + blk - 2)
        v[:, sl] = rng.standard_normal((B, sl.stop - sl.start)) * np.maximum(p[:, sl], 1e-2)
        h = 1e-7
        fd = (f(p + h * v) - f(p - h * v)) / (2 * h)
        an = np.sum(grad * v, axis=1)
        # the forward's own accuracy (KKT tolerance 1e-11) over h sets an absolute floor of ~1e-6
        scale = np.maximum(np.sum(np.abs(grad * v), axis=1), 1.0)
        assert np.all(np.abs(an - fd) <= 1e-5 * scale), (blk, np.max(np.abs(an - fd) / scale))


def _gradcheck_rows(ev, N, B, rng, broadcast):
    o = consts_of(ev)
    s = solver(ev, N)
    for _ in range(50):
        lm, lr, gam = draw(rng, o, N, 8 * B)
        if broadcast:
            lm[:] = lm[0]
            lr[:] = lr[0]
        w, _ = s.solve_lompc_batch(lm, lr, gam)
        rows = _nondegenerate(o, N, lm, lr, gam, w, 1e-4)
        if len(rows) >= B:
            rows = rows[:B]
            return s, lm[rows], lr[rows], gam[rows]
    raise AssertionError("no nondegenerate rows found")


@pytest.mark.parametrize("mode", ["per_row", "broadcast_lmbd", "scalar_lmbd_r"])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_gradcheck(ev, mode):
    N = 12
    rng = np.random.default_rng(40 + (ev == "large"))
    s, lm, lr, gam = _gradcheck_rows(ev, N, 3, rng, mode != "per_row")
    lm_t = T(lm[0] if mode == "broadcast_lmbd" else lm).requires_grad_()
    lr_t = T(lr[:1] if mode == "scalar_lmbd_r" else lr).requires_grad_()
    ga_t = T(gam).requires_grad_()
    assert torch.autograd.gradcheck(lambda a, b, c: s.solve_lompc_diff(a, b, c), (lm_t, lr_t, ga_t),
                                    eps=1e-6, atol=1e-6, rtol=1e-5)


# ----------------------------------------------------------------------------------- broadcast and subsets
def _loss_grads(s, lm, lr, gam, gw, gc, req=(True, True, True)):
    leaves = [x.clone().requires_grad_(r) for x, r in zip((lm, lr, gam), req)]
    w, cost = s.solve_lompc_diff(*leaves)
    ((w * gw).sum() + (cost * gc).sum()).backward()
    return w, cost, [x.grad for x in leaves]


@pytest.mark.parametrize("ev", ["small", "large"])
def test_broadcast_gradient_is_the_sum_of_row_gradients(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(60 + (ev == "large"))
    lm, lr, gam = draw(rng, o, N, 777)
    gw, gc = T(rng.standard_normal((777, N))), T(rng.standard_normal(777))
    _, _, (b_lm, b_lr, b_ga) = _loss_grads(s, T(lm[0]), T(lr[:1]), T(gam), gw, gc)
    _, _, (r_lm, r_lr, r_ga) = _loss_grads(s, T(np.repeat(lm[:1], 777, 0)), T(np.repeat(lr[:1], 777)), T(gam), gw, gc)
    assert b_lm.shape == (3 * N,) and b_lr.shape == (1,)
    for a, r in ((b_lm, r_lm.sum(0)), (b_lr, r_lr.sum(0, keepdim=True))):
        assert torch.max(torch.abs(a - r)) <= 1e-12 * max(1.0, float(torch.max(torch.abs(r))))
    assert torch.equal(b_ga, r_ga)
    # a python-float lmbd_r is a constant broadcast scalar
    w, _ = s.solve_lompc_diff(T(lm[0]), float(lr[0]), T(gam))
    assert torch.equal(w, s.solve_lompc_batch(T(lm[0]), T(lr[:1]), T(gam))[0])


@pytest.mark.parametrize("ev", ["small", "large"])
def test_every_subset_of_needs_input_grad(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(70 + (ev == "large"))
    for bc in (False, True):
        lm, lr, gam = draw(rng, o, N, 50)
        lm_t, lr_t = (T(lm[0]), T(lr[:1])) if bc else (T(lm), T(lr))
        gw, gc = T(rng.standard_normal((50, N))), T(rng.standard_normal(50))
        _, _, full = _loss_grads(s, lm_t, lr_t, T(gam), gw, gc)
        for req in itertools.product((False, True), repeat=3):
            if not any(req):
                continue
            _, _, got = _loss_grads(s, lm_t, lr_t, T(gam), gw, gc, req)
            for r, g, f in zip(req, got, full):
                assert (g is None) if not r else torch.equal(g, f), (bc, req)


# ------------------------------------------------------------------------------------------- batch shapes
@pytest.mark.parametrize("ev,N", [("small", 24), ("large", 24), ("large", 512)])
def test_batch_composition_gives_the_same_bits(ev, N):
    """B = 0, 1, 31, 32, 33 and 70,001 (a partial last CTA); N = 512 large EV runs CTAs narrower than a warp.
    A row gives the same bits alone and inside any batch (the same w is passed in)."""
    o, s = consts_of(ev), solver(ev, N)
    rng = np.random.default_rng(80 + N)
    Bmax = 70001 if N == 24 else 333
    lm, lr, gam = draw(rng, o, N, Bmax)
    lm[Bmax // 2:] *= 0.05
    w = s.solve_lompc_batch(T(lm), T(lr), T(gam))[0]
    gw, gc = rng.standard_normal((Bmax, N)), rng.standard_normal(Bmax)
    _, big, _ = solve_and_vjp(s, lm, lr, gam, gw, gc, w)
    probe = [0, 1, 30, 31, 32, 33, Bmax // 2, Bmax - 2, Bmax - 1]
    for B in (1, 31, 32, 33):
        _, part, _ = solve_and_vjp(s, lm[:B], lr[:B], gam[:B], gw[:B], gc[:B], w[:B].contiguous())
        for a, r in zip(part, big):
            assert np.array_equal(a, r[:B])
    for b in probe:
        _, one, _ = solve_and_vjp(s, lm[b:b + 1], lr[b:b + 1], gam[b:b + 1], gw[b:b + 1], gc[b:b + 1],
                                  w[b:b + 1].contiguous())
        for a, r in zip(one, big):
            assert np.array_equal(a, r[b:b + 1])
    check_rows(o, N, lm, lr, gam, np_(w), gw, gc, big, rows=probe)
    _, empty, st = solve_and_vjp(s, lm[:0], lr[:0], gam[:0], gw[:0], gc[:0], w[:0])
    assert empty[0].shape == (0, 3 * N) and st.shape == (0,)
    wd, cd = s.solve_lompc_diff(T(lm[:0]).requires_grad_(), T(lr[:0]), T(gam[:0]))
    assert wd.shape == (0, N) and cd.shape == (0,)


# ------------------------------------------------------------------------------------------- active sets
def _prices_for(o, N, w, gam, target_mult):
    """Prices (lmbd3 = lmbd_r = 0) that make w the solution: on fixed coordinates -(Hw+g) = target_mult (inside the
    subdifferential), on free ones the KKT equation with the segment's slope."""
    d, c, _, _, _ = orc.lompc_problem_data(N, o, np.zeros(3 * N), 0.0, gam)
    Hw = orc.dense_hessian(N, d, c) @ w
    g = -Hw - target_mult  # g_k = theta (l1 - l2) - c gamma (N - k)
    x = (g + c * gam * np.arange(N, 0, -1)) / o.theta
    lm = np.zeros(3 * N)
    lm[:N] = np.maximum(x, 0) + 0.1
    lm[N:2 * N] = np.maximum(-x, 0) + 0.1
    return lm


@pytest.mark.parametrize("ev", ["small", "large"])
def test_active_set_edges(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    brk, slope = orc._segments(o)
    wm = o.w_max
    rng = np.random.default_rng(90 + (ev == "large"))
    cases = {}
    # all free: w strictly inside one segment (the first for the large EV), multiplier = minus that slope
    w_free = wm * (0.03 + 0.08 * rng.random(N))
    cases["all_free"] = (_prices_for(o, N, w_free, 0.7, slope[0]), 0.0, 0.7)
    # all at 0: gamma = 0 and lmbd1 > lmbd2
    lm0 = np.zeros(3 * N)
    lm0[:N] = 1.0
    cases["all_zero"] = (lm0, 0.0, 0.0)
    # all at w_max: a large price for not charging
    lmx = np.zeros(3 * N)
    lmx[N:2 * N] = 100 * o.theta
    cases["all_wmax"] = (lmx, 0.0, o.y_max)
    if ev == "large":  # every coordinate on the breakpoint 0.5 w_max, multipliers mid-interval
        cases["all_interior"] = (_prices_for(o, N, np.full(N, brk[2]), 0.6, 0.5 * (slope[1] + slope[2])), 0.0, 0.6)
        lmd = 0.05 * o.theta * rng.random(3 * N)
        lmd[2 * N:] = 0.0
        cases["free_d0"] = (lmd, 0.0, 0.5)
    lm = np.stack([c[0] for c in cases.values()])
    lr = np.array([c[1] for c in cases.values()])
    gam = np.array([c[2] for c in cases.values()])
    B = len(gam)
    gw, gc = rng.standard_normal((B, N)), rng.standard_normal(B)
    w, got, st = solve_and_vjp(s, lm, lr, gam, gw, gc)
    assert (st == 0).all()
    fixed = np.array([classify(o, w[b]) for b in range(B)])
    names = list(cases)
    at = {n: i for i, n in enumerate(names)}
    assert not fixed[at["all_free"]].any()
    assert np.all(w[at["all_zero"]] == 0.0) and fixed[at["all_zero"]].all()
    assert np.allclose(w[at["all_wmax"]], wm, atol=1e-9 * wm) and fixed[at["all_wmax"]].all()
    if ev == "large":
        assert np.allclose(w[at["all_interior"]], brk[2], atol=1e-9 * wm) and fixed[at["all_interior"]].all()
        assert (~fixed[at["free_d0"]]).any()
    check_rows(o, N, lm, lr, gam, w, gw, gc, got)
    # fully fixed rows: the w part vanishes, the cost part is the envelope gradient alone
    for n in ("all_zero", "all_wmax") + (("all_interior",) if ev == "large" else ()):
        b = at[n]
        ref = vjp_dense(N, o, lm[b], lr[b], gam[b], w[b], None, gc[b])
        assert np.array_equal(got[0][b], ref[0]) or np.max(np.abs(got[0][b] - ref[0])) <= 1e-12 * np.max(np.abs(ref[0]))


# ------------------------------------------------------------------------------- upstream and invalid input
@pytest.mark.parametrize("ev", ["small", "large"])
def test_upstream_on_one_output_and_nan_isolation(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(100 + (ev == "large"))
    lm, lr, gam = draw(rng, o, N, 40)
    gw, gc = rng.standard_normal((40, N)), rng.standard_normal(40)
    w, only_w, _ = solve_and_vjp(s, lm, lr, gam, gw, None)
    check_rows(o, N, lm, lr, gam, w, gw, None, only_w)
    _, only_c, _ = solve_and_vjp(s, lm, lr, gam, None, gc, w)
    check_rows(o, N, lm, lr, gam, w, None, gc, only_c)
    _, both, _ = solve_and_vjp(s, lm, lr, gam, gw, gc, w)
    gw_nan = gw.copy()
    gw_nan[7, 5] = np.nan
    _, nan, _ = solve_and_vjp(s, lm, lr, gam, gw_nan, gc, w)
    others = np.arange(40) != 7
    for a, r in zip(nan, both):
        assert np.array_equal(a[others], r[others])
    assert np.isnan(nan[0][7]).any() and np.isnan(nan[2][7])
    # autograd with the cost alone used: grad_w is None inside the backward
    lm_t = T(lm).requires_grad_()
    _, cost = s.solve_lompc_diff(lm_t, T(lr), T(gam))
    (cost * T(gc)).sum().backward()
    assert np.array_equal(np_(lm_t.grad), only_c[0])


@pytest.mark.parametrize("ev", ["small", "large"])
def test_invalid_rows_get_zero_gradients_and_a_status(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(110 + (ev == "large"))
    lm, lr, gam = draw(rng, o, N, 12)
    gw, gc = rng.standard_normal((12, N)), rng.standard_normal(12)
    w, clean, _ = solve_and_vjp(s, lm, lr, gam, gw, gc)
    lm2, lr2, gam2 = lm.copy(), lr.copy(), gam.copy()
    lm2[1, 3] = -1.0
    gam2[2] = np.nan
    gam2[3] = o.y_max + 0.01
    lr2[4] = -0.5
    lm2[5, 2 * N + 1] = np.nan
    _, got, st = solve_and_vjp(s, lm2, lr2, gam2, gw, gc, w)
    ST = _native
    assert list(st[:6]) == [0, ST.ST_NEGATIVE, ST.ST_NEGATIVE, ST.ST_BAD_GAMMA, ST.ST_NEGATIVE, ST.ST_NEGATIVE]
    assert (st[6:] == 0).all()
    for a, r in zip(got, clean):
        assert np.all(a[1:6] == 0.0)
        assert np.array_equal(a[[0] + list(range(6, 12))], r[[0] + list(range(6, 12))])
    # the autograd forward raises like solve_lompc_batch's host path: the first bad row decides
    gam_bad = gam[:4].copy()
    gam_bad[3] = o.y_max + 0.01
    with pytest.raises(AssertionError):
        s.solve_lompc_diff(T(lm[:4]).requires_grad_(), T(lr[:4]), T(gam_bad))
    with pytest.raises(ValueError):
        s.solve_lompc_diff(T(lm2[:4]).requires_grad_(), T(lr[:4]), T(gam_bad))


# --------------------------------------------------------------------------------- determinism and identity
@pytest.mark.parametrize("ev", ["small", "large"])
def test_deterministic_and_identical_to_the_plain_solve(ev):
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(120 + (ev == "large"))
    lm, lr, gam = draw(rng, o, N, 5000)
    gw, gc = rng.standard_normal((5000, N)), rng.standard_normal(5000)
    w, a, _ = solve_and_vjp(s, lm, lr, gam, gw, gc)
    _, b, _ = solve_and_vjp(s, lm, lr, gam, gw, gc, w)
    side = torch.cuda.Stream(DEV)
    with torch.cuda.stream(side):
        _, c, _ = solve_and_vjp(s, lm, lr, gam, gw, gc, w)
    side.synchronize()
    for x, y, z in zip(a, b, c):
        assert np.array_equal(x, y) and np.array_equal(x, z)
    wd, cd = s.solve_lompc_diff(T(lm).requires_grad_(), T(lr), T(gam))
    wp, cp = s.solve_lompc_batch(T(lm), T(lr), T(gam))
    assert torch.equal(wd.detach(), wp) and torch.equal(cd.detach(), cp)


# ------------------------------------------------------------------------------------- the project's use case
@pytest.mark.parametrize("ev", ["small", "large"])
def test_group_tracking_error_gradient(ev):
    """d/d(lmbd, lmbd_r) of ||mean_i w(lmbd, gamma_i) - w_ref||^2 in the A_bar metric (price_solver.py:205-209:
    v'A'Av + kappa v'v, kappa = lmbd_r / delta) for a 70-EV group at N = 24 with broadcast prices."""
    N, o = 24, consts_of(ev)
    s = solver(ev, N)
    rng = np.random.default_rng(130 + (ev == "large"))
    n = 70
    lm = 0.3 * o.theta * rng.random(3 * N)
    lr = 0.5 * o.delta
    gam = o.y_max - (0.2 + 0.3 * rng.random(n))
    w_ref = o.w_max * 0.4 * rng.random(N)
    lm_t, lr_t = T(lm).requires_grad_(), T([lr]).requires_grad_()
    w, _ = s.solve_lompc_diff(lm_t, lr_t, T(gam))
    v = w.mean(0) - T(w_ref)
    loss = (torch.cumsum(v, 0) ** 2).sum() + lr_t[0] / o.delta * (v * v).sum()
    loss.backward()
    # oracle: the chain rule by hand, vjp_dense per EV
    wn = np_(w)
    vn = wn.mean(0) - w_ref
    A = np.tril(np.ones((N, N)))
    gbar = 2 * (A.T @ A @ vn + lr / o.delta * vn) / n
    ref_lm, ref_lr = np.zeros(3 * N), (vn @ vn) / o.delta
    for i in range(n):
        r = vjp_dense(N, o, lm, lr, gam[i], wn[i], gbar)
        ref_lm += r[0]
        ref_lr += r[1]
    assert np.max(np.abs(np_(lm_t.grad) - ref_lm)) <= 1e-9 * max(1.0, np.max(np.abs(ref_lm)))
    assert abs(float(lr_t.grad[0]) - ref_lr) <= 1e-9 * max(1.0, abs(ref_lr))
    assert np.max(np.abs(ref_lm)) > 1e-6  # the loss does depend on the prices here
