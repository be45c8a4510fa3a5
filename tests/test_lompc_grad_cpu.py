"""The gradient of the LoMPC solve, on the CPU: the dense reference VJP (``vjp_dense``, which the GPU tests compare
the kernel with) against central finite differences of the exact active-set oracle.

Parameters p = (lmbd[3N], lmbd_r, gamma).  Where the active set is locally constant, dw_B = 0 and
dw_F = -H_FF^-1 (dg_F + dd_F .* w_F); the cost gradient follows from the envelope theorem (include/lompc_b200.h,
DESIGN.md section 2).  Finite differences are taken along directions of p and compared only at points whose
active set cannot change within the step: every free coordinate at least 1e-6 w_max from a breakpoint and every
fixed coordinate's multiplier at least 1e-6 (relative) inside its interval."""
import numpy as np
import pytest

from oracle import lompc_oracle as orc


def classify(consts, w, band=None):
    """Fixed coordinates of w: K1's binding rule (lompc_solve.cuh), the same comparisons as the VJP kernel."""
    wm = consts.w_max
    band = 1e-9 * wm if band is None else band
    brk, _ = orc._segments(consts)
    fixed = (w <= band) | (w >= brk[-1] - band)
    for b in brk[1:-1]:
        fixed |= (w >= b - band) & (w <= b + band)
    return fixed


def vjp_dense(N, consts, lmbd, lmbd_r, gamma, w, grad_w=None, grad_cost=None, band=None):
    """Reference vector-Jacobian product of the LoMPC solve at its solution w: dense solve on H_FF.
    Returns (grad_lmbd[3N], grad_lmbd_r, grad_gamma) of  grad_w'w + grad_cost * cost."""
    th, wm = consts.theta, consts.w_max
    q = 3 * th / (4 * wm)
    d, c, _, _, _ = orc.lompc_problem_data(N, consts, lmbd, lmbd_r, gamma)
    gw = np.zeros(N) if grad_w is None else np.asarray(grad_w, dtype=np.float64)
    gc = 0.0 if grad_cost is None else float(grad_cost)
    free = ~classify(consts, w, band)
    z = np.zeros(N)
    if free.any():
        H = orc.dense_hessian(N, d, c)
        z[free] = np.linalg.solve(H[np.ix_(free, free)], gw[free])
    s = np.cumsum(w)
    g_lm = np.concatenate([-th * z + gc * th * w, th * z + gc * th * (wm - w), -2 * q * z * w + gc * q * w * w])
    g_lr = -2 * th ** 2 * (z @ w) + gc * th ** 2 * (w @ w)
    g_ga = c * (np.arange(N, 0, -1) @ z) - gc * c * np.sum(s)
    return g_lm, float(g_lr), float(g_ga)


def margins(N, consts, lmbd, lmbd_r, gamma, w):
    """(free margin / w_max, fixed-multiplier margin / scale, kinds of the fixed coordinates) at the solution w."""
    d, c, g, _, _ = orc.lompc_problem_data(N, consts, lmbd, lmbd_r, gamma)
    grad = orc.dense_hessian(N, d, c) @ w + g
    brk, slope = orc._segments(consts)
    nseg = len(slope)
    scale = max(1.0, float(np.max(np.abs(g))) + float(slope[-1]))
    fixed = classify(consts, w)
    free_m, fix_m, kinds = np.inf, np.inf, set()
    for k in range(N):
        if not fixed[k]:
            free_m = min(free_m, float(np.min(np.abs(w[k] - brk))) / consts.w_max)
            continue
        i = int(np.argmin(np.abs(w[k] - brk)))
        kinds.add("zero" if i == 0 else ("wmax" if i == nseg else "interior"))
        s_lo = slope[i - 1] if i > 0 else -np.inf
        s_hi = slope[i] if i < nseg else np.inf
        fix_m = min(fix_m, float(min(-grad[k] - s_lo, s_hi + grad[k])) / scale)
    return free_m, fix_m, kinds


def draw(rng, N, consts, price, lr_pos, regime="random"):
    """One point drawn like tests/test_lompc_gpu.py (test_lompc.py:34-36 prices), or the closed-loop scale."""
    th = consts.theta
    lm = (th if regime == "random" else 0.05 * th) * rng.random(3 * N)
    if price == "linear":
        lm[2 * N:] = 0.0
    lr = 3 * N * consts.delta * rng.random() if lr_pos else 0.0
    gam = consts.y_max * rng.random()
    return lm, lr, gam


def solve(N, consts, lm, lr, gam):
    return orc.solve_active_set(N, consts, lm, lr, gam)[0]


def fd_directional(N, consts, p, v, gw, gc, h):
    """Central difference of grad_w'w + grad_cost * cost along v, p = (lmbd, lmbd_r, gamma) flattened."""
    def f(x):
        lm, lr, gam = x[:3 * N], x[3 * N], x[3 * N + 1]
        w = solve(N, consts, lm, lr, gam)
        return gw @ w + gc * orc.lompc_cost(N, consts, w, lm, lr, gam)
    return (f(p + h * v) - f(p - h * v)) / (2 * h)


def directions(rng, N, p, lr_pos, price):
    """Block directions (lmbd1, lmbd2, lmbd3, lmbd_r, gamma) and one mixed direction, scaled like p."""
    vs = []
    for blk in range(3):
        if blk == 2 and price == "linear":
            continue
        v = np.zeros(3 * N + 2)
        v[blk * N:(blk + 1) * N] = rng.standard_normal(N) * np.maximum(p[blk * N:(blk + 1) * N], 1e-3)
        vs.append(v)
    if lr_pos:
        v = np.zeros(3 * N + 2)
        v[3 * N] = p[3 * N]
        vs.append(v)
    v = np.zeros(3 * N + 2)
    v[3 * N + 1] = 1.0
    vs.append(v)
    return vs


def consts_of(ev):
    return orc.small_ev_consts() if ev == "small" else orc.large_ev_consts()


def _seed(ev, N, price, lr_pos):
    return 1000 * N + 10 * (ev == "large") + 2 * (price == "linear") + lr_pos


def _points(ev, N, price, lr_pos, seed):
    rng = np.random.default_rng(seed)
    o = consts_of(ev)
    pts = [draw(rng, N, o, price, lr_pos) for _ in range(5)]
    # one point that charges at full rate early on (coordinates at w_max) and one at the closed-loop scale
    lm, lr, gam = draw(rng, N, o, price, lr_pos)
    lm[:N] *= 0.02
    pts.append((lm, lr * 0.1, o.y_max - 1e-3))
    pts.append(draw(rng, N, o, price, lr_pos, "closed"))
    return rng, o, pts


@pytest.mark.parametrize("lr_pos", [False, True])
@pytest.mark.parametrize("price", ["linear", "convex"])
@pytest.mark.parametrize("N", [12, 24])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_vjp_dense_against_finite_differences(ev, N, price, lr_pos):
    rng, o, pts = _points(ev, N, price, lr_pos, _seed(ev, N, price, lr_pos))
    used = 0
    for lm, lr, gam in pts:
        w = solve(N, o, lm, lr, gam)
        free_m, fix_m, kinds = margins(N, o, lm, lr, gam, w)
        if free_m < 1e-6 or fix_m < 1e-6:
            continue
        used += 1
        gw = rng.standard_normal(N)
        gc = float(rng.standard_normal())
        g_lm, g_lr, g_ga = vjp_dense(N, o, lm, lr, gam, w, gw, gc)
        grad = np.concatenate([g_lm, [g_lr, g_ga]])
        p = np.concatenate([lm, [lr, gam]])
        for v in directions(rng, N, p, lr_pos, price):
            an = grad @ v
            fd = fd_directional(N, o, p, v, gw, gc, 1e-7)
            scale = np.abs(grad) @ np.abs(v)
            assert abs(an - fd) <= 2e-6 * max(scale, 1e-12), (ev, N, price, lr_pos, an, fd, scale)
    assert used >= 4, f"only {used} of {len(pts)} points are far enough from an active-set change"


def test_qualifying_points_cover_every_kind_of_fixed_coordinate():
    """The comparisons above include coordinates fixed at 0, at w_max and (large EV) at an interior breakpoint."""
    seen = set()
    for ev in ("small", "large"):
        for N in (12, 24):
            for price in ("linear", "convex"):
                for lr_pos in (False, True):
                    _, o, pts = _points(ev, N, price, lr_pos, _seed(ev, N, price, lr_pos))
                    for lm, lr, gam in pts:
                        w = solve(N, o, lm, lr, gam)
                        free_m, fix_m, kinds = margins(N, o, lm, lr, gam, w)
                        if free_m >= 1e-6 and fix_m >= 1e-6:
                            seen.update((ev, k) for k in kinds)
    for ev in ("small", "large"):
        assert (ev, "zero") in seen and (ev, "wmax") in seen, seen
    assert ("large", "interior") in seen, seen


def _segments_inner(o):
    """Breakpoints to pin a coordinate at: 0 (small EV), 0 and the interior pwl breakpoints (large EV)."""
    brk, _ = orc._segments(o)
    return brk[:-1]


def weakly_active_point(N, o, lm, lr, gam, b):
    """A point where a coordinate sits on breakpoint b with its multiplier at the end of its interval: raise lmbd1_k
    of the first coordinate above b until w_k just reaches b (w_k is nonincreasing in lmbd1_k), by bisection."""
    w = solve(N, o, lm, lr, gam)
    k = int(np.flatnonzero(w > b + 1e-6 * o.w_max)[0])
    lo, hi = lm[k], lm[k] + 1.0
    while solve(N, o, np.where(np.arange(3 * N) == k, hi, lm), lr, gam)[k] > b:
        hi += 10 * (hi - lo)
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        if solve(N, o, np.where(np.arange(3 * N) == k, mid, lm), lr, gam)[k] > b:
            lo = mid
        else:
            hi = mid
    return np.where(np.arange(3 * N) == k, hi, lm), lr, gam


@pytest.mark.parametrize("ev", ["small", "large"])
def test_cost_gradient_at_degenerate_points(ev):
    """The envelope-theorem cost gradient against central finite differences of cost o solve, also where the active
    set changes inside the step: w = 0 everywhere (gamma = 0), zero prices, sparse closed-loop-scale prices, and
    coordinates pinned weakly active on 0 and on every interior pwl breakpoint.  The cost is C^1 with a Lipschitz gradient, so the differences converge there too.  (The oracle accepts
    parameters a step below zero.)"""
    o = consts_of(ev)
    N = 12
    rng = np.random.default_rng(7 + (ev == "large"))
    pts = [(np.zeros(3 * N), 0.0, 0.0), (np.zeros(3 * N), 0.0, o.y_max - 1e-3)]
    for _ in range(4):
        lm = 0.05 * o.theta * rng.random(3 * N) * (rng.random(3 * N) < 0.5)
        pts.append((lm, 0.0, (o.y_max - 1e-3) * rng.random()))
    lm, lr, gam = draw(rng, N, o, "convex", True)
    lm[:N] *= 0.02  # charge hard, so that some coordinate lies above every breakpoint
    for b in _segments_inner(o):
        pts.append(weakly_active_point(N, o, lm, 0.1 * lr, o.y_max - 1e-3, b))
    degenerate = 0
    for lm, lr, gam in pts:
        w = solve(N, o, lm, lr, gam)
        free_m, fix_m, _ = margins(N, o, lm, lr, gam, w)
        degenerate += free_m < 1e-6 or fix_m < 1e-6
        g_lm, g_lr, g_ga = vjp_dense(N, o, lm, lr, gam, w, None, 1.0)
        grad = np.concatenate([g_lm, [g_lr, g_ga]])
        p = np.concatenate([lm, [lr, gam]])
        for i in list(range(0, 3 * N, 5)) + [3 * N, 3 * N + 1]:
            v = np.zeros(3 * N + 2)
            v[i] = 1.0
            h = 1e-8
            fd = fd_directional(N, o, p, v, np.zeros(N), 1.0, h)
            # a kink inside the step leaves an O(h L) error (L: Lipschitz constant of the gradient, up to ~c N^3 in
            # gamma), and the cost's rounding error is divided by h
            cost = orc.lompc_cost(N, o, w, lm, lr, gam)
            tol = 1e-5 * max(1.0, abs(grad[i])) + 4e-16 * max(1.0, abs(cost)) / h
            assert abs(grad[i] - fd) <= tol, (ev, i, grad[i], fd, tol)
    assert degenerate >= 1 + len(_segments_inner(o))


@pytest.mark.parametrize("ev", ["small", "large"])
def test_w_jacobian_in_g_is_symmetric(ev):
    """dw/dg = -E H_FF^-1 E' is symmetric: u'Jv = v'Ju, and Jv matches finite differences of the solve along g."""
    o = consts_of(ev)
    N = 24
    rng = np.random.default_rng(31 + (ev == "large"))
    checked = 0
    for _ in range(6):
        lm, lr, gam = draw(rng, N, o, "convex", True)
        w = solve(N, o, lm, lr, gam)
        free_m, fix_m, _ = margins(N, o, lm, lr, gam, w)
        u, v = rng.standard_normal(N), rng.standard_normal(N)
        z_u = -vjp_dense(N, o, lm, lr, gam, w, u)[0][:N] / o.theta  # dL/dlmbd1 = -theta z
        z_v = -vjp_dense(N, o, lm, lr, gam, w, v)[0][:N] / o.theta
        assert abs(u @ z_v - v @ z_u) <= 1e-12 * max(1.0, np.abs(u) @ np.abs(z_v))
        if free_m < 1e-6 or fix_m < 1e-6:
            continue
        checked += 1
        h = 1e-7
        dl = np.concatenate([v / o.theta, np.zeros(2 * N)])  # g = theta (lmbd1 - lmbd2) + ...: dg = v
        jv = (solve(N, o, lm + h * dl, lr, gam) - solve(N, o, lm - h * dl, lr, gam)) / (2 * h)
        assert np.max(np.abs(jv + z_v)) <= 1e-6 * max(1.0, np.max(np.abs(z_v)))
    assert checked >= 3
