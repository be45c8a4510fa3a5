"""The gradient of the grouped LoMPC solve, on the CPU: the dense reference (``group_vjp_dense``, which the GPU tests
compare lompc_group_vjp_dev with) against central finite differences of the exact active-set oracle's group means.

Group g owns EVs [off[g], off[g+1]); all of them see the prices lmbd[g], lmbd_r[g] and differ in gamma_i.  With
upstream gradients grad_w[B,N] on the EVs' w and grad_w_avg[G,N] on the group means, the upstream on w_i is
grad_w[i] + grad_w_avg[g] / n_g, and the group gradients are the sums of ``vjp_dense`` over the group's EVs
(DESIGN.md section 2).  Finite differences are compared only at points where every EV of the group has margin
(``margins``), so that no active set changes within the step."""
import numpy as np
import pytest

from oracle import lompc_oracle as orc
from test_lompc_grad_cpu import consts_of, margins, solve, vjp_dense


def group_vjp_dense(N, consts, off, lmbd, lmbd_r, gamma, w, grad_w=None, grad_w_avg=None):
    """Reference VJP of the grouped solve: (grad_lmbd[G,3N], grad_lmbd_r[G], grad_gamma[B]) of
    sum grad_w .* w + sum grad_w_avg .* w_avg, summed over each group's EVs in EV order."""
    G, B = len(off) - 1, len(gamma)
    g_lm, g_lr, g_ga = np.zeros((G, 3 * N)), np.zeros(G), np.zeros(B)
    for g in range(G):
        n = off[g + 1] - off[g]
        for i in range(off[g], off[g + 1]):
            gw = np.zeros(N) if grad_w is None else np.array(grad_w[i], dtype=np.float64)
            if grad_w_avg is not None:
                gw = gw + grad_w_avg[g] / n
            r = vjp_dense(N, consts, lmbd[g], lmbd_r[g], gamma[i], w[i], gw)
            g_lm[g] += r[0]
            g_lr[g] += r[1]
            g_ga[i] = r[2]
    return g_lm, g_lr, g_ga


def group_solve(N, consts, off, lmbd, lmbd_r, gamma):
    """(w[B,N], w_avg[G,N]) by the exact oracle; an empty group's mean is 0."""
    G = len(off) - 1
    w = np.array([solve(N, consts, lmbd[g], lmbd_r[g], gamma[i]) for g in range(G) for i in range(off[g], off[g + 1])])
    w = w.reshape(len(gamma), N)
    w_avg = np.array([w[off[g]:off[g + 1]].mean(0) if off[g + 1] > off[g] else np.zeros(N) for g in range(G)])
    return w, w_avg


def margin_groups(rng, N, o, price, sizes, tries=60):
    """Group prices (random scale, lmbd_r > 0 in every other group) and gammas whose EVs all have margin >= 1e-6."""
    lm, lr, gam = [], [], []
    for g, n in enumerate(sizes):
        lmg = o.theta * rng.random(3 * N)
        if price == "linear":
            lmg[2 * N:] = 0.0
        lrg = 3 * N * o.delta * rng.random() if g % 2 else 0.0
        got = []
        for _ in range(tries):
            ga = o.y_max * rng.random()
            w = solve(N, o, lmg, lrg, ga)
            if min(margins(N, o, lmg, lrg, ga, w)[:2]) >= 1e-6:
                got.append(ga)
                if len(got) == n:
                    break
        assert len(got) == n, f"only {len(got)} EVs with margin for group {g}"
        lm.append(lmg)
        lr.append(lrg)
        gam += got
    return np.array(lm), np.array(lr), np.array(gam)


@pytest.mark.parametrize("price", ["linear", "convex"])
@pytest.mark.parametrize("N", [12, 24])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_group_vjp_dense_against_finite_differences(ev, N, price):
    o = consts_of(ev)
    rng = np.random.default_rng(2000 + N + 7 * (ev == "large") + 3 * (price == "linear"))
    sizes = [3, 2]
    off = np.concatenate([[0], np.cumsum(sizes)])
    lm, lr, gam = margin_groups(rng, N, o, price, sizes)
    G, B = len(sizes), len(gam)
    w, w_avg = group_solve(N, o, off, lm, lr, gam)
    gw, ga = rng.standard_normal((B, N)), rng.standard_normal((G, N))
    for up_w, up_a in ((gw, None), (None, ga), (gw, ga)):
        g_lm, g_lr, g_ga = group_vjp_dense(N, o, off, lm, lr, gam, w, up_w, up_a)

        def f(lm_, lr_, gam_):
            w_, wa_ = group_solve(N, o, off, lm_, lr_, gam_)
            return (0.0 if up_w is None else np.sum(up_w * w_)) + (0.0 if up_a is None else np.sum(up_a * wa_))

        h = 1e-7
        dirs = []
        for g in range(G):
            for blk in range(3 if price == "convex" else 2):
                v = np.zeros_like(lm)
                v[g, blk * N:(blk + 1) * N] = rng.standard_normal(N) * np.maximum(lm[g, blk * N:(blk + 1) * N], 1e-3)
                dirs.append((v, np.zeros(G), np.zeros(B)))
            if lr[g] > 0:
                u = np.zeros(G)
                u[g] = lr[g]
                dirs.append((np.zeros_like(lm), u, np.zeros(B)))
        dirs.append((np.zeros_like(lm), np.zeros(G), rng.standard_normal(B) * 1e-1))
        for v_lm, v_lr, v_ga in dirs:
            an = np.sum(g_lm * v_lm) + g_lr @ v_lr + g_ga @ v_ga
            fd = (f(lm + h * v_lm, lr + h * v_lr, gam + h * v_ga) - f(lm - h * v_lm, lr - h * v_lr, gam - h * v_ga)) / (2 * h)
            scale = np.sum(np.abs(g_lm * v_lm)) + np.abs(g_lr) @ np.abs(v_lr) + np.abs(g_ga) @ np.abs(v_ga)
            assert abs(an - fd) <= 2e-6 * max(scale, 1e-12), (ev, N, price, an, fd, scale)


def test_group_vjp_dense_is_the_sum_of_per_ev_rows_and_empty_groups_are_zero():
    """Group structure of the reference itself: an upstream on w_avg alone equals the per-EV vjp_dense rows with
    grad_w_avg[g] / n_g as their upstream, summed; an empty group gets zeros; grad_gamma stays per EV."""
    N, o = 12, consts_of("large")
    rng = np.random.default_rng(5)
    off = np.array([0, 2, 2, 5])
    lm = o.theta * rng.random((3, 3 * N))
    lr = np.array([0.0, 0.3, 0.1])
    gam = o.y_max * rng.random(5)
    w, w_avg = group_solve(N, o, off, lm, lr, gam)
    assert np.array_equal(w_avg[1], np.zeros(N))
    ga = rng.standard_normal((3, N))
    g_lm, g_lr, g_ga = group_vjp_dense(N, o, off, lm, lr, gam, w, None, ga)
    assert np.all(g_lm[1] == 0.0) and g_lr[1] == 0.0
    for g in (0, 2):
        rows = [vjp_dense(N, o, lm[g], lr[g], gam[i], w[i], ga[g] / (off[g + 1] - off[g])) for i in range(off[g], off[g + 1])]
        assert np.allclose(g_lm[g], sum(r[0] for r in rows), rtol=0, atol=1e-15 * (1 + np.abs(g_lm[g]).max()))
        assert np.array_equal(g_ga[off[g]:off[g + 1]], np.array([r[2] for r in rows]))
