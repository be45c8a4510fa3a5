"""Every kernel the K1 dispatcher can pick, held to the exact oracle.

``launch_solve`` / ``launch_solve_reg_variant`` (csrc/lompc_api.cu) and the solve set's ``set_launch``
(csrc/lompc_warp_api.cu) choose between the warp-cooperative kernel, the register kernel in three CTA shapes
(64 x 4, 256 x 1, bulk-copied rows), and the any-N shared-memory kernel, by horizon, batch size, EV type, buffer
alignment and call kind (plain, broadcast prices, group mode with fused epilogues, solve set).  The tests below
reach each of those paths at the shapes where they go wrong - horizons without a compiled kernel, partial last
CTAs, the 65,536-QP switch, misaligned caller buffers, empty groups and segments, lanes of one warp in different
regimes - and compare against ``oracle.lompc_oracle`` (exact active set + KKT certificate), against the per-object
path or against a float64 numpy restatement of the reference's formulas."""
import numpy as np
import pytest

from oracle import lompc_oracle as orc
from oracle import price_oracle as po

pytestmark = pytest.mark.gpu

W_RTOL = 1e-9   # relative to w_max
C_RTOL = 1e-10  # relative to max(1, |cost|)


def _consts(ev):
    from chargingstation.lompc import LoMPCConstants
    o = orc.small_ev_consts() if ev == "small" else orc.large_ev_consts()
    return o, LoMPCConstants(o.delta, o.theta, o.y_max, o.w_max, o.ev_type)


def _regimes(o, N, B, seed):
    """Thirds of the batch: test_lompc.py:34-36 prices, closed-loop-scale sparse prices, linear prices."""
    rng = np.random.default_rng(seed)
    th = o.theta
    lm = np.zeros((B, 3 * N))
    lr = np.zeros(B)
    gam = o.y_max * rng.random(B)
    a, b = B // 3, 2 * B // 3
    lm[:a] = th * rng.random((a, 3 * N))
    lr[:a] = 3 * N * o.delta * rng.random(a)
    lm[a:b] = 0.05 * th * rng.random((b - a, 3 * N)) * (rng.random((b - a, 3 * N)) < 0.5)
    lm[b:, :2 * N] = 0.05 * th * rng.random((B - b, 2 * N))
    return lm, lr, gam


def _solver(N, ev, variant=0):
    from chargingstation.lompc import LoMPC
    o, c = _consts(ev)
    s = LoMPC(N, c)
    s.set_kernel_variant(variant)
    return o, s


def _sample(B, per_third):
    """Indices spread over the three regimes of _regimes, always with the first and the last QP."""
    cuts = [0, B // 3, 2 * B // 3, B]
    idx = [0, B - 1]
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        if hi > lo:
            idx += list(np.linspace(lo, hi - 1, per_third).astype(int))
    return sorted(set(idx))


def _check_oracle(N, o, w, cost, lm, lr, gam, idx):
    for b in idx:
        lmb = lm if lm.ndim == 1 else lm[b]
        lrb = float(lr if np.ndim(lr) == 0 else lr[b])
        wo, co, _ = orc.solve_active_set(N, o, lmb, lrb, float(gam[b]))
        assert np.max(np.abs(w[b] - wo)) <= W_RTOL * o.w_max, (N, b, np.max(np.abs(w[b] - wo)))
        if cost is not None:
            assert abs(cost[b] - co) <= C_RTOL * max(1.0, abs(co)), (N, b, cost[b], co)
        # (coordinates within the kernels' binding band, 1e-9 w_max, of a breakpoint count as on it; the bound pays
        # sqrt(N) * 1e-9 w_max for that)
        _, dist = orc.kkt_certificate(N, o, w[b], lmb, lrb, float(gam[b]), band=1e-9)
        assert dist <= 1e-8, (N, b, dist)


def _check_info(o, w, info):
    assert np.all(info["status"] == 0), np.flatnonzero(info["status"])[:8]
    assert info["kkt_res"].max() <= 1e-10
    assert w.min() >= 0.0 and w.max() <= o.w_max


# ------------------------------------------------------------------------------------------------------------------
# A. Horizons: the any-N kernel (no barrier, layout [k*T + t]) at every width the launcher can choose
# ------------------------------------------------------------------------------------------------------------------
HORIZONS = [1, 2, 3, 7, 12, 13, 24, 36, 47, 48, 96, 100, 129, 130, 151, 152, 168, 256, 512]


@pytest.mark.parametrize("B", [37, 18945])
@pytest.mark.parametrize("N", HORIZONS)
@pytest.mark.parametrize("ev", ["small", "large"])
def test_any_n_kernel_horizons(ev, N, B):
    """Horizons without a compiled kernel run the any-N kernel in automatic mode; the compiled ones (12, 24, 48, 96)
    are forced onto it.  18,945 QPs give the widest CTA that fits the horizon with a partial last CTA (T = 128 up to
    N ~ 32, 16 threads at N = 168, 8 at 512); 37 QPs one or two narrow CTAs.  Above N = 129 (large EV) / 151 (small
    EV) not even 32 threads fit the shared memory."""
    o, s = _solver(N, ev, 1 if N in (12, 24, 48, 96) else 0)
    lm, lr, gam = _regimes(o, N, B, 1000 + 7 * N + (ev == "large"))
    w, cost, info = s.solve_lompc_batch(lm, lr, gam, return_info=True)
    _check_info(o, w, info)
    per = 4 if N <= 100 else 2
    _check_oracle(N, o, w, cost, lm, lr, gam, _sample(B, per))


@pytest.mark.parametrize("ev", ["small", "large"])
def test_any_n_kernel_longest_horizon(ev):
    """N = 4096, the longest horizon lompc_create accepts: one QP per CTA (7 or 6 columns of 4096 doubles)."""
    N = 4096
    o, s = _solver(N, ev)
    rng = np.random.default_rng(44 + (ev == "large"))
    lm = o.theta * rng.random((2, 3 * N))
    lm[1] *= 0.05 * (rng.random(3 * N) < 0.5)
    lr = np.array([3 * N * o.delta * rng.random(), 0.0])
    gam = o.y_max * rng.random(2)
    w, cost, info = s.solve_lompc_batch(lm, lr, gam, return_info=True)
    _check_info(o, w, info)
    for b in range(2):
        _, dist = orc.kkt_certificate(N, o, w[b], lm[b], lr[b], gam[b])
        assert dist <= 1e-8, (b, dist)


@pytest.mark.parametrize("N", [36, 168])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_phase_split_price_loop_at_uncompiled_horizons(ev, N):
    """compute_optimal_prices (price_solver.py:79-174) at horizons with no device-resident loop: the phase-split loop,
    the any-N kernel in group mode (shared prices, skip mask, warm starts) and group_step_kernel<0>, with an empty
    group among the others.  Iteration counts equal the oracle's, prices within 1e-6."""
    from chargingstation import settings
    from chargingstation.price_solver import PriceSolver
    settings.PRINT_LEVEL = 0
    o, c = _consts(ev)
    rng = np.random.default_rng(N + 5 * (ev == "large"))
    counts = np.array([1, 5, 0, 17])
    G = len(counts)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    spans = [0.0, 0.02, 0.0, 0.1]
    y0 = np.concatenate([0.3 + sp * rng.random(n) for n, sp in zip(counts, spans)])
    # references the EVs can follow (the response to some price at gamma_sc, perturbed): loops of a few iterations
    w_ref = np.zeros((G, N))
    for g in range(G):
        lam = 0.05 * o.theta * rng.random(3 * N) * (rng.random(3 * N) < 0.5)
        w_ref[g] = orc.solve_active_set(N, o, lam, 0.0, 0.5)[0] * (1 + 0.2 * rng.random(N))
    max_iter = 40 if N <= 128 else 12  # (the Python oracle solves every EV of every iteration)
    ps = PriceSolver(N, c, "linear-convex")
    prices, st = ps.compute_optimal_prices_batch(off, y0, w_ref, np.zeros(G), np.zeros((G, 3 * N)), max_iter=max_iter)
    for g in np.flatnonzero(counts):
        ora = po.PriceOracle(N, o, "linear-convex", fast=N <= 128)
        ora.set_charge_levels(y0[off[g]: off[g + 1]])
        lam_o, st_o = ora.compute_optimal_prices(w_ref[g], 0.0, max_iter=max_iter)
        assert st["iter"][g] == st_o["iter"], (g, st["iter"][g], st_o["iter"])
        small = np.abs(lam_o) <= 1e3
        err = np.abs(prices[g] - lam_o)
        assert np.max(err[small]) <= 1e-6 * max(1.0, np.max(np.abs(lam_o[small]))), (g, np.max(err[small]))
        assert np.all(err[~small] <= 1e-3 * np.abs(lam_o[~small])), g


def test_price_loop_beyond_the_group_step_scratch_is_refused():
    """The price step keeps 2 x (3r + 9N) doubles per CTA in shared memory: above N ~ 750 that is more than a CTA can
    have.  The loop refuses such a horizon with ValueError (not a failed launch) and the process stays usable."""
    from chargingstation import settings
    from chargingstation.price_solver import PriceSolver
    settings.PRINT_LEVEL = 0
    o, c = _consts("small")
    rng = np.random.default_rng(7)
    y0 = 0.3 + 0.05 * rng.random(4)
    ps = PriceSolver(1024, c, "linear-convex")
    # (the LoMPC solves of that horizon themselves run: the columns of 8 threads do not fit, those of 4 do)
    lm = 0.05 * o.theta * rng.random((2, 3 * 1024))
    w, cost, info = ps.lompc.solve_lompc_batch(lm, np.zeros(2), np.array([0.2, 0.6]), return_info=True)
    _check_info(o, w, info)
    for b in range(2):
        assert orc.kkt_certificate(1024, o, w[b], lm[b], 0.0, [0.2, 0.6][b])[1] <= 1e-8
    ps.set_charge_levels(y0)
    with pytest.raises(ValueError):
        ps.compute_optimal_prices(0.5 * o.w_max * rng.random(1024), 0.0)
    N = 24
    ps = PriceSolver(N, c, "linear-convex")
    ps.set_loop_mode(1)  # the same phase-split loop, at a horizon where it fits
    ps.set_charge_levels(y0)
    w_ref = 0.5 * o.w_max * rng.random(N)
    lam, st = ps.compute_optimal_prices(w_ref, 0.0)
    ora = po.PriceOracle(N, o, "linear-convex", fast=True)
    ora.set_charge_levels(y0)
    lam_o, st_o = ora.compute_optimal_prices(w_ref, 0.0)
    assert st["iter"] == st_o["iter"]
    small = np.abs(lam_o) <= 1e3
    assert np.max(np.abs(lam - lam_o)[small]) <= 1e-6 * max(1.0, np.max(np.abs(lam_o[small])))


# ------------------------------------------------------------------------------------------------------------------
# B. Register-kernel shapes and layouts (N = 12, 24)
# ------------------------------------------------------------------------------------------------------------------
REG_BATCHES = [1, 255, 256, 257, 65535, 65536, 70001]


def _expected_auto_variant(N, ev, B):
    """The register-kernel shape automatic mode takes for plain rows (None: the warp-cooperative kernel)."""
    if B <= (4096 if N == 12 else 6144):
        return None
    if N == 24 and B >= 65536:
        return 9
    return 7 if (ev == "large" and B >= 65536) else 4


@pytest.mark.parametrize("B", REG_BATCHES)
@pytest.mark.parametrize("N", [12, 24])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_register_kernel_shapes_are_bit_identical(ev, N, B):
    """Variants 4 (64 x 4), 7 (256 x 1) and 9 (bulk-copied rows) run the same solve_reg with warps aligned at 32 in
    every shape: same bits for w, iterations, status and residual; the cost is re-summed in each epilogue (1e-12).
    Automatic mode equals the shape it picks."""
    o, _ = _consts(ev)
    lm, lr, gam = _regimes(o, N, B, 2000 + B + N + (ev == "large"))
    res = {}
    for v in (4, 7, 9, 0):
        _, s = _solver(N, ev, v)
        res[v] = s.solve_lompc_batch(lm, lr, gam, return_info=True)
    w4, c4, i4 = res[4]
    _check_info(o, w4, i4)
    for v in (7, 9):
        w, cst, info = res[v]
        assert np.array_equal(w, w4), (v, np.abs(w - w4).max())
        assert np.array_equal(info["iters"], i4["iters"]) and np.array_equal(info["status"], i4["status"]), v
        assert np.array_equal(info["kkt_res"], i4["kkt_res"]), v
        assert np.max(np.abs(cst - c4) / np.maximum(1.0, np.abs(c4))) <= 1e-12, v
    wa, ca, ia = res[0]
    _check_info(o, wa, ia)
    av = _expected_auto_variant(N, ev, B)
    if av is None:  # the warp-cooperative kernel: same decisions, other rounding
        assert np.max(np.abs(wa - w4)) <= 1e-12 * o.w_max
    else:
        assert np.array_equal(wa, res[av][0]) and np.array_equal(ia["iters"], res[av][2]["iters"]), av
        assert np.max(np.abs(ca - res[av][1]) / np.maximum(1.0, np.abs(res[av][1]))) <= 1e-12
    _check_oracle(N, o, w4, c4, lm, lr, gam, _sample(B, 3))


@pytest.mark.parametrize("N", [12, 24])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_register_kernel_broadcast_prices_and_invalid_last_row(ev, N):
    """Broadcast prices (lmbd_stride = 0, price_solver.py:203-204) on a grid of 256-thread CTAs equal the tiled rows;
    one NaN in the last QP of the partial last CTA is reported (ValueError) by every shape."""
    o, _ = _consts(ev)
    B = 70001
    rng = np.random.default_rng(31 + N + (ev == "large"))
    lm1 = 0.05 * o.theta * rng.random(3 * N) * (rng.random(3 * N) < 0.5)
    lr1 = 0.0 if ev == "large" else 2.0
    gam = o.y_max * rng.random(B)
    _, s = _solver(N, ev)
    wb, cb, ib = s.solve_lompc_batch(lm1, lr1, gam, return_info=True)
    wt, ct, it_ = s.solve_lompc_batch(np.tile(lm1, (B, 1)), np.full(B, lr1), gam, return_info=True)
    _check_info(o, wb, ib)
    assert np.array_equal(wb, wt) and np.array_equal(ib["iters"], it_["iters"])
    assert np.max(np.abs(cb - ct) / np.maximum(1.0, np.abs(ct))) <= 1e-12
    _check_oracle(N, o, wb, cb, lm1, lr1, gam, [0, 1, 65535, 65536, B - 2, B - 1])
    lm, lr, gam = _regimes(o, N, B, 77 + N)
    lm[B - 1, 3 * N - 1] = np.nan
    for v in (0, 4, 7, 9):
        s.set_kernel_variant(v)
        with pytest.raises(ValueError):
            s.solve_lompc_batch(lm, lr, gam)


@pytest.mark.parametrize("N", [12, 24])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_register_kernel_misaligned_buffers(ev, N):
    """Price rows and result rows at an odd storage offset (not 16-byte aligned): the register kernels load and store
    them per element instead of in pairs (and the bulk-copy kernel is not eligible).  Results are the bits of the
    aligned call, the doubles next to the views stay untouched."""
    import torch
    from chargingstation.lompc import LoMPC
    o, c = _consts(ev)
    dev = torch.device("cuda:0")
    s = LoMPC(N, c)
    for B in (65535, 65536):
        lm, lr, gam = _regimes(o, N, B, 500 + B + N)
        lm_al = torch.from_numpy(lm).to(dev)
        lr_d = torch.from_numpy(lr).to(dev)
        gam_d = torch.from_numpy(gam).to(dev)
        lm_buf = torch.full((B * 3 * N + 2,), float("nan"), dtype=torch.float64, device=dev)
        lm_mis = lm_buf[1:1 + B * 3 * N].view(B, 3 * N)
        lm_mis.copy_(lm_al)
        w_buf = torch.full((B * N + 2,), float("nan"), dtype=torch.float64, device=dev)
        w_mis = w_buf[1:1 + B * N].view(B, N)
        assert lm_mis.data_ptr() % 16 == 8 and w_mis.data_ptr() % 16 == 8
        for v in (0, 4, 7, 9):
            s.set_kernel_variant(v)
            w_a, c_a, i_a = s.solve_lompc_batch(lm_al, lr_d, gam_d, return_info=True)
            w_buf[1:-1] = float("nan")
            cost_m = torch.empty(B, dtype=torch.float64, device=dev)
            _, c_m, i_m = s.solve_lompc_batch(lm_mis, lr_d, gam_d, return_info=True, out=(w_mis, cost_m))
            torch.cuda.synchronize()
            assert torch.equal(w_mis, w_a), (B, v, (w_mis - w_a).abs().max().item())
            assert torch.equal(i_m["iters"], i_a["iters"]) and torch.equal(i_m["kkt_res"], i_a["kkt_res"]), (B, v)
            # (an aligned call of 65,536 rows at N = 24 takes the bulk-copy kernel, whose epilogue re-sums the cost)
            assert ((c_m - c_a).abs() / c_a.abs().clamp(min=1.0)).max().item() <= 1e-12, (B, v)
            assert torch.equal(i_m["status"], i_a["status"]) and int(i_a["status"].max()) == 0, (B, v)
            assert torch.isnan(w_buf[0]) and torch.isnan(w_buf[-1]), (B, v)
            assert torch.isnan(lm_buf[0]) and torch.isnan(lm_buf[-1]), (B, v)
        w = w_a.cpu().numpy()
        _check_oracle(N, o, w, c_a.cpu().numpy(), lm, lr, gam, [0, B // 2, B - 1])


# ------------------------------------------------------------------------------------------------------------------
# C. Group mode and the fused epilogues (error norm, w0, price0)
# ------------------------------------------------------------------------------------------------------------------
def _group_inputs(o, N, counts, seed):
    rng = np.random.default_rng(seed)
    G = len(counts)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    y0 = 0.05 + 0.8 * rng.random(int(off[-1]))
    lmbd = np.zeros((G, 3 * N))
    lmbd[0::2] = o.theta * rng.random((len(range(0, G, 2)), 3 * N))
    lmbd[1::2] = 0.05 * o.theta * rng.random((len(range(1, G, 2)), 3 * N)) * (rng.random((len(range(1, G, 2)), 3 * N)) < 0.5)
    lmbd_r = np.where(np.arange(G) % 3 == 0, 0.0, 3 * N * o.delta * rng.random(G))
    w_ref = o.w_max * rng.random((G, N))
    return off, y0, lmbd, lmbd_r, w_ref


def _group_outputs(ps, off, y0, lmbd, lmbd_r, w_ref):
    """get_w0_price0_batch and price_w_err_dev (through ctypes) on the same groups."""
    import torch
    from chargingstation import _native
    N, G, B = ps.N, len(off) - 1, int(off[-1])
    w0, p0 = ps.get_w0_price0_batch(off, y0, lmbd, lmbd_r)
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    d_off, d_gam, d_lm, d_lr, d_wr = t(off), t(ps.consts.y_max - y0), t(lmbd), t(lmbd_r), t(w_ref)
    w_avg = torch.full((G, N), float("nan"), dtype=torch.float64, device=dev)
    e_max, e0, e_avg = (torch.full((G,), float("nan"), dtype=torch.float64, device=dev) for _ in range(3))
    w0_b = torch.full((B,), float("nan"), dtype=torch.float64, device=dev)
    rc = ps._lib.price_w_err_dev(ps._h, G, B, d_off.data_ptr(), d_gam.data_ptr(), d_lm.data_ptr(), d_lr.data_ptr(),
                                 d_wr.data_ptr(), w_avg.data_ptr(), e_max.data_ptr(), e0.data_ptr(), e_avg.data_ptr(),
                                 w0_b.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _native.raise_for(rc)
    torch.cuda.synchronize()
    return {"w0": w0, "price0": p0, "w0_err_path": w0_b.cpu().numpy(), "w_avg": w_avg.cpu().numpy(),
            "w_err_max": e_max.cpu().numpy(), "w0_err": e0.cpu().numpy(), "w_avg_err": e_avg.cpu().numpy()}


def _group_reference(o, N, off, y0, lmbd, lmbd_r, w_ref, variant):
    """price_solver.get_w_err / get_w0_price0 restated in float64 numpy on QPs solved through the plain path."""
    G = len(off) - 1
    counts = np.diff(off)
    grp = np.repeat(np.arange(G), counts)
    _, s = _solver(N, o.ev_type, variant)
    lm_ev, lr_ev, gam = lmbd[grp], lmbd_r[grp], o.y_max - y0
    w, cost, info = s.solve_lompc_batch(lm_ev, lr_ev, gam, return_info=True)
    _check_info(o, w, info)
    q = 3 * o.theta / (4 * o.w_max)
    x0 = w[:, 0]
    p0_ev = (o.theta * (x0 * lm_ev[:, 0] + (o.w_max - x0) * lm_ev[:, N]) + q * x0 * x0 * lm_ev[:, 2 * N]
             + o.theta ** 2 * x0 * x0 * lr_ev)                      # lompc.py:164-170
    ref = {"w": w, "cost": cost, "lm_ev": lm_ev, "lr_ev": lr_ev, "gam": gam, "price0": np.full(G, np.nan),
           "w_avg": np.full((G, N), np.nan), "w_err_max": np.full(G, np.nan), "w0_err": np.full(G, np.nan),
           "w_avg_err": np.full(G, np.nan)}

    def a_norm(v, kap):  # sqrt(v' (A'A + kappa I) v), A = tril(ones)
        return np.sqrt(np.sum(np.cumsum(v, axis=-1) ** 2, axis=-1) + kap * np.sum(v * v, axis=-1))

    for g in np.flatnonzero(counts):  # (sums in EV order, as price_solver.py:205 adds them)
        sl = slice(off[g], off[g + 1])
        kap = lmbd_r[g] / o.delta
        ref["price0"][g] = np.cumsum(p0_ev[sl])[-1] / counts[g]
        wa = np.cumsum(w[sl], axis=0)[-1] / counts[g]
        ref["w_avg"][g] = wa
        ref["w_err_max"][g] = np.max(a_norm(w[sl] - w_ref[g], kap))
        ref["w_avg_err"][g] = a_norm(wa - w_ref[g], kap)
        ref["w0_err"][g] = abs(wa[0] - w_ref[g, 0])
    return ref


def _close(a, b, rtol, floor):
    return np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(b), floor))


@pytest.mark.parametrize("N", [12, 24, 36, 48, 96])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_group_mode_epilogues(ev, N):
    """get_w0_price0 (price_solver.py:272-285) and _get_w_err (:196-214) for groups of 1, 2, 0, 63, 64, 65 and 300 EVs:
    the thread kernels (64 x 4 at N = 12, 24; the any-N kernel otherwise) with group rows, w0 / price0 / error-norm
    epilogues, against the same QPs solved through the plain path.  Removing the empty group changes no other
    group's numbers."""
    from chargingstation.price_solver import PriceSolver
    o, c = _consts(ev)
    counts = [1, 2, 0, 63, 64, 65, 300]
    off, y0, lmbd, lmbd_r, w_ref = _group_inputs(o, N, counts, 60 + N + (ev == "large"))
    ps = PriceSolver(N, c, "linear-convex")
    out = _group_outputs(ps, off, y0, lmbd, lmbd_r, w_ref)
    ref = _group_reference(o, N, off, y0, lmbd, lmbd_r, w_ref, 4 if N in (12, 24) else 1)
    _assert_group_outputs(o, off, out, ref)
    B = int(off[-1])
    _check_oracle(N, o, ref["w"], ref["cost"], ref["lm_ev"], ref["lr_ev"], ref["gam"], list(range(0, B, 41)) + [B - 1])
    # the same groups without the empty one
    keep = [g for g in range(len(counts)) if counts[g] > 0]
    off2 = np.concatenate([[0], np.cumsum([counts[g] for g in keep])]).astype(np.int32)
    out2 = _group_outputs(ps, off2, y0, lmbd[keep], lmbd_r[keep], w_ref[keep])
    assert np.array_equal(out2["w0"], out["w0"]) and np.array_equal(out2["w0_err_path"], out["w0_err_path"])
    for k in ("price0", "w_err_max", "w0_err", "w_avg_err", "w_avg"):
        assert np.array_equal(out2[k], out[k][keep]), k


@pytest.mark.parametrize("N", [12, 24])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_group_mode_epilogues_full_grid(ev, N):
    """70,000 EVs in group mode: the large EV takes the 256 x 1 register kernel (>= 65,536 QPs)."""
    from chargingstation.price_solver import PriceSolver
    o, c = _consts(ev)
    counts = [1, 2, 0, 63, 64, 65, 70000 - 195]
    off, y0, lmbd, lmbd_r, w_ref = _group_inputs(o, N, counts, 90 + N + (ev == "large"))
    ps = PriceSolver(N, c, "linear-convex")
    out = _group_outputs(ps, off, y0, lmbd, lmbd_r, w_ref)
    ref = _group_reference(o, N, off, y0, lmbd, lmbd_r, w_ref, 4)
    _assert_group_outputs(o, off, out, ref)
    B = int(off[-1])
    _check_oracle(N, o, ref["w"], ref["cost"], ref["lm_ev"], ref["lr_ev"], ref["gam"], [0, 1, 3, 131, 195, 40000, B - 1])


def _assert_group_outputs(o, off, out, ref):
    ne = np.flatnonzero(np.diff(off))
    w0_ref = ref["w"][:, 0]
    assert np.max(np.abs(out["w0"] - w0_ref)) <= 1e-12 * o.w_max
    assert np.max(np.abs(out["w0_err_path"] - w0_ref)) <= 1e-12 * o.w_max
    assert _close(out["price0"][ne], ref["price0"][ne], 1e-12, 1e-300), (out["price0"][ne], ref["price0"][ne])
    assert _close(out["w_avg"][ne], ref["w_avg"][ne], 1e-11, o.w_max)
    for k in ("w_err_max", "w0_err", "w_avg_err"):
        assert _close(out[k][ne], ref[k][ne], 1e-11, o.w_max), (k, out[k][ne], ref[k][ne])


# ------------------------------------------------------------------------------------------------------------------
# D. Warp-kernel edge cases at 4, 16 and 32 lanes per QP
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [12, 48, 96])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_warp_kernel_edge_cases(ev, N):
    from chargingstation.lompc import LoMPC
    o, c = _consts(ev)
    solver = LoMPC(N, c)
    solver.set_kernel_variant(8)
    thread = LoMPC(N, c)
    thread.set_kernel_variant(4 if N == 12 else 1)
    z = np.zeros(3 * N)
    w, cost = solver.solve_lompc(z, 0.0, 0.0)
    assert np.all(w == 0.0) and cost == 0.0
    w, cost = solver.solve_lompc(z, 0.0, o.y_max)
    wo, co, _ = orc.solve_active_set(N, o, z, 0.0, o.y_max)
    assert np.max(np.abs(w - wo)) <= W_RTOL * o.w_max and abs(cost - co) <= C_RTOL * abs(co)
    big = np.concatenate([1e4 * np.ones(N), np.zeros(2 * N)])
    assert np.all(solver.solve_lompc(big, 0.0, 0.5)[0] == 0.0)
    neg = np.concatenate([np.zeros(N), 1e4 * np.ones(N), np.zeros(N)])
    assert np.all(solver.solve_lompc(neg, 0.0, 0.5)[0] == o.w_max)
    rng = np.random.default_rng(4 + N)
    cases = []
    # gamma = 0 and gamma = y_max with random prices
    lm = o.theta * rng.random((8, 3 * N))
    cases.append((lm, 3 * N * o.delta * rng.random(8), np.r_[np.zeros(4), np.full(4, o.y_max)]))
    # regulariser-size prices (lmbd3 ~ 1e11 where w ~ 0)
    lm = 0.05 * o.theta * rng.random((8, 3 * N))
    lm[:, 2 * N::3] = 1e11
    cases.append((lm, np.zeros(8), o.y_max * rng.random(8)))
    # exact-zero stage curvature (large EV: lmbd_r = 0 and lmbd3_k = 0)
    lm = 0.05 * o.theta * rng.random((8, 3 * N)) * (rng.random((8, 3 * N)) < 0.5)
    lm[:, 2 * N:] *= rng.random((8, N)) < 0.3
    cases.append((lm, np.zeros(8), o.y_max * rng.random(8)))
    for lm, lr, gam in cases:
        w, cost, info = solver.solve_lompc_batch(lm, lr, gam, return_info=True)
        assert np.all(info["status"] == 0)
        w_t, cost_t = thread.solve_lompc_batch(lm, lr, gam)
        assert np.max(np.abs(w - w_t)) <= 1e-11 * o.w_max
        assert np.max(np.abs(cost - cost_t) / np.maximum(1, np.abs(cost_t))) <= 1e-12
        _check_oracle(N, o, w, cost, lm, lr, gam, range(len(gam)))
    # per-QP status and the reference's exceptions (lompc.py:78-90)
    lm = o.theta * rng.random((5, 3 * N))
    with pytest.raises(AssertionError):
        solver.solve_lompc_batch(lm, 0.0, np.array([0.1, 0.2, o.y_max + 0.01, 0.3, 0.4]))
    lm2 = lm.copy()
    lm2[3, 7] = -1.0
    with pytest.raises(ValueError):
        solver.solve_lompc_batch(lm2, 0.0, np.full(5, 0.2))
    lm2[3, 7] = np.nan
    with pytest.raises(ValueError):
        solver.solve_lompc_batch(lm2, 0.0, np.full(5, 0.2))
    lm2[3, 7] = 0.1
    with pytest.raises((ValueError, AssertionError)):
        solver.solve_lompc_batch(lm2, 0.0, np.array([0.2, 0.2, np.nan, 0.2, 0.2]))


@pytest.mark.parametrize("N", [12, 48, 96])
@pytest.mark.parametrize("ev", ["small", "large"])
def test_warp_kernel_mixed_regimes_in_one_warp(ev, N):
    """Consecutive QPs cycle through gamma = 0, lmbd3 = 1e11, zero stage curvature (lmbd_r = 0, sparse lmbd3) and test
    prices, so every warp holds lane groups in different regimes iterating in lock step.  Each QP matches its solve
    alone (B = 1) and the oracle."""
    o, s = _solver(N, ev, 8)
    rng = np.random.default_rng(70 + N + (ev == "large"))
    B = 64
    lm = np.zeros((B, 3 * N))
    lr = np.zeros(B)
    gam = o.y_max * rng.random(B)
    for b in range(B):
        kind = b % 4
        if kind == 0:
            lm[b] = o.theta * rng.random(3 * N)
            lr[b] = 3 * N * o.delta * rng.random()
            gam[b] = 0.0
        elif kind == 1:
            lm[b] = 0.05 * o.theta * rng.random(3 * N)
            lm[b, 2 * N::3] = 1e11
        elif kind == 2:
            lm[b] = 0.05 * o.theta * rng.random(3 * N) * (rng.random(3 * N) < 0.5)
            lm[b, 2 * N:] *= rng.random(N) < 0.3
        else:
            lm[b] = o.theta * rng.random(3 * N)
            lr[b] = 3 * N * o.delta * rng.random()
    w, cost, info = s.solve_lompc_batch(lm, lr, gam, return_info=True)
    _check_info(o, w, info)
    for b in range(B):
        w1, c1, i1 = s.solve_lompc_batch(lm[b:b + 1], lr[b:b + 1], gam[b:b + 1], return_info=True)
        assert i1["status"][0] == 0
        assert np.max(np.abs(w[b] - w1[0])) <= 1e-11 * o.w_max, (b, np.max(np.abs(w[b] - w1[0])))
        assert abs(cost[b] - c1[0]) <= 1e-12 * max(1.0, abs(c1[0])), b
    _check_oracle(N, o, w, cost, lm, lr, gam, range(B))


# ------------------------------------------------------------------------------------------------------------------
# E. Solve set: 1..4 segments, empty segments, every launch mode
# ------------------------------------------------------------------------------------------------------------------
# (EV types, batch sizes): one segment; three with an empty first one (mapped host blocks where the warp kernel
# exists); four with an empty middle one and 9,500 QPs (staged copies, one warp launch); four with an empty last one
# and 18,000 QPs (N = 12, 24: one thread-kernel launch per segment + the status reduction)
SET_LAYOUTS = {
    "one": (["small"], [301]),
    "three_empty_first": (["large", "small", "large"], [0, 517, 300]),
    "four_empty_mid": (["small", "large", "large", "small"], [3000, 0, 2500, 4000]),
    "four_empty_last": (["large", "small", "small", "large"], [6000, 5000, 7000, 0]),
}


def _set_uses_warp_kernel(N, total):
    return N in (48, 96) or (N in (12, 24) and total <= 16384)


def _object_uses_warp_kernel(N, B):
    return N in (48, 96) or (N == 12 and B <= 4096) or (N == 24 and B <= 6144)


@pytest.mark.parametrize("layout", list(SET_LAYOUTS))
@pytest.mark.parametrize("N", [12, 24, 36, 48, 96])
def test_solve_set_segments(N, layout):
    import torch
    from chargingstation.lompc import LoMPC, LoMPCSet
    evs, sizes = SET_LAYOUTS[layout]
    consts = [_consts(ev) for ev in evs]
    solvers = [LoMPC(N, c) for _, c in consts]
    sset = LoMPCSet(solvers, sizes)
    total = sum(sizes)
    data = []
    for i, (o, _) in enumerate(consts):
        lm, lr, gam = _regimes(o, N, sizes[i], 300 + 11 * i + N)
        sset.lmbd[i][:], sset.lmbd_r[i][:], sset.gamma[i][:] = lm, lr, gam
        data.append((lm, lr, gam))
    sset.solve(info=True)
    for i, (o, _) in enumerate(consts):
        B = sizes[i]
        if B == 0:
            continue
        lm, lr, gam = data[i]
        w, cost, info = solvers[i].solve_lompc_batch(lm, lr, gam, return_info=True)
        assert np.all(sset.status[i] == 0) and sset.kkt_res[i].max() <= 1e-10, i
        if _set_uses_warp_kernel(N, total) == _object_uses_warp_kernel(N, B):
            assert np.array_equal(sset.w[i], w) and np.array_equal(sset.cost[i], cost), i
            assert np.array_equal(sset.iters[i], info["iters"]) and np.array_equal(sset.kkt_res[i], info["kkt_res"]), i
        else:
            assert np.max(np.abs(sset.w[i] - w)) <= 1e-12 * o.w_max, i
            assert np.max(np.abs(sset.cost[i] - cost) / np.maximum(1.0, np.abs(cost))) <= 1e-12, i
        _check_oracle(N, o, sset.w[i], sset.cost[i], lm, lr, gam, _sample(B, 2 if N <= 48 else 1))
    results = [(sset.w[i].copy(), sset.cost[i].copy()) for i in range(len(sizes))]

    # solve_dev_at: two caller-owned block pairs with the set's layout, solved back to back
    dev = torch.device("cuda:0")
    data2 = [(lm, 0.5 * lr, 0.5 * gam) for lm, lr, gam in data]
    blocks = []
    for epoch, dset in ((7, data), (9, data2)):
        inb = torch.zeros(sset.h2d_bytes // 8, dtype=torch.float64, device=dev)
        outb = torch.zeros(sset.d2h_bytes // 8, dtype=torch.float64, device=dev)
        inb.view(torch.int64)[0] = epoch
        for i, (lm, lr, gam) in enumerate(dset):
            o_lm, o_lr, o_ga, _, _ = sset.offsets(i)
            B = sizes[i]
            inb[o_lm // 8: o_lm // 8 + B * 3 * N] = torch.from_numpy(lm.reshape(-1)).to(dev)
            inb[o_lr // 8: o_lr // 8 + B] = torch.from_numpy(lr).to(dev)
            inb[o_ga // 8: o_ga // 8 + B] = torch.from_numpy(gam).to(dev)
        blocks.append((epoch, inb, outb))
    stream = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    for _, inb, outb in blocks:
        sset.solve_dev_at(inb.data_ptr(), outb.data_ptr(), stream)
    torch.cuda.synchronize()
    for i in range(len(sizes)):
        sset.lmbd[i][:], sset.lmbd_r[i][:], sset.gamma[i][:] = data2[i]
    sset.solve()
    results2 = [(sset.w[i].copy(), sset.cost[i].copy()) for i in range(len(sizes))]
    for (epoch, _, outb), res in zip(blocks, (results, results2)):
        out = outb.cpu().numpy()
        assert int(out[:1].view(np.int64)[0]) == 4 * epoch  # epoch * 4 + worst status (OK)
        for i in range(len(sizes)):
            _, _, _, o_w, o_c = sset.offsets(i)
            B = sizes[i]
            assert np.array_equal(out[o_w // 8: o_w // 8 + B * N].reshape(B, N), res[i][0]), (epoch, i)
            assert np.array_equal(out[o_c // 8: o_c // 8 + B], res[i][1]), (epoch, i)

    if layout == "four_empty_mid":  # error conventions with the failure in the third / the last segment
        for i in range(len(sizes)):
            sset.lmbd[i][:], sset.lmbd_r[i][:], sset.gamma[i][:] = data[i]
        sset.lmbd[2][sizes[2] - 1, 5] = np.nan
        with pytest.raises(ValueError):
            sset.solve()
        sset.lmbd[2][sizes[2] - 1, 5] = 0.1
        sset.gamma[3][sizes[3] - 1] = consts[3][0].y_max + 0.01
        with pytest.raises(AssertionError):
            sset.solve()
        sset.gamma[3][sizes[3] - 1] = 0.2
        sset.solve()
        w, _ = solvers[3].solve_lompc_batch(sset.lmbd[3].copy(), sset.lmbd_r[3].copy(), sset.gamma[3].copy())
        assert np.max(np.abs(sset.w[3] - w)) <= 1e-12 * consts[3][0].w_max
