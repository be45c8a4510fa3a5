"""Drop-in mirror of the reference's ``chargingstation/price_solver.py`` (class,
method names, arguments, return types, ``prev_prices`` warm start and the
``solver_stats`` keys of price_solver.py:16-285), with every cvxpy solve and
Python loop over EVs replaced by the batched sm_100a kernels behind
``include/lompc_b200.h``.

Added (not in the reference): ``PriceSolver.compute_optimal_prices_batch`` /
``get_w0_price0_batch`` - the same computations for G independent groups
(EV partitions, stations, scenarios) in one device-resident loop."""
from __future__ import annotations

import ctypes as C

import numpy as np

from chargingstation import _native
from chargingstation.lompc import LoMPC, LoMPCConstants
from chargingstation.price_regularizer import PriceRegularizer
from chargingstation.settings import (MAX_PRICE_SOLVER_ITERATIONS,
                                      PRICE_SOLVER_EPS_REG,
                                      PRICE_SOLVER_EPS_TOL,
                                      PRICE_SOLVER_TOL_TYPE)
from chargingstation import settings


def tol_type_max(tol_type: str | None, default: str) -> int:
    """The C ABI's tol_type_max flag for a tolerance type of the price loop's convergence test
    (settings.PRICE_SOLVER_TOL_TYPE, price_solver.py:121-128): "avg" (error of the mean response) or "max" (largest
    error of a single EV).  None takes ``default``, the module constant, as the reference does."""
    if tol_type is None:
        return 1 if default == "max" else 0
    if tol_type not in ("avg", "max"):
        raise ValueError(f'tol_type must be "avg" or "max", not {tol_type!r}')
    return 1 if tol_type == "max" else 0


class PriceSolver:
    def __init__(self, N: int, consts: LoMPCConstants, price_type: str, device: int = 0) -> None:
        """
        Inputs:
            N:          Horizon length.
            consts:     LoMPC constants.
            price_type: "linear" or "linear-convex".
        """
        assert (price_type == "linear") or (price_type == "linear-convex")
        self.lompc = LoMPC(N, consts, device=device)
        self._set_constants(N, consts, price_type)
        self.price_reg = PriceRegularizer(self.N, self.r, device=device)
        self.device = int(device)
        self._lib = _native.load()
        self._h = self.lompc._h

    def _set_constants(self, N: int, consts: LoMPCConstants, price_type: str) -> None:
        # price_solver.py:42-64
        self.nEVs = None
        self.N = N
        if price_type == "linear":
            self.r = 2 * self.N
        else:
            self.r = 3 * self.N
        self.consts = consts
        self.price_type = price_type
        # Initialize charge levels.
        self.y0 = None
        self.y0_rng = None
        self.gamma_sc = None
        self.gamma_sm = None
        # Initialize prices.
        self.prev_prices = np.zeros((self.r,))
        # LoMPC input matrix, y = A w + y_0 1.
        self.A = self.lompc.get_input_mat()
        # Gradient descent regularization weight.
        self.eps_reg = PRICE_SOLVER_EPS_REG
        # Gradient descent tolerance.
        self.eps_tol = PRICE_SOLVER_EPS_TOL
        # Strong convexity modulus.
        self.m = self.lompc.get_sc_modulus()

    # ------------------------------------------------------------------ helpers
    def _torch(self):
        import torch
        return torch, torch.device("cuda", self.device)

    def _dev(self, x, dtype=None):
        torch, dev = self._torch()
        t = torch.from_numpy(np.ascontiguousarray(x)) if isinstance(x, np.ndarray) else x
        if dtype is not None:
            t = t.to(dtype)
        return t.to(dev).contiguous()

    def _stream(self):
        torch, dev = self._torch()
        return torch.cuda.current_stream(dev).cuda_stream

    # ----------------------------------------------------- reference interface
    def set_charge_levels(self, y0: np.ndarray) -> None:
        """
        Inputs:
            y0: (nEVs,) ndarray: EV normalized SoC array.
        """
        assert all(y0 >= 0) and all(y0 <= self.consts.y_max)
        assert len(y0.shape) == 1
        self.nEVs = len(y0)
        self.y0 = y0
        self.y0_rng = (np.max(self.y0) - np.min(self.y0)) / 2  # = \bar{\Gamma}
        self.gamma_sc = self.consts.y_max - (np.max(self.y0) + np.min(self.y0)) / 2
        self.gamma_sm = self.consts.y_max - np.mean(self.y0)

    def compute_optimal_prices(self, w_ref: np.ndarray, lmbd_r: float) -> tuple[np.ndarray, dict]:
        """
        Inputs:
            w_ref:  Reference w vector (team-optimal solution) from the BiMPC.
            lmbd_r: Robustness price parameter.
        Outputs:
            lmbd:           Optimal unit price (incentive) vector.
            solver_stats:   Additional solver info.

        solver_stats is a dict with keys
            iter:                           Number of solver iterations.
            price_before_reg:               Price before regularization.
            price_after_reg:                Price after regularization.
            dual_cost_decrease_actual:      Decrease in -\\tilde{g}^*.
            dual_cost_decrease_predicted:   Decrease in -\\tilde{g}^*(., \\lambda^k).
        """
        w_ref = np.asarray(w_ref, dtype=np.float64)
        assert w_ref.shape == (self.N,)
        prev = np.zeros((1, 3 * self.N))
        prev[0, : self.r] = self.prev_prices
        prices, stats = self.compute_optimal_prices_batch(
            np.array([0, self.nEVs], dtype=np.int32), self.y0, w_ref[None, :], np.array([float(lmbd_r)]),
            prev, history=True)
        lmbd_k = prices[0]
        it = int(stats["iter"][0])
        if settings.PRINT_LEVEL >= 1:  # price_solver.py:150-164
            _, w0_err_bound = self.get_robustness_bounds(lmbd_r)
            _, w0_err, _ = self._get_w_err(lmbd_k, lmbd_r, w_ref, None)
            print(f"w0-error      : {w0_err:13.8f} | w0 error bound: {w0_err_bound:13.8f}")
        # Update previous prices.
        self.prev_prices = lmbd_k[: self.r]
        nrec = min(it, stats["hist_ac"].shape[1])
        solver_stats = {
            "iter": it,
            "price_before_reg": float(stats["price_before_reg"][0]),
            "price_after_reg": float(stats["price_after_reg"][0]),
            "dual_cost_decrease_actual": stats["hist_ac"][0, :nrec].copy(),
            "dual_cost_decrease_predicted": stats["hist_pred"][0, :nrec].copy(),
        }
        return lmbd_k, solver_stats

    def set_loop_mode(self, mode: int = 0) -> None:
        """Kernel behind ``compute_optimal_prices`` (include/lompc_b200.h: price_set_loop_mode): 0 automatic,
        1 phase-split loop, 2 parametric one-warp-per-group loop (EVs between two pivots with the same active
        set are interpolated), 3 thread-per-EV loop."""
        _native.raise_for(self._lib.price_set_loop_mode(self._h, int(mode)))

    def last_pivot_overflows(self) -> int:
        """Groups of the last parametric loop whose pivot pool ran out (their stuck intervals were solved EV by EV:
        exact, informational)."""
        return int(self._lib.price_last_cycles(self._h, 5))

    def last_nnqp_cap_hits(self) -> int:
        """Groups of the last device-resident loop whose price step hit the cap of its active-set iteration."""
        return int(self._lib.price_last_cycles(self._h, 6))

    def last_nnqp_fallbacks(self) -> int:
        """Groups of the last device-resident loop whose price step took the Lawson-Hanson fallback (informational)."""
        return int(self._lib.price_last_cycles(self._h, 8))

    def _warn_inexact(self) -> None:
        n = self.last_nnqp_cap_hits()
        q = int(self._lib.price_last_cycles(self._h, 7))
        if n or q:
            import warnings
            warnings.warn(f"price loop: {n} group(s) with a price step stopped at its iteration cap, "
                          f"{q} LoMPC solve(s) without status OK - prices may be inexact", RuntimeWarning, stacklevel=3)

    def get_gamma_sc(self) -> float:
        return self.gamma_sc

    def get_gamma_sm(self) -> float:
        return self.gamma_sm

    def get_robustness_bounds(self, lmbd_r: float) -> tuple[float, float]:
        kappa = lmbd_r / self.consts.delta + 1e-5
        w_err_bound = np.sqrt(self.N) * self.y0_rng + self.eps_tol
        w0_err_bound = w_err_bound * np.min((1, 1 / np.sqrt(kappa)))
        return w_err_bound, w0_err_bound

    def _get_w_inner_product_metric(self, lmbd_r: float) -> tuple[np.ndarray, np.ndarray]:
        kappa = lmbd_r / self.consts.delta
        A_bar = self.A.T @ self.A + kappa * np.eye(self.N)
        A_bar_inv = np.linalg.inv(A_bar)
        return A_bar, A_bar_inv

    def _get_w_err(self, lmbd: np.ndarray, lmbd_r: float, w_ref: np.ndarray, A_bar: np.ndarray
                   ) -> tuple[float, float, float]:
        """price_solver.py:196-214 (A_bar is implied by lmbd_r; the argument is kept for the signature)."""
        torch, dev = self._torch()
        lm = np.zeros((1, 3 * self.N))
        lm[0, : len(lmbd)] = lmbd
        off = self._dev(np.array([0, self.nEVs], dtype=np.int32))
        gamma = self._dev(self.consts.y_max - self.y0)
        out = torch.empty((3,), dtype=torch.float64, device=dev)
        # keep every device buffer referenced until the call has been issued
        lm_d, lr_d = self._dev(lm), self._dev(np.array([float(lmbd_r)]))
        wr_d = self._dev(np.asarray(w_ref, dtype=np.float64))
        rc = self._lib.price_w_err_dev(
            self._h, 1, self.nEVs, off.data_ptr(), gamma.data_ptr(), lm_d.data_ptr(), lr_d.data_ptr(),
            wr_d.data_ptr(), None, out[0:].data_ptr(), out[1:].data_ptr(), out[2:].data_ptr(), None,
            self._stream())
        _native.raise_for(rc)
        w_err_max, w0_err, w_avg_err = out.cpu().numpy()
        return float(w_err_max), float(w0_err), float(w_avg_err)

    def _price_gradient_descent_step(self, A_bar_inv: np.ndarray, w_ref: np.ndarray, w: np.ndarray,
                                     lmbd: np.ndarray, lmbd_r: float = None) -> np.ndarray:
        """price_solver.py:216-246.  The reference passes A_bar_inv; this mirror recovers
        kappa = lmbd_r/delta from it (A_bar_inv[0,0] is monotone in kappa) unless lmbd_r is given."""
        torch, dev = self._torch()
        if lmbd_r is None:
            # (A'A + kappa I)^{-1}: recover kappa from the trace identity tr(A_bar) = tr(A'A) + N kappa
            A_bar = np.linalg.inv(A_bar_inv)
            lmbd_r = max(0.0, (np.trace(A_bar) - np.trace(self.A.T @ self.A)) / self.N) * self.consts.delta
        lm = np.zeros((1, 3 * self.N))
        lm[0, : self.r] = lmbd
        lm_d = self._dev(lm)
        dec = torch.empty((1,), dtype=torch.float64, device=dev)
        st = torch.zeros((1,), dtype=torch.int32, device=dev)
        wr_d = self._dev(np.asarray(w_ref, dtype=np.float64))
        w_d = self._dev(np.asarray(w, dtype=np.float64))
        lr_d = self._dev(np.array([float(lmbd_r)]))
        rc = self._lib.price_step_dev(self._h, 1, self.r, wr_d.data_ptr(), w_d.data_ptr(), lr_d.data_ptr(),
                                      lm_d.data_ptr(), dec.data_ptr(), st.data_ptr(), self._stream())
        _native.raise_for(rc)
        if int(st.item()) != 0:
            raise RuntimeError("price step: active-set iteration cap reached")
        return lm_d.cpu().numpy()[0, : self.r], float(dec.item())

    def _regularize_prices(self, w: np.ndarray, lmbd: np.ndarray) -> np.ndarray:
        """
        w should be optimal for lmbd, i.e., w = w*(lmbd).
        """
        torch, dev = self._torch()
        lm = np.zeros((1, 3 * self.N))
        lm[0, : self.r] = lmbd
        lm_d = self._dev(lm)
        pp = torch.empty((2,), dtype=torch.float64, device=dev)
        w_d = self._dev(np.asarray(w, dtype=np.float64))
        rc = self._lib.price_regularize_dev(self._h, 1, self.r, w_d.data_ptr(), lm_d.data_ptr(),
                                            pp[0:].data_ptr(), pp[1:].data_ptr(), self._stream())
        _native.raise_for(rc)
        return lm_d.cpu().numpy()[0, : self.r]

    def get_w0_price0(self, lmbd: np.ndarray, lmbd_r: float) -> tuple[np.ndarray, float]:
        lm = np.zeros((1, 3 * self.N))
        lm[0, : self.r] = lmbd
        w0, price0 = self.get_w0_price0_batch(np.array([0, self.nEVs], dtype=np.int32), self.y0, lm,
                                              np.array([float(lmbd_r)]))
        return w0, float(price0[0])

    # ------------------------------------------------------- batched extension
    def compute_optimal_prices_batch(self, group_off, y0, w_ref, lmbd_r, prev_prices, history: bool = False,
                                     max_iter: int = MAX_PRICE_SOLVER_ITERATIONS, tol_type: str | None = None):
        """``compute_optimal_prices`` for G groups at once.

        group_off: int32 [G+1], EVs sorted by group.  y0: [B] SoCs.  w_ref: [G, N].
        lmbd_r: [G].  prev_prices: [G, 3N] warm start (zero padded for "linear").
        tol_type: "avg" or "max" (the convergence test, price_solver.py:121-128); None = PRICE_SOLVER_TOL_TYPE.
        Returns (prices [G, 3N] numpy, stats dict of arrays: iter, price_before_reg,
        price_after_reg, w_k [G, N], total_iters; with ``history`` also hist_ac /
        hist_pred [G, cap])."""
        tol_max = tol_type_max(tol_type, PRICE_SOLVER_TOL_TYPE)
        torch, dev = self._torch()
        N = self.N
        group_off = np.ascontiguousarray(group_off, dtype=np.int32)
        G = len(group_off) - 1
        y0 = np.ascontiguousarray(y0, dtype=np.float64)
        B = int(group_off[-1])
        assert y0.shape == (B,)
        # the assert of set_charge_levels (price_solver.py:71) is re-checked on the device
        prices = self._dev(np.ascontiguousarray(prev_prices, dtype=np.float64).reshape(G, 3 * N).copy())
        w_ref_d = self._dev(np.ascontiguousarray(w_ref, dtype=np.float64).reshape(G, N))
        lr_d = self._dev(np.ascontiguousarray(lmbd_r, dtype=np.float64).reshape(G))
        off_d = self._dev(group_off)
        y0_d = self._dev(y0)
        iters = torch.empty((G,), dtype=torch.int32, device=dev)
        pre = torch.zeros((G,), dtype=torch.float64, device=dev)
        post = torch.zeros((G,), dtype=torch.float64, device=dev)
        w_k = torch.zeros((G, N), dtype=torch.float64, device=dev)
        cap = max_iter if history else 0
        hist_ac = torch.zeros((G, max(cap, 1)), dtype=torch.float64, device=dev) if history else None
        hist_pred = torch.zeros((G, max(cap, 1)), dtype=torch.float64, device=dev) if history else None
        total = C.c_int32(0)
        rc = self._lib.price_solve_dev(
            self._h, G, B, off_d.data_ptr(), y0_d.data_ptr(), w_ref_d.data_ptr(), lr_d.data_ptr(), self.r,
            int(max_iter), tol_max, float(self.eps_reg), float(self.eps_tol),
            prices.data_ptr(), iters.data_ptr(), pre.data_ptr(), post.data_ptr(), w_k.data_ptr(),
            hist_ac.data_ptr() if history else None, hist_pred.data_ptr() if history else None, cap,
            C.byref(total), self._stream())
        _native.raise_for(rc)
        self._warn_inexact()
        stats = {"iter": iters.cpu().numpy(), "price_before_reg": pre.cpu().numpy(),
                 "price_after_reg": post.cpu().numpy(), "w_k": w_k.cpu().numpy(), "total_iters": total.value}
        if history:
            stats["hist_ac"] = hist_ac.cpu().numpy()
            stats["hist_pred"] = hist_pred.cpu().numpy()
        return prices.cpu().numpy(), stats

    def get_w0_price0_batch(self, group_off, y0, lmbd, lmbd_r):
        """``get_w0_price0`` for G groups: returns (w0 [B], price0 [G])."""
        torch, dev = self._torch()
        N = self.N
        group_off = np.ascontiguousarray(group_off, dtype=np.int32)
        G = len(group_off) - 1
        B = int(group_off[-1])
        y0 = np.ascontiguousarray(y0, dtype=np.float64)
        assert np.all(y0 >= 0) and np.all(y0 <= self.consts.y_max)
        gamma = self._dev(self.consts.y_max - y0)
        w0 = torch.zeros((B,), dtype=torch.float64, device=dev)
        p0 = torch.zeros((G,), dtype=torch.float64, device=dev)
        off_d = self._dev(group_off)
        lm_d = self._dev(np.ascontiguousarray(lmbd, dtype=np.float64).reshape(G, 3 * N))
        lr_d = self._dev(np.ascontiguousarray(lmbd_r, dtype=np.float64).reshape(G))
        rc = self._lib.price_w0_price0_dev(self._h, G, B, off_d.data_ptr(), gamma.data_ptr(), lm_d.data_ptr(),
                                           lr_d.data_ptr(), w0.data_ptr(), p0.data_ptr(), self._stream())
        _native.raise_for(rc)
        return w0.cpu().numpy(), p0.cpu().numpy()
