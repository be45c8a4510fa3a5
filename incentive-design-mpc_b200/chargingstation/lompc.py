"""Drop-in mirror of the reference's ``chargingstation/lompc.py`` (class and
method names, argument meaning, return types and error behaviour as in
lompc.py:12-187), with the cvxpy/CLARABEL solve replaced by the batched
sm_100a kernel behind ``include/lompc_b200.h``.

Added (not in the reference): ``LoMPC.solve_lompc_batch`` - the same solve for
a whole batch of (lmbd, lmbd_r, gamma) triples in one kernel launch; the scalar
``solve_lompc`` is that call with B = 1.  ``LoMPC.solve_lompc_diff`` / ``solve_lompc_vjp`` - the same solve with
a device-side vector-Jacobian product (chargingstation/autodiff.py)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from chargingstation import _native
from chargingstation.settings import (MAX_BAT_CHARGE_RATE, MAX_MAX_BAT_SOC,
                                      MIN_MAX_BAT_SOC)


@dataclass
class LoMPCConstants:
    """
    delta:      Relative weight of charging cost.
    theta:      Battery capacity [kWh].
    y_max:      Maximum allowed state of charge (SoC) as a fraction of capacity.
    w_max:      Maximum fraction of charge replenished per time step (normalized charging rate).
    ev_type:    EV type, either "small" or "large".
    """

    delta: float
    theta: float
    y_max: float
    w_max: float
    ev_type: str


def _is_torch_cuda(x) -> bool:
    return type(x).__module__.startswith("torch") and getattr(x, "is_cuda", False)


class LoMPC:
    def __init__(self, N: int, consts: LoMPCConstants, device: int = 0) -> None:
        """
        Inputs:
            N:      LoMPC horizon length.
            consts: LoMPC constants.
            device: CUDA device ordinal (extension; the reference is CPU-only).
        """
        # lompc.py:36-38
        assert (consts.y_max >= MIN_MAX_BAT_SOC) and (consts.y_max <= MAX_MAX_BAT_SOC)
        assert (consts.w_max >= 0) and (consts.w_max <= MAX_BAT_CHARGE_RATE)
        assert (consts.ev_type == "small") or (consts.ev_type == "large")
        self._set_constants(N, consts)
        self._lib = _native.load()
        self._h = C.c_void_p()
        rc = self._lib.lompc_create(
            self.N, float(self.delta), float(self.theta), float(self.y_max), float(self.w_max),
            _native.EV_LARGE if self.ev_type == "large" else _native.EV_SMALL, int(device),
            C.byref(self._h))
        _native.raise_for(rc)
        self.device = int(device)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._lib.lompc_destroy(h)
            self._h = C.c_void_p()

    def _set_constants(self, N: int, consts: LoMPCConstants) -> None:
        # lompc.py:59-71
        self.N = N
        self.delta = consts.delta
        self.theta = consts.theta
        self.y_max = consts.y_max
        self.w_max = consts.w_max
        self.ev_type = consts.ev_type
        # Scaling factor for the quadratic electricity cost.
        self.q_scale = 3 * self.theta / (4 * self.w_max)
        # LoMPC input matrix, y = A w.
        self.A = np.tril(np.ones((self.N, self.N)))
        # Strong convexity modulus.
        self.m = 2 * self.delta * self.theta ** 2

    # ------------------------------------------------------------------ solves
    def set_solver_options(self, max_iter: int = 200, tol: float = 1e-11) -> None:
        _native.raise_for(self._lib.lompc_set_options(self._h, int(max_iter), float(tol)))

    def set_kernel_variant(self, variant: int = 0) -> None:
        """0 = automatic; 1 = any-N shared-memory kernel; 2..7 = register-kernel shapes (tuning);
        8 = the warp-cooperative latency kernel; 9 = the register kernel with bulk-copied rows (include/lompc_b200.h)."""
        _native.raise_for(self._lib.lompc_set_kernel_variant(self._h, int(variant)))

    def solve_lompc(self, lmbd: np.ndarray, lmbd_r: float, gamma: float) -> tuple[np.ndarray, float]:
        """
        Inputs:
            lmbd:   Unit price (incentive) vector.
            lmbd_r: Robustness price parameter.
            gamma:  Fraction of battery capacity remaining to be charged.
        Outputs:
            w_opt:      Optimal w vector.
            cost_opt:   Optimal cost.
        """
        lmbd = np.ascontiguousarray(lmbd, dtype=np.float64)
        assert lmbd.shape == (3 * self.N,)
        # lompc.py:87 asserts first; then cvxpy validates the nonneg Parameters (lompc.py:78-82).
        assert gamma <= self.y_max
        if not (np.all(lmbd >= 0) and lmbd_r >= 0 and gamma >= 0):  # NaN is rejected too, as cvxpy does
            raise ValueError("Parameter value must be nonnegative.")
        w, cost = self.solve_lompc_batch(lmbd[None, :], np.array([lmbd_r], dtype=np.float64),
                                         np.array([gamma], dtype=np.float64))
        return w[0], float(cost[0])

    def solve_lompc_batch(self, lmbd, lmbd_r, gamma, return_info: bool = False, out=None, wait: bool = True):
        """Batched ``solve_lompc``.

        lmbd:   [B, 3N] or [3N] (one price vector broadcast to the batch, the
                ``_get_w_err`` case of price_solver.py:203-204).
        lmbd_r: [B] or scalar.   gamma: [B].
        numpy inputs  -> numpy outputs (host entry point, copies included);
        torch CUDA fp64 tensors -> torch CUDA tensors (device entry point,
        asynchronous on the current torch stream, no status check).
        Returns (w[B, N], cost[B]) and, with ``return_info``, a dict with
        ``status``, ``iters`` and ``kkt_res`` per QP.  ``out=(w, cost)`` reuses
        preallocated (e.g. pinned) output buffers.  ``wait=False`` (numpy path) only
        enqueues the copies and the kernel on this object's stream - call ``wait()``
        before reading the outputs; independent LoMPC objects overlap that way."""
        if _is_torch_cuda(gamma):
            return self._solve_batch_torch(lmbd, lmbd_r, gamma, return_info, out)
        N = self.N
        gamma = np.ascontiguousarray(np.atleast_1d(gamma), dtype=np.float64)
        B = gamma.shape[0]
        lmbd = np.ascontiguousarray(lmbd, dtype=np.float64)
        if lmbd.ndim == 1:
            assert lmbd.shape == (3 * N,)
            lm_stride = 0
        else:
            assert lmbd.shape == (B, 3 * N)
            lm_stride = 3 * N
        lmbd_r = np.ascontiguousarray(np.atleast_1d(lmbd_r), dtype=np.float64)
        if lmbd_r.shape[0] == 1 and B != 1:
            lr_stride = 0
        else:
            assert lmbd_r.shape == (B,)
            lr_stride = 1 if B > 1 else 0
        if out is not None:
            w, cost = out
            assert w.shape == (B, N) and cost.shape == (B,) and w.dtype == np.float64
            assert w.flags.c_contiguous and cost.flags.c_contiguous
        else:
            w = np.empty((B, N), dtype=np.float64)
            cost = np.empty((B,), dtype=np.float64)
        if return_info:
            status = np.empty((B,), dtype=np.int32)
            iters = np.empty((B,), dtype=np.int32)
            kkt = np.empty((B,), dtype=np.float64)
            ptrs = (status.ctypes.data, iters.ctypes.data, kkt.ctypes.data)
        else:
            ptrs = (None, None, None)  # the C side still fetches and checks the status
        fn = self._lib.lompc_solve_batch_host if wait else self._lib.lompc_solve_batch_host_async
        rc = fn(self._h, B, lmbd.ctypes.data, lm_stride, lmbd_r.ctypes.data, lr_stride,
                gamma.ctypes.data, w.ctypes.data, cost.ctypes.data, *ptrs)
        _native.raise_for(rc)
        if not wait:
            self._pending = (lmbd, lmbd_r, gamma, w, cost, ptrs)  # keep the host buffers alive
        if return_info:
            return w, cost, {"status": status, "iters": iters, "kkt_res": kkt}
        return w, cost

    def _solve_batch_torch(self, lmbd, lmbd_r, gamma, return_info, out=None):
        import torch

        N = self.N
        B = gamma.shape[0]
        dev = gamma.device
        assert gamma.dtype == torch.float64 and gamma.is_contiguous()
        assert lmbd.dtype == torch.float64 and lmbd.is_contiguous() and lmbd.device == dev
        lm_stride = 0 if lmbd.dim() == 1 else 3 * N
        assert lmbd.shape == ((3 * N,) if lm_stride == 0 else (B, 3 * N))
        if not torch.is_tensor(lmbd_r):
            lmbd_r = torch.full((1,), float(lmbd_r), dtype=torch.float64, device=dev)
        assert lmbd_r.dtype == torch.float64 and lmbd_r.device == dev
        lr_stride = 0 if lmbd_r.numel() == 1 else 1
        if out is not None:
            w, cost = out
            assert w.shape == (B, N) and w.is_contiguous() and cost.shape == (B,)
        else:
            w = torch.empty((B, N), dtype=torch.float64, device=dev)
            cost = torch.empty((B,), dtype=torch.float64, device=dev)
        if return_info:
            status = torch.empty((B,), dtype=torch.int32, device=dev)
            iters = torch.empty((B,), dtype=torch.int32, device=dev)
            kkt = torch.empty((B,), dtype=torch.float64, device=dev)
            ptrs = (status.data_ptr(), iters.data_ptr(), kkt.data_ptr())
        else:
            ptrs = (None, None, None)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = self._lib.lompc_solve_batch_dev(
            self._h, B, lmbd.data_ptr(), lm_stride, lmbd_r.data_ptr(), lr_stride,
            gamma.data_ptr(), w.data_ptr(), cost.data_ptr(), *ptrs, stream)
        _native.raise_for(rc)
        if return_info:
            return w, cost, {"status": status, "iters": iters, "kkt_res": kkt}
        return w, cost

    def solve_lompc_diff(self, lmbd, lmbd_r, gamma):
        """Differentiable ``solve_lompc_batch`` on fp64 CUDA tensors that may require grad (chargingstation/autodiff.py).

        lmbd: [B, 3N] or [3N] (broadcast); lmbd_r: [B], a one-element tensor (broadcast) or a float; gamma: [B].
        Returns (w[B, N], cost[B]); raises like ``solve_lompc`` on an invalid or unconverged QP (one host sync).
        Backward: one ``lompc_vjp_dev`` launch; a broadcast input receives the batch sum of the per-QP gradients.
        A coordinate of w within 1e-9 w_max of a breakpoint counts as fixed; at a weakly active coordinate, where w
        is not differentiable, the gradient is that of this active set (one of the one-sided derivatives)."""
        import torch

        from chargingstation.autodiff import LoMPCSolveFunction

        if not torch.is_tensor(lmbd_r):
            lmbd_r = torch.full((1,), float(lmbd_r), dtype=torch.float64, device=gamma.device)
        return LoMPCSolveFunction.apply(self, lmbd.contiguous(), lmbd_r.contiguous(), gamma.contiguous())

    def solve_lompc_vjp(self, lmbd, lmbd_r, gamma, w, grad_w=None, grad_cost=None, return_info: bool = False):
        """Vector-Jacobian product of ``solve_lompc_batch`` outside autograd (``lompc_vjp_dev``, asynchronous on the
        current torch stream).  ``w`` is the solution at (lmbd, lmbd_r, gamma); grad_w[B, N] / grad_cost[B] are
        the upstream gradients (None = zero).  Returns per-QP rows (grad_lmbd[B, 3N], grad_lmbd_r[B],
        grad_gamma[B]) even for broadcast inputs, and with ``return_info`` a dict with the per-QP ``status``
        (rows with invalid parameters get zero gradients and the solve's status code).  Same active-set
        convention as ``solve_lompc_diff``."""
        import torch

        from chargingstation.autodiff import lompc_vjp

        if not torch.is_tensor(lmbd_r):
            lmbd_r = torch.full((1,), float(lmbd_r), dtype=torch.float64, device=gamma.device)
        status = torch.empty(gamma.shape, dtype=torch.int32, device=gamma.device) if return_info else None
        grads = lompc_vjp(self, lmbd, lmbd_r, gamma, w, grad_w, grad_cost, status=status)
        return (*grads, {"status": status}) if return_info else grads

    def wait(self) -> None:
        """Completes a ``solve_lompc_batch(..., wait=False)``; raises like the blocking call."""
        rc = self._lib.lompc_host_wait(self._h)
        self._pending = None
        _native.raise_for(rc)

    # --------------------------------------------------------------- accessors
    def get_sc_modulus(self) -> float:
        return self.m

    def get_input_mat(self) -> np.ndarray:
        return self.A

    def get_price0(self, w: np.ndarray, lmbd: np.ndarray, lmbd_r: float) -> float:
        # lompc.py:164-170
        price0 = (
            self.theta * (w[0] * lmbd[0] + (self.w_max - w[0]) * lmbd[self.N])
            + self.q_scale * w[0] ** 2 * lmbd[2 * self.N]
            + self.theta ** 2 * w[0] ** 2 * lmbd_r
        )
        return price0

    def phi(self, w: np.ndarray) -> np.ndarray:
        assert w.shape == (self.N,)
        # Linear + quadratic prices are given by: lmbd @ phi(w).  (lompc.py:172-177)
        return np.hstack(
            (self.theta * w, self.theta * (self.w_max - w), self.q_scale * (w * w))
        )

    def Dphi(self, w: np.ndarray) -> np.ndarray:
        assert w.shape == (self.N,)
        # lompc.py:179-187
        return np.vstack(
            (self.theta * np.eye(self.N), -self.theta * np.eye(self.N),
             2 * self.q_scale * np.diag(w))
        )


class LoMPCSet:
    """The QPs of several ``LoMPC`` objects (e.g. a station's small-EV and large-EV solver,
    charging_station.py:59-60) solved by ONE kernel launch with ONE copy each way
    (``lompc_set_*`` in include/lompc_b200.h).  Not in the reference: it replaces the
    caller-side loops over ``LoMPC.solve_lompc`` (test/test_lompc.py:30-40,
    price_solver.py:203-204) for callers that hold their inputs in host memory.

    The set owns packed pinned-host and device blocks; ``lmbd[i]``, ``lmbd_r[i]``,
    ``gamma[i]`` are numpy views of segment ``i`` of the pinned input block (write the
    inputs IN PLACE), ``w[i]`` / ``cost[i]`` views of the pinned output block (valid
    after ``solve()``), so neither side makes a staging copy."""

    def __init__(self, solvers, batch_sizes) -> None:
        solvers = list(solvers)
        batch_sizes = [int(b) for b in batch_sizes]
        assert len(solvers) == len(batch_sizes) and 1 <= len(solvers) <= 4
        assert all(s.N == solvers[0].N and s.device == solvers[0].device for s in solvers)
        self.solvers, self.batch_sizes = solvers, batch_sizes
        self.N, self.device = solvers[0].N, solvers[0].device
        self._lib = _native.load()
        self._h = C.c_void_p()
        hs = (C.c_void_p * len(solvers))(*[s._h for s in solvers])
        Bs = (C.c_int64 * len(solvers))(*batch_sizes)
        _native.raise_for(self._lib.lompc_set_create(hs, len(solvers), Bs, C.byref(self._h)))
        N = self.N
        self.lmbd, self.lmbd_r, self.gamma, self.w, self.cost = [], [], [], [], []
        self.status, self.iters, self.kkt_res = [], [], []
        self._dev_ptrs = []

        def view(ptr, shape, ctype, dtype):
            n = int(np.prod(shape))
            if n == 0:
                return np.empty(shape, dtype=dtype)
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(n,)).reshape(shape)

        for i, B in enumerate(batch_sizes):
            p = [C.c_void_p() for _ in range(5)]
            _native.raise_for(self._lib.lompc_set_buffers(self._h, 0, i, *[C.byref(x) for x in p]))
            self.lmbd.append(view(p[0], (B, 3 * N), C.c_double, np.float64))
            self.lmbd_r.append(view(p[1], (B,), C.c_double, np.float64))
            self.gamma.append(view(p[2], (B,), C.c_double, np.float64))
            self.w.append(view(p[3], (B, N), C.c_double, np.float64))
            self.cost.append(view(p[4], (B,), C.c_double, np.float64))
            q = [C.c_void_p() for _ in range(3)]
            _native.raise_for(self._lib.lompc_set_info_buffers(self._h, i, *[C.byref(x) for x in q]))
            self.status.append(view(q[0], (B,), C.c_int32, np.int32))
            self.iters.append(view(q[1], (B,), C.c_int32, np.int32))
            self.kkt_res.append(view(q[2], (B,), C.c_double, np.float64))
            d = [C.c_void_p() for _ in range(5)]
            _native.raise_for(self._lib.lompc_set_buffers(self._h, 1, i, *[C.byref(x) for x in d]))
            self._dev_ptrs.append(tuple(x.value for x in d))
        self.h2d_bytes = int(self._lib.lompc_set_bytes(self._h, 0))
        self.d2h_bytes = int(self._lib.lompc_set_bytes(self._h, 1))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._lib.lompc_set_destroy(h)
            self._h = C.c_void_p()

    def solve(self, info: bool = False) -> None:
        """Host round trip (one H2D copy, one launch, one D2H copy, synchronised); raises like ``solve_lompc``."""
        _native.raise_for(self._lib.lompc_set_solve_host(self._h, 1 if info else 0))

    def solve_async(self, info: bool = False) -> None:
        _native.raise_for(self._lib.lompc_set_solve_host_async(self._h, 1 if info else 0))

    def wait(self) -> None:
        _native.raise_for(self._lib.lompc_set_wait(self._h))

    def upload(self, stream: int = 0) -> None:
        """Copies the pinned input block to the device block (asynchronous on ``stream``)."""
        _native.raise_for(self._lib.lompc_set_copy(self._h, 0, stream))

    def download(self, stream: int = 0) -> None:
        _native.raise_for(self._lib.lompc_set_copy(self._h, 1, stream))

    def solve_dev(self, stream: int = 0, info: bool = False) -> None:
        """Launch only, device block to device block, asynchronous on ``stream`` (a raw cudaStream_t)."""
        _native.raise_for(self._lib.lompc_set_solve_dev(self._h, 1 if info else 0, stream))

    def solve_dev_at(self, in_block: int, out_block: int, stream: int = 0) -> None:
        """The set's launch on caller-owned device blocks of ``h2d_bytes`` / ``d2h_bytes`` bytes laid out like the
        set's own (``offsets(i)``): many resident batches can be solved back to back."""
        _native.raise_for(self._lib.lompc_set_solve_dev_at(self._h, in_block, out_block, stream))

    def offsets(self, i: int):
        """Byte offsets of segment ``i``: (lmbd, lmbd_r, gamma) in the input block, (w, cost) in the output block."""
        o = (C.c_int64 * 5)()
        _native.raise_for(self._lib.lompc_set_offsets(self._h, i, o))
        return tuple(int(x) for x in o)

    def device_pointers(self, i: int):
        """(lmbd, lmbd_r, gamma, w, cost) device addresses of segment ``i``."""
        return self._dev_ptrs[i]
