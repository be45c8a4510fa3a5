"""Differentiable batched LoMPC solve (not in the reference; its cvxpy problem is DPP-parametrised in lmbd, lmbd_r
and gamma, lompc.py:74-90, so cvxpy / cvxpylayers can differentiate it).

``LoMPCSolveFunction`` is a ``torch.autograd.Function``: its forward is the torch device path of
``LoMPC.solve_lompc_batch``, its backward one launch of ``lompc_vjp_dev`` (include/lompc_b200.h), a Riccati solve
with the upstream gradient as right-hand side on the free coordinates of w (DESIGN.md section 2).

Active-set convention: a coordinate of w within 1e-9 w_max of a breakpoint (0, w_max, an interior large-EV pwl
breakpoint) counts as fixed.  At a weakly active coordinate w is not differentiable; the gradient returned there
is that of the classified active set, one of the one-sided derivatives.  The cost gradient is exact everywhere."""
from __future__ import annotations

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from chargingstation import _native


def raise_for_status(status: torch.Tensor) -> None:
    """Raises like the host entry point (``lompc_host_wait``) for the per-QP status of a device solve: the first
    bad gamma (AssertionError) or negative parameter (ValueError) in row order, else a non-converged QP
    (RuntimeError)."""
    st = status.cpu().numpy()
    bad = np.flatnonzero((st == _native.ST_BAD_GAMMA) | (st == _native.ST_NEGATIVE))
    if bad.size:
        _native.raise_for(_native.ERR_GAMMA if st[bad[0]] == _native.ST_BAD_GAMMA else _native.ERR_NEGATIVE)
    if (st == _native.ST_MAXITER).any():
        _native.raise_for(_native.ERR_NOT_CONVERGED)


def _f64_on(x, dev, shape, name):
    assert torch.is_tensor(x) and x.dtype == torch.float64 and x.device == dev, f"{name}: fp64 tensor on {dev}"
    assert tuple(x.shape) == tuple(shape), f"{name}: shape {tuple(x.shape)}, expected {tuple(shape)}"
    return x.contiguous()


def lompc_vjp(solver, lmbd, lmbd_r, gamma, w, grad_w=None, grad_cost=None, need=(True, True, True), status=None):
    """One ``lompc_vjp_dev`` launch on the current torch stream.  Returns per-QP (grad_lmbd[B,3N], grad_lmbd_r[B],
    grad_gamma[B]); an entry whose flag in ``need`` is false is None and is not computed."""
    N = solver.N
    dev = gamma.device
    B = gamma.shape[0]
    gamma = _f64_on(gamma, dev, (B,), "gamma")
    lmbd = _f64_on(lmbd, dev, (3 * N,) if lmbd.dim() == 1 else (B, 3 * N), "lmbd")
    lmbd_r = _f64_on(lmbd_r, dev, lmbd_r.shape, "lmbd_r")
    assert lmbd_r.numel() == 1 or tuple(lmbd_r.shape) == (B,), "lmbd_r: scalar or [B]"
    w = _f64_on(w, dev, (B, N), "w")
    grad_w = None if grad_w is None else _f64_on(grad_w, dev, (B, N), "grad_w")
    grad_cost = None if grad_cost is None else _f64_on(grad_cost, dev, (B,), "grad_cost")
    out = [torch.empty(shape, dtype=torch.float64, device=dev) if want else None
           for want, shape in zip(need, ((B, 3 * N), (B,), (B,)))]
    if status is not None:
        assert status.dtype == torch.int32 and status.device == dev and tuple(status.shape) == (B,)
    if B == 0:  # (an empty tensor has no storage to point at)
        return tuple(x.zero_() if x is not None else None for x in out)

    def ptr(x):
        return None if x is None else x.data_ptr()

    rc = solver._lib.lompc_vjp_dev(
        solver._h, B, lmbd.data_ptr(), 0 if lmbd.dim() == 1 else 3 * N, lmbd_r.data_ptr(),
        0 if lmbd_r.numel() == 1 else 1, gamma.data_ptr(), w.data_ptr(), ptr(grad_w), ptr(grad_cost),
        ptr(out[0]), ptr(out[1]), ptr(out[2]), ptr(status), torch.cuda.current_stream(dev).cuda_stream)
    _native.raise_for(rc)
    return tuple(out)


class LoMPCSolveFunction(torch.autograd.Function):
    """(w[B,N], cost[B]) = solve(lmbd, lmbd_r, gamma) with a backward pass.  lmbd: [B,3N] or [3N] (broadcast),
    lmbd_r: [B] or a one-element tensor (broadcast), gamma: [B]; fp64 CUDA tensors.  The gradient of a broadcast
    input is the (deterministic) sum over the batch of the per-QP gradients."""

    @staticmethod
    def forward(ctx, solver, lmbd, lmbd_r, gamma):
        if gamma.shape[0] == 0:  # (an empty tensor has no storage to point at)
            w, cost = gamma.new_empty((0, solver.N)), gamma.new_empty((0,))
        else:
            w, cost, info = solver.solve_lompc_batch(lmbd, lmbd_r, gamma, return_info=True)
            raise_for_status(info["status"])
        ctx.solver = solver
        ctx.save_for_backward(lmbd, lmbd_r, gamma, w)
        ctx.set_materialize_grads(False)
        return w, cost

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_w, grad_cost):
        lmbd, lmbd_r, gamma, w = ctx.saved_tensors
        need = ctx.needs_input_grad[1:]
        if not any(need) or (grad_w is None and grad_cost is None):
            return (None, None, None, None)
        g_lm, g_lr, g_ga = lompc_vjp(ctx.solver, lmbd, lmbd_r, gamma, w, grad_w, grad_cost, need)
        if g_lm is not None and lmbd.dim() == 1:
            g_lm = g_lm.sum(dim=0)
        if g_lr is not None:
            g_lr = (g_lr.sum(dim=0) if lmbd_r.numel() == 1 else g_lr).reshape(lmbd_r.shape)
        return None, g_lm, g_lr, g_ga
