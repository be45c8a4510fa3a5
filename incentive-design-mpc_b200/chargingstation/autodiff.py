"""Differentiable batched LoMPC solve (not in the reference; its cvxpy problem is DPP-parametrised in lmbd, lmbd_r
and gamma, lompc.py:74-90, so cvxpy / cvxpylayers can differentiate it).

``LoMPCSolveFunction`` is a ``torch.autograd.Function``: its forward is the torch device path of
``LoMPC.solve_lompc_batch``, its backward one launch of ``lompc_vjp_dev`` (include/lompc_b200.h), a Riccati solve
with the upstream gradient as right-hand side on the free coordinates of w (DESIGN.md section 2).
``LoMPCGroupSolveFunction`` is the same for G groups of EVs that share their group's prices (the price loop's
structure): forward ``lompc_group_solve_dev`` (w and the group means), backward one ``lompc_group_vjp_dev`` call that
writes the [G, 3N] gradient directly, summed over each group's EVs in EV order.

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


def _ptr(x):
    return None if x is None else x.data_ptr()


def group_offsets_checked(group_off, B):
    """(offsets the kernels can run on, a device flag that is 1 if ``group_off`` is not 0 = off[0] <= ... <= off[G] = B).
    The kernels get a clamped, non-decreasing copy, so a malformed array is reported at the caller's next host sync
    (``raise_for_group_status``) and is never read out of bounds."""
    assert torch.is_tensor(group_off) and group_off.dtype == torch.int32 and group_off.is_cuda and group_off.dim() == 1 \
        and group_off.numel() >= 1, "group_off: int32 CUDA tensor [G+1]"
    off = group_off.contiguous()
    safe = torch.cummax(off.clamp(0, B), 0)[0]
    safe[0] = 0
    safe[-1] = B
    bad = (safe != off).any().to(torch.int32).reshape(1)
    return safe.contiguous(), bad


def raise_for_group_status(bad_off, status):
    """One host sync for a grouped solve: ValueError for malformed offsets, then ``raise_for_status``."""
    st = torch.cat([bad_off, status]).cpu()
    if int(st[0]):
        raise ValueError("group_off must satisfy 0 = off[0] <= off[1] <= ... <= off[G] = B")
    raise_for_status(st[1:])


def lompc_group_solve(solver, off, lmbd, lmbd_r, gamma):
    """One ``lompc_group_solve_dev`` call on the current torch stream: (w[B,N], w_avg[G,N], status[B])."""
    N = solver.N
    dev = gamma.device
    G, B = off.numel() - 1, gamma.shape[0]
    w = torch.empty((B, N), dtype=torch.float64, device=dev)
    w_avg = torch.empty((G, N), dtype=torch.float64, device=dev)
    status = torch.empty((B,), dtype=torch.int32, device=dev)
    rc = solver._lib.lompc_group_solve_dev(
        solver._h, G, B, off.data_ptr(), _ptr(lmbd) if G else None, _ptr(lmbd_r) if G else None,
        _ptr(gamma) if B else None, _ptr(w) if B else None, _ptr(w_avg) if G else None, _ptr(status) if B else None,
        torch.cuda.current_stream(dev).cuda_stream)
    _native.raise_for(rc)
    return w, w_avg, status


def lompc_group_vjp(solver, off, lmbd, lmbd_r, gamma, w, grad_w=None, grad_w_avg=None, need=(True, True, True),
                    status=None):
    """One ``lompc_group_vjp_dev`` call on the current torch stream.  Returns (grad_lmbd[G,3N], grad_lmbd_r[G],
    grad_gamma[B]); an entry whose flag in ``need`` is false is None and is not computed."""
    N = solver.N
    dev = gamma.device
    G, B = off.numel() - 1, gamma.shape[0]
    out = [torch.empty(shape, dtype=torch.float64, device=dev) if want else None
           for want, shape in zip(need, ((G, 3 * N), (G,), (B,)))]
    grad_w = None if grad_w is None else _f64_on(grad_w, dev, (B, N), "grad_w")
    grad_w_avg = None if grad_w_avg is None else _f64_on(grad_w_avg, dev, (G, N), "grad_w_avg")

    def p(x, n):
        return _ptr(x) if n else None
    rc = solver._lib.lompc_group_vjp_dev(
        solver._h, G, B, off.data_ptr(), p(lmbd, G), p(lmbd_r, G), p(gamma, B), p(w, B), p(grad_w, B),
        p(grad_w_avg, G), p(out[0], G), p(out[1], G), p(out[2], B), p(status, B),
        torch.cuda.current_stream(dev).cuda_stream)
    _native.raise_for(rc)
    return tuple(out)


class LoMPCGroupSolveFunction(torch.autograd.Function):
    """(w[B,N], w_avg[G,N]) = the grouped solve of G price rows over B EVs sorted by group, with a backward pass.
    group_off: int32 CUDA [G+1]; lmbd: [G,3N]; lmbd_r: [G] or a one-element tensor (broadcast to every group);
    gamma: [B]; fp64 CUDA tensors.  The gradient of a broadcast lmbd_r is the sum over the groups."""

    @staticmethod
    def forward(ctx, solver, group_off, lmbd, lmbd_r, gamma):
        N = solver.N
        dev = gamma.device
        B = gamma.shape[0]
        off, bad = group_offsets_checked(group_off, B)
        G = off.numel() - 1
        gamma = _f64_on(gamma, dev, (B,), "gamma")
        lmbd = _f64_on(lmbd, dev, (G, 3 * N), "lmbd")
        lmbd_r = _f64_on(lmbd_r, dev, lmbd_r.shape, "lmbd_r")
        assert lmbd_r.numel() == 1 or tuple(lmbd_r.shape) == (G,), "lmbd_r: one element or [G]"
        lr_g = lmbd_r.reshape(1).expand(G).contiguous() if lmbd_r.numel() == 1 else lmbd_r
        w, w_avg, status = lompc_group_solve(solver, off, lmbd, lr_g, gamma)
        raise_for_group_status(bad, status)
        ctx.solver = solver
        ctx.lr_shape = lmbd_r.shape
        ctx.lr_broadcast = lmbd_r.numel() == 1
        ctx.save_for_backward(off, lmbd, lr_g, gamma, w)
        ctx.set_materialize_grads(False)
        return w, w_avg

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_w, grad_w_avg):
        off, lmbd, lr_g, gamma, w = ctx.saved_tensors
        need = ctx.needs_input_grad[2:]
        if not any(need) or (grad_w is None and grad_w_avg is None):
            return (None,) * 5
        g_lm, g_lr, g_ga = lompc_group_vjp(ctx.solver, off, lmbd, lr_g, gamma, w, grad_w, grad_w_avg, need)
        if g_lr is not None and ctx.lr_broadcast:
            g_lr = g_lr.sum(dim=0).reshape(ctx.lr_shape)
        return None, None, g_lm, g_lr, g_ga
