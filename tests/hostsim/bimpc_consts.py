"""Host build of the per-station mode of csrc/bimpc_solve.cuh (test infrastructure only): the twin of
bimpc_solve_kernel<true>, next to the uniform twin ``hostsim.bimpc_solve``."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from hostsim import CSRC, _build, _p


def _lib():
    return C.CDLL(_build("bimpc_hostsim_consts", [os.path.join(CSRC, "bimpc_solve.cuh")]))


def bimpc_solve_consts(consts, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, omega, tol=1e-9,
                       max_iter=100):
    """The per-station mode of csrc/bimpc_solve.cuh on the host: `consts` holds one oracle BiConsts per station (they
    share N, P and the EV constants), `omega` [S, N] each station's stage weights."""
    lib = _lib()
    fn = lib.bimpc_hostsim_solve_consts
    fn.restype = C.c_int
    fn.argtypes = [C.c_int, C.c_int] + [C.c_double] * 4 + [C.c_int] + [C.c_void_p] * 21 + [C.c_double, C.c_int]
    c = consts[0]
    S = len(consts)
    assert all((k.N, k.P, k.theta_s, k.theta_l, k.w_max_s, k.w_max_l) == (c.N, c.P, c.theta_s, c.theta_l, c.w_max_s,
                                                                          c.w_max_l) for k in consts)
    arrs = [np.ascontiguousarray(np.atleast_2d(np.asarray(v, dtype=np.float64)))
            for v in (Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm)]
    assert arrs[0].shape[0] == S
    x0 = np.ascontiguousarray(np.atleast_1d(np.asarray(x0, dtype=np.float64)))
    demand = np.ascontiguousarray(np.atleast_2d(np.asarray(demand, dtype=np.float64)))
    omega = np.ascontiguousarray(omega, dtype=np.float64).reshape(S, c.N)
    st5 = [np.array([getattr(k, f) for k in consts], dtype=np.float64)
           for f in ("delta", "c_g", "u_g_max", "u_b_max", "x_max")]
    ct = np.array([k.cost_type for k in consts], dtype=np.int32)
    ws = np.zeros((S, c.P, c.N))
    wl = np.zeros((S, c.P, c.N))
    ug = np.zeros((S, c.N))
    st = np.zeros(S, dtype=np.int32)
    it = np.zeros(S, dtype=np.int32)
    obj = np.zeros(S)
    rc = fn(c.N, c.P, c.theta_s, c.theta_l, c.w_max_s, c.w_max_l, S, *[_p(v) for v in st5], _p(ct), _p(omega),
            *[_p(v) for v in arrs], _p(x0), _p(demand), _p(ws), _p(wl), _p(ug), _p(st), _p(it), _p(obj), tol, max_iter)
    assert rc == 0, rc
    return ws, wl, ug, {"status": st, "iters": it, "objective": obj}


def stage_weights_loop(N, cost_type, exp_rate):
    """The stage weights of the loop bimpc_create ran before bimpc_stage_weights existed."""
    lib = _lib()
    fn = lib.bimpc_hostsim_stage_weights_loop
    fn.restype = None
    fn.argtypes = [C.c_int, C.c_int, C.c_double, C.c_void_p]
    om = np.empty(N)
    fn(N, cost_type, exp_rate, _p(om))
    return om
