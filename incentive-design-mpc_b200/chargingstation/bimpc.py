"""Drop-in mirror of the reference's ``chargingstation/bimpc.py`` (upper-level,
team-optimal MPC): same enum, dataclasses, constructor asserts, ``solve_bimpc`` signature
and return shapes (bimpc.py:12-295).  The convex program cvxpy hands to CLARABEL
(bimpc.py:114,287) is solved by the batched sm_100a interior-point kernel behind
``include/bimpc_b200.h`` (``csrc/bimpc_solve.cuh``): one station per CTA, block-tridiagonal
Cholesky over the horizon.  There is no CPU fallback.

Added (not in the reference): ``BiMPC.solve_bimpc_batch`` - S stations in one launch, optionally each with
its own ``BiMPCConstants``."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from enum import Enum

import numpy as np

from chargingstation import _native
from chargingstation.lompc import LoMPCConstants


class BiMPCChargingCostType(Enum):
    WEIGHTED = 0
    UNWEIGHTED = 1
    EXP_UNWEIGHTED = 2


@dataclass
class BiMPCConstants:
    """
    delta:              Relative weight of charging cost.
    c_g:                Electricity generation cost coefficient.
    u_g_max:            Maximum electricity generation per timestep.
    u_b_max:            Maximum charge/discharge rate of the storage battery.
    x_max:              Battery storage capacity.
    charging_cost_type: Enum of type BiMPCChargingCostType.
    exp_rate:           Rate of expoenential growth for EXP_UNWEIGHTED charging cost.
    """

    delta: float
    c_g: float
    u_g_max: float
    u_b_max: float
    x_max: float
    charging_cost_type: BiMPCChargingCostType
    exp_rate: float = 1  # Use np.Inf if only the cost at the final timestep is needed.


@dataclass
class BiMPCParameters:
    """
    Mp_s:       Number of small EVs in each partition.
    Mp_l:       Number of large EVs in each partition.
    beta_s:     Robustness bounds, for each partition of small EVs.
    beta_l:     Robustness bounds, for each partition of large EVs.
    gamma_sm:   Average fraction of battery capacity to be charged, for each partition of small EVs.
    gamma_lm:   Average fraction of battery capacity to be charged, for each partition of large EVs.
    x0:         Current charge of the storage battery.
    demand:     External electricity demand forecast for the control horizon.
    """

    Mp_s: np.ndarray
    Mp_l: np.ndarray
    beta_s: np.ndarray
    beta_l: np.ndarray
    gamma_sm: np.ndarray
    gamma_lm: np.ndarray
    x0: float
    demand: np.ndarray


# the scalar fields of BiMPCConstants that may differ from station to station (with the cost type and exp_rate)
SCALAR_FIELDS = ("delta", "c_g", "u_g_max", "u_b_max", "x_max")


def check_constants(consts_bi: BiMPCConstants, station: int | None = None) -> None:
    """The asserts of bimpc.py:79-84 (AssertionError) and the cost-type check of bimpc.py:231
    (NotImplementedError).  ``station``: the index the message names."""
    where = "" if station is None else f"station {station}: "
    for f in SCALAR_FIELDS:
        v = getattr(consts_bi, f)
        assert v >= 0, f"{where}BiMPCConstants.{f} must be >= 0, got {v}"
    assert consts_bi.exp_rate >= 1, f"{where}BiMPCConstants.exp_rate must be >= 1, got {consts_bi.exp_rate}"
    if not isinstance(consts_bi.charging_cost_type, BiMPCChargingCostType):
        raise NotImplementedError(f"{where}unknown charging cost type {consts_bi.charging_cost_type!r}")  # bimpc.py:231


def station_constants(consts, S: int) -> dict:
    """Checks one ``BiMPCConstants`` per station (``check_constants``, naming the station) and returns them as arrays:
    delta, c_g, u_g_max, u_b_max, x_max, exp_rate (float64 [S]), cost_type (int32 [S]) and the list itself
    ("consts")."""
    assert not isinstance(consts, BiMPCConstants), f"expected one BiMPCConstants per station ({S}), got one in all"
    consts = list(consts)
    assert len(consts) == S, f"expected one BiMPCConstants per station ({S}), got {len(consts)}"
    for s, c in enumerate(consts):
        check_constants(c, s)
    out = {f: np.array([float(getattr(c, f)) for c in consts], dtype=np.float64) for f in SCALAR_FIELDS + ("exp_rate",)}
    out["cost_type"] = np.array([c.charging_cost_type.value for c in consts], dtype=np.int32)
    out["consts"] = consts
    return out


def stage_weights(lib, N: int, cost_type: int, exp_rate: float) -> np.ndarray:
    """The [N] stage weights of the charging cost (bimpc.py:255-257) as the library builds them for a handle
    (``bimpc_stage_weights``): a per-station row has the bits of the handle's."""
    om = np.empty(N)
    _native.raise_for(lib.bimpc_stage_weights(int(N), int(cost_type), float(exp_rate), om.ctypes.data_as(C.c_void_p)))
    return om


class BiMPC:
    def __init__(self, N: int, P: int, consts_bi: BiMPCConstants, consts_s: LoMPCConstants,
                 consts_l: LoMPCConstants, device: int = 0) -> None:
        """
        Inputs:
            N:                  Horizon length.
            P:                  Number of partitions per EV type.
            consts_bi:          BiMPC constants.
            consts_s:           LoMPC constants for small EVs.
            consts_l:           LoMPC constants for large EVs.
        """
        check_constants(consts_bi)  # bimpc.py:79-84, 231
        self.N, self.P = N, P
        self.delta = consts_bi.delta
        self.c_g = consts_bi.c_g
        self.u_g_max = consts_bi.u_g_max
        self.u_b_max = consts_bi.u_b_max
        self.x_max = consts_bi.x_max
        self.exp_rate = consts_bi.exp_rate * 1.0
        self.charging_cost_type = consts_bi.charging_cost_type
        self.theta_s, self.theta_l = consts_s.theta, consts_l.theta
        self.w_max_s, self.w_max_l = consts_s.w_max, consts_l.w_max
        # BiMPC input matrix, x = A u_b + x0 1.
        self.A = np.tril(np.ones((N, N)))
        self.device = int(device)
        self._lib = _native.load()
        h = C.c_void_p()
        rc = self._lib.bimpc_create(N, P, float(self.delta), float(self.c_g), float(self.u_g_max),
                                    float(self.u_b_max), float(self.x_max), self.charging_cost_type.value,
                                    float(self.exp_rate), float(self.theta_s), float(self.theta_l),
                                    float(self.w_max_s), float(self.w_max_l), self.device, C.byref(h))
        _native.raise_for(rc)
        self._h = h
        self.last_info = {}

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                self._lib.bimpc_destroy(h)
            except Exception:
                pass

    def get_bat_input_mat(self) -> np.ndarray:
        return self.A

    def set_options(self, max_iter: int = 100, tol: float = 1e-9) -> None:
        _native.raise_for(self._lib.bimpc_set_options(self._h, int(max_iter), float(tol)))

    def solve_bimpc(self, params: BiMPCParameters) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """
        Inputs:
            params: BiMPC problem parameters.
        Outputs:
            w_hat_s_opt:    Team-optimal electricity output for small EVs.
            w_hat_l_opt:    Team-optimal electricity output for large EVs.
            u_g_opt:        Team-optimal electricity generation.
        """
        P, N = self.P, self.N
        # bimpc.py:278-283
        assert (params.Mp_s.shape == (P,)) and (params.Mp_l.shape == (P,))
        assert (params.beta_s.shape == (P,)) and (params.beta_l.shape == (P,))
        assert (params.gamma_sm.shape == (P,)) and (params.gamma_lm.shape == (P,))
        assert params.demand.shape == (N,)
        ws, wl, ug, info = self.solve_bimpc_batch(params.Mp_s[None], params.Mp_l[None], params.beta_s[None],
                                                  params.beta_l[None], params.gamma_sm[None],
                                                  params.gamma_lm[None], np.array([float(params.x0)]),
                                                  params.demand[None])
        self.last_info = {k: v[0] for k, v in info.items()}
        if self.last_info["status"] != 0:
            # the reference hands back the .value of unsolved cvxpy variables, i.e. None (bimpc.py:288-291), and its
            # caller fails on the first slice; the last iterate stays available through solve_bimpc_batch
            return None, None, None
        return ws[0], wl[0], ug[0]

    def solve_bimpc_batch(self, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, consts=None):
        """``solve_bimpc`` for S stations: every argument has a leading station axis
        ([S,P] / [S] / [S,N]).  Returns (w_hat_s [S,P,N], w_hat_l [S,P,N], u_g [S,N], info)
        with info = {status, iters, objective} arrays of length S.

        consts: None, or one ``BiMPCConstants`` per station (same units as the constructor's).  Station s
        then solves with its own delta, c_g, limits, cost type and exp_rate, with the bits a BiMPC created
        with ``consts[s]`` gives it; N, P and the EV constants stay this object's.  Each is checked like
        the constructor's constants before any device work."""
        P, N = self.P, self.N
        ins = [np.ascontiguousarray(v, dtype=np.float64) for v in (Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm)]
        S = ins[0].shape[0]
        sc = None if consts is None else station_constants(consts, S)
        for v in ins:
            assert v.shape == (S, P)
            if np.any(v < 0):  # nonneg cv.Parameters, bimpc.py:122-140
                raise ValueError("negative value for a nonneg BiMPC parameter")
        x0 = np.ascontiguousarray(x0, dtype=np.float64).reshape(S)
        demand = np.ascontiguousarray(demand, dtype=np.float64)
        assert demand.shape == (S, N)
        if np.any(demand < 0):
            raise ValueError("negative demand (nonneg cv.Parameter, bimpc.py:131)")
        ws = np.empty((S, P, N))
        wl = np.empty((S, P, N))
        ug = np.empty((S, N))
        st = np.empty(S, dtype=np.int32)
        it = np.empty(S, dtype=np.int32)
        obj = np.empty(S)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        if sc is None:
            rc = self._lib.bimpc_solve_batch_host(self._h, S, *[p(v) for v in ins], p(x0), p(demand), p(ws), p(wl),
                                                  p(ug), p(st), p(it), p(obj))
        else:
            rc = self._lib.bimpc_solve_batch_consts_host(
                self._h, S, *[p(sc[f]) for f in SCALAR_FIELDS + ("cost_type", "exp_rate")], *[p(v) for v in ins], p(x0),
                p(demand), p(ws), p(wl), p(ug), p(st), p(it), p(obj))
        if rc != _native.ERR_NOT_CONVERGED:
            _native.raise_for(rc)
        # a failed solve yields None in the reference (.value of an unsolved variable, bimpc.py:288-291); the batch
        # call reports it per station in info["status"], warns, and returns the last iterate of those stations
        if rc == _native.ERR_NOT_CONVERGED or np.any(st != 0):
            import warnings
            warnings.warn(f"BiMPC: {int(np.count_nonzero(st))} of {S} station(s) not solved to tolerance "
                          "(infeasible or iteration cap) - see info['status']", RuntimeWarning, stacklevel=2)
        return ws, wl, ug, {"status": st, "iters": it, "objective": obj}
