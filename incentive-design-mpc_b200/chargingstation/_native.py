"""ctypes binding of ``liblompc_b200.so`` (C ABI: ``include/lompc_b200.h``,
``include/bimpc_b200.h``, ``include/fleet_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` (or ``make -C
incentive-design-mpc_b200/csrc``).  Loading fails loudly if it is missing:
this package has no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LOMPC_B200_LIB: another build of the same library (tuning sweeps build variants next to the default one)
LIB_PATH = os.environ.get("LOMPC_B200_LIB") or os.path.join(os.path.dirname(_HERE), "csrc", "liblompc_b200.so")

OK = 0
ERR_CONSTS, ERR_ARG, ERR_CUDA, ERR_GAMMA, ERR_NEGATIVE, ERR_NOT_CONVERGED, ERR_NO_DEVICE = (
    -1, -2, -3, -4, -5, -6, -7)
EV_SMALL, EV_LARGE = 0, 1
ST_OK, ST_MAXITER, ST_BAD_GAMMA, ST_NEGATIVE = 0, 1, 2, 3

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)

# name -> (restype, argtypes); every symbol include/lompc_b200.h declares.
SIGNATURES = {
    "lompc_version": (C.c_char_p, []),
    "lompc_strerror": (C.c_char_p, [C.c_int]),
    "lompc_last_cuda_error": (C.c_char_p, []),
    "lompc_device_count": (C.c_int, []),
    "lompc_create": (C.c_int, [C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int,
                               C.c_int, C.POINTER(C.c_void_p)]),
    "lompc_destroy": (C.c_int, [C.c_void_p]),
    "lompc_sc_modulus": (C.c_double, [C.c_void_p]),
    "lompc_set_options": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "lompc_set_kernel_variant": (C.c_int, [C.c_void_p, C.c_int]),
    "lompc_solve_batch_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                        C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "lompc_solve_batch_host": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                         C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "lompc_solve_batch_host_async": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                               C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p]),
    "lompc_host_wait": (C.c_int, [C.c_void_p]),
    "lompc_vjp_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64] +
                      [C.c_void_p] * 9),
    "lompc_group_solve_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64] + [C.c_void_p] * 8),
    "lompc_group_vjp_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64] + [C.c_void_p] * 12),
    "lompc_launch_count": (C.c_int64, []),
    "lompc_set_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_void_p)]),
    "lompc_set_destroy": (C.c_int, [C.c_void_p]),
    "lompc_set_buffers": (C.c_int, [C.c_void_p, C.c_int, C.c_int] + [C.POINTER(C.c_void_p)] * 5),
    "lompc_set_info_buffers": (C.c_int, [C.c_void_p, C.c_int] + [C.POINTER(C.c_void_p)] * 3),
    "lompc_set_solve_host_async": (C.c_int, [C.c_void_p, C.c_int]),
    "lompc_set_wait": (C.c_int, [C.c_void_p]),
    "lompc_set_solve_host": (C.c_int, [C.c_void_p, C.c_int]),
    "lompc_set_solve_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "lompc_set_solve_dev_at": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lompc_set_offsets": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int64)]),
    "lompc_set_copy": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "lompc_set_bytes": (C.c_int64, [C.c_void_p, C.c_int]),
    "price_group_stats_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64] + [C.c_void_p] * 7),
    "price_w_err_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64] + [C.c_void_p] * 11),
    "price_step_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int] + [C.c_void_p] * 7),
    "price_regularize_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int] + [C.c_void_p] * 5),
    "price_lp_rows_dev": (C.c_int, [C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 5),
    "price_solve_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.c_void_p]),
    "price_solve_chain_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double] +
                              [C.c_void_p] * 6 + [C.POINTER(C.c_int32), C.c_void_p]),
    "price_set_loop_mode": (C.c_int, [C.c_void_p, C.c_int]),
    "price_last_qp_solves": (C.c_int64, [C.c_void_p]),
    "price_last_cycles": (C.c_int64, [C.c_void_p, C.c_int]),
    "price_debug_force_nnqp_fallback": (C.c_int, [C.c_int]),
    "price_debug_pivot_pool": (C.c_int, [C.c_int]),
    "price_debug_record_errors": (C.c_int, [C.c_void_p, C.c_void_p]),
    "price_debug_force_compact_step": (C.c_int, [C.c_int]),
    "price_shard_begin": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_int, C.c_int, C.c_double, C.c_double] + [C.c_void_p] * 10 +
                          [C.c_int, C.c_void_p]),
    "price_shard_start": (C.c_int, [C.c_void_p, C.c_void_p]),
    "price_shard_ev_phase": (C.c_int, [C.c_void_p, C.c_void_p]),
    "price_shard_group_phase": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.c_void_p]),
    "price_shard_group_phase_async": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "price_shard_poll": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int32)]),
    "lompc_ipc_alloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(C.c_void_p), C.c_void_p]),
    "lompc_ipc_open": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "lompc_ipc_close": (C.c_int, [C.c_int, C.c_void_p]),
    "lompc_ipc_free": (C.c_int, [C.c_int, C.c_void_p]),
    "price_shard_attach_peers": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_size_t]),
    "price_shard_uses_peers": (C.c_int, [C.c_void_p]),
    "price_shard_local_sums": (C.c_int, [C.c_void_p, C.c_int]),
    "price_shard_finish": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "price_w0_price0_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64] + [C.c_void_p] * 7),
    "lompc_measure_fp64_peak": (C.c_int, [C.c_int, C.c_int, _dp, _dp]),
    # include/bimpc_b200.h
    "bimpc_create": (C.c_int, [C.c_int, C.c_int] + [C.c_double] * 5 + [C.c_int] + [C.c_double] * 5 +
                     [C.c_int, C.POINTER(C.c_void_p)]),
    "bimpc_destroy": (C.c_int, [C.c_void_p]),
    "bimpc_set_options": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "bimpc_solve_batch_dev": (C.c_int, [C.c_void_p, C.c_int32] + [C.c_void_p] * 15),
    "bimpc_solve_batch_host": (C.c_int, [C.c_void_p, C.c_int32] + [C.c_void_p] * 14),
    "bimpc_stage_weights": (C.c_int, [C.c_int, C.c_int, C.c_double, C.c_void_p]),
    "bimpc_solve_batch_consts_dev": (C.c_int, [C.c_void_p, C.c_int32] + [C.c_void_p] * 22),
    "bimpc_solve_batch_consts_host": (C.c_int, [C.c_void_p, C.c_int32] + [C.c_void_p] * 21),
    # include/fleet_b200.h
    "fleet_partition_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 9),
    "fleet_partition_sized_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 10),
    "fleet_bimpc_params_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_int32] + [C.c_double] * 5 +
                               [C.c_void_p] * 8 + [C.c_int32, C.c_int32] + [C.c_void_p] * 9),
    "fleet_bimpc_params_sized_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p] +
                                     [C.c_double] * 4 + [C.c_void_p] * 8 + [C.c_int32, C.c_int32] + [C.c_void_p] * 9),
    "fleet_wref_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 3),
    "fleet_keep_prices_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32] + [C.c_void_p] * 7),
    "fleet_apply_charge_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double,
                                         C.c_double, C.c_int64, C.c_int32, C.c_int32] + [C.c_void_p] * 9),
    "fleet_apply_charge_sized_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_double,
                                               C.c_double, C.c_double, C.c_int64, C.c_int32, C.c_int32] +
                                     [C.c_void_p] * 9),
    "fleet_battery_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double] +
                          [C.c_void_p] * 4 + [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "fleet_battery_sized_dev": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_void_p] +
                                [C.c_void_p] * 4 + [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Loads the shared library once and types every entry point."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` or `make -C incentive-design-mpc_b200/csrc` (no CPU fallback exists)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def strerror(code: int) -> str:
    lib = load()
    msg = lib.lompc_strerror(code).decode()
    if code == ERR_CUDA:
        msg += ": " + lib.lompc_last_cuda_error().decode()
    return msg


def raise_for(code: int) -> None:
    """Maps C error codes onto the reference's exception types (SURVEY.md 8b)."""
    if code == OK:
        return
    msg = strerror(code)
    if code in (ERR_CONSTS, ERR_GAMMA):
        raise AssertionError(msg)  # Python asserts in lompc.py:36-38,87
    if code == ERR_NEGATIVE:
        raise ValueError(msg)  # cvxpy nonneg Parameter, lompc.py:78-82
    if code == ERR_ARG:
        raise ValueError(msg)
    raise RuntimeError(msg)
