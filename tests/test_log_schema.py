"""SURVEY.md 8 row f4: the `logs` dict of the closed loop (charging_station.py:118-149) and the `solver_stats` of
PriceSolver.compute_optimal_prices (price_solver.py:167-173) keep the reference's schema, so that its plot scripts
(example/real_time_price_control_plots.py:24-305, plots/plots.py:115-127) can read a pickle written here.  The
schema is a committed fixture parsed from the reference's sources (tests/golden/gen_log_schema.py)."""
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SCHEMA = json.load(open(os.path.join(GOLD, "log_schema.json")))


def test_consumers_only_read_keys_the_schema_produces():
    for key in SCHEMA["consumed"]:
        parts = key.split(".")
        if parts[0] == "solver_stats":
            assert parts[1] in SCHEMA["solver_stats"], key
        elif len(parts) == 1:
            assert parts[0] in SCHEMA["logs"], key
        else:
            assert parts[1] in SCHEMA["logs"][parts[0]], key


def _check_logs(logs, P, Tf):
    assert set(logs) == set(SCHEMA["logs"])
    for top, sub in SCHEMA["logs"].items():
        if sub is None:
            continue
        assert set(logs[top]) == set(sub), top
        for name, spec in sub.items():
            val = logs[top][name]
            dims = tuple({"P": P, "Tf": Tf}[d] for d in spec["dims"])
            if dims:
                assert isinstance(val, np.ndarray) and val.shape == dims, (top, name, getattr(val, "shape", None))
                assert (val.dtype.kind in "iu") == spec["int"], (top, name, val.dtype)
            else:
                assert np.ndim(val) == 0 and float(val) == int(val), (top, name)


@pytest.mark.gpu
def test_station_and_fleet_logs_and_solver_stats_follow_the_schema(tmp_path):
    import pickle
    from chargingstation import settings
    from chargingstation.charging_station import ChargingStation
    from chargingstation.example.real_time_price_control import get_chargingstation_consts
    from chargingstation.fleet import ChargingStationFleet
    from chargingstation.price_solver import PriceSolver
    settings.PRINT_LEVEL = 0
    consts = get_chargingstation_consts(3)
    np.random.seed(0)
    cs = ChargingStation(consts)
    logs = cs.simulate()
    _check_logs(logs, consts.npartitions, 3)
    # the example pickles the dict (real_time_price_control.py:88-93): it must survive the round trip
    path = tmp_path / "logs.pkl"
    with open(path, "wb") as f:
        pickle.dump(logs, f)
    with open(path, "rb") as f:
        _check_logs(pickle.load(f), consts.npartitions, 3)
    # what _plot_graphs computes first from it (real_time_price_control_plots.py:37-60) works
    Mp_s, w_s = logs["statistics"]["Mp_s"], logs["inputs"]["w_s"]
    assert np.sum(Mp_s * w_s, axis=0).shape == (3,)
    niter = logs["statistics"]["niter_s"]
    assert niter[niter >= 1].ndim == 1
    fleet = ChargingStationFleet(consts, 2, seed=0, rng="numpy")
    fleet.simulate()
    _check_logs(fleet.station_logs(1), consts.npartitions, 3)
    # solver_stats (price_solver.py:167-173), read by plots/plots.py:125-127
    ps = PriceSolver(12, consts.small_EV_consts, "linear-convex")
    ps.set_charge_levels(np.array([0.3, 0.32, 0.35]))
    _, st = ps.compute_optimal_prices(0.1 * np.ones(12), 0.0)
    assert set(st) == set(SCHEMA["solver_stats"])
    assert len(st["dual_cost_decrease_actual"]) == st["iter"] == len(st["dual_cost_decrease_predicted"])
