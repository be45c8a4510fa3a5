"""Seeded BiMPC instances shared by the CPU (oracle / host-simulated kernel) and GPU tests."""
import numpy as np

from oracle import bimpc_oracle as bo

# MediumTermLoadForecast of the reference's bundled CSV (data rows 31-54), see demand_data.py
FORECAST_24 = np.array([73822, 70492, 69346, 67924, 67239, 67297, 67663, 69463, 72885, 77079, 80526, 84550,
                        87982, 90588, 92603, 94458, 95772, 95887, 94438, 92268, 89947, 85908, 80634, 76068], float)


def draw_station(rng, c: bo.BiConsts, empty: bool = True, active_s=None, active_l=None, track_empty: bool = False):
    """One station's BiMPCParameters tuple in the ranges charging_station.py:187-220 produces.

    active_s / active_l: indices of the partitions that hold EVs (at least one each); every other partition of that
    type is empty.  None keeps the drawn sizes (with the last small and the first large partition emptied if
    `empty`).  track_empty: empty partitions keep a charging target gamma > 0 instead of 0."""
    N, P = c.N, c.P
    M2 = 500
    Bcap = (c.theta_s + c.theta_l) * M2
    Mp_s = rng.multinomial(M2, np.ones(P) / P) / Bcap
    Mp_l = rng.multinomial(M2, np.ones(P) / P) / Bcap
    if empty and P > 3:
        Mp_s[-1] = 0.0
        Mp_l[0] = 0.0
    for Mp, act in ((Mp_s, active_s), (Mp_l, active_l)):
        if act is not None:
            keep = np.zeros(P, dtype=bool)
            keep[list(act)] = True
            Mp[:] = np.where(keep, Mp + 1.0 / Bcap, 0.0)
    dem = np.resize(np.roll(FORECAST_24, int(rng.integers(24))), N) * 0.25 / Bcap
    edges = np.linspace(0.3, 0.9, P + 1)
    g = 0.9 - edges[:-1] - (edges[1] - edges[0]) * rng.random(P)
    beta_s = (np.sqrt(12) * 0.5 * (edges[1] - edges[0]) * rng.random(P) + 0.01) * 0.1
    beta_l = (np.sqrt(12) * 0.5 * (edges[1] - edges[0]) * rng.random(P) + 0.01) * 0.1
    gs, gl = (g, g.copy()) if track_empty else (g * (Mp_s > 0), g * (Mp_l > 0))
    return (Mp_s, Mp_l, beta_s, beta_l, gs, gl, 0.1 * rng.random(), dem)


def stack(stations):
    return [np.stack([np.asarray(s[i], dtype=float) for s in stations]) for i in range(8)]
