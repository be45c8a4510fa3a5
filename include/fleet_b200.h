/*
 * fleet_b200.h -- C ABI of the device-resident closed loop over S charging stations
 * (SURVEY.md section 8 f2; BASELINE.json configs[3]).  These entry points are the
 * plumbing kernels between the optimisation kernels of lompc_b200.h / bimpc_b200.h;
 * each replaces a NumPy fragment of reference chargingstation/charging_station.py, batched
 * over stations.  All pointers are DEVICE pointers, calls are asynchronous on `stream`.
 *
 * Layout.  Per EV type a station holds M EVs: SoC y[S,M], partition index idx[S,M].  The
 * price loop wants EVs sorted by group; groups are numbered PARTITION-MAJOR, g = p*S + s,
 * so that "partition p of every station" is one contiguous slice of groups and of EVs
 * (the reference solves the partitions of an EV type one after the other with a shared
 * warm start, charging_station.py:273-304).
 *
 * Stations of different sizes.  The *_sized_dev entry points take nevs[S] (device, 1 <=
 * nevs[s] <= M; values outside [0, M] are clamped to it) and/or Bcap[S] (device, > 0):
 * station s owns the first nevs[s] slots of its row of M, and the padding slots of y, idx
 * and replace_mask are neither read nor written.  The EV-sorted arrays (y_sorted, perm and
 * what the price loops build on them) hold real EVs only, so off[P*S] = sum(nevs).  The
 * uniform entry points are the same kernels with nevs[s] = M and Bcap[s] = Bcap for every
 * station.
 */
#ifndef FLEET_B200_H
#define FLEET_B200_H

#include <stdint.h>

#include "lompc_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ChargingStation._update_indices (charging_station.py:111-116) for S stations, then the
 * sort of the EVs by group: idx[S,M] is updated in place (an SoC outside every partition
 * keeps its index), counts[P*S] (partition-major), off[P*S+1] = exclusive scan,
 * off_rebased[P,(S+1)] = per-partition offsets starting at 0, y_sorted[S*M] and
 * perm[S*M] (sorted position -> EV index inside its station; order inside a group = EV
 * order, as y[idx == p] in the reference).  edges[P+1] = partition boundaries.           */
int fleet_partition_dev(int device, int32_t S, int32_t M, int32_t P, const double* edges, const double* y,
                        int32_t* idx, int32_t* counts, int32_t* off, int32_t* off_rebased,
                        double* y_sorted, int32_t* perm, void* stream);
/* The same for stations of nevs[s] EVs: only slots j < nevs[s] of a row are assigned and
 * sorted; counts, off, off_rebased, y_sorted and perm[sum(nevs)] cover real EVs only.      */
int fleet_partition_sized_dev(int device, int32_t S, int32_t M, int32_t P, const int32_t* nevs, const double* edges,
                              const double* y, int32_t* idx, int32_t* counts, int32_t* off, int32_t* off_rebased,
                              double* y_sorted, int32_t* perm, void* stream);

/* BiMPCParameters of every station (charging_station.py:187-220): Mp = counts / Bcap,
 * beta = the w0 bound of PriceSolver.get_robustness_bounds (price_solver.py:182-186) from
 * y0_rng, gamma_m = gamma_sm (0 for an empty partition), x0 = x, demand = profile[s, t : t +
 * N_bi] / Bcap.  Group arrays are partition-major [P*S]; outputs are station-major [S,P].  */
int fleet_bimpc_params_dev(int device, int32_t S, int32_t P, int32_t N_bi, int32_t N_lo, double Bcap,
                           double eps_tol, double lmbd_r, double delta_s, double delta_l,
                           const int32_t* counts_s, const int32_t* counts_l, const double* y0_rng_s,
                           const double* y0_rng_l, const double* gamma_sm_s, const double* gamma_sm_l,
                           const double* x, const double* demand_profile, int32_t profile_len, int32_t t,
                           double* Mp_s, double* Mp_l, double* beta_s, double* beta_l, double* gamma_s,
                           double* gamma_l, double* x0, double* demand, void* stream);
/* The same with each station's own capacity: Mp = counts / Bcap[s], demand = profile / Bcap[s]. */
int fleet_bimpc_params_sized_dev(int device, int32_t S, int32_t P, int32_t N_bi, int32_t N_lo, const double* Bcap,
                                 double eps_tol, double lmbd_r, double delta_s, double delta_l,
                                 const int32_t* counts_s, const int32_t* counts_l, const double* y0_rng_s,
                                 const double* y0_rng_l, const double* gamma_sm_s, const double* gamma_sm_l,
                                 const double* x, const double* demand_profile, int32_t profile_len, int32_t t,
                                 double* Mp_s, double* Mp_l, double* beta_s, double* beta_l, double* gamma_s,
                                 double* gamma_l, double* x0, double* demand, void* stream);

/* w_ref of every group = the first N_lo steps of the BiMPC plan (charging_station.py:269):
 * w_ref[(p*S+s), k] = w_hat[s, p, k].                                                      */
int fleet_wref_dev(int device, int32_t S, int32_t P, int32_t N_bi, int32_t N_lo, const double* w_hat,
                   double* w_ref, void* stream);

/* Keeps the price rows of one partition slice: dst[s,:] = src[s,:] if the group (p, s) is
 * non-empty, else 0 (prices_s = np.zeros(...), charging_station.py:270), and
 * price_red[s] = post - pre or NaN for an empty group (charging_station.py:422-433).       */
int fleet_keep_prices_dev(int device, int32_t S, int32_t row, const int32_t* counts_p, const double* src,
                          double* dst, const double* price_pre, const double* price_post,
                          double* price_red, void* stream);

/* ChargingStation._update_state (charging_station.py:329-365) for one EV type of every
 * station: y[s, perm] += w0_sorted; EVs above MIN_FULL_CHARGE_FRACTION * y_max are replaced
 * by a new EV with SoC uniform in [y0_min, y0_max) when rng_seed >= 0 (counter-based
 * generator keyed by (seed, type, station, EV, t)); with rng_seed < 0 the replacement is
 * left to the host (parity runs on np.random) and only `replace_mask[S,M]` is written.
 * Also: w_sum[S] = sum of w0 of the station, w_mean[P*S] = mean first-step charge per group
 * (logs["inputs"]["w_s"], charging_station.py:381-385), ncharged[S] += replaced EVs.        */
int fleet_apply_charge_dev(int device, int32_t S, int32_t M, int32_t P, double full_level, double y0_min,
                           double y0_max, int64_t rng_seed, int32_t ev_type, int32_t t, const int32_t* off,
                           const int32_t* perm, const double* w0_sorted, double* y, int32_t* replace_mask,
                           double* w_sum, double* w_mean, int32_t* ncharged, void* stream);
/* The same for stations of nevs[s] EVs: departures, arrivals and replace_mask cover slots
 * j < nevs[s] only (the generator key keeps the EV's slot in its station).                 */
int fleet_apply_charge_sized_dev(int device, int32_t S, int32_t M, int32_t P, const int32_t* nevs, double full_level,
                                 double y0_min, double y0_max, int64_t rng_seed, int32_t ev_type, int32_t t,
                                 const int32_t* off, const int32_t* perm, const double* w0_sorted, double* y,
                                 int32_t* replace_mask, double* w_sum, double* w_mean, int32_t* ncharged,
                                 void* stream);

/* Battery update (charging_station.py:353-365, ADD_RESIDUAL_CHARGE_TO_BATTERY = False):
 * x[s] += u_g[s,0] + (-theta_s w_sum_s[s] - theta_l w_sum_l[s] - profile[s,t]) / Bcap.      */
int fleet_battery_dev(int device, int32_t S, int32_t N_bi, double theta_s, double theta_l, double Bcap,
                      const double* u_g, const double* w_sum_s, const double* w_sum_l,
                      const double* demand_profile, int32_t profile_len, int32_t t, double* x,
                      void* stream);
/* The same with each station's own capacity: ... / Bcap[s].                               */
int fleet_battery_sized_dev(int device, int32_t S, int32_t N_bi, double theta_s, double theta_l, const double* Bcap,
                            const double* u_g, const double* w_sum_s, const double* w_sum_l,
                            const double* demand_profile, int32_t profile_len, int32_t t, double* x, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FLEET_B200_H */
