/*
 * bimpc_b200.h -- C ABI of the batched upper-level BiMPC (one convex program per
 * charging station and time step), the caller of the lower-level price loop
 * (SURVEY.md section 8 a12 / f1).  Replaces reference chargingstation/bimpc.py:
 * BiMPC.__init__ (bimpc.py:62-114) and BiMPC.solve_bimpc (bimpc.py:267-292), batched
 * over S independent stations.  Same conventions and error codes as lompc_b200.h.
 */
#ifndef BIMPC_B200_H
#define BIMPC_B200_H

#include <stdint.h>

#include "lompc_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* BiMPCChargingCostType (bimpc.py:12-15) */
#define BIMPC_COST_WEIGHTED 0
#define BIMPC_COST_UNWEIGHTED 1
#define BIMPC_COST_EXP_UNWEIGHTED 2

/* per-station status written by the kernel */
#define BIMPC_ST_OK 0
#define BIMPC_ST_MAXITER 1    /* also: infeasible program (cvxpy would return None, bimpc.py:288-291) */
#define BIMPC_ST_BREAKDOWN 2  /* Newton matrix lost positive definiteness */

typedef struct bimpc_handle bimpc_t;

/* Replaces BiMPC.__init__ / _set_constants (bimpc.py:62-141): N = horizon, P = partitions
 * per EV type.  LOMPC_ERR_CONSTS when one of the asserts of bimpc.py:79-84 fails or the
 * cost type is unknown (NotImplementedError, bimpc.py:231); LOMPC_ERR_ARG when the
 * problem does not fit one CTA's shared memory (N <= 48).                              */
int bimpc_create(int N, int P, double delta, double c_g, double u_g_max, double u_b_max,
                 double x_max, int cost_type, double exp_rate, double theta_s, double theta_l,
                 double w_max_s, double w_max_l, int device, bimpc_t** out);
int bimpc_destroy(bimpc_t* h);

/* Interior-point knobs (defaults: max_iter 100, tol 1e-9 on the dual residual relative to
 * the gradient scale, on the primal residual and on the mean complementarity).          */
int bimpc_set_options(bimpc_t* h, int max_iter, double tol);

/* Replaces BiMPC.solve_bimpc (bimpc.py:267-292) for S stations.  Inputs are the fields of
 * BiMPCParameters (bimpc.py:44-58), one row per station: Mp_s, Mp_l, beta_s, beta_l,
 * gamma_sm, gamma_lm [S,P]; x0 [S]; demand [S,N].  Outputs: w_hat_s, w_hat_l [S,P,N],
 * u_g [S,N], status, iters [S]; objective [S] may be NULL.  DEVICE pointers, asynchronous
 * on `stream`.                                                                          */
int bimpc_solve_batch_dev(bimpc_t* h, int32_t S, const double* Mp_s, const double* Mp_l,
                          const double* beta_s, const double* beta_l, const double* gamma_sm,
                          const double* gamma_lm, const double* x0, const double* demand,
                          double* w_hat_s, double* w_hat_l, double* u_g, int32_t* status,
                          int32_t* iters, double* objective, void* stream);

/* Same call with HOST pointers: copies in, solves, copies out, synchronises.  Returns
 * LOMPC_ERR_NOT_CONVERGED if any station ended with a status other than BIMPC_ST_OK
 * (outputs are still written).                                                          */
int bimpc_solve_batch_host(bimpc_t* h, int32_t S, const double* Mp_s, const double* Mp_l,
                           const double* beta_s, const double* beta_l, const double* gamma_sm,
                           const double* gamma_lm, const double* x0, const double* demand,
                           double* w_hat_s, double* w_hat_l, double* u_g, int32_t* status,
                           int32_t* iters, double* objective);

/* Stage weights of the charging cost for horizon N (bimpc.py:255-257): omega[k] =
 * exp_rate^(k-N+1) for BIMPC_COST_EXP_UNWEIGHTED, 1 otherwise; omega holds N doubles (host).
 * bimpc_create builds the handle's weights with this function, so a row built here for the
 * same cost type and exp_rate has the handle's bits.  LOMPC_ERR_CONSTS for an unknown cost
 * type or exp_rate < 1 (or NaN); LOMPC_ERR_ARG for N < 1 or a NULL omega.               */
int bimpc_stage_weights(int N, int cost_type, double exp_rate, double* omega);

/* bimpc_solve_batch_dev with one set of BiMPC constants per station: delta, c_g, u_g_max,
 * u_b_max, x_max [S], cost_type [S] and the stage weights omega [S,N] (a row of
 * bimpc_stage_weights for the station's cost type and exp_rate).  Same units as the
 * handle's constants (normalised by each station's own capacity).  These calls IGNORE the
 * handle's delta, c_g, u_g_max, u_b_max, x_max, cost type and exp_rate; they use its N, P,
 * theta_s, theta_l, w_max_s, w_max_l and options.  Station s solves exactly as a handle
 * created with its constants would solve it alone (same bits).  A station whose constants
 * are negative or not finite, whose cost type is not 0..2 or whose omega row is not finite
 * gets status BIMPC_ST_BREAKDOWN; the other stations are unaffected.  A NULL pointer among
 * the constants returns LOMPC_ERR_ARG and launches nothing.  DEVICE pointers, asynchronous
 * on `stream`.                                                                          */
int bimpc_solve_batch_consts_dev(bimpc_t* h, int32_t S, const double* delta, const double* c_g,
                                 const double* u_g_max, const double* u_b_max, const double* x_max,
                                 const int32_t* cost_type, const double* omega, const double* Mp_s,
                                 const double* Mp_l, const double* beta_s, const double* beta_l,
                                 const double* gamma_sm, const double* gamma_lm, const double* x0,
                                 const double* demand, double* w_hat_s, double* w_hat_l, double* u_g,
                                 int32_t* status, int32_t* iters, double* objective, void* stream);

/* The same call with HOST pointers, like bimpc_solve_batch_host.  Takes exp_rate [S] in place
 * of omega and builds each station's weights with bimpc_stage_weights; a station whose cost
 * type or exp_rate that function refuses gets status BIMPC_ST_BREAKDOWN.                */
int bimpc_solve_batch_consts_host(bimpc_t* h, int32_t S, const double* delta, const double* c_g,
                                  const double* u_g_max, const double* u_b_max, const double* x_max,
                                  const int32_t* cost_type, const double* exp_rate, const double* Mp_s,
                                  const double* Mp_l, const double* beta_s, const double* beta_l,
                                  const double* gamma_sm, const double* gamma_lm, const double* x0,
                                  const double* demand, double* w_hat_s, double* w_hat_l, double* u_g,
                                  int32_t* status, int32_t* iters, double* objective);

#ifdef __cplusplus
}
#endif
#endif /* BIMPC_B200_H */
