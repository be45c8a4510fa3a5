// Host compilation of the per-station mode of the BiMPC kernel body (csrc/bimpc_solve.cuh with BIMPC_HOSTSIM,
// solve_station<true>): one "thread" per station, barriers are no-ops.  TEST INFRASTRUCTURE ONLY - lets the CPU test
// suite check the per-station algorithm against the dense oracle and against the uniform mode without a GPU; the
// product library never contains this code path.
#define BIMPC_HOSTSIM 1
#include <stdlib.h>
#include <cmath>
#include "bimpc_solve.cuh"

// The same kernel body in its per-station mode (bimpc_solve_kernel<true>): station s solves with delta[s], ...,
// cost_type[s] and its row of omega [S,N].  The handle-wide constants the per-station mode must not read are NaN.
extern "C" int bimpc_hostsim_solve_consts(int N, int P, double theta_s, double theta_l, double w_max_s,
                                          double w_max_l, int S, const double* delta, const double* c_g,
                                          const double* u_g_max, const double* u_b_max, const double* x_max,
                                          const int32_t* cost_type, const double* omega, const double* Mp_s,
                                          const double* Mp_l, const double* beta_s, const double* beta_l,
                                          const double* gamma_sm, const double* gamma_lm, const double* x0,
                                          const double* demand, double* w_hat_s, double* w_hat_l, double* u_g,
                                          int32_t* status, int32_t* iters, double* objective, double tol,
                                          int max_iter) {
  if (N > bimpc::kMaxN) return -2;
  const double nan = __builtin_nan("");
  bimpc::BiConsts c{N, P, nan, nan, nan, nan, nan, -1, theta_s, theta_l, w_max_s, w_max_l};
  bimpc::BiArgs a{S, nullptr, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand,
                  w_hat_s, w_hat_l, u_g, status, iters, objective, tol, max_iter, nullptr, nullptr,
                  delta, c_g, u_g_max, u_b_max, x_max, cost_type, omega};
  const size_t n = bimpc::scratch_doubles(N, P, 1);
  double* sm = (double*)malloc(n * sizeof(double));
  double* li = (double*)malloc(bimpc::global_scratch_doubles(N, P) * sizeof(double));
  if (!sm || !li) return -1;
  for (int s = 0; s < S; ++s) bimpc::solve_station<true>(c, a, s, sm, li, 0, 1);
  free(sm);
  free(li);
  return 0;
}

// The stage-weight loop bimpc_create ran before it called bimpc_stage_weights (kept to check that the two agree bit
// for bit).
extern "C" void bimpc_hostsim_stage_weights_loop(int N, int cost_type, double exp_rate, double* omega) {
  for (int k = 0; k < N; ++k) omega[k] = 1.0;
  if (cost_type == 2)
    for (int k = 0; k < N; ++k) omega[k] = std::pow(exp_rate, (double)(k - N + 1));
}
