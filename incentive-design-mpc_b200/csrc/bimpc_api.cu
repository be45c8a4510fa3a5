// C ABI of the batched BiMPC (see include/bimpc_b200.h).
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "bimpc_b200.h"
#include "bimpc_solve.cuh"
#include "lompc_common.cuh"

#define CK(call)                                                        \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) return lompc_detail::cuda_fail(e__, #call); \
  } while (0)

struct bimpc_handle {
  bimpc::BiConsts c;
  int device;
  int max_iter;
  double tol;
  double* omega;  // device [N]
  int threads;
  size_t smem;
  int ctas_per_sm, sms;
  int ctas_per_sm_st;  // of the per-station kernel
  double* li;     // [grid, N, np] inverse-factor scratch of the kernel
  void* ws;       // grow-only device workspace of the _host entry point
  size_t ws_bytes;
};

extern "C" {

int bimpc_stage_weights(int N, int cost_type, double exp_rate, double* omega) {
  if (N < 1 || !omega) return LOMPC_ERR_ARG;
  if (cost_type < 0 || cost_type > 2 || !(exp_rate >= 1)) return LOMPC_ERR_CONSTS;
  // exp_rate^(k-N+1) (bimpc.py:255-257), ones otherwise
  for (int k = 0; k < N; ++k) omega[k] = 1.0;
  if (cost_type == BIMPC_COST_EXP_UNWEIGHTED)
    for (int k = 0; k < N; ++k) omega[k] = std::pow(exp_rate, (double)(k - N + 1));
  return LOMPC_OK;
}

int bimpc_create(int N, int P, double delta, double c_g, double u_g_max, double u_b_max,
                 double x_max, int cost_type, double exp_rate, double theta_s, double theta_l,
                 double w_max_s, double w_max_l, int device, bimpc_t** out) {
  if (!out || N < 1 || P < 1) return LOMPC_ERR_ARG;
  *out = nullptr;
  // bimpc.py:79-84
  if (!(delta >= 0) || !(c_g >= 0) || !(u_g_max >= 0) || !(u_b_max >= 0) || !(x_max >= 0) || !(exp_rate >= 1))
    return LOMPC_ERR_CONSTS;
  if (cost_type < 0 || cost_type > 2) return LOMPC_ERR_CONSTS;  // NotImplementedError, bimpc.py:231
  if (!(theta_s > 0) || !(theta_l > 0) || !(w_max_s > 0) || !(w_max_l > 0)) return LOMPC_ERR_ARG;
  if (N > bimpc::kMaxN) return LOMPC_ERR_ARG;
  if (lompc_device_count() <= device || device < 0) return LOMPC_ERR_NO_DEVICE;
  CK(cudaSetDevice(device));
  bimpc_handle* h = new (std::nothrow) bimpc_handle();
  if (!h) return LOMPC_ERR_ARG;
  h->c = bimpc::BiConsts{N, P, delta, c_g, u_g_max, u_b_max, x_max, cost_type, theta_s, theta_l, w_max_s, w_max_l};
  h->device = device;
  h->max_iter = 100;
  h->tol = 1e-9;
  h->threads = bimpc::kThreads;
  h->smem = bimpc::scratch_doubles(N, P, h->threads) * sizeof(double);
  h->ws = nullptr;
  h->ws_bytes = 0;
  h->li = nullptr;
  h->omega = nullptr;
  cudaDeviceProp prop;
  if (cudaError_t e = cudaGetDeviceProperties(&prop, device); e != cudaSuccess) {
    delete h;
    return lompc_detail::cuda_fail(e, "cudaGetDeviceProperties");
  }
  h->sms = prop.multiProcessorCount;
  if (h->smem > (size_t)prop.sharedMemPerBlockOptin) {
    delete h;
    return LOMPC_ERR_ARG;
  }
  // The opt-in is a per-device attribute of the FUNCTION, shared by every handle: always ask for the device's
  // maximum, so that a later, smaller handle cannot lower the limit under an earlier, larger one.
  for (auto kernel : {bimpc::bimpc_solve_kernel<false>, bimpc::bimpc_solve_kernel<true>})
    if (cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)prop.sharedMemPerBlockOptin);
        e != cudaSuccess) {
      delete h;
      return lompc_detail::cuda_fail(e, "cudaFuncSetAttribute(bimpc_solve_kernel)");
    }
  // from here on a failing CUDA call releases the handle and whatever it already owns
#define CKH(call)                                        \
  do {                                                   \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) {                            \
      bimpc_destroy(h);                                  \
      return lompc_detail::cuda_fail(e__, #call);        \
    }                                                    \
  } while (0)
  int occ = 1, occ_st = 1;
  CKH(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bimpc::bimpc_solve_kernel<false>, h->threads, h->smem));
  CKH(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_st, bimpc::bimpc_solve_kernel<true>, h->threads, h->smem));
  h->ctas_per_sm = occ < 1 ? 1 : occ;
  h->ctas_per_sm_st = occ_st < 1 ? 1 : occ_st;
  const int ctas_max = h->ctas_per_sm > h->ctas_per_sm_st ? h->ctas_per_sm : h->ctas_per_sm_st;
  CKH(cudaMalloc(&h->li, (size_t)h->sms * ctas_max * bimpc::global_scratch_doubles(N, P) * sizeof(double)));
  std::vector<double> om(N);
  bimpc_stage_weights(N, cost_type, exp_rate, om.data());
  CKH(cudaMalloc(&h->omega, N * sizeof(double)));
  CKH(cudaMemcpy(h->omega, om.data(), N * sizeof(double), cudaMemcpyHostToDevice));
#undef CKH
  *out = h;
  return LOMPC_OK;
}

int bimpc_destroy(bimpc_t* h) {
  if (!h) return LOMPC_OK;
  cudaSetDevice(h->device);
  if (h->omega) cudaFree(h->omega);
  if (h->li) cudaFree(h->li);
  if (h->ws) cudaFree(h->ws);
  delete h;
  return LOMPC_OK;
}

int bimpc_set_options(bimpc_t* h, int max_iter, double tol) {
  if (!h || max_iter < 1 || !(tol > 0.0)) return LOMPC_ERR_ARG;
  h->max_iter = max_iter;
  h->tol = tol;
  return LOMPC_OK;
}

}  // extern "C"

namespace {

bool null_arg(bimpc_t* h, int32_t S, const double* Mp_s, const double* Mp_l, const double* beta_s,
              const double* beta_l, const double* gamma_sm, const double* gamma_lm, const double* x0,
              const double* demand, double* w_hat_s, double* w_hat_l, double* u_g, int32_t* status, int32_t* iters) {
  return !h || S < 0 || !Mp_s || !Mp_l || !beta_s || !beta_l || !gamma_sm || !gamma_lm || !x0 || !demand ||
         !w_hat_s || !w_hat_l || !u_g || !status || !iters;
}

// Per-station constants of the _consts entry points (device pointers), or none.
struct StationConsts {
  const double *delta, *c_g, *u_g_max, *u_b_max, *x_max;
  const int32_t* cost_type;
  const double* omega;
};

int launch(bimpc_t* h, int32_t S, const StationConsts* sc, const double* Mp_s, const double* Mp_l,
           const double* beta_s, const double* beta_l, const double* gamma_sm, const double* gamma_lm,
           const double* x0, const double* demand, double* w_hat_s, double* w_hat_l, double* u_g, int32_t* status,
           int32_t* iters, double* objective, void* stream) {
  if (S == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  bimpc::BiArgs a{S, h->omega, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand,
                  w_hat_s, w_hat_l, u_g, status, iters, objective, h->tol, h->max_iter, nullptr, h->li};
  int grid = h->sms * (sc ? h->ctas_per_sm_st : h->ctas_per_sm);  // persistent CTAs, one station at a time each
  if (grid > S) grid = S;
  if (sc) {
    a.st_delta = sc->delta;
    a.st_c_g = sc->c_g;
    a.st_u_g_max = sc->u_g_max;
    a.st_u_b_max = sc->u_b_max;
    a.st_x_max = sc->x_max;
    a.st_cost_type = sc->cost_type;
    a.st_omega = sc->omega;
    bimpc::bimpc_solve_kernel<true><<<grid, h->threads, h->smem, static_cast<cudaStream_t>(stream)>>>(h->c, a);
  } else {
    bimpc::bimpc_solve_kernel<false><<<grid, h->threads, h->smem, static_cast<cudaStream_t>(stream)>>>(h->c, a);
  }
  lompc_detail::count_launch();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

// The _host entry points: copy in, solve, copy out, synchronise.  `exp_rate` != NULL: per-station constants on the
// host (`sc` holds host pointers, its omega is built here).
int solve_host(bimpc_t* h, int32_t S, const StationConsts* sc, const double* exp_rate, const double* Mp_s,
               const double* Mp_l, const double* beta_s, const double* beta_l, const double* gamma_sm,
               const double* gamma_lm, const double* x0, const double* demand, double* w_hat_s, double* w_hat_l,
               double* u_g, int32_t* status, int32_t* iters, double* objective) {
  if (S == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  const int N = h->c.N, P = h->c.P;
  const size_t sp = (size_t)S * P * 8, sn = (size_t)S * N * 8, spn = (size_t)S * P * N * 8, s1 = (size_t)S * 8;
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t total = 6 * al(sp) + al(s1) + al(sn) + 2 * al(spn) + al(sn) + 2 * al((size_t)S * 4) + al(s1);
  if (sc) total += 5 * al(s1) + al((size_t)S * 4) + al(sn);
  if (h->ws_bytes < total) {
    if (h->ws) CK(cudaFree(h->ws));
    h->ws = nullptr;
    h->ws_bytes = 0;
    CK(cudaMalloc(&h->ws, total + total / 4));
    h->ws_bytes = total + total / 4;
  }
  char* p = static_cast<char*>(h->ws);
  auto take = [&](size_t bytes) { char* q = p; p += al(bytes); return q; };
  double* d_in[6];
  const double* h_in[6] = {Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm};
  cudaStream_t s = 0;
  for (int i = 0; i < 6; ++i) {
    d_in[i] = (double*)take(sp);
    CK(cudaMemcpyAsync(d_in[i], h_in[i], sp, cudaMemcpyHostToDevice, s));
  }
  double* d_x0 = (double*)take(s1);
  double* d_dem = (double*)take(sn);
  double* d_ws = (double*)take(spn);
  double* d_wl = (double*)take(spn);
  double* d_ug = (double*)take(sn);
  int32_t* d_st = (int32_t*)take((size_t)S * 4);
  int32_t* d_it = (int32_t*)take((size_t)S * 4);
  double* d_obj = (double*)take(s1);
  CK(cudaMemcpyAsync(d_x0, x0, s1, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_dem, demand, sn, cudaMemcpyHostToDevice, s));
  StationConsts dsc{};
  std::vector<double> om;
  if (sc) {
    // a station whose cost type or exp_rate bimpc_stage_weights refuses gets NaN weights: the kernel gives it status 2
    om.assign((size_t)S * N, NAN);
    for (int i = 0; i < S; ++i)
      if (bimpc_stage_weights(N, sc->cost_type[i], exp_rate[i], om.data() + (size_t)i * N) != LOMPC_OK)
        for (int k = 0; k < N; ++k) om[(size_t)i * N + k] = NAN;
    const double* h5[5] = {sc->delta, sc->c_g, sc->u_g_max, sc->u_b_max, sc->x_max};
    double* d5[5];
    for (int i = 0; i < 5; ++i) {
      d5[i] = (double*)take(s1);
      CK(cudaMemcpyAsync(d5[i], h5[i], s1, cudaMemcpyHostToDevice, s));
    }
    int32_t* d_ct = (int32_t*)take((size_t)S * 4);
    double* d_om = (double*)take(sn);
    CK(cudaMemcpyAsync(d_ct, sc->cost_type, (size_t)S * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_om, om.data(), sn, cudaMemcpyHostToDevice, s));
    dsc = StationConsts{d5[0], d5[1], d5[2], d5[3], d5[4], d_ct, d_om};
  }
  int rc = launch(h, S, sc ? &dsc : nullptr, d_in[0], d_in[1], d_in[2], d_in[3], d_in[4], d_in[5], d_x0, d_dem, d_ws,
                  d_wl, d_ug, d_st, d_it, d_obj, s);
  if (rc) return rc;
  CK(cudaMemcpyAsync(w_hat_s, d_ws, spn, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(w_hat_l, d_wl, spn, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(u_g, d_ug, sn, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(status, d_st, (size_t)S * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(iters, d_it, (size_t)S * 4, cudaMemcpyDeviceToHost, s));
  if (objective) CK(cudaMemcpyAsync(objective, d_obj, s1, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  for (int i = 0; i < S; ++i)
    if (status[i] != BIMPC_ST_OK) return LOMPC_ERR_NOT_CONVERGED;
  return LOMPC_OK;
}

}  // namespace

extern "C" {

int bimpc_solve_batch_dev(bimpc_t* h, int32_t S, const double* Mp_s, const double* Mp_l,
                          const double* beta_s, const double* beta_l, const double* gamma_sm,
                          const double* gamma_lm, const double* x0, const double* demand,
                          double* w_hat_s, double* w_hat_l, double* u_g, int32_t* status,
                          int32_t* iters, double* objective, void* stream) {
  if (null_arg(h, S, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, w_hat_s, w_hat_l, u_g, status, iters))
    return LOMPC_ERR_ARG;
  return launch(h, S, nullptr, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, w_hat_s, w_hat_l, u_g,
                status, iters, objective, stream);
}

int bimpc_solve_batch_host(bimpc_t* h, int32_t S, const double* Mp_s, const double* Mp_l,
                           const double* beta_s, const double* beta_l, const double* gamma_sm,
                           const double* gamma_lm, const double* x0, const double* demand,
                           double* w_hat_s, double* w_hat_l, double* u_g, int32_t* status,
                           int32_t* iters, double* objective) {
  if (null_arg(h, S, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, w_hat_s, w_hat_l, u_g, status, iters))
    return LOMPC_ERR_ARG;
  return solve_host(h, S, nullptr, nullptr, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, w_hat_s,
                    w_hat_l, u_g, status, iters, objective);
}

int bimpc_solve_batch_consts_dev(bimpc_t* h, int32_t S, const double* delta, const double* c_g,
                                 const double* u_g_max, const double* u_b_max, const double* x_max,
                                 const int32_t* cost_type, const double* omega, const double* Mp_s,
                                 const double* Mp_l, const double* beta_s, const double* beta_l,
                                 const double* gamma_sm, const double* gamma_lm, const double* x0,
                                 const double* demand, double* w_hat_s, double* w_hat_l, double* u_g,
                                 int32_t* status, int32_t* iters, double* objective, void* stream) {
  if (null_arg(h, S, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, w_hat_s, w_hat_l, u_g, status, iters))
    return LOMPC_ERR_ARG;
  if (!delta || !c_g || !u_g_max || !u_b_max || !x_max || !cost_type || !omega) return LOMPC_ERR_ARG;
  const StationConsts sc{delta, c_g, u_g_max, u_b_max, x_max, cost_type, omega};
  return launch(h, S, &sc, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, w_hat_s, w_hat_l, u_g, status,
                iters, objective, stream);
}

int bimpc_solve_batch_consts_host(bimpc_t* h, int32_t S, const double* delta, const double* c_g,
                                  const double* u_g_max, const double* u_b_max, const double* x_max,
                                  const int32_t* cost_type, const double* exp_rate, const double* Mp_s,
                                  const double* Mp_l, const double* beta_s, const double* beta_l,
                                  const double* gamma_sm, const double* gamma_lm, const double* x0,
                                  const double* demand, double* w_hat_s, double* w_hat_l, double* u_g,
                                  int32_t* status, int32_t* iters, double* objective) {
  if (null_arg(h, S, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, w_hat_s, w_hat_l, u_g, status, iters))
    return LOMPC_ERR_ARG;
  if (!delta || !c_g || !u_g_max || !u_b_max || !x_max || !cost_type || !exp_rate) return LOMPC_ERR_ARG;
  const StationConsts sc{delta, c_g, u_g_max, u_b_max, x_max, cost_type, nullptr};
  return solve_host(h, S, &sc, exp_rate, Mp_s, Mp_l, beta_s, beta_l, gamma_sm, gamma_lm, x0, demand, w_hat_s,
                    w_hat_l, u_g, status, iters, objective);
}

}  // extern "C"
