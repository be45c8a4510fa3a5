// Plumbing kernels of the device-resident closed loop over S stations (include/fleet_b200.h):
// partition assignment + sort, BiMPC parameter assembly, reference gathering, plant update.
// All of it is byte/index shuffling over [S, M] arrays: coalesced loads, one CTA per station
// where a station-wide reduction is needed, fixed-order reductions (results do not depend on
// the launch geometry).  Stations may hold fewer EVs than the row stride M (nevs[s]) and
// carry their own capacity (Bcap[s]); the uniform entry points run the same kernels with
// null arrays, which stand for nevs[s] = M and the scalar Bcap.
#include <cmath>

#include "fleet_b200.h"
#include "lompc_common.cuh"

#define CK(call)                                                        \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) return lompc_detail::cuda_fail(e__, #call); \
  } while (0)

namespace {

constexpr int kMaxP = 64;

inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

// EVs of station s: the first nevs[s] slots of its row of M (clamped to [0, M], so that no
// index leaves the row), or all M when nevs is null (every station the same size).
__device__ __forceinline__ int station_evs(const int32_t* __restrict__ nevs, int s, int M) {
  return nevs ? min(max(nevs[s], 0), M) : M;
}

// Total EV capacity of station s: Bcap_s[s], or the fleet-wide Bcap when Bcap_s is null.
__device__ __forceinline__ double station_bcap(const double* __restrict__ Bcap_s, int s, double Bcap) {
  return Bcap_s ? Bcap_s[s] : Bcap;
}

// charging_station.py:111-116, one CTA per station.
__global__ void assign_kernel(int S, int M, int P, const int32_t* __restrict__ nevs, const double* __restrict__ edges,
                              const double* __restrict__ y, int32_t* __restrict__ idx, int32_t* __restrict__ counts) {
  __shared__ int hist[kMaxP];
  __shared__ double e[kMaxP + 1];
  const int s = blockIdx.x;
  const int n = station_evs(nevs, s, M);
  for (int p = threadIdx.x; p <= P; p += blockDim.x) e[p] = edges[p];
  for (int p = threadIdx.x; p < P; p += blockDim.x) hist[p] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = y[(size_t)s * M + i];
    int p = idx[(size_t)s * M + i];
    for (int q = 0; q < P; ++q)
      if (v >= e[q] && v <= e[q + 1]) p = q;  // the last matching partition wins
    idx[(size_t)s * M + i] = p;
    atomicAdd(&hist[p], 1);
  }
  __syncthreads();
  for (int p = threadIdx.x; p < P; p += blockDim.x) counts[(size_t)p * S + s] = hist[p];
}

// Exclusive scan of counts[n] by ONE CTA of 1024 threads (n = P*S is tens of thousands);
// also the per-partition rebased offsets.
__global__ void __launch_bounds__(1024) scan_kernel(int n, int S, int P, const int32_t* __restrict__ counts,
                                                    int32_t* __restrict__ off, int32_t* __restrict__ rebased) {
  __shared__ int part[1024];
  const int T = blockDim.x, t = threadIdx.x;
  const int per = (n + T - 1) / T;
  const int lo = min(t * per, n), hi = min(lo + per, n);
  int sum = 0;
  for (int i = lo; i < hi; ++i) sum += counts[i];
  part[t] = sum;
  __syncthreads();
  for (int d = 1; d < T; d <<= 1) {  // Hillis-Steele inclusive scan of the partials
    const int v = (t >= d) ? part[t - d] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  int run = part[t] - sum;
  for (int i = lo; i < hi; ++i) {
    off[i] = run;
    run += counts[i];
  }
  if (t == T - 1) off[n] = part[T - 1];
  __syncthreads();
  // rebased[p][s] = off[p*S+s] - off[p*S], s = 0..S
  for (int i = t; i < P * (S + 1); i += T) {
    const int p = i / (S + 1), s = i - p * (S + 1);
    rebased[i] = off[p * S + s] - off[p * S];
  }
}

// Stable gather of one group's EVs: thread (s, p) walks its station's EVs in order.
__global__ void gather_kernel(int S, int M, int P, const int32_t* __restrict__ nevs, const int32_t* __restrict__ idx,
                              const double* __restrict__ y, const int32_t* __restrict__ off,
                              double* __restrict__ y_sorted, int32_t* __restrict__ perm) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= S * P) return;
  const int s = i / P, p = i - s * P;
  const int n = station_evs(nevs, s, M);
  int pos = off[(size_t)p * S + s];
  const int32_t* ix = idx + (size_t)s * M;
  const double* ys = y + (size_t)s * M;
  for (int ev = 0; ev < n; ++ev)
    if (ix[ev] == p) {
      y_sorted[pos] = ys[ev];
      perm[pos] = ev;
      ++pos;
    }
}

__global__ void bimpc_params_kernel(int S, int P, int N_bi, int N_lo, double Bcap, const double* __restrict__ Bcap_s,
                                    double eps_tol, double lmbd_r,
                                    double delta_s, double delta_l, const int32_t* __restrict__ counts_s,
                                    const int32_t* __restrict__ counts_l, const double* __restrict__ y0_rng_s,
                                    const double* __restrict__ y0_rng_l, const double* __restrict__ gsm_s,
                                    const double* __restrict__ gsm_l, const double* __restrict__ x,
                                    const double* __restrict__ profile, int profile_len, int t,
                                    double* __restrict__ Mp_s, double* __restrict__ Mp_l, double* __restrict__ beta_s,
                                    double* __restrict__ beta_l, double* __restrict__ gamma_s,
                                    double* __restrict__ gamma_l, double* __restrict__ x0,
                                    double* __restrict__ demand) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < S * P) {
    const int s = i / P, p = i - s * P;
    const size_t g = (size_t)p * S + s;
    const double bc = station_bcap(Bcap_s, s, Bcap);
    const double sq = sqrt((double)N_lo);
    {  // price_solver.py:182-186: w0 bound = (sqrt(N) y0_rng + eps_tol) min(1, 1/sqrt(kappa)), kappa = lmbd_r/delta + 1e-5
      const int n = counts_s[g];
      Mp_s[i] = n / bc;
      beta_s[i] = n > 0 ? (sq * y0_rng_s[g] + eps_tol) * fmin(1.0, 1.0 / sqrt(lmbd_r / delta_s + 1e-5)) : 0.0;
      gamma_s[i] = n > 0 ? gsm_s[g] : 0.0;
    }
    {
      const int n = counts_l[g];
      Mp_l[i] = n / bc;
      beta_l[i] = n > 0 ? (sq * y0_rng_l[g] + eps_tol) * fmin(1.0, 1.0 / sqrt(lmbd_r / delta_l + 1e-5)) : 0.0;
      gamma_l[i] = n > 0 ? gsm_l[g] : 0.0;
    }
  }
  if (i < S * N_bi) {
    const int s = i / N_bi, k = i - s * N_bi;
    demand[i] = profile[(size_t)s * profile_len + t + k] / station_bcap(Bcap_s, s, Bcap);
  }
  if (i < S) x0[i] = x[i];
}

__global__ void wref_kernel(int S, int P, int N_bi, int N_lo, const double* __restrict__ w_hat,
                            double* __restrict__ w_ref) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)S * P * N_lo) return;
  const int k = (int)(i % N_lo);
  const int64_t g = i / N_lo;
  const int p = (int)(g / S), s = (int)(g - (int64_t)p * S);
  w_ref[i] = w_hat[((size_t)s * P + p) * N_bi + k];
}

__global__ void keep_prices_kernel(int S, int row, const int32_t* __restrict__ counts_p, const double* __restrict__ src,
                                   double* __restrict__ dst, const double* __restrict__ pre,
                                   const double* __restrict__ post, double* __restrict__ red) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)S * row) return;
  const int s = (int)(i / row);
  const bool full = counts_p[s] > 0;
  dst[i] = full ? src[i] : 0.0;
  if (i % row == 0 && red) red[s] = full ? post[s] - pre[s] : nan("");
}

// splitmix64-style counter hash -> uniform double in [0, 1)
__device__ __forceinline__ double counter_uniform(uint64_t seed, uint64_t a, uint64_t b, uint64_t c, uint64_t d) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (a + 1) + 0xBF58476D1CE4E5B9ull * (b + 1) +
               0x94D049BB133111EBull * (c + 1) + 0xD6E8FEB86659FD93ull * (d + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  z = (z ^ (z >> 33)) * 0xFF51AFD7ED558CCDull;
  z = z ^ (z >> 33);
  return (double)(z >> 11) * 0x1.0p-53;
}

// charging_station.py:329-349 for one EV type, one CTA (256 threads) per station.
__global__ void __launch_bounds__(256) apply_charge_kernel(
    int S, int M, int P, const int32_t* __restrict__ nevs, double full_level, double y0_min, double y0_max,
    long long rng_seed, int ev_type, int t, const int32_t* __restrict__ off, const int32_t* __restrict__ perm,
    const double* __restrict__ w0_sorted, double* __restrict__ y, int32_t* __restrict__ replace_mask,
    double* __restrict__ w_sum, double* __restrict__ w_mean, int32_t* __restrict__ ncharged) {
  __shared__ double red[256];
  __shared__ int cnt[256];
  const int s = blockIdx.x, tid = threadIdx.x;
  const int n = station_evs(nevs, s, M);
  double* ys = y + (size_t)s * M;
  // per group (fixed order inside the group): mean first-step charge, and the scatter
  for (int p = tid; p < P; p += blockDim.x) {
    const int b0 = off[(size_t)p * S + s], b1 = off[(size_t)p * S + s + 1];
    double sum = 0.0;
    for (int b = b0; b < b1; ++b) {
      const double w = w0_sorted[b];
      sum += w;
      ys[perm[b]] += w;
    }
    if (w_mean) w_mean[(size_t)p * S + s] = b1 > b0 ? sum / (b1 - b0) : 0.0;
    red[p] = sum;
  }
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int p = 0; p < P; ++p) tot += red[p];
    w_sum[s] = tot;
  }
  // departures / arrivals
  int mine = 0;
  for (int ev = tid; ev < n; ev += blockDim.x) {
    const bool leave = ys[ev] > full_level;
    if (replace_mask) replace_mask[(size_t)s * M + ev] = leave;
    if (leave) {
      ++mine;
      if (rng_seed >= 0)
        ys[ev] = y0_min + (y0_max - y0_min) * counter_uniform((uint64_t)rng_seed, ev_type, s, ev, t);
    }
  }
  cnt[tid] = mine;
  __syncthreads();
  if (tid == 0) {
    int tot = 0;
    for (int i = 0; i < blockDim.x; ++i) tot += cnt[i];
    ncharged[s] += tot;
  }
}

__global__ void battery_kernel(int S, int N_bi, double theta_s, double theta_l, double Bcap,
                               const double* __restrict__ Bcap_s, const double* __restrict__ u_g,
                               const double* __restrict__ ws, const double* __restrict__ wl,
                               const double* __restrict__ profile, int profile_len, int t, double* __restrict__ x) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const double u0_b = u_g[(size_t)s * N_bi] +
                      (-theta_s * ws[s] - theta_l * wl[s] - profile[(size_t)s * profile_len + t]) /
                          station_bcap(Bcap_s, s, Bcap);
  x[s] += u0_b;
}

int prep(int device) {
  if (lompc_device_count() <= device || device < 0) return LOMPC_ERR_NO_DEVICE;
  CK(cudaSetDevice(device));
  return LOMPC_OK;
}

// One launcher per job; the uniform entry points pass nevs = null (every station M EVs) or
// Bcap_s = null (the scalar Bcap), the sized ones pass the per-station arrays.
int partition(int device, int32_t S, int32_t M, int32_t P, const int32_t* nevs, const double* edges, const double* y,
              int32_t* idx, int32_t* counts, int32_t* off, int32_t* off_rebased, double* y_sorted, int32_t* perm,
              void* stream) {
  if (S < 1 || M < 1 || P < 1 || P > kMaxP || !edges || !y || !idx || !counts || !off || !off_rebased ||
      !y_sorted || !perm)
    return LOMPC_ERR_ARG;
  int rc = prep(device);
  if (rc) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  assign_kernel<<<S, 128, 0, s>>>(S, M, P, nevs, edges, y, idx, counts);
  lompc_detail::count_launch();
  scan_kernel<<<1, 1024, 0, s>>>(P * S, S, P, counts, off, off_rebased);
  lompc_detail::count_launch();
  gather_kernel<<<nblk((int64_t)S * P, 128), 128, 0, s>>>(S, M, P, nevs, idx, y, off, y_sorted, perm);
  lompc_detail::count_launch();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

int bimpc_params(int device, int32_t S, int32_t P, int32_t N_bi, int32_t N_lo, double Bcap, const double* Bcap_s,
                 double eps_tol, double lmbd_r, double delta_s, double delta_l, const int32_t* counts_s,
                 const int32_t* counts_l, const double* y0_rng_s, const double* y0_rng_l, const double* gamma_sm_s,
                 const double* gamma_sm_l, const double* x, const double* demand_profile, int32_t profile_len,
                 int32_t t, double* Mp_s, double* Mp_l, double* beta_s, double* beta_l, double* gamma_s,
                 double* gamma_l, double* x0, double* demand, void* stream) {
  if (S < 1 || P < 1 || N_bi < 1 || N_lo < 1 || !(Bcap_s || Bcap > 0) || !counts_s || !counts_l || !y0_rng_s ||
      !y0_rng_l || !gamma_sm_s || !gamma_sm_l || !x || !demand_profile || t < 0 || t + N_bi > profile_len || !Mp_s ||
      !Mp_l || !beta_s || !beta_l || !gamma_s || !gamma_l || !x0 || !demand)
    return LOMPC_ERR_ARG;
  int rc = prep(device);
  if (rc) return rc;
  const int64_t n = (int64_t)S * (P > N_bi ? P : N_bi);
  bimpc_params_kernel<<<nblk(n, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      S, P, N_bi, N_lo, Bcap, Bcap_s, eps_tol, lmbd_r, delta_s, delta_l, counts_s, counts_l, y0_rng_s, y0_rng_l,
      gamma_sm_s, gamma_sm_l, x, demand_profile, profile_len, t, Mp_s, Mp_l, beta_s, beta_l, gamma_s, gamma_l, x0,
      demand);
  lompc_detail::count_launch();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

int apply_charge(int device, int32_t S, int32_t M, int32_t P, const int32_t* nevs, double full_level, double y0_min,
                 double y0_max, int64_t rng_seed, int32_t ev_type, int32_t t, const int32_t* off, const int32_t* perm,
                 const double* w0_sorted, double* y, int32_t* replace_mask, double* w_sum, double* w_mean,
                 int32_t* ncharged, void* stream) {
  if (S < 1 || M < 1 || P < 1 || P > 256 || !off || !perm || !w0_sorted || !y || !w_sum || !ncharged)
    return LOMPC_ERR_ARG;
  if (rng_seed < 0 && !replace_mask) return LOMPC_ERR_ARG;
  int rc = prep(device);
  if (rc) return rc;
  apply_charge_kernel<<<S, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      S, M, P, nevs, full_level, y0_min, y0_max, (long long)rng_seed, ev_type, t, off, perm, w0_sorted, y,
      replace_mask, w_sum, w_mean, ncharged);
  lompc_detail::count_launch();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

int battery(int device, int32_t S, int32_t N_bi, double theta_s, double theta_l, double Bcap, const double* Bcap_s,
            const double* u_g, const double* w_sum_s, const double* w_sum_l, const double* demand_profile,
            int32_t profile_len, int32_t t, double* x, void* stream) {
  if (S < 1 || !u_g || !w_sum_s || !w_sum_l || !demand_profile || t < 0 || t >= profile_len || !x)
    return LOMPC_ERR_ARG;
  int rc = prep(device);
  if (rc) return rc;
  battery_kernel<<<nblk(S, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      S, N_bi, theta_s, theta_l, Bcap, Bcap_s, u_g, w_sum_s, w_sum_l, demand_profile, profile_len, t, x);
  lompc_detail::count_launch();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

}  // namespace

extern "C" {

int fleet_partition_dev(int device, int32_t S, int32_t M, int32_t P, const double* edges, const double* y,
                        int32_t* idx, int32_t* counts, int32_t* off, int32_t* off_rebased,
                        double* y_sorted, int32_t* perm, void* stream) {
  return partition(device, S, M, P, nullptr, edges, y, idx, counts, off, off_rebased, y_sorted, perm, stream);
}

int fleet_partition_sized_dev(int device, int32_t S, int32_t M, int32_t P, const int32_t* nevs, const double* edges,
                              const double* y, int32_t* idx, int32_t* counts, int32_t* off, int32_t* off_rebased,
                              double* y_sorted, int32_t* perm, void* stream) {
  if (!nevs) return LOMPC_ERR_ARG;
  return partition(device, S, M, P, nevs, edges, y, idx, counts, off, off_rebased, y_sorted, perm, stream);
}

int fleet_bimpc_params_dev(int device, int32_t S, int32_t P, int32_t N_bi, int32_t N_lo, double Bcap,
                           double eps_tol, double lmbd_r, double delta_s, double delta_l,
                           const int32_t* counts_s, const int32_t* counts_l, const double* y0_rng_s,
                           const double* y0_rng_l, const double* gamma_sm_s, const double* gamma_sm_l,
                           const double* x, const double* demand_profile, int32_t profile_len, int32_t t,
                           double* Mp_s, double* Mp_l, double* beta_s, double* beta_l, double* gamma_s,
                           double* gamma_l, double* x0, double* demand, void* stream) {
  return bimpc_params(device, S, P, N_bi, N_lo, Bcap, nullptr, eps_tol, lmbd_r, delta_s, delta_l, counts_s, counts_l,
                      y0_rng_s, y0_rng_l, gamma_sm_s, gamma_sm_l, x, demand_profile, profile_len, t, Mp_s, Mp_l,
                      beta_s, beta_l, gamma_s, gamma_l, x0, demand, stream);
}

int fleet_bimpc_params_sized_dev(int device, int32_t S, int32_t P, int32_t N_bi, int32_t N_lo, const double* Bcap,
                                 double eps_tol, double lmbd_r, double delta_s, double delta_l,
                                 const int32_t* counts_s, const int32_t* counts_l, const double* y0_rng_s,
                                 const double* y0_rng_l, const double* gamma_sm_s, const double* gamma_sm_l,
                                 const double* x, const double* demand_profile, int32_t profile_len, int32_t t,
                                 double* Mp_s, double* Mp_l, double* beta_s, double* beta_l, double* gamma_s,
                                 double* gamma_l, double* x0, double* demand, void* stream) {
  if (!Bcap) return LOMPC_ERR_ARG;
  return bimpc_params(device, S, P, N_bi, N_lo, 0.0, Bcap, eps_tol, lmbd_r, delta_s, delta_l, counts_s, counts_l,
                      y0_rng_s, y0_rng_l, gamma_sm_s, gamma_sm_l, x, demand_profile, profile_len, t, Mp_s, Mp_l,
                      beta_s, beta_l, gamma_s, gamma_l, x0, demand, stream);
}

int fleet_wref_dev(int device, int32_t S, int32_t P, int32_t N_bi, int32_t N_lo, const double* w_hat,
                   double* w_ref, void* stream) {
  if (S < 1 || P < 1 || N_lo < 1 || N_bi < N_lo || !w_hat || !w_ref) return LOMPC_ERR_ARG;
  int rc = prep(device);
  if (rc) return rc;
  wref_kernel<<<nblk((int64_t)S * P * N_lo, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(S, P, N_bi, N_lo,
                                                                                             w_hat, w_ref);
  lompc_detail::count_launch();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

int fleet_keep_prices_dev(int device, int32_t S, int32_t row, const int32_t* counts_p, const double* src,
                          double* dst, const double* price_pre, const double* price_post,
                          double* price_red, void* stream) {
  if (S < 1 || row < 1 || !counts_p || !src || !dst) return LOMPC_ERR_ARG;
  if (price_red && (!price_pre || !price_post)) return LOMPC_ERR_ARG;
  int rc = prep(device);
  if (rc) return rc;
  keep_prices_kernel<<<nblk((int64_t)S * row, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      S, row, counts_p, src, dst, price_pre, price_post, price_red);
  lompc_detail::count_launch();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

int fleet_apply_charge_dev(int device, int32_t S, int32_t M, int32_t P, double full_level, double y0_min,
                           double y0_max, int64_t rng_seed, int32_t ev_type, int32_t t, const int32_t* off,
                           const int32_t* perm, const double* w0_sorted, double* y, int32_t* replace_mask,
                           double* w_sum, double* w_mean, int32_t* ncharged, void* stream) {
  return apply_charge(device, S, M, P, nullptr, full_level, y0_min, y0_max, rng_seed, ev_type, t, off, perm, w0_sorted,
                      y, replace_mask, w_sum, w_mean, ncharged, stream);
}

int fleet_apply_charge_sized_dev(int device, int32_t S, int32_t M, int32_t P, const int32_t* nevs, double full_level,
                                 double y0_min, double y0_max, int64_t rng_seed, int32_t ev_type, int32_t t,
                                 const int32_t* off, const int32_t* perm, const double* w0_sorted, double* y,
                                 int32_t* replace_mask, double* w_sum, double* w_mean, int32_t* ncharged,
                                 void* stream) {
  if (!nevs) return LOMPC_ERR_ARG;
  return apply_charge(device, S, M, P, nevs, full_level, y0_min, y0_max, rng_seed, ev_type, t, off, perm, w0_sorted,
                      y, replace_mask, w_sum, w_mean, ncharged, stream);
}

int fleet_battery_dev(int device, int32_t S, int32_t N_bi, double theta_s, double theta_l, double Bcap,
                      const double* u_g, const double* w_sum_s, const double* w_sum_l,
                      const double* demand_profile, int32_t profile_len, int32_t t, double* x,
                      void* stream) {
  return battery(device, S, N_bi, theta_s, theta_l, Bcap, nullptr, u_g, w_sum_s, w_sum_l, demand_profile, profile_len,
                 t, x, stream);
}

int fleet_battery_sized_dev(int device, int32_t S, int32_t N_bi, double theta_s, double theta_l, const double* Bcap,
                            const double* u_g, const double* w_sum_s, const double* w_sum_l,
                            const double* demand_profile, int32_t profile_len, int32_t t, double* x, void* stream) {
  if (!Bcap) return LOMPC_ERR_ARG;
  return battery(device, S, N_bi, theta_s, theta_l, 0.0, Bcap, u_g, w_sum_s, w_sum_l, demand_profile, profile_len, t,
                 x, stream);
}

}  // extern "C"
