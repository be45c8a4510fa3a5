// Vector-Jacobian product of the grouped LoMPC solve (lompc_group_vjp_dev, include/lompc_b200.h), sm_100a, fp64.
//
// EVs are sorted by group: group g owns EVs [off[g], off[g+1]) and all of them see the group's prices lmbd[g]
// (3N) and lmbd_r[g]; they differ only in gamma_i.  The forward pass returns w_i and w_avg_g = mean_i w_i.  For
// upstream gradients grad_w[B,N] and grad_w_avg[G,N] the upstream on w_i (i in g) is
//   gw_i = grad_w[i] + grad_w_avg[g] / n_g,
// z_i is the adjoint of lompc_vjp_kernel for that gw_i (same classification, same recursion: vjp_qp of lompc_vjp.cuh), and
//   dL/dlmbd1_g = -theta sum_i z_i,  dL/dlmbd2_g = theta sum_i z_i,  dL/dlmbd3_g = -2q sum_i z_i .* w_i,
//   dL/dlmbd_r,g = -2 theta^2 sum_i z_i'w_i,  dL/dgamma_i = c sum_k (N - k) z_i,k.
// Two launches, no atomics: group_vjp_ev_kernel (one EV per thread) writes z_i and z_i'w_i to a workspace,
// group_vjp_sum_kernel (one thread per (group, stage)) adds them in EV order.  A group's result depends only on its
// own EVs, so it has the same bits whatever else is in the batch.
#pragma once
#include "lompc_common.cuh"
#include "lompc_vjp.cuh"

namespace lompc {

struct GroupVjpArgs {
  int G;
  int64_t B;
  const int32_t* off;         // [G+1]
  const double* lmbd;         // [G,3N]
  const double* lmbd_r;       // [G]
  const double* gamma;        // [B]
  const double* w;            // [B,N]
  const double* grad_w;       // [B,N] or NULL (zero)
  const double* grad_w_avg;   // [G,N] or NULL (zero)
  double* z;                  // [B,N] workspace: the adjoints (0 for an invalid EV)
  double* zw;                 // [B]   workspace: z_i'w_i (0 for an invalid EV)
  double* grad_gamma;         // [B] or NULL
  int32_t* status;            // [B] or NULL
  double* grad_lmbd;          // [G,3N] or NULL
  double* grad_lmbd_r;        // [G] or NULL
};

// One EV per thread; shared-memory columns as lompc_vjp_kernel (kVjpArrays * N doubles per thread).
template <int NSEG>
__global__ void __launch_bounds__(128) group_vjp_ev_kernel(const Consts cs, const GroupVjpArgs a) {
  extern __shared__ double smem[];
  const int T = blockDim.x;
  const int t = threadIdx.x;
  const int64_t b = (int64_t)blockIdx.x * T + t;
  if (b >= a.B) return;  // no block-level sync below
  vjp_qp<NSEG, true>(cs, a, smem + t, T, b);
}

// One thread per (group, stage): the group's sums in EV order (eight loads in flight, as colsum_body).  Thread k = 0
// also forms the lmbd_r gradient.  An empty group gets zeros.  A stage with z = 0 (fixed, or an invalid EV) adds
// nothing to z.*w: the w of an invalid EV may be NaN.
__global__ void group_vjp_sum_kernel(const Consts cs, const GroupVjpArgs a) {
  const int N = cs.N;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.G * N) return;
  const int g = (int)(idx / N), k = (int)(idx % N);
  const int b0 = a.off[g], b1 = a.off[g + 1];
  if (a.grad_lmbd) {
    const double* zc = a.z + k;
    const double* wc = a.w + k;
    double sz = 0.0, szw = 0.0;
    int b = b0;
    for (; b + 8 <= b1; b += 8) {
      double zv[8], wv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        zv[u] = zc[(int64_t)(b + u) * N];
        wv[u] = wc[(int64_t)(b + u) * N];
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        sz += zv[u];
        szw = zv[u] != 0.0 ? fma(zv[u], wv[u], szw) : szw;
      }
    }
    for (; b < b1; ++b) {
      const double zb = zc[(int64_t)b * N];
      sz += zb;
      szw = zb != 0.0 ? fma(zb, wc[(int64_t)b * N], szw) : szw;
    }
    double* gl = a.grad_lmbd + (int64_t)g * (3 * N);
    gl[k] = -cs.theta * sz;
    gl[N + k] = cs.theta * sz;
    gl[2 * N + k] = -2.0 * cs.q_scale * szw;
  }
  if (k == 0 && a.grad_lmbd_r) {
    double s = 0.0;
    int b = b0;
    for (; b + 8 <= b1; b += 8) {
      double v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = a.zw[b + u];
#pragma unroll
      for (int u = 0; u < 8; ++u) s += v[u];
    }
    for (; b < b1; ++b) s += a.zw[b];
    a.grad_lmbd_r[g] = -2.0 * cs.theta2 * s;
  }
}

}  // namespace lompc
