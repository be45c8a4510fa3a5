// Vector-Jacobian product of the batched LoMPC solve (K1, lompc_solve.cuh), one QP per thread (sm_100a, fp64).
//
// The QP of K1 is  min 1/2 w'Hw + g'w + kappa0 + psi(w)  over 0 <= w <= w_max, with
//   H = diag(d) + c A'A,  d_k = 2(lmbd_r theta^2 + q lmbd3_k) [+ 2 theta^2/0.81 small EV],
//   g_k = theta (lmbd1_k - lmbd2_k) - c gamma (N - k),  c = 2 delta theta^2,  q = 3 theta / (4 w_max),
// and psi the large-EV pwl, piecewise LINEAR (no curvature).  Given the solution w, a coordinate is FIXED
// (set B) when it lies within band = 1e-9 w_max of a breakpoint (0, w_max or an interior pwl breakpoint: the
// binding rule of K1's backward sweep) and FREE (set F) otherwise.  Where the active set is locally constant,
// dw_B = 0 and dw_F = -H_FF^-1 (dg_F + dd_F .* w_F).  So for an upstream gradient gw[N] on w, with
// z = the solution of H_FF z_F = gw_F, z_B = 0:
//   dL/dlmbd1 = -theta z,  dL/dlmbd2 = theta z,  dL/dlmbd3 = -2q z.*w,
//   dL/dlmbd_r = -2 theta^2 sum_k z_k w_k,  dL/dgamma = c sum_k (N - k) z_k.
// For an upstream gradient gc on the cost as K1 returns it (kappa0 included, no 1/2 c N gamma^2 term), the
// envelope theorem gives, at every point:
//   dcost/dlmbd1 = theta w,  dcost/dlmbd2 = theta (w_max - w),  dcost/dlmbd3 = q w.^2,
//   dcost/dlmbd_r = theta^2 sum w.^2,  dcost/dgamma = -c sum_k s_k,  s = cumsum(w).
//
// Non-differentiable points: at a weakly active coordinate (on a breakpoint with its multiplier at an end of
// the subdifferential interval) w is not differentiable in the prices.  The kernel returns the derivative of
// the active set it classifies from w with the band above, which is one of the one-sided derivatives there.
//
// H_FF z = gw_F is solved as the scalar-state control problem  min 1/2 sum d_k z_k^2 + c/2 sum sigma_k^2 - gw'z,
// sigma_k = sigma_{k-1} + z_k, z_B = 0: with M = c + P_{k+1} (P_N = 0, r_N = 0), the backward pass is
//   fixed stage: P_k = M, r_k = r_{k+1};   free stage: P_k = d M / (d + M), r_k = (d r_{k+1} + M gw_k) / (d + M),
// and the forward pass z_k = -(M_k sigma_{k-1} + r_{k+1} - gw_k) / (d_k + M_k) on free stages.  d + M >= c > 0,
// so the recursion exists for d_k = 0 stages too, and P <= c N keeps it in range for every N.
#pragma once
#include "lompc_common.cuh"

namespace lompc {

struct VjpArgs {
  int64_t B;
  const double* lmbd;  // [rows, 3N], row stride lmbd_stride (0: one row for the whole batch)
  int64_t lmbd_stride;
  const double* lmbd_r;  // stride lmbd_r_stride (0: one scalar)
  int64_t lmbd_r_stride;
  const double* gamma;      // [B]
  const double* w;          // [B, N] the solution of the forward solve
  const double* grad_w;     // [B, N] or NULL (zero)
  const double* grad_cost;  // [B] or NULL (zero)
  double* grad_lmbd;        // [B, 3N] or NULL
  double* grad_lmbd_r;      // [B] or NULL
  double* grad_gamma;       // [B] or NULL
  int32_t* status;          // [B] or NULL: LOMPC_ST_OK, or the K1 status of an invalid row
};

// Per-stage vectors of the recursion, one column per thread ([k*T + t]): M_k, r_{k+1} - gw_k, 1/(d_k + M_k)
// (0 on fixed stages) and w_k.
constexpr int kVjpArrays = 4;

template <int NSEG>
__global__ void __launch_bounds__(128) lompc_vjp_kernel(const Consts cs, const VjpArgs a) {
  extern __shared__ double smem[];
  const int T = blockDim.x;
  const int t = threadIdx.x;
  const int N = cs.N;
  const int64_t b = (int64_t)blockIdx.x * T + t;
  if (b >= a.B) return;  // no block-level sync below

  double* MM = smem + t;
  double* RR = MM + (size_t)N * T;
  double* IV = RR + (size_t)N * T;
  double* WW = IV + (size_t)N * T;

  const double* lm = a.lmbd + b * a.lmbd_stride;
  const double lr = a.lmbd_r[b * a.lmbd_r_stride];
  const double gam = a.gamma[b];
  const double* wr = a.w + b * (int64_t)N;
  const double* gw = a.grad_w ? a.grad_w + b * (int64_t)N : nullptr;
  const double gc = a.grad_cost ? a.grad_cost[b] : 0.0;
  const double c = cs.c, wmax = cs.w_max;
  const double band = 1e-9 * wmax;  // K1's binding band (lompc_solve.cuh)
  double blo[NSEG + 1], bhi[NSEG + 1];
#pragma unroll
  for (int i = 0; i <= NSEG; ++i) {
    blo[i] = cs.brk[i] - band;
    bhi[i] = cs.brk[i] + band;
  }

  // ---- backward pass: validation (as K1), classification, Riccati recursion of H_FF z = gw_F ----------------
  int st = LOMPC_ST_OK;
  if (!(gam >= 0.0) || !(lr >= 0.0)) st = LOMPC_ST_NEGATIVE;
  double P = 0.0, r = 0.0;
  for (int k = N - 1; k >= 0; --k) {
    const double l1 = lm[k], l2 = lm[N + k], l3 = lm[2 * N + k];
    if (!(l1 >= 0.0) || !(l2 >= 0.0) || !(l3 >= 0.0)) st = LOMPC_ST_NEGATIVE;
    const double wk = wr[k];
    WW[k * T] = wk;
    if (!gw) continue;
    const double d = 2.0 * (lr * cs.theta2 + cs.q_scale * l3) + cs.d_base;
    const double g = gw[k];
    bool fixed = wk <= band || wk >= blo[NSEG];
#pragma unroll
    for (int j = 1; j < NSEG; ++j) fixed |= (wk >= blo[j]) && (wk <= bhi[j]);
    const double M = c + P;
    MM[k * T] = M;
    RR[k * T] = r - g;
    if (fixed) {
      IV[k * T] = 0.0;
      P = M;
    } else {
      const double iv = fast_rcp(d + M);
      IV[k * T] = iv;
      P = d * M * iv;
      r = fma(d, r, M * g) * iv;
    }
  }
  if (gam > cs.y_max) st = LOMPC_ST_BAD_GAMMA;
  if (a.status) a.status[b] = st;
  const bool ok = st == LOMPC_ST_OK;

  // ---- forward pass: z, then the gradients ---------------------------------------------------------------
  double* gl = a.grad_lmbd ? a.grad_lmbd + b * (int64_t)(3 * N) : nullptr;
  const double th = cs.theta, q = cs.q_scale;
  double sigma = 0.0, s = 0.0, zw = 0.0, zn = 0.0, ww = 0.0, ss = 0.0;
  for (int k = 0; k < N; ++k) {
    const double wk = WW[k * T];
    const double z = gw ? -fma(MM[k * T], sigma, RR[k * T]) * IV[k * T] : 0.0;
    sigma += z;
    s += wk;
    zw = fma(z, wk, zw);
    zn = fma((double)(N - k), z, zn);
    ww = fma(wk, wk, ww);
    ss += s;
    if (gl) {
      gl[k] = ok ? fma(gc * th, wk, -th * z) : 0.0;
      gl[N + k] = ok ? fma(gc * th, wmax - wk, th * z) : 0.0;
      gl[2 * N + k] = ok ? q * wk * fma(gc, wk, -2.0 * z) : 0.0;
    }
  }
  if (a.grad_lmbd_r) a.grad_lmbd_r[b] = ok ? cs.theta2 * fma(gc, ww, -2.0 * zw) : 0.0;
  if (a.grad_gamma) a.grad_gamma[b] = ok ? c * fma(-gc, ss, zn) : 0.0;
}

}  // namespace lompc
