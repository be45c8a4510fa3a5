// K6: batched upper-level BiMPC (reference chargingstation/bimpc.py:142-292), one station
// per CTA.  The convex program
//
//   min  c_g sum_k u[k]^1.7 + delta sum_q sum_k omega_k a_q (cumsum(w_q)_k - gamma_q)^2
//   s.t. 0 <= w_q <= wmax_q,  0 <= u <= u_g_max,                               (bimpc.py:143-186)
//        v = u - demand - sum_q m_q w_q,   |v -+ d e1| <= u_b_max,             (bimpc.py:188-203)
//        d <= x0 + cumsum(v) <= x_max - d                                      (bimpc.py:205-218)
//
// (q = 0..2P-1: P small-EV then P large-EV partitions, m_q = theta_q Mp_q) is solved with a
// Mehrotra predictor-corrector interior-point method (cvxpy hands the same program to
// CLARABEL's interior point, bimpc.py:114,287).  The (2P+1)N x (2P+1)N Newton matrix
//     K = diag(E) + blockdiag_q(A' D_q A) + Ub' (diag(D1) + A' diag(D2) A) Ub,
//     A = tril(ones),  Ub = [-m_0 I .. -m_{2P-1} I,  I]
// is dense, but in CUMULATIVE coordinates xi_k = (cumsum(w_0)_k .. cumsum(w_{2P-1})_k, cumsum(u)_k)
// (the MPC states: energy delivered per partition and generated so far) it is block
// TRIDIAGONAL over the horizon with (2P+1) x (2P+1) blocks
//     Diag_k = diag(E_k + E_{k+1} + D_k) + (D2_k + D1_k + D1_{k+1}) a a',   a = (-m, 1)
//     Off_k  = -diag(E_k) - D1_k a a'
// and is factorised by a block Cholesky sweep over the stages (backward stable: with the
// reference's exponential stage weights 5^(k-N+1) the blocks H_q span 11 decades and a
// Woodbury / dual-decomposition solve through H_q^{-1} loses the Newton direction).  Only the
// inverse triangular factors of the diagonal blocks are stored (packed); the off-diagonal
// blocks are diagonal + rank one and are applied on the fly.
//
// The body is written as thread-strided loops separated by block barriers and uses no warp
// intrinsics, so that tests/hostsim can compile this very file for the host with one
// "thread" (BIMPC_HOSTSIM) and check the algorithm against the dense oracle without a GPU.
#pragma once
#include <math.h>
#include <stdint.h>
#ifdef BIMPC_TRACE
#include <stdio.h>
#endif

#ifdef BIMPC_HOSTSIM
#define BI_FN inline
#define BI_HD inline
#define BI_SYNC() ((void)0)
#define BI_SUBSUM(v, nsub) ((void)0)
#define BI_RCP(x) (1.0 / (x))
#else
#define BI_FN __device__ __forceinline__
#define BI_HD __host__ __device__ inline
#define BI_SYNC() __syncthreads()
#define BI_RCP(x) bimpc::fast_rcp_dev(x)
// sum over the `nsub` (1 or 4) adjacent lanes that share one matrix row
#define BI_SUBSUM(v, nsub)                        \
  do {                                            \
    if ((nsub) == 4) {                            \
      v += __shfl_xor_sync(0xffffffffu, v, 1);    \
      v += __shfl_xor_sync(0xffffffffu, v, 2);    \
    }                                             \
  } while (0)
#endif

#if defined(BIMPC_PROFILE) && !defined(BIMPC_HOSTSIM)
#define BI_TIC(slot) long long bi_t_##slot = clock64()
#define BI_TOC(slot) if (tid == 0) a.prof[slot] += clock64() - bi_t_##slot
#else
#define BI_TIC(slot) ((void)0)
#define BI_TOC(slot) ((void)0)
#endif

namespace bimpc {

#ifndef BIMPC_HOSTSIM
// reciprocal of a positive, well-scaled double: MUFU seed + one cubic Newton step (~1 ulp)
__device__ __forceinline__ double fast_rcp_dev(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double e = fma(-x, y, 1.0);
  const double t = fma(e, e, e);
  return fma(y, t, y);
}
#endif

#ifndef BIMPC_THREADS
#define BIMPC_THREADS 128
#endif
// Stations per SM: the kernel hides the latency of its dependent, barrier-separated steps only by the number of
// resident WARPS.  Measured on the BiMPC phase of a 4,096-station closed-loop step (round 2): 3 stations x 128 threads
// (166 registers, all state in shared memory) 47.3 ms; 4 x 128 (register cap 128: no spills; 5 of the 9 state
// vectors in global scratch so that 4 x 52 KB fit) 38.6 ms; 5 x 128 (96 registers, 16 B of spills, 7 vectors) 38.5 ms;
// 6 x 128 (80 registers, 48 B of spills, all 9) 48.4 ms.  Fewer threads per station at the same number of warps per
// SM (4 x 96, 5 x 64, 6 x 64) changes nothing (48.3 / 48.7 / 48.9 ms).
#ifndef BIMPC_MINB
#define BIMPC_MINB 4
#endif
#ifndef BIMPC_GVEC
#define BIMPC_GVEC 5
#endif
constexpr int kThreads = BIMPC_THREADS;  // threads per station
constexpr int kMinBlocks = BIMPC_MINB;   // stations per SM the register allocation is asked to allow
// Of the nine [2P, N] vectors of a station's state (iterate, slacks, multipliers, residual, directions, barrier
// diagonal) the last kGlobalVecs live in the CTA's global scratch (L2-resident, touched by thread-strided loops only)
// instead of shared memory, so that more stations share an SM.
constexpr int kGlobalVecs = BIMPC_GVEC;
constexpr int kMaxN = 48;  // horizon cap (scratch of one station must fit 227 KB of shared memory)

struct BiConsts {
  int N, P;
  double delta, c_g, u_g_max, u_b_max, x_max;
  int cost_type;  // 0 WEIGHTED, 1 UNWEIGHTED, 2 EXP_UNWEIGHTED (bimpc.py:12-15)
  double theta_s, theta_l, w_max_s, w_max_l;
};

struct BiArgs {
  int S;                  // stations
  const double* omega;    // [N] stage weights of the charging cost (bimpc.py:255-257)
  const double* Mp_s;     // [S,P] normalised partition sizes (BiMPCParameters, bimpc.py:44-58)
  const double* Mp_l;
  const double* beta_s;   // [S,P]
  const double* beta_l;
  const double* gamma_sm; // [S,P]
  const double* gamma_lm;
  const double* x0;       // [S]
  const double* demand;   // [S,N]
  double* w_hat_s;        // [S,P,N]
  double* w_hat_l;        // [S,P,N]
  double* u_g;            // [S,N]
  int32_t* status;        // [S] 0 ok, 1 iteration cap, 2 numerical breakdown
  int32_t* iters;         // [S]
  double* objective;      // [S] or NULL
  double tol;
  int max_iter;
  long long* prof;        // BIMPC_PROFILE builds only: cycle counters
  double* li_scratch;     // [CTAs, global_scratch_doubles()] packed inverse factors of the diagonal blocks [+ state
                          // vectors] (global memory, L2-resident: keeping them out of shared memory lets several
                          // stations share an SM)
};

// Doubles of per-CTA global scratch: the packed inverse factors of the N diagonal blocks + the state vectors that are
// kept out of shared memory.
BI_HD size_t global_scratch_doubles(int N, int P) {
  const size_t nb = 2 * (size_t)P + 1;
  return (size_t)N * (nb * (nb + 1) / 2) + (size_t)kGlobalVecs * 2 * P * N;
}

// Number of doubles of scratch one station needs (shared memory on the device).
BI_HD size_t scratch_doubles(int N, int P, int T) {
  const int Q2 = 2 * P, QN = Q2 * N, nb = Q2 + 1;
  return (size_t)(9 - kGlobalVecs) * QN + (size_t)(QN + N) + 2 * (size_t)(nb * (nb + 1) / 2) + 2 * (size_t)nb * nb +
         (size_t)40 * N + 8 * (size_t)nb + 3 * (size_t)T + 5 * Q2 + 16;
}

// Deterministic block reduction of (sum, max, min): partials in tid order.
BI_FN void block_reduce(double* RED, int tid, int T, double& sum, double& mx, double& mn) {
  RED[tid] = sum;
  RED[T + tid] = mx;
  RED[2 * T + tid] = mn;
  BI_SYNC();
#ifndef BIMPC_HOSTSIM
  // Every thread needs the three results; computing them once per thread cost 8 % of the kernel's instructions at fleet
  // scale (ncu, round 2).  Per WARP instead: lane 0 runs the ordered sum (same additions in the same order - the
  // result does not change) and broadcasts it; maximum and minimum do not depend on the order and are folded by shuffles.
  const unsigned full = 0xffffffffu;
  const int lane = tid & 31;
  double s = 0.0;
  if (lane == 0)
    for (int i = 0; i < T; ++i) s += RED[i];
  s = __shfl_sync(full, s, 0);
  double a = RED[T + lane], b = RED[2 * T + lane];
  for (int i = lane + 32; i < T; i += 32) {
    a = fmax(a, RED[T + i]);
    b = fmin(b, RED[2 * T + i]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    a = fmax(a, __shfl_xor_sync(full, a, o));
    b = fmin(b, __shfl_xor_sync(full, b, o));
  }
#else
  double s = 0.0, a = RED[T], b = RED[2 * T];
  for (int i = 0; i < T; ++i) {
    s += RED[i];
    a = fmax(a, RED[T + i]);
    b = fmin(b, RED[2 * T + i]);
  }
#endif
  BI_SYNC();
  sum = s;
  mx = a;
  mn = b;
}

// Partial dot products on a packed lower-triangular matrix L (row i starts at i(i+1)/2): the
// `nsub` lanes that share row i take the terms part, part + nsub, ... and are summed with
// BI_SUBSUM.  row: sum_{j<=i} L[i][j] x[j];   col: sum_{l>=i} L[l][i] x[l].
BI_FN double row_part(const double* L, int i, const double* x, int part, int nsub) {
  const double* r = L + i * (i + 1) / 2;
  double a0 = 0.0, a1 = 0.0;
  int j = part;
  for (; j + nsub <= i; j += 2 * nsub) {
    a0 += r[j] * x[j];
    a1 += r[j + nsub] * x[j + nsub];
  }
  if (j <= i) a0 += r[j] * x[j];
  return a0 + a1;
}
BI_FN double col_part(const double* L, int i, int nb, const double* x, int part, int nsub) {
  double a0 = 0.0, a1 = 0.0;
  int l = i + part;
  for (; l + nsub < nb; l += 2 * nsub) {
    a0 += L[l * (l + 1) / 2 + i] * x[l];
    a1 += L[(l + nsub) * (l + nsub + 1) / 2 + i] * x[l + nsub];
  }
  if (l < nb) a0 += L[l * (l + 1) / 2 + i] * x[l];
  return a0 + a1;
}
BI_FN double vec_dot(const double* a, const double* b, int n) {
#ifndef BIMPC_HOSTSIM
  // The same four accumulator chains and the same final additions as the loop below (same bits), formed once per
  // WARP - lanes 0-3 run one chain each - instead of once per thread: every thread of the CTA needs the value, and
  // 128 copies of a 25-term dot product were 16 % of the kernel's instructions at fleet scale (ncu, round 2).
  // Every lane of the warp must call.
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  double acc = 0.0;
  if (lane < 4) {
    const int n4 = n & ~3;
    for (int j = lane; j < n4; j += 4) acc = fma(a[j], b[j], acc);
    if (lane == 0)
      for (int j = n4; j < n; ++j) acc = fma(a[j], b[j], acc);
  }
  const double pr = acc + __shfl_down_sync(full, acc, 1);  // lane 0: a0 + a1, lane 2: a2 + a3
  const double r = pr + __shfl_down_sync(full, pr, 2);     // lane 0: (a0 + a1) + (a2 + a3)
  return __shfl_sync(full, r, 0);
#else
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  int j = 0;
  for (; j + 3 < n; j += 4) {
    a0 += a[j] * b[j];
    a1 += a[j + 1] * b[j + 1];
    a2 += a[j + 2] * b[j + 2];
    a3 += a[j + 3] * b[j + 3];
  }
  for (; j < n; ++j) a0 += a[j] * b[j];
  return (a0 + a1) + (a2 + a3);
#endif
}

// One station.  `sm` = scratch_doubles(N, P, T) doubles private to this CTA.
BI_FN void solve_station(const BiConsts& c, const BiArgs& a, int st_idx, double* sm, double* LI, int tid, int T) {
  const int N = c.N, P = c.P;
  // all 2P partition blocks size the scratch; the loops run over the ACTIVE ones only (see below)
  const int Q2max = 2 * P, QNmax = Q2max * N, nbmax = Q2max + 1, npmax = nbmax * (nbmax + 1) / 2;
  // matrix-vector products: `nsub` adjacent lanes share one row (T >= 128), else one thread per row
  const int nsub = (T >= 128) ? 4 : 1, row = tid / nsub, part = tid - row * nsub, rows_pp = T / nsub;
  // dense block operations: thread (tx, ty) = (column, row group)
  const int nx = T < 32 ? T : 32, tx = tid % nx, ty = tid / nx, ny = T / nx;
  // ---- carve
  // the nine [Q2,N] state vectors: slot v < 9 - kGlobalVecs in shared memory, the others in the CTA's global scratch
  // (behind the inverse factors); ordered so that the ones the factorisation and the solves read stay on chip
  double* gvec = LI + (size_t)N * npmax;
  auto vec_at = [&](int v) {
    return v < 9 - kGlobalVecs ? sm + (size_t)v * QNmax : gvec + (size_t)(v - (9 - kGlobalVecs)) * QNmax;
  };
  double* EW = vec_at(0);        // barrier diagonal z1/s1 + z2/s2
  double* DX = vec_at(1);        // Newton right-hand side, then the current direction, w block
  double* W = vec_at(2);         // [Q2,N] iterate
  double* S1 = vec_at(3);        // slack / multiplier of w >= 0
  double* Z1 = vec_at(4);
  double* S2 = vec_at(5);        // slack / multiplier of w <= wmax
  double* Z2 = vec_at(6);
  double* DXA = vec_at(7);       // affine direction, w block
  double* RDW = vec_at(8);       // dual residual, w block
  double* XI = sm + (size_t)(9 - kGlobalVecs) * QNmax;  // [N,nb] block-tridiagonal solve vector (cumulative coordinates)
  double* LPS = XI + QNmax + N;  // [2,np] shared-memory copy of the inverse factor of the last two stages
  double* SW = LPS + 2 * (size_t)npmax;  // [nb,nb] Schur complement of the current stage
  double* XW = SW + nbmax * nbmax;  // [nb,nb] the identity the elimination turns into the inverse factor
  double* pk = XW + nbmax * nbmax;  // per-k vectors
  double* U = pk;             pk += N;
  double* S3 = pk;            pk += N;
  double* Z3 = pk;            pk += N;
  double* S4 = pk;            pk += N;
  double* Z4 = pk;            pk += N;
  double* S5 = pk;            pk += N;
  double* Z5 = pk;            pk += N;
  double* S6 = pk;            pk += N;
  double* Z6 = pk;            pk += N;
  double* S7 = pk;            pk += N;
  double* Z7 = pk;            pk += N;
  double* S8 = pk;            pk += N;
  double* Z8 = pk;            pk += N;
  double* V = pk;             pk += N;  // u_b
  double* XX = pk;            pk += N;  // battery state
  double* RDU = pk;           pk += N;
  double* HU = pk;            pk += N;
  double* D1 = pk;            pk += N;
  double* D2 = pk;            pk += N;
  double* BU = pk;            pk += N;  // right-hand side, then the current direction, u block
  double* DXUA = pk;          pk += N;
  double* DV = pk;            pk += N;
  double* DVA = pk;           pk += N;
  double* DXX = pk;           pk += N;
  double* DXXA = pk;          pk += N;
  double* NU = pk;            pk += N;
  double* YV = pk;            pk += N;
  double* T56 = pk;           pk += N;
  double* T78 = pk;           pk += N;
  double* DEM = pk;           pk += N;
  double* OM = pk;            pk += N;
  pk += 9 * N;                          // (spare, keeps the 40 N budget)
  double* AV = pk;            pk += nbmax;  // a = (-m, 1)
  double* LA = pk;            pk += nbmax;  // Linv_{k-1} a
  double* TL = pk;            pk += nbmax;  // T' la
  pk += nbmax;
  double* TV1 = pk;           pk += nbmax;
  double* TV2 = pk;           pk += nbmax;
  pk += 2 * nbmax;
  double* RED = pk;           pk += 3 * T;
  double* MQ = pk;            pk += Q2max;   // m_q
  double* AQ = pk;            pk += Q2max;   // a_q
  double* GQ = pk;            pk += Q2max;   // gamma_q
  double* WMX = pk;           pk += Q2max;   // wmax_q
  double* QIDX = pk;          pk += Q2max;   // active block -> partition index (small P, then large P)

  // ---- station data
  const double x0 = a.x0[st_idx];
  // d = theta_s (Mp_s . beta_s) + theta_l (Mp_l . beta_l)   (bimpc.py:195-197); every thread
  // evaluates the scalar itself, in the same order
  double dot_s = 0.0, dot_l = 0.0;
  for (int p = 0; p < P; ++p) {
    dot_s += a.Mp_s[(size_t)st_idx * P + p] * a.beta_s[(size_t)st_idx * P + p];
    dot_l += a.Mp_l[(size_t)st_idx * P + p] * a.beta_l[(size_t)st_idx * P + p];
  }
  const double derr = c.theta_s * dot_s + c.theta_l * dot_l;
  // A partition with no EVs (m_q = 0) and nothing to track (gamma_q = 0, or zero cost weight) is
  // decoupled from the rest of the program and its optimum is w_q = 0: it is left out of the
  // Newton system (the block size 2P+1 shrinks to active+1; early in a simulation only a third
  // of the partitions is populated).  Thread 0 builds the compact list.
  // It also checks that every input is finite: a NaN drops out of the fmax / fmin of the residual maxima and the
  // ratio test, and a partition left out here is never read again, so a non-finite input could otherwise come back
  // as a converged solve.  Such a station gets status 2.
  if (tid == 0) {
    int cnt = 0;
    bool finite = isfinite(x0) && isfinite(derr);  // derr: every Mp and beta
    for (int k = 0; k < N; ++k) finite = finite && isfinite(a.demand[(size_t)st_idx * N + k]);
    for (int q = 0; q < Q2max; ++q) {
      const bool small = q < P;
      const int p = small ? q : q - P;
      const double mp = small ? a.Mp_s[(size_t)st_idx * P + p] : a.Mp_l[(size_t)st_idx * P + p];
      const double th = small ? c.theta_s : c.theta_l;
      const double gq = small ? a.gamma_sm[(size_t)st_idx * P + p] : a.gamma_lm[(size_t)st_idx * P + p];
      const double aq = c.cost_type == 0 ? (th * mp) * (th * mp) : 1.0;
      finite = finite && isfinite(gq);
      if (th * mp == 0.0 && (gq == 0.0 || aq == 0.0)) continue;
      MQ[cnt] = th * mp;
      AQ[cnt] = aq;
      GQ[cnt] = gq;
      WMX[cnt] = small ? c.w_max_s : c.w_max_l;
      AV[cnt] = -th * mp;
      QIDX[cnt] = (double)q;
      ++cnt;
    }
    AV[cnt] = 1.0;
    RED[0] = (double)cnt;
    RED[1] = finite ? 1.0 : 0.0;
  }
  BI_SYNC();
  const int Q2 = (int)RED[0], QN = Q2 * N, nb = Q2 + 1, np = nb * (nb + 1) / 2;
  const bool finite_in = RED[1] != 0.0;
  BI_SYNC();
  for (int k = tid; k < N; k += T) {
    DEM[k] = a.demand[(size_t)st_idx * N + k];
    OM[k] = a.omega[k];
  }
  BI_SYNC();
  double om_sum = 0.0;
  for (int k = 0; k < N; ++k) om_sum += OM[k];
  double scale_g = 1.0;
  for (int q = 0; q < Q2; ++q) scale_g = fmax(scale_g, 2.0 * c.delta * AQ[q] * fabs(GQ[q]) * om_sum);
  const double mtot = (double)(2 * QN + 6 * N);

  // ---- starting point: box centre, slacks max(h - Gx, 1e-2), multipliers 1
  for (int i = tid; i < QN; i += T) {
    const int q = i / N;
    W[i] = 0.5 * WMX[q];
    S1[i] = fmax(0.5 * WMX[q], 1e-2);
    S2[i] = fmax(0.5 * WMX[q], 1e-2);
    Z1[i] = 1.0;
    Z2[i] = 1.0;
  }
  for (int k = tid; k < N; k += T) {
    U[k] = 0.5 * c.u_g_max;
    S3[k] = fmax(0.5 * c.u_g_max, 1e-2);
    S4[k] = fmax(0.5 * c.u_g_max, 1e-2);
    Z3[k] = Z4[k] = Z5[k] = Z6[k] = Z7[k] = Z8[k] = 1.0;
  }
  BI_SYNC();
  for (int k = tid; k < N; k += T) {
    double v = U[k] - DEM[k];
    for (int q = 0; q < Q2; ++q) v -= MQ[q] * W[q * N + k];
    V[k] = v;
  }
  BI_SYNC();
  for (int k = tid; k < N; k += T) {
    double x = x0;
    for (int j = 0; j <= k; ++j) x += V[j];
    const double e1 = (k == 0) ? derr : 0.0;
    S5[k] = fmax(V[k] + c.u_b_max - e1, 1e-2);
    S6[k] = fmax(c.u_b_max - e1 - V[k], 1e-2);
    S7[k] = fmax(x - derr, 1e-2);
    S8[k] = fmax(c.x_max - derr - x, 1e-2);
  }
  BI_SYNC();

  int it = 0, status = 1;
  double mu = 0.0;
  for (;; ++it) {
    if (!finite_in) {
      status = 2;
      break;
    }
    BI_TIC(0);
    // ---- A. primal quantities and the gradient of the charging cost
    for (int q = tid; q < Q2; q += T) {
      // grad_q = 2 delta a_q A' (omega .* (A w_q - gamma_q)):  forward cumsum, then reverse
      double s = 0.0;
      for (int k = 0; k < N; ++k) {
        s += W[q * N + k];
        RDW[q * N + k] = OM[k] * (s - GQ[q]);
      }
      double r = 0.0;
      const double f = 2.0 * c.delta * AQ[q];
      for (int k = N - 1; k >= 0; --k) {
        r += RDW[q * N + k];
        RDW[q * N + k] = f * r;
      }
    }
    for (int k = tid; k < N; k += T) {
      double v = U[k] - DEM[k];
      for (int q = 0; q < Q2; ++q) v -= MQ[q] * W[q * N + k];
      V[k] = v;
      T56[k] = Z6[k] - Z5[k];
      T78[k] = Z8[k] - Z7[k];
    }
    BI_SYNC();
    for (int k = tid; k < N; k += T) {
      double x = x0;
      for (int j = 0; j <= k; ++j) x += V[j];
      XX[k] = x;
      double y = T56[k];
      for (int j = N - 1; j >= k; --j) y += T78[j];
      YV[k] = y;
    }
    BI_SYNC();
    // ---- B. residuals
    double r_sz = 0.0, r_max = 0.0, r_dummy = 0.0, rp_max = 0.0;
    for (int i = tid; i < QN; i += T) {
      const int q = i / N, k = i - q * N;
      const double rd = RDW[i] - Z1[i] + Z2[i] - MQ[q] * YV[k];
      RDW[i] = rd;
      r_max = fmax(r_max, fabs(rd));
      rp_max = fmax(rp_max, fmax(fabs(S1[i] - W[i]), fabs(W[i] + S2[i] - WMX[q])));
      r_sz += S1[i] * Z1[i] + S2[i] * Z2[i];
    }
    for (int k = tid; k < N; k += T) {
      const double u = fmax(U[k], 1e-300);
      const double rd = 1.7 * c.c_g * pow(u, 0.7) - Z3[k] + Z4[k] + YV[k];
      RDU[k] = rd;
      r_max = fmax(r_max, fabs(rd));
      const double e1 = (k == 0) ? derr : 0.0;
      double m = fmax(fabs(S3[k] - U[k]), fabs(U[k] + S4[k] - c.u_g_max));
      m = fmax(m, fabs(-V[k] + S5[k] - (c.u_b_max - e1)));
      m = fmax(m, fabs(V[k] + S6[k] - (c.u_b_max - e1)));
      m = fmax(m, fabs(-XX[k] + S7[k] + derr));
      m = fmax(m, fabs(XX[k] + S8[k] - (c.x_max - derr)));
      rp_max = fmax(rp_max, m);
      r_sz += S3[k] * Z3[k] + S4[k] * Z4[k] + S5[k] * Z5[k] + S6[k] * Z6[k] + S7[k] * Z7[k] + S8[k] * Z8[k];
    }
    // two maxima travel through one reduction: (sum, max, min) = (s'z, max|rd|, -max|rp|)
    r_dummy = -rp_max;
    block_reduce(RED, tid, T, r_sz, r_max, r_dummy);
    rp_max = -r_dummy;
    mu = r_sz / mtot;
#ifdef BIMPC_TRACE
    printf("it %d rd %.3e rp %.3e mu %.3e\n", it, r_max, rp_max, mu);
#endif
    if (r_max <= a.tol * scale_g && rp_max <= a.tol && mu <= a.tol) {
      status = 0;
      break;
    }
    if (it >= a.max_iter) break;
    if (!(mu == mu) || !(r_max == r_max)) {  // NaN
      status = 2;
      break;
    }

    BI_TOC(0);
    BI_TIC(1);
    // ---- C. factorisation: block Cholesky of the stage-ordered Newton matrix
    for (int i = tid; i < QN; i += T) EW[i] = Z1[i] / S1[i] + Z2[i] / S2[i];
    for (int k = tid; k < N; k += T) {
      const double u = fmax(U[k], 1e-300);
      HU[k] = 1.7 * 0.7 * c.c_g * pow(u, -0.3) + Z3[k] / S3[k] + Z4[k] / S4[k];
      D1[k] = Z5[k] / S5[k] + Z6[k] / S6[k];
      D2[k] = Z7[k] / S7[k] + Z8[k] / S8[k];
    }
    BI_SYNC();
    // E_k[i]: barrier diagonal of stage k in block order (partitions, then u)
    auto Ek = [&](int k, int i) { return k >= N ? 0.0 : (i < Q2 ? EW[i * N + k] : HU[k]); };
    bool ok = true;
    for (int k = 0; k < N; ++k) {
      const double* Lp = LPS + (size_t)((k - 1) & 1) * np;  // previous stage (k >= 1), shared-memory copy
      const double d1k = D1[k], d1n = (k + 1 < N) ? D1[k + 1] : 0.0;
      BI_TIC(4);
      if (k >= 1) {
        for (int i0 = 0; i0 < nb; i0 += rows_pp) {  // la = Linv_{k-1} a
          const int i = i0 + row;
          double v = (i < nb) ? row_part(Lp, i, AV, part, nsub) : 0.0;
          BI_SUBSUM(v, nsub);
          if (i < nb && part == 0) LA[i] = v;
        }
        BI_SYNC();
        for (int i0 = 0; i0 < nb; i0 += rows_pp) {  // tl = T' la,  T = Linv_{k-1} diag(E_k)
          const int i = i0 + row;
          double v = (i < nb) ? col_part(Lp, i, nb, LA, part, nsub) : 0.0;
          BI_SUBSUM(v, nsub);
          if (i < nb && part == 0) TL[i] = v * Ek(k, i);
        }
        BI_SYNC();
      }
      BI_TOC(4);
      BI_TIC(5);
      const double ll = (k >= 1) ? vec_dot(LA, LA, nb) : 0.0;
      const double rho = D2[k] + d1k + d1n;
      // Schur complement S_k = Diag_k - Off_k Linv' Linv Off_k (full symmetric storage) and X = I;
      // thread (tx, ty): column tx (+32, ...), rows ty, ty + ny, ...
      for (int i = ty; i < nb; i += ny) {
        const double eki = Ek(k, i), di = d1k * AV[i];
        for (int j = tx; j < nb; j += nx) {
          XW[i * nb + j] = (i == j) ? 1.0 : 0.0;
          if (j > i) continue;
          double v = rho * AV[i] * AV[j];
          if (i == j) v += eki + Ek(k + 1, i) + (i < Q2 ? 2.0 * c.delta * AQ[i] * OM[k] : 0.0);
          if (k >= 1) {
            double t0 = 0.0, t1 = 0.0;  // (Linv' Linv)[i][j], i >= j
            int l = i, o = i * (i + 1) / 2;
            for (; l + 1 < nb; l += 2) {
              t0 += Lp[o + i] * Lp[o + j];
              o += l + 1;
              t1 += Lp[o + i] * Lp[o + j];
              o += l + 2;
            }
            if (l < nb) t0 += Lp[o + i] * Lp[o + j];
            const double tt = (t0 + t1) * (eki * Ek(k, j));
            const double dj = d1k * AV[j];
            v -= tt + TL[i] * dj + di * TL[j] + ll * di * dj;
          }
          SW[i * nb + j] = v;
          SW[j * nb + i] = v;
        }
      }
      BI_SYNC();
      BI_TOC(5);
      BI_TIC(6);
      // Gaussian elimination of [S | I] without pivoting (S is SPD): the row operations that
      // triangularise S turn I into the unit-lower inverse factor; scaling row i by
      // 1/sqrt(pivot_i) gives Linv = chol(S)^{-1}.  One barrier per pivot; in step j thread
      // (tx, ty) updates column tx of rows j+1+ty, j+1+ty+ny, ... (columns <= j belong to X,
      // the others to S).
      for (int j = 0; j < nb; ++j) {
        const double piv = SW[j * nb + j];
        if (!(piv > 0.0)) ok = false;
        const double rp = BI_RCP(piv > 0.0 ? piv : 1.0);
        for (int cidx = tx; cidx < nb; cidx += nx) {
          double* M = (cidx <= j) ? XW : SW;
          const double pr = M[j * nb + cidx];
          for (int i = j + 1 + ty; i < nb; i += ny) M[i * nb + cidx] -= (SW[i * nb + j] * rp) * pr;
        }
        BI_SYNC();
      }
      BI_TOC(6);
      BI_TIC(7);
      for (int i = tid; i < nb; i += T) TV1[i] = 1.0 / sqrt(SW[i * nb + i]);
      BI_SYNC();
      double* Lk = LI + (size_t)k * np;
      double* Lks = LPS + (size_t)(k & 1) * np;
      for (int i = ty; i < nb; i += ny) {
        const double rs = TV1[i];
        for (int j = tx; j <= i; j += nx) {
          const double v = XW[i * nb + j] * rs;
          Lk[i * (i + 1) / 2 + j] = v;
          Lks[i * (i + 1) / 2 + j] = v;
        }
      }
      BI_SYNC();
      BI_TOC(7);
    }
    if (!ok) {
      status = 2;
      break;
    }

    BI_TOC(1);
    // (outW, outU) = K^{-1} (inW, inU) through the block factorisation; in and out may alias.
    auto lin_solve = [&](const double* inW, const double* inU, double* outW, double* outU) {
      // right-hand side in cumulative coordinates: b~_k = b_k - b_{k+1}
      for (int e = tid; e < N * nb; e += T) {
        const int k = e / nb, i = e - k * nb;
        const double b0 = i < Q2 ? inW[i * N + k] : inU[k];
        const double b1 = (k + 1 < N) ? (i < Q2 ? inW[i * N + k + 1] : inU[k + 1]) : 0.0;
        XI[e] = b0 - b1;
      }
      BI_SYNC();
      // forward: y_k = Linv_k (b~_k - Off_k Linv_{k-1}' y_{k-1})
      for (int k = 0; k < N; ++k) {
        double* x = XI + k * nb;
        if (k >= 1) {
          const double* Lp = LI + (size_t)(k - 1) * np;
          const double* yp = XI + (k - 1) * nb;
          for (int i0 = 0; i0 < nb; i0 += rows_pp) {
            const int i = i0 + row;
            double v = (i < nb) ? col_part(Lp, i, nb, yp, part, nsub) : 0.0;
            BI_SUBSUM(v, nsub);
            if (i < nb && part == 0) TV1[i] = v;
          }
          BI_SYNC();
          const double at = vec_dot(AV, TV1, nb);
          for (int i = tid; i < nb; i += T) TV2[i] = x[i] + Ek(k, i) * TV1[i] + D1[k] * AV[i] * at;
        } else {
          for (int i = tid; i < nb; i += T) TV2[i] = x[i];
        }
        BI_SYNC();
        const double* Lk = LI + (size_t)k * np;
        for (int i0 = 0; i0 < nb; i0 += rows_pp) {
          const int i = i0 + row;
          double v = (i < nb) ? row_part(Lk, i, TV2, part, nsub) : 0.0;
          BI_SUBSUM(v, nsub);
          if (i < nb && part == 0) x[i] = v;
        }
        BI_SYNC();
      }
      // backward: xi_k = Linv_k' (y_k - Linv_k Off_{k+1} xi_{k+1})
      for (int k = N - 1; k >= 0; --k) {
        double* x = XI + k * nb;
        const double* Lk = LI + (size_t)k * np;
        if (k + 1 < N) {
          const double* xn = XI + (k + 1) * nb;
          const double ax = vec_dot(AV, xn, nb);
          for (int i = tid; i < nb; i += T) TV1[i] = -(Ek(k + 1, i) * xn[i] + D1[k + 1] * AV[i] * ax);
          BI_SYNC();
          for (int i0 = 0; i0 < nb; i0 += rows_pp) {
            const int i = i0 + row;
            double v = (i < nb) ? row_part(Lk, i, TV1, part, nsub) : 0.0;
            BI_SUBSUM(v, nsub);
            if (i < nb && part == 0) TV2[i] = x[i] - v;
          }
        } else {
          for (int i = tid; i < nb; i += T) TV2[i] = x[i];
        }
        BI_SYNC();
        for (int i0 = 0; i0 < nb; i0 += rows_pp) {
          const int i = i0 + row;
          double v = (i < nb) ? col_part(Lk, i, nb, TV2, part, nsub) : 0.0;
          BI_SUBSUM(v, nsub);
          if (i < nb && part == 0) x[i] = v;
        }
        BI_SYNC();
      }
      // back to stage increments: dx_k = xi_k - xi_{k-1}
      for (int e = tid; e < N * nb; e += T) {
        const int k = e / nb, i = e - k * nb;
        const double v = XI[e] - (k >= 1 ? XI[e - nb] : 0.0);
        if (i < Q2) outW[i * N + k] = v;
        else outU[k] = v;
      }
      BI_SYNC();
    };

    BI_TIC(3);
    // ---- D..G: predictor (pass 0) and corrector (pass 1)
    double sigma_mu = 0.0, alpha = 1.0;
    for (int pass = 0; pass < 2; ++pass) {
      // complementarity target rc_i = s z [+ ds_a dz_a - sigma mu]; xi_i = (z rp - rc)/s
      auto rc_of = [&](double s, double z, double rp, double ga) {
        double rc = s * z;
        if (pass == 1) {
          const double dsa = -rp - ga;
          const double dza = (-s * z - z * dsa) / s;
          rc += dsa * dza - sigma_mu;
        }
        return rc;
      };
      for (int k = tid; k < N; k += T) {
        const double e1 = (k == 0) ? derr : 0.0;
        const double rp5 = -V[k] + S5[k] - (c.u_b_max - e1), rp6 = V[k] + S6[k] - (c.u_b_max - e1);
        const double rp7 = -XX[k] + S7[k] + derr, rp8 = XX[k] + S8[k] - (c.x_max - derr);
        const double x5 = (Z5[k] * rp5 - rc_of(S5[k], Z5[k], rp5, -DVA[k])) / S5[k];
        const double x6 = (Z6[k] * rp6 - rc_of(S6[k], Z6[k], rp6, DVA[k])) / S6[k];
        const double x7 = (Z7[k] * rp7 - rc_of(S7[k], Z7[k], rp7, -DXXA[k])) / S7[k];
        const double x8 = (Z8[k] * rp8 - rc_of(S8[k], Z8[k], rp8, DXXA[k])) / S8[k];
        T56[k] = x6 - x5;
        T78[k] = x8 - x7;
      }
      BI_SYNC();
      for (int k = tid; k < N; k += T) {
        double y = T56[k];
        for (int j = N - 1; j >= k; --j) y += T78[j];
        NU[k] = y;  // y_xi (NU is free until tau has been formed)
      }
      BI_SYNC();
      for (int i = tid; i < QN; i += T) {
        const int q = i / N, k = i - q * N;
        const double rp1 = S1[i] - W[i], rp2 = W[i] + S2[i] - WMX[q];
        const double x1 = (Z1[i] * rp1 - rc_of(S1[i], Z1[i], rp1, -DXA[i])) / S1[i];
        const double x2 = (Z2[i] * rp2 - rc_of(S2[i], Z2[i], rp2, DXA[i])) / S2[i];
        DX[i] = -RDW[i] + x1 - x2 + MQ[q] * NU[k];
      }
      for (int k = tid; k < N; k += T) {
        const double rp3 = S3[k] - U[k], rp4 = U[k] + S4[k] - c.u_g_max;
        const double x3 = (Z3[k] * rp3 - rc_of(S3[k], Z3[k], rp3, -DXUA[k])) / S3[k];
        const double x4 = (Z4[k] * rp4 - rc_of(S4[k], Z4[k], rp4, DXUA[k])) / S4[k];
        BU[k] = -RDU[k] + x3 - x4 - NU[k];
      }
      BI_SYNC();
      // dx = K^{-1} b (in place; the block Cholesky is backward stable, no refinement needed)
      BI_TIC(2);
      lin_solve(DX, BU, DX, BU);
      BI_TOC(2);
      for (int k = tid; k < N; k += T) {
        double v = BU[k];
        for (int q = 0; q < Q2; ++q) v -= MQ[q] * DX[q * N + k];
        DV[k] = v;
      }
      BI_SYNC();
      for (int k = tid; k < N; k += T) {
        double x = 0.0;
        for (int j = 0; j <= k; ++j) x += DV[j];
        DXX[k] = x;
      }
      BI_SYNC();
      // ---- ratio test (and, on the predictor pass, mu_aff)
      double amin = 1e300, dummy_s = 0.0, dummy_m = 0.0;
      auto ratio = [&](double s, double z, double rp, double g, double ga) {
        const double rc = rc_of(s, z, rp, ga);
        const double ds = -rp - g;
        const double dz = (-rc - z * ds) / s;
        if (ds < 0.0) amin = fmin(amin, -s / ds);
        if (dz < 0.0) amin = fmin(amin, -z / dz);
      };
      for (int i = tid; i < QN; i += T) {
        const int q = i / N;
        const double rp1 = S1[i] - W[i], rp2 = W[i] + S2[i] - WMX[q];
        ratio(S1[i], Z1[i], rp1, -DX[i], -DXA[i]);
        ratio(S2[i], Z2[i], rp2, DX[i], DXA[i]);
      }
      for (int k = tid; k < N; k += T) {
        const double e1 = (k == 0) ? derr : 0.0;
        ratio(S3[k], Z3[k], S3[k] - U[k], -BU[k], -DXUA[k]);
        ratio(S4[k], Z4[k], U[k] + S4[k] - c.u_g_max, BU[k], DXUA[k]);
        ratio(S5[k], Z5[k], -V[k] + S5[k] - (c.u_b_max - e1), -DV[k], -DVA[k]);
        ratio(S6[k], Z6[k], V[k] + S6[k] - (c.u_b_max - e1), DV[k], DVA[k]);
        ratio(S7[k], Z7[k], -XX[k] + S7[k] + derr, -DXX[k], -DXXA[k]);
        ratio(S8[k], Z8[k], XX[k] + S8[k] - (c.x_max - derr), DXX[k], DXXA[k]);
      }
      block_reduce(RED, tid, T, dummy_s, dummy_m, amin);
      if (pass == 0) {
        const double a_aff = fmin(1.0, amin);
        double acc = 0.0, d1 = 0.0, d2 = 0.0;
        auto muaff = [&](double s, double z, double rp, double g) {
          const double ds = -rp - g;
          const double dz = (-s * z - z * ds) / s;
          acc += (s + a_aff * ds) * (z + a_aff * dz);
        };
        for (int i = tid; i < QN; i += T) {
          const int q = i / N;
          muaff(S1[i], Z1[i], S1[i] - W[i], -DX[i]);
          muaff(S2[i], Z2[i], W[i] + S2[i] - WMX[q], DX[i]);
          DXA[i] = DX[i];
        }
        for (int k = tid; k < N; k += T) {
          const double e1 = (k == 0) ? derr : 0.0;
          muaff(S3[k], Z3[k], S3[k] - U[k], -BU[k]);
          muaff(S4[k], Z4[k], U[k] + S4[k] - c.u_g_max, BU[k]);
          muaff(S5[k], Z5[k], -V[k] + S5[k] - (c.u_b_max - e1), -DV[k]);
          muaff(S6[k], Z6[k], V[k] + S6[k] - (c.u_b_max - e1), DV[k]);
          muaff(S7[k], Z7[k], -XX[k] + S7[k] + derr, -DXX[k]);
          muaff(S8[k], Z8[k], XX[k] + S8[k] - (c.x_max - derr), DXX[k]);
          DXUA[k] = BU[k];
          DVA[k] = DV[k];
          DXXA[k] = DXX[k];
        }
        block_reduce(RED, tid, T, acc, d1, d2);
        const double mu_aff = acc / mtot;
        const double sg = mu_aff / mu;
        sigma_mu = sg * sg * sg * mu;
      } else {
        alpha = fmin(1.0, 0.99 * amin);
#ifdef BIMPC_TRACE
        printf("   alpha %.4f sigma_mu %.3e\n", alpha, sigma_mu);
#endif
      }
    }
    // ---- G. step (pass == 1 semantics for rc: DXA etc. still hold the affine direction)
    {
      auto upd = [&](double& s, double& z, double rp, double g, double ga) {
        const double dsa = -rp - ga;
        const double dza = (-s * z - z * dsa) / s;
        const double rc = s * z + dsa * dza - sigma_mu;
        const double ds = -rp - g;
        const double dz = (-rc - z * ds) / s;
        s += alpha * ds;
        z += alpha * dz;
      };
      for (int i = tid; i < QN; i += T) {
        const int q = i / N;
        const double rp1 = S1[i] - W[i], rp2 = W[i] + S2[i] - WMX[q];
        upd(S1[i], Z1[i], rp1, -DX[i], -DXA[i]);
        upd(S2[i], Z2[i], rp2, DX[i], DXA[i]);
        W[i] += alpha * DX[i];
      }
      for (int k = tid; k < N; k += T) {
        const double e1 = (k == 0) ? derr : 0.0;
        const double rp3 = S3[k] - U[k], rp4 = U[k] + S4[k] - c.u_g_max;
        const double rp5 = -V[k] + S5[k] - (c.u_b_max - e1), rp6 = V[k] + S6[k] - (c.u_b_max - e1);
        const double rp7 = -XX[k] + S7[k] + derr, rp8 = XX[k] + S8[k] - (c.x_max - derr);
        upd(S3[k], Z3[k], rp3, -BU[k], -DXUA[k]);
        upd(S4[k], Z4[k], rp4, BU[k], DXUA[k]);
        upd(S5[k], Z5[k], rp5, -DV[k], -DVA[k]);
        upd(S6[k], Z6[k], rp6, DV[k], DVA[k]);
        upd(S7[k], Z7[k], rp7, -DXX[k], -DXXA[k]);
        upd(S8[k], Z8[k], rp8, DXX[k], DXXA[k]);
        U[k] += alpha * BU[k];
      }
      BI_SYNC();
    }
    BI_TOC(3);
  }

  // ---- outputs (clipped into the box like the oracle; inactive partitions: w = 0)
  for (int i = tid; i < P * N; i += T) {
    a.w_hat_s[(size_t)st_idx * P * N + i] = 0.0;
    a.w_hat_l[(size_t)st_idx * P * N + i] = 0.0;
  }
  BI_SYNC();
  for (int i = tid; i < QN; i += T) {
    const int cq = i / N, k = i - cq * N, q = (int)QIDX[cq];
    const double x = fmin(fmax(W[i], 0.0), WMX[cq]);
    if (q < P) a.w_hat_s[((size_t)st_idx * P + q) * N + k] = x;
    else a.w_hat_l[((size_t)st_idx * P + (q - P)) * N + k] = x;
  }
  for (int k = tid; k < N; k += T) a.u_g[(size_t)st_idx * N + k] = fmin(fmax(U[k], 0.0), c.u_g_max);
  if (tid == 0) {
    a.status[st_idx] = status;
    a.iters[st_idx] = it;
  }
  if (a.objective) {
    // c_g sum u^1.7 + delta sum_q a_q sum_k omega_k (cumsum(w_q)_k - gamma_q)^2, by thread 0
    BI_SYNC();
    if (tid == 0) {
      double f = 0.0;
      for (int k = 0; k < N; ++k) f += c.c_g * pow(fmax(U[k], 0.0), 1.7);
      for (int q = 0; q < Q2; ++q) {
        double s = 0.0;
        for (int k = 0; k < N; ++k) {
          s += W[q * N + k];
          f += c.delta * AQ[q] * OM[k] * (s - GQ[q]) * (s - GQ[q]);
        }
      }
      a.objective[st_idx] = f;
    }
  }

}

#ifndef BIMPC_HOSTSIM
__global__ void __launch_bounds__(kThreads, kMinBlocks) bimpc_solve_kernel(const BiConsts c, const BiArgs a) {
  extern __shared__ double bimpc_smem[];
  for (int s = blockIdx.x; s < a.S; s += gridDim.x) {
    solve_station(c, a, s, bimpc_smem, a.li_scratch + (size_t)blockIdx.x * global_scratch_doubles(c.N, c.P), threadIdx.x,
                  blockDim.x);
    __syncthreads();
  }
}
#endif

}  // namespace bimpc
