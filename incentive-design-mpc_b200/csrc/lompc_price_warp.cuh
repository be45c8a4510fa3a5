// K5, parametric variant (SURVEY.md section 8 row f3): PriceSolver.compute_optimal_prices
// (reference price_solver.py:79-174) for one group (station, EV type, partition) by ONE WARP,
// exploiting that the EVs of a group share their prices and differ only in the scalar gamma_i
// (price_solver.py:196-214): the QP's linear term is affine in gamma, so its solution is
// PIECEWISE AFFINE in gamma - affine on every critical region (= set of gammas with the same
// active set: which breakpoint / which piece every stage sits on), and critical regions are
// intervals.  Two EVs whose solutions carry the same piece codes lie in one region, and so does
// every EV between them: their solutions are the linear interpolation of the two, and the SUM the
// price loop needs (w_avg, price_solver.py:205-210) is
//     count * w_a + (sum(gamma_i) - count * gamma_a) / (gamma_b - gamma_a) * (w_b - w_a)
// from two prefix sums over the sorted gammas - no solve per EV.
//
// Per MM iteration: the EVs are sorted by gamma once per group; the warp solves the extreme EVs and the
// "virtual EV" at gamma_sc (price_solver.py:106,132; it is the midpoint of the gamma range) with the
// warp-cooperative K1 (lompc_solve_warp.cuh: QPW = 32 / (N/3) QPs per round, warm-started from the
// previous iteration or from the neighbouring pivot), compares the piece codes of neighbouring pivots,
// and splits only the intervals whose ends disagree - (QPW + 1)-way, so that every round of the solver
// is full and a region boundary among n EVs is located in log_{QPW+1}(n) rounds.  A group of ~95 EVs
// spans 1.6-1.8 regions at the closed loop's prices.  Then lane 0 runs the convergence test and the warp
// the exact price step (price_step_warp) exactly as in lompc_price_fused.cuh.  One warp per CTA, ~12 KB
// of shared memory, compact rolled code (the thread-per-EV kernels stream ~100 KB of unrolled code per
// iteration and are instruction-fetch bound at fleet scale).
#pragma once
#include "lompc_common.cuh"
#include "lompc_price.cuh"
#include "lompc_price_fused.cuh"
#include "lompc_solve_warp.cuh"

namespace lompc {

#ifndef LOMPC_K3_FLEET_UNROLL
#define LOMPC_K3_FLEET_UNROLL 4
#endif
#ifndef LOMPC_CHAIN_MINB
#define LOMPC_CHAIN_MINB 1
#endif
// Test hook: pivot slots the parametric loop may use (price_debug_pivot_pool(); 32 = all).  A small pool makes the
// direct jobs of group_loop_warp, which a full pool needs about once in 10^4 groups, the common case.
__device__ int g_pivot_pool = 32;
// Test hook: [G] device arrays (price_debug_record_errors()) that receive, per group, w_err_max and w_avg_err of the
// last convergence test of a parametric "max" loop; NULL = off.
__device__ double* g_record_err_max = nullptr;
__device__ double* g_record_err_avg = nullptr;
constexpr int kMaxPivots = 32;  // solved EVs kept at a time (3 permanent: lowest gamma, virtual, highest gamma)
constexpr int kQueueCap = 64;   // intervals between neighbouring pivots waiting for their verdict

// A-bar-norm of w - w_ref (price_solver.py:207), w = wa + t (wb - wa): the formula and summation order of the
// thread-per-EV loop (lompc_price_fused.cuh), so that a solved EV (t = 0) gives the same error there and here.
template <int N>
__device__ __forceinline__ double ev_err_warp(const double* wa, const double* wb, const double t, const double* wref,
                                              const double kappa) {
  double cum = 0.0, e2 = 0.0;
  for (int k = 0; k < N; ++k) {
    const double v = wa[k] + t * (wb[k] - wa[k]) - wref[k];
    cum += v;
    e2 += cum * cum + kappa * v * v;
  }
  return sqrt(e2);
}

template <int N>
struct WarpLoopSmem {
  // doubles
  static constexpr int oLM = 0;                      // [3N] current prices
  static constexpr int oWREF = oLM + 3 * N;          // [N]
  static constexpr int oWSUM = oWREF + N;            // [N]
  static constexpr int oWS = oWSUM + N;              // price-step scratch, 18N
  static constexpr int oPW = oWS + 18 * N;           // [kMaxPivots][N] pivot solutions
  static constexpr int oPG = oPW + kMaxPivots * N;   // [kMaxPivots] pivot gammas
  static constexpr int oSC = oPG + kMaxPivots;       // 8 scalars
  static constexpr int kDoubles = oSC + 8;
  // then ints PFA / PLB [kMaxPivots]; bytes: PC[kMaxPivots][N], queues 2 x 2 x kQueueCap, WSB[3N]
  static constexpr size_t bytes =
      (size_t)kDoubles * 8 + 3 * kMaxPivots * 4 + kMaxPivots * N + 4 * kQueueCap + 3 * N + 32;
};

// The loop of ONE group by one warp.  Same contract as group_loop_body (lompc_price_fused.cuh).  N = 12, 24 (the closed
// loop's horizons) and 48, 96 (configs[4]'s: 16 / 32 lanes per QP, 2 / 1 QPs per warp pass).
// Scratch in global memory (a.w_scratch rows b0 .., N doubles per EV): the sorted gammas and their
// prefix sums (2n + 1 doubles; the launcher sizes the rows so that this fits for every n >= 1).
// MAXTOL: the "max" tolerance type (price_solver.py:121-128), the largest error of a single EV.  Within a critical
// region w is affine in gamma, so the error is convex in gamma on every interpolated interval and its largest value
// over the interval's EVs is at the first or the last of them: the maximum over the group is the maximum over the real
// EVs solved (pivots, direct jobs) and those two EVs of every interpolated interval.  The virtual EV is not an EV of
// the group and never enters it.  A separate instantiation, so that the "avg" kernels carry none of this code.
template <int N, int NSEG, bool MAXTOL>
__device__ __forceinline__ bool group_loop_warp(const Consts& cs, const FusedArgs& a, const int g, double* smem,
                                                const double* p_in, double* p_out, double* p_out2) {
  constexpr int SPL = 3, LPQ = N / SPL, QPW = 32 / LPQ;
  static_assert(N % SPL == 0 && (32 % LPQ == 0) && N <= 96, "N = 12, 24, 48, 96");
  constexpr int NW = (N + 31) / 32;  // stages per lane in the sums over the group (lane l: stages l, l + 32, ...)
  const int lane = threadIdx.x;
  const int b0 = a.group_off[g], b1 = a.group_off[g + 1];
  const int n = b1 - b0;
  if (n <= 0) {
    if (lane == 0) a.iters[g] = -1;
    return false;
  }
  using L = WarpLoopSmem<N>;
  double* LM = smem + L::oLM;
  double* WREF = smem + L::oWREF;
  double* WSUM = smem + L::oWSUM;
  double* WS = smem + L::oWS;
  double* PW = smem + L::oPW;
  double* PG = smem + L::oPG;
  double* SC = smem + L::oSC;
  int* PFA = reinterpret_cast<int*>(smem + L::kDoubles);  // first EV index after the pivot
  int* PLB = PFA + kMaxPivots;                             // last EV index before the pivot
  int* PIT = PLB + kMaxPivots;                             // K1 iterations of the slot's last solve (statistics)
  unsigned char* PC = reinterpret_cast<unsigned char*>(PIT + kMaxPivots);  // [slot][N] piece codes
  unsigned char* Q0 = PC + kMaxPivots * N;                 // interval queues (ping-pong): endpoints a, b
  unsigned char* Q1 = Q0 + 2 * kQueueCap;
  unsigned char* WSB = Q1 + 2 * kQueueCap;                 // [r] free set of the price step
  double* WK = PW + N;                                     // slot 1 = the virtual EV: w_k of price_solver.py:106,132
  double* GS = a.w_scratch + (size_t)b0 * N + (size_t)2 * g;  // [n] sorted gammas (2 extra doubles per group before it)
  double* GPS = GS + n;                                    // [n + 1] prefix sums of GS
  const unsigned full = 0xffffffffu;

  // ---- set_charge_levels (price_solver.py:66-77) + sort of the gammas (rank sort, once per group)
  double mn = 1e300, mx = -1e300;
  bool bad = false;
  for (int i = lane; i < n; i += 32) {
    const double y = a.y0[b0 + i];
    if (!(y >= 0.0 && y <= cs.y_max)) bad = true;
    mn = fmin(mn, y);
    mx = fmax(mx, y);
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) {
    mn = fmin(mn, __shfl_xor_sync(full, mn, d));
    mx = fmax(mx, __shfl_xor_sync(full, mx, d));
  }
  if (__any_sync(full, bad)) {
    if (lane == 0) atomicExch(a.flags + 1, 1);
  }
  for (int i = lane; i < n; i += 32) {
    const double yi = a.y0[b0 + i];
    int rank = 0;  // gamma ascending = y0 descending; ties by index
    for (int j = 0; j < n; ++j) {
      const double yj = a.y0[b0 + j];
      rank += (yj > yi) || (yj == yi && j < i);
    }
    GS[rank] = cs.y_max - yi;
  }
  for (int k = lane; k < 3 * N; k += 32) LM[k] = p_in[k];
  for (int k = lane; k < N; k += 32) WREF[k] = a.w_ref[(size_t)g * N + k];
  __syncwarp();
  if (lane == 0) {  // prefix sums of the sorted gammas
    double acc = 0.0;
    GPS[0] = 0.0;
    for (int i = 0; i < n; ++i) {
      acc += GS[i];
      GPS[i + 1] = acc;
    }
  }
  const double y0_rng = (mx - mn) / 2;
  const double gamma_sc = cs.y_max - (mx + mn) / 2;
  const double lr = a.lmbd_r[g];
  const double kappa = lr / cs.delta;
  const double tolg = sqrt((double)N) * y0_rng + a.eps_tol;  // price_solver.py:184
  abar_factor<(N <= 24 ? N : 0)>(N, kappa, WS + 3 * a.r + 6 * N, lane);
  __syncwarp();
  // position of the virtual EV in the sorted list: EVs [0, vpos) have gamma <= gamma_sc
  int vpos;
  {
    int lo = 0, hi = n;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (GS[mid] <= gamma_sc) lo = mid + 1; else hi = mid;
    }
    // the list order is EV 0 <= virtual <= EV n - 1: gamma_sc is the midpoint of the range, but with (nearly) equal
    // SoCs it rounds onto the largest gamma and the search lands behind the last EV - which would then be counted
    // twice (inside the first interval and as the pivot of the last one)
    vpos = n > 1 ? max(1, min(lo, n - 1)) : 1;
  }
  // permanent pivots: slot 0 = EV 0 (lowest gamma), slot 1 = virtual EV, slot 2 = EV n - 1 (n > 1)
  const int nperm = n > 1 ? 3 : 2;
  if (lane == 0) {
    PG[0] = GS[0]; PFA[0] = 1; PLB[0] = -1;
    PG[1] = gamma_sc; PFA[1] = vpos; PLB[1] = vpos - 1;
    PG[2] = GS[n - 1]; PFA[2] = n; PLB[2] = n - 2;
  }
  for (int k = lane; k < 3 * N; k += 32) PW[k] = 0.0;
  __syncwarp();

  const int pool_n = g_pivot_pool;
  const unsigned pool = pool_n >= 32 ? 0xffffffffu : ((1u << (pool_n < nperm + 1 ? nperm + 1 : pool_n)) - 1u);
  double dual_cost = 0.0, lamdiff = 0.0, dec_pred = 0.0;  // lane 0
  int it = 0, nnqp_bad = 0, flag = 0;
  unsigned long long solves = 0, rounds = 0, k1_iters = 0;
  long long cyc_qp = 0, cyc_step = 0, cyc_solve = 0;
  int overflowed = 0;
  for (;; ++it) {
    const long long t_a = clock64();
    // ================= LoMPC pass: pivots, splitting, interpolated sum =================
    // warp-uniform registers: slot masks, 2-bit reference counts (intervals that use a slot), queue length
    unsigned used = (1u << nperm) - 1u, solved = 0u;
    unsigned long long refs = 0ull;
    unsigned char *QR = Q0, *QW = Q1;
    int qn = nperm - 1;
    if (lane == 0) {
      QR[0] = 0; QR[1] = 1;
      QR[2] = 1; QR[3] = 2;
    }
    double wsum[NW];  // lane l, slot u: sum over the group's EVs of w_i[l + 32 u]
#pragma unroll
    for (int u = 0; u < NW; ++u) wsum[u] = 0.0;
    [[maybe_unused]] double emax = 0.0;  // MAXTOL: largest EV error this lane has evaluated in this pass
    // direct job: EVs [dj_first, dj_first + dj_cnt) of an interval (dj_sa, dj_sb) that found no free pivot slots are
    // solved one by one into the (idle) price-step scratch - exact, just without the saving
    int dj_first = 0, dj_cnt = 0, dj_sa = 0, dj_sb = 0;
    auto release = [&](int sx) {  // an interval lets go of an endpoint; slots nobody holds return to the pool
      if (sx >= nperm) {
        const unsigned long long rc = (refs >> (2 * sx)) & 3ull;
        refs -= 1ull << (2 * sx);
        if (rc == 1ull) {
          used &= ~(1u << sx);
          solved &= ~(1u << sx);
        }
      }
    };
    __syncwarp();
    for (;;) {
      // ---- solve phase: up to QPW unsolved pivots (or EVs of the direct job) per round, one per lane group
      unsigned pending = used & ~solved;
      const bool direct = !pending && dj_cnt > 0;
      if (pending || direct) {
        int my_slot = -1, q = 0;
        unsigned batch = 0u;
        if (direct) {
          q = dj_cnt < QPW ? dj_cnt : QPW;
          if (lane / LPQ < q) my_slot = lane / LPQ;  // (a row of the scratch, not a pivot slot)
        } else {
          for (unsigned m = pending; m && q < QPW; m &= m - 1, ++q) {
            const int s = __ffs(m) - 1;
            if (lane / LPQ == q) my_slot = s;
            batch |= 1u << s;
          }
        }
        solves += (unsigned long long)q;
        ++rounds;
        WarpProblem P;
        const int s = my_slot < 0 ? 0 : my_slot;
        P.lm = LM;
        P.lr = lr;
        P.gam = direct ? GS[dj_first + s] : PG[s];
        // (a new pivot holds a copy of a neighbour's solution; a direct solve starts from the interval's left end)
        P.w_init = direct ? PW + dj_sa * N : ((it > 0 || s >= nperm) ? PW + s * N : nullptr);
        P.w_out = direct ? WS + s * N : PW + s * N;
        P.cost_out = (!direct && s == 1) ? SC + 0 : nullptr;
        P.status = nullptr;
        P.iters = (a.qp_count && !direct) ? PIT + s : nullptr;
        P.kkt_res = nullptr;
        P.codes_out = direct ? nullptr : PC + s * N;
        P.tol = a.qp_tol;
        P.max_iter = a.qp_max_iter;
        int st;
        const long long t_s = clock64();
        solve_warp_core<N, NSEG, SPL>(cs, P, my_slot >= 0, lane, st);
        cyc_solve += clock64() - t_s;
        if (__any_sync(full, my_slot >= 0 && st != LOMPC_ST_OK)) {
          if (lane == 0) atomicAdd(a.flags + 3, 1);
        }
        __syncwarp();
        if constexpr (MAXTOL) {  // one solved EV per lane: the direct job's rows, or the real EVs of the batch
          int sv = -1;
          if (direct) {
            if (lane < q) sv = lane;
          } else {
            int t = 0;
            for (unsigned m = batch & ~2u; m; m &= m - 1, ++t)
              if (t == lane) sv = __ffs(m) - 1;
          }
          if (sv >= 0) {
            const double* w = direct ? WS + sv * N : PW + sv * N;
            emax = fmax(emax, ev_err_warp<N>(w, w, 0.0, WREF, kappa));
          }
        }
        if (direct) {
          for (int t = 0; t < q; ++t)
#pragma unroll
            for (int u = 0; u < NW; ++u)
              if (lane + 32 * u < N) wsum[u] += WS[t * N + lane + 32 * u];
          dj_first += q;
          dj_cnt -= q;
          if (dj_cnt == 0) {
            release(dj_sa);
            release(dj_sb);
          }
          __syncwarp();
          continue;
        }
        // the real EVs just solved count once themselves
        for (unsigned m = batch & ~2u; m; m &= m - 1) {
          const int sv = __ffs(m) - 1;
#pragma unroll
          for (int u = 0; u < NW; ++u)
            if (lane + 32 * u < N) wsum[u] += PW[sv * N + lane + 32 * u];
        }
        if (a.qp_count)
          for (unsigned m = batch; m; m &= m - 1) k1_iters += (unsigned long long)PIT[__ffs(m) - 1];
        solved |= batch;
        continue;
      }
      // ---- verdicts: neighbouring pivots with the same codes (or nothing in between) are interpolated,
      //      the others are split (QPW + 1)-way
      bool progressed = false;
      int wn = 0;
      for (int e = 0; e < qn; ++e) {
        const int sa = QR[2 * e], sb = QR[2 * e + 1];
        const int fa = PFA[sa], lb = PLB[sb];
        const int cnt = lb - fa + 1;
        bool same = true;
        if (cnt > 0) {
          bool diff = false;
#pragma unroll
          for (int u = 0; u < NW; ++u)
            if (lane + 32 * u < N) diff |= PC[sa * N + lane + 32 * u] != PC[sb * N + lane + 32 * u];
          same = !__any_sync(full, diff);
        }
        if (cnt <= 0 || same) {
          if (cnt > 0) {
            const double ga = PG[sa], gb = PG[sb];
            const double sg = GPS[lb + 1] - GPS[fa];
            const double coef = gb > ga ? (sg - cnt * ga) / (gb - ga) : 0.0;
#pragma unroll
            for (int u = 0; u < NW; ++u)
              if (lane + 32 * u < N) {
                const double wa = PW[sa * N + lane + 32 * u], wb = PW[sb * N + lane + 32 * u];
                wsum[u] += cnt * wa + coef * (wb - wa);
              }
            if constexpr (MAXTOL) {  // the interval's first (lane 0) and last (lane 1) EV, on the interpolant
              if (lane < 2) {
                const double gi = GS[lane == 0 ? fa : lb];
                emax = fmax(emax, ev_err_warp<N>(PW + sa * N, PW + sb * N, gb > ga ? (gi - ga) / (gb - ga) : 0.0,
                                                 WREF, kappa));
              }
            }
          }
          release(sa);
          release(sb);
          progressed = true;
          continue;
        }
        const int k = cnt < QPW ? cnt : QPW;  // new pivots inside the interval
        const unsigned freem = ~used & pool;   // kMaxPivots == 32: every clear bit is a free slot
        if (__popc(freem) >= k && wn + (k + 1) + (qn - e - 1) <= kQueueCap) {
          int prev = sa;
          unsigned fm = freem;
          for (int t = 1; t <= k; ++t) {
            const int sn = __ffs(fm) - 1;
            fm &= fm - 1;
            const int idx = fa + (int)(((long long)t * cnt) / (k + 1));
            used |= 1u << sn;
            refs |= 2ull << (2 * sn);
            if (lane == 0) {
              PG[sn] = GS[idx];
              PFA[sn] = idx + 1;
              PLB[sn] = idx - 1;
              QW[2 * wn] = (unsigned char)prev;
              QW[2 * wn + 1] = (unsigned char)sn;
            }
#pragma unroll
            for (int u = 0; u < NW; ++u)  // warm start: the left end's solution
              if (lane + 32 * u < N) PW[sn * N + lane + 32 * u] = PW[sa * N + lane + 32 * u];
            ++wn;
            prev = sn;
          }
          if (lane == 0) {
            QW[2 * wn] = (unsigned char)prev;
            QW[2 * wn + 1] = (unsigned char)sb;
          }
          ++wn;
          progressed = true;
        } else {  // no room now: the interval waits
          if (lane == 0) {
            QW[2 * wn] = (unsigned char)sa;
            QW[2 * wn + 1] = (unsigned char)sb;
          }
          ++wn;
        }
      }
      qn = wn;
      {
        unsigned char* t = QR;
        QR = QW;
        QW = t;
      }
      __syncwarp();
      if (qn == 0 && dj_cnt == 0) break;
      if (!progressed && !(used & ~solved) && dj_cnt == 0) {
        // pool exhausted (about one group in 10^4 on the first step of a fleet): every slot is an endpoint of a
        // waiting interval.  The last interval of the queue becomes the direct job; finishing it and, if need be, its
        // neighbours (consecutive in the queue) returns their shared endpoints to the pool.
        --qn;
        dj_sa = QR[2 * qn];
        dj_sb = QR[2 * qn + 1];
        dj_first = PFA[dj_sa];
        dj_cnt = PLB[dj_sb] - dj_first + 1;
        overflowed = 1;
      }
    }
#pragma unroll
    for (int u = 0; u < NW; ++u)
      if (lane + 32 * u < N) WSUM[lane + 32 * u] = wsum[u];
    __syncwarp();
    // ================= lane 0: bookkeeping of the previous step, convergence test; all lanes: price step =================
    flag = 0;
    const long long t_b = clock64();
    cyc_qp += t_b - t_a;
    if constexpr (MAXTOL) {
#pragma unroll
      for (int d = 16; d >= 1; d >>= 1) emax = fmax(emax, __shfl_xor_sync(full, emax, d));
    }
    if (lane == 0) {
      const double cost_sc = SC[0];
      if (it > 0 && a.hist_ac && it - 1 < a.hist_cap) {  // price_solver.py:135-139
        a.hist_ac[(size_t)g * a.hist_cap + it - 1] = cost_sc - dual_cost + lamdiff;
        a.hist_pred[(size_t)g * a.hist_cap + it - 1] = dec_pred;
      }
      dual_cost = cost_sc;
      if (it >= a.max_iter) {
        flag = 2;  // the loop ran out: `iter` ends at max_iter - 1 (price_solver.py:111)
      } else {
        double w_avg_err, w0_err;
        price_errors(N, kappa, WSUM, (double)n, WREF, w_avg_err, w0_err);
        if constexpr (MAXTOL) {
          if (emax <= tolg) flag = 1;  // price_solver.py:125 ("max" tolerance type)
          if (g_record_err_max) {
            g_record_err_max[g] = emax;
            g_record_err_avg[g] = w_avg_err;
          }
        } else {
          if (w_avg_err <= tolg) flag = 1;  // price_solver.py:125 ("avg" tolerance type)
        }
      }
    }
    flag = __shfl_sync(full, flag, 0);
    if (flag != 0) break;
    {
      int st;
      // (unrolled recursions for the horizons of the closed loop - 4 stages per trip in launches of several waves,
      // where the code size counts (K3Unroll), all of them otherwise -, rolled ones for the long horizons of the sweep)
      if (N <= 24 && a.compact_step)
        price_step_warp<(N <= 24 ? N : 0), LOMPC_K3_FLEET_UNROLL>(cs, a.r, kappa, a.eps_reg, LM, WK, WREF, WS, WSB, lane,
                                                                  it == 0, it > 0, a.hist_ac != nullptr, true, lamdiff,
                                                                  dec_pred, st);
      else
        price_step_warp<(N <= 24 ? N : 0)>(cs, a.r, kappa, a.eps_reg, LM, WK, WREF, WS, WSB, lane, it == 0, it > 0,
                                           a.hist_ac != nullptr, true, lamdiff, dec_pred, st);
      nnqp_bad |= st;
    }
    __syncwarp();
    cyc_step += clock64() - t_b;
  }
  // ---- regularisation (price_solver.py:145-147) and outputs
  if (lane == 0) {
    a.iters[g] = (flag == 2) ? a.max_iter - 1 : it;
    double pre, post;
    regularize_core(cs, a.r, WK, LM, pre, post);
    a.price_pre[g] = pre;
    a.price_post[g] = post;
    if (nnqp_bad & 1) atomicAdd(a.flags, 1);
    if (nnqp_bad & 2) atomicAdd(a.flags + 17, 1);  // groups that took the NNQP fallback (informational)
    if (overflowed) atomicAdd(a.flags + 16, 1);  // informational (flags[4..15] hold the 64-bit counters)
    atomicMax(a.flags + 2, it);
    if (a.qp_count) {
      atomicAdd(a.qp_count, solves);
      atomicAdd(a.qp_count + 1, (unsigned long long)cyc_solve);  // cycles inside the K1 rounds (summed over groups)
      atomicAdd(a.qp_count + 2, (unsigned long long)cyc_step);  // cycles in the price steps
      atomicAdd(a.qp_count + 3, k1_iters);                      // K1 iterations summed over the solves
      atomicAdd(a.qp_count + 4, rounds);                        // solver rounds ...
      atomicAdd(a.qp_count + 5, (unsigned long long)(it + 1));  // ... over this many LoMPC passes
    }
  }
  __syncwarp();
  for (int k = lane; k < 3 * N; k += 32) {
    p_out[k] = LM[k];
    if (p_out2) p_out2[k] = LM[k];
  }
  if (a.w_k_out)
    for (int k = lane; k < N; k += 32) a.w_k_out[(size_t)g * N + k] = WK[k];
  __syncwarp();
  return true;
}

// Grid = the groups: one warp (= one CTA) per group.  MAXTOL = "max" tolerance type (a.tol_type_max).
template <int N, bool MAXTOL>
__global__ void __launch_bounds__(32, LOMPC_CHAIN_MINB) price_group_warp_kernel(const __grid_constant__ Consts cs,
                                                                 const __grid_constant__ FusedArgs a) {
  extern __shared__ double smem[];
  const int g = blockIdx.x;
  double* row = a.prices + (size_t)g * 3 * N;
  if (cs.large)
    group_loop_warp<N, 4, MAXTOL>(cs, a, g, smem, row, row, nullptr);
  else
    group_loop_warp<N, 1, MAXTOL>(cs, a, g, smem, row, row, nullptr);
}

// Grid = the stations: one warp per station walks its P partitions in the reference's warm-start order
// (see price_station_chain_kernel in lompc_price_fused.cuh).
template <int N, bool MAXTOL>
__global__ void __launch_bounds__(32, LOMPC_CHAIN_MINB) price_station_chain_warp_kernel(const __grid_constant__ Consts cs,
                                                                         const __grid_constant__ FusedArgs a) {
  extern __shared__ double smem[];
  const int S = a.chain_S, s = a.chain_order ? a.chain_order[blockIdx.x] : (int)blockIdx.x;
  double* prev = a.chain_prev + (size_t)s * 3 * N;
  for (int p = 0; p < a.chain_P; ++p) {
    const int g = p * S + s;
    double* row = a.prices + (size_t)g * 3 * N;
    const bool solved = cs.large ? group_loop_warp<N, 4, MAXTOL>(cs, a, g, smem, prev, prev, row)
                                 : group_loop_warp<N, 1, MAXTOL>(cs, a, g, smem, prev, prev, row);
    if (!solved)
      for (int k = threadIdx.x; k < 3 * N; k += 32) row[k] = 0.0;
    __syncwarp();
  }
}

// Phase-split loop, second half of a group phase in ONE launch: the gamma_sc solves of iteration `it`
// (price_solver.py:132, the warp-cooperative K1 in group mode: row = group, warm start from w_k) followed, per group,
// by bookkeep_kernel's work (price_solver.py:135-137: the actual decrease from the cost this lane group has just
// written, the new dual cost, the histories).  Warp 0 also publishes the active-group count of the iteration to the
// host's ring and resets the counter: the launch is stream-ordered after group_step_kernel(it), and nothing else touches
// the counter before group_step_kernel(it + 1), which is ordered after this launch.  Same arithmetic as the two
// launches it replaces; a launch (and its place on the side stream's critical path) less per iteration.
template <int N>
__global__ void __launch_bounds__(32, 1) sc_solve_bookkeep_kernel(const __grid_constant__ Consts cs,
                                                                  const __grid_constant__ SolveArgs a,
                                                                  const __grid_constant__ PriceArgs p, const int it) {
  constexpr int SPL = 3, LPQ = N / SPL, QPW = 32 / LPQ;
  const int lane = threadIdx.x;
  const int64_t b = (int64_t)blockIdx.x * QPW + lane / LPQ;
  const bool live = b < a.B;
  if (blockIdx.x == 0 && lane == 0 && p.publish_ring) {
    volatile int32_t* slot = p.publish_ring + 2 * (it % p.publish_slots);
    slot[1] = *p.n_active;
    __threadfence_system();
    slot[0] = it + 1;
    *p.n_active = 0;
  }
  int st;
  if (cs.large)
    solve_warp<N, 4, SPL>(cs, a, b, live, lane, st);
  else
    solve_warp<N, 1, SPL>(cs, a, b, live, lane, st);
  if (live && (lane & (LPQ - 1)) == 0 && !p.skip[b]) {  // the lane that stored cost_out[b] (group b)
    const double cn = a.cost_out[b];
    const double ac = cn - p.dual_cost[b] + p.lamdiff_phi[b];
    p.dual_cost[b] = cn;
    if (p.hist_ac && it < p.hist_cap) {
      p.hist_ac[(size_t)b * p.hist_cap + it] = ac;
      p.hist_pred[(size_t)b * p.hist_cap + it] = p.dec_pred[b];
    }
  }
}

}  // namespace lompc
