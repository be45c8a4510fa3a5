/*
 * lompc_b200.h -- C ABI of the B200-native lower-level MPC (LoMPC) hot path.
 *
 * The reference (AkshayThiru/incentive-design-mpc) has no FFI of its own: the
 * boundary of this path is its Python class API (SURVEY.md section 8b).  Each
 * entry point below names the reference method it replaces (file:line relative
 * to the reference tree).  The Python mirror of those classes, in
 * incentive-design-mpc_b200/chargingstation/, binds this header with ctypes;
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions: plain C, fp64, row-major, B = batch.  Functions return 0 on
 * success or a negative LOMPC_ERR_* code; they never throw.  "_dev" entry
 * points take DEVICE pointers and are asynchronous on `stream` (a
 * cudaStream_t passed as void*); "_host" entry points take HOST pointers and
 * do the host<->device copies themselves and synchronise before returning.
 * A handle is bound to one (EV type, horizon N, device); it is not
 * thread-safe (neither are the reference's objects, SURVEY.md 8b).
 */
#ifndef LOMPC_B200_H
#define LOMPC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LOMPC_OK 0
#define LOMPC_ERR_CONSTS (-1)      /* lompc.py:36-38 asserts  -> AssertionError */
#define LOMPC_ERR_ARG (-2)         /* bad pointer / size / shape */
#define LOMPC_ERR_CUDA (-3)        /* CUDA runtime failure (see lompc_last_cuda_error) */
#define LOMPC_ERR_GAMMA (-4)       /* gamma > y_max, lompc.py:87 -> AssertionError */
#define LOMPC_ERR_NEGATIVE (-5)    /* nonneg cv.Parameter got < 0, lompc.py:78-82 -> ValueError */
#define LOMPC_ERR_NOT_CONVERGED (-6)
#define LOMPC_ERR_NO_DEVICE (-7)   /* no CUDA device: there is NO CPU fallback */

#define LOMPC_EV_SMALL 0
#define LOMPC_EV_LARGE 1

/* per-QP status written by the solve kernels */
#define LOMPC_ST_OK 0
#define LOMPC_ST_MAXITER 1
#define LOMPC_ST_BAD_GAMMA 2
#define LOMPC_ST_NEGATIVE 3

typedef struct lompc_handle lompc_t;

/* Library / build information. */
const char* lompc_version(void);
const char* lompc_strerror(int code);
const char* lompc_last_cuda_error(void);
int lompc_device_count(void);

/* Replaces LoMPC.__init__ / _set_constants (lompc.py:30-71): validates the
 * constants exactly like lompc.py:36-38 (LOMPC_ERR_CONSTS), derives q_scale
 * (lompc.py:67) and the strong-convexity modulus m (lompc.py:71).           */
int lompc_create(int N, double delta, double theta, double y_max, double w_max,
                 int ev_type, int device, lompc_t** out);
int lompc_destroy(lompc_t* h);

/* LoMPC.get_sc_modulus (lompc.py:158). */
double lompc_sc_modulus(const lompc_t* h);

/* Solver knobs (defaults: max_iter 200, tol 1e-11 relative KKT residual). */
int lompc_set_options(lompc_t* h, int max_iter, double tol);

/* Kernel choice: 0 = automatic (register-resident kernel for N = 12, 24 - 64 threads x 4 CTAs per SM; large EV
 * on grids that fill the GPU: one 256-thread CTA per SM; plain batches of >= 65,536 QPs at N = 24: the same
 * kernel with bulk-copied rows, see 9 - and the any-N shared-memory kernel otherwise),
 * 1 = always the any-N kernel (every N that lompc_create accepts, 1..4096: up to 128 threads per CTA, fewer where
 * N's columns do not fit - below 32 threads above N = 129 large EV / 151 small EV, down to one thread at N = 4096), 4 / 7 = one register-kernel shape regardless of the batch size (4 = 64 threads x
 * 4 CTAs per SM, 7 = 256 x 1; the other shapes of round 1's sweep are no longer compiled: LOMPC_ERR_ARG);
 * 8 = the warp-cooperative latency kernel (one QP per group of N/3 lanes, time-parallel sweeps; N = 12, 24,
 * 48, 96), which automatic mode picks for batches too small to fill the GPU with one QP per thread;
 * 9 = the register kernel with every row moved by the bulk-copy engine (cp.async.bulk into shared memory, one copy per
 * row, result rows by bulk stores; N = 12, 24; batches that are not plain 16-byte aligned rows - broadcast prices, the
 * group mode of the price loop, fused error outputs - run on the default shape). */
int lompc_set_kernel_variant(lompc_t* h, int variant);

/* Replaces LoMPC.solve_lompc (lompc.py:137-156), batched over B independent
 * QPs.  lmbd: B rows of 3N prices (row stride lmbd_stride doubles; 0 =
 * broadcast ONE price vector to the whole batch, the _get_w_err case
 * price_solver.py:203-204).  lmbd_r: stride 0 = one scalar for all.
 * gamma[B].  Outputs: w_out[B,N], cost_out[B] (the full objective including
 * theta*w_max*sum(lmbd2), as self.cost.value lompc.py:155); optional (may be
 * NULL) status[B], iters[B], kkt_res[B] (relative KKT residual).             */
int lompc_solve_batch_dev(lompc_t* h, int64_t B, const double* lmbd, int64_t lmbd_stride,
                          const double* lmbd_r, int64_t lmbd_r_stride, const double* gamma,
                          double* w_out, double* cost_out, int32_t* status, int32_t* iters,
                          double* kkt_res, void* stream);

/* Vector-Jacobian product of lompc_solve_batch_dev: for B solved QPs (w[B,N] = their solutions) and upstream
 * gradients grad_w[B,N] on w and grad_cost[B] on the cost (either may be NULL = zero), writes per QP
 *   grad_lmbd[B,3N], grad_lmbd_r[B], grad_gamma[B]   (each may be NULL: not computed)
 * = the gradient of  sum_k grad_w[b,k] w[b,k] + grad_cost[b] cost[b]  with respect to that QP's lmbd row, lmbd_r
 * and gamma.  lmbd / lmbd_r take the strides of lompc_solve_batch_dev (0 = broadcast); the outputs are per-QP rows
 * even then (a caller that broadcast sums them over the batch).  One QP per thread, two O(N) sweeps (a Riccati
 * solve with the upstream gradient as right-hand side, DESIGN.md section 2).  Asynchronous on `stream`, DEVICE
 * pointers; every N that lompc_create accepts.
 * Classification: a coordinate of w within 1e-9 w_max of a breakpoint (0, w_max, an interior large-EV pwl
 * breakpoint) is fixed, the others are free; the w-gradient is that of this active set.  At a weakly active
 * coordinate (multiplier at an end of its interval) w is not differentiable; the result is then one of the
 * one-sided derivatives.  The cost gradient (envelope theorem) holds at every point.
 * A row with a negative or NaN parameter or gamma > y_max gets zero gradients and the solve's status code in the
 * optional status[B] (LOMPC_ST_NEGATIVE / LOMPC_ST_BAD_GAMMA; LOMPC_ST_OK otherwise).                           */
int lompc_vjp_dev(lompc_t* h, int64_t B, const double* lmbd, int64_t lmbd_stride,
                  const double* lmbd_r, int64_t lmbd_r_stride, const double* gamma,
                  const double* w, const double* grad_w, const double* grad_cost,
                  double* grad_lmbd, double* grad_lmbd_r, double* grad_gamma,
                  int32_t* status, void* stream);

/* Same call with HOST buffers: copies in, solves, copies out, synchronises.
 * Returns LOMPC_ERR_GAMMA / LOMPC_ERR_NEGATIVE / LOMPC_ERR_NOT_CONVERGED if
 * any QP reported that status (outputs are still written).                  */
int lompc_solve_batch_host(lompc_t* h, int64_t B, const double* lmbd, int64_t lmbd_stride,
                           const double* lmbd_r, int64_t lmbd_r_stride, const double* gamma,
                           double* w_out, double* cost_out, int32_t* status, int32_t* iters,
                           double* kkt_res);

/* The host call in two halves, so that independent handles (the two EV types, several batches)
 * overlap their copies and kernels: _async enqueues copies-in, the solve and copies-out on the
 * handle's own stream and returns; lompc_host_wait blocks until they are done and returns what
 * lompc_solve_batch_host would have.  Host buffers must stay alive (and should be pinned) until
 * the wait; one pending call per handle.                                                       */
int lompc_solve_batch_host_async(lompc_t* h, int64_t B, const double* lmbd, int64_t lmbd_stride,
                                 const double* lmbd_r, int64_t lmbd_r_stride, const double* gamma,
                                 double* w_out, double* cost_out, int32_t* status, int32_t* iters,
                                 double* kkt_res);
int lompc_host_wait(lompc_t* h);

/* ------------------------------------------------------------------------
 * Solve set: the QPs of SEVERAL LoMPC objects (the small-EV and the large-EV
 * solver of a station, charging_station.py:59-60) solved by ONE kernel launch,
 * with ONE host->device and ONE device->host copy per call.  Replaces the
 * caller-side loops over LoMPC.solve_lompc (lompc.py:137-156; the timing loop
 * of test/test_lompc.py:30-40, the EV loops of price_solver.py:203-204,
 * 280-281) when the caller holds the inputs in host memory.
 *
 * The set owns four packed blocks - pinned host in / out, device in / out - and
 * hands out typed views of them: the caller writes lmbd / lmbd_r / gamma of
 * segment i IN PLACE into the host (or device) views and reads w / cost from
 * the output views, so no staging copy is made on either side.
 *   in  block: [epoch u64 | pad] then per segment lmbd[B_i,3N] lmbd_r[B_i] gamma[B_i]
 *   out block: [summary u64 | pad] then per segment w[B_i,N] cost[B_i]
 *   info block (optional third copy): per segment status[B_i] iters[B_i] kkt_res[B_i]
 * Every segment starts 256-byte aligned.  The worst per-QP status of a call is
 * reduced on the device into the summary word (tagged with the call's epoch,
 * so nothing is cleared between calls) and mapped onto the return code exactly
 * like lompc_solve_batch_host.  All handles must share N and the device.
 * ------------------------------------------------------------------------ */
typedef struct lompc_set lompc_set_t;
#define LOMPC_SET_MAX_SEGMENTS 4

int lompc_set_create(lompc_t* const* handles, int n_handles, const int64_t* batch_sizes, lompc_set_t** out);
int lompc_set_destroy(lompc_set_t* s);
/* Views of segment i (any out-pointer may be NULL).  which: 0 = pinned host blocks, 1 = device blocks. */
int lompc_set_buffers(lompc_set_t* s, int which, int i, double** lmbd, double** lmbd_r, double** gamma,
                      double** w, double** cost);
/* Per-QP diagnostics of segment i (pinned host views; filled by a solve with want_info != 0). */
int lompc_set_info_buffers(lompc_set_t* s, int i, int32_t** status, int32_t** iters, double** kkt_res);
/* Host round trip: copy the in block to the device, solve every segment in one launch, copy the out block
 * (and, with want_info, the info block) back, on the set's own stream.  _async enqueues and returns;
 * lompc_set_wait synchronises and returns LOMPC_ERR_GAMMA / _NEGATIVE / _NOT_CONVERGED like
 * lompc_solve_batch_host.  lompc_set_solve_host = both.  The sequence is captured once as a CUDA graph
 * (environment LOMPC_SET_NO_GRAPH=1: plain stream calls).  Sets of up to 8,192 QPs skip the copy engine
 * altogether: the pinned host blocks are mapped into the device's address space, the kernel loads its inputs
 * from them and stores w / cost / status into them over PCIe ("zero copy": the same bytes cross the bus, but
 * the transfer overlaps the solves and two copy launches disappear; measured 34 us against 44 us per 1,024-QP
 * call).  LOMPC_SET_MAPPED=0 forces the staged H2D copy -> launch -> D2H copy.                        */
int lompc_set_solve_host_async(lompc_set_t* s, int want_info);
int lompc_set_wait(lompc_set_t* s);
int lompc_set_solve_host(lompc_set_t* s, int want_info);
/* Launch only: inputs / outputs are the set's DEVICE blocks, asynchronous on `stream`.  summary_out (DEVICE
 * u64, may be NULL) receives epoch*4 + worst status; the epoch is read from the device in block.     */
int lompc_set_solve_dev(lompc_set_t* s, int want_info, void* stream);
/* The same launch on CALLER-OWNED device blocks that follow the set's layout (lompc_set_bytes gives their sizes,
 * lompc_set_offsets the byte offsets of segment i: lmbd, lmbd_r, gamma inside the in block, w, cost inside the out
 * block): lets a caller keep many batches resident and solve them back to back.  The first 8 bytes of out_block
 * receive epoch*4 + worst status, the epoch being read from the first 8 bytes of in_block.                     */
int lompc_set_solve_dev_at(lompc_set_t* s, void* in_block, void* out_block, void* stream);
int lompc_set_offsets(const lompc_set_t* s, int i, int64_t* offsets /*[5]*/);
/* Copies between the host and device blocks (which: 0 = in block host->device, 1 = out block device->host),
 * asynchronous on `stream`: for callers that mix the host views with lompc_set_solve_dev.            */
int lompc_set_copy(lompc_set_t* s, int which, void* stream);
/* Bytes of one call's host->device / device->host copies (without the info block). */
int64_t lompc_set_bytes(const lompc_set_t* s, int which);

/* ------------------------------------------------------------------------
 * Price loop (reference price_solver.py / price_regularizer.py), batched over
 * G independent groups = (station, EV type, partition) triples.  EVs are sorted
 * by group; group g owns EVs [group_off[g], group_off[g+1]).  All pointers are
 * DEVICE pointers; prices are stored as G rows of 3N doubles (the last N are
 * zero for price type "linear", like lmbd_k in price_solver.py:102-104).
 * ------------------------------------------------------------------------ */

/* PriceSolver.set_charge_levels (price_solver.py:66-77) for every group:
 * y0_rng, gamma_sc, gamma_sm [G] and gamma_i = y_max - y0_i [B]
 * (price_solver.py:201).  Synchronises; LOMPC_ERR_CONSTS if some y0 is outside
 * [0, y_max] (the assert of price_solver.py:71).                             */
int price_group_stats_dev(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off,
                          const double* y0, double* gamma, double* y0_rng, double* gamma_sc,
                          double* gamma_sm, void* stream);

/* PriceSolver._get_w_err (price_solver.py:196-214) for every group: solves the
 * B LoMPC QPs with their group's prices and reduces.  Outputs (any may be
 * NULL): w_avg[G,N], w_err_max[G], w0_err[G], w_avg_err[G], w0[B].            */
int price_w_err_dev(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off,
                    const double* gamma, const double* lmbd, const double* lmbd_r,
                    const double* w_ref, double* w_avg, double* w_err_max, double* w0_err,
                    double* w_avg_err, double* w0, void* stream);

/* PriceSolver._price_gradient_descent_step (price_solver.py:216-246): exact
 * solution of the non-negative QP for every group.  r = 2N or 3N.  lmbd[G,3N]
 * is updated in place; dual_decrease[G] = predicted decrease (:244).          */
int price_step_dev(lompc_t* h, int32_t G, int r, const double* w_ref, const double* w_k,
                   const double* lmbd_r, double* lmbd, double* dual_decrease, int32_t* status,
                   void* stream);

/* PriceSolver._regularize_prices -> PriceRegularizer.solve_price_regularization
 * (price_solver.py:248-255, price_regularizer.py:68-85) in closed form; lmbd is
 * replaced by the regularised prices; price_pre/post = phi(w_k) @ lmbd before
 * and after (price_solver.py:145,147).                                        */
int price_regularize_dev(lompc_t* h, int32_t G, int r, const double* w_k, double* lmbd,
                         double* price_pre, double* price_post, void* stream);

/* PriceRegularizer.solve_price_regularization (price_regularizer.py:68-85) for a
 * constraint matrix of the pattern A = [diag(a_0) ... diag(a_{nb-1})] (a, c:
 * [nb,N]; b: [N]; x out: [nb,N]; DEVICE pointers).  LOMPC_ERR_ARG if a row is
 * infeasible.  Synchronises.                                                 */
int price_lp_rows_dev(int device, int N, int nb, const double* a, const double* b, const double* c,
                      double* x, void* stream);

/* PriceSolver.compute_optimal_prices (price_solver.py:79-174) for every group.
 * prices[G,3N]: in = warm start (prev_prices), out = regularised prices.
 * iters[G] = value of `iter` at exit; price_pre/post[G]; optional (NULL ok)
 * hist_ac/hist_pred[G,hist_cap] = dual_cost_decrease_actual/predicted per
 * iteration; w_k_out[G,N] = LoMPC solution at gamma_sc for the last
 * un-regularised prices.  Returns after the stream has drained.  tol_type_max = 1 for settings "max", 0 for "avg". */
int price_solve_dev(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off, const double* y0,
                    const double* w_ref, const double* lmbd_r, int r, int max_iter,
                    int tol_type_max, double eps_reg, double eps_tol, double* prices,
                    int32_t* iters, double* price_pre, double* price_post, double* w_k_out,
                    double* hist_ac, double* hist_pred, int hist_cap, int32_t* total_iters,
                    void* stream);

/* compute_optimal_prices along the reference's WARM-START CHAIN, for S stations with P partitions
 * each: the PriceSolver object of an EV type is shared by its partitions, so partition p starts from
 * the prices of the last non-empty partition solved before it (price_solver.py:56,104,166;
 * charging_station.py:273-304).  Groups are numbered partition-major, g = p*S + s; group_off[P*S+1],
 * w_ref[P*S,N], lmbd_r[P*S], iters / price_pre / price_post[P*S].  prev_prices[S,3N] is the carried
 * warm start (in: PriceSolver.prev_prices of every station, out: the same after the step);
 * prices[P*S,3N] receives every group's regularised prices (zeros for an empty group,
 * charging_station.py:270; its iters = -1).  One CTA per station runs its P loops back to back, so
 * stations do not wait for each other (N = 12, 24; N = 48, 96 with the parametric loop; otherwise the same
 * chain runs as P phase-split loops, one per partition slice).  station_order[S] (may be NULL) = a permutation of the stations:
 * the order in which CTAs pick them up (longest expected chains first shortens the tail).
 * Synchronises; max_group_iters = length of the longest loop.                                       */
int price_solve_chain_dev(lompc_t* h, int32_t S, int32_t P, int64_t B, const int32_t* group_off, const double* y0,
                          const double* w_ref, const double* lmbd_r, int r, int max_iter, int tol_type_max,
                          double eps_reg, double eps_tol, double* prev_prices, double* prices, int32_t* iters,
                          double* price_pre, double* price_post, const int32_t* station_order,
                          int32_t* max_group_iters, void* stream);

/* price_solve_dev / price_solve_chain_dev run, for the compiled horizons (N = 12, 24; N = 48, 96 with the parametric
 * loop), ONE kernel that iterates every group to convergence on the device, for either tolerance type.  Loop modes:
 * 0 = automatic (the parametric loop); 1 = the phase-split loop below (any N; the path a multi-GPU caller drives);
 * 2 = the PARAMETRIC loop, one warp per group: the EVs of a group differ only in gamma and the QP's solution is
 * piecewise affine in it, so only the extreme EVs, the virtual EV (gamma_sc) and the EVs that bracket a change of
 * active set are solved and the rest is interpolated (SURVEY.md 8 row f3; price_solver.py:196-214 - for "max" the
 * error of an interpolated stretch of EVs is convex in gamma, so its largest value is at the stretch's first or last
 * EV); 3 = the thread-per-EV loop, one CTA per group (N = 12, 24; the phase-split loop at other horizons).  All give
 * the same iteration counts and prices up to rounding.  price_last_qp_solves = LoMPC QPs solved by the last fused call;
 * price_last_cycles(h, 5) = groups of the last parametric call whose pool of 32 pivot slots ran out (about one group in
 * 10^4 on a fleet's first step; the EVs of the stuck intervals are then solved one by one: exact, informational),
 * price_last_cycles(h, 6) = groups of the last device-resident call whose price step (price_solver.py:216-246) ended
 * inexact (its primal-dual active-set iteration cycles on about one degenerate step in 10^6; it then falls back to
 * Lawson-Hanson's iteration, and only a cap hit THERE counts), price_last_cycles(h, 7) = LoMPC solves of that call
 * that ended without status OK (both 0 in every run so far; the Python mirror warns on either),
 * price_last_cycles(h, 8) = groups that took the fallback (informational).
 * price_debug_force_nnqp_fallback: test hook - non-zero sends EVERY price step of the current device through the
 * fallback (the parity tests of the price loop are run both ways); price_debug_pivot_pool: test hook - the pivot
 * slots the parametric loop may use (4..32, default 32), so that a test can make slot shortage the common case;
 * price_debug_record_errors: test hook - while set (both non-NULL: device arrays [G] of the current device; both NULL:
 * off), every group of a parametric "max" loop writes the w_err_max and w_avg_err of its last convergence test
 * (price_solver.py:196-214).  With max_iter = 1 these are the errors at the warm-start prices. */
int price_set_loop_mode(lompc_t* h, int mode);
int64_t price_last_qp_solves(const lompc_t* h);
/* SM cycles of the last fused call summed over groups: which = 0 LoMPC passes, 1 price steps. */
int64_t price_last_cycles(const lompc_t* h, int which);
int price_debug_force_nnqp_fallback(int on);
int price_debug_pivot_pool(int slots);
int price_debug_record_errors(double* w_err_max, double* w_avg_err);
/* Test hook: non-zero makes every device-resident loop take the code path of fleet-scale launches (the compact price
 * step: recursions unrolled 4 stages per trip; automatic from 1,184 groups / stations per launch). */
int price_debug_force_compact_step(int on);

/* The same loop cut into the phases between which a multi-GPU caller
 * all-reduces, for EVs sharded over ranks (each rank passes its LOCAL EVs and
 * LOCAL group_off; a group may be empty on a rank).  Per handle one session at
 * a time.  Caller-owned DEVICE buffers carry the cross-rank quantities:
 *   stat_min/max/sum/cnt[G]  after price_shard_begin : all-reduce MIN/MAX/SUM/SUM
 *   w_sum[G,N]               after price_shard_ev_phase : all-reduce SUM
 *   err_max[G]               after price_shard_ev_phase : all-reduce MAX ("max" tolerance type only)
 * (price_solver.py:66-77 and :199-210 are the reductions being distributed).
 * price_shard_start validates the REDUCED statistics (the assert of price_solver.py:71), so a y0 outside
 * [0, y_max] makes every rank return LOMPC_ERR_CONSTS together (a rank-local check would leave the others
 * waiting in the next all-reduce).
 * price_shard_group_phase runs the convergence test, the price step and the
 * gamma_sc solve on every rank identically (replicated, deterministic) and
 * returns the number of still-active groups; stop when it is 0.              */
int price_shard_begin(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off, const double* y0,
                      const double* w_ref, const double* lmbd_r, int r, int max_iter, int tol_type_max,
                      double eps_reg, double eps_tol, double* prices, int32_t* iters, double* stat_min,
                      double* stat_max, double* stat_sum, double* stat_cnt, double* w_sum, double* err_max,
                      double* hist_ac, double* hist_pred, int hist_cap, void* stream);
int price_shard_start(lompc_t* h, void* stream);
int price_shard_ev_phase(lompc_t* h, void* stream);
int price_shard_group_phase(lompc_t* h, int it, int32_t* n_active, void* stream);
/* The same phase WITHOUT the host round trip, for a loop that keeps the GPU fed: _async only enqueues (the
 * number of still-active groups is published into a pinned ring by the device); price_shard_poll returns 1 and
 * that number once iteration `it` has been published, 0 if not yet (wait = 0), or spins on the pinned word
 * until it has (wait != 0) - it never makes a synchronising CUDA call.  Groups that have converged are skipped
 * on the device, so iterations enqueued beyond convergence cost launches only.  The ring holds 64 iterations:
 * poll iteration `it` before enqueuing iteration it + 64.                                              */
int price_shard_group_phase_async(lompc_t* h, int it, void* stream);
int price_shard_poll(lompc_t* h, int it, int wait, int32_t* n_active);
int price_shard_finish(lompc_t* h, double* price_pre, double* price_post, double* w_k_out, void* stream);

/* The aggregate exchange WITHOUT a collective library call: the per-group partial sums travel over NVLink peer
 * memory.  Every rank allocates one region with lompc_ipc_alloc (>= 1024 + 2*G*N*8 bytes; the 64-byte CUDA IPC
 * handle is what the ranks exchange, e.g. with one all_gather at set-up), opens the other ranks' regions with
 * lompc_ipc_open and hands the `world` device pointers (its own at index `rank`) to price_shard_attach_peers.
 * From then on price_shard_ev_phase writes the partial sums into the rank's own region and raises a flag on every
 * rank, and price_shard_group_phase_async starts by waiting for the flags of all ranks and adding the partials in
 * rank order straight out of the peers' memory (bit-identical on every rank): the caller does NOT all-reduce w_sum
 * any more ("avg" tolerance type; with "max" the session falls back to the caller's all-reduces).  A rank that
 * does not deliver within 2 s makes price_shard_finish return LOMPC_ERR_CUDA instead of hanging the GPU.
 * world <= 1 detaches.  One GPU per rank (kernels of different ranks wait on each other).                    */
int lompc_ipc_alloc(int device, size_t bytes, void** dev_ptr, unsigned char* handle_out /*[64]*/);
int lompc_ipc_open(int device, const unsigned char* handle /*[64]*/, void** dev_ptr);
int lompc_ipc_close(int device, void* dev_ptr);
int lompc_ipc_free(int device, void* dev_ptr);
int price_shard_attach_peers(lompc_t* h, int rank, int world, void* const* regions, size_t region_bytes);
/* 1 if the current / last session exchanges through peer memory (the caller then skips its all-reduce). */
int price_shard_uses_peers(const lompc_t* h);
/* Call after price_shard_begin when THIS rank holds every EV of every group (world size 1, the reduction of
 * price_solver.py:199-210 has nothing to add): the group phase then forms the per-group column sums itself (same
 * additions in EV order) and price_shard_ev_phase neither launches the column-sum kernel nor fills w_sum / err_max.
 * Ignored while peers are attached.  Session-scoped: price_shard_begin resets it. */
int price_shard_local_sums(lompc_t* h, int on);

/* PriceSolver.get_w0_price0 (price_solver.py:272-285) for every group:
 * w0[B] = first-step charge of each EV, price0[G] = mean first-step price.    */
int price_w0_price0_dev(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off,
                        const double* gamma, const double* lmbd, const double* lmbd_r,
                        double* w0, double* price0, void* stream);

/* Measures the device's FP64 FMA peak (TFLOP/s, FMA = 2 flops) with a
 * register-resident DFMA chain kernel: the roofline denominator of this
 * FP64-bound path (MEASURED_PEAKS.json has no FP64 figure).                 */
int lompc_measure_fp64_peak(int device, int iters, double* tflops_out, double* ms_out);

/* Number of kernels this library has launched since load (bench.py's
 * gpu_launches claim is read from here).                                    */
int64_t lompc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* LOMPC_B200_H */
