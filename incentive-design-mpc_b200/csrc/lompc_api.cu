// C ABI of the B200-native LoMPC hot path (see include/lompc_b200.h).
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>

#include "lompc_common.cuh"
#include "lompc_solve.cuh"
#include "lompc_solve_reg.cuh"
#include "lompc_vjp.cuh"
#include "lompc_price.cuh"
#include "lompc_price_fused.cuh"
#include "lompc_price_warp.cuh"

namespace {

constexpr bool kParametricLoopByDefault = true;  // parity: tests/test_fullsize_gpu.py, tools/compare_loop_modes.py; timing: DESIGN.md 4
std::atomic<bool> g_force_compact_step{false};  // test hook: price_debug_force_compact_step()
constexpr int kRingSlots = 64;  // iterations the pinned n_active ring of the sharded price loop can hold

thread_local char g_cuda_err[256] = "";
std::atomic<int64_t> g_launches{0};

int cuda_fail(cudaError_t e, const char* what) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
  return LOMPC_ERR_CUDA;
}
#define CK(call)                                   \
  do {                                             \
    cudaError_t e__ = (call);                      \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

// settings.py:7-9
constexpr double kMinMaxBatSoc = 0.75;
constexpr double kMaxMaxBatSoc = 0.9;
constexpr double kMaxBatChargeRate = 0.25;

}  // namespace

namespace lompc_detail {
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
int cuda_fail(cudaError_t e, const char* what) { return ::cuda_fail(e, what); }
}  // namespace lompc_detail

struct PriceSession {  // state of one (possibly sharded) compute_optimal_prices run
  bool active = false;
  int G = 0, max_iter = 0, ev_passes = 0;
  int64_t B = 0;
  const int32_t* group_off = nullptr;
  int32_t *group_of = nullptr, *skip = nullptr, *nst = nullptr, *nact = nullptr, *empty = nullptr;
  double *gamma = nullptr, *w_ev = nullptr, *err_ev = nullptr, *y0_rng = nullptr, *gamma_sc = nullptr,
         *gamma_sm = nullptr, *w_k = nullptr, *e_avg = nullptr, *e_0 = nullptr, *dual_cost = nullptr,
         *cost_new = nullptr, *lamdiff = nullptr, *decp = nullptr;
  unsigned char* wsb = nullptr;
  double *stat_min = nullptr, *stat_max = nullptr, *stat_sum = nullptr, *stat_cnt = nullptr;
  lompc::PriceArgs p;
  bool peer = false;            // the aggregate is exchanged through peer memory (price_shard_attach_peers)
  bool local_sums = false;      // this rank holds every EV: column sums inside the group step (price_shard_local_sums)
  unsigned long long tag0 = 0;  // flag value of iteration 0 of this session, minus one
};

struct lompc_handle {
  lompc::Consts cs;
  int device;
  int max_iter;
  double tol;
  double delta;
  // grow-only device workspace for the _host entry points
  void* ws;
  size_t ws_bytes;
  cudaStream_t hstream;       // stream of the host entry points (non-blocking, created on first use)
  int32_t* hst;               // pinned status buffer used when the caller passes status = NULL
  size_t hst_cap;
  int64_t pending_B;          // batch of the enqueued, not yet awaited host call
  const int32_t* pending_status;
  // grow-only device workspace of the price loop + pinned poll word
  int variant;  // 0 auto, 1 = any-N shared-memory kernel, 2.. = register-kernel variants
  int loop_mode;  // price loop: 0 auto (fused one-CTA-per-group kernel when compiled for N), 1 = phase-split host loop
  int last_qp_failures;               // LoMPC solves of that loop that ended without status OK (never observed)
  int last_nnqp_fallbacks;            // groups of that loop that took the Lawson-Hanson fallback of the price step
  int last_nnqp_cap_hits;             // groups of the last device-resident loop whose price step hit its active-set cap
  int last_pivot_overflows;           // groups of the last parametric loop whose pivot pool overflowed (expected 0)
  unsigned long long last_qp_solves;  // LoMPC QPs solved by the last fused price loop
  unsigned long long last_cycles[5];  // its SM cycles in the LoMPC passes / the price steps (summed over groups),
                                      // K1 iterations summed over its solves, warp passes with no K1 iteration, warp passes
  void* pws;
  size_t pws_bytes;
  int32_t* poll;  // pinned host
  int32_t* ring;  // pinned host ring of (tag, n_active) pairs, written by publish_active_kernel
  lompc::PeerView peers;        // world == 0: not attached
  size_t peer_region_bytes;
  unsigned long long peer_sessions;
  void* rws;      // reduction buffers of the single-GPU price loop
  size_t rws_bytes;
  // side stream of the pipelined phase-split loop (price_shard_group_phase_async): the gamma_sc solve and the
  // bookkeeping of iteration `it` run beside the EV phase of iteration it + 1 (created on first use)
  cudaStream_t side;
  cudaEvent_t ev_fork, ev_join;
  bool side_pending;  // work enqueued on `side` that the caller's stream has not waited for yet
  PriceSession ses;
};

namespace {

// One bit per device ordinal (< 64): "this kernel's shared-memory opt-in has been set on that device".
// Devices beyond 63 simply set the attribute on every launch.
inline bool device_flag_test(const std::atomic<uint64_t>& m, int dev) {
  return dev < 64 && ((m.load(std::memory_order_acquire) >> dev) & 1u);
}
inline void device_flag_set(std::atomic<uint64_t>& m, int dev) {
  if (dev < 64) m.fetch_or(uint64_t(1) << dev, std::memory_order_release);
}

int ensure_ws(lompc_handle* h, size_t bytes) {
  if (h->ws_bytes >= bytes) return LOMPC_OK;
  if (h->ws) CK(cudaFree(h->ws));
  h->ws = nullptr;
  h->ws_bytes = 0;
  size_t want = bytes + bytes / 4;
  CK(cudaMalloc(&h->ws, want));
  h->ws_bytes = want;
  return LOMPC_OK;
}

// Register-resident kernel for the compile-time horizons (variants: see lompc_set_kernel_variant).
template <int N, int NSEG, int T, int MINB, bool GREG>
int launch_solve_reg(const lompc_handle* h, const lompc::SolveArgs& a, cudaStream_t stream) {
  constexpr size_t smem = lompc::RegSmem<N, NSEG, T, GREG>::bytes;
  // the opt-in is a per-device (per-context) attribute of the function: one flag per device ordinal
  static std::atomic<uint64_t> configured{0};
  if (!device_flag_test(configured, h->device)) {
    CK(cudaFuncSetAttribute(lompc::lompc_solve_reg_kernel<N, NSEG, T, MINB, GREG>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    device_flag_set(configured, h->device);
  }
  const int64_t blocks = (a.B + T - 1) / T;
  lompc::SolveArgs av = a;
  av.vec16 = (reinterpret_cast<uintptr_t>(a.lmbd) % 16 == 0) && (a.lmbd_stride % 2 == 0) &&
             (reinterpret_cast<uintptr_t>(a.w_out) % 16 == 0);
  lompc::lompc_solve_reg_kernel<N, NSEG, T, MINB, GREG><<<(unsigned)blocks, T, smem, stream>>>(h->cs, av);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CK(cudaGetLastError());
  return LOMPC_OK;
}

// The register kernel with the rows moved by the bulk-copy engine (lompc_solve_reg_tma_kernel): plain batches only.
inline bool tma_rows_ok(const lompc::SolveArgs& a, int N) {
  return !a.group_of && !a.skip && !a.w_init && !a.err_out && !a.w0_out && !a.price0_out && a.w_out &&
         a.lmbd_stride == 3 * N && a.lmbd_r_stride == 1 && reinterpret_cast<uintptr_t>(a.lmbd) % 16 == 0 &&
         reinterpret_cast<uintptr_t>(a.w_out) % 16 == 0;
}

template <int N, int NSEG, int T, int MINB, bool OUT_ALIAS>
int launch_solve_reg_tma(const lompc_handle* h, const lompc::SolveArgs& a, cudaStream_t stream) {
  constexpr size_t smem = lompc::RegTmaSmem<N, NSEG, T, OUT_ALIAS>::bytes;
  static_assert(smem <= 227 * 1024, "shared memory of one CTA");
  static std::atomic<uint64_t> configured{0};
  if (!device_flag_test(configured, h->device)) {
    CK(cudaFuncSetAttribute(lompc::lompc_solve_reg_tma_kernel<N, NSEG, T, MINB, OUT_ALIAS>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    device_flag_set(configured, h->device);
  }
  const int64_t blocks = (a.B + T - 1) / T;
  lompc::lompc_solve_reg_tma_kernel<N, NSEG, T, MINB, OUT_ALIAS><<<(unsigned)blocks, T, smem, stream>>>(h->cs, a);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CK(cudaGetLastError());
  return LOMPC_OK;
}

template <int N, int NSEG>
int launch_solve_reg_variant(const lompc_handle* h, const lompc::SolveArgs& a, cudaStream_t stream) {
  if (h->variant == 9 && tma_rows_ok(a, N)) {  // bulk-copy rows (batches that are not plain rows: the default below)
    if constexpr (NSEG > 1)
      return launch_solve_reg_tma<N, NSEG, 128, 2, true>(h, a, stream);
    else
      return launch_solve_reg_tma<N, NSEG, 64, 4, false>(h, a, stream);
  }
  switch (h->variant) {
    // (the other shapes of round 1's sweep - 64x4 with g in shared memory, 128x3, 64x5, 128x2 - lost everywhere and
    // are no longer compiled; their numbers are kept)
    case 2: case 3: case 5: case 6: return LOMPC_ERR_ARG;
    case 4: return launch_solve_reg<N, NSEG, 64, 4, true>(h, a, stream);
    case 7: return launch_solve_reg<N, NSEG, 256, 1, true>(h, a, stream);
    default:
      // measured on B200 (tools/sweep_variants.sh, r1j): W, d AND g in registers (255 registers, no spills; KK,
      // kappa, parked iterate [, 1/(d+Q)] in shared memory), 8 warps per SM.  Small EV: 4 CTAs of 64 threads (the
      // 24 KB loop body fits the instruction cache; small CTAs keep the tail short).  Large EV: the unrolled loop
      // body is 50 KB and the kernel is instruction-fetch bound (ncu: no_instruction = 36 % of the stall samples,
      // spread evenly over the body) unless the warps of an SM run in step and share the fetched lines: ONE CTA of
      // 256 threads per SM (+17..21 % over 4 x 64) once the grid fills the GPU; latency-bound grids keep 64.
      // Grids that fill the GPU at N = 24: rows by the bulk-copy engine (lompc_solve_reg_tma_kernel).  Measured
      // (tools/time_k1.py, us per launch, per-thread loads / bulk copies): 65,536 QPs 41.0 / 38.9 small, 65.5 / 59.4
      // large; 262,144: 116.7 / 104.4, 202.8 / 182.3; 524,288: 215.0 / 188.4 (2.44 -> 2.78 G QP/s), 389.1 / 344.1
      // (1.35 -> 1.52 G).  Below that (16,384: 18.4 / 18.4, 30.7 / 32.8) and at N = 12, where a row is 288 B and the
      // two CTA barriers cost more than the copies save (524,288 QPs: 94.4 / 110.6 us), the loads stay per-thread.
      // CTA shape with bulk-copied rows (524,288 QPs): small EV 64 x 4: 188.4 us, 128 x 2: 194.6, 256 x 1: 229.3; large
      // EV 128 x 2: 325.6 us (1.61 G QP/s), 64 x 4: 327.7, 256 x 1: 340.0 - two CTAs per SM cover each other's load
      // and store phases, which the one-CTA shape the per-thread-load kernel prefers cannot.
      if constexpr (N == 24) {
        if (a.B >= 65536 && tma_rows_ok(a, N)) {
          if constexpr (NSEG > 1)
            return launch_solve_reg_tma<N, NSEG, 128, 2, true>(h, a, stream);
          else
            return launch_solve_reg_tma<N, NSEG, 64, 4, false>(h, a, stream);
        }
      }
      if (NSEG > 1 && a.B >= 65536) return launch_solve_reg<N, NSEG, 256, 1, true>(h, a, stream);
      return launch_solve_reg<N, NSEG, 64, 4, true>(h, a, stream);
  }
}

// Batches below this many QPs go to the warp-cooperative kernel (lompc_solve_warp.cuh) in automatic mode: one QP
// per thread needs ~150 k QPs to fill the GPU (148 SMs x 8 warps x 32 lanes x a few waves), below that
// its warps sit alone on their schedulers and the time-parallel sweeps win.  Measured (tools/time_k1.py, N = 24,
// us per launch, warp / thread kernel): 512 QPs 12.3 / 16.4 small, 16.4 / 22.5 large; 4,096: 14.3 / 16.4,
// 18.4 / 24.6; 8,192: 20.5 / 18.4, 28.6 / 28.7; 16,384: 30.7 / 18.4, 43.0 / 30.7.
// N = 12: 4,096 QPs 10.2 / 10.2 (small), 16,384: 16.4 / 12.3.  N = 48 and 96 have no register kernel: the warp kernel
// beats the any-N shared-memory kernel at every batch size measured (16,384 QPs, small EV: 57 vs 92 us at N = 48,
// 119 vs 457 us at N = 96; 65,536: 197 vs 231, 430 vs 1,584), so it takes all of them.
inline int64_t warp_kernel_max_batch(int N) {
  return N == 12 ? 4096 : (N == 24 ? 6144 : INT64_MAX);
}

// Threads per CTA of the one-QP-per-thread kernels with per-stage columns in shared memory ([k*T + t], qp_bytes per
// QP): the size that keeps most warps resident per SM (shared memory is the limit), capped at 128; small batches use
// small blocks so that more SMs take part.
int any_n_cta_width(size_t qp_bytes, int64_t B) {
  int T = 32;
  {
    size_t best = 0;
    for (int cand = 32; cand <= 128; cand <<= 1) {
      const size_t per_cta = qp_bytes * cand + 1024;
      const size_t warps = (size_t)(227 * 1024 / per_cta) * (cand / 32);
      if (warps >= best && per_cta <= 227 * 1024) {
        best = warps;
        T = cand;
      }
    }
  }
  while (T > 32 && (B + T - 1) / T < 148) T >>= 1;
  // Horizons whose columns do not fit 32 threads (K1: N > 129 large EV, N > 151 small EV): the largest power of two
  // that fits.  The kernels have no barrier and their layout is [k*T + t], so any T works; at T = 1 every N <= 4096
  // fits.  (The throughput of these partial-warp CTAs has not been measured.)
  while (T > 1 && qp_bytes * T > 227 * 1024) T >>= 1;
  return T;
}

template <int NSEG>
int launch_solve(const lompc_handle* h, const lompc::SolveArgs& a, cudaStream_t stream) {
  const int N = h->cs.N;
  {
    // plain batched solves and the group mode of the phase-split price loop (shared prices, skip mask, warm
    // starts); the fused epilogues (error norm, first-step price) stay on the thread kernels
    const bool plain = !a.err_out && !a.w0_out && !a.price0_out && a.w_out;
    const int spl = 3;
    const bool want = h->variant == 8 || (h->variant == 0 && a.B <= warp_kernel_max_batch(N));
    if (plain && want && lompc_detail::warp_kernel_supports(N, spl)) {
      lompc::WarpArgs wa;
      memset(&wa, 0, sizeof(wa));
      wa.nsegs = 1;
      wa.seg[0].cs = h->cs;
      wa.seg[0].a = a;
      return lompc_detail::launch_k1_warp(h->device, N, spl, wa, stream);
    }
  }
  if (h->variant != 1) {
    if (N == 24) return launch_solve_reg_variant<24, NSEG>(h, a, stream);
    if (N == 12) return launch_solve_reg_variant<12, NSEG>(h, a, stream);
  }
  const int T = any_n_cta_width(lompc::SmemLayout<NSEG>::bytes(N, 1), a.B);
  const size_t smem = lompc::SmemLayout<NSEG>::bytes(N, T);
  if (smem > 227 * 1024) return LOMPC_ERR_ARG;
  static std::atomic<uint64_t> configured{0};  // per device ordinal (the attribute is per context)
  if (!device_flag_test(configured, h->device)) {
    CK(cudaFuncSetAttribute(lompc::lompc_solve_kernel<NSEG>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    device_flag_set(configured, h->device);
  }
  const int64_t blocks = (a.B + T - 1) / T;
  lompc::lompc_solve_kernel<NSEG><<<(unsigned)blocks, T, smem, stream>>>(h->cs, a);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CK(cudaGetLastError());
  return LOMPC_OK;
}

template <int NSEG>
int launch_vjp(const lompc_handle* h, const lompc::VjpArgs& a, cudaStream_t stream) {
  const int N = h->cs.N;
  const size_t qp_bytes = (size_t)lompc::kVjpArrays * N * sizeof(double);
  const int T = any_n_cta_width(qp_bytes, a.B);
  const size_t smem = qp_bytes * T;
  if (smem > 227 * 1024) return LOMPC_ERR_ARG;
  static std::atomic<uint64_t> configured{0};  // per device ordinal (the attribute is per context)
  if (!device_flag_test(configured, h->device)) {
    CK(cudaFuncSetAttribute(lompc::lompc_vjp_kernel<NSEG>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    device_flag_set(configured, h->device);
  }
  const int64_t blocks = (a.B + T - 1) / T;
  lompc::lompc_vjp_kernel<NSEG><<<(unsigned)blocks, T, smem, stream>>>(h->cs, a);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CK(cudaGetLastError());
  return LOMPC_OK;
}

}  // namespace

namespace lompc_detail {
HandleView handle_view(const lompc_t* h) { return HandleView{&h->cs, h->device, h->max_iter, h->tol, h->variant}; }
int launch_k1(const lompc_t* h, const lompc::SolveArgs& a, cudaStream_t s) {
  return h->cs.large ? launch_solve<4>(h, a, s) : launch_solve<1>(h, a, s);
}
}  // namespace lompc_detail

extern "C" {

const char* lompc_version(void) { return "lompc_b200 0.2 (sm_100a)"; }

const char* lompc_strerror(int code) {
  switch (code) {
    case LOMPC_OK: return "ok";
    case LOMPC_ERR_CONSTS: return "invalid LoMPC constants (lompc.py:36-38)";
    case LOMPC_ERR_ARG: return "invalid argument";
    case LOMPC_ERR_CUDA: return "CUDA error";
    case LOMPC_ERR_GAMMA: return "gamma > y_max (lompc.py:87)";
    case LOMPC_ERR_NEGATIVE: return "negative value for a nonneg parameter (lompc.py:78-82)";
    case LOMPC_ERR_NOT_CONVERGED: return "solver did not converge";
    case LOMPC_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
    default: return "unknown error";
  }
}

const char* lompc_last_cuda_error(void) { return g_cuda_err; }

int lompc_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int64_t lompc_launch_count(void) { return g_launches.load(); }

int lompc_create(int N, double delta, double theta, double y_max, double w_max, int ev_type,
                 int device, lompc_t** out) {
  if (!out || N < 1 || N > 4096) return LOMPC_ERR_ARG;
  *out = nullptr;
  // lompc.py:36-38
  if (!(y_max >= kMinMaxBatSoc && y_max <= kMaxMaxBatSoc)) return LOMPC_ERR_CONSTS;
  if (!(w_max >= 0.0 && w_max <= kMaxBatChargeRate)) return LOMPC_ERR_CONSTS;
  if (ev_type != LOMPC_EV_SMALL && ev_type != LOMPC_EV_LARGE) return LOMPC_ERR_CONSTS;
  if (!(w_max > 0.0) || !(theta > 0.0) || !(delta > 0.0)) return LOMPC_ERR_ARG;
  if (lompc_device_count() <= device || device < 0) return LOMPC_ERR_NO_DEVICE;

  lompc_handle* h = new (std::nothrow) lompc_handle();
  if (!h) return LOMPC_ERR_ARG;
  lompc::Consts& cs = h->cs;
  memset(&cs, 0, sizeof(cs));
  cs.N = N;
  cs.large = ev_type == LOMPC_EV_LARGE;
  cs.delta = delta;
  cs.theta = theta;
  cs.w_max = w_max;
  cs.y_max = y_max;
  cs.c = 2.0 * delta * theta * theta;       // lompc.py:71
  cs.q_scale = 3.0 * theta / (4.0 * w_max);  // lompc.py:67
  cs.theta2 = theta * theta;
  if (!cs.large) {
    cs.d_base = 2.0 * theta * theta / 0.81;  // theta^2 * sum_squares(w / 0.9), lompc.py:107
    cs.nseg = 1;
    cs.brk[0] = 0.0;
    cs.brk[1] = w_max;
    cs.slope[0] = 0.0;
  } else {
    // (theta*w_max)^2 * sum max(0, x-.125, 1.5x-.375, 2x-.75), x = w/w_max  (lompc.py:109-116)
    cs.d_base = 0.0;
    cs.nseg = 4;
    const double brk_rel[5] = {0.0, 0.125, 0.5, 0.75, 1.0};
    const double slope_rel[4] = {0.0, 1.0, 1.5, 2.0};
    const double per_w = (theta * w_max) * (theta * w_max) / w_max;
    for (int i = 0; i <= 4; ++i) cs.brk[i] = brk_rel[i] * w_max;
    cs.brk[4] = w_max;
    for (int j = 0; j < 4; ++j) cs.slope[j] = per_w * slope_rel[j];
  }
  h->device = device;
  h->max_iter = 200;
  h->tol = 1e-11;
  h->delta = delta;
  h->ws = nullptr;
  h->ws_bytes = 0;
  h->hstream = nullptr;
  h->hst = nullptr;
  h->hst_cap = 0;
  h->pending_B = 0;
  h->pending_status = nullptr;
  h->variant = 0;
  h->loop_mode = 0;
  h->last_qp_solves = 0;
  h->last_pivot_overflows = 0;
  h->last_nnqp_cap_hits = 0;
  h->last_qp_failures = 0;
  h->last_nnqp_fallbacks = 0;
  for (auto& c : h->last_cycles) c = 0;
  h->pws = nullptr;
  h->pws_bytes = 0;
  h->poll = nullptr;
  h->ring = nullptr;
  memset(&h->peers, 0, sizeof(h->peers));
  h->peer_region_bytes = 0;
  h->peer_sessions = 0;
  h->rws = nullptr;
  h->rws_bytes = 0;
  *out = h;
  return LOMPC_OK;
}

int lompc_destroy(lompc_t* h) {
  if (!h) return LOMPC_OK;
  cudaSetDevice(h->device);
  if (h->hstream) {
    cudaStreamSynchronize(h->hstream);
    cudaStreamDestroy(h->hstream);
  }
  if (h->side) {
    cudaStreamSynchronize(h->side);
    cudaStreamDestroy(h->side);
    cudaEventDestroy(h->ev_fork);
    cudaEventDestroy(h->ev_join);
  }
  if (h->hst) cudaFreeHost(h->hst);
  if (h->ws) cudaFree(h->ws);
  if (h->pws) cudaFree(h->pws);
  if (h->poll) cudaFreeHost(h->poll);
  if (h->ring) cudaFreeHost(h->ring);
  if (h->rws) cudaFree(h->rws);
  delete h;
  return LOMPC_OK;
}

double lompc_sc_modulus(const lompc_t* h) { return h ? h->cs.c : NAN; }

int lompc_set_options(lompc_t* h, int max_iter, double tol) {
  if (!h || max_iter < 1 || !(tol > 0.0)) return LOMPC_ERR_ARG;
  h->max_iter = max_iter;
  h->tol = tol;
  return LOMPC_OK;
}

int lompc_set_kernel_variant(lompc_t* h, int variant) {
  if (!h || variant < 0 || variant > 9 || variant == 2 || variant == 3 || variant == 5 || variant == 6) return LOMPC_ERR_ARG;
  h->variant = variant;
  return LOMPC_OK;
}

int price_set_loop_mode(lompc_t* h, int mode) {
  if (!h || mode < 0 || mode > 3) return LOMPC_ERR_ARG;
  h->loop_mode = mode;
  return LOMPC_OK;
}

int64_t price_last_qp_solves(const lompc_t* h) { return h ? (int64_t)h->last_qp_solves : 0; }

int price_debug_force_nnqp_fallback(int on) {
  CK(cudaMemcpyToSymbol(lompc::g_nnqp_force_fallback, &on, sizeof(int)));
  return LOMPC_OK;
}

int price_debug_force_compact_step(int on) {
  g_force_compact_step.store(on != 0, std::memory_order_relaxed);
  return LOMPC_OK;
}

int price_debug_pivot_pool(int slots) {
  if (slots < 4 || slots > 32) return LOMPC_ERR_ARG;
  CK(cudaMemcpyToSymbol(lompc::g_pivot_pool, &slots, sizeof(int)));
  return LOMPC_OK;
}

int price_debug_record_errors(double* w_err_max, double* w_avg_err) {
  if (!w_err_max != !w_avg_err) return LOMPC_ERR_ARG;
  CK(cudaMemcpyToSymbol(lompc::g_record_err_max, &w_err_max, sizeof(double*)));
  CK(cudaMemcpyToSymbol(lompc::g_record_err_avg, &w_avg_err, sizeof(double*)));
  return LOMPC_OK;
}

int64_t price_last_cycles(const lompc_t* h, int which) {
  if (h && which == 5) return h->last_pivot_overflows;
  if (h && which == 6) return h->last_nnqp_cap_hits;
  if (h && which == 7) return h->last_qp_failures;
  if (h && which == 8) return h->last_nnqp_fallbacks;
  return (h && which >= 0 && which < 5) ? (int64_t)h->last_cycles[which] : 0;
}

int lompc_solve_batch_dev(lompc_t* h, int64_t B, const double* lmbd, int64_t lmbd_stride,
                          const double* lmbd_r, int64_t lmbd_r_stride, const double* gamma,
                          double* w_out, double* cost_out, int32_t* status, int32_t* iters,
                          double* kkt_res, void* stream) {
  if (!h || B < 0 || !lmbd || !lmbd_r || !gamma || !w_out || !cost_out) return LOMPC_ERR_ARG;
  if (lmbd_stride != 0 && lmbd_stride < 3 * (int64_t)h->cs.N) return LOMPC_ERR_ARG;
  if (lmbd_r_stride != 0 && lmbd_r_stride != 1) return LOMPC_ERR_ARG;
  if (B == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  lompc::SolveArgs a;
  a.B = B;
  a.lmbd = lmbd;
  a.lmbd_stride = lmbd_stride;
  a.lmbd_r = lmbd_r;
  a.lmbd_r_stride = lmbd_r_stride;
  a.gamma = gamma;
  a.w_out = w_out;
  a.cost_out = cost_out;
  a.status = status;
  a.iters = iters;
  a.kkt_res = kkt_res;
  a.max_iter = h->max_iter;
  a.tol = h->tol;
  a.group_of = nullptr;
  a.skip = nullptr;
  a.w_ref = nullptr;
  a.err_out = nullptr;
  a.w0_out = nullptr;
  a.price0_out = nullptr;
  a.w_init = nullptr;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return h->cs.large ? launch_solve<4>(h, a, s) : launch_solve<1>(h, a, s);
}

int lompc_vjp_dev(lompc_t* h, int64_t B, const double* lmbd, int64_t lmbd_stride, const double* lmbd_r,
                  int64_t lmbd_r_stride, const double* gamma, const double* w, const double* grad_w,
                  const double* grad_cost, double* grad_lmbd, double* grad_lmbd_r, double* grad_gamma,
                  int32_t* status, void* stream) {
  if (!h || B < 0 || !lmbd || !lmbd_r || !gamma || !w) return LOMPC_ERR_ARG;
  if (lmbd_stride != 0 && lmbd_stride < 3 * (int64_t)h->cs.N) return LOMPC_ERR_ARG;
  if (lmbd_r_stride != 0 && lmbd_r_stride != 1) return LOMPC_ERR_ARG;
  if (B == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  lompc::VjpArgs a;
  a.B = B;
  a.lmbd = lmbd;
  a.lmbd_stride = lmbd_stride;
  a.lmbd_r = lmbd_r;
  a.lmbd_r_stride = lmbd_r_stride;
  a.gamma = gamma;
  a.w = w;
  a.grad_w = grad_w;
  a.grad_cost = grad_cost;
  a.grad_lmbd = grad_lmbd;
  a.grad_lmbd_r = grad_lmbd_r;
  a.grad_gamma = grad_gamma;
  a.status = status;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return h->cs.large ? launch_vjp<4>(h, a, s) : launch_vjp<1>(h, a, s);
}

// Host entry point in two halves: enqueue (copies in, kernel, copies out on the handle's own
// non-blocking stream) and wait (synchronise, map the per-QP status onto the return code).
int lompc_solve_batch_host_async(lompc_t* h, int64_t B, const double* lmbd, int64_t lmbd_stride,
                                 const double* lmbd_r, int64_t lmbd_r_stride, const double* gamma,
                                 double* w_out, double* cost_out, int32_t* status, int32_t* iters,
                                 double* kkt_res) {
  if (!h || B < 0 || !lmbd || !lmbd_r || !gamma || !w_out || !cost_out) return LOMPC_ERR_ARG;
  h->pending_B = 0;
  if (B == 0) return LOMPC_OK;
  const int N = h->cs.N;
  if (lmbd_stride != 0 && lmbd_stride != 3 * (int64_t)N) return LOMPC_ERR_ARG;
  if (lmbd_r_stride != 0 && lmbd_r_stride != 1) return LOMPC_ERR_ARG;
  CK(cudaSetDevice(h->device));
  if (!h->hstream) CK(cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking));
  const size_t n_lm = (lmbd_stride ? (size_t)B : 1) * 3 * N;
  const size_t n_lr = lmbd_r_stride ? (size_t)B : 1;
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t o_lm = 0;
  const size_t o_lr = o_lm + al(n_lm * 8);
  const size_t o_ga = o_lr + al(n_lr * 8);
  const size_t o_w = o_ga + al((size_t)B * 8);
  const size_t o_c = o_w + al((size_t)B * N * 8);
  const size_t o_k = o_c + al((size_t)B * 8);
  const size_t o_st = o_k + al((size_t)B * 8);
  const size_t o_it = o_st + al((size_t)B * 4);
  const size_t total = o_it + al((size_t)B * 4);
  int rc = ensure_ws(h, total);
  if (rc) return rc;
  if (!status) {  // the status is always fetched: it carries the reference's error conventions
    if (h->hst_cap < (size_t)B) {
      if (h->hst) CK(cudaFreeHost(h->hst));
      h->hst = nullptr;
      h->hst_cap = 0;
      CK(cudaMallocHost(&h->hst, (size_t)B * 4 + 1024));
      h->hst_cap = (size_t)B + 256;
    }
    status = h->hst;
  }
  char* ws = static_cast<char*>(h->ws);
  cudaStream_t s = h->hstream;
  CK(cudaMemcpyAsync(ws + o_lm, lmbd, n_lm * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(ws + o_lr, lmbd_r, n_lr * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(ws + o_ga, gamma, (size_t)B * 8, cudaMemcpyHostToDevice, s));
  rc = lompc_solve_batch_dev(h, B, (const double*)(ws + o_lm), lmbd_stride,
                             (const double*)(ws + o_lr), lmbd_r_stride, (const double*)(ws + o_ga),
                             (double*)(ws + o_w), (double*)(ws + o_c), (int32_t*)(ws + o_st),
                             (int32_t*)(ws + o_it), (double*)(ws + o_k), s);
  if (rc) return rc;
  CK(cudaMemcpyAsync(w_out, ws + o_w, (size_t)B * N * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(cost_out, ws + o_c, (size_t)B * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(status, ws + o_st, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
  if (iters) CK(cudaMemcpyAsync(iters, ws + o_it, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
  if (kkt_res) CK(cudaMemcpyAsync(kkt_res, ws + o_k, (size_t)B * 8, cudaMemcpyDeviceToHost, s));
  h->pending_B = B;
  h->pending_status = status;
  return LOMPC_OK;
}

int lompc_host_wait(lompc_t* h) {
  if (!h) return LOMPC_ERR_ARG;
  if (!h->hstream || h->pending_B == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->hstream));
  const int64_t B = h->pending_B;
  const int32_t* st = h->pending_status;
  h->pending_B = 0;
  int rc = LOMPC_OK;
  for (int64_t i = 0; i < B; ++i) {
    if (st[i] == LOMPC_ST_BAD_GAMMA) { rc = LOMPC_ERR_GAMMA; break; }
    if (st[i] == LOMPC_ST_NEGATIVE) { rc = LOMPC_ERR_NEGATIVE; break; }
    if (st[i] == LOMPC_ST_MAXITER) rc = LOMPC_ERR_NOT_CONVERGED;
  }
  return rc;
}

int lompc_solve_batch_host(lompc_t* h, int64_t B, const double* lmbd, int64_t lmbd_stride,
                           const double* lmbd_r, int64_t lmbd_r_stride, const double* gamma,
                           double* w_out, double* cost_out, int32_t* status, int32_t* iters,
                           double* kkt_res) {
  int rc = lompc_solve_batch_host_async(h, B, lmbd, lmbd_stride, lmbd_r, lmbd_r_stride, gamma, w_out, cost_out,
                                        status, iters, kkt_res);
  if (rc) return rc;
  return lompc_host_wait(h);
}


// ------------------------------------------------------------------------------
// Price loop
// ------------------------------------------------------------------------------
}  // extern "C" (helpers below are internal)

namespace {

struct Carver {  // carves aligned sub-buffers out of one allocation
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<char*>(b)) {}
  template <typename T>
  T* take(size_t n) {
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += (n * sizeof(T) + 255) & ~(size_t)255;
    return p;
  }
};

int ensure_pws(lompc_handle* h, size_t bytes) {
  if (!h->poll) CK(cudaMallocHost(&h->poll, 128));
  if (h->pws_bytes >= bytes) return LOMPC_OK;
  if (h->pws) CK(cudaFree(h->pws));
  h->pws = nullptr;
  h->pws_bytes = 0;
  const size_t want = bytes + bytes / 8;
  CK(cudaMalloc(&h->pws, want));
  h->pws_bytes = want;
  return LOMPC_OK;
}

// K1 in group mode (shared prices per group, optional skip mask and fused epilogues).
int launch_group_solve(const lompc_handle* h, int64_t B, const double* lmbd, const double* lmbd_r,
                       const double* gamma, const int32_t* group_of, const int32_t* skip,
                       const double* w_ref, double* w_out, double* cost_out, double* err_out,
                       double* w0_out, double* price0_out, cudaStream_t s, const double* w_init = nullptr) {
  if (B == 0) return LOMPC_OK;
  lompc::SolveArgs a;
  a.B = B;
  a.lmbd = lmbd;
  a.lmbd_stride = 3 * (int64_t)h->cs.N;
  a.lmbd_r = lmbd_r;
  a.lmbd_r_stride = 1;
  a.gamma = gamma;
  a.w_out = w_out;
  a.cost_out = cost_out;
  a.status = nullptr;
  a.iters = nullptr;
  a.kkt_res = nullptr;
  a.max_iter = h->max_iter;
  a.tol = h->tol;
  a.group_of = group_of;
  a.skip = skip;
  a.w_ref = w_ref;
  a.err_out = err_out;
  a.w0_out = w0_out;
  a.price0_out = price0_out;
  a.w_init = w_init;
  return h->cs.large ? launch_solve<4>(h, a, s) : launch_solve<1>(h, a, s);
}

inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

// group_step_kernel: one warp per group, 2 warps per CTA, scratch in dynamic shared memory
int launch_group_step(const lompc_handle* h, const lompc::PriceArgs& p, int it, cudaStream_t s) {
  const int N = h->cs.N, wpc = 2;
  const size_t smem = (size_t)wpc * (lompc::price_step_scratch_doubles(N, p.r) + (p.r + 7) / 8) * sizeof(double);
  // the scratch of two warps grows with N: above N ~ 750 it exceeds the shared-memory opt-in (not a CUDA failure)
  if (smem > 227 * 1024) return LOMPC_ERR_ARG;
  // (the horizons of the closed loop and of BASELINE configs[2] get the unrolled recursions of the price step)
  if (N == 24) {
    lompc::group_step_kernel<24><<<nblk(p.G, wpc), 32 * wpc, smem, s>>>(h->cs, p, it);
  } else if (N == 12) {
    lompc::group_step_kernel<12><<<nblk(p.G, wpc), 32 * wpc, smem, s>>>(h->cs, p, it);
  } else {
    if (smem > 48 * 1024) {
      CK(cudaFuncSetAttribute(lompc::group_step_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    lompc::group_step_kernel<0><<<nblk(p.G, wpc), 32 * wpc, smem, s>>>(h->cs, p, it);
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CK(cudaGetLastError());
  return LOMPC_OK;
}
#define COUNT_LAUNCH() g_launches.fetch_add(1, std::memory_order_relaxed)

}  // namespace

extern "C" {

int price_group_stats_dev(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off,
                          const double* y0, double* gamma, double* y0_rng, double* gamma_sc,
                          double* gamma_sm, void* stream) {
  if (!h || G < 0 || B < 0 || !group_off || !y0 || !gamma || !y0_rng || !gamma_sc || !gamma_sm)
    return LOMPC_ERR_ARG;
  if (G == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int rc = ensure_pws(h, 256);
  if (rc) return rc;
  int32_t* bad = static_cast<int32_t*>(h->pws);
  CK(cudaMemsetAsync(bad, 0, 4, s));
  lompc::group_stats_kernel<<<nblk(G, 128), 128, 0, s>>>(h->cs, G, group_off, y0, gamma, y0_rng, gamma_sc,
                                                        gamma_sm, bad);
  COUNT_LAUNCH();
  CK(cudaMemcpyAsync(h->poll, bad, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return h->poll[0] ? LOMPC_ERR_CONSTS : LOMPC_OK;
}

int price_w_err_dev(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off,
                    const double* gamma, const double* lmbd, const double* lmbd_r,
                    const double* w_ref, double* w_avg, double* w_err_max, double* w0_err,
                    double* w_avg_err, double* w0, void* stream) {
  if (!h || G < 0 || B < 0 || !group_off || !gamma || !lmbd || !lmbd_r || !w_ref) return LOMPC_ERR_ARG;
  if (G == 0 || B == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int N = h->cs.N;
  Carver sz(nullptr);
  sz.take<int32_t>(B); sz.take<double>((size_t)B * N); sz.take<double>(B);
  sz.take<double>((size_t)G * N); sz.take<double>(G); sz.take<double>(G); sz.take<double>(G);
  sz.take<int32_t>(G); sz.take<int32_t>(G); sz.take<int32_t>(G); sz.take<int32_t>(1); sz.take<double>(G);
  int rc = ensure_pws(h, sz.off);
  if (rc) return rc;
  Carver cv(h->pws);
  int32_t* group_of = cv.take<int32_t>(B);
  double* w_ev = cv.take<double>((size_t)B * N);
  double* err_ev = cv.take<double>(B);
  double* t_wavg = cv.take<double>((size_t)G * N);
  double* t_emax = cv.take<double>(G);
  double* t_e0 = cv.take<double>(G);
  double* t_eavg = cv.take<double>(G);
  int32_t* skip = cv.take<int32_t>(G);
  int32_t* iters = cv.take<int32_t>(G);
  int32_t* nst = cv.take<int32_t>(G);
  int32_t* nact = cv.take<int32_t>(1);
  double* y0r = cv.take<double>(G);
  lompc::group_of_kernel<<<nblk(B, 256), 256, 0, s>>>(B, G, group_off, group_of);
  COUNT_LAUNCH();
  lompc::init_groups_kernel<<<nblk(G, 128), 128, 0, s>>>(G, 1, group_off, skip, iters, nst);
  COUNT_LAUNCH();
  rc = launch_group_solve(h, B, lmbd, lmbd_r, gamma, group_of, skip, w_ref, w_ev, nullptr, err_ev, w0,
                          nullptr, s);
  if (rc) return rc;
  double* wa = w_avg ? w_avg : t_wavg;
  double* em = w_err_max ? w_err_max : t_emax;
  lompc::colsum_kernel<<<nblk((int64_t)G * N, 128), 128, 0, s>>>(N, G, group_off, skip, w_ev, err_ev, wa, em, 0);
  COUNT_LAUNCH();
  // errors via the step kernel's first phase with an infinite tolerance (every group "converges")
  CK(cudaMemsetAsync(y0r, 0x7f, (size_t)G * 8, s));  // 0x7f7f... = 1.4e306
  lompc::PriceArgs p{};
  p.G = G; p.r = 3 * N; p.tol_type_max = 0; p.eps_reg = 0.01; p.eps_tol = 0.0;
  p.group_off = group_off; p.w_ref = w_ref; p.lmbd_r = lmbd_r; p.y0_rng = y0r;
  p.w_avg = wa; p.w_err_max = em; p.w_avg_err = w_avg_err ? w_avg_err : t_eavg;
  p.w0_err = w0_err ? w0_err : t_e0; p.skip = skip; p.iters = iters; p.nnqp_status = nst; p.n_active = nact;
  return launch_group_step(h, p, 0, s);
}

int price_step_dev(lompc_t* h, int32_t G, int r, const double* w_ref, const double* w_k,
                   const double* lmbd_r, double* lmbd, double* dual_decrease, int32_t* status,
                   void* stream) {
  if (!h || G < 0 || !w_ref || !w_k || !lmbd_r || !lmbd) return LOMPC_ERR_ARG;
  const int N = h->cs.N;
  if (r != 2 * N && r != 3 * N) return LOMPC_ERR_ARG;
  if (G == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Carver sz(nullptr);
  sz.take<double>((size_t)G * N); sz.take<double>(G); sz.take<double>(G); sz.take<double>(G); sz.take<double>(G);
  sz.take<double>(G); sz.take<double>(G); sz.take<int32_t>(G); sz.take<int32_t>(G); sz.take<int32_t>(G);
  sz.take<int32_t>(1); sz.take<unsigned char>((size_t)r * G);
  int rc = ensure_pws(h, sz.off);
  if (rc) return rc;
  Carver cv(h->pws);
  double* w_avg = cv.take<double>((size_t)G * N);
  double* y0r = cv.take<double>(G);
  double* e1 = cv.take<double>(G);
  double* e2 = cv.take<double>(G);
  double* e3 = cv.take<double>(G);
  double* lamdiff = cv.take<double>(G);
  double* decp = cv.take<double>(G);
  int32_t* skip = cv.take<int32_t>(G);
  int32_t* iters = cv.take<int32_t>(G);
  int32_t* nst = cv.take<int32_t>(G);
  int32_t* nact = cv.take<int32_t>(1);
  unsigned char* wsb = cv.take<unsigned char>((size_t)r * G);
  CK(cudaMemsetAsync(skip, 0, (size_t)G * 4, s));
  // force the step: w_avg = +huge so that the error test never passes
  CK(cudaMemsetAsync(w_avg, 0x7f, (size_t)G * N * 8, s));
  CK(cudaMemsetAsync(y0r, 0, (size_t)G * 8, s));
  lompc::PriceArgs p{};
  p.G = G; p.r = r; p.tol_type_max = 0; p.eps_reg = 0.01; p.eps_tol = 0.01;
  p.w_ref = w_ref; p.lmbd_r = lmbd_r; p.y0_rng = y0r; p.lmbd = lmbd; p.w_k = const_cast<double*>(w_k);
  p.w_avg = w_avg; p.w_err_max = e1; p.w_avg_err = e2; p.w0_err = e3; p.lamdiff_phi = lamdiff;
  p.dec_pred = dual_decrease ? dual_decrease : decp; p.skip = skip; p.iters = iters;
  p.nnqp_status = status ? status : nst; p.n_active = nact; p.wsb = wsb; p.cold = 1; p.want_dec = 1;
  return launch_group_step(h, p, 1, s);
}

int price_regularize_dev(lompc_t* h, int32_t G, int r, const double* w_k, double* lmbd,
                         double* price_pre, double* price_post, void* stream) {
  if (!h || G < 0 || !w_k || !lmbd || !price_pre || !price_post) return LOMPC_ERR_ARG;
  const int N = h->cs.N;
  if (r != 2 * N && r != 3 * N) return LOMPC_ERR_ARG;
  if (G == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  lompc::regularize_kernel<<<nblk(G, 128), 128, 0, s>>>(h->cs, G, r, w_k, lmbd, price_pre, price_post, nullptr);
  COUNT_LAUNCH();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

// ---- sharded price loop: the pieces of compute_optimal_prices between which a multi-GPU
// caller all-reduces (include/lompc_b200.h).  State lives in the handle (one session at a time).
static int shard_join_side(lompc_t* h, cudaStream_t s);

int price_shard_begin(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off, const double* y0,
                      const double* w_ref, const double* lmbd_r, int r, int max_iter, int tol_type_max,
                      double eps_reg, double eps_tol, double* prices, int32_t* iters, double* stat_min,
                      double* stat_max, double* stat_sum, double* stat_cnt, double* w_sum, double* err_max,
                      double* hist_ac, double* hist_pred, int hist_cap, void* stream) {
  if (!h || G < 0 || B < 0 || !group_off || (!y0 && B > 0) || !w_ref || !lmbd_r || !prices || !iters ||
      !stat_min || !stat_max || !stat_sum || !stat_cnt || !w_sum || !err_max)
    return LOMPC_ERR_ARG;
  const int N = h->cs.N;
  if ((r != 2 * N && r != 3 * N) || max_iter < 1) return LOMPC_ERR_ARG;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  {
    int rcj = shard_join_side(h, s);  // (a previous session that ended without price_shard_finish)
    if (rcj) return rcj;
  }
  PriceSession& S = h->ses;
  S = PriceSession{};
  S.G = G; S.B = B; S.group_off = group_off; S.max_iter = max_iter;
  if (G == 0) { S.active = true; return LOMPC_OK; }
  auto carve = [&](Carver& cv) {
    S.group_of = cv.take<int32_t>(B); S.gamma = cv.take<double>(B); S.w_ev = cv.take<double>((size_t)B * N);
    S.err_ev = cv.take<double>(B); S.y0_rng = cv.take<double>(G); S.gamma_sc = cv.take<double>(G);
    S.gamma_sm = cv.take<double>(G); S.w_k = cv.take<double>((size_t)G * N);
    S.e_avg = cv.take<double>(G); S.e_0 = cv.take<double>(G); S.dual_cost = cv.take<double>(G);
    S.cost_new = cv.take<double>(G); S.lamdiff = cv.take<double>(G); S.decp = cv.take<double>(G);
    S.skip = cv.take<int32_t>(G); S.nst = cv.take<int32_t>(G); S.nact = cv.take<int32_t>(4);
    S.empty = cv.take<int32_t>(G);
    S.wsb = cv.take<unsigned char>((size_t)r * G);
  };
  Carver sz(nullptr);
  carve(sz);
  int rc = ensure_pws(h, sz.off);
  if (rc) return rc;
  Carver cv(h->pws);
  carve(cv);
  S.stat_min = stat_min; S.stat_max = stat_max; S.stat_sum = stat_sum; S.stat_cnt = stat_cnt;
  lompc::PriceArgs& p = S.p;
  p = lompc::PriceArgs{};
  p.G = G; p.r = r; p.tol_type_max = tol_type_max; p.eps_reg = eps_reg; p.eps_tol = eps_tol;
  p.group_off = group_off; p.w_ref = w_ref; p.lmbd_r = lmbd_r; p.y0_rng = S.y0_rng; p.lmbd = prices;
  p.w_k = S.w_k; p.w_avg = w_sum; p.cnt = stat_cnt; p.w_err_max = err_max; p.w_avg_err = S.e_avg; p.w0_err = S.e_0;
  p.dual_cost = S.dual_cost; p.cost_new = S.cost_new; p.lamdiff_phi = S.lamdiff; p.dec_pred = S.decp;
  p.skip = S.skip; p.iters = iters; p.nnqp_status = S.nst; p.n_active = S.nact;
  p.hist_ac = (hist_ac && hist_pred && hist_cap > 0) ? hist_ac : nullptr;
  p.hist_pred = hist_pred; p.hist_cap = hist_cap; p.wsb = S.wsb;
  CK(cudaMemsetAsync(S.nact, 0, 16, s));
  if (B > 0) {
    lompc::group_of_kernel<<<nblk(B, 256), 256, 0, s>>>(B, G, group_off, S.group_of);
    COUNT_LAUNCH();
  }
  lompc::group_stats_local_kernel<<<nblk(G, 128), 128, 0, s>>>(h->cs, G, group_off, y0, S.gamma, stat_min, stat_max,
                                                              stat_sum, stat_cnt, S.nact + 1);
  COUNT_LAUNCH();
  if (p.hist_ac) {
    CK(cudaMemsetAsync(hist_ac, 0, (size_t)G * hist_cap * 8, s));
    CK(cudaMemsetAsync(hist_pred, 0, (size_t)G * hist_cap * 8, s));
  }
  CK(cudaGetLastError());
  S.peer = h->peers.world > 1 && !tol_type_max &&
           lompc::kPeerFlagBytes + 2 * (size_t)G * N * sizeof(double) <= h->peer_region_bytes;
  if (S.peer) {
    S.tag0 = (++h->peer_sessions) << 20;  // every rank opens its sessions in the same order
    p.peer_world = h->peers.world;
    p.peer_rank = h->peers.rank;
    for (int r = 0; r < h->peers.world; ++r) p.peer_region[r] = h->peers.region[r];
    p.blocks_done = reinterpret_cast<unsigned int*>(S.nact + 3);
    p.peer_tag0 = S.tag0;
    p.peer_timeout = S.nact + 2;
  }
  S.active = true;
  return LOMPC_OK;
}

// Group-step arguments of the session: with every EV on this rank the step forms the column sums itself.
static lompc::PriceArgs shard_fused_sums(const lompc_t* h) {
  const PriceSession& S = h->ses;
  lompc::PriceArgs pa = S.p;
  if (S.local_sums && !S.peer) {
    pa.cs_w_ev = S.w_ev;
    pa.cs_err_ev = S.p.tol_type_max ? S.err_ev : nullptr;
    pa.cs_off = S.group_off;
  }
  return pa;
}

// The caller's stream waits for whatever the pipelined group phase left running on the side stream.
static int shard_join_side(lompc_t* h, cudaStream_t s) {
  if (!h->side_pending) return LOMPC_OK;
  CK(cudaStreamWaitEvent(s, h->ev_join, 0));
  h->side_pending = false;
  return LOMPC_OK;
}

int price_shard_start(lompc_t* h, void* stream) {
  if (!h || !h->ses.active) return LOMPC_ERR_ARG;
  PriceSession& S = h->ses;
  if (S.G == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  lompc::stats_finalize_kernel<<<nblk(S.G, 128), 128, 0, s>>>(h->cs, S.G, S.max_iter, S.stat_min, S.stat_max,
                                                             S.stat_sum, S.stat_cnt, S.y0_rng, S.gamma_sc,
                                                             S.gamma_sm, S.skip, S.p.iters, S.nst, S.empty, S.nact + 1);
  COUNT_LAUNCH();
  // the one synchronising check of a solve: y0 outside [0, y_max] anywhere in the (all-reduced) statistics
  CK(cudaMemcpyAsync(h->poll, S.nact, 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  // The stream is idle: every count the previous loop published has landed.  Clear the ring, so that price_shard_poll
  // cannot take the tag a previous loop left in a slot for this loop's iteration of the same number.
  if (h->ring) memset(h->ring, 0, kRingSlots * 2 * sizeof(int32_t));
  if (h->poll[1]) {
    S.active = false;
    return LOMPC_ERR_CONSTS;  // price_solver.py:71, raised by every rank
  }
  // w_k, dual_cost = solve_lompc(lmbd_k, lmbd_r, gamma_sc)   (price_solver.py:106)
  return launch_group_solve(h, S.G, S.p.lmbd, S.p.lmbd_r, S.gamma_sc, nullptr, S.skip, nullptr, S.w_k,
                            S.dual_cost, nullptr, nullptr, nullptr, s);
}

int price_shard_ev_phase(lompc_t* h, void* stream) {
  if (!h || !h->ses.active) return LOMPC_ERR_ARG;
  PriceSession& S = h->ses;
  if (S.G == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int N = h->cs.N;
  const bool need_err = S.p.tol_type_max != 0;
  // _get_w_err (price_solver.py:112,196-214): the EV solves and the per-group column sums
  // (from the second pass on every QP starts from its solution at the previous prices)
  int rc = launch_group_solve(h, S.B, S.p.lmbd, S.p.lmbd_r, S.gamma, S.group_of, S.skip, S.p.w_ref, S.w_ev,
                              nullptr, need_err ? S.err_ev : nullptr, nullptr, nullptr, s,
                              S.ev_passes > 0 ? S.w_ev : nullptr);
  if (rc) return rc;
  const int it = S.ev_passes++;
  // the per-group column sums: into the caller's w_sum buffer (which it all-reduces), or - peer exchange - into
  // buffer it & 1 of this rank's peer region, followed by the flag on every rank
  if (S.local_sums && !S.peer) return LOMPC_OK;  // the group step forms the sums itself (shard_fused_sums)
  if (S.peer) {
    double* sums = reinterpret_cast<double*>(h->peers.region[h->peers.rank] + lompc::kPeerFlagBytes) +
                   (size_t)(it & 1) * S.G * N;
    lompc::colsum_signal_kernel<<<nblk((int64_t)S.G * N, 128), 128, 0, s>>>(N, S.G, S.group_off, S.skip, S.w_ev, sums,
                                                                           S.p, S.tag0 + (unsigned long long)it + 1);
  } else {
    lompc::colsum_kernel<<<nblk((int64_t)S.G * N, 128), 128, 0, s>>>(N, S.G, S.group_off, S.skip, S.w_ev,
                                                                    need_err ? S.err_ev : nullptr, S.p.w_avg,
                                                                    S.p.w_err_max, 1);
  }
  COUNT_LAUNCH();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

int price_shard_group_phase(lompc_t* h, int it, int32_t* n_active, void* stream) {
  if (!h || !h->ses.active || !n_active) return LOMPC_ERR_ARG;
  PriceSession& S = h->ses;
  *n_active = 0;
  if (S.G == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  {
    int rcj = shard_join_side(h, s);
    if (rcj) return rcj;
  }
  CK(cudaMemsetAsync(S.nact, 0, 4, s));
  {
    int rc0 = launch_group_step(h, shard_fused_sums(h), it, s);
    if (rc0) return rc0;
  }
  CK(cudaMemcpyAsync(h->poll, S.nact, 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (h->poll[1]) return LOMPC_ERR_CONSTS;  // y0 outside [0, y_max], price_solver.py:71
  *n_active = h->poll[0];
  if (h->poll[0] == 0) return LOMPC_OK;
  // w_k, dual_cost_new = solve_lompc(lmbd_k_new, lmbd_r, gamma_sc)   (price_solver.py:132)
  int rc = launch_group_solve(h, S.G, S.p.lmbd, S.p.lmbd_r, S.gamma_sc, nullptr, S.skip, nullptr, S.w_k,
                              S.cost_new, nullptr, nullptr, nullptr, s, S.w_k);
  if (rc) return rc;
  lompc::bookkeep_kernel<<<nblk(S.G, 128), 128, 0, s>>>(S.p, it);
  COUNT_LAUNCH();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

// price_shard_group_phase without the host round trip: enqueues the convergence test, the price step, the
// gamma_sc solve and the bookkeeping of iteration `it` and PUBLISHES the number of still-active groups into a
// pinned ring that price_shard_poll reads.  Converged groups are skipped on the device (every kernel tests the
// group's flag), so iterations enqueued beyond convergence are no-ops.
int price_shard_group_phase_async(lompc_t* h, int it, void* stream) {
  if (!h || !h->ses.active || it < 0) return LOMPC_ERR_ARG;
  PriceSession& S = h->ses;
  if (S.G == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!h->ring) {
    CK(cudaMallocHost(&h->ring, kRingSlots * 2 * sizeof(int32_t)));
    memset(h->ring, 0, kRingSlots * 2 * sizeof(int32_t));
  }
  // three launches per group phase: the step (which, with peers attached, first gathers the ranks' partial sums),
  // the gamma_sc solve, and the bookkeeping (which publishes the active count to the host ring and resets it)
  lompc::PriceArgs pa = shard_fused_sums(h);
  pa.publish_ring = h->ring;
  pa.publish_slots = kRingSlots;
  // The gamma_sc solve and the bookkeeping of this iteration are needed by the NEXT group step only (w_k, the reset
  // active count), not by the next EV phase (which reads the prices and skip flags the step just wrote, and touches
  // none of w_k / cost_new / dual_cost / the histories / the counter): they go to a side stream, beside the EV
  // solves and column sums of iteration it + 1, and the next group step (or price_shard_finish) joins them.  Same
  // kernels, same inputs, same results; one ~10 us launch of 1,024 QPs less on the critical path of an iteration.
  // LOMPC_SHARD_OVERLAP=0 keeps everything on the caller's stream.
  static const bool overlap = [] { const char* e = getenv("LOMPC_SHARD_OVERLAP"); return !(e && e[0] == '0'); }();
  {
    int rcj = shard_join_side(h, s);  // iteration it - 1's gamma_sc solve and bookkeeping
    if (rcj) return rcj;
    int rc0 = launch_group_step(h, pa, it, s);
    if (rc0) return rc0;
  }
  cudaStream_t t = s;
  if (overlap) {
    if (!h->side) {
      CK(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
      CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    t = h->side;
    CK(cudaEventRecord(h->ev_fork, s));
    CK(cudaStreamWaitEvent(t, h->ev_fork, 0));
  }
  // gamma_sc solve + bookkeeping: one launch where the warp-cooperative K1 would take the solve anyway
  // (LOMPC_SHARD_FUSED_BK=0: always the two launches)
  static const bool fuse_bk = [] { const char* e = getenv("LOMPC_SHARD_FUSED_BK"); return !(e && e[0] == '0'); }();
  const int N = h->cs.N;
  const bool sc_on_warps = lompc_detail::warp_kernel_supports(N, 3) &&
                           (h->variant == 8 || (h->variant == 0 && S.G <= warp_kernel_max_batch(N)));
  if (fuse_bk && sc_on_warps) {
    lompc::SolveArgs a;
    memset(&a, 0, sizeof(a));
    a.B = S.G;
    a.lmbd = S.p.lmbd;
    a.lmbd_stride = 3 * (int64_t)N;
    a.lmbd_r = S.p.lmbd_r;
    a.lmbd_r_stride = 1;
    a.gamma = S.gamma_sc;
    a.w_out = S.w_k;
    a.cost_out = S.cost_new;
    a.max_iter = h->max_iter;
    a.tol = h->tol;
    a.skip = S.skip;
    a.w_init = S.w_k;
    const int qpw = 32 / (N / 3);
    const unsigned warps = (unsigned)((S.G + qpw - 1) / qpw);
    switch (N) {
      case 12: lompc::sc_solve_bookkeep_kernel<12><<<warps, 32, 0, t>>>(h->cs, a, pa, it); break;
      case 24: lompc::sc_solve_bookkeep_kernel<24><<<warps, 32, 0, t>>>(h->cs, a, pa, it); break;
      case 48: lompc::sc_solve_bookkeep_kernel<48><<<warps, 32, 0, t>>>(h->cs, a, pa, it); break;
      case 96: lompc::sc_solve_bookkeep_kernel<96><<<warps, 32, 0, t>>>(h->cs, a, pa, it); break;
      default: return LOMPC_ERR_ARG;
    }
    COUNT_LAUNCH();
  } else {
    int rc = launch_group_solve(h, S.G, S.p.lmbd, S.p.lmbd_r, S.gamma_sc, nullptr, S.skip, nullptr, S.w_k,
                                S.cost_new, nullptr, nullptr, nullptr, t, S.w_k);
    if (rc) return rc;
    lompc::bookkeep_kernel<<<nblk(S.G, 128), 128, 0, t>>>(pa, it);
    COUNT_LAUNCH();
  }
  CK(cudaGetLastError());
  if (overlap) {
    CK(cudaEventRecord(h->ev_join, t));
    h->side_pending = true;
  }
  return LOMPC_OK;
}

// Number of active groups after iteration `it` if the device has published it (returns 1), else 0 (wait == 0)
// or spins on the pinned slot until it has (wait != 0; no synchronising CUDA call is made).  The ring holds kRingSlots
// iterations: poll iteration `it` before enqueuing iteration it + kRingSlots.
int price_shard_poll(lompc_t* h, int it, int wait, int32_t* n_active) {
  if (!h || !n_active || it < 0) return LOMPC_ERR_ARG;
  *n_active = 0;
  if (h->ses.G == 0) return 1;
  if (!h->ring) return 0;
  volatile int32_t* slot = h->ring + 2 * (it % kRingSlots);
  const auto t0 = std::chrono::steady_clock::now();
  for (unsigned spins = 1; slot[0] != it + 1; ++spins) {
    if (!wait) return 0;
    if ((spins & 0xfffffu) == 0) {  // now and then: do not spin for ever on a dead context or a stuck peer
      const cudaError_t e = cudaPeekAtLastError();
      if (e != cudaSuccess) return cuda_fail(e, "price_shard_poll");
      if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(30)) {
        snprintf(g_cuda_err, sizeof(g_cuda_err), "price_shard_poll: iteration %d was not published within 30 s", it);
        return LOMPC_ERR_CUDA;
      }
    }
  }
  *n_active = slot[1];
  return 1;
}

int price_shard_finish(lompc_t* h, double* price_pre, double* price_post, double* w_k_out, void* stream) {
  if (!h || !h->ses.active || !price_pre || !price_post) return LOMPC_ERR_ARG;
  PriceSession& S = h->ses;
  S.active = false;
  if (S.G == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int N = h->cs.N;
  {
    int rcj = shard_join_side(h, s);
    if (rcj) return rcj;
  }
  // price_solver.py:145-147
  // (empty groups keep their price row: no EV, no solve - charging_station.py:277,293)
  lompc::regularize_kernel<<<nblk(S.G, 128), 128, 0, s>>>(h->cs, S.G, S.p.r, S.w_k, S.p.lmbd, price_pre, price_post,
                                                         S.empty);
  COUNT_LAUNCH();
  if (w_k_out) CK(cudaMemcpyAsync(w_k_out, S.w_k, (size_t)S.G * N * 8, cudaMemcpyDeviceToDevice, s));
  CK(cudaGetLastError());
  if (S.peer) {
    CK(cudaMemcpyAsync(h->poll, S.nact, 16, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (h->poll[2]) {
      snprintf(g_cuda_err, sizeof(g_cuda_err), "peer exchange: a rank did not deliver its partial sums within 2 s");
      return LOMPC_ERR_CUDA;
    }
    return LOMPC_OK;
  }
  CK(cudaStreamSynchronize(s));
  return LOMPC_OK;
}

// ---- peer-memory plumbing (CUDA IPC) of the sharded price loop ----
int lompc_ipc_alloc(int device, size_t bytes, void** dev_ptr, unsigned char* handle_out) {
  if (!dev_ptr || !handle_out || bytes == 0) return LOMPC_ERR_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the ABI carries the handle as 64 bytes");
  CK(cudaSetDevice(device));
  CK(cudaMalloc(dev_ptr, bytes));
  CK(cudaMemset(*dev_ptr, 0, bytes));
  cudaIpcMemHandle_t hd;
  CK(cudaIpcGetMemHandle(&hd, *dev_ptr));
  memcpy(handle_out, &hd, 64);
  return LOMPC_OK;
}

int lompc_ipc_open(int device, const unsigned char* handle, void** dev_ptr) {
  if (!dev_ptr || !handle) return LOMPC_ERR_ARG;
  CK(cudaSetDevice(device));
  cudaIpcMemHandle_t hd;
  memcpy(&hd, handle, 64);
  CK(cudaIpcOpenMemHandle(dev_ptr, hd, cudaIpcMemLazyEnablePeerAccess));
  return LOMPC_OK;
}

int lompc_ipc_close(int device, void* dev_ptr) {
  if (!dev_ptr) return LOMPC_OK;
  CK(cudaSetDevice(device));
  CK(cudaIpcCloseMemHandle(dev_ptr));
  return LOMPC_OK;
}

int lompc_ipc_free(int device, void* dev_ptr) {
  if (!dev_ptr) return LOMPC_OK;
  CK(cudaSetDevice(device));
  CK(cudaFree(dev_ptr));
  return LOMPC_OK;
}

int price_shard_uses_peers(const lompc_t* h) { return (h && h->ses.peer) ? 1 : 0; }

int price_shard_local_sums(lompc_t* h, int on) {
  if (!h || !h->ses.active) return LOMPC_ERR_ARG;
  h->ses.local_sums = on != 0;
  return LOMPC_OK;
}

int price_shard_attach_peers(lompc_t* h, int rank, int world, void* const* regions, size_t region_bytes) {
  if (!h || world < 0 || world > lompc::kMaxPeers || (world > 0 && (!regions || rank < 0 || rank >= world)))
    return LOMPC_ERR_ARG;
  if (h->ses.active) return LOMPC_ERR_ARG;  // not in the middle of a session
  memset(&h->peers, 0, sizeof(h->peers));
  h->peer_region_bytes = 0;
  if (world <= 1) return LOMPC_OK;
  if (region_bytes <= lompc::kPeerFlagBytes) return LOMPC_ERR_ARG;
  h->peers.rank = rank;
  h->peers.world = world;
  for (int r = 0; r < world; ++r) {
    if (!regions[r]) return LOMPC_ERR_ARG;
    h->peers.region[r] = static_cast<char*>(regions[r]);
  }
  h->peer_region_bytes = region_bytes;
  return LOMPC_OK;
}

}  // extern "C"

namespace {

template <int N, int NSEG, int T, int MINB, bool GREG>
int launch_fused(lompc_handle* h, const lompc::FusedArgs& a, cudaStream_t s) {
  constexpr size_t smem = lompc::FusedSmem<N, NSEG, T, GREG>::bytes;
  static std::atomic<uint64_t> configured{0};  // per device ordinal
  if (!device_flag_test(configured, h->device)) {
    CK(cudaFuncSetAttribute(lompc::price_group_loop_kernel<N, NSEG, T, MINB, GREG>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute(lompc::price_station_chain_kernel<N, NSEG, T, MINB, GREG>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    device_flag_set(configured, h->device);
  }
  if (a.chain_P > 0)
    lompc::price_station_chain_kernel<N, NSEG, T, MINB, GREG><<<(unsigned)a.chain_S, T, smem, s>>>(h->cs, a);
  else
    lompc::price_group_loop_kernel<N, NSEG, T, MINB, GREG><<<(unsigned)a.G, T, smem, s>>>(h->cs, a);
  COUNT_LAUNCH();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

// The parametric loop (lompc_price_warp.cuh): one warp per group / per station; the "max" tolerance type has its own
// instantiation.
template <int N>
int launch_fused_warp(lompc_handle* h, const lompc::FusedArgs& a, cudaStream_t s) {
  constexpr size_t smem = lompc::WarpLoopSmem<N>::bytes;
  static_assert(smem <= 48 * 1024, "no shared-memory opt-in needed");
  if (a.tol_type_max) {
    if (a.chain_P > 0)
      lompc::price_station_chain_warp_kernel<N, true><<<(unsigned)a.chain_S, 32, smem, s>>>(h->cs, a);
    else
      lompc::price_group_warp_kernel<N, true><<<(unsigned)a.G, 32, smem, s>>>(h->cs, a);
  } else if (a.chain_P > 0) {
    lompc::price_station_chain_warp_kernel<N, false><<<(unsigned)a.chain_S, 32, smem, s>>>(h->cs, a);
  } else {
    lompc::price_group_warp_kernel<N, false><<<(unsigned)a.G, 32, smem, s>>>(h->cs, a);
  }
  COUNT_LAUNCH();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

// Is there a device-resident loop for this handle?  N = 12, 24: the parametric and the thread-per-EV kernels; N = 48,
// 96: the parametric kernel only (loop mode 0 or 2).  Otherwise: the phase-split loop.  Both tolerance types alike.
inline bool has_fused_loop(const lompc_handle* h) {
  if (h->variant == 1 || h->loop_mode == 1) return false;
  const int N = h->cs.N;
  if (N == 12 || N == 24) return true;
  return (N == 48 || N == 96) && (h->loop_mode == 2 || (h->loop_mode == 0 && kParametricLoopByDefault));
}

// compute_optimal_prices for whole groups resident on this GPU: one CTA per group, no host loop.
int price_solve_fused(lompc_handle* h, const lompc::FusedArgs& a, cudaStream_t s) {
  const int N = h->cs.N;
  // loop mode 2 = the parametric one-warp-per-group loop, 3 = the thread-per-EV loop; 0 = automatic
  const bool parametric = h->loop_mode == 2 || (h->loop_mode == 0 && kParametricLoopByDefault);
  if (parametric) {
    if (N == 24) return launch_fused_warp<24>(h, a, s);
    if (N == 12) return launch_fused_warp<12>(h, a, s);
    if (N == 48) return launch_fused_warp<48>(h, a, s);
    if (N == 96) return launch_fused_warp<96>(h, a, s);
  }
  if (h->cs.large) {
    if (N == 24) return launch_fused<24, 4, 64, 4, true>(h, a, s);
    if (N == 12) return launch_fused<12, 4, 64, 4, true>(h, a, s);
  } else {
    if (N == 24) return launch_fused<24, 1, 64, 4, false>(h, a, s);
    if (N == 12) return launch_fused<12, 1, 64, 4, false>(h, a, s);
  }
  return LOMPC_ERR_ARG;
}

// Fused, device-resident loop (lompc_price_fused.cuh): one CTA per group, or - chain_P > 0 - one CTA
// per station running its chain_P partitions in the reference's warm-start order.
int price_solve_fused_entry(lompc_handle* h, int32_t G, int64_t B, const int32_t* group_off, const double* y0,
                            const double* w_ref, const double* lmbd_r, int r, int max_iter, int tol_type_max,
                            double eps_reg, double eps_tol, double* prices, int32_t* iters, double* price_pre,
                            double* price_post, double* w_k_out, double* hist_ac, double* hist_pred, int hist_cap,
                            int32_t* total_iters, int chain_S, int chain_P, double* chain_prev,
                            const int32_t* chain_order, void* stream) {
  {
    if ((r != 2 * h->cs.N && r != 3 * h->cs.N) || max_iter < 1) return LOMPC_ERR_ARG;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int rc = ensure_pws(h, 256 + ((size_t)(B + G) * h->cs.N + 2 * (size_t)G + 8) * sizeof(double));
    if (rc) return rc;
    int32_t* flags = static_cast<int32_t*>(h->pws);
    CK(cudaMemsetAsync(flags, 0, 128, s));
    const bool hist = hist_ac && hist_pred && hist_cap > 0;
    if (hist) {
      CK(cudaMemsetAsync(hist_ac, 0, (size_t)G * hist_cap * 8, s));
      CK(cudaMemsetAsync(hist_pred, 0, (size_t)G * hist_cap * 8, s));
    }
    lompc::FusedArgs a{};
    a.G = G; a.r = r; a.tol_type_max = tol_type_max; a.eps_reg = eps_reg; a.eps_tol = eps_tol;
    a.max_iter = max_iter; a.qp_tol = h->tol; a.qp_max_iter = h->max_iter; a.group_off = group_off; a.y0 = y0;
    a.w_ref = w_ref; a.lmbd_r = lmbd_r; a.prices = prices; a.iters = iters; a.price_pre = price_pre;
    a.price_post = price_post; a.w_k_out = w_k_out; a.hist_ac = hist ? hist_ac : nullptr; a.hist_pred = hist_pred;
    a.hist_cap = hist_cap; a.flags = flags;
    a.qp_count = reinterpret_cast<unsigned long long*>(flags + 4);
    a.w_scratch = reinterpret_cast<double*>(static_cast<char*>(h->pws) + 256);
    a.B = B;
    a.chain_S = chain_S; a.chain_P = chain_P; a.chain_prev = chain_prev; a.chain_order = chain_order;
    a.compact_step = g_force_compact_step.load(std::memory_order_relaxed) ||
                     (chain_P > 0 ? chain_S : G) >= 2 * 148 * 4;  // CTAs of the launch vs. 2 resident waves
    rc = price_solve_fused(h, a, s);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h->poll, flags, 128, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    h->last_pivot_overflows = h->poll[16];
    h->last_nnqp_cap_hits = h->poll[0];
    h->last_qp_failures = h->poll[3];
    h->last_nnqp_fallbacks = h->poll[17];
    if (total_iters) *total_iters = h->poll[2];
    h->last_qp_solves = *reinterpret_cast<unsigned long long*>(h->poll + 4);
    h->last_cycles[0] = *reinterpret_cast<unsigned long long*>(h->poll + 6);
    h->last_cycles[1] = *reinterpret_cast<unsigned long long*>(h->poll + 8);
    for (int i = 2; i < 5; ++i) h->last_cycles[i] = *reinterpret_cast<unsigned long long*>(h->poll + 6 + 2 * i);
    if (h->poll[1]) return LOMPC_ERR_CONSTS;  // y0 outside [0, y_max], price_solver.py:71
    if (h->poll[3]) return LOMPC_ERR_NOT_CONVERGED;  // some LoMPC solve inside the loop did not converge
    return LOMPC_OK;
  }
}

}  // namespace

extern "C" {

int price_solve_dev(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off, const double* y0,
                    const double* w_ref, const double* lmbd_r, int r, int max_iter,
                    int tol_type_max, double eps_reg, double eps_tol, double* prices,
                    int32_t* iters, double* price_pre, double* price_post, double* w_k_out,
                    double* hist_ac, double* hist_pred, int hist_cap, int32_t* total_iters,
                    void* stream) {
  if (!h || G < 0 || B < 0 || !group_off || !y0 || !w_ref || !lmbd_r || !prices || !iters ||
      !price_pre || !price_post)
    return LOMPC_ERR_ARG;
  if (total_iters) *total_iters = 0;
  if (G == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  if (has_fused_loop(h))
    return price_solve_fused_entry(h, G, B, group_off, y0, w_ref, lmbd_r, r, max_iter, tol_type_max, eps_reg, eps_tol,
                                   prices, iters, price_pre, price_post, w_k_out, hist_ac, hist_pred, hist_cap,
                                   total_iters, 0, 0, nullptr, nullptr, stream);
  // phase-split loop (any horizon; also the path a multi-GPU caller drives, see price_shard_*):
  // the reduction buffers live in a second grow-only allocation of the handle
  const int N = h->cs.N;
  const size_t need = ((size_t)G * (N + 5) + 64) * sizeof(double);
  if (h->rws_bytes < need) {
    if (h->rws) CK(cudaFree(h->rws));
    h->rws = nullptr;
    h->rws_bytes = 0;
    CK(cudaMalloc(&h->rws, need + need / 8));
    h->rws_bytes = need + need / 8;
  }
  double* rb = static_cast<double*>(h->rws);
  double *smin = rb, *smax = rb + G, *ssum = rb + 2 * (size_t)G, *scnt = rb + 3 * (size_t)G,
         *emax = rb + 4 * (size_t)G, *wsum = rb + 5 * (size_t)G;
  int rc = price_shard_begin(h, G, B, group_off, y0, w_ref, lmbd_r, r, max_iter, tol_type_max, eps_reg, eps_tol,
                             prices, iters, smin, smax, ssum, scnt, wsum, emax, hist_ac, hist_pred, hist_cap, stream);
  if (rc) return rc;
  h->ses.local_sums = true;  // one process, every EV here
  rc = price_shard_start(h, stream);
  if (rc) return rc;
  // The host never synchronises inside the loop: iteration `it` is enqueued while the device may still be kDepth
  // iterations behind; the active-group count of every iteration comes back through the pinned ring, and the loop
  // ends at the first iteration that published 0 (converged groups are skipped on the device, so the iterations
  // enqueued beyond that point are no-ops).  Same counts as the synchronous loop (price_shard_group_phase).
  constexpr int kDepth = 4;
  static_assert(kDepth < kRingSlots, "the ring must hold the iterations in flight");
  int done_at = -1, it = 0;
  for (; it < max_iter && done_at < 0; ++it) {
    rc = price_shard_ev_phase(h, stream);
    if (rc) return rc;
    rc = price_shard_group_phase_async(h, it, stream);
    if (rc) return rc;
    if (it >= kDepth) {
      int32_t nact = 0;
      rc = price_shard_poll(h, it - kDepth, 1, &nact);
      if (rc < 0) return rc;
      if (nact == 0) done_at = it - kDepth;
    }
  }
  for (int j = (it > kDepth ? it - kDepth : 0); j < it && done_at < 0; ++j) {  // drain what is still in flight
    int32_t nact = 0;
    rc = price_shard_poll(h, j, 1, &nact);
    if (rc < 0) return rc;
    if (nact == 0) done_at = j;
  }
  if (total_iters) *total_iters = done_at >= 0 ? done_at : max_iter;
  return price_shard_finish(h, price_pre, price_post, w_k_out, stream);
}

int price_solve_chain_dev(lompc_t* h, int32_t S, int32_t P, int64_t B, const int32_t* group_off, const double* y0,
                          const double* w_ref, const double* lmbd_r, int r, int max_iter, int tol_type_max,
                          double eps_reg, double eps_tol, double* prev_prices, double* prices, int32_t* iters,
                          double* price_pre, double* price_post, const int32_t* station_order,
                          int32_t* max_group_iters, void* stream) {
  if (!h || S < 1 || P < 1 || B < 0 || !group_off || !y0 || !w_ref || !lmbd_r || !prev_prices || !prices || !iters ||
      !price_pre || !price_post)
    return LOMPC_ERR_ARG;
  if (max_group_iters) *max_group_iters = 0;
  CK(cudaSetDevice(h->device));
  if (!has_fused_loop(h)) {
    // no fused kernel for this horizon: the same chain as P phase-split loops, one per partition slice
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int N = h->cs.N;
    // rebased offsets of the current slice live in the handle's second grow-only allocation
    // (price_solve_dev below uses the first one)
    const size_t need = (size_t)(S + 1) * sizeof(int32_t) + ((size_t)S * (N + 5) + 64) * sizeof(double);
    if (h->rws_bytes < need) {
      if (h->rws) CK(cudaFree(h->rws));
      h->rws = nullptr;
      h->rws_bytes = 0;
      CK(cudaMalloc(&h->rws, need + need / 8));
      h->rws_bytes = need + need / 8;
    }
    int32_t* reb = reinterpret_cast<int32_t*>(static_cast<char*>(h->rws) +
                                              ((h->rws_bytes - (size_t)(S + 1) * sizeof(int32_t)) & ~(size_t)15));
    int rc = LOMPC_OK;
    for (int p = 0; p < P && rc == LOMPC_OK; ++p) {
      const int32_t* off_p = group_off + (size_t)p * S;
      int32_t ends[2] = {0, 0};
      cudaError_t e = cudaMemcpyAsync(&ends[0], off_p, 4, cudaMemcpyDeviceToHost, s);
      if (e == cudaSuccess) e = cudaMemcpyAsync(&ends[1], off_p + S, 4, cudaMemcpyDeviceToHost, s);
      if (e == cudaSuccess) e = cudaStreamSynchronize(s);
      if (e != cudaSuccess) { rc = cuda_fail(e, "price_solve_chain_dev"); break; }
      const size_t g0 = (size_t)p * S;
      if (ends[1] > ends[0]) {
        lompc::rebase_offsets_kernel<<<nblk(S + 1, 128), 128, 0, s>>>(S, off_p, reb);
        COUNT_LAUNCH();
        int32_t tot = 0;
        rc = price_solve_dev(h, S, ends[1] - ends[0], reb, y0 + ends[0], w_ref + g0 * N, lmbd_r + g0, r, max_iter,
                             tol_type_max, eps_reg, eps_tol, prev_prices, iters + g0, price_pre + g0, price_post + g0,
                             nullptr, nullptr, nullptr, 0, &tot, stream);
        if (max_group_iters && tot > *max_group_iters) *max_group_iters = tot;
      } else {
        e = cudaMemsetAsync(iters + g0, 0xff, (size_t)S * 4, s);  // -1: empty partition
        if (e != cudaSuccess) { rc = cuda_fail(e, "price_solve_chain_dev"); break; }
      }
      lompc::chain_rows_kernel<<<nblk((int64_t)S * 3 * N, 256), 256, 0, s>>>(S, 3 * N, off_p, prev_prices,
                                                                             prices + g0 * 3 * N);
      COUNT_LAUNCH();
    }
    cudaStreamSynchronize(s);
    return rc;
  }
  return price_solve_fused_entry(h, S * P, B, group_off, y0, w_ref, lmbd_r, r, max_iter, tol_type_max, eps_reg, eps_tol,
                                 prices, iters, price_pre, price_post, nullptr, nullptr, nullptr, 0, max_group_iters, S,
                                 P, prev_prices, station_order, stream);
}

int price_lp_rows_dev(int device, int N, int nb, const double* a, const double* b, const double* c,
                      double* x, void* stream) {
  if (N < 0 || nb < 1 || !a || !b || !c || !x) return LOMPC_ERR_ARG;
  if (lompc_device_count() <= device || device < 0) return LOMPC_ERR_NO_DEVICE;
  if (N == 0) return LOMPC_OK;
  CK(cudaSetDevice(device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int32_t* st = nullptr;
  CK(cudaMalloc(&st, 4));
  CK(cudaMemsetAsync(st, 0, 4, s));
  lompc::lp_rows_kernel<<<nblk(N, 128), 128, 0, s>>>(N, nb, a, b, c, x, st);
  COUNT_LAUNCH();
  int32_t hst = 0;
  cudaError_t e = cudaMemcpyAsync(&hst, st, 4, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  cudaFree(st);
  if (e != cudaSuccess) return cuda_fail(e, "price_lp_rows_dev");
  return hst ? LOMPC_ERR_ARG : LOMPC_OK;
}

int price_w0_price0_dev(lompc_t* h, int32_t G, int64_t B, const int32_t* group_off,
                        const double* gamma, const double* lmbd, const double* lmbd_r,
                        double* w0, double* price0, void* stream) {
  if (!h || G < 0 || B < 0 || !group_off || !gamma || !lmbd || !lmbd_r || !w0 || !price0) return LOMPC_ERR_ARG;
  if (G == 0 || B == 0) return LOMPC_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Carver sz(nullptr);
  sz.take<int32_t>(B); sz.take<double>(B);
  int rc = ensure_pws(h, sz.off);
  if (rc) return rc;
  Carver cv(h->pws);
  int32_t* group_of = cv.take<int32_t>(B);
  double* p0_ev = cv.take<double>(B);
  lompc::group_of_kernel<<<nblk(B, 256), 256, 0, s>>>(B, G, group_off, group_of);
  COUNT_LAUNCH();
  rc = launch_group_solve(h, B, lmbd, lmbd_r, gamma, group_of, nullptr, nullptr, nullptr, nullptr, nullptr, w0,
                          p0_ev, s);
  if (rc) return rc;
  lompc::mean_kernel<<<nblk(G, 128), 128, 0, s>>>(G, group_off, p0_ev, price0);
  COUNT_LAUNCH();
  CK(cudaGetLastError());
  return LOMPC_OK;
}

}  // extern "C"
