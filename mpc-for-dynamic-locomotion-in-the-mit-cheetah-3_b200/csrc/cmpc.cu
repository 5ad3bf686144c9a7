// cmpc.cu - C ABI (include/cmpc.h) over the sm_100a kernels in cmpc_kernels.cuh.
// No torch types, no CPU fallback: every entry point fails with CMPC_ERR_NO_DEVICE /
// CMPC_ERR_CUDA when the CUDA device or the kernels are unavailable.
#include "../../include/cmpc.h"
#include "cmpc_kernels.cuh"
#include "cmpc_cluster.cuh"
#include "cmpc_riccati.cuh"

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                  \
  do {                                                                                  \
    cudaError_t e_ = (expr);                                                            \
    if (e_ != cudaSuccess)                                                              \
      return fail(CMPC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                  __FILE__, __LINE__);                                                  \
  } while (0)

// ---- horizon Gram matrices (fp64 on the host, once per handle) -------------------------
// M_a[j][j'] = 2 sum_{k>max(j,j')}^{N} ( w_pos,a dt^4 (k-1-j)(k-1-j') + w_vel,a dt^2 )
// axes 0-2: Theta (rotated frame) with omega weights, axes 3-5: p with v weights.
void axis_gram(int N, double dt, const float* w, std::vector<double>& M) {
  M.assign((size_t)6 * N * N, 0.0);
  for (int a = 0; a < 6; ++a) {
    const double wp = w[a];                          // w[0:3] Theta, w[3:6] p
    const double wv = w[6 + a];                      // w[6:9] omega, w[9:12] v
    for (int j = 0; j < N; ++j)
      for (int j2 = 0; j2 < N; ++j2) {
        double acc = 0.0;
        for (int k = (j > j2 ? j : j2) + 1; k <= N; ++k)
          acc += wp * dt * dt * dt * dt * (double)(k - 1 - j) * (double)(k - 1 - j2) + wv * dt * dt;
        M[((size_t)a * N + j) * N + j2] = 2.0 * acc;
      }
  }
}

// Makes `dev` current for the lifetime of the guard and restores the caller's device afterwards
// (a handle on device k must not change the calling thread's current device, which is torch's too).
struct DeviceGuard {
  int prev = -1, dev;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int d) : dev(d) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (prev >= 0 && prev != dev) cudaSetDevice(prev);
  }
};
#define DEVICE_GUARD(h)                                                                   \
  DeviceGuard guard_((h)->cfg.device);                                                    \
  if (guard_.err != cudaSuccess)                                                          \
    return fail(CMPC_ERR_CUDA, "cudaSetDevice(%d) failed: %s", (h)->cfg.device, cudaGetErrorString(guard_.err))

struct Staging {
  char* h_in = nullptr;    // pinned
  char* h_out = nullptr;   // pinned
  char* d_in = nullptr;
  char* d_out = nullptr;
  size_t in_bytes = 0, out_bytes = 0;
  cudaStream_t streams[2] = {nullptr, nullptr};
  cudaStream_t copy2 = nullptr;   // second copy stream of the async path (a second copy engine)
  cudaEvent_t h2d2[2] = {};
  cudaStream_t d2h = nullptr;     // results of the async path back to the caller's buffers
  cudaEvent_t solved[2] = {};
  char* d_async_out[2] = {nullptr, nullptr};
  // result copies of the latest submission, not enqueued yet (see flush_results)
  struct Pending {
    bool active = false;
    int32_t ticket = 0, B = 0;
    int arena = 0;
    float* U = nullptr; float* X = nullptr; int32_t* iters = nullptr;
    float* pri = nullptr; float* dua = nullptr; int32_t* status = nullptr;
  } pending;
  int cap = 0;             // problems
  cudaEvent_t done[8] = {};   // cmpc_solve_host_async: completion of the last 8 submissions
  int32_t next_ticket = 0;
  char* d_async_in[2] = {nullptr, nullptr};   // double-buffered device copies of the inputs of the async path
  size_t async_in_bytes = 0;
  cudaEvent_t h2d[2] = {};
};

}  // namespace

struct cmpc_handle {
  cmpc_config cfg;
  int NK = 0;                       // horizon of the solve kernel (cfg.N, or the next compiled one)
  float* d_pad_r = nullptr;         // NK-layout scratch of a padded horizon (NK != cfg.N)
  uint8_t* d_pad_mask = nullptr;
  float* d_pad_xdes = nullptr;
  float* d_pad_U = nullptr;
  float* d_pad_X = nullptr;
  int hist_slots = 0;
  float* d_Minv = nullptr;
  float* d_Mg = nullptr;
  float* d_warm_x = nullptr;
  float* d_warm_y = nullptr;
  uint8_t* d_warm_valid = nullptr;
  float* d_score = nullptr;      // LPT scheduling scratch
  int32_t* d_order = nullptr;
  int32_t* d_hist = nullptr;
  int32_t* d_sched = nullptr;       // persistent-launch scheduling state, one block of kSchedInts per LPT slot range
  float4* d_cache_pinv = nullptr;   // cfg.cache_factorization
  float* d_cache_r = nullptr;
  uint8_t* d_cache_mask = nullptr;
  float* d_cache_meta = nullptr;
  uint8_t* d_cache_hit = nullptr;
  Staging st;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // cfg.time_kernel
  bool timed = false;
  std::atomic<int64_t> launches{0};
};

extern "C" {   // the definition sits inside the extern "C" block below, so the declaration carries C linkage too
namespace {
int flush_results(cmpc_handle* h);   // async host path, defined with it
}
}

namespace {

using SolveLaunch = cudaError_t (*)(const cmpc::SolveParams&, cudaStream_t);
using CondenseLaunch = cudaError_t (*)(const cmpc::CondenseParams&, cudaStream_t);
using ScoreLaunch = cudaError_t (*)(const cmpc::ScoreParams&, cudaStream_t);

// Programmatic dependent launch: the kernel may be scheduled while its predecessor in the stream is
// still running (its CTAs wait in griddepcontrol.wait before they touch global memory), which hides the
// launch latency between the two scheduling kernels and the solve kernel.  CMPC_NO_PDL=1 turns it off.
bool use_pdl() {
  static const bool on = std::getenv("CMPC_NO_PDL") == nullptr;
  return on;
}
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = use_pdl() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// Batches of 1.5-4 waves of resident CTAs (SCHED instantiations, with the LPT order: p.sched is set by
// schedule_batch) keep their hardest ranks on reserved, half-empty SMs (see "work distribution" in solve_kernel).
// CMPC_NO_RESERVE=1 / CMPC_HARD_SM=<n> are experiment switches.
template <int N, int SPLIT, int MINB, int R = 1, bool CACHE = false, bool TC = false, bool SCHED = false>
cudaError_t launch_solve(const cmpc::SolveParams& p_in, cudaStream_t s) {
  auto kernel = cmpc::solve_kernel<N, SPLIT, MINB, R, CACHE, TC, false>;
  constexpr int THREADS = cmpc::Geo<N, SPLIT, R>::THREADS;
  // 24 KB of static shared memory per CTA: MINB resident CTAs need the 196 KB carve-out (86 % of 228 KB); the
  // remaining 60 KB of L1 hold the register spills of the ADMM loop (CMPC_CARVEOUT=<percent> overrides)
  static const int carve_pct = std::getenv("CMPC_CARVEOUT") ? std::atoi(std::getenv("CMPC_CARVEOUT")) : 70;
  if (TC) {
    static const cudaError_t carve = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve_pct);
    if (carve != cudaSuccess) return carve;
  }
  cmpc::SolveParams p = p_in;
  if constexpr (SCHED) {
    auto skernel = cmpc::solve_kernel<N, SPLIT, MINB, R, CACHE, TC, true>;
    static const cudaError_t scarve = TC ? cudaFuncSetAttribute(skernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve_pct) : cudaSuccess;
    if (scarve != cudaSuccess) return scarve;
    static const int per_sm = [&] {      // resident CTAs of this kernel per SM
      int per = 0;
      return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, skernel, THREADS, 0) == cudaSuccess ? per : 0;
    }();
    static const int nsm = [&] {
      int dev = 0, n = 0;
      return cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess ? n : 0;
    }();
    const int wave = nsm * per_sm;       // CTAs the device holds at once
    static const bool reserve_on = std::getenv("CMPC_NO_RESERVE") == nullptr;
    static const int hard_sm = std::getenv("CMPC_HARD_SM") ? std::atoi(std::getenv("CMPC_HARD_SM")) : 32;
    // every reserved SM must receive its kHardSlots hard workers in the first wave (B > wave), and the other
    // SMs must be able to drain the main queue meanwhile
    // ... and only batches of 1.5-4 waves gain (scripts/gpu_reserve_sizes.py, 3 seeds per size, trot / mixed gaits:
    // 1536-3584 problems +2...+7 %; 1024 and >= 4096 problems -1...-6 %: in a long launch the hardest problems are over
    // long before the end, and the rank assignment costs every CTA two L2 round trips)
    if (p.sched && reserve_on && hard_sm > 0 && per_sm > cmpc::kHardSlots && nsm >= 2 * hard_sm && 2 * p.B > 3 * wave && p.B <= 4 * wave &&
        hard_sm * cmpc::kHardSlots <= p.B / 4) {
      p.n_hard_sm = hard_sm;
      p.n_hard = hard_sm * cmpc::kHardSlots;
      const int sleepers = hard_sm * (per_sm - cmpc::kHardSlots);   // as many spare CTAs as can sleep on the reserved SMs
      return launch_pdl(skernel, dim3((unsigned)(p.B + sleepers)), dim3(THREADS), 0, s, p);
    }
  }
  p.sched = nullptr;
  return launch_pdl(kernel, dim3((unsigned)p.B), dim3(THREADS), 0, s, p);
}
// one thread-block cluster of CL CTAs per problem (long horizons, see cmpc_cluster.cuh)
template <int NL, int CL, int SPLIT, int MINB>
cudaError_t launch_solve_cluster(const cmpc::SolveParams& p, cudaStream_t s) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(p.B * CL), 1, 1);
  cfg.blockDim = dim3(cmpc::CGeo<NL, CL, SPLIT>::THREADS, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, cmpc::solve_cluster_kernel<NL, CL, SPLIT, MINB>, p);
}
// stage-wise (Riccati) kernel: dynamic shared memory above the 48 KB default needs the opt-in
template <int N, int MINB>
cudaError_t launch_solve_riccati(const cmpc::SolveParams& p, cudaStream_t s) {
  using G_ = cmpc::RGeo<N>;
  static cudaError_t attr = cudaFuncSetAttribute(cmpc::solve_riccati_kernel<N, MINB>,
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G_::SMEM_BYTES);
  if (attr != cudaSuccess) return attr;
  return launch_pdl(cmpc::solve_riccati_kernel<N, MINB>, dim3((unsigned)p.B), dim3(G_::THREADS), G_::SMEM_BYTES, s, p);
}
template <int N>
cudaError_t launch_score(const cmpc::ScoreParams& p, cudaStream_t s) {
  return launch_pdl(cmpc::score_kernel<N>, dim3((unsigned)((p.B + 127) / 128)), dim3(128), 0, s, p);
}
template <int N>
cudaError_t launch_condense(const cmpc::CondenseParams& p, cudaStream_t s) {
  cmpc::condense_kernel<N><<<p.B, 256, 0, s>>>(p);
  return cudaGetLastError();
}

constexpr int kVariants = 6;
struct HorizonEntry {
  int N;
  SolveLaunch solve[kVariants];   // thread-layout variants (nullptr = not compiled)
  CondenseLaunch condense;
  ScoreLaunch score;
  SolveLaunch solve_cached;       // default layout with the factorisation cache compiled in, or nullptr
};

// Horizons with compiled kernels.  Dense kernels <N, SPLIT, MINB, R>: a thread owns an R x (6N/SPLIT)
// register tile of the 6N x 6N wrench matrix (R rows, one of SPLIT column slices), <= 96 floats.
// Slot 0 is the default kernel of the horizon:
//   N <= 16: dense single-CTA kernel (cmpc_kernels.cuh); N = 10: <10, 1, MINB = 6, 1, CACHE, TC, SCHED> = factorisation
//            sweep on the tensor cores (cmpc_tc.cuh), 6 CTAs/SM at 168 registers, reserved-SM rank assignment for
//            batches of 1.5-4 waves; slot 1 = the SIMT sweep at 8 CTAs/SM (round-1 layout), slot 2 = tensor-core sweep
//            at 8 CTAs/SM / 128 registers (scripts/gpu_tc_exp.py, gpu_carve_exp.py, gpu_reserve_exp.py);
//   N >= 20: stage-wise Riccati kernel (cmpc_riccati.cuh), measured on B200 against the dense / cluster
//            kernels: N=20 1.5x at 16384 problems (equal at 4096), N=30 2.25x (config 4), N=40 3.4x, N=60 5.2x
//            (scripts/gpu_riccati_exp.py, gpu_n20_kernels.py).
// Slot 2 of N = 20 / 30 is the thread-block-cluster kernel on the same horizon, slot 5 the "other"
// formulation (Riccati for N = 10, dense / cluster for N >= 20): tests compare the kernels on the same
// problems.  The remaining slots hold alternative dense layouts that were measured SLOWER (N=10: 8.4-10.7
// vs 12.4 M solves/s; N=30: 703 k vs 764 k) and are only compiled with -DCMPC_EXTRA_LAYOUTS
// (cmpc_has_variant tells).  Any other horizon N <= 60 runs padded on the next compiled one (pad_kernel).
#ifdef CMPC_EXTRA_LAYOUTS
#define CMPC_X(...) __VA_ARGS__
#else
#define CMPC_X(...) nullptr
#endif
const HorizonEntry kHorizons[] = {
    {4, {launch_solve<4, 1, 8>}, launch_condense<4>, launch_score<4>, nullptr},
    {5, {launch_solve<5, 1, 8>}, launch_condense<5>, launch_score<5>, nullptr},
    {8, {launch_solve<8, 1, 8>}, launch_condense<8>, launch_score<8>, nullptr},
    {10, {launch_solve<10, 1, 6, 1, false, true, true>, launch_solve<10, 1, 8>, launch_solve<10, 1, 8, 1, false, true, true>,
          CMPC_X(launch_solve<10, 2, 8, 2>), CMPC_X(launch_solve<10, 5, 8, 5>), launch_solve_riccati<10, 8>},
     launch_condense<10>, launch_score<10>, launch_solve<10, 1, 6, 1, true, true, true>},
    {12, {launch_solve<12, 2, 4>, nullptr, nullptr, nullptr, nullptr, launch_solve_riccati<12, 8>}, launch_condense<12>, launch_score<12>, nullptr},
    {16, {launch_solve<16, 2, 3>, nullptr, nullptr, nullptr, nullptr, launch_solve_riccati<16, 8>}, launch_condense<16>, launch_score<16>, nullptr},
    {20, {launch_solve_riccati<20, 6>, CMPC_X(launch_solve<20, 3, 1>), launch_solve_cluster<10, 2, 2, 3>, nullptr, nullptr,
          launch_solve<20, 2, 2>},
     launch_condense<20>, launch_score<20>, nullptr},
    {30, {launch_solve_riccati<30, 4>, CMPC_X(launch_solve<30, 3, 1>), launch_solve_cluster<10, 3, 3, 2>,
          CMPC_X(launch_solve<30, 6, 1, 2>), CMPC_X(launch_solve<30, 3, 1, 2>), launch_solve<30, 6, 1, 3>},
     launch_condense<30>, launch_score<30>, launch_solve<30, 6, 1, 3, true>},
    {40, {launch_solve_riccati<40, 3>, nullptr, nullptr, nullptr, nullptr, launch_solve_cluster<10, 4, 4, 1>},
     nullptr, launch_score<40>, nullptr},
    {60, {launch_solve_riccati<60, 2>, nullptr, nullptr, nullptr, nullptr, launch_solve_cluster<10, 6, 6, 1>},
     nullptr, launch_score<60>, nullptr},
};
constexpr int kMaxHorizon = 60;

const HorizonEntry* find_horizon(int N) {
  for (const auto& e : kHorizons)
    if (e.N == N) return &e;
  return nullptr;
}
// the compiled horizon a user horizon runs on: itself, or the next larger one (padded)
const HorizonEntry* kernel_horizon(int N) {
  if (N < 1) return nullptr;
  for (const auto& e : kHorizons)
    if (e.N >= N) return &e;
  return nullptr;
}

SolveLaunch pick_solve(const cmpc_handle* h) {
  const cmpc_config& c = h->cfg;
  const HorizonEntry* e = find_horizon(h->NK);
  if (c.cache_factorization && e->solve_cached) return e->solve_cached;
  const int v = (c.kernel_variant >= 0 && c.kernel_variant < kVariants) ? c.kernel_variant : 0;
  return e->solve[v] ? e->solve[v] : e->solve[0];
}

void fill_solve_params(const cmpc_handle* h, cmpc::SolveParams& p) {
  const cmpc_config& c = h->cfg;
  p.warm_x = h->d_warm_x;
  p.warm_y = h->d_warm_y;
  p.warm_valid = h->d_warm_valid;
  p.Minv = h->d_Minv;
  p.Mg = h->d_Mg;
  p.dt = c.dt;
  p.inv_mass = 1.0f / c.mass;
  for (int i = 0; i < 3; ++i) p.ib[i] = c.ibody_inv[i];
  for (int i = 0; i < 13; ++i) p.w[i] = c.w[i];
  p.r_weight = c.r_weight;
  p.f_min = c.f_min;
  p.f_max = c.f_max;
  p.rho = c.rho;
  p.sigma = c.sigma;
  p.alpha = c.alpha;
  p.eps_abs = c.eps_abs;
  p.eps_rel = c.eps_rel;
  p.max_iter = c.max_iter;
  p.check_every = c.check_every;
  p.refresh_every = c.refresh_every;
  p.warm_mode = c.warm_mode;
  p.adaptive_rho_interval = c.adaptive_rho_interval;
  p.adaptive_rho_tolerance = c.adaptive_rho_tolerance;
  p.rho_min = c.rho_min;
  p.rho_max = c.rho_max;
  static const float floor_ = std::getenv("CMPC_RHO_FLOOR") ? (float)std::atof(std::getenv("CMPC_RHO_FLOOR")) : cmpc::kRhoAdaptFloor;
  p.rho_adapt_floor = floor_;
  p.cache_pinv = h->d_cache_pinv;      // nullptr unless cfg.cache_factorization
  p.cache_r = h->d_cache_r;
  p.cache_mask = h->d_cache_mask;
  p.cache_meta = h->d_cache_meta;
  p.cache_tol_r = c.cache_tol_r;
  p.cache_tol_yaw = c.cache_tol_yaw;
  p.cache_max_iter = c.cache_max_iter;
  p.cache_hit = h->d_cache_hit;
  p.n_eff = c.N;                       // < NK on a padded horizon
}

// Enqueue the LPT ordering of a batch (2 small kernels) and point p.order at it.  The scratch
// (score, order, histogram) is carved out by the batch's slot range, so that disjoint slot ranges
// of one handle may be solved concurrently on different streams: order/score live at
// [slot0, slot0 + B), the histogram at slot0 / lpt_schedule (two disjoint ranges of >= lpt_schedule
// slots each cannot share that quotient).
int schedule_batch(cmpc_handle* h, cmpc::SolveParams& p, cudaStream_t s) {
  p.order = nullptr;
  p.sched = nullptr;
  if (!h->cfg.lpt_schedule || p.B < h->cfg.lpt_schedule) return CMPC_OK;
  if ((reinterpret_cast<uintptr_t>(p.r) & 15u) != 0) return CMPC_OK;   // score_kernel reads r with 16-byte loads
  const cmpc_config& c = h->cfg;
  const int hist_slot = p.slot0 / c.lpt_schedule;
  if (hist_slot >= h->hist_slots) return CMPC_OK;
  cmpc::ScoreParams sp{};
  sp.x0 = p.x0; sp.r = p.r; sp.mask = p.mask; sp.Mg = h->d_Mg; sp.mu = p.mu;
  static const int score_mode = std::getenv("CMPC_SCORE") ? std::atoi(std::getenv("CMPC_SCORE")) : 0;   // experiment switch
  sp.mode = score_mode;
  sp.score = h->d_score + p.slot0;
  sp.hist = h->d_hist + 64 * hist_slot;
  sp.B = p.B;
  sp.inv_mass = 1.0f / c.mass;
  for (int i = 0; i < 3; ++i) sp.ib[i] = c.ibody_inv[i];
  // (one fused single-CTA score+sort kernel was measured slower than these two launches:
  // its dependent load rounds cost more than the kernel boundary it saves)
  CUDA_TRY(find_horizon(h->NK)->score(sp, s));
  CUDA_TRY(launch_pdl(cmpc::order_kernel, dim3(1), dim3(1024), 0, s, (const float*)sp.score, sp.hist,
                      h->d_order + p.slot0, p.B));
  h->launches.fetch_add(2);
  p.order = h->d_order + p.slot0;
  p.sched = h->d_sched + (size_t)cmpc::kSchedInts * hist_slot;   // used by the dense kernels for batches of 1.5-4 waves
  return CMPC_OK;
}

// pad -> schedule -> solve -> unpad of one batch on one stream; all pointers are device-visible
// (device memory, or page-locked host memory mapped into the device's address space)
int solve_device(cmpc_handle* h, int B, int slot0, const float* x0, const float* r, const uint8_t* mask,
                 const float* x_des, const float* mu, float* U, float* X, int32_t* iters, float* pri_res,
                 float* dua_res, int32_t* status, cudaStream_t s, bool timed, bool plain_launch = false) {
  const int N = h->cfg.N, NK = h->NK;
  cmpc::SolveParams p{};
  fill_solve_params(h, p);
  p.x0 = x0; p.mu = mu; p.iters = iters; p.pri_res = pri_res; p.dua_res = dua_res; p.status = status;
  p.B = B;
  p.slot0 = slot0;
  if (NK == N) {
    p.r = r; p.mask = mask; p.x_des = x_des; p.U = U; p.X = X;
  } else {
    cmpc::PadParams pp{};
    pp.r = r; pp.mask = mask; pp.x_des = x_des;
    pp.r_k = h->d_pad_r + (size_t)slot0 * 12 * NK;
    pp.mask_k = h->d_pad_mask + (size_t)slot0 * NK;
    pp.x_des_k = h->d_pad_xdes + (size_t)slot0 * 13 * (NK + 1);
    pp.B = B; pp.N = N; pp.NK = NK;
    const long long items = (long long)B * (12 * NK + 13 * (NK + 1) + NK);
    cmpc::pad_kernel<<<(unsigned)((items + 255) / 256), 256, 0, s>>>(pp);
    CUDA_TRY(cudaGetLastError());
    h->launches.fetch_add(1);
    p.r = pp.r_k; p.mask = pp.mask_k; p.x_des = pp.x_des_k;
    p.U = h->d_pad_U + (size_t)slot0 * 12 * NK;
    p.X = X ? h->d_pad_X + (size_t)slot0 * 13 * (NK + 1) : nullptr;
  }
  int rc = schedule_batch(h, p, s);
  if (rc) return rc;
  if (plain_launch) p.sched = nullptr;   // chunked host path: the launch shares the device with its sibling chunk
  static const bool dbg = std::getenv("CMPC_DEBUG_CLOCKS") != nullptr;   // developer aid, synchronous
  if (dbg) { CUDA_TRY(cudaMalloc(&p.dbg_clk, 32 * sizeof(long long))); CUDA_TRY(cudaMemset(p.dbg_clk, 0, 32 * sizeof(long long))); }
  static const char* tl_path = std::getenv("CMPC_DEBUG_TIMELINE");          // developer aid, synchronous
  if (tl_path) { CUDA_TRY(cudaMalloc(&p.dbg_tl, (size_t)B * 4 * sizeof(long long))); CUDA_TRY(cudaMemset(p.dbg_tl, 0, (size_t)B * 4 * sizeof(long long))); }
  if (timed) {
    if (!h->ev0) { CUDA_TRY(cudaEventCreate(&h->ev0)); CUDA_TRY(cudaEventCreate(&h->ev1)); }
    CUDA_TRY(cudaEventRecord(h->ev0, s));
  }
  CUDA_TRY(pick_solve(h)(p, s));
  if (timed) {
    CUDA_TRY(cudaEventRecord(h->ev1, s));
    h->timed = true;
  }
  h->launches.fetch_add(1);
  if (tl_path) {   // per-CTA timeline of this launch: [B][4] int64 (start ns, end ns, SM, iterations), launch order
    std::vector<long long> tl((size_t)B * 4);
    CUDA_TRY(cudaStreamSynchronize(s));   // the launching stream may be a non-blocking one
    CUDA_TRY(cudaMemcpy(tl.data(), p.dbg_tl, tl.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    cudaFree(p.dbg_tl);
    if (FILE* f = std::fopen(tl_path, "wb")) { std::fwrite(tl.data(), sizeof(long long), tl.size(), f); std::fclose(f); }
  }
  if (dbg) {
    long long c[32];
    CUDA_TRY(cudaMemcpy(c, p.dbg_clk, sizeof c, cudaMemcpyDeviceToHost));
    cudaFree(p.dbg_clk);
    if (c[8] || c[9])
      std::fprintf(stderr, "cmpc riccati clocks (CTA 0, totals): setup %lld factor %lld | legA+check %lld P1 %lld sweeps+barrier %lld "
                           "(backward %lld forward %lld adjoint %lld) legB %lld | exit %lld\n",
                   c[8], c[9], c[11], c[12], c[17], c[13], c[15], c[16], c[18], c[19]);
    std::fprintf(stderr, "cmpc clocks (CTA 0): load %lld geometry %lld P-build %lld sweep %lld init %lld admm %lld output %lld\n",
                 c[1] - c[0], c[2] - c[1], c[3] - c[2], c[4] - c[3], c[5] - c[4], c[6] - c[5], c[7] - c[6]);
  }
  if (NK != N) {
    cmpc::UnpadParams up{};
    up.U_k = p.U; up.X_k = p.X; up.U = U; up.X = X; up.B = B; up.N = N; up.NK = NK;
    const long long items = (long long)B * (12 * N + (X ? 13 * (N + 1) : 0));
    cmpc::unpad_kernel<<<(unsigned)((items + 255) / 256), 256, 0, s>>>(up);
    CUDA_TRY(cudaGetLastError());
    h->launches.fetch_add(1);
  }
  return CMPC_OK;
}

int check_batch(const cmpc_handle* h, int B, int slot0) {
  if (!h) return fail(CMPC_ERR_INVALID, "null handle");
  if (B < 0 || slot0 < 0 || (int64_t)slot0 + B > h->cfg.max_batch)
    return fail(CMPC_ERR_INVALID, "batch [%d,%d) outside the handle's %d slots", slot0, slot0 + B,
                h->cfg.max_batch);
  return CMPC_OK;
}

}  // namespace

extern "C" {

int cmpc_version(void) { return CMPC_VERSION_MAJOR * 1000 + CMPC_VERSION_MINOR; }

const char* cmpc_last_error(void) { return g_err.c_str(); }

int cmpc_supported_horizons(int32_t* out, int32_t cap) {
  int n = 0;
  for (const auto& e : kHorizons) {
    if (out && n < cap) out[n] = e.N;
    ++n;
  }
  return n;
}

int cmpc_max_horizon(void) { return kMaxHorizon; }

int cmpc_kernel_horizon(int32_t N) {
  const HorizonEntry* e = kernel_horizon(N);
  return e ? e->N : fail(CMPC_ERR_UNSUPPORTED, "horizon N=%d is outside 1..%d", N, kMaxHorizon);
}

int cmpc_has_variant(int32_t N, int32_t variant) {
  const HorizonEntry* e = kernel_horizon(N);
  if (!e || variant < 0 || variant >= kVariants) return 0;
  return e->solve[variant] != nullptr ? 1 : 0;
}

int cmpc_default_config(cmpc_config* cfg, int32_t N, int32_t max_batch) {
  if (!cfg) return fail(CMPC_ERR_INVALID, "null config");
  std::memset(cfg, 0, sizeof *cfg);
  cfg->N = N;
  cfg->max_batch = max_batch;
  cfg->dt = 0.01f;                      // world.getTimeStep(), reference src/main.py:37
  cfg->mass = 8.885f;                   // src/mpc.py:71
  cfg->ibody_inv[0] = 1.0f / 0.24f;     // src/mpc.py:73-76
  cfg->ibody_inv[1] = 1.0f;
  cfg->ibody_inv[2] = 1.0f;
  const float w[13] = {1e4f, 2.7e4f, 1e4f, 2.7e5f, 2.7e5f, 2.7e5f, 1e4f,
                       1e4f, 1e4f, 1.6e4f, 1.6e4f, 1.6e4f, 0.f};   // src/mpc.py:121-134
  std::memcpy(cfg->w, w, sizeof w);
  cfg->r_weight = 0.0f;                 // src/mpc.py:121
  cfg->f_min = 3.0f;                    // src/mpc.py:45-46
  cfg->f_max = 100.0f;
  // rho_0 follows the scale of H, which grows with the horizon (measured on the Lite3
  // workloads: 0.5 is best at N=10, 1-3 at N=30, 2-8 at N=60)
  const HorizonEntry* he = kernel_horizon(N);
  const bool stagewise = he && he->N >= 20;          // default kernel = Riccati (slot 0 of kHorizons)
  cfg->rho = 0.05f * (float)N;
  cfg->sigma = 1e-6f;
  cfg->alpha = 1.6f;
  cfg->eps_abs = 1e-3f;                 // OSQP defaults (reference keeps them)
  cfg->eps_rel = 1e-3f;
  cfg->max_iter = 1000;                 // src/mpc.py:51
  cfg->check_every = 5;
  cfg->refresh_every = 5;
  cfg->warm_mode = CMPC_WARM_PRIMAL;
  cfg->adaptive_rho_interval = 25;      // OSQP adapts rho too (adaptive_rho = 1 by default)
  // refactorise when rho moves by more than this factor.  A dense refactorisation costs ~40 (N=10) to ~80
  // (N=30) iterations, a Riccati one ~6: with the stage-wise kernel a tight tolerance pays (measured,
  // scripts/gpu_ric_rho_sweep.py: N=30 3.49 -> 2.47 ms per 4096 problems, N=60 8.27 -> 4.81 ms per 512; the
  // hardest problem drops from 580 to 385 and from 860 to 485 iterations.  A larger rho_0 = 0.1 N is faster
  // still (N=60: 3.95 ms) but stops at objectives 4-5 % above the optimum instead of < 2 %: not adopted)
  cfg->adaptive_rho_tolerance = stagewise ? 1.5f : 3.0f;
  cfg->rho_min = 0.1f * cfg->rho;       // fp32 Woodbury form loses accuracy for rho << |H|
  cfg->rho_max = 300.0f;                // problems with far-away duals want rho ~ 100
  cfg->lpt_schedule = 1024;             // hardest-first launch order for batches >= this size
  cfg->device = 0;
  cfg->host_zero_copy = 1;              // pinned caller buffers are accessed in place
  cfg->cache_factorization = 0;         // closed-loop callers switch it on (rollout.py)
  cfg->cache_tol_r = 2e-3f;
  cfg->cache_tol_yaw = 2e-3f;
  cfg->cache_max_iter = 30;
  return CMPC_OK;
}

int cmpc_create(const cmpc_config* cfg, cmpc_handle** out) {
  if (!cfg || !out) return fail(CMPC_ERR_INVALID, "null argument");
  *out = nullptr;
  const cmpc_config& c = *cfg;
  const HorizonEntry* he = kernel_horizon(c.N);
  if (!he)
    return fail(CMPC_ERR_UNSUPPORTED, "horizon N=%d is outside 1..%d (largest compiled kernel)", c.N, kMaxHorizon);
  if (c.max_batch <= 0) return fail(CMPC_ERR_INVALID, "max_batch must be positive");
  if (!(c.dt > 0) || !(c.mass > 0) || !(c.rho > 0) || !(c.sigma >= 0) || !(c.alpha > 0 && c.alpha < 2))
    return fail(CMPC_ERR_INVALID, "dt, mass, rho must be > 0, sigma >= 0, 0 < alpha < 2");
  if (!(c.f_min >= 0.f) || !(c.f_min <= c.f_max)) return fail(CMPC_ERR_INVALID, "0 <= f_min <= f_max required");
  if (c.max_iter < 0 || c.check_every <= 0 || c.refresh_every < 0)
    return fail(CMPC_ERR_INVALID, "max_iter >= 0, check_every > 0, refresh_every >= 0 required");
  if (c.warm_mode < 0 || c.warm_mode > 2) return fail(CMPC_ERR_INVALID, "bad warm_mode");
  if (c.cache_factorization && (!(c.cache_tol_r >= 0.f) || !(c.cache_tol_yaw >= 0.f) || c.cache_max_iter < 0))
    return fail(CMPC_ERR_INVALID, "cache tolerances and cache_max_iter must be >= 0");
  if (c.cache_factorization && c.refresh_every > 0 && c.check_every % c.refresh_every != 0)
    return fail(CMPC_ERR_INVALID, "with cache_factorization the termination test must run on a freshly "
                                  "recomputed gradient: check_every must be a multiple of refresh_every");
  if (c.lpt_schedule < 0) return fail(CMPC_ERR_INVALID, "lpt_schedule must be >= 0");
  if (c.adaptive_rho_interval < 0 || (c.adaptive_rho_interval > 0 && !(c.adaptive_rho_tolerance > 1.f)))
    return fail(CMPC_ERR_INVALID, "adaptive_rho_interval >= 0 and adaptive_rho_tolerance > 1 required");
  if (!(c.rho_min > 0.f) || !(c.rho_min <= c.rho_max)) return fail(CMPC_ERR_INVALID, "0 < rho_min <= rho_max required");
  for (int i = 0; i < 12; ++i)
    if (!(c.w[i] >= 0)) return fail(CMPC_ERR_INVALID, "state weights must be >= 0");
  if (c.w[6] != c.w[7])
    return fail(CMPC_ERR_UNSUPPORTED,
                "the wrench-space form needs equal x/y angular-velocity weights (w[6]==w[7])");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(CMPC_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
  }
  if (c.device < 0 || c.device >= ndev) return fail(CMPC_ERR_INVALID, "device %d of %d", c.device, ndev);
  DeviceGuard guard_(c.device);
  if (guard_.err != cudaSuccess)
    return fail(CMPC_ERR_CUDA, "cudaSetDevice(%d) failed: %s", c.device, cudaGetErrorString(guard_.err));

  const int Nu = c.N, N = he->N;       // user horizon, kernel horizon (N > Nu: padded, see pad_kernel)
  std::vector<double> Mu, Miu;
  axis_gram(Nu, (double)c.dt, c.w, Mu);
  Miu = Mu;
  for (int a = 0; a < 6; ++a) {
    // plain Gauss-Jordan with the textbook sign handling
    double* A = Miu.data() + (size_t)a * Nu * Nu;
    std::vector<double> aug((size_t)Nu * 2 * Nu, 0.0);
    for (int i = 0; i < Nu; ++i) {
      for (int j = 0; j < Nu; ++j) aug[(size_t)i * 2 * Nu + j] = A[i * Nu + j];
      aug[(size_t)i * 2 * Nu + Nu + i] = 1.0;
    }
    for (int k = 0; k < Nu; ++k) {
      const double piv = aug[(size_t)k * 2 * Nu + k];
      if (!(piv > 0.0) || !std::isfinite(piv))
        return fail(CMPC_ERR_INVALID, "horizon Gram matrix of axis %d is not positive definite "
                                      "(position and velocity weight both zero?)", a);
      for (int j = 0; j < 2 * Nu; ++j) aug[(size_t)k * 2 * Nu + j] /= piv;
      for (int i = 0; i < Nu; ++i) {
        if (i == k) continue;
        const double f = aug[(size_t)i * 2 * Nu + k];
        if (f == 0.0) continue;
        for (int j = 0; j < 2 * Nu; ++j) aug[(size_t)i * 2 * Nu + j] -= f * aug[(size_t)k * 2 * Nu + j];
      }
    }
    for (int i = 0; i < Nu; ++i)
      for (int j = 0; j < Nu; ++j) A[i * Nu + j] = aug[(size_t)i * 2 * Nu + Nu + j];
  }
  // embed into the kernel horizon: blockdiag(M_Nu, I) per axis (the tail stages are all-swing, their
  // wrench rows decouple; any positive definite filler works)
  std::vector<float> Mf((size_t)6 * N * N, 0.f), Mif((size_t)6 * N * N, 0.f);
  for (int a = 0; a < 6; ++a)
    for (int i = 0; i < N; ++i)
      for (int j = 0; j < N; ++j) {
        const size_t o = ((size_t)a * N + i) * N + j;
        if (i < Nu && j < Nu) {
          Mf[o] = (float)Mu[((size_t)a * Nu + i) * Nu + j];
          Mif[o] = (float)Miu[((size_t)a * Nu + i) * Nu + j];
        } else if (i == j) {
          Mf[o] = 1.f;
          Mif[o] = 1.f;
        }
      }

  cmpc_handle* h = new cmpc_handle();
  h->cfg = c;
  h->NK = N;
  h->hist_slots = c.lpt_schedule > 0 ? c.max_batch / c.lpt_schedule + 1 : 1;
  const size_t mbytes = sizeof(float) * 6 * N * N;
  const size_t slots = (size_t)c.max_batch;
  cudaError_t e;
  if ((e = cudaMalloc(&h->d_Minv, mbytes)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_Mg, mbytes)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_warm_x, slots * 12 * N * sizeof(float))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_warm_y, slots * 12 * N * sizeof(float))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_warm_valid, slots)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_score, slots * sizeof(float))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_order, slots * sizeof(int32_t))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_hist, (size_t)h->hist_slots * 64 * sizeof(int32_t))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_sched, (size_t)h->hist_slots * cmpc::kSchedInts * sizeof(int32_t))) != cudaSuccess ||
      (e = cudaMemset(h->d_sched, 0, (size_t)h->hist_slots * cmpc::kSchedInts * sizeof(int32_t))) != cudaSuccess ||
      (e = cudaMemcpy(h->d_Minv, Mif.data(), mbytes, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(h->d_Mg, Mf.data(), mbytes, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemset(h->d_warm_x, 0, slots * 12 * N * sizeof(float))) != cudaSuccess ||
      (e = cudaMemset(h->d_warm_y, 0, slots * 12 * N * sizeof(float))) != cudaSuccess ||
      (e = cudaMemset(h->d_warm_valid, 0, slots)) != cudaSuccess ||
      (e = cudaMemset(h->d_hist, 0, (size_t)h->hist_slots * 64 * sizeof(int32_t))) != cudaSuccess) {
    cmpc_destroy(h);
    return fail(CMPC_ERR_CUDA, "device allocation failed: %s", cudaGetErrorString(e));
  }
  if (c.cache_factorization && !find_horizon(N)->solve_cached) {
    cmpc_destroy(h);
    return fail(CMPC_ERR_UNSUPPORTED, "cache_factorization is compiled for the N = 10 and N = 30 kernels only");
  }
  if (N != Nu) {
    if ((e = cudaMalloc(&h->d_pad_r, slots * 12 * N * sizeof(float))) != cudaSuccess ||
        (e = cudaMalloc(&h->d_pad_mask, slots * N)) != cudaSuccess ||
        (e = cudaMalloc(&h->d_pad_xdes, slots * 13 * (N + 1) * sizeof(float))) != cudaSuccess ||
        (e = cudaMalloc(&h->d_pad_U, slots * 12 * N * sizeof(float))) != cudaSuccess ||
        (e = cudaMalloc(&h->d_pad_X, slots * 13 * (N + 1) * sizeof(float))) != cudaSuccess) {
      cmpc_destroy(h);
      return fail(CMPC_ERR_CUDA, "padded-horizon scratch allocation failed: %s", cudaGetErrorString(e));
    }
  }
  if (c.cache_factorization) {
    // a tile row is padded to a multiple of 4 SPLIT floats, SPLIT <= 6 in the compiled layouts
    const size_t NW = 6 * (size_t)N, per_entry = NW * (NW + 20) * sizeof(float);
    const size_t entries = slots;
    if ((e = cudaMalloc(&h->d_cache_pinv, entries * per_entry)) != cudaSuccess ||
        (e = cudaMalloc(&h->d_cache_r, entries * 12 * N * sizeof(float))) != cudaSuccess ||
        (e = cudaMalloc(&h->d_cache_mask, entries * N)) != cudaSuccess ||
        (e = cudaMalloc(&h->d_cache_meta, entries * 4 * sizeof(float))) != cudaSuccess ||
        (e = cudaMalloc(&h->d_cache_hit, slots)) != cudaSuccess ||
        (e = cudaMemset(h->d_cache_hit, 0, slots)) != cudaSuccess ||
        (e = cudaMemset(h->d_cache_meta, 0, entries * 4 * sizeof(float))) != cudaSuccess) {
      cmpc_destroy(h);
      return fail(CMPC_ERR_CUDA, "factorisation cache allocation failed: %s", cudaGetErrorString(e));
    }
  }
  *out = h;
  return CMPC_OK;
}

int cmpc_destroy(cmpc_handle* h) {
  if (!h) return CMPC_OK;
  DeviceGuard guard_(h->cfg.device);
  cudaFree(h->d_pad_r);
  cudaFree(h->d_pad_mask);
  cudaFree(h->d_pad_xdes);
  cudaFree(h->d_pad_U);
  cudaFree(h->d_pad_X);
  cudaFree(h->d_Minv);
  cudaFree(h->d_Mg);
  cudaFree(h->d_warm_x);
  cudaFree(h->d_warm_y);
  cudaFree(h->d_warm_valid);
  cudaFree(h->d_score);
  cudaFree(h->d_order);
  cudaFree(h->d_hist);
  cudaFree(h->d_sched);
  cudaFree(h->d_cache_pinv);
  cudaFree(h->d_cache_r);
  cudaFree(h->d_cache_mask);
  cudaFree(h->d_cache_meta);
  cudaFree(h->d_cache_hit);
  if (h->st.h_in) cudaFreeHost(h->st.h_in);
  if (h->st.h_out) cudaFreeHost(h->st.h_out);
  cudaFree(h->st.d_in);
  cudaFree(h->st.d_out);
  for (auto& s : h->st.streams)
    if (s) cudaStreamDestroy(s);
  if (h->st.pending.active) { flush_results(h); cudaStreamSynchronize(h->st.d2h); }
  for (auto& e : h->st.done)
    if (e) cudaEventDestroy(e);
  for (auto& e : h->st.h2d)
    if (e) cudaEventDestroy(e);
  for (auto& e : h->st.h2d2)
    if (e) cudaEventDestroy(e);
  if (h->st.copy2) cudaStreamDestroy(h->st.copy2);
  if (h->st.d2h) cudaStreamDestroy(h->st.d2h);
  for (auto& e : h->st.solved)
    if (e) cudaEventDestroy(e);
  for (auto& q : h->st.d_async_out) cudaFree(q);
  for (auto& q : h->st.d_async_in) cudaFree(q);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  delete h;
  return CMPC_OK;
}

int64_t cmpc_launch_count(const cmpc_handle* h) { return h ? h->launches.load() : 0; }

int cmpc_accumulate_stats(cmpc_handle* h, int32_t B, int32_t slot0, const int32_t* iters,
                          const int32_t* status, uint64_t* acc, void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (B == 0) return CMPC_OK;
  if (!iters || !status || !acc) return fail(CMPC_ERR_INVALID, "null pointer");
  DEVICE_GUARD(h);
  cmpc::stats_kernel<<<(B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      iters, status, h->d_cache_hit ? h->d_cache_hit + slot0 : nullptr, B,
      reinterpret_cast<unsigned long long*>(acc));
  CUDA_TRY(cudaGetLastError());
  h->launches.fetch_add(1);
  return CMPC_OK;
}

int cmpc_get_cache_meta(cmpc_handle* h, int32_t B, int32_t slot0, float* meta, void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!meta) return fail(CMPC_ERR_INVALID, "null pointer");
  if (!h->d_cache_meta) return fail(CMPC_ERR_INVALID, "the handle was created without cache_factorization");
  DEVICE_GUARD(h);
  CUDA_TRY(cudaMemcpyAsync(meta, h->d_cache_meta + (size_t)slot0 * 4, (size_t)B * 4 * sizeof(float),
                           cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return CMPC_OK;
}

int cmpc_last_kernel_ms(cmpc_handle* h, float* ms) {
  if (!h || !ms) return fail(CMPC_ERR_INVALID, "null argument");
  if (!h->timed) return fail(CMPC_ERR_INVALID, "no timed solve yet (set cfg.time_kernel and call cmpc_solve)");
  CUDA_TRY(cudaEventSynchronize(h->ev1));
  CUDA_TRY(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  return CMPC_OK;
}

int cmpc_solve(cmpc_handle* h, int32_t B, int32_t slot0, const float* x0, const float* r,
               const uint8_t* mask, const float* x_des, const float* mu, float* U, float* X,
               int32_t* iters, float* pri_res, float* dua_res, int32_t* status, void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (B == 0) return CMPC_OK;
  if (!x0 || !r || !mask || !x_des || !mu || !U) return fail(CMPC_ERR_INVALID, "null input/output pointer");
  DEVICE_GUARD(h);
  return solve_device(h, B, slot0, x0, r, mask, x_des, mu, U, X, iters, pri_res, dua_res, status,
                      (cudaStream_t)stream, h->cfg.time_kernel != 0);
}

int cmpc_condense(cmpc_handle* h, int32_t B, const float* x0, const float* r, const uint8_t* mask,
                  const float* x_des, float* H, float* g, void* stream) {
  if (!h) return fail(CMPC_ERR_INVALID, "null handle");
  if (B < 0) return fail(CMPC_ERR_INVALID, "negative batch");
  if (B == 0) return CMPC_OK;
  if (!x0 || !r || !mask || !x_des || !H || !g) return fail(CMPC_ERR_INVALID, "null pointer");
  DEVICE_GUARD(h);
  cmpc::CondenseParams p{};
  const cmpc_config& c = h->cfg;
  p.x0 = x0; p.r = r; p.mask = mask; p.x_des = x_des; p.H = H; p.g = g; p.Mg = h->d_Mg;
  p.B = B;
  p.dt = c.dt;
  p.inv_mass = 1.0f / c.mass;
  for (int i = 0; i < 3; ++i) p.ib[i] = c.ibody_inv[i];
  for (int i = 0; i < 13; ++i) p.w[i] = c.w[i];
  p.r_weight = c.r_weight;
  if (h->NK != c.N || !find_horizon(c.N)->condense)
    return fail(CMPC_ERR_UNSUPPORTED, "cmpc_condense (dense H export, inspection path) is compiled for "
                "N in {4,5,8,10,12,16,20,30} only, not N=%d", c.N);
  CUDA_TRY(find_horizon(c.N)->condense(p, (cudaStream_t)stream));
  h->launches.fetch_add(1);
  return CMPC_OK;
}

namespace {
void fill_gait(const cmpc_handle* h, const cmpc_gait_tables* g, cmpc::GaitTables& o) {
  o.plan_pos = g->plan_pos; o.feet_id = g->feet_id; o.ss = g->ss; o.ds = g->ds;
  o.v_ref = g->v_ref; o.omega_ref = g->omega_ref; o.rp0 = g->rp0;
  o.S = g->S; o.total_steps = g->total_steps; o.step_height = g->step_height; o.g = g->g;
  o.dt = h->cfg.dt;
}
int check_gait(const cmpc_gait_tables* g) {
  if (!g || !g->plan_pos || !g->feet_id || !g->ss || !g->ds || !g->v_ref || !g->omega_ref || !g->rp0)
    return fail(CMPC_ERR_INVALID, "null gait table pointer");
  if (g->S <= 0) return fail(CMPC_ERR_INVALID, "gait tables need at least one step");
  return CMPC_OK;
}
}  // namespace

int cmpc_assemble(cmpc_handle* h, int32_t B, const cmpc_gait_tables* gt, const int32_t* tick,
                  const float* x, const float* yaw_start, const float* com_start, float* x_des,
                  float* r, uint8_t* mask, void* stream) {
  if (!h) return fail(CMPC_ERR_INVALID, "null handle");
  if (B < 0) return fail(CMPC_ERR_INVALID, "negative batch");
  int rc = check_gait(gt);
  if (rc) return rc;
  if (B == 0) return CMPC_OK;
  if (!tick || !x || !yaw_start || !com_start || !x_des || !r || !mask)
    return fail(CMPC_ERR_INVALID, "null pointer");
  DEVICE_GUARD(h);
  cmpc::AssembleParams p{};
  fill_gait(h, gt, p.gt);
  p.tick = tick; p.x = x; p.yaw_start = yaw_start; p.com_start = com_start;
  p.x_des = x_des; p.r = r; p.mask = mask; p.B = B; p.N = h->cfg.N;
  {
    const long long total = (long long)B * (p.N + 1);
    cmpc::assemble_kernel<<<(unsigned)((total + 127) / 128), 128, 0, (cudaStream_t)stream>>>(p);
    CUDA_TRY(cudaGetLastError());
  }
  h->launches.fetch_add(1);
  return CMPC_OK;
}

int cmpc_plant_step(cmpc_handle* h, int32_t B, const cmpc_gait_tables* gt, int32_t* tick, float* x,
                    const float* r, const float* U, const float* x_des, float* yaw_start,
                    float* com_start, float* track_err, void* stream) {
  if (!h) return fail(CMPC_ERR_INVALID, "null handle");
  if (B < 0) return fail(CMPC_ERR_INVALID, "negative batch");
  int rc = check_gait(gt);
  if (rc) return rc;
  if (!tick || ((!x || !r || !U || !x_des || !yaw_start || !com_start || !track_err) && B > 0))
    return fail(CMPC_ERR_INVALID, "null pointer");
  DEVICE_GUARD(h);
  cudaStream_t s = (cudaStream_t)stream;
  if (B > 0) {
    cmpc::PlantParams p{};
    fill_gait(h, gt, p.gt);
    p.tick = tick; p.x = x; p.r = r; p.U = U; p.x_des = x_des; p.yaw_start = yaw_start;
    p.com_start = com_start; p.track_err = track_err; p.B = B; p.N = h->cfg.N;
    p.inv_mass = 1.0f / h->cfg.mass;
    for (int i = 0; i < 3; ++i) p.ib[i] = h->cfg.ibody_inv[i];
    cmpc::plant_kernel<<<(B + 127) / 128, 128, 0, s>>>(p);
    CUDA_TRY(cudaGetLastError());
  }
  cmpc::tick_kernel<<<1, 1, 0, s>>>(tick);
  CUDA_TRY(cudaGetLastError());
  h->launches.fetch_add(B > 0 ? 2 : 1);
  return CMPC_OK;
}

int cmpc_leg_torques(cmpc_handle* h, int32_t B, const cmpc_gait_tables* gt, const int32_t* tick,
                     const float* U, const float* J, const float* Jdot, const float* Mleg,
                     const float* cg, const float* dq, const float* foot_pos, const float* foot_vel,
                     const float* kp, const float* kd, float* tau, float* p_des, uint8_t* stance,
                     void* stream) {
  if (!h) return fail(CMPC_ERR_INVALID, "null handle");
  if (B < 0) return fail(CMPC_ERR_INVALID, "negative batch");
  int rc = check_gait(gt);
  if (rc) return rc;
  if (B == 0) return CMPC_OK;
  if (!tick || !U || !J || !Jdot || !Mleg || !cg || !dq || !foot_pos || !foot_vel || !kp || !kd || !tau)
    return fail(CMPC_ERR_INVALID, "null pointer");
  DEVICE_GUARD(h);
  cmpc::LegParams p{};
  fill_gait(h, gt, p.gt);
  p.tick = tick; p.U = U; p.J = J; p.Jdot = Jdot; p.Mleg = Mleg; p.cg = cg; p.dq = dq;
  p.foot_pos = foot_pos; p.foot_vel = foot_vel; p.tau = tau; p.p_des = p_des; p.stance = stance;
  p.B = B; p.N = h->cfg.N;
  for (int i = 0; i < 3; ++i) { p.kp[i] = kp[i]; p.kd[i] = kd[i]; }
  cmpc::leg_torque_kernel<<<(4 * B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  h->launches.fetch_add(1);
  return CMPC_OK;
}

int cmpc_leg_kinematics(cmpc_handle* h, int32_t B, const float* base_pos, const float* theta,
                        const float* v_base, const float* w_base, const float* q, const float* dq,
                        float* foot_pos, float* foot_vel, float* J, float* Jdot, float* Mleg, float* cg,
                        float gravity, void* stream) {
  if (!h) return fail(CMPC_ERR_INVALID, "null handle");
  if (B < 0) return fail(CMPC_ERR_INVALID, "negative batch");
  if (B == 0) return CMPC_OK;
  if (!base_pos || !theta || !v_base || !w_base || !q || !dq || !foot_pos || !foot_vel || !J || !Jdot)
    return fail(CMPC_ERR_INVALID, "null pointer");
  DEVICE_GUARD(h);
  cmpc::KinParams p{};
  p.base_pos = base_pos; p.theta = theta; p.v_base = v_base; p.w_base = w_base; p.q = q; p.dq = dq;
  p.foot_pos = foot_pos; p.foot_vel = foot_vel; p.J = J; p.Jdot = Jdot; p.Mleg = Mleg; p.cg = cg;
  p.B = B; p.g = gravity;
  cmpc::leg_kinematics_kernel<<<(4 * B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  h->launches.fetch_add(1);
  return CMPC_OK;
}

int cmpc_fp32_peak(int32_t device, float* tflops) {
  if (!tflops) return fail(CMPC_ERR_INVALID, "null pointer");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(CMPC_ERR_NO_DEVICE, "no CUDA device visible");
  }
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop{};
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  const int grid = prop.multiProcessorCount * 8, iters = 4096;
  float* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, (size_t)grid * 256 * sizeof(float)));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  float best = 0.f;
  for (int rep = 0; rep < 5; ++rep) {
    CUDA_TRY(cudaEventRecord(e0));
    cmpc::fma_peak_kernel<<<grid, 256>>>(d, iters, 0.999f, 0.001f);
    CUDA_TRY(cudaEventRecord(e1));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    const double flop = 2.0 * 64.0 * iters * 256.0 * grid;
    const float tf = (float)(flop / (ms * 1e-3) / 1e12);
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *tflops = best;
  return CMPC_OK;
}

// ---- host-buffer path -------------------------------------------------------------------
namespace {
struct Layout {   // byte offsets of one chunk of C problems inside the in/out arenas
  size_t x0, r, xdes, mu, mask, in_total;
  size_t U, X, iters, pri, dua, status, out_total;
};
Layout make_layout(int N, int C, bool withX) {
  Layout L{};
  auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
  size_t o = 0;
  L.x0 = o; o = al(o + (size_t)C * 13 * 4);
  L.r = o; o = al(o + (size_t)C * 12 * N * 4);
  L.xdes = o; o = al(o + (size_t)C * 13 * (N + 1) * 4);
  L.mu = o; o = al(o + (size_t)C * 4);
  L.mask = o; o = al(o + (size_t)C * N);
  L.in_total = o;
  o = 0;
  L.U = o; o = al(o + (size_t)C * 12 * N * 4);
  L.iters = o; o = al(o + (size_t)C * 4);
  L.pri = o; o = al(o + (size_t)C * 4);
  L.dua = o; o = al(o + (size_t)C * 4);
  L.status = o; o = al(o + (size_t)C * 4);
  L.X = o; if (withX) o = al(o + (size_t)C * 13 * (N + 1) * 4);
  L.out_total = o;
  return L;
}
}  // namespace

namespace {
// true if `ptr` is page-locked host memory the DMA engines can read/write directly;
// *dev (optional) receives the address under which kernels on the current device see it
bool is_pinned(const void* ptr, void** dev = nullptr) {
  if (dev) *dev = nullptr;
  if (!ptr) return true;
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  if (at.type != cudaMemoryTypeHost) return false;
  if (dev) *dev = at.devicePointer;
  return true;
}
}  // namespace

namespace {
// Result copies of the async host path.  They are enqueued one submission late - after the NEXT submission's input
// copies, or by cmpc_host_wait - because a copy that waits for its solve sits at the head of its hardware queue for
// the whole solve, and when the driver maps the input-copy streams onto that queue too (it varies from process
// to process) the next step's inputs wait behind it and the steps serialise (measured: 0.25 / 0.27 / 0.32 instead
// of 0.23 ms per step, the delay being the copy time of whichever stream shared the queue).
int flush_results(cmpc_handle* h) {
  Staging& st = h->st;
  Staging::Pending& q = st.pending;
  if (!q.active) return CMPC_OK;
  const int N = h->cfg.N;
  const Layout Lo = make_layout(N, h->cfg.max_batch, true);
  const char* dout = st.d_async_out[q.arena];
  const size_t B = (size_t)q.B;
  CUDA_TRY(cudaStreamWaitEvent(st.d2h, st.solved[q.arena], 0));
  CUDA_TRY(cudaMemcpyAsync(q.U, dout + Lo.U, B * 12 * N * 4, cudaMemcpyDeviceToHost, st.d2h));
  if (q.X) CUDA_TRY(cudaMemcpyAsync(q.X, dout + Lo.X, B * 13 * (N + 1) * 4, cudaMemcpyDeviceToHost, st.d2h));
  if (q.iters) CUDA_TRY(cudaMemcpyAsync(q.iters, dout + Lo.iters, B * 4, cudaMemcpyDeviceToHost, st.d2h));
  if (q.pri) CUDA_TRY(cudaMemcpyAsync(q.pri, dout + Lo.pri, B * 4, cudaMemcpyDeviceToHost, st.d2h));
  if (q.dua) CUDA_TRY(cudaMemcpyAsync(q.dua, dout + Lo.dua, B * 4, cudaMemcpyDeviceToHost, st.d2h));
  if (q.status) CUDA_TRY(cudaMemcpyAsync(q.status, dout + Lo.status, B * 4, cudaMemcpyDeviceToHost, st.d2h));
  CUDA_TRY(cudaEventRecord(st.done[q.ticket & 7], st.d2h));   // a ticket completes when its results are in host memory
  q.active = false;
  return CMPC_OK;
}
}  // namespace

namespace {
// Page-locked caller buffers: one launch over the whole batch, every CTA pulls its own
// ~1.1 KB record over PCIe and pushes its results back, so the transfers overlap the
// solve CTA by CTA and no copy is ever enqueued.  All accesses of the kernel to these
// buffers are coalesced and touch every byte once.  Returns 1 when the batch was enqueued on
// the host-path stream, 0 when the buffers are not all page-locked, < 0 on error.
int enqueue_zero_copy(cmpc_handle* h, int32_t B, int32_t slot0, const float* x0, const float* r,
                      const uint8_t* mask, const float* x_des, const float* mu, float* U, float* X,
                      int32_t* iters, float* pri_res, float* dua_res, int32_t* status) {
  Staging& st = h->st;
  void *dx0, *dr, *dmask, *dxd, *dmu, *dU, *dX, *dit, *dpr, *ddu, *dst;
  const bool ok = is_pinned(x0, &dx0) && is_pinned(r, &dr) && is_pinned(mask, &dmask) &&
                  is_pinned(x_des, &dxd) && is_pinned(mu, &dmu) && is_pinned(U, &dU) &&
                  is_pinned(X, &dX) && is_pinned(iters, &dit) && is_pinned(pri_res, &dpr) &&
                  is_pinned(dua_res, &ddu) && is_pinned(status, &dst);
  if (!(ok && dx0 && dr && dmask && dxd && dmu && dU)) return 0;
  if (!st.streams[0]) {
    if (cudaStreamCreateWithFlags(&st.streams[0], cudaStreamNonBlocking) != cudaSuccess)
      return fail(CMPC_ERR_CUDA, "stream creation failed");
  }
  const int rc = solve_device(h, B, slot0, (const float*)dx0, (const float*)dr, (const uint8_t*)dmask,
                              (const float*)dxd, (const float*)dmu, (float*)dU, (float*)dX, (int32_t*)dit,
                              (float*)dpr, (float*)ddu, (int32_t*)dst, st.streams[0], false);
  return rc ? (rc < 0 ? rc : -rc) : 1;
}
}  // namespace

int cmpc_solve_host(cmpc_handle* h, int32_t B, int32_t slot0, const float* x0, const float* r,
                    const uint8_t* mask, const float* x_des, const float* mu, float* U, float* X,
                    int32_t* iters, float* pri_res, float* dua_res, int32_t* status) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (B == 0) return CMPC_OK;
  if (!x0 || !r || !mask || !x_des || !mu || !U) return fail(CMPC_ERR_INVALID, "null input/output pointer");
  DEVICE_GUARD(h);
  const int N = h->cfg.N;
  Staging& st = h->st;
  rc = flush_results(h);      // an asynchronous submission may still owe its result copies
  if (rc) return rc;
  if (h->cfg.host_zero_copy) {
    rc = enqueue_zero_copy(h, B, slot0, x0, r, mask, x_des, mu, U, X, iters, pri_res, dua_res, status);
    if (rc < 0) return rc;
    if (rc == 1) {
      CUDA_TRY(cudaStreamSynchronize(st.streams[0]));
      return CMPC_OK;
    }
  }
  // Two chunks on two streams: H2D(1) overlaps solve(0), D2H(0) overlaps solve(1).  More
  // chunks would give every chunk its own straggler tail.
  const int nchunk = B >= 2048 ? 2 : 1;
  const int C = (B + nchunk - 1) / nchunk;
  // page-locked caller buffers are copied directly by the DMA engines; pageable ones are
  // staged through the handle's pinned arenas
  const bool in_pinned = is_pinned(x0) && is_pinned(r) && is_pinned(mask) && is_pinned(x_des) && is_pinned(mu);
  const bool out_pinned = is_pinned(U) && is_pinned(X) && is_pinned(iters) && is_pinned(pri_res) &&
                          is_pinned(dua_res) && is_pinned(status);
  const Layout L = make_layout(N, C, true);
  if (st.cap < C || !st.d_in) {
    if (st.h_in) cudaFreeHost(st.h_in);
    if (st.h_out) cudaFreeHost(st.h_out);
    cudaFree(st.d_in);
    cudaFree(st.d_out);
    st.h_in = st.h_out = st.d_in = st.d_out = nullptr;
    st.cap = 0;
    const size_t nb = 2;   // arenas per direction (= max chunks)
    CUDA_TRY(cudaMallocHost(&st.h_in, L.in_total * nb));
    CUDA_TRY(cudaMallocHost(&st.h_out, L.out_total * nb));
    CUDA_TRY(cudaMalloc(&st.d_in, L.in_total * nb));
    CUDA_TRY(cudaMalloc(&st.d_out, L.out_total * nb));
    st.in_bytes = L.in_total;
    st.out_bytes = L.out_total;
    st.cap = C;
    for (auto& s : st.streams)
      if (!s) CUDA_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  }
  const Layout La = make_layout(N, st.cap, true);   // arena strides use the allocated capacity
  const size_t nx = (size_t)13 * (N + 1), nu = (size_t)12 * N;
  for (int ci = 0; ci < nchunk; ++ci) {
    const int lo = ci * C, n = (lo + C <= B ? C : B - lo);
    if (n <= 0) break;
    cudaStream_t s = st.streams[ci];
    char* hin = st.h_in + (size_t)ci * st.in_bytes;
    char* din = st.d_in + (size_t)ci * st.in_bytes;
    char* dout = st.d_out + (size_t)ci * st.out_bytes;
    char* hout = st.h_out + (size_t)ci * st.out_bytes;
    if (in_pinned) {
      CUDA_TRY(cudaMemcpyAsync(din + La.x0, x0 + (size_t)lo * 13, (size_t)n * 13 * 4, cudaMemcpyHostToDevice, s));
      CUDA_TRY(cudaMemcpyAsync(din + La.r, r + (size_t)lo * nu, (size_t)n * nu * 4, cudaMemcpyHostToDevice, s));
      CUDA_TRY(cudaMemcpyAsync(din + La.xdes, x_des + (size_t)lo * nx, (size_t)n * nx * 4, cudaMemcpyHostToDevice, s));
      CUDA_TRY(cudaMemcpyAsync(din + La.mu, mu + lo, (size_t)n * 4, cudaMemcpyHostToDevice, s));
      CUDA_TRY(cudaMemcpyAsync(din + La.mask, mask + (size_t)lo * N, (size_t)n * N, cudaMemcpyHostToDevice, s));
    } else {
      std::memcpy(hin + La.x0, x0 + (size_t)lo * 13, (size_t)n * 13 * 4);
      std::memcpy(hin + La.r, r + (size_t)lo * nu, (size_t)n * nu * 4);
      std::memcpy(hin + La.xdes, x_des + (size_t)lo * nx, (size_t)n * nx * 4);
      std::memcpy(hin + La.mu, mu + lo, (size_t)n * 4);
      std::memcpy(hin + La.mask, mask + (size_t)lo * N, (size_t)n * N);
      CUDA_TRY(cudaMemcpyAsync(din, hin, La.in_total, cudaMemcpyHostToDevice, s));
    }
    rc = solve_device(h, n, slot0 + lo, (const float*)(din + La.x0), (const float*)(din + La.r),
                      (const uint8_t*)(din + La.mask), (const float*)(din + La.xdes),
                      (const float*)(din + La.mu), (float*)(dout + La.U),
                      X ? (float*)(dout + La.X) : nullptr, (int32_t*)(dout + La.iters),
                      (float*)(dout + La.pri), (float*)(dout + La.dua), (int32_t*)(dout + La.status), s, false,
                      nchunk > 1);
    if (rc) return rc;
    if (out_pinned) {
      CUDA_TRY(cudaMemcpyAsync(U + (size_t)lo * nu, dout + La.U, (size_t)n * nu * 4, cudaMemcpyDeviceToHost, s));
      if (X) CUDA_TRY(cudaMemcpyAsync(X + (size_t)lo * nx, dout + La.X, (size_t)n * nx * 4, cudaMemcpyDeviceToHost, s));
      if (iters) CUDA_TRY(cudaMemcpyAsync(iters + lo, dout + La.iters, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
      if (pri_res) CUDA_TRY(cudaMemcpyAsync(pri_res + lo, dout + La.pri, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
      if (dua_res) CUDA_TRY(cudaMemcpyAsync(dua_res + lo, dout + La.dua, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
      if (status) CUDA_TRY(cudaMemcpyAsync(status + lo, dout + La.status, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    } else {
      const size_t out_n = X ? La.out_total : La.X;
      CUDA_TRY(cudaMemcpyAsync(hout, dout, out_n, cudaMemcpyDeviceToHost, s));
    }
  }
  for (int ci = 0; ci < nchunk; ++ci) {
    const int lo = ci * C, n = (lo + C <= B ? C : B - lo);
    if (n <= 0) break;
    CUDA_TRY(cudaStreamSynchronize(st.streams[ci]));
    if (out_pinned) continue;
    const char* hout = st.h_out + (size_t)ci * st.out_bytes;
    std::memcpy(U + (size_t)lo * nu, hout + La.U, (size_t)n * nu * 4);
    if (X) std::memcpy(X + (size_t)lo * nx, hout + La.X, (size_t)n * nx * 4);
    if (iters) std::memcpy(iters + lo, hout + La.iters, (size_t)n * 4);
    if (pri_res) std::memcpy(pri_res + lo, hout + La.pri, (size_t)n * 4);
    if (dua_res) std::memcpy(dua_res + lo, hout + La.dua, (size_t)n * 4);
    if (status) std::memcpy(status + lo, hout + La.status, (size_t)n * 4);
  }
  return CMPC_OK;
}


int cmpc_solve_host_async(cmpc_handle* h, int32_t B, int32_t slot0, const float* x0, const float* r,
                          const uint8_t* mask, const float* x_des, const float* mu, float* U, float* X,
                          int32_t* iters, float* pri_res, float* dua_res, int32_t* status, int32_t* ticket) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!ticket) return fail(CMPC_ERR_INVALID, "null ticket pointer");
  if (!x0 || !r || !mask || !x_des || !mu || !U) return fail(CMPC_ERR_INVALID, "null input/output pointer");
  if (!h->cfg.host_zero_copy) return fail(CMPC_ERR_UNSUPPORTED, "cmpc_solve_host_async needs cfg.host_zero_copy");
  DEVICE_GUARD(h);
  Staging& st = h->st;
  for (auto& s : st.streams)
    if (!s) CUDA_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  const int32_t t = st.next_ticket;
  static const bool engine_copies = std::getenv("CMPC_ASYNC_ZERO_COPY") == nullptr;   // experiment switch
  if (B > 0 && engine_copies) {
    // Inputs go through the copy engines into one of two device arenas while the previous submission is being
    // solved (SM-issued reads of host memory top out at ~16 GB/s, the engines move the same 4.6 MB at ~50 GB/s,
    // and a solve on device-resident inputs is 0.1 ms shorter); the results are still written in place.
    void *dU, *dX, *dit, *dpr, *ddu, *dst;
    const bool ok = is_pinned(x0) && is_pinned(r) && is_pinned(mask) && is_pinned(x_des) && is_pinned(mu) &&
                    is_pinned(U, &dU) && is_pinned(X, &dX) && is_pinned(iters, &dit) && is_pinned(pri_res, &dpr) &&
                    is_pinned(dua_res, &ddu) && is_pinned(status, &dst);
    if (!ok || !dU) return fail(CMPC_ERR_UNSUPPORTED, "cmpc_solve_host_async needs page-locked buffers (use cmpc_solve_host)");
    const int N = h->cfg.N;
    const Layout L = make_layout(N, h->cfg.max_batch, false);
    if (!st.d_async_in[0]) {
      for (int a = 0; a < 2; ++a) {
        CUDA_TRY(cudaMalloc(&st.d_async_in[a], L.in_total));
        CUDA_TRY(cudaEventCreateWithFlags(&st.h2d[a], cudaEventDisableTiming));
      }
      st.async_in_bytes = L.in_total;
    }
    const int a = t & 1;
    char* din = st.d_async_in[a];
    cudaStream_t cs = st.streams[1], ks = st.streams[0];
    // two copy streams (two copy engines): x_des on one, the rest on the other
    static const bool two_engines = std::getenv("CMPC_ASYNC_ONE_COPY_STREAM") == nullptr;   // experiment switch
    if (!st.copy2) {
      CUDA_TRY(cudaStreamCreateWithFlags(&st.copy2, cudaStreamNonBlocking));
      for (auto& e : st.h2d2) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    cudaStream_t cs2 = two_engines ? st.copy2 : cs;
    if (t >= 2) {   // the solve that read this arena last
      CUDA_TRY(cudaStreamWaitEvent(cs, st.done[(t - 2) & 7], 0));
      if (two_engines) CUDA_TRY(cudaStreamWaitEvent(cs2, st.done[(t - 2) & 7], 0));
    }
    CUDA_TRY(cudaMemcpyAsync(din + L.xdes, x_des, (size_t)B * 13 * (N + 1) * 4, cudaMemcpyHostToDevice, cs2));
    CUDA_TRY(cudaMemcpyAsync(din + L.r, r, (size_t)B * 12 * N * 4, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpyAsync(din + L.x0, x0, (size_t)B * 13 * 4, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpyAsync(din + L.mu, mu, (size_t)B * 4, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpyAsync(din + L.mask, mask, (size_t)B * N, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaEventRecord(st.h2d[a], cs));
    CUDA_TRY(cudaStreamWaitEvent(ks, st.h2d[a], 0));
    if (two_engines) {
      CUDA_TRY(cudaEventRecord(st.h2d2[a], cs2));
      CUDA_TRY(cudaStreamWaitEvent(ks, st.h2d2[a], 0));
    }
    // Results: into a device arena, then back with the copy engines on their own stream while the next submission
    // is solved (CMPC_ASYNC_INPLACE_RESULTS=1: written in place into the page-locked buffers by the kernel instead;
    // on part of the boxes of this pool that costs 0.04 ms per step)
    static const bool engine_results = std::getenv("CMPC_ASYNC_INPLACE_RESULTS") == nullptr;
    if (!engine_results) {
      rc = solve_device(h, B, slot0, (const float*)(din + L.x0), (const float*)(din + L.r), (const uint8_t*)(din + L.mask),
                        (const float*)(din + L.xdes), (const float*)(din + L.mu), (float*)dU, (float*)dX, (int32_t*)dit,
                        (float*)dpr, (float*)ddu, (int32_t*)dst, ks, false);
      if (rc) return rc;
    } else {
      const Layout Lo = make_layout(N, h->cfg.max_batch, true);
      if (!st.d2h) {
        CUDA_TRY(cudaStreamCreateWithFlags(&st.d2h, cudaStreamNonBlocking));
        for (int q = 0; q < 2; ++q) {
          CUDA_TRY(cudaMalloc(&st.d_async_out[q], Lo.out_total));
          CUDA_TRY(cudaEventCreateWithFlags(&st.solved[q], cudaEventDisableTiming));
        }
      }
      char* dout = st.d_async_out[a];
      rc = flush_results(h);        // the previous submission's result copies: behind this one's input copies
      if (rc) return rc;
      if (t >= 2) CUDA_TRY(cudaStreamWaitEvent(ks, st.done[(t - 2) & 7], 0));   // its results have left this arena
      rc = solve_device(h, B, slot0, (const float*)(din + L.x0), (const float*)(din + L.r), (const uint8_t*)(din + L.mask),
                        (const float*)(din + L.xdes), (const float*)(din + L.mu), (float*)(dout + Lo.U),
                        X ? (float*)(dout + Lo.X) : nullptr, iters ? (int32_t*)(dout + Lo.iters) : nullptr,
                        pri_res ? (float*)(dout + Lo.pri) : nullptr, dua_res ? (float*)(dout + Lo.dua) : nullptr,
                        status ? (int32_t*)(dout + Lo.status) : nullptr, ks, false);
      if (rc) return rc;
      CUDA_TRY(cudaEventRecord(st.solved[a], ks));
      cudaEvent_t& evd = st.done[t & 7];
      if (!evd) CUDA_TRY(cudaEventCreateWithFlags(&evd, cudaEventDisableTiming));
      Staging::Pending& q = st.pending;
      q.active = true; q.ticket = t; q.B = B; q.arena = a;
      q.U = U; q.X = X; q.iters = iters; q.pri = pri_res; q.dua = dua_res; q.status = status;
      st.next_ticket++;
      *ticket = t;
      return CMPC_OK;
    }
  } else if (B > 0) {
    rc = enqueue_zero_copy(h, B, slot0, x0, r, mask, x_des, mu, U, X, iters, pri_res, dua_res, status);
    if (rc < 0) return rc;
    if (rc == 0) return fail(CMPC_ERR_UNSUPPORTED, "cmpc_solve_host_async needs page-locked buffers (use cmpc_solve_host)");
  }
  rc = flush_results(h);      // tickets complete in submission order
  if (rc) return rc;
  st.next_ticket++;
  cudaEvent_t& ev = st.done[t & 7];
  if (!ev) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  CUDA_TRY(cudaEventRecord(ev, (B == 0 && st.d2h) ? st.d2h : st.streams[0]));   // tickets complete in submission order
  *ticket = t;
  return CMPC_OK;
}

int cmpc_host_wait(cmpc_handle* h, int32_t ticket) {
  if (!h) return fail(CMPC_ERR_INVALID, "null handle");
  Staging& st = h->st;
  if (ticket < 0 || ticket >= st.next_ticket) return fail(CMPC_ERR_INVALID, "unknown ticket %d", ticket);
  DEVICE_GUARD(h);
  if (st.pending.active && st.pending.ticket <= ticket) {
    const int rc = flush_results(h);
    if (rc) return rc;
  }
  if (st.next_ticket - ticket > 8) {     // its event was reused: submissions complete in order, wait for the oldest kept
    CUDA_TRY(cudaEventSynchronize(st.done[st.next_ticket & 7]));
    return CMPC_OK;
  }
  CUDA_TRY(cudaEventSynchronize(st.done[ticket & 7]));
  return CMPC_OK;
}

int cmpc_reset_warm_async(cmpc_handle* h, int32_t B, int32_t slot0, const uint8_t* slot_mask, void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (B == 0) return CMPC_OK;
  DEVICE_GUARD(h);
  cmpc::reset_warm_kernel<<<(B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      h->d_warm_valid, h->d_cache_meta, slot_mask, slot0, B);
  CUDA_TRY(cudaGetLastError());
  h->launches.fetch_add(1);
  return CMPC_OK;
}

int cmpc_reset_warm(cmpc_handle* h, const uint8_t* slot_mask) {
  if (!h) return fail(CMPC_ERR_INVALID, "null handle");
  DEVICE_GUARD(h);
  // host-synchronous form: ordered against EVERY stream of the device (solves may be in flight on
  // non-blocking streams, which the legacy default stream does not wait for)
  CUDA_TRY(cudaDeviceSynchronize());
  const int slots = h->cfg.max_batch;
  uint8_t* d_mask = nullptr;
  if (slot_mask) {
    CUDA_TRY(cudaMalloc(&d_mask, (size_t)slots));
    cudaError_t e = cudaMemcpy(d_mask, slot_mask, (size_t)slots, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      cudaFree(d_mask);
      return fail(CMPC_ERR_CUDA, "cudaMemcpy of the slot mask failed: %s", cudaGetErrorString(e));
    }
  }
  cmpc::reset_warm_kernel<<<(slots + 255) / 256, 256>>>(h->d_warm_valid, h->d_cache_meta, d_mask, 0, slots);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  cudaFree(d_mask);
  if (e != cudaSuccess) return fail(CMPC_ERR_CUDA, "reset_warm failed: %s", cudaGetErrorString(e));
  h->launches.fetch_add(1);
  return CMPC_OK;
}

// the handle keeps warm x / y in the kernel horizon's layout [slots][NK][12]; callers use [B][N][12]
int cmpc_get_warm(cmpc_handle* h, int32_t B, int32_t slot0, float* x, float* y, void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!x) return fail(CMPC_ERR_INVALID, "null pointer");
  if (B == 0) return CMPC_OK;
  DEVICE_GUARD(h);
  const size_t wu = (size_t)h->cfg.N * 12 * 4, wk = (size_t)h->NK * 12 * 4;
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaMemcpy2DAsync(x, wu, h->d_warm_x + (size_t)slot0 * 12 * h->NK, wk, wu, (size_t)B,
                             cudaMemcpyDeviceToDevice, s));
  if (y)
    CUDA_TRY(cudaMemcpy2DAsync(y, wu, h->d_warm_y + (size_t)slot0 * 12 * h->NK, wk, wu, (size_t)B,
                               cudaMemcpyDeviceToDevice, s));
  return CMPC_OK;
}

int cmpc_set_warm(cmpc_handle* h, int32_t B, int32_t slot0, const float* x, const float* y,
                  void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!x) return fail(CMPC_ERR_INVALID, "null pointer");
  if (B == 0) return CMPC_OK;
  DEVICE_GUARD(h);
  const size_t wu = (size_t)h->cfg.N * 12 * 4, wk = (size_t)h->NK * 12 * 4;
  cudaStream_t s = (cudaStream_t)stream;
  float* wx = h->d_warm_x + (size_t)slot0 * 12 * h->NK;
  float* wy = h->d_warm_y + (size_t)slot0 * 12 * h->NK;
  if (wk != wu) CUDA_TRY(cudaMemsetAsync(wx, 0, wk * B, s));      // padded stages carry no force
  CUDA_TRY(cudaMemcpy2DAsync(wx, wk, x, wu, wu, (size_t)B, cudaMemcpyDeviceToDevice, s));
  CUDA_TRY(cudaMemsetAsync(wy, 0, wk * B, s));
  if (y) CUDA_TRY(cudaMemcpy2DAsync(wy, wk, y, wu, wu, (size_t)B, cudaMemcpyDeviceToDevice, s));
  CUDA_TRY(cudaMemsetAsync(h->d_warm_valid + slot0, 1, (size_t)B, s));
  return CMPC_OK;
}

}  // extern "C"
