// cmpc.cu - C ABI (include/cmpc.h) over the sm_100a kernels in cmpc_kernels.cuh.
// No torch types, no CPU fallback: every entry point fails with CMPC_ERR_NO_DEVICE /
// CMPC_ERR_CUDA when the CUDA device or the kernels are unavailable.
#include "../../include/cmpc.h"
#include "cmpc_kernels.cuh"
#include "cmpc_launch.cuh"
#include "cmpc_riccati.cuh"

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
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

// per-slot data a handle has received; kBody, kContact, kWeights, kForce and kStage select the solve kernels compiled
// with that flag (kForce is always set with kWeights, kStage with kForce), a wrench adds a pass before and after the
// solve (cmpc_wrench.cu)
enum Feature : unsigned { kBody = 1, kContact = 2, kWeights = 4, kWrench = 8, kForce = 16, kStage = 32 };
constexpr unsigned kSolveFeatures = kBody | kContact | kWeights | kForce | kStage;

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
  float4* d_body = nullptr;         // [slots][kBodyF4] per-slot rigid body, filled with cfg's body at create
  float4* d_contact = nullptr;      // [slots][NK][4][kContactF4] per-leg-stage contact, allocated by the first
                                    // cmpc_set_contact
  float4* d_weights = nullptr;      // [slots][kWeightF4] per-slot cost weights, allocated by the first cmpc_set_weights
  float* d_w_Minv = nullptr;        // [slots][6][NK][NK] their M^-1 and M (NK <= kWeightTableMaxN only)
  float* d_w_Mg = nullptr;
  float* d_wrench = nullptr;        // [slots][N][6] per-stage external force and torque, allocated by the first
                                    // cmpc_set_wrench
  float* d_wrench_xdes = nullptr;   // [slots][13 (N + 1)] their shifted x_des (NK == N; padded horizons shift
                                    // d_pad_xdes in place)
  float4* d_force = nullptr;        // [slots][NK][4] per-leg-stage force reference {f_ref, w_f}, allocated by the
                                    // first cmpc_set_force_ref
  float4* d_wstage = nullptr;       // [slots][NK][kStageF4] per-stage state weights w[0..11], allocated by the first
                                    // cmpc_set_stage_weights
  std::atomic<unsigned> features{0};   // kBody | kContact | kWeights | kWrench | kForce | kStage, set by the first
                                       // cmpc_set_body / _contact / _weights / _wrench / _force_ref / _stage_weights:
                                       // launch the kernels of that feature set (handle_features)
  std::mutex feature_alloc;            // the first cmpc_set_contact / _weights / _wrench / _force_ref /
                                       // _stage_weights (init_feature)
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

namespace cmpc {
template const SolveRow* solve_rows<false, false, false>();   // the plain solve kernels
}  // namespace cmpc

namespace {

using cmpc::SolveLaunch;
using cmpc::launch_pdl;
using CondenseLaunch = cudaError_t (*)(const cmpc::CondenseParams&, cudaStream_t);
using ScoreLaunch = cudaError_t (*)(const cmpc::ScoreParams&, cudaStream_t);

template <int N>
cudaError_t launch_score(const cmpc::ScoreParams& p, cudaStream_t s) {
  return launch_pdl(cmpc::score_kernel<N>, dim3((unsigned)((p.B + 127) / 128)), dim3(128), 0, s, p);
}
template <int N>
cudaError_t launch_condense(const cmpc::CondenseParams& p, cudaStream_t s) {
  cmpc::condense_kernel<N><<<p.B, 256, 0, s>>>(p);
  return cudaGetLastError();
}

struct HorizonEntry {
  int N;
  CondenseLaunch condense;  // or nullptr
  ScoreLaunch score;
};

// Horizons with compiled kernels; their solve launchers are row i of solve_rows (cmpc_launch.cuh, one instantiation
// per feature set, see solve_row).  Any other horizon N <= 60 runs padded on the next compiled one (pad_kernel).
const HorizonEntry kHorizons[] = {
    {4, launch_condense<4>, launch_score<4>},
    {5, launch_condense<5>, launch_score<5>},
    {8, launch_condense<8>, launch_score<8>},
    {10, launch_condense<10>, launch_score<10>},
    {12, launch_condense<12>, launch_score<12>},
    {16, launch_condense<16>, launch_score<16>},
    {20, launch_condense<20>, launch_score<20>},
    {30, launch_condense<30>, launch_score<30>},
    {40, nullptr, launch_score<40>},
    {60, nullptr, launch_score<60>},
};
static_assert(sizeof kHorizons / sizeof kHorizons[0] == cmpc::kNumHorizons, "one row of solve_rows per horizon");
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

// the per-slot data a handle has received (Feature bits)
unsigned handle_features(const cmpc_handle* h) { return h->features.load(); }

// The solve launchers of compiled horizon e for a handle with features f.  The CONTACT and WEIGHTS kernels are
// compiled with BODY only, the FORCE kernels with BODY + WEIGHTS only, the STAGE kernels with BODY + WEIGHTS + FORCE
// only (see fill_solve_params).  Every feature set has a row for every horizon; kWrench selects none.
const cmpc::SolveRow& solve_row(const HorizonEntry* e, unsigned f) {
  using Rows = const cmpc::SolveRow* (*)();
  static constexpr Rows kRows[8] = {   // index: f without kForce
      cmpc::solve_rows<false, false, false>, cmpc::solve_rows<true, false, false>,
      cmpc::solve_rows<true, true, false>,   cmpc::solve_rows<true, true, false>,
      cmpc::solve_rows<true, false, true>,   cmpc::solve_rows<true, false, true>,
      cmpc::solve_rows<true, true, true>,    cmpc::solve_rows<true, true, true>,
  };
  static constexpr Rows kForceRows[2] = {   // index: f has kContact
      cmpc::solve_rows<true, false, true, true>, cmpc::solve_rows<true, true, true, true>,
  };
  static constexpr Rows kStageRows[2] = {   // index: f has kContact
      cmpc::solve_rows<true, false, true, true, true>, cmpc::solve_rows<true, true, true, true, true>,
  };
  const Rows rows = f & kStage   ? kStageRows[(f & kContact) ? 1 : 0]
                    : f & kForce ? kForceRows[(f & kContact) ? 1 : 0]
                                 : kRows[f & (kBody | kContact | kWeights)];
  return rows()[e - kHorizons];
}

SolveLaunch pick_solve(const cmpc_handle* h, unsigned f) {
  const cmpc_config& c = h->cfg;
  const cmpc::SolveRow& row = solve_row(find_horizon(h->NK), f);
  if (c.cache_factorization && row.cached) return row.cached;
  if (c.kernel_variant == 5 && row.other) return row.other;
  return row.solve;
}

// the parameters of the kernels of feature set f (handle_features, read once per solve, so that these and
// pick_solve's kernel agree while another thread publishes a feature)
void fill_solve_params(const cmpc_handle* h, unsigned f, cmpc::SolveParams& p) {
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
  p.cache_pinv = h->d_cache_pinv;      // nullptr unless cfg.cache_factorization
  p.cache_r = h->d_cache_r;
  p.cache_mask = h->d_cache_mask;
  p.cache_meta = h->d_cache_meta;
  p.cache_tol_r = c.cache_tol_r;
  p.cache_tol_yaw = c.cache_tol_yaw;
  p.cache_max_iter = c.cache_max_iter;
  p.cache_hit = h->d_cache_hit;
  p.n_eff = c.N;                       // < NK on a padded horizon
  // the CONTACT and WEIGHTS kernels exist with BODY only: a handle with contacts or weights and no body runs them on
  // the configuration's body, which every slot of d_body holds until cmpc_set_body (bit-identical to the plain
  // kernels' body); kForce comes with kWeights (cmpc_set_force_ref), kStage with both (cmpc_set_stage_weights)
  const bool weights = f & kWeights;
  p.contact = f & kContact ? h->d_contact : nullptr;
  if (f & kForce) p.force = h->d_force;   // in place of Minv, which the FORCE kernels do not read
  if (f & kStage) p.wstage = h->d_wstage;   // in place of Mg, which the STAGE kernels do not read
  p.weights = weights ? h->d_weights : nullptr;
  p.w_Minv = weights ? h->d_w_Minv : nullptr;
  p.w_Mg = weights ? h->d_w_Mg : nullptr;
  p.body = f & kSolveFeatures ? h->d_body : nullptr;
}

// Enqueue the LPT ordering of a batch (2 small kernels) and point p.order at it.  The scratch
// (score, order, histogram) is carved out by the batch's slot range, so that disjoint slot ranges
// of one handle may be solved concurrently on different streams: order/score live at
// [slot0, slot0 + B), the histogram at slot0 / lpt_schedule (two disjoint ranges of >= lpt_schedule
// slots each cannot share that quotient).
int schedule_batch(cmpc_handle* h, unsigned f, cmpc::SolveParams& p, cudaStream_t s) {
  p.order = nullptr;
  p.sched = nullptr;
  if (!h->cfg.lpt_schedule || p.B < h->cfg.lpt_schedule) return CMPC_OK;
  if ((reinterpret_cast<uintptr_t>(p.r) & 15u) != 0) return CMPC_OK;   // score_kernel reads r with 16-byte loads
  const cmpc_config& c = h->cfg;
  const int hist_slot = p.slot0 / c.lpt_schedule;
  if (hist_slot >= h->hist_slots) return CMPC_OK;
  cmpc::ScoreParams sp{};
  sp.x0 = p.x0; sp.r = p.r; sp.mask = p.mask; sp.Mg = h->d_Mg; sp.mu = p.mu;
  sp.score = h->d_score + p.slot0;
  sp.hist = h->d_hist + 64 * hist_slot;
  sp.B = p.B;
  sp.inv_mass = 1.0f / c.mass;
  for (int i = 0; i < 3; ++i) sp.ib[i] = c.ibody_inv[i];
  sp.body = p.body ? p.body + (size_t)cmpc::kBodyF4 * p.slot0 : nullptr;
  sp.weights = p.weights ? p.weights + (size_t)cmpc::kWeightF4 * p.slot0 : nullptr;
  sp.wstage = f & kStage ? h->d_wstage + (size_t)cmpc::kStageF4 * h->NK * p.slot0 : nullptr;
  sp.dt = c.dt;
  sp.n_eff = c.N;
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

// pad -> wrench shift -> schedule -> solve -> unpad -> wrench finish of one batch on one stream; all pointers are
// device-visible (device memory, or page-locked host memory mapped into the device's address space)
int solve_device(cmpc_handle* h, int B, int slot0, const float* x0, const float* r, const uint8_t* mask,
                 const float* x_des, const float* mu, float* U, float* X, int32_t* iters, float* pri_res,
                 float* dua_res, int32_t* status, cudaStream_t s, bool timed, bool plain_launch = false) {
  const int N = h->cfg.N, NK = h->NK;
  const unsigned f = handle_features(h);
  cmpc::SolveParams p{};
  fill_solve_params(h, f, p);
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
  // a known external wrench: the same QP on x_des - phi (wrench_shift_kernel), X + phi afterwards
  cmpc::WrenchParams wp{};
  if (f & kWrench) {
    wp.x0 = x0; wp.x_des = p.x_des; wp.X = X; wp.status = status;
    wp.x_des_out = NK == N ? h->d_wrench_xdes + (size_t)slot0 * 13 * (N + 1) : const_cast<float*>(p.x_des);
    wp.wrench = h->d_wrench + (size_t)slot0 * 6 * N;
    wp.body = h->d_body + (size_t)cmpc::kBodyF4 * slot0;
    wp.B = B; wp.N = N; wp.NK = NK; wp.dt = h->cfg.dt;
    CUDA_TRY(cmpc::wrench_shift(wp, s));
    h->launches.fetch_add(1);
    p.x_des = wp.x_des_out;
  }
  int rc = schedule_batch(h, f, p, s);
  if (rc) return rc;
  if (plain_launch) p.sched = nullptr;   // chunked host path: the launch shares the device with its sibling chunk
  if (timed) {
    if (!h->ev0) { CUDA_TRY(cudaEventCreate(&h->ev0)); CUDA_TRY(cudaEventCreate(&h->ev1)); }
    CUDA_TRY(cudaEventRecord(h->ev0, s));
  }
  CUDA_TRY(pick_solve(h, f)(p, h->cfg.device, s));
  if (timed) {
    CUDA_TRY(cudaEventRecord(h->ev1, s));
    h->timed = true;
  }
  h->launches.fetch_add(1);
  if (NK != N) {
    cmpc::UnpadParams up{};
    up.U_k = p.U; up.X_k = p.X; up.U = U; up.X = X; up.B = B; up.N = N; up.NK = NK;
    const long long items = (long long)B * (12 * N + (X ? 13 * (N + 1) : 0));
    cmpc::unpad_kernel<<<(unsigned)((items + 255) / 256), 256, 0, s>>>(up);
    CUDA_TRY(cudaGetLastError());
    h->launches.fetch_add(1);
  }
  if ((f & kWrench) && (X || status)) {
    CUDA_TRY(cmpc::wrench_finish(wp, s));
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

// A device array of a feature, allocated by the feature's first call.
struct FeatureArray {
  void** ptr;     // the handle's pointer
  size_t bytes;   // 0: not allocated
};

// The first call of the feature `bit` (cmpc_set_contact, cmpc_set_weights: `fn`) allocates its arrays and fills every
// slot with the "never set" state (`init` enqueues one kernel on s) before any solve, on any stream, can read them:
// host-synchronous, so refused inside a graph capture.  The arrays are freed on failure.  The caller publishes the
// bit once it has enqueued its store kernel.
template <typename Init>
int init_feature(cmpc_handle* h, unsigned bit, const char* fn, cudaStream_t s,
                 std::initializer_list<FeatureArray> arrays, Init init) {
  if (handle_features(h) & bit) return CMPC_OK;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  CUDA_TRY(cudaStreamIsCapturing(s, &cap));
  if (cap != cudaStreamCaptureStatusNone)
    return fail(CMPC_ERR_INVALID, "the first %s of a handle allocates: call it once outside a graph capture", fn);
  std::lock_guard<std::mutex> lock(h->feature_alloc);
  if (*arrays.begin()->ptr) return CMPC_OK;   // allocated by a concurrent or an earlier first call
  cudaError_t e = cudaSuccess;
  for (const FeatureArray& a : arrays)
    if (e == cudaSuccess && a.bytes) e = cudaMalloc(a.ptr, a.bytes);
  if (e == cudaSuccess) e = init();
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) {
    for (const FeatureArray& a : arrays) {
      cudaFree(*a.ptr);
      *a.ptr = nullptr;
    }
    return fail(CMPC_ERR_CUDA, "%s: array initialisation failed: %s", fn, cudaGetErrorString(e));
  }
  h->launches.fetch_add(1);
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
  if (!e) return 0;
  return variant == 0 || (variant == 5 && solve_row(e, 0).other) ? 1 : 0;
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
  const bool stagewise = he && he->N >= 20;          // default kernel = Riccati (see kHorizons)
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
  {
    // every slot starts with the configuration's body, so slots never given one solve as before
    const float bd[4 * cmpc::kBodyF4] = {1.0f / c.mass, c.ibody_inv[0], 0.f, 0.f, 0.f, c.ibody_inv[1], 0.f, 0.f, 0.f,
                                         c.ibody_inv[2], 0.f, 0.f};
    std::vector<float> fill(slots * 4 * cmpc::kBodyF4);
    for (size_t i = 0; i < slots; ++i) std::memcpy(fill.data() + i * 4 * cmpc::kBodyF4, bd, sizeof bd);
    if ((e = cudaMalloc(&h->d_body, fill.size() * sizeof(float))) != cudaSuccess ||
        (e = cudaMemcpy(h->d_body, fill.data(), fill.size() * sizeof(float), cudaMemcpyHostToDevice)) != cudaSuccess) {
      cmpc_destroy(h);
      return fail(CMPC_ERR_CUDA, "body array allocation failed: %s", cudaGetErrorString(e));
    }
  }
  if (c.cache_factorization && !solve_row(he, 0).cached) {
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
  // the host path may still have work in flight: the result copies owed to the last asynchronous submission
  // are enqueued and every host-path stream is drained before any stream or buffer goes away
  if (h->st.pending.active) flush_results(h);
  for (cudaStream_t s : {h->st.streams[0], h->st.streams[1], h->st.copy2, h->st.d2h})
    if (s) cudaStreamSynchronize(s);
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
  cudaFree(h->d_body);
  cudaFree(h->d_contact);
  cudaFree(h->d_weights);
  cudaFree(h->d_w_Minv);
  cudaFree(h->d_w_Mg);
  cudaFree(h->d_wrench);
  cudaFree(h->d_wrench_xdes);
  cudaFree(h->d_force);
  cudaFree(h->d_wstage);
  if (h->st.h_in) cudaFreeHost(h->st.h_in);
  if (h->st.h_out) cudaFreeHost(h->st.h_out);
  cudaFree(h->st.d_in);
  cudaFree(h->st.d_out);
  for (auto& s : h->st.streams)
    if (s) cudaStreamDestroy(s);
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

int cmpc_set_body(cmpc_handle* h, int32_t B, int32_t slot0, const float* mass, const float* ibody_inv,
                  void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!mass || !ibody_inv) return fail(CMPC_ERR_INVALID, "null pointer");
  if (B == 0) return CMPC_OK;
  DEVICE_GUARD(h);
  cmpc::set_body_kernel<<<(B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(mass, ibody_inv, h->d_body,
                                                                           h->d_cache_meta, slot0, B);
  CUDA_TRY(cudaGetLastError());
  h->launches.fetch_add(1);
  h->features.fetch_or(kBody);
  return CMPC_OK;
}

int cmpc_set_contact(cmpc_handle* h, int32_t B, int32_t slot0, const float* normal, const float* mu,
                     const float* f_min, const float* f_max, void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!normal || !mu || !f_min || !f_max) return fail(CMPC_ERR_INVALID, "null pointer");
  if (B == 0) return CMPC_OK;
  DEVICE_GUARD(h);
  const cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)h->cfg.max_batch * h->NK * 4;   // leg-stages
  rc = init_feature(h, kContact, "cmpc_set_contact", s,
                    {{(void**)&h->d_contact, n * cmpc::kContactF4 * sizeof(float4)}},
                    [&] { return cmpc::init_contact(h->d_contact, h->cfg.f_min, h->cfg.f_max, n, s); });
  if (rc) return rc;
  CUDA_TRY(cmpc::store_contact(normal, mu, f_min, f_max, h->d_contact, slot0, B, h->cfg.N, h->NK, s));
  h->launches.fetch_add(1);
  h->features.fetch_or(kContact);
  return CMPC_OK;
}

namespace {
// The first cmpc_set_weights or cmpc_set_force_ref (`fn`) of a handle: allocate the weight storage and give every slot
// the handle's weight record and Gram tables (init_feature).
int init_weight_storage(cmpc_handle* h, const char* fn, cudaStream_t s) {
  const cmpc_config& c = h->cfg;
  const size_t slots = (size_t)c.max_batch;
  // the Gram tables exist for the kernel horizons that read them
  const size_t tbytes = h->NK <= cmpc::kWeightTableMaxN ? slots * 6 * h->NK * h->NK * sizeof(float) : 0;
  return init_feature(h, kWeights, fn, s,
                      {{(void**)&h->d_weights, slots * cmpc::kWeightF4 * sizeof(float4)},
                       {(void**)&h->d_w_Minv, tbytes},
                       {(void**)&h->d_w_Mg, tbytes}},
                      [&] {
                        // every slot gets the handle's record and Gram tables
                        float rec[4 * cmpc::kWeightF4] = {};
                        for (int i = 0; i < 13; ++i) rec[i] = c.w[i];
                        rec[13] = c.r_weight;
                        return cmpc::init_weights(h->d_weights, h->d_w_Minv, h->d_w_Mg, rec, h->d_Minv, h->d_Mg,
                                                  c.max_batch, h->NK, s);
                      });
}
}  // namespace

int cmpc_set_weights(cmpc_handle* h, int32_t B, int32_t slot0, const float* w, const float* r_weight, void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!w || !r_weight) return fail(CMPC_ERR_INVALID, "null pointer");
  if (B == 0) return CMPC_OK;
  DEVICE_GUARD(h);
  const cudaStream_t s = (cudaStream_t)stream;
  const cmpc_config& c = h->cfg;
  rc = init_weight_storage(h, "cmpc_set_weights", s);
  if (rc) return rc;
  // a handle with stage weights: w goes to every stage of the slots' tables too
  float4* wstage = handle_features(h) & kStage ? h->d_wstage : nullptr;
  CUDA_TRY(cmpc::store_weights(w, 0, r_weight, h->d_weights, wstage, h->d_w_Minv, h->d_w_Mg, h->d_cache_meta, slot0, B,
                               c.N, h->NK, c.dt, c.device, s));
  h->launches.fetch_add(1);
  h->features.fetch_or(kWeights);
  return CMPC_OK;
}

int cmpc_set_wrench(cmpc_handle* h, int32_t B, int32_t slot0, const float* force, const float* torque, void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!force || !torque) return fail(CMPC_ERR_INVALID, "null pointer");
  if (B == 0) return CMPC_OK;
  DEVICE_GUARD(h);
  const cudaStream_t s = (cudaStream_t)stream;
  const cmpc_config& c = h->cfg;
  const size_t slots = (size_t)c.max_batch, bytes = slots * 6 * c.N * sizeof(float);
  // a padded horizon shifts its own NK-layout copy of x_des (d_pad_xdes) in place
  const size_t xbytes = h->NK == c.N ? slots * 13 * (c.N + 1) * sizeof(float) : 0;
  rc = init_feature(h, kWrench, "cmpc_set_wrench", s,
                    {{(void**)&h->d_wrench, bytes}, {(void**)&h->d_wrench_xdes, xbytes}},
                    [&] { return cudaMemsetAsync(h->d_wrench, 0, bytes, s); });   // every slot: zero wrench
  if (rc) return rc;
  CUDA_TRY(cmpc::store_wrench(force, torque, h->d_wrench, slot0, B, c.N, s));
  h->launches.fetch_add(1);
  h->features.fetch_or(kWrench);
  return CMPC_OK;
}

int cmpc_set_force_ref(cmpc_handle* h, int32_t B, int32_t slot0, const float* f_ref, const float* weight,
                       void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!f_ref || !weight) return fail(CMPC_ERR_INVALID, "null pointer");
  if (B == 0) return CMPC_OK;
  DEVICE_GUARD(h);
  const cudaStream_t s = (cudaStream_t)stream;
  const cmpc_config& c = h->cfg;
  // the FORCE kernels are compiled with WEIGHTS: a handle without weights gets the configuration's in every slot,
  // which give the answers of the configuration's weights bit for bit
  rc = init_weight_storage(h, "cmpc_set_force_ref", s);
  if (rc) return rc;
  const size_t bytes = (size_t)c.max_batch * h->NK * 4 * sizeof(float4);
  rc = init_feature(h, kForce, "cmpc_set_force_ref", s, {{(void**)&h->d_force, bytes}},
                    [&] { return cudaMemsetAsync(h->d_force, 0, bytes, s); });   // every slot: zero weight
  if (rc) return rc;
  CUDA_TRY(cmpc::store_force_ref(f_ref, weight, h->d_force, h->d_cache_meta, slot0, B, c.N, h->NK, s));
  h->launches.fetch_add(1);
  h->features.fetch_or(kWeights | kForce);
  return CMPC_OK;
}

int cmpc_set_stage_weights(cmpc_handle* h, int32_t B, int32_t slot0, const float* w, const float* r_weight,
                           void* stream) {
  int rc = check_batch(h, B, slot0);
  if (rc) return rc;
  if (!w || !r_weight) return fail(CMPC_ERR_INVALID, "null pointer");
  if (B == 0) return CMPC_OK;
  DEVICE_GUARD(h);
  const cudaStream_t s = (cudaStream_t)stream;
  const cmpc_config& c = h->cfg;
  // the STAGE kernels are compiled with WEIGHTS + FORCE: a handle without weights gets the configuration's in every
  // slot, one without force references zero weight in every slot (both give the answers of no such call bit for bit)
  rc = init_weight_storage(h, "cmpc_set_stage_weights", s);
  if (rc) return rc;
  const size_t fbytes = (size_t)c.max_batch * h->NK * 4 * sizeof(float4);
  rc = init_feature(h, kForce, "cmpc_set_stage_weights", s, {{(void**)&h->d_force, fbytes}},
                    [&] { return cudaMemsetAsync(h->d_force, 0, fbytes, s); });
  if (rc) return rc;
  // every slot's stages start from its weight record (the configuration's, or those of an earlier cmpc_set_weights)
  const size_t bytes = (size_t)c.max_batch * h->NK * cmpc::kStageF4 * sizeof(float4);
  rc = init_feature(h, kStage, "cmpc_set_stage_weights", s, {{(void**)&h->d_wstage, bytes}},
                    [&] { return cmpc::init_stage_weights(h->d_wstage, h->d_weights, c.max_batch, c.N, h->NK, s); });
  if (rc) return rc;
  CUDA_TRY(cmpc::store_weights(w, 13, r_weight, h->d_weights, h->d_wstage, h->d_w_Minv, h->d_w_Mg, h->d_cache_meta,
                               slot0, B, c.N, h->NK, c.dt, c.device, s));
  h->launches.fetch_add(1);
  h->features.fetch_or(kWeights | kForce | kStage);
  return CMPC_OK;
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
  const unsigned f = handle_features(h);
  p.body = f & kBody ? h->d_body : nullptr;   // slots [0, B)
  if (f & kWeights) {                         // slots [0, B); condense horizons have per-slot tables
    p.weights = h->d_weights;
    p.w_Mg = h->d_w_Mg;
  }
  p.wrench = f & kWrench ? h->d_wrench : nullptr;   // slots [0, B)
  p.force = f & kForce ? h->d_force : nullptr;      // slots [0, B)
  p.wstage = f & kStage ? h->d_wstage : nullptr;    // slots [0, B)
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
    const unsigned f = handle_features(h);
    p.body = f & kBody ? h->d_body : nullptr;       // slots [0, B)
    p.wrench = f & kWrench ? h->d_wrench : nullptr;   // stage 0 of slots [0, B)
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
  if (B == 0) {
    rc = flush_results(h);      // tickets complete in submission order
    if (rc) return rc;
    st.next_ticket++;
    cudaEvent_t& ev = st.done[t & 7];
    if (!ev) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(ev, st.d2h ? st.d2h : st.streams[0]));
    *ticket = t;
    return CMPC_OK;
  }
  // Inputs go through the copy engines into one of two device arenas while the previous submission is being
  // solved (SM-issued reads of host memory top out at ~16 GB/s, the engines move the same 4.6 MB at ~50 GB/s,
  // and a solve on device-resident inputs is 0.1 ms shorter).
  void* dU;
  const bool ok = is_pinned(x0) && is_pinned(r) && is_pinned(mask) && is_pinned(x_des) && is_pinned(mu) &&
                  is_pinned(U, &dU) && is_pinned(X) && is_pinned(iters) && is_pinned(pri_res) &&
                  is_pinned(dua_res) && is_pinned(status);
  if (!ok || !dU) return fail(CMPC_ERR_UNSUPPORTED, "cmpc_solve_host_async needs page-locked buffers (use cmpc_solve_host)");
  const int N = h->cfg.N;
  const Layout L = make_layout(N, h->cfg.max_batch, false);
  const Layout Lo = make_layout(N, h->cfg.max_batch, true);
  if (!st.d_async_in[0]) {
    for (int a = 0; a < 2; ++a) {
      CUDA_TRY(cudaMalloc(&st.d_async_in[a], L.in_total));
      CUDA_TRY(cudaEventCreateWithFlags(&st.h2d[a], cudaEventDisableTiming));
    }
    st.async_in_bytes = L.in_total;
  }
  if (!st.copy2) {
    CUDA_TRY(cudaStreamCreateWithFlags(&st.copy2, cudaStreamNonBlocking));
    for (auto& e : st.h2d2) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  if (!st.d2h) {
    CUDA_TRY(cudaStreamCreateWithFlags(&st.d2h, cudaStreamNonBlocking));
    for (int q = 0; q < 2; ++q) {
      CUDA_TRY(cudaMalloc(&st.d_async_out[q], Lo.out_total));
      CUDA_TRY(cudaEventCreateWithFlags(&st.solved[q], cudaEventDisableTiming));
    }
  }
  const int a = t & 1;
  char* din = st.d_async_in[a];
  char* dout = st.d_async_out[a];
  // two copy streams (two copy engines): x_des on one, the rest on the other
  cudaStream_t cs = st.streams[1], cs2 = st.copy2, ks = st.streams[0];
  if (t >= 2) {   // the solve that read this arena last
    CUDA_TRY(cudaStreamWaitEvent(cs, st.done[(t - 2) & 7], 0));
    CUDA_TRY(cudaStreamWaitEvent(cs2, st.done[(t - 2) & 7], 0));
  }
  CUDA_TRY(cudaMemcpyAsync(din + L.xdes, x_des, (size_t)B * 13 * (N + 1) * 4, cudaMemcpyHostToDevice, cs2));
  CUDA_TRY(cudaMemcpyAsync(din + L.r, r, (size_t)B * 12 * N * 4, cudaMemcpyHostToDevice, cs));
  CUDA_TRY(cudaMemcpyAsync(din + L.x0, x0, (size_t)B * 13 * 4, cudaMemcpyHostToDevice, cs));
  CUDA_TRY(cudaMemcpyAsync(din + L.mu, mu, (size_t)B * 4, cudaMemcpyHostToDevice, cs));
  CUDA_TRY(cudaMemcpyAsync(din + L.mask, mask, (size_t)B * N, cudaMemcpyHostToDevice, cs));
  CUDA_TRY(cudaEventRecord(st.h2d[a], cs));
  CUDA_TRY(cudaStreamWaitEvent(ks, st.h2d[a], 0));
  CUDA_TRY(cudaEventRecord(st.h2d2[a], cs2));
  CUDA_TRY(cudaStreamWaitEvent(ks, st.h2d2[a], 0));
  // Results: into a device arena, then back with the copy engines on their own stream while the next submission
  // is solved (measured against the kernel writing them in place into the page-locked buffers: that cost
  // 0.04 ms per step on part of the boxes)
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
