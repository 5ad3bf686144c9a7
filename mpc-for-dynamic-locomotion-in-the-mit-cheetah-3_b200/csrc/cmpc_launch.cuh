// cmpc_launch.cuh - host-side launchers of the solve kernels and the one list of them per compiled horizon
// (solve_rows), instantiated for each feature set by cmpc.cu (a handle that has never received a body, a contact or
// weights), cmpc_body.cu (BODY, see cmpc_set_body), cmpc_contact.cu (BODY + CONTACT, see cmpc_set_contact) and
// cmpc_weights.cu (BODY + WEIGHTS and BODY + CONTACT + WEIGHTS, see cmpc_set_weights), cmpc_force.cu (the same two
// with FORCE, see cmpc_set_force_ref) and cmpc_stage.cu (those with STAGE, see cmpc_set_stage_weights).  A wrench (cmpc_set_wrench) selects no solve kernel: cmpc_wrench.cu shifts x_des
// before the solve and corrects X after it.
#pragma once
#include "cmpc_kernels.cuh"
#include "cmpc_riccati.cuh"

#include <mutex>

namespace cmpc {

using SolveLaunch = cudaError_t (*)(const SolveParams&, int device, cudaStream_t);

// Programmatic dependent launch: the kernel may be scheduled while its predecessor in the stream is
// still running (its CTAs wait in griddepcontrol.wait before they touch global memory), which hides the
// launch latency between the two scheduling kernels and the solve kernel.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// One-time set-up of a kernel on one device.  Function attributes and occupancy are per device and one
// process may hold handles on several GPUs, so each launcher keeps one PerDevice table and runs its
// set-up the first time it launches on a device ordinal.
constexpr int kMaxDevices = 64;
struct PerDevice {
  std::once_flag once[kMaxDevices];
  cudaError_t err[kMaxDevices] = {};
  int per_sm[kMaxDevices] = {};   // resident CTAs of the kernel per SM
  int nsm[kMaxDevices] = {};      // SMs of the device
};
template <typename Init>
cudaError_t set_up_once(PerDevice& t, int dev, Init init) {
  if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
  std::call_once(t.once[dev], [&] { t.err[dev] = init(t.per_sm[dev], t.nsm[dev]); });
  return t.err[dev];
}

// Batches of 1.5-4 waves of resident CTAs (SCHED instantiations, with the LPT order: p.sched is set by
// schedule_batch) keep their hardest ranks on kHardSm reserved, half-empty SMs (see "work distribution" in
// solve_kernel).
constexpr int kHardSm = 32;
template <int N, int SPLIT, int MINB, int R = 1, bool CACHE = false, bool TC = false, bool SCHED = false, bool BODY = false,
          bool CONTACT = false, bool WEIGHTS = false, bool FORCE = false, bool STAGE = false>
cudaError_t launch_solve(const SolveParams& p_in, int dev, cudaStream_t s) {
  auto kernel = solve_kernel<N, SPLIT, MINB, R, CACHE, TC, false, BODY, CONTACT, WEIGHTS, FORCE, STAGE>;
  constexpr int THREADS = Geo<N, SPLIT, R>::THREADS;
  // 24 KB of static shared memory per CTA: MINB resident CTAs need the 196 KB carve-out (86 % of 228 KB); the
  // remaining 60 KB of L1 hold the register spills of the ADMM loop
  constexpr int kCarveoutPct = 70;
  static PerDevice setup;
  const cudaError_t e = set_up_once(setup, dev, [&](int& per_sm, int& nsm) {
    cudaError_t r = TC ? cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, kCarveoutPct)
                       : cudaSuccess;
    if constexpr (SCHED) {
      auto skernel = solve_kernel<N, SPLIT, MINB, R, CACHE, TC, true, BODY, CONTACT, WEIGHTS, FORCE, STAGE>;
      if (TC && r == cudaSuccess)
        r = cudaFuncSetAttribute(skernel, cudaFuncAttributePreferredSharedMemoryCarveout, kCarveoutPct);
      if (r == cudaSuccess) r = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, skernel, THREADS, 0);
      if (r == cudaSuccess) r = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    }
    return r;
  });
  if (e != cudaSuccess) return e;
  SolveParams p = p_in;
  if constexpr (SCHED) {
    auto skernel = solve_kernel<N, SPLIT, MINB, R, CACHE, TC, true, BODY, CONTACT, WEIGHTS, FORCE, STAGE>;
    const int per_sm = setup.per_sm[dev], nsm = setup.nsm[dev];
    const int wave = nsm * per_sm;       // CTAs the device holds at once
    // every reserved SM must receive its kHardSlots hard workers in the first wave (B > wave), and the other
    // SMs must be able to drain the main queue meanwhile
    // ... and only batches of 1.5-4 waves gain (3 seeds per size, trot / mixed gaits: 1536-3584 problems
    // +2...+7 %; 1024 and >= 4096 problems -1...-6 %: in a long launch the hardest problems are over long before
    // the end, and the rank assignment costs every CTA two L2 round trips; profiles/r02_reserved_sm_by_batch_size.jsonl)
    if (p.sched && per_sm > kHardSlots && nsm >= 2 * kHardSm && 2 * p.B > 3 * wave && p.B <= 4 * wave &&
        kHardSm * kHardSlots <= p.B / 4) {
      p.n_hard_sm = kHardSm;
      p.n_hard = kHardSm * kHardSlots;
      const int sleepers = kHardSm * (per_sm - kHardSlots);   // as many spare CTAs as can sleep on the reserved SMs
      return launch_pdl(skernel, dim3((unsigned)(p.B + sleepers)), dim3(THREADS), 0, s, p);
    }
  }
  p.sched = nullptr;
  return launch_pdl(kernel, dim3((unsigned)p.B), dim3(THREADS), 0, s, p);
}
// stage-wise (Riccati) kernel: dynamic shared memory above the 48 KB default needs the opt-in
template <int N, int MINB, bool BODY = false, bool CONTACT = false, bool WEIGHTS = false, bool FORCE = false,
          bool STAGE = false>
cudaError_t launch_solve_riccati(const SolveParams& p, int dev, cudaStream_t s) {
  using G_ = RGeo<N, WEIGHTS, FORCE, STAGE>;
  auto kernel = solve_riccati_kernel<N, MINB, BODY, CONTACT, WEIGHTS, FORCE, STAGE>;
  static PerDevice setup;
  const cudaError_t e = set_up_once(setup, dev, [&](int&, int&) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G_::SMEM_BYTES);
  });
  if (e != cudaSuccess) return e;
  return launch_pdl(kernel, dim3((unsigned)p.B), dim3(G_::THREADS), G_::SMEM_BYTES, s, p);
}

// The solve launchers of one compiled horizon.
struct SolveRow {
  SolveLaunch solve;    // default kernel of the horizon
  SolveLaunch other;    // the other formulation (cfg.kernel_variant = 5), or nullptr
  SolveLaunch cached;   // default kernel with the factorisation cache compiled in, or nullptr
};
constexpr int kNumHorizons = 10;

// The solve launchers of every compiled horizon for one feature set, row i for horizon kHorizons[i].N (cmpc.cu).
// Dense kernels <N, SPLIT, MINB, R>: a thread owns an R x (6N/SPLIT) register tile of the 6N x 6N wrench matrix
// (R rows, one of SPLIT column slices), <= 96 floats.  Default kernel of the horizon:
//   N <= 16: dense single-CTA kernel (cmpc_kernels.cuh); N = 10: <10, 1, MINB = 6, 1, CACHE, TC, SCHED> = factorisation
//            sweep on the tensor cores (cmpc_tc.cuh), 6 CTAs/SM at 168 registers, reserved-SM rank assignment for
//            batches of 1.5-4 waves (measured faster than the SIMT sweep and than the tensor-core sweep at 8 CTAs/SM:
//            profiles/r02_tc_sweep_vs_simt.jsonl, r02_occupancy_carveout_exp.jsonl, r02_reserved_sm_policy.jsonl);
//   N >= 20: stage-wise Riccati kernel (cmpc_riccati.cuh), measured on B200 against the dense kernel and a
//            thread-block-cluster kernel: N=20 1.5x at 16384 problems (equal at 4096), N=30 2.25x (config 4),
//            N=40 3.4x, N=60 5.2x (profiles/r02_riccati_vs_dense.jsonl).
// `other` is the other formulation where both fit (Riccati for N <= 16, dense for N = 20 / 30): tests compare
// the two kernels on the same problems.
// Each translation unit instantiates only its own feature sets (BODY, CONTACT, WEIGHTS, FORCE, STAGE): cmpc.cu the
// plain kernels (0,0,0,0,0) of a handle that has never received a body, a contact, weights, force references or stage
// weights, cmpc_body.cu (1,0,0,0,0), cmpc_contact.cu (1,1,0,0,0), cmpc_weights.cu (1,0,1,0,0) and (1,1,1,0,0),
// cmpc_force.cu (1,0,1,1,0) and (1,1,1,1,0), cmpc_stage.cu (1,0,1,1,1) and (1,1,1,1,1); CONTACT and WEIGHTS are
// compiled with BODY only, FORCE with BODY + WEIGHTS only, STAGE with BODY + WEIGHTS + FORCE only.  The compiler's
// inlining decisions depend on what else a module holds: in one module with the BODY kernels the plain N = 30 dense
// kernels stopped inlining their factorisation.
template <bool BODY, bool CONTACT, bool WEIGHTS, bool FORCE = false, bool STAGE = false>
const SolveRow* solve_rows() {
  constexpr bool B = BODY, C = CONTACT, W = WEIGHTS, F = FORCE, S = STAGE;
  static const SolveRow rows[] = {
      {launch_solve<4, 1, 8, 1, false, false, false, B, C, W, F, S>, nullptr, nullptr},
      {launch_solve<5, 1, 8, 1, false, false, false, B, C, W, F, S>, nullptr, nullptr},
      {launch_solve<8, 1, 8, 1, false, false, false, B, C, W, F, S>, nullptr, nullptr},
      {launch_solve<10, 1, 6, 1, false, true, true, B, C, W, F, S>, launch_solve_riccati<10, 8, B, C, W, F, S>,
       launch_solve<10, 1, 6, 1, true, true, true, B, C, W, F, S>},
      {launch_solve<12, 2, 4, 1, false, false, false, B, C, W, F, S>, launch_solve_riccati<12, 8, B, C, W, F, S>, nullptr},
      {launch_solve<16, 2, 3, 1, false, false, false, B, C, W, F, S>, launch_solve_riccati<16, 8, B, C, W, F, S>, nullptr},
      {launch_solve_riccati<20, 6, B, C, W, F, S>, launch_solve<20, 2, 2, 1, false, false, false, B, C, W, F, S>, nullptr},
      {launch_solve_riccati<30, 4, B, C, W, F, S>, launch_solve<30, 6, 1, 3, false, false, false, B, C, W, F, S>,
       launch_solve<30, 6, 1, 3, true, false, false, B, C, W, F, S>},
      {launch_solve_riccati<40, 3, B, C, W, F, S>, nullptr, nullptr},
      {launch_solve_riccati<60, 2, B, C, W, F, S>, nullptr, nullptr},
  };
  static_assert(sizeof rows / sizeof rows[0] == kNumHorizons);
  return rows;
}
extern template const SolveRow* solve_rows<false, false, false>();   // cmpc.cu
extern template const SolveRow* solve_rows<true, false, false>();    // cmpc_body.cu
extern template const SolveRow* solve_rows<true, true, false>();     // cmpc_contact.cu
extern template const SolveRow* solve_rows<true, false, true>();     // cmpc_weights.cu
extern template const SolveRow* solve_rows<true, true, true>();      // cmpc_weights.cu
extern template const SolveRow* solve_rows<true, false, true, true>();   // cmpc_force.cu
extern template const SolveRow* solve_rows<true, true, true, true>();    // cmpc_force.cu
extern template const SolveRow* solve_rows<true, false, true, true, true>();   // cmpc_stage.cu
extern template const SolveRow* solve_rows<true, true, true, true, true>();    // cmpc_stage.cu

// cmpc_contact.cu: fill n leg-stage records with the "never set" state (init_contact_kernel), and store the
// contacts of slots [slot0, slot0 + B) of a handle with horizon N and kernel horizon NK (set_contact_kernel)
cudaError_t init_contact(float4* contact, float f_min, float f_max, size_t n, cudaStream_t s);
cudaError_t store_contact(const float* normal, const float* mu, const float* f_min, const float* f_max,
                          float4* contact, int slot0, int B, int N, int NK, cudaStream_t s);

// cmpc_weights.cu: give `slots` slots the handle's weight record `rec` and Gram tables Minv / Mg ([6][NK][NK], or
// nullptr when the handle has no per-slot tables) (init_weights_kernel), and store the weights of slots
// [slot0, slot0 + B) of a handle with horizon N and kernel horizon NK (set_weights_kernel); w_Minv / w_Mg are
// nullptr for NK > kWeightTableMaxN.  `w` holds one row of 13 per slot (ws = 0, cmpc_set_weights) or one per stage
// (ws = 13, [B][N][13], cmpc_set_stage_weights); a handle with stage weights passes its table `wstage`
// ([slots][NK][kStageF4]), which receives every stage's row, else nullptr.
cudaError_t init_weights(float4* weights, float* w_Minv, float* w_Mg, const float rec[4 * kWeightF4],
                         const float* Minv, const float* Mg, int slots, int NK, cudaStream_t s);
cudaError_t store_weights(const float* w, int ws, const float* r_weight, float4* weights, float4* wstage,
                          float* w_Minv, float* w_Mg, float* cache_meta, int slot0, int B, int N, int NK, float dt,
                          int dev, cudaStream_t s);
// cmpc_weights.cu: give every one of `slots` slots of the stage table wstage its weight record's w[0..11] on stages
// [0, N) and zeros on the padding stages [N, NK) (init_stage_weights_kernel)
cudaError_t init_stage_weights(float4* wstage, const float4* weights, int slots, int N, int NK, cudaStream_t s);

// cmpc_force.cu: store the force references f_ref [B,N,4,3] and weights [B,N,4] of slots [slot0, slot0 + B) at the
// kernel horizon's stride NK into force ([slots][NK][4] float4) and invalidate their cached factors (set_force_ref_kernel)
cudaError_t store_force_ref(const float* f_ref, const float* weight, float4* force, float* cache_meta, int slot0, int B,
                            int N, int NK, cudaStream_t s);

// cmpc_wrench.cu: the pre- and post-pass of a solve of a handle with wrenches (cmpc_set_wrench), one CTA per problem
struct WrenchParams {
  const float* x0;        // [B,13]
  const float* x_des;     // [B,NK+1,13] read by wrench_shift ...
  float* x_des_out;       // ... which writes x_des - phi here (may be x_des itself)
  float* X;               // [B,N+1,13] wrench_finish adds phi (or nullptr)
  int32_t* status;        // [B] wrench_finish reports invalid wrenches (or nullptr)
  const float* wrench;    // the batch's slots of the wrench array, [B][N][6]
  const float4* body;     // the batch's slots of the body array, [B][kBodyF4]
  int32_t B, N, NK;       // batch, horizon, kernel horizon
  float dt;
};
// store the wrenches force, torque [B,N,3] of slots [slot0, slot0 + B) (set_wrench_kernel)
cudaError_t store_wrench(const float* force, const float* torque, float* wrench, int slot0, int B, int N,
                         cudaStream_t s);
cudaError_t wrench_shift(const WrenchParams& p, cudaStream_t s);    // wrench_shift_kernel, PDL launch
cudaError_t wrench_finish(const WrenchParams& p, cudaStream_t s);   // wrench_finish_kernel

}  // namespace cmpc
