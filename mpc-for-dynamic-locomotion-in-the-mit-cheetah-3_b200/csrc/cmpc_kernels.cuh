// cmpc_kernels.cuh - sm_100a device code of the batched convex-MPC solver.
//
// Problem (reference src/mpc.py:64-173): single-rigid-body dynamics linearised over N
// stages, quadratic tracking cost on the 12 states, forces of swing legs pinned to zero,
// fz in [f_min, f_max] and a friction pyramid |fx|,|fy| <= mu fz per stance leg.
//
// Formulation used on the GPU (DESIGN.md section 3).  After eliminating the states the
// cost depends on the forces u only through the 6N-vector of per-stage wrenches
//     w = G u,   w_j = [ Rz I^-1 sum_l [r_jl]x f_jl ;  sum_l f_jl / m ]
//     H = G' M G,  M = blockdiag over 6 axes of constant N x N Gram matrices (host, fp64).
// OSQP-style ADMM (x-update / relaxation / dual update of Stellato et al. 2020) with the
// constraint copy z = u kept in the friction frustum C = {fz in [f_min,f_max], |fx|,|fy| <= mu fz}
// by an exact Euclidean projection.  The x-update needs K^-1, K = H + (sigma + rho) I = d^-1 I + G'MG;
// by the matrix-inversion lemma
//     K^-1 = d I - d^2 G' P^-1 G,    P = M^-1 + d G G'   (6N x 6N, SPD).
// One CTA per problem:
//   * "leg threads"   (4N): one per leg-stage, keep that leg's x(3), z(3), y(3) in registers;
//   * "wrench threads"(6N*SPLIT): own one row (slice) of P, invert it in registers with a
//     symmetric Gauss-Jordan sweep whose pivot rows are broadcast through shared memory,
//     then apply P^-1 once per ADMM iteration.
// The iteration is written in residual-correction form (K d = -r_dual - rho r_prim,
// x += alpha d) so fp32 solve errors do not accumulate, and uses M G d = P^-1 s to keep the
// wrench-space gradient v = M G x up to date without a second matrix-vector product.
#pragma once
#include <cuda_runtime.h>
// Packed fp32 FMA (sm_100 FFMA2, fma.rn.f32x2) in the sweep and in the P^-1 application: two row
// entries per instruction, bit-identical results.  Measured on B200: config 2
// 0.294 -> 0.281 ms per 4096-problem batch, config 3 shard 0.684 -> 0.654 ms.
#include <stdint.h>
#include <type_traits>

#include "cmpc_tc.cuh"

namespace cmpc {

// Below this level both normalised residuals are fp32 rounding noise and their ratio carries no
// information: rho stops adapting (a run with eps = 0 would otherwise let rho drift on noise and
// lose accuracy).  Every finite tolerance >= 1e-5 exits long before, so iterates are unchanged.
constexpr float kRhoAdaptFloor = 1e-6f;

// scheduling state of a SCHED launch: [0] next main rank, [1] next hard rank, [2] CTAs that left,
// [3] reserved-SM tickets, then per SM id (< kSchedSm): arrivals, role (0 unknown, 1 reserved, 2 normal),
// hard problems in flight, hard workers that have made their take
constexpr int kSchedSm = 256;
constexpr int kSchedInts = 16 + 4 * kSchedSm;
constexpr int kHardSlots = 4;         // CTAs of a reserved SM that serve the hard queue

struct SolveParams {
  const float* __restrict__ x0;
  const float* __restrict__ r;
  const uint8_t* __restrict__ mask;
  const float* __restrict__ x_des;
  const float* __restrict__ mu;
  float* __restrict__ U;
  float* __restrict__ X;
  int32_t* __restrict__ iters;
  float* __restrict__ pri_res;
  float* __restrict__ dua_res;
  int32_t* __restrict__ status;
  float* __restrict__ warm_x;         // [slots][N][12]
  float* __restrict__ warm_y;         // [slots][N][4][3]
  uint8_t* __restrict__ warm_valid;   // [slots]
  union {
    const float* __restrict__ Minv;   // [6][N][N], read by the dense kernels without WEIGHTS
    // per-leg-stage force references (cmpc_set_force_ref), read by the FORCE instantiations only, which are compiled
    // with WEIGHTS and read M^-1 from w_Minv: [slots][N][4] float4 = {f_ref (world frame), w_f}; w_f is NaN on every
    // leg-stage of a slot stored with an invalid entry.  In Minv's place so that the parameter block keeps its size:
    // a larger one changes the machine code of the kernels that copy it to local memory (the N = 30 dense ones).
    const float4* __restrict__ force;
  };
  union {
    const float* __restrict__ Mg;     // [6][N][N], read by the dense kernels without WEIGHTS
    // per-stage state weights (cmpc_set_stage_weights), read by the STAGE instantiations only, which are compiled
    // with WEIGHTS and read M from w_Mg: [slots][N][kStageF4] float4 = w[0..11] of stage i + 1 (zero on padding
    // stages).  In Mg's place for the reason given at `force`.
    const float4* __restrict__ wstage;
  };
  const int32_t* __restrict__ order;  // launch order (hardest first) or nullptr
  int32_t B;
  int32_t slot0;
  int32_t n_eff;                      // stages that carry cost (<= N; the rest is all-swing padding, 0 = N)
  float dt, inv_mass;
  float ib[3];
  float w[13];
  float r_weight, f_min, f_max, rho, sigma, alpha, eps_abs, eps_rel;
  int32_t max_iter, check_every, refresh_every, warm_mode;
  int32_t adaptive_rho_interval;      // 0 = fixed rho
  float adaptive_rho_tolerance;
  float rho_min, rho_max;             // clamp of the adapted rho (fp32 stability of the Woodbury form)
  // batches of 1.5-4 waves: CTAs take their launch-order rank when they start; the first n_hard ranks
  // (the hardest by the LPT score) go to kHardSlots CTAs on each of n_hard_sm reserved SMs, whose other CTAs
  // wait until those problems are done (see "work distribution" in solve_kernel)
  int32_t* sched;                     // kSchedInts ints of scheduling state, all zero between launches
  int32_t n_hard, n_hard_sm;
  // factorisation cache (closed-loop use, cfg.cache_factorization): -P^-1 of each slot's last
  // factorisation with the data it was computed for; nullptr = off
  float4* __restrict__ cache_pinv;    // [slots][NW*NWP/4 float4], laid out [tile piece][thread]
  float* __restrict__ cache_r;        // [slots][12 N] lever arms of that factorisation
  uint8_t* __restrict__ cache_mask;   // [slots][N]
  float* __restrict__ cache_meta;     // [slots][4]: rho, yaw, valid, reused by the last launch
  float cache_tol_r, cache_tol_yaw;
  int32_t cache_max_iter;             // a solve that needs more iterations invalidates its cache entry
  uint8_t* __restrict__ cache_hit;         // [slots] 1 if the last launch reused a cached factor
  // per-slot rigid body (cmpc_set_body), read by the BODY instantiations only: [slots][kBodyF4] float4 =
  // {1/m, Ib^-1 row-major (9), 0, 0}; 1/m is NaN for a slot stored with an invalid body
  const float4* __restrict__ body;
  // per-leg-stage contact surface (cmpc_set_contact), read by the CONTACT instantiations only:
  // [slots][N][4][kContactF4] float4 = {n (unit), mu}, {f_min, f_max, 0, 0}; see load_contact
  const float4* __restrict__ contact;
  // per-slot cost weights (cmpc_set_weights), read by the WEIGHTS instantiations only: [slots][kWeightF4] float4 =
  // {w[0..12], r_weight, 0, 0}; r_weight is NaN for a slot stored with invalid weights
  const float4* __restrict__ weights;
  // the slots' horizon Gram matrices M^-1 and M, [slots][6][N][N] each in the layout of Minv / Mg (read by the
  // dense WEIGHTS instantiations; allocated for kernel horizons N <= 30 only)
  const float* __restrict__ w_Minv;
  const float* __restrict__ w_Mg;
};
// the size every solve kernel is compiled with (see `force`): a new field goes into a union with one that the kernels
// reading it do not read
static_assert(sizeof(SolveParams) == 400, "the parameter block keeps its size");
constexpr int kBodyF4 = 3;     // float4 per slot of the body array
constexpr int kContactF4 = 2;   // float4 per leg-stage of the contact array
constexpr int kWeightF4 = 4;    // float4 per slot of the weight array
constexpr int kStageF4 = 3;     // float4 per stage of the stage-weight array (w[0..11])
constexpr int kWeightTableMaxN = 30;   // largest kernel horizon with per-slot Gram tables (dense and condense kernels)

// entry i of slot `slot`'s weight record {w[0..12], r_weight} (WEIGHTS instantiations)
__device__ __forceinline__ float slot_weight(const SolveParams& p, int slot, int i) {
  return __ldg(reinterpret_cast<const float*>(p.weights + (size_t)slot * kWeightF4) + i);
}

// Thread geometry.  Every "row thread" owns R rows of P (rows rp + q*NWR, q < R: same axis,
// stages N/R apart) restricted to one of SPLIT column slices, i.e. an R x COLS register tile.
// One broadcast 16-byte shared-memory load of the pivot row / rhs feeds 4R FMAs: R = 1 makes
// the sweep shared-memory-bandwidth bound (measured: a warp-uniform LDS.128 costs 2.4 cycles of
// the SM's shared-memory pipe, 15 of them per 60 FMAs), R = 2 halves that traffic.
template <int N, int SPLIT, int R = 1>
struct Geo {
  static_assert(N % R == 0, "rows of one thread must share their axis");
  static constexpr int NW = 6 * N;                                  // wrench dimension
  static constexpr int NWR = NW / R;                                // row groups
  static constexpr int NWP = ((NW + 4 * SPLIT - 1) / (4 * SPLIT)) * (4 * SPLIT);
  static constexpr int COLS = NWP / SPLIT;                          // row slice per thread
  static constexpr int NLEG = 4 * N;
  static constexpr int ROWT = NWR * SPLIT;                          // threads owning P rows
  static constexpr int TMAX = ROWT > NLEG ? ROWT : NLEG;
  static constexpr int THREADS = ((TMAX + 31) / 32) * 32;
  static constexpr int WARPS = THREADS / 32;
  static constexpr int LWARPS = (NLEG + 31) / 32;                   // warps that own leg threads
  static constexpr int NX = 13 * (N + 1);
};

// a[i] for a runtime i by selects (a dynamically indexed register array goes to local memory)
__device__ __forceinline__ float pick6(const float a[6], int i) {
  float e = a[0];
#pragma unroll
  for (int q = 1; q < 6; ++q) e = (i == q) ? a[q] : e;
  return e;
}

// Programmatic dependent launch (see launch_pdl in cmpc.cu): wait until every kernel launched before
// this one in the stream has completed and its writes are visible; a no-op for ordinary launches.
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// allow the next kernel of the stream to be scheduled (it still waits for this one in its own wait)
__device__ __forceinline__ void grid_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }

__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}

// (a[2l], a[2l+1]) for l = 0..2 by selects: a dynamically indexed register array would be
// demoted to local memory (a store + load round trip per ADMM iteration)
__device__ __forceinline__ float2 pick_pair(const float a[6], int l) {
  return make_float2(l == 0 ? a[0] : (l == 1 ? a[2] : a[4]), l == 0 ? a[1] : (l == 1 ? a[3] : a[5]));
}

__device__ __forceinline__ float warp_max_nonneg(float v) {
  // v >= 0 (or NaN): IEEE bit patterns of non-negative floats order like unsigned ints,
  // NaN (0x7fc00000) sorts above every finite value so it propagates.
  return __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(v)));
}

// Per-leg geometry: Ghat = Rz * (Rz diag(ib) Rz') * [r]x   (torque rows of G, rotated frame)
__device__ __forceinline__ void leg_map(float c, float s, const float ib[3], float rx, float ry,
                                        float rz, float G[3][3]) {
  // S = [r]x
  const float S[3][3] = {{0.f, -rz, ry}, {rz, 0.f, -rx}, {-ry, rx, 0.f}};
  float A[3][3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {   // A = diag(ib) * Rz' * S
    A[0][k] = ib[0] * (c * S[0][k] + s * S[1][k]);
    A[1][k] = ib[1] * (-s * S[0][k] + c * S[1][k]);
    A[2][k] = ib[2] * S[2][k];
  }
  float T[3][3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {   // T = Rz * A  (= I_hat^-1 [r]x, reference src/mpc.py:78,103)
    T[0][k] = c * A[0][k] - s * A[1][k];
    T[1][k] = s * A[0][k] + c * A[1][k];
    T[2][k] = A[2][k];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {   // Ghat = Rz * T
    G[0][k] = c * T[0][k] - s * T[1][k];
    G[1][k] = s * T[0][k] + c * T[1][k];
    G[2][k] = T[2][k];
  }
}

// leg_map with a full body-frame inverse inertia ib (3x3 row-major): A = ib * Rz' * S with the same
// q = Rz' S columns as leg_map, so a diagonal ib only adds exact zeros and gives leg_map's values
__device__ __forceinline__ void leg_map_full(float c, float s, const float* ib, float rx, float ry,
                                             float rz, float G[3][3]) {
  const float S[3][3] = {{0.f, -rz, ry}, {rz, 0.f, -rx}, {-ry, rx, 0.f}};
  float A[3][3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float q0 = c * S[0][k] + s * S[1][k];
    const float q1 = -s * S[0][k] + c * S[1][k];
    const float q2 = S[2][k];
#pragma unroll
    for (int i = 0; i < 3; ++i) A[i][k] = ib[3 * i] * q0 + ib[3 * i + 1] * q1 + ib[3 * i + 2] * q2;
  }
  float T[3][3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    T[0][k] = c * A[0][k] - s * A[1][k];
    T[1][k] = s * A[0][k] + c * A[1][k];
    T[2][k] = A[2][k];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    G[0][k] = c * T[0][k] - s * T[1][k];
    G[1][k] = s * T[0][k] + c * T[1][k];
    G[2][k] = T[2][k];
  }
}

// Exact Euclidean projection onto the friction frustum {fz in [fmin, fmax], |fx|,|fy| <= mu fz}
// (inv1 = 1/(1+mu^2), inv2 = 1/(1+2mu^2)): the same arithmetic as the `project` lambdas of the plain solve
// kernels, which keep their own copy (calling this function reorders a select in their SASS)
__device__ __forceinline__ void project_frustum(float wx, float wy, float wz, float mu, float inv1, float inv2,
                                                float fmin, float fmax, float& zx, float& zy, float& zz) {
  const float ax = fabsf(wx), ay = fabsf(wy);
  const float big = fmaxf(ax, ay), small = fminf(ax, ay);
  const float f2 = (wz + mu * big) * inv1;
  const float f1 = (wz + mu * (ax + ay)) * inv2;
  float fz = (mu * wz >= big) ? wz : ((mu * f2 >= small) ? f2 : f1);
  fz = fminf(fmaxf(fz, fmin), fmax);
  const float lim = mu * fz;
  zx = fminf(fmaxf(wx, -lim), lim);
  zy = fminf(fmaxf(wy, -lim), lim);
  zz = fz;
}

// The constraint of one leg-stage of a CONTACT instantiation, held in registers through the ADMM loop: the
// frustum above in the contact frame R = [t1 t2 n] of the leg's ground.  The projection onto R C is R P_C(R' w).
struct LegContact {
  float t1[3], t2[3], n[3];
  float mu, inv1, inv2, fmin, fmax;
};

// Build a leg-stage's constraint from its record (cmpc_set_contact, set_contact_kernel).  A record never set has
// mu < 0: the call's mu (the record holds world axes and the configuration's bounds).  The frame: t1 = the
// normalised part of e_x orthogonal to n, or of e_y when n is within 45 degrees of e_x; t2 = n x t1.  For
// n = (0,0,1) every product with 1 or 0 is exact, so R is the identity and the projection is the world-axis one.
__device__ __forceinline__ void load_contact(const float4* rec, float call_mu, LegContact& c) {
  const float4 a = __ldg(rec), b = __ldg(rec + 1);
  c.n[0] = a.x; c.n[1] = a.y; c.n[2] = a.z;
  c.mu = a.w < 0.f ? call_mu : a.w;              // NaN (an invalid record) stays NaN
  c.fmin = b.x;
  c.fmax = b.y;
  c.inv1 = 1.f / (1.f + c.mu * c.mu);
  c.inv2 = 1.f / (1.f + 2.f * c.mu * c.mu);
  const bool ex = a.x * a.x <= 0.5f;
  const float e = ex ? a.x : a.y;                // e . n
  const float v0 = (ex ? 1.f : 0.f) - e * a.x, v1 = (ex ? 0.f : 1.f) - e * a.y, v2 = -e * a.z;
  const float len = sqrtf(v0 * v0 + v1 * v1 + v2 * v2);
  c.t1[0] = v0 / len; c.t1[1] = v1 / len; c.t1[2] = v2 / len;
  c.t2[0] = a.y * c.t1[2] - a.z * c.t1[1];
  c.t2[1] = a.z * c.t1[0] - a.x * c.t1[2];
  c.t2[2] = a.x * c.t1[1] - a.y * c.t1[0];
}

__device__ __forceinline__ void project_contact(const LegContact& c, float wx, float wy, float wz, float& zx,
                                                float& zy, float& zz) {
  const float a = c.t1[0] * wx + c.t1[1] * wy + c.t1[2] * wz;
  const float b = c.t2[0] * wx + c.t2[1] * wy + c.t2[2] * wz;
  const float d = c.n[0] * wx + c.n[1] * wy + c.n[2] * wz;
  float pa, pb, pd;
  project_frustum(a, b, d, c.mu, c.inv1, c.inv2, c.fmin, c.fmax, pa, pb, pd);
  zx = c.t1[0] * pa + c.t2[0] * pb + c.n[0] * pd;
  zy = c.t1[1] * pa + c.t2[1] * pb + c.n[1] * pd;
  zz = c.t1[2] * pa + c.t2[2] * pb + c.n[2] * pd;
}

// Tracking error of the free response at stage k on wrench axis a (position-like and
// velocity-like part; angular velocity error rotated by Rz):  e = free response - x_des.
// In double: the inputs are fp32, their differences are exact, and the linear term h below is a
// sum of N terms of size ~1e3 whose rounding in fp32 (~1e-3 absolute) is NOT harmless - the
// wrench components with the smallest cost curvature (2 w_pos dt^4 ~ 3e-3 per N^2) move by
// gradient error / curvature, i.e. by tenths of a newton at N = 60 (measured, scripts/gpu_tight_diag.py).
__device__ __forceinline__ void stage_error(int k, int a, const float* sx0, const float* sxd, float c,
                                            float s, float dt, double& e_pos, double& e_vel) {
  const float* xd = sxd + 13 * k;
  const double kf = (double)k, dtd = (double)dt, cd = (double)c, sd = (double)s;
  if (a < 3) {
    const double w0x = sx0[6], w0y = sx0[7], wdx = xd[6], wdy = xd[7];
    const double rw0 = a == 0 ? (cd * w0x - sd * w0y) : (a == 1 ? (sd * w0x + cd * w0y) : (double)sx0[8]);
    const double rwd = a == 0 ? (cd * wdx - sd * wdy) : (a == 1 ? (sd * wdx + cd * wdy) : (double)xd[8]);
    e_pos = ((double)sx0[a] - (double)xd[a]) + kf * dtd * rw0;
    e_vel = rw0 - rwd;
  } else {
    const int aa = a - 3;
    double pf = ((double)sx0[3 + aa] - (double)xd[3 + aa]) + kf * dtd * (double)sx0[9 + aa];
    double vf = (double)sx0[9 + aa] - (double)xd[9 + aa];
    if (aa == 2) {
      const double g = sx0[12];
      pf += 0.5 * kf * (kf - 1.0) * dtd * dtd * g;
      vf += kf * dtd * g;
    }
    e_pos = pf;
    e_vel = vf;
  }
}

// Linear term of the wrench-space cost: h[6j+a] = 2 sum_{k>j} (w_pos,k d^2 (k-1-j) e_pos + w_vel,k d e_vel),
// stages k <= n_eff only (the rest of a padded horizon carries no cost).  Stage k's weights are
// w[ws (k-1) ...]: ws = 0 for one row for every stage, 12 for per-stage rows (cmpc_set_stage_weights).
template <int N>
__device__ __forceinline__ float wrench_linear_term(int j, int a, const float* sx0,
                                                    const float* sxd, float c, float s,
                                                    const float* w, int ws, float dt, int n_eff) {
  const double dtd = dt;      // w[0:3] Theta, w[3:6] p, w[6:9] omega, w[9:12] v
  double acc = 0.0;
  for (int k = j + 1; k <= n_eff; ++k) {
    const double wp = w[ws * (k - 1) + a], wv = w[ws * (k - 1) + 6 + a];
    double e_pos, e_vel;
    stage_error(k, a, sx0, sxd, c, s, dt, e_pos, e_vel);
    acc += 2.0 * (wp * dtd * dtd * (double)(k - 1 - j) * e_pos + wv * dtd * e_vel);
  }
  return (float)acc;
}

// ---------------------------------------------------------------------------------------
// Fused condense + factor + ADMM kernel.  One CTA per problem.
// ---------------------------------------------------------------------------------------
// CACHE compiles the factorisation cache in (closed-loop instantiations); the default
// instantiation carries none of its state through the register-limited ADMM loop.
// TC runs the factorisation sweep on the tensor cores (cmpc_tc.cuh; one 64-thread CTA, 6N <= 64).
// SCHED compiles the reserved-SM rank assignment in (p.sched; see "work distribution" below).
// BODY reads the problem's rigid body from its slot of p.body instead of p.inv_mass / p.ib.
// CONTACT projects each leg-stage onto its own contact surface from p.contact (LegContact).
// WEIGHTS reads the problem's cost weights and Gram tables from its slot of p.weights / p.w_Minv / p.w_Mg
// instead of p.w / p.r_weight / p.Minv / p.Mg.
// FORCE adds each stance leg-stage's force reference from p.force: w_f ||f - f_ref||^2, so 2 w_f joins the leg's
// curvature (d, the 2 r_weight x gradient term) and -2 w_f f_ref its linear term.
// STAGE reads the state weights of every stage from p.wstage in the linear term h; M and M^-1 are the slot's w_Mg /
// w_Minv, which cmpc_set_stage_weights builds from the same stage weights.
template <int N, int SPLIT, int MINB, int R, bool CACHE, bool TC = false, bool SCHED = false, bool BODY = false,
          bool CONTACT = false, bool WEIGHTS = false, bool FORCE = false, bool STAGE = false>
__global__ void __launch_bounds__((Geo<N, SPLIT, R>::THREADS), MINB)
solve_kernel(const SolveParams p) {
  using G_ = Geo<N, SPLIT, R>;
  constexpr int NW = G_::NW, NWP = G_::NWP, COLS = G_::COLS, NLEG = G_::NLEG, NWR = G_::NWR;
  constexpr int THREADS = G_::THREADS, LWARPS = G_::LWARPS, NX = G_::NX;
  static_assert(!TC || (SPLIT == 1 && R == 1 && THREADS == kTcN && NW <= kTcN), "tensor-core sweep: one row per thread, 64 threads");
  static_assert(!FORCE || (BODY && WEIGHTS), "force references are compiled with BODY + WEIGHTS only");
  static_assert(!STAGE || FORCE, "stage weights are compiled with BODY + WEIGHTS + FORCE only");
  __shared__ __align__(16) float s_P[TC ? tc_smem_floats<NW>() : 4];   // row <-> fragment staging of the tensor-core sweep
  // FORCE: this thread's {-2 w_f f_ref, 2 w_f}, zero on swing legs and non-leg threads (each thread reads its own)
  __shared__ __align__(16) float4 s_fr[FORCE ? THREADS : 1];

  __shared__ __align__(16) float s_x0[BODY ? 16 + 4 * kBodyF4 : 16];   // x0 (13); WEIGHTS: 2 r_weight at 13; FORCE: w_f of leg-stage 0 at 14 (NaN: invalid slot); BODY: the slot's body at 16
  __shared__ __align__(16) float s_xd[NX + 3];         // x_des; reused to stage U at the end
  __shared__ __align__(16) float s_r[3 * NLEG];        // lever arms as loaded (coalesced)
  __shared__ __align__(16) float s_G[NLEG][12];        // Ghat (9) + dxy, dz, pad per leg
  __shared__ __align__(16) float s_rowA[NWP + 4];      // pivot-row double buffer (+ 1/pivot): two
  __shared__ __align__(16) float s_rowB[NWP + 4];      // arrays, so loads of one never alias stores to the other
  __shared__ __align__(16) float s_s[NWP];             // wrench-space rhs  s = G D^-1 b
  __shared__ __align__(16) float s_q[SPLIT][NWP];      // q = P^-1 s as SPLIT partial sums
  __shared__ __align__(16) float s_v[NWP];             // exact gradient M G x (refresh)
  __shared__ __align__(16) float s_h[NWP];             // linear term h
  __shared__ __align__(16) float s_S[NWP];             // Jacobi scaling 1/sqrt(P_ii) of the sweep
  __shared__ float s_red[2][LWARPS][8];
  __shared__ __align__(8) float s_dump[2 * THREADS];   // scratch target of lanes that own no wrench pair
  __shared__ float s_gl[3 * NLEG];                      // G' h per leg (read at check iterations only)
  __shared__ float s_pre[2][6 * (N + 1)];              // prefix sums for the X output
  __shared__ double s_e[2][NW];                         // stage errors of the linear term (fp64)
  __shared__ int s_mask[N];

  __shared__ int s_item;
  __shared__ int s_sm[2];                 // SCHED, thread 0: SM id, hard item in flight
  if (!SCHED && (int)blockIdx.x >= p.B) return;
  grid_dependency_wait();
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const bool leg_warp = warp < LWARPS;   // warp-uniform: warps without leg threads skip leg phases

  // ---- work distribution --------------------------------------------------------------------------
  // !SCHED: CTA i solves rank i of the launch order.  SCHED: still one problem per CTA, but a CTA takes
  // its rank when it starts, by the role of the SM it landed on.  A CTA's iteration latency doubles
  // between an idle and a full SM (gpu_iter_latency.py) and the batch ends when its hardest problem does,
  // so the n_hard hardest ranks are kept off the full SMs: the first n_hard_sm SMs to report are reserved,
  // the first kHardSlots CTAs of a reserved SM take ranks from the hard queue, and every other CTA that
  // lands there sleeps until this SM's hard problems are solved (it holds a CTA slot but no issue slots;
  // the hardware keeps placing the remaining CTAs on the other SMs).  Everybody
  // else takes the next main rank, or a hard one when the main queue is empty.  The grid has as many CTAs
  // more than ranks as there can be sleepers, so a sleeper that wakes up to empty queues leaves without
  // work instead of starting one of the last problems late.  Thread 0 only; nothing stays in registers.
  int item = (int)blockIdx.x;
  if constexpr (SCHED) {
    if (tid == 0) {
      int* S = p.sched;
      const int nh = p.n_hard, nm = p.B - nh;
      int sm_id, role = 2, arrival = kHardSlots;
      asm volatile("mov.u32 %0, %smid;" : "=r"(sm_id));
      if (sm_id >= kSchedSm) sm_id = kSchedSm - 1;
      int* running = S + 16 + 2 * kSchedSm + sm_id;
      {
        // the role of an SM is fixed by its first CTA; CTAs of later waves on the ordinary SMs (the common case)
        // pay one load for it, and only reserved SMs count their arrivals further
        volatile int* rp_ = S + 16 + kSchedSm + sm_id;
        role = *rp_;
        if (role != 2) {
          arrival = atomicAdd(S + 16 + sm_id, 1);
          if (arrival == 0) {
            role = atomicAdd(S + 3, 1) < p.n_hard_sm ? 1 : 2;
            atomicExch(S + 16 + kSchedSm + sm_id, role);
          } else {
            while ((role = *rp_) == 0) __nanosleep(100);   // the first CTA of this SM is about to set it
          }
        }
      }
      int got = p.B, hard = 0;
      const bool reserved = role == 1, hard_worker = reserved && arrival < kHardSlots;
      // A sleeper waits for this SM only: for its kHardSlots hard workers (they arrived before it and do not
      // block) to have made their take, and for the hard problems they took to be solved.  It never waits for
      // the queues, so no CTA placement by the hardware (other kernels on the device) can stall the launch.
      int* settled = S + 16 + 3 * kSchedSm + sm_id;
      if (reserved && !hard_worker) {
        unsigned ns = 250;              // back off to ~4 us between polls: a hard problem runs for 50-250 us
        while (*(volatile int*)settled < kHardSlots || *(volatile int*)running > 0) {
          __nanosleep(ns);
          if (ns < 4000) ns *= 2;
        }
      }
      if (hard_worker) {
        if (atomicAdd(S + 1, 0) < nh) {
          atomicAdd(running, 1);
          const int h = atomicAdd(S + 1, 1);
          if (h < nh) { got = h; hard = 1; }
          else atomicSub(running, 1);
        }
        __threadfence();                // `running` is up before this worker counts as settled
        atomicAdd(settled, 1);
      }
      if (got == p.B) {
        const int m = atomicAdd(S, 1);
        if (m < nm) got = nh + m;
      }
      if (got == p.B && nh > 0 && atomicAdd(S + 1, 0) < nh) { const int h = atomicAdd(S + 1, 1); if (h < nh) got = h; }   // main queue empty: a hard rank may be left
      s_item = got;
      s_sm[0] = sm_id; s_sm[1] = hard;
    }
    __syncthreads();
    item = s_item;
  }
  if (!SCHED || item < p.B) {   // SCHED launches a few CTAs more than ranks: a CTA that wakes up to empty queues just leaves
  const int b = p.order ? p.order[item] : item;
  const int slot = p.slot0 + b;

  // ---- phase 0: stage the per-problem record (coalesced 4-byte loads, every byte requested
  // once: the record may live in page-locked HOST memory, see cmpc_solve_host) --------------
  for (int i = tid; i < 13; i += THREADS) s_x0[i] = __ldg(p.x0 + (size_t)b * 13 + i);
  for (int i = tid; i < NX; i += THREADS) s_xd[i] = __ldg(p.x_des + (size_t)b * NX + i);
  for (int i = tid; i < 3 * NLEG; i += THREADS) s_r[i] = __ldg(p.r + (size_t)b * 3 * NLEG + i);
  for (int i = tid; i < N; i += THREADS) s_mask[i] = (int)__ldg(p.mask + (size_t)b * N + i);
  for (int i = tid; i < NWP; i += THREADS) { s_s[i] = 0.f; s_v[i] = 0.f; s_h[i] = 0.f; s_S[i] = 0.f; }
  if constexpr (BODY) {
    if (tid < kBodyF4) reinterpret_cast<float4*>(s_x0 + 16)[tid] = __ldg(p.body + (size_t)slot * kBodyF4 + tid);
  }
  // the slot's force weight, read from shared memory where it is used (a register through the ADMM loop
  // would cost the N = 10 kernels a spill)
  if constexpr (WEIGHTS) {
    if (tid == 0) s_x0[13] = 2.f * slot_weight(p, slot, 13);
  }
  const float mu = __ldg(p.mu + b);
  // issue every other global load of this problem now so that their DRAM latencies overlap
  const bool is_leg = tid < NLEG;
  float wx_in[3] = {0.f, 0.f, 0.f};
  float wy_in[3] = {0.f, 0.f, 0.f};
  const bool warm = p.warm_mode != 0 && p.warm_valid[slot] != 0;
  if (is_leg) {
    if (warm) {
      const float* wx = p.warm_x + ((size_t)slot * NLEG + tid) * 3;
      wx_in[0] = wx[0]; wx_in[1] = wx[1]; wx_in[2] = wx[2];
      if (p.warm_mode == 2) {
        const float* wy = p.warm_y + ((size_t)slot * NLEG + tid) * 3;
        wy_in[0] = wy[0]; wy_in[1] = wy[1]; wy_in[2] = wy[2];
      }
    }
  }
  float4 fr_in = make_float4(0.f, 0.f, 0.f, 0.f);   // FORCE: this leg-stage's {f_ref, w_f}
  if constexpr (FORCE) {
    if (is_leg) fr_in = __ldg(p.force + (size_t)slot * NLEG + tid);
    if (tid == 0) s_x0[14] = fr_in.w;
  }
  __syncthreads();

  // Factorisation cache: P depends on the lever arms, the contact masks, the yaw and rho only.
  // When none of them moved (a standing robot, or any stretch with a static contact schedule),
  // the cached -P^-1 is reused as is: the iteration is in residual-correction form, so an
  // inexact K^-1 changes the convergence rate but not the fixed point or the stopping test.
  bool reuse = false;
  const size_t cslot = (size_t)slot;
  if (CACHE && p.cache_pinv) {
    const float* meta = p.cache_meta + cslot * 4;
    bool ok = meta[2] != 0.f && meta[0] == p.rho && fabsf(meta[1] - s_x0[2]) <= p.cache_tol_yaw;
    for (int i = tid; i < 3 * NLEG; i += THREADS)
      ok = ok && fabsf(s_r[i] - p.cache_r[cslot * 3 * NLEG + i]) <= p.cache_tol_r;
    for (int i = tid; i < N; i += THREADS) ok = ok && s_mask[i] == (int)p.cache_mask[cslot * N + i];
    reuse = __syncthreads_and(ok) != 0;
    if (tid == 0) { p.cache_meta[cslot * 4 + 3] = reuse ? 1.f : 0.f; p.cache_hit[slot] = reuse ? 1 : 0; }
  }
  bool cached_fresh = false;          // this launch stored a new factorisation of the CURRENT data
  bool used_cache = false;            // the iteration runs on a reused (possibly slightly stale) factor

  float sn, cs;
  sincosf(s_x0[2], &sn, &cs);
  const float im = BODY ? s_x0[16] : p.inv_mass;
  const float alpha = p.alpha;
  float rho = p.rho;
  float rho_inv = 1.f / rho;

  // ---- phase 1: leg geometry, linear term -----------------------------------------------
  const int lj = tid >> 2, ll = tid & 3;            // stage, leg of a leg thread
  bool stance = false;
  float Gh[3][3];
  float dinv = 0.f;                                  // d = 1/(sigma + 2 r_weight + rho), 0 on swing legs
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int k = 0; k < 3; ++k) Gh[a][k] = 0.f;
  if (is_leg) {
    stance = (s_mask[lj] >> ll) & 1;
    if constexpr (BODY) leg_map_full(cs, sn, s_x0 + 17, s_r[3 * tid], s_r[3 * tid + 1], s_r[3 * tid + 2], Gh);
    else leg_map(cs, sn, p.ib, s_r[3 * tid], s_r[3 * tid + 1], s_r[3 * tid + 2], Gh);
    if (!stance) {
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int k = 0; k < 3; ++k) Gh[a][k] = 0.f;
    }
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int k = 0; k < 3; ++k) s_G[tid][3 * a + k] = Gh[a][k];
    s_G[tid][11] = stance ? 1.f : 0.f;
  }
  if constexpr (FORCE) {   // swing leg-stages ignore their entries
    const float w2 = 2.f * fr_in.w;
    s_fr[tid] = stance ? make_float4(-w2 * fr_in.x, -w2 * fr_in.y, -w2 * fr_in.z, w2) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const bool is_row = tid < G_::ROWT;
  const int rs = SPLIT == 1 ? 0 : tid / NWR;         // slice-major layout: column slice,
  const int rp = tid - rs * NWR;                     // first row (rows rp + q NWR, q < R)
  const int rj0 = rp / 6, ra = rp % 6;               // stage of the first row, axis of all R rows
  const int n_eff = p.n_eff > 0 ? p.n_eff : N;
  {
    // linear term h in two steps: the 6N stage errors once (one (k, a) per thread), then the
    // suffix sums over k > j - the same terms in the same order as wrench_linear_term(), in double
    double* e_pos = &s_e[0][0];           // [N][6]
    double* e_vel = &s_e[1][0];
    for (int i = tid; i < NW; i += THREADS) {
      double ep = 0.0, ev = 0.0;
      if (i / 6 + 1 <= n_eff) stage_error(i / 6 + 1, i % 6, s_x0, s_xd, cs, sn, p.dt, ep, ev);
      e_pos[i] = ep;
      e_vel[i] = ev;
    }
    __syncthreads();
    for (int i = tid; i < NW; i += THREADS) {
      const int j = i / 6, a = i % 6;
      const double dt = p.dt;
      double acc = 0.0;
      if constexpr (STAGE) {   // stage k's weights: row k - 1 of the slot's table
        const float* ws = reinterpret_cast<const float*>(p.wstage + (size_t)slot * N * kStageF4);
        for (int k = j + 1; k <= N; ++k) {
          const double wp = __ldg(ws + 12 * (k - 1) + a), wv = __ldg(ws + 12 * (k - 1) + 6 + a);
          acc += 2.0 * (wp * dt * dt * (double)(k - 1 - j) * e_pos[6 * (k - 1) + a] + wv * dt * e_vel[6 * (k - 1) + a]);
        }
      } else {
        double wp, wv;
        if constexpr (WEIGHTS) {
          wp = slot_weight(p, slot, a);
          wv = slot_weight(p, slot, 6 + a);
        } else {
          wp = p.w[a];
          wv = p.w[6 + a];
        }
        for (int k = j + 1; k <= N; ++k)
          acc += 2.0 * (wp * dt * dt * (double)(k - 1 - j) * e_pos[6 * (k - 1) + a] + wv * dt * e_vel[6 * (k - 1) + a]);
      }
      s_h[i] = (float)acc;
    }
  }
  __syncthreads();

  // ---- phases 2+3 as a re-runnable step (adaptive rho refactorises) ------------------------
  float row[R][COLS];
  constexpr int TILE4 = R * COLS / 4;                   // 16-byte pieces of a thread's tile
  auto factorize = [&]() {
  // d of this leg for the current rho (K = H + (sigma + rho) I on the stance forces)
  if constexpr (FORCE) dinv = stance ? 1.f / (p.sigma + (s_x0[13] + s_fr[tid].w) + rho) : 0.f;
  else if constexpr (WEIGHTS) dinv = stance ? 1.f / (p.sigma + s_x0[13] + rho) : 0.f;
  else dinv = stance ? 1.f / (p.sigma + 2.f * p.r_weight + rho) : 0.f;
  if (is_leg) s_G[tid][9] = dinv;
  __syncthreads();
  if (reuse) {                                          // CTA-uniform; only the first call can hit
    reuse = false;
    used_cache = true;
    if (is_row) {
      const float4* src = p.cache_pinv + cslot * TILE4 * G_::ROWT + tid;
#pragma unroll
      for (int q = 0; q < R; ++q)
#pragma unroll
        for (int c = 0; c < COLS; c += 4) {
          const float4 v = __ldg(src + (size_t)((q * COLS + c) / 4) * G_::ROWT);
          row[q][c] = v.x; row[q][c + 1] = v.y; row[q][c + 2] = v.z; row[q][c + 3] = v.w;
        }
    }
    return;
  }
  used_cache = false;   // from here on the factor is a fresh one of the current data
  // ---- phase 2: P = M^-1 + E (R x COLS register tiles) -------------------------------------
  // E_j[ra][a'] = sum_l sum_c Gp[ra][c] d Gp[a'][c],  Gp = [Ghat ; I/m]
  float E[R][6];
  float sc[R], diag[R], rdiag[R];
  const float* mi[R];
#pragma unroll
  for (int q = 0; q < R; ++q) {
    const int rj = rj0 + q * (N / R);
    if constexpr (WEIGHTS)
      mi[q] = p.w_Minv + (size_t)slot * 6 * N * N + ((size_t)(is_row ? ra : 0) * N + (is_row ? rj : 0)) * N;
    else
      mi[q] = p.Minv + ((size_t)(is_row ? ra : 0) * N + (is_row ? rj : 0)) * N;
#pragma unroll
    for (int a2 = 0; a2 < 6; ++a2) E[q][a2] = 0.f;
    sc[q] = 1.f; diag[q] = 1.f; rdiag[q] = 1.f;
    if (is_row) {
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        const float* g = s_G[4 * rj + l];
        const float d = g[9];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float mine = (ra < 3 ? g[3 * ra + c] : (ra - 3 == c ? im : 0.f)) * d;
#pragma unroll
          for (int a2 = 0; a2 < 3; ++a2) E[q][a2] += mine * g[3 * a2 + c];
          E[q][3 + c] += mine * im;
        }
      }
      // Jacobi scaling: the sweep runs on S P S (unit diagonal, pivots <= 1); its fused special
      // cases lose log2(pivot) bits when pivots are >> 1
      const float pii = __ldg(mi[q] + rj) + pick6(E[q], ra);
      sc[q] = rsqrtf(pii);
      diag[q] = pii * sc[q] * sc[q];
      rdiag[q] = __fdividef(1.f, diag[q]);
      if (rs == 0) s_S[rp + q * NWR] = sc[q];
    }
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < R; ++q)
#pragma unroll
    for (int c = 0; c < COLS; ++c) row[q][c] = 0.f;
  if (is_row) {
    // column of tile entry c: col = rs COLS + c = 6 j2 + a2, with j2, a2 advanced from those
    // of the slice start by compile-time steps (no runtime division per entry)
    const int bj = (rs * COLS) / 6, ba = (rs * COLS) % 6;
#pragma unroll
    for (int q = 0; q < R; ++q) {
      const int rj = rj0 + q * (N / R);
#pragma unroll
      for (int c = 0; c < COLS; ++c) {
        const int col = rs * COLS + c;
        int a2 = ba + c % 6, j2 = bj + c / 6;
        if (a2 >= 6) { a2 -= 6; ++j2; }
        float v = 0.f;
        if (col < NW) {
          if (a2 == ra) v = __ldg(mi[q] + j2);
          if (j2 == rj) v += pick6(E[q], a2);
          v *= sc[q] * s_S[col];
        }
        row[q][c] = v;
      }
    }
  }
  // Scheduling fence between the tile build and the sweep: without it the compiler interleaves the two and
  // the N = 10 kernel is 3.7 % slower on B200 (0.2314 against 0.2232 ms per 4096-problem batch).
  asm volatile("" ::: "memory");

  // ---- phase 3: symmetric Gauss-Jordan sweep, rows in registers -> row = -P^-1 ------------
  // Step k: the owners of row k (one thread per column slice) publish it through shared memory
  // with entry k replaced by a_kk - 1, plus d = 1/a_kk.  EVERY thread then runs the same FMA
  // stream on each of its rows
  //     row[c] += nf * p'[c],   nf = -a_ik d  (other rows),   nf = d - 1  (the pivot row itself)
  // which yields a_ic - a_ik a_kc / a_kk, a_ik / a_kk in column k, and d * p' for the pivot row.
  // Only the pivot row's own diagonal comes out as 2 - d instead of -d; the true diagonal of
  // every row is therefore tracked in a register (`diag`, also the next pivot) and the constant
  // +2 on the in-row copy is removed once at the end.  No divergent special-case path, no
  // dynamic register indexing (the pivot loop is split by the row slot q0 that holds the pivot).
  // The owners of the NEXT pivot row store it while they update it (one predicated 16-byte
  // store after every 4R FMAs) instead of after the update: a barrier waits for the stores in
  // flight to drain, and 15 back-to-back stores of one lane in front of it cost more than the
  // update itself (measured: 410 cycles per pivot on an otherwise idle SM).
  if constexpr (TC) {
    tc_sweep<NW, COLS>(row[0], s_P, tid);      // row = -(S P S)^-1
  } else {
    auto publish_tail = [&](float* nbuf, int kn, float dg, float rdg) {
      if (kn / COLS == rs) {   // this slice holds the pivot (stores of one thread stay ordered)
        nbuf[kn] = dg - 1.f;
        nbuf[NWP] = rdg;
      }
    };
    auto sweep_step = [&](auto q0c, auto qnc, auto parc, int kk, int kn_local, bool has_next) {
      constexpr int q0 = decltype(q0c)::value, qn = decltype(qnc)::value;
      constexpr bool odd = decltype(parc)::value != 0;     // pivot parity picks the buffer statically
      const float* buf = odd ? s_rowB : s_rowA;
      float* nbuf = odd ? s_rowA : s_rowB;
      if (is_row) {
        const float d = buf[NWP];
        float nf[R];
  #pragma unroll
        for (int q = 0; q < R; ++q) {
          const float m = buf[rp + q * NWR];
          const bool own = q == q0 && rp == kk;
          nf[q] = own ? d - 1.f : -m * d;
          diag[q] = own ? -d : fmaf(nf[q], m, diag[q]);
          rdiag[q] = __fdividef(1.f, diag[q]);
        }
        const bool pub = has_next && rp == kn_local;
        const float* pr = buf + rs * COLS;
  #pragma unroll
        for (int c = 0; c < COLS; c += 4) {
          const float4 pv = *reinterpret_cast<const float4*>(pr + c);
  #pragma unroll
          for (int q = 0; q < R; ++q) {
            // packed fp32 FMA (sm_100 FFMA2): two row entries per instruction
            const float2 nn = make_float2(nf[q], nf[q]);
            const float2 lo = __ffma2_rn(nn, make_float2(pv.x, pv.y), make_float2(row[q][c], row[q][c + 1]));
            const float2 hi = __ffma2_rn(nn, make_float2(pv.z, pv.w), make_float2(row[q][c + 2], row[q][c + 3]));
            row[q][c] = lo.x; row[q][c + 1] = lo.y; row[q][c + 2] = hi.x; row[q][c + 3] = hi.y;
          }
          if (pub)
            *reinterpret_cast<float4*>(nbuf + rs * COLS + c) =
                make_float4(row[qn][c], row[qn][c + 1], row[qn][c + 2], row[qn][c + 3]);
        }
        if (pub) publish_tail(nbuf, qn * NWR + kn_local, diag[qn], rdiag[qn]);
      }
      __syncthreads();
    };
    if (is_row && rp == 0) {   // pivot 0
  #pragma unroll
      for (int c = 0; c < COLS; c += 4)
        *reinterpret_cast<float4*>(s_rowA + rs * COLS + c) = make_float4(row[0][c], row[0][c + 1], row[0][c + 2], row[0][c + 3]);
      publish_tail(s_rowA, 0, diag[0], rdiag[0]);
    }
    __syncthreads();
    {
      static_assert(NWR % 2 == 0, "pivots are processed in (even, odd) pairs");
      using I0 = std::integral_constant<int, 0>;
      using I1 = std::integral_constant<int, 1>;
      auto blocks = [&](auto self, auto q0c) -> void {
        constexpr int q0 = decltype(q0c)::value;
        constexpr int qn = q0 + 1 < R ? q0 + 1 : q0;
        for (int kk = 0; kk + 2 < NWR; kk += 2) {
          sweep_step(q0c, q0c, I0{}, kk, kk + 1, true);
          sweep_step(q0c, q0c, I1{}, kk + 1, kk + 2, true);
        }
        sweep_step(q0c, q0c, I0{}, NWR - 2, NWR - 1, true);
        sweep_step(q0c, std::integral_constant<int, qn>{}, I1{}, NWR - 1, 0, q0 + 1 < R);
        if constexpr (q0 + 1 < R) self(self, std::integral_constant<int, q0 + 1>{});
      };
      blocks(blocks, I0{});
    }
  }
  if (is_row) {   // remove the +2 of the in-row diagonal copy, undo the Jacobi scaling
#pragma unroll
    for (int q = 0; q < R; ++q)
#pragma unroll
      for (int c = 0; c < COLS; ++c) {
        const int col = rs * COLS + c;
        const float v = (!TC && col == rp + q * NWR) ? diag[q] : row[q][c];
        row[q][c] = v * sc[q] * (col < NW ? s_S[col] : 0.f);
      }
    if (CACHE && p.cache_pinv) {
      float4* dst = p.cache_pinv + cslot * TILE4 * G_::ROWT + tid;
#pragma unroll
      for (int q = 0; q < R; ++q)
#pragma unroll
        for (int c = 0; c < COLS; c += 4)
          dst[(size_t)((q * COLS + c) / 4) * G_::ROWT] = make_float4(row[q][c], row[q][c + 1], row[q][c + 2], row[q][c + 3]);
    }
  }
  if (CACHE && p.cache_pinv) {
    cached_fresh = true;
    if (tid == 0) p.cache_meta[cslot * 4] = rho;   // the cached factor belongs to this rho
  }
  __syncthreads();
  };
  factorize();

  // ---- phase 4: initial iterate -----------------------------------------------------------
  const float fmin = p.f_min, fmax = p.f_max;
  const float inv1 = 1.f / (1.f + mu * mu), inv2 = 1.f / (1.f + 2.f * mu * mu);
  LegContact lc{};
  bool bad_contact = false;          // a leg-stage of this slot was stored invalid (mu = NaN, set_contact_kernel)
  if constexpr (CONTACT) {
    if (is_leg) load_contact(p.contact + ((size_t)slot * NLEG + tid) * kContactF4, mu, lc);
    else lc = LegContact{{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}, mu, inv1, inv2, fmin, fmax};
    bad_contact = __syncthreads_or(!(lc.mu == lc.mu)) != 0;
  }
  // exact projection onto the friction frustum: minimise over fz the 1-D convex residual
  // (fx, fy are clamped to +-mu fz), three linear pieces, then clamp fz to [f_min, f_max]
  auto project = [&](float wx, float wy, float wz, float& zx, float& zy, float& zz) {
    if constexpr (CONTACT) {
      project_contact(lc, wx, wy, wz, zx, zy, zz);
    } else {
      const float ax = fabsf(wx), ay = fabsf(wy);
      const float big = fmaxf(ax, ay), small = fminf(ax, ay);
      const float f2 = (wz + mu * big) * inv1;
      const float f1 = (wz + mu * (ax + ay)) * inv2;
      float fz = (mu * wz >= big) ? wz : ((mu * f2 >= small) ? f2 : f1);
      fz = fminf(fmaxf(fz, fmin), fmax);
      const float lim = mu * fz;
      zx = fminf(fmaxf(wx, -lim), lim);
      zy = fminf(fmaxf(wy, -lim), lim);
      zz = fz;
    }
  };
  float x[3] = {0.f, 0.f, 0.f};
  float y[3] = {0.f, 0.f, 0.f};
  float z[3] = {0.f, 0.f, 0.f};
  float vh[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // v + h,  v = M G x  (wrench-space gradient)
  float glmax = 0.f;                               // max |G' h| of this leg (G' h itself lives in s_gl)
  auto init_iterate = [&]() {
#pragma unroll
    for (int a = 0; a < 6; ++a) vh[a] = 0.f;
    if (is_leg) {
      float gl[3] = {0.f, 0.f, 0.f};               // linear term of this leg:  G' h
      if (stance) {
#pragma unroll
        for (int a = 0; a < 6; ++a) vh[a] = s_h[6 * lj + a];     // h of this stage (v = 0 at x = 0)
#pragma unroll
        for (int k = 0; k < 3; ++k)
          gl[k] = Gh[0][k] * vh[0] + Gh[1][k] * vh[1] + Gh[2][k] * vh[2] + im * vh[3 + k];
        if constexpr (FORCE) {   // + -2 w_f f_ref: the whole linear term g of this force
          const float4 fr = s_fr[tid];
          gl[0] += fr.x; gl[1] += fr.y; gl[2] += fr.z;
        }
        x[0] = x[1] = x[2] = 0.f;
        y[0] = y[1] = y[2] = 0.f;
        if (warm) {
          x[0] = wx_in[0]; x[1] = wx_in[1]; x[2] = wx_in[2];
          y[0] = wy_in[0]; y[1] = wy_in[1]; y[2] = wy_in[2];
        }
        project(x[0], x[1], x[2], z[0], z[1], z[2]);
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) s_gl[3 * tid + k] = gl[k];   // only this thread reads it back
      glmax = fmaxf(fabsf(gl[0]), fmaxf(fabsf(gl[1]), fabsf(gl[2])));
    }
  };
  init_iterate();

  // exact wrench-space gradient  v = M (G x)  (uniform: every thread takes part)
  auto refresh_gradient = [&]() {
    if (leg_warp) {   // whole warps: every lane executes the shuffles (Gh = x = 0 on non-leg lanes)
      float wv[6];
#pragma unroll
      for (int a = 0; a < 3; ++a)
        wv[a] = quad_sum(Gh[a][0] * x[0] + Gh[a][1] * x[1] + Gh[a][2] * x[2]);
#pragma unroll
      for (int k = 0; k < 3; ++k) wv[3 + k] = quad_sum(x[k] * im);
      *reinterpret_cast<float2*>((is_leg && ll < 3) ? s_s + 6 * lj + 2 * ll : s_dump + 2 * tid) = pick_pair(wv, ll);
    }
    __syncthreads();
    for (int i = tid; i < NW; i += THREADS) {
      const int a_ = i % 6;
      const float* mg;
      if constexpr (WEIGHTS) mg = p.w_Mg + (size_t)slot * 6 * N * N + (size_t)(a_ * N + i / 6) * N;
      else mg = p.Mg + (size_t)(a_ * N + i / 6) * N;
      float acc = 0.f;
#pragma unroll
      for (int j2 = 0; j2 < N; ++j2) acc = fmaf(__ldg(mg + j2), s_s[6 * j2 + a_], acc);
      s_v[i] = acc;
    }
    __syncthreads();
    if (is_leg && stance) {
#pragma unroll
      for (int a = 0; a < 6; ++a) vh[a] = s_v[6 * lj + a] + s_h[6 * lj + a];
    }
    // no barrier here: s_v is next written by the next refresh, at least two barriers from now
  };
  if (warm) refresh_gradient();

  // constant part of the dual tolerance: ||G' h||_inf
  float ng = 0.f;
  {
    float m = glmax;
    if (leg_warp) {
      m = warp_max_nonneg(m);
      if (lane == 0) s_red[1][warp][0] = m;
    }
    __syncthreads();
#pragma unroll
    for (int wv = 0; wv < LWARPS; ++wv) ng = fmaxf(ng, s_red[1][wv][0]);
    __syncthreads();
  }

  // ---- phase 5: ADMM ------------------------------------------------------------------------
  int it = 0;
  int status = 0;
  float pri = 0.f, dua = 0.f;
  const float two_rw = 2.f * p.r_weight;   // WEIGHTS: s_x0[13]
  int rho_updates = 0;
  int next_chk = 0;
  int next_ref = p.refresh_every > 0 ? p.refresh_every : -1;
  int next_adp = p.adaptive_rho_interval > 0 ? p.adaptive_rho_interval : -1;
  for (;;) {
    if (it == next_ref) {
      next_ref += p.refresh_every;
      refresh_gradient();
    }
    const bool adapt_now = it == next_adp;
    if (adapt_now) next_adp += p.adaptive_rho_interval;
    const bool chk = it == next_chk || it >= p.max_iter || adapt_now;
    if (it == next_chk) next_chk += p.check_every;
    // leg phase A: residuals of the current iterate, rhs of the correction equation
    float t[3] = {0.f, 0.f, 0.f};
    float st_[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    if (leg_warp) {   // whole warps (all-zero state on non-leg lanes) so the shuffles are convergent
      float gr[3], rp[3];
      float trw = two_rw;
      if constexpr (WEIGHTS) trw = s_x0[13];
      float fl[3] = {0.f, 0.f, 0.f};
      if constexpr (FORCE) {   // (2 r_weight + 2 w_f) x - 2 w_f f_ref; a zero weight adds exact zeros
        const float4 fr = s_fr[tid];
        trw += fr.w;
        fl[0] = fr.x; fl[1] = fr.y; fl[2] = fr.z;
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        // (H x + g)_k = G'(v + h) + 2 r_weight x
        gr[k] = Gh[0][k] * vh[0] + Gh[1][k] * vh[1] + Gh[2][k] * vh[2] + im * vh[3 + k] + trw * x[k];
        if constexpr (FORCE) gr[k] += fl[k];
        rp[k] = x[k] - z[k];
        // K dlt = -(Hx + g + y) - rho (x - z)
        t[k] = -dinv * (gr[k] + y[k] + rho * rp[k]);
      }
      float sv[6];
#pragma unroll
      for (int a = 0; a < 3; ++a)
        sv[a] = quad_sum(Gh[a][0] * t[0] + Gh[a][1] * t[1] + Gh[a][2] * t[2]);
#pragma unroll
      for (int k = 0; k < 3; ++k) sv[3 + k] = quad_sum(t[k] * im);
      // every lane stores (no branch on the critical path): lanes without a pair hit the scratch row
      *reinterpret_cast<float2*>((is_leg && ll < 3) ? s_s + 6 * lj + 2 * ll : s_dump + 2 * tid) = pick_pair(sv, ll);
      if (chk) {
        float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, sum = 0.f;
        if (stance) {
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            const float rd = gr[k] + y[k];
            m0 = fmaxf(m0, fabsf(rp[k]));                                   // primal residual
            m1 = fmaxf(m1, fabsf(rd));                                      // dual residual
            m2 = fmaxf(m2, fmaxf(fabsf(x[k]), fabsf(z[k])));                // max(|x|,|z|)
            m3 = fmaxf(m3, fmaxf(fabsf(gr[k] - s_gl[3 * tid + k]), fabsf(y[k])));       // max(|Hx|,|y|)
            sum += x[k] + rd;
          }
        }
        st_[0] = m0; st_[1] = m1; st_[2] = m2; st_[3] = m3;
        st_[4] = fabsf(sum * 0.f);      // NaN / Inf guard: any non-finite value makes this NaN
#pragma unroll
        for (int k = 0; k < 5; ++k) {
          const float m = warp_max_nonneg(st_[k]);
          if (lane == 0) s_red[0][warp][k] = m;
        }
      }
    }
    __syncthreads();
    if (chk) {
      float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, m4 = 0.f;
#pragma unroll
      for (int wv = 0; wv < LWARPS; ++wv) {
        m0 = fmaxf(m0, s_red[0][wv][0]);
        m1 = fmaxf(m1, s_red[0][wv][1]);
        m2 = fmaxf(m2, s_red[0][wv][2]);
        m3 = fmaxf(m3, s_red[0][wv][3]);
        m4 += s_red[0][wv][4];
      }
      pri = m0;
      dua = m1;
      const float eps_p = p.eps_abs + p.eps_rel * m2;
      const float eps_d = p.eps_abs + p.eps_rel * fmaxf(m3, ng);
      // an invalid body (1/m = NaN, see set_body_kernel), contact or weight set (r_weight = NaN, see
      // set_weights_kernel) fails the problem also when no stance force carries it
      // or force reference (w_f = NaN, see set_force_ref_kernel)
      const bool nonfinite = !(m4 == 0.f) || !(m0 == m0) || !(m1 == m1) || (BODY && !(im == im)) ||
                             (CONTACT && bad_contact) || (WEIGHTS && !(s_x0[13] == s_x0[13])) ||
                             (FORCE && !(s_x0[14] == s_x0[14]));
      const bool converged = pri <= eps_p && dua <= eps_d;
      // a reused factor that is too stale for this problem (slow or blown up): factorise the
      // current data and go on.  Shares the one in-loop factorize() call with the rho adaptation.
      const bool stale = used_cache && !converged && (nonfinite || it >= p.cache_max_iter);
      bool refactor = stale;
      if (stale) {
        used_cache = false;
        if (nonfinite) {                       // restart from the cold iterate: x = y = 0, v = 0
#pragma unroll
          for (int k = 0; k < 3; ++k) { x[k] = 0.f; y[k] = 0.f; z[k] = 0.f; }
          if (is_leg && stance) project(0.f, 0.f, 0.f, z[0], z[1], z[2]);
#pragma unroll
          for (int a = 0; a < 6; ++a) vh[a] = (is_leg && stance) ? s_h[6 * lj + a] : 0.f;
        }
      } else {
        if (nonfinite) { status = -1; break; }
        if (converged) { status = 1; break; }
        if (it >= p.max_iter) { status = 0; break; }
        if (adapt_now) {
          // OSQP's rho adaptation: balance the normalised primal and dual residuals
          const float pr_n = m0 / (m2 + 1e-10f);
          const float du_n = m1 / (fmaxf(m3, ng) + 1e-10f);
          float rn = rho * sqrtf(pr_n / (du_n + 1e-10f));
          rn = fminf(fmaxf(rn, p.rho_min), p.rho_max);
          if (fmaxf(pr_n, du_n) > kRhoAdaptFloor &&
            (rn > rho * p.adaptive_rho_tolerance || rn * p.adaptive_rho_tolerance < rho)) {
            rho = rn;
            rho_inv = 1.f / rho;
            ++rho_updates;
            refactor = true;
          }
        }
      }
      if (refactor) {
        factorize();     // uniform: every thread of the CTA sees the same statistics
        continue;        // redo phase A of this iterate with the new factor
      }
    }
    // wrench phase: q = P^-1 s   (row holds -P^-1); each slice publishes its partial sum
    if (is_row) {
      float acc[R][4];
#pragma unroll
      for (int q = 0; q < R; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
      const float* sp = s_s + rs * COLS;
#pragma unroll
      for (int c = 0; c < COLS; c += 4) {
        const float4 sv4 = *reinterpret_cast<const float4*>(sp + c);
#pragma unroll
        for (int q = 0; q < R; ++q) {
          const float2 lo = __ffma2_rn(make_float2(row[q][c], row[q][c + 1]), make_float2(sv4.x, sv4.y), make_float2(acc[q][0], acc[q][1]));
          const float2 hi = __ffma2_rn(make_float2(row[q][c + 2], row[q][c + 3]), make_float2(sv4.z, sv4.w), make_float2(acc[q][2], acc[q][3]));
          acc[q][0] = lo.x; acc[q][1] = lo.y; acc[q][2] = hi.x; acc[q][3] = hi.y;
        }
      }
#pragma unroll
      for (int q = 0; q < R; ++q)
        s_q[rs][rp + q * NWR] = -((acc[q][0] + acc[q][1]) + (acc[q][2] + acc[q][3]));
    }
    __syncthreads();
    // leg phase B: x-update, relaxed projection, dual update.  Whole leg warps run it without a
    // divergent branch: swing legs and padding lanes carry zero state (d = 0, G = 0), so the same
    // instruction stream leaves their x and y at 0; only z is masked after the projection.
    if (leg_warp) {
      const int lq = is_leg ? 6 * lj : 0;
      float qv[6];
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        float acc = s_q[0][lq + a];
#pragma unroll
        for (int sl = 1; sl < SPLIT; ++sl) acc += s_q[sl][lq + a];
        qv[a] = acc;
      }
#pragma unroll
      for (int a = 0; a < 6; ++a) vh[a] = fmaf(alpha, qv[a], vh[a]);
      float w3[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float dl = t[k] - dinv * (Gh[0][k] * qv[0] + Gh[1][k] * qv[1] + Gh[2][k] * qv[2] + im * qv[3 + k]);
        const float xt = x[k] + dl;
        x[k] = fmaf(alpha, dl, x[k]);      // OSQP: x <- alpha x~ + (1 - alpha) x
        const float zh = alpha * xt + (1.f - alpha) * z[k];
        w3[k] = fmaf(y[k], rho_inv, zh);
      }
      project(w3[0], w3[1], w3[2], z[0], z[1], z[2]);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        z[k] = stance ? z[k] : 0.f;
        y[k] = rho * (w3[k] - z[k]);
      }
    }
    ++it;
  }
  (void)rho_updates;

  // ---- phase 6: outputs -----------------------------------------------------------------------
  if (is_leg) {
    s_xd[3 * tid] = x[0]; s_xd[3 * tid + 1] = x[1]; s_xd[3 * tid + 2] = x[2];   // staged, stored below
    float* wx = p.warm_x + ((size_t)slot * NLEG + tid) * 3;
    wx[0] = x[0]; wx[1] = x[1]; wx[2] = x[2];
    float* wy = p.warm_y + ((size_t)slot * NLEG + tid) * 3;
    wy[0] = y[0]; wy[1] = y[1]; wy[2] = y[2];
  }
  if (CACHE && p.cache_pinv) {
    if (cached_fresh) {
      for (int i = tid; i < 3 * NLEG; i += THREADS) p.cache_r[cslot * 3 * NLEG + i] = s_r[i];
      for (int i = tid; i < N; i += THREADS) p.cache_mask[cslot * N + i] = (uint8_t)s_mask[i];
    }
    if (tid == 0) {
      float* meta = p.cache_meta + cslot * 4;
      if (cached_fresh) meta[1] = s_x0[2];
      // keep the entry only for healthy solves: a slow or failed one refactorises next time
      const bool keep = status == 1 && it <= p.cache_max_iter && (cached_fresh || meta[2] != 0.f);
      meta[2] = keep ? 1.f : 0.f;
    }
  }
  if (tid == 0) {
    if (p.iters) p.iters[b] = it;
    if (p.pri_res) p.pri_res[b] = pri;
    if (p.dua_res) p.dua_res[b] = dua;
    if (p.status) p.status[b] = status;
    p.warm_valid[slot] = status >= 0 ? 1 : 0;
  }
  __syncthreads();
  for (int i = tid; i < 3 * NLEG; i += THREADS) p.U[(size_t)b * 3 * NLEG + i] = s_xd[i];
  if (p.X) {
    // predicted states X = free response + forced response of the wrench sequence w = G x
    __syncthreads();
    if (leg_warp) {
      float wv[6];
#pragma unroll
      for (int a = 0; a < 3; ++a)
        wv[a] = quad_sum(Gh[a][0] * x[0] + Gh[a][1] * x[1] + Gh[a][2] * x[2]);
#pragma unroll
      for (int k = 0; k < 3; ++k) wv[3 + k] = quad_sum(x[k] * im);
      if (is_leg && ll < 3)
        *reinterpret_cast<float2*>(s_s + 6 * lj + 2 * ll) = pick_pair(wv, ll);
    }
    __syncthreads();
    // prefix sums of the wrench sequence per axis: c1[k] = sum_{j<k} w_j, c2[k] = sum_{j<k} (k-1-j) w_j
    // (6 threads, serial in k: measured faster than one (axis, k) pair per thread)
    float* c1 = &s_pre[0][0];            // [6][N+1]
    float* c2 = &s_pre[1][0];
    if (tid < 6) {
      float a1 = 0.f, a2 = 0.f;
      c1[tid * (N + 1)] = 0.f;
      c2[tid * (N + 1)] = 0.f;
      for (int k = 1; k <= N; ++k) {
        a2 += a1;
        a1 += s_s[6 * (k - 1) + tid];
        c1[tid * (N + 1) + k] = a1;
        c2[tid * (N + 1) + k] = a2;
      }
    }
    __syncthreads();
    const float dt = p.dt, g = s_x0[12];
    for (int o = tid; o < NX; o += THREADS) {
      const int k = o / 13, cidx = o % 13;
      const float kf = (float)k;
      float val;
      if (cidx == 12) {
        val = g;
      } else if (cidx < 3) {           // Theta_k = Theta_0 + k d Rz w0 + d^2 sum (k-1-j) tau^_j
        const float rw0 = cidx == 0 ? (cs * s_x0[6] - sn * s_x0[7])
                                    : (cidx == 1 ? (sn * s_x0[6] + cs * s_x0[7]) : s_x0[8]);
        val = s_x0[cidx] + kf * dt * rw0 + dt * dt * c2[cidx * (N + 1) + k];
      } else if (cidx < 6) {           // p_k
        const int aa = cidx - 3;
        val = s_x0[cidx] + kf * dt * s_x0[9 + aa] + dt * dt * c2[(3 + aa) * (N + 1) + k];
        if (aa == 2) val += 0.5f * kf * (kf - 1.f) * dt * dt * g;
      } else if (cidx < 9) {           // omega_k = omega_0 + d Rz' sum tau^_j
        const float sx = c1[k], sy = c1[(N + 1) + k], sz = c1[2 * (N + 1) + k];
        const int aa = cidx - 6;
        const float rot = aa == 0 ? (cs * sx + sn * sy) : (aa == 1 ? (-sn * sx + cs * sy) : sz);
        val = s_x0[cidx] + dt * rot;
      } else {                         // v_k
        const int aa = cidx - 9;
        val = s_x0[cidx] + dt * c1[(3 + aa) * (N + 1) + k];
        if (aa == 2) val += kf * dt * g;
      }
      p.X[(size_t)b * NX + o] = val;
    }
  }
  }
  if constexpr (SCHED) {
    if (tid == 0) {
      if (s_sm[1]) atomicSub(p.sched + 16 + 2 * kSchedSm + s_sm[0], 1);   // wakes this SM's sleepers when it was the last
      __threadfence();
      s_sm[1] = atomicAdd(p.sched + 2, 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    if (s_sm[1]) {   // the last CTA to leave zeroes the scheduling state for the next launch
      for (int i = tid; i < kSchedInts; i += THREADS) p.sched[i] = 0;
    }
  }
}

// Forced response of a known external wrench sequence (cmpc_set_wrench) at stage k: the offsets phi[12] it adds to
// Theta, p, omega, v of the free response of x0 (g is unchanged).  eps = the slot's record [n][6]: per stage the
// world-frame force F and torque tau about the CoM (stages >= n carry none).  The conventions are the solve kernels':
// yaw frozen at x0 (c, s from sincosf(x0[2])), the body {1/m = im, Ib^-1 row-major = ib}; stage j's wrench in wrench
// axes is Rz (Rz Ib^-1 Rz') tau (leg_map_full's map of [r]x f) and F / m; with the fp32 prefix sums
// c1[k] = sum_{j<k} of it and c2[k] = sum_{j<k} (k-1-j) of it, in the order of the kernels' X output:
//   Theta += d^2 c2_ang,  p += d^2 c2_lin,  omega += d Rz' c1_ang,  v += d c1_lin.
// The QP with the wrench is the QP without it on x_des - phi, and its X is that QP's X + phi (DESIGN.md section 4).
__device__ __forceinline__ void wrench_response(int k, int n, const float* eps, float c, float s, float dt, float im,
                                                const float* ib, float phi[12]) {
  float a1[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, a2[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int j = 0; j < k; ++j) {
#pragma unroll
    for (int a = 0; a < 6; ++a) a2[a] += a1[a];
    if (j >= n) continue;
    const float* e = eps + 6 * j;
    const float q0 = c * e[3] + s * e[4], q1 = -s * e[3] + c * e[4], q2 = e[5];   // Rz' tau
    float A[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) A[i] = ib[3 * i] * q0 + ib[3 * i + 1] * q1 + ib[3 * i + 2] * q2;
    const float T0 = c * A[0] - s * A[1], T1 = s * A[0] + c * A[1];
    a1[0] += c * T0 - s * T1;
    a1[1] += s * T0 + c * T1;
    a1[2] += A[2];
#pragma unroll
    for (int i = 0; i < 3; ++i) a1[3 + i] += e[i] * im;
  }
#pragma unroll
  for (int a = 0; a < 6; ++a) phi[a] = dt * dt * a2[a];
  phi[6] = dt * (c * a1[0] + s * a1[1]);
  phi[7] = dt * (-s * a1[0] + c * a1[1]);
  phi[8] = dt * a1[2];
#pragma unroll
  for (int i = 0; i < 3; ++i) phi[9 + i] = dt * a1[3 + i];
}

// Everything below is compiled once, in cmpc.cu; cmpc_body.cu needs only the solve kernels above.
#ifndef CMPC_SOLVE_KERNELS_ONLY

// ---------------------------------------------------------------------------------------
// Longest-processing-time-first launch order.  ADMM iteration counts vary by 20x inside a
// batch and one CTA owns one problem, so the kernel's makespan is set by where the slowest
// problems start.  A cheap conditioning score (mean diagonal of H = G'MG over the stance
// legs of the first and last stage, times their squared horizontal lever arms over mu)
// predicts them well (hard problems have 2-3x the score);
// problems are bucketed by quarter-octaves of the score and launched hardest first.
// ---------------------------------------------------------------------------------------
struct ScoreParams {
  const float* __restrict__ x0;
  const float* __restrict__ r;
  const uint8_t* __restrict__ mask;
  const float* __restrict__ Mg;
  const float* __restrict__ mu;
  float* __restrict__ score;
  int32_t* __restrict__ hist;   // [64], zeroed by the host before the launch
  int32_t B;
  float inv_mass;
  float ib[3];
  const float4* __restrict__ body;   // per-problem body [B][kBodyF4] (slots [slot0, slot0 + B)), or nullptr
  const float4* __restrict__ weights;   // per-problem weights [B][kWeightF4] (slots [slot0, slot0 + B)), or nullptr
  // per-problem stage weights [B][N][kStageF4] (slots [slot0, slot0 + B)), or nullptr; replace weights' state weights
  const float4* __restrict__ wstage;
  float dt;
  int32_t n_eff;                        // stages of the user horizon (<= N; the rest is padding)
};

__device__ __forceinline__ int score_bucket(float s) {
  const float l = log2f(fmaxf(s, 1e-6f));
  int q = (int)((l + 10.f) * 4.f);
  return q < 0 ? 0 : (q > 63 ? 63 : q);
}

// Mean over the stance legs of the first and last stage of the squared horizontal lever arm, over mu.  Measured
// on the iteration counts of configs 2 / 3 (profiles/r02_lpt_score_study.txt), for the product with the mean
// diagonal of H (the score): 93 / 72 of the 96 hardest of 3000 problems in the first 384 ranks against
// 83 / 59 for the mean diagonal of H alone, and no 235-iteration problem among the last ranks of a mixed-gait
// batch (the lever arms alone find the hard problems as well but rank the easy ones worse).
template <int N>
__device__ __forceinline__ float problem_score_arms(const ScoreParams& p, int b) {
  float acc = 0.f;
  int cnt = 0;
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int j = e == 0 ? 0 : N - 1;
    const int m = __ldg(p.mask + (size_t)b * N + j);
    const float4* rq = reinterpret_cast<const float4*>(p.r + ((size_t)b * N + j) * 12);
    const float4 q0 = __ldg(rq), q1 = __ldg(rq + 1), q2 = __ldg(rq + 2);
    const float rr[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
#pragma unroll
    for (int l = 0; l < 4; ++l)
      if ((m >> l) & 1) {
        acc += rr[3 * l] * rr[3 * l] + rr[3 * l + 1] * rr[3 * l + 1];
        ++cnt;
      }
  }
  return cnt ? acc / ((float)cnt * fmaxf(__ldg(p.mu + b), 1e-3f)) : 0.f;
}

template <int N>
__device__ __forceinline__ float problem_score(const ScoreParams& p, int b) {
  const float arms = problem_score_arms<N>(p, b);
  float sn, cs;
  sincosf(__ldg(p.x0 + (size_t)b * 13 + 2), &sn, &cs);
  float bd[4 * kBodyF4];
  if (p.body) {
#pragma unroll
    for (int i = 0; i < kBodyF4; ++i) {
      const float4 v = __ldg(p.body + (size_t)b * kBodyF4 + i);
      bd[4 * i] = v.x; bd[4 * i + 1] = v.y; bd[4 * i + 2] = v.z; bd[4 * i + 3] = v.w;
    }
  }
  const float im = p.body ? bd[0] : p.inv_mass;
  float acc = 0.f;
  int cnt = 0;
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int j = e == 0 ? 0 : N - 1;
    const int m = __ldg(p.mask + (size_t)b * N + j);
    float md[6];
    if (p.wstage) {
      // M_a[j][j] of the problem's stage weights, j = 0 or N - 1: 2 sum_{k>j} (w_pos,k dt^4 (k-1-j)^2 + w_vel,k dt^2)
      // (1 on the padding stages, as in the embedded tables)
      const float* ws = reinterpret_cast<const float*>(p.wstage + (size_t)b * N * kStageF4);
      const float d2 = p.dt * p.dt;
#pragma unroll
      for (int a = 0; a < 6; ++a) md[a] = 0.f;
      for (int k = j + 1; k <= p.n_eff; ++k) {
        const float m = (float)(k - 1 - j);
#pragma unroll
        for (int a = 0; a < 6; ++a) md[a] += 2.f * (__ldg(ws + 12 * (k - 1) + a) * d2 * d2 * m * m + __ldg(ws + 12 * (k - 1) + 6 + a) * d2);
      }
      if (j >= p.n_eff) {
#pragma unroll
        for (int a = 0; a < 6; ++a) md[a] = 1.f;
      }
    } else if (p.weights) {
      // M_a[j][j] of the problem's weights in closed form: 2 sum_{m<n} (w_pos dt^4 m^2 + w_vel dt^2), n = n_eff - j
      // stages (1 on the padding stages, as in the embedded tables)
      const float* wr = reinterpret_cast<const float*>(p.weights + (size_t)b * kWeightF4);
      const float n = (float)(p.n_eff - j), s2 = (n - 1.f) * n * (2.f * n - 1.f) / 6.f, d2 = p.dt * p.dt;
#pragma unroll
      for (int a = 0; a < 6; ++a)
        md[a] = j < p.n_eff ? 2.f * (__ldg(wr + a) * d2 * d2 * s2 + __ldg(wr + 6 + a) * d2 * n) : 1.f;
    } else {
#pragma unroll
      for (int a = 0; a < 6; ++a) md[a] = __ldg(p.Mg + ((size_t)a * N + j) * N + j);
    }
    // the stage's 12 lever-arm floats as three 16-byte loads (48 B records are 16-B aligned);
    // few, wide requests also when the batch is read in place from page-locked host memory
    const float4* rq = reinterpret_cast<const float4*>(p.r + ((size_t)b * N + j) * 12);
    const float4 q0 = __ldg(rq), q1 = __ldg(rq + 1), q2 = __ldg(rq + 2);
    const float rr[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      if (!((m >> l) & 1)) continue;
      float G[3][3];
      if (p.body) leg_map_full(cs, sn, bd + 1, rr[3 * l], rr[3 * l + 1], rr[3 * l + 2], G);
      else leg_map(cs, sn, p.ib, rr[3 * l], rr[3 * l + 1], rr[3 * l + 2], G);
#pragma unroll
      for (int c = 0; c < 3; ++c)
        acc += G[0][c] * G[0][c] * md[0] + G[1][c] * G[1][c] * md[1] + G[2][c] * G[2][c] * md[2] +
               im * im * md[3 + c];
      cnt += 3;
    }
  }
  return cnt ? arms * acc / (float)cnt : 0.f;
}

template <int N>
__global__ void __launch_bounds__(128) score_kernel(const ScoreParams p) {
  grid_dependency_wait();
  grid_launch_dependents();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  const float sc = problem_score<N>(p, b);
  p.score[b] = sc;
  atomicAdd(p.hist + score_bucket(sc), 1);
}

__global__ void __launch_bounds__(1024) order_kernel(const float* __restrict__ score,
                                                     int32_t* __restrict__ hist,
                                                     int32_t* __restrict__ order, int32_t B) {
  __shared__ int offs[64];
  grid_dependency_wait();
  grid_launch_dependents();
  if (threadIdx.x == 0) {       // descending exclusive scan: hardest bucket first
    int run = 0;
    for (int q = 63; q >= 0; --q) { offs[q] = run; run += hist[q]; hist[q] = 0; }  // re-armed
  }
  __syncthreads();
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const int pos = atomicAdd(&offs[score_bucket(score[b])], 1);
    order[pos] = b;
  }
}

// ---------------------------------------------------------------------------------------
// Dense condensed QP export: H [B,12N,12N], g [B,12N]  (parity / inspection path)
// grid = (B), block = 256
// ---------------------------------------------------------------------------------------
struct CondenseParams {
  const float* __restrict__ x0;
  const float* __restrict__ r;
  const uint8_t* __restrict__ mask;
  const float* __restrict__ x_des;
  float* __restrict__ H;
  float* __restrict__ g;
  const float* __restrict__ Mg;   // [6][N][N]
  int32_t B;
  float dt, inv_mass;
  float ib[3];
  float w[13];
  float r_weight;
  const float4* __restrict__ body;   // per-problem body [B][kBodyF4] (slots [0, B)), or nullptr
  // per-problem weights [B][kWeightF4] and their Gram tables M [B][6][N][N] (slots [0, B)), or nullptr
  const float4* __restrict__ weights;
  const float* __restrict__ w_Mg;
  const float* __restrict__ wrench;   // per-problem external wrench [B][N][6] (slots [0, B)), or nullptr
  const float4* __restrict__ force;   // per-problem force references [B][N][4] {f_ref, w_f} (slots [0, B)), or nullptr
  // per-problem stage weights [B][N][kStageF4] (slots [0, B)), or nullptr; replace weights' state weights in h (M is
  // w_Mg, built from them)
  const float4* __restrict__ wstage;
};

template <int N>
__global__ void __launch_bounds__(256) condense_kernel(const CondenseParams p) {
  constexpr int NLEG = 4 * N, NU = 12 * N, NX = 13 * (N + 1), NW = 6 * N;
  __shared__ float s_x0[16];
  __shared__ float s_xd[NX];
  __shared__ float s_Gp[NLEG][3][6];     // Gp' : per leg, per force component c, the 6 wrench rows
  __shared__ float s_h[NW];
  __shared__ float s_M[6][N][N];
  __shared__ float s_w[12 * N + 1];      // the state weights: one row (13), or one per stage (12 N)
  const int b = blockIdx.x, tid = threadIdx.x;
  if (b >= p.B) return;
  const float* wrec = p.weights ? reinterpret_cast<const float*>(p.weights + (size_t)b * kWeightF4) : nullptr;
  const float* Mg = wrec ? p.w_Mg + (size_t)b * 6 * N * N : p.Mg;
  const float* wst = p.wstage ? reinterpret_cast<const float*>(p.wstage + (size_t)b * N * kStageF4) : nullptr;
  const int ws = wst ? 12 : 0;
  for (int i = tid; i < 13; i += 256) s_x0[i] = __ldg(p.x0 + (size_t)b * 13 + i);
  if (wst) {
    for (int i = tid; i < 12 * N; i += 256) s_w[i] = __ldg(wst + i);
  } else {
    for (int i = tid; i < 13; i += 256) s_w[i] = wrec ? __ldg(wrec + i) : p.w[i];
  }
  for (int i = tid; i < NX; i += 256) s_xd[i] = __ldg(p.x_des + (size_t)b * NX + i);
  for (int i = tid; i < 6 * N * N; i += 256) (&s_M[0][0][0])[i] = __ldg(Mg + i);
  const float r_weight = wrec ? __ldg(wrec + 13) : p.r_weight;
  __syncthreads();
  float sn, cs;
  sincosf(s_x0[2], &sn, &cs);
  const float* bd = p.body ? reinterpret_cast<const float*>(p.body + (size_t)b * kBodyF4) : nullptr;
  const float im = bd ? __ldg(bd) : p.inv_mass;
  if (p.wrench) {   // the QP with the wrench is the QP on x_des - phi (wrench_response)
    if (tid <= N) {
      float ibw[9], phi[12];
      for (int i = 0; i < 9; ++i) ibw[i] = bd ? __ldg(bd + 1 + i) : (i % 4 == 0 ? p.ib[i / 4] : 0.f);
      wrench_response(tid, N, p.wrench + (size_t)b * 6 * N, cs, sn, p.dt, im, ibw, phi);
      for (int i = 0; i < 12; ++i) s_xd[13 * tid + i] -= phi[i];
    }
    __syncthreads();
  }
  for (int t = tid; t < NLEG; t += 256) {
    const int j = t >> 2, l = t & 3;
    const bool stance = (__ldg(p.mask + (size_t)b * N + j) >> l) & 1;
    const float* rp = p.r + ((size_t)b * NLEG + t) * 3;
    float Gh[3][3];
    if (bd) {
      float ib[9];
      for (int i = 0; i < 9; ++i) ib[i] = __ldg(bd + 1 + i);
      leg_map_full(cs, sn, ib, __ldg(rp), __ldg(rp + 1), __ldg(rp + 2), Gh);
    } else {
      leg_map(cs, sn, p.ib, __ldg(rp), __ldg(rp + 1), __ldg(rp + 2), Gh);
    }
    for (int c = 0; c < 3; ++c) {
      for (int a = 0; a < 3; ++a) s_Gp[t][c][a] = stance ? Gh[a][c] : 0.f;
      for (int a = 0; a < 3; ++a) s_Gp[t][c][3 + a] = (stance && a == c) ? im : 0.f;
    }
  }
  for (int i = tid; i < NW; i += 256)
    s_h[i] = wrench_linear_term<N>(i / 6, i % 6, s_x0, s_xd, cs, sn, s_w, ws, p.dt, N);
  __syncthreads();
  // the force reference of stance force u: w_f ||f - f_ref||^2 adds 2 w_f to H's diagonal and -2 w_f f_ref to g
  const float* fref = p.force ? reinterpret_cast<const float*>(p.force + (size_t)b * NLEG) : nullptr;
  // g = G' h
  for (int u = tid; u < NU; u += 256) {
    const int t = u / 3, c = u % 3, j = t >> 2;
    float acc = 0.f;
#pragma unroll
    for (int a = 0; a < 6; ++a) acc += s_Gp[t][c][a] * s_h[6 * j + a];
    if (fref && s_Gp[t][c][3 + c] != 0.f) acc += -2.f * __ldg(fref + 4 * t + 3) * __ldg(fref + 4 * t + c);
    p.g[(size_t)b * NU + u] = acc;
  }
  // H = G' M G  (+ 2 r_weight + 2 w_f on the diagonal of stance forces); float4 stores along rows
  float* Hb = p.H + (size_t)b * NU * NU;
  for (int e = tid; e < NU * (NU / 4); e += 256) {
    const int row = e / (NU / 4), c4 = (e % (NU / 4)) * 4;
    const int t1 = row / 3, c1 = row % 3, j1 = t1 >> 2;
    float out[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int col = c4 + q;
      const int t2 = col / 3, c2 = col % 3, j2 = t2 >> 2;
      float acc = 0.f;
#pragma unroll
      for (int a = 0; a < 6; ++a) acc += s_Gp[t1][c1][a] * s_M[a][j1][j2] * s_Gp[t2][c2][a];
      if (row == col && s_Gp[t1][c1][3 + c1] != 0.f) {
        acc += 2.f * r_weight;
        if (fref) acc += 2.f * __ldg(fref + 4 * t1 + 3);
      }
      out[q] = acc;
    }
    *reinterpret_cast<float4*>(Hb + (size_t)row * NU + c4) = make_float4(out[0], out[1], out[2], out[3]);
  }
}

// ---------------------------------------------------------------------------------------
// On-device parameter assembly and SRBD plant step (SURVEY.md section 8f.1 / 8f.2).
// Replaces the Python loops of reference src/mpc.py:178-255 (x_des, lever arms, contact
// schedule) with one thread per (robot, stage); contact masks are integer arithmetic and
// bit-exact with src/footstep_planner.py:226-246.
// ---------------------------------------------------------------------------------------
struct GaitTables {
  const float* __restrict__ plan_pos;    // [B,S,4,3]
  const uint8_t* __restrict__ feet_id;   // [B,S] stance bits of the single-support part
  const int32_t* __restrict__ ss;        // [B]
  const int32_t* __restrict__ ds;        // [B]
  const float* __restrict__ v_ref;       // [B,3]
  const float* __restrict__ omega_ref;   // [B]
  const float* __restrict__ rp0;         // [B,2] initial roll, pitch
  int32_t S, total_steps;
  float step_height, g, dt;
};

// foot position the MPC look-ahead uses at tick `tk` (reference MPC.update_r_num,
// src/mpc.py:306-318 + src/foot_trajectory_generator.py:27-96) and the stance bits of that tick
__device__ __forceinline__ int lookahead(const GaitTables& gt, int b, int tk, float foot[4][3]) {
  const int ss = gt.ss[b], period = ss + gt.ds[b];
  int step = tk / period;
  if (step > gt.S - 1) step = gt.S - 1;
  const int tin = tk - step * period;
  const int bits = (tin < ss) ? (int)gt.feet_id[(size_t)b * gt.S + step] : 0xF;
  const int nxt = step + 1 < gt.S ? step + 1 : gt.S - 1;
  const float* p0 = gt.plan_pos + ((size_t)b * gt.S + step) * 12;
  const float* p1 = gt.plan_pos + ((size_t)b * gt.S + nxt) * 12;
  const float ts = 0.8f * (float)ss, t = (float)tin;
  const float u = t / ts;
  const float blend = u * u * (3.f - 2.f * u);                // -2 u^3 + 3 u^2
  const float bump = 16.f * gt.step_height * u * u * (u - 1.f) * (u - 1.f);   // 16h (u^4 - 2u^3 + u^2)
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    const bool stance = (bits >> l) & 1;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float a = p0[3 * l + k], c = p1[3 * l + k];
      float v = a;
      if (!stance && step != 0) {
        if (t >= ts) v = c;
        else v = (k == 2) ? a + bump : a + (c - a) * blend;
      }
      foot[l][k] = v;
    }
  }
  return bits;
}

struct AssembleParams {
  GaitTables gt;
  const int32_t* __restrict__ tick;      // [1] current tick (device)
  const float* __restrict__ x;           // [B,13] measured state
  const float* __restrict__ yaw_start;   // [B]
  const float* __restrict__ com_start;   // [B,3]
  float* __restrict__ x_des;             // [B,N+1,13]
  float* __restrict__ r;                 // [B,N,4,3]
  uint8_t* __restrict__ mask;            // [B,N]
  int32_t B, N;                          // any horizon (runtime)
};

__global__ void __launch_bounds__(128) assemble_kernel(const AssembleParams p) {
  const int N = p.N;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.B * (N + 1)) return;
  const int b = idx / (N + 1), i = idx % (N + 1);
  const GaitTables& gt = p.gt;
  const int t = *p.tick;
  const int period = gt.ss[b] + gt.ds[b];
  int step_now = t / period;
  if (step_now > gt.S - 1) step_now = gt.S - 1;
  const bool last = step_now == gt.total_steps - 1;          // src/mpc.py:181-183
  const float vx = last ? 0.f : gt.v_ref[3 * b], vy = last ? 0.f : gt.v_ref[3 * b + 1],
              vz = last ? 0.f : gt.v_ref[3 * b + 2], om = last ? 0.f : gt.omega_ref[b];
  const float fi = (float)i;
  float* xd = p.x_des + ((size_t)b * (N + 1) + i) * 13;       // src/mpc.py:202-214
  const float cx = p.com_start[3 * b] + fi * vx * gt.dt, cy = p.com_start[3 * b + 1] + fi * vy * gt.dt,
              cz = p.com_start[3 * b + 2] + fi * vz * gt.dt;
  xd[0] = gt.rp0[2 * b]; xd[1] = gt.rp0[2 * b + 1]; xd[2] = p.yaw_start[b] + fi * om * gt.dt;
  xd[3] = cx; xd[4] = cy; xd[5] = cz;
  xd[6] = 0.f; xd[7] = 0.f; xd[8] = om;
  xd[9] = vx; xd[10] = vy; xd[11] = vz; xd[12] = gt.g;
  if (i == N) return;
  float foot[4][3];
  const int bits = lookahead(gt, b, t + i, foot);
  p.mask[(size_t)b * N + i] = (uint8_t)bits;                  // src/mpc.py:249-254
  const float* xs = p.x + (size_t)b * 13;
  const float ox = i == 0 ? xs[3] : cx, oy = i == 0 ? xs[4] : cy, oz = i == 0 ? xs[5] : cz;
  float* rr = p.r + ((size_t)b * N + i) * 12;                 // src/mpc.py:218-239
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    rr[3 * l] = foot[l][0] - ox; rr[3 * l + 1] = foot[l][1] - oy; rr[3 * l + 2] = foot[l][2] - oz;
  }
}

// SRBD forward-Euler plant with the applied first-stage forces and the true lever arms
// (the same model the MPC predicts with, reference src/mpc.py:86-117), plus the reference
// accumulator update of src/mpc.py:261-262 and a running tracking-error sum.
struct PlantParams {
  GaitTables gt;
  int32_t* __restrict__ tick;            // [1], advanced by thread 0 of block 0 of the NEXT kernel
  float* __restrict__ x;                 // [B,13]
  const float* __restrict__ r;           // [B,N,4,3] (stage 0 is used)
  const float* __restrict__ U;           // [B,N,12]
  const float* __restrict__ x_des;       // [B,N+1,13]
  float* __restrict__ yaw_start;
  float* __restrict__ com_start;
  float* __restrict__ track_err;         // [B,2] accumulated |p - p_des|^2, |Theta - Theta_des|^2
  int32_t B, N;
  float inv_mass;
  float ib[3];
  const float4* __restrict__ body;       // per-robot body [B][kBodyF4] (slots [0, B)), or nullptr
  const float* __restrict__ wrench;      // per-robot external wrench [B][N][6] (slots [0, B); stage 0 is applied),
                                         // or nullptr
};

__global__ void __launch_bounds__(128) plant_kernel(const PlantParams p) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  const GaitTables& gt = p.gt;
  const int t = *p.tick;
  float* x = p.x + (size_t)b * 13;
  const float* u = p.U + (size_t)b * p.N * 12;
  const float* r0 = p.r + (size_t)b * p.N * 12;
  const float* xd = p.x_des + (size_t)b * (p.N + 1) * 13;
  float sn, cs;
  sincosf(x[2], &sn, &cs);
  // net force and torque
  float fx = 0.f, fy = 0.f, fz = 0.f, tx = 0.f, ty = 0.f, tz = 0.f;
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    const float ax = u[3 * l], ay = u[3 * l + 1], az = u[3 * l + 2];
    const float rx = r0[3 * l], ry = r0[3 * l + 1], rz = r0[3 * l + 2];
    fx += ax; fy += ay; fz += az;
    tx += ry * az - rz * ay; ty += rz * ax - rx * az; tz += rx * ay - ry * ax;
  }
  if (p.wrench) {   // the known external force and torque of stage 0 (cmpc_set_wrench)
    const float* e = p.wrench + (size_t)b * p.N * 6;
    fx += e[0]; fy += e[1]; fz += e[2];
    tx += e[3]; ty += e[4]; tz += e[5];
  }
  // omega_dot = Rz Ib^-1 Rz' tau
  float bx, by, bz, im = p.inv_mass;
  if (p.body) {
    const float4* bq = p.body + (size_t)b * kBodyF4;
    const float4 b0 = __ldg(bq), b1 = __ldg(bq + 1), b2 = __ldg(bq + 2);
    const float q0 = cs * tx + sn * ty, q1 = -sn * tx + cs * ty, q2 = tz;
    im = b0.x;
    bx = b0.y * q0 + b0.z * q1 + b0.w * q2;
    by = b1.x * q0 + b1.y * q1 + b1.z * q2;
    bz = b1.w * q0 + b2.x * q1 + b2.y * q2;
  } else {
    bx = p.ib[0] * (cs * tx + sn * ty); by = p.ib[1] * (-sn * tx + cs * ty); bz = p.ib[2] * tz;
  }
  const float wdx = cs * bx - sn * by, wdy = sn * bx + cs * by, wdz = bz;
  const float dt = gt.dt;
  const float wx = x[6], wy = x[7], wz = x[8];
  // tracking error of the state the controller saw
  const float ep = (x[3] - xd[3]) * (x[3] - xd[3]) + (x[4] - xd[4]) * (x[4] - xd[4]) + (x[5] - xd[5]) * (x[5] - xd[5]);
  const float et = (x[0] - xd[0]) * (x[0] - xd[0]) + (x[1] - xd[1]) * (x[1] - xd[1]) + (x[2] - xd[2]) * (x[2] - xd[2]);
  p.track_err[2 * b] += ep;
  p.track_err[2 * b + 1] += et;
  // X+ = X + dt (A X + B u):  Theta' = Rz w, p' = v, w' = I^-1 tau, v' = f/m + g e_z
  x[0] += dt * (cs * wx - sn * wy);
  x[1] += dt * (sn * wx + cs * wy);
  x[2] += dt * wz;
  x[3] += dt * x[9]; x[4] += dt * x[10]; x[5] += dt * x[11];
  x[6] += dt * wdx; x[7] += dt * wdy; x[8] += dt * wdz;
  x[9] += dt * fx * im; x[10] += dt * fy * im; x[11] += dt * (fz * im + x[12]);
  // reference accumulators (src/mpc.py:261-262), zeroed references during the last planned step
  const int period = gt.ss[b] + gt.ds[b];
  int step_now = t / period;
  if (step_now > gt.S - 1) step_now = gt.S - 1;
  if (step_now != gt.total_steps - 1) {
    p.com_start[3 * b] += gt.v_ref[3 * b] * dt;
    p.com_start[3 * b + 1] += gt.v_ref[3 * b + 1] * dt;
    p.com_start[3 * b + 2] += gt.v_ref[3 * b + 2] * dt;
    p.yaw_start[b] += gt.omega_ref[b] * dt;
  }
}

__global__ void tick_kernel(int32_t* tick) { *tick += 1; }

// ---------------------------------------------------------------------------------------
// Any horizon (reference src/main.py:41 accepts any params['N']): a horizon N without a compiled
// solve kernel runs on the next compiled horizon NK > N.  The extra stages are all-swing (no
// unknowns) and carry no cost (SolveParams::n_eff = N; the horizon Gram matrices are those of N
// with an identity tail), so the padded problem has exactly the optimum of the N-stage problem.
// pad_kernel copies a batch of user-layout records [B,N,...] into NK-layout scratch, unpad_kernel
// copies U / X back.  One thread per float of the wider layout, coalesced on that side.
// ---------------------------------------------------------------------------------------
struct PadParams {
  const float* __restrict__ r;        // [B,N,12]
  const uint8_t* __restrict__ mask;   // [B,N]
  const float* __restrict__ x_des;    // [B,N+1,13]
  float* __restrict__ r_k;            // [B,NK,12]
  uint8_t* __restrict__ mask_k;       // [B,NK]
  float* __restrict__ x_des_k;        // [B,NK+1,13]
  int32_t B, N, NK;
};

__global__ void __launch_bounds__(256) pad_kernel(const PadParams p) {
  const int per = 12 * p.NK + 13 * (p.NK + 1) + p.NK;       // work items per problem
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)p.B * per) return;
  const int b = (int)(gid / per);
  int i = (int)(gid - (long long)b * per);
  if (i < 12 * p.NK) {
    p.r_k[(size_t)b * 12 * p.NK + i] = i < 12 * p.N ? __ldg(p.r + (size_t)b * 12 * p.N + i) : 0.f;
    return;
  }
  i -= 12 * p.NK;
  if (i < 13 * (p.NK + 1)) {
    const int k = i / 13, c = i - 13 * k;
    const int ks = k <= p.N ? k : p.N;                      // hold the last desired state (it has no weight)
    p.x_des_k[(size_t)b * 13 * (p.NK + 1) + i] = __ldg(p.x_des + ((size_t)b * (p.N + 1) + ks) * 13 + c);
    return;
  }
  i -= 13 * (p.NK + 1);
  p.mask_k[(size_t)b * p.NK + i] = i < p.N ? __ldg(p.mask + (size_t)b * p.N + i) : (uint8_t)0;
}

struct UnpadParams {
  const float* __restrict__ U_k;      // [B,NK,12]
  const float* __restrict__ X_k;      // [B,NK+1,13] or nullptr
  float* __restrict__ U;              // [B,N,12]
  float* __restrict__ X;              // [B,N+1,13] or nullptr
  int32_t B, N, NK;
};

__global__ void __launch_bounds__(256) unpad_kernel(const UnpadParams p) {
  const int nu = 12 * p.N, nx = p.X ? 13 * (p.N + 1) : 0, per = nu + nx;
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)p.B * per) return;
  const int b = (int)(gid / per);
  const int i = (int)(gid - (long long)b * per);
  if (i < nu) p.U[(size_t)b * nu + i] = p.U_k[(size_t)b * 12 * p.NK + i];
  else p.X[(size_t)b * nx + (i - nu)] = p.X_k[(size_t)b * 13 * (p.NK + 1) + (i - nu)];
}

// forget the warm start (and the cached factorisation) of the slots whose mask byte is set
__global__ void __launch_bounds__(256) reset_warm_kernel(uint8_t* __restrict__ warm_valid,
                                                         float* __restrict__ cache_meta,
                                                         const uint8_t* __restrict__ slot_mask,
                                                         int32_t slot0, int32_t B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  if (slot_mask && !slot_mask[i]) return;
  warm_valid[slot0 + i] = 0;
  if (cache_meta) cache_meta[(size_t)(slot0 + i) * 4 + 2] = 0.f;
}

// store the bodies of slots [slot0, slot0 + B) (cmpc_set_body) and invalidate their cached factors, which
// were computed with the previous body.  An invalid body (mass not finite and positive, or a non-finite entry
// of Ib^-1) is stored with 1/m = NaN, which every solve of the slot reports through its non-finite guard.
__global__ void __launch_bounds__(256) set_body_kernel(const float* __restrict__ mass,
                                                       const float* __restrict__ ibody_inv,
                                                       float4* __restrict__ body, float* __restrict__ cache_meta,
                                                       int32_t slot0, int32_t B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const float m = mass[i];
  float ib[9];
  bool ok = isfinite(m) && m > 0.f;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    ib[k] = ibody_inv[(size_t)i * 9 + k];
    ok = ok && isfinite(ib[k]);
  }
  const float im = ok ? __frcp_rn(m) : __int_as_float(0x7fc00000);   // correctly rounded, = 1.0f / m on the host
  float4* d = body + (size_t)(slot0 + i) * kBodyF4;
  d[0] = make_float4(im, ib[0], ib[1], ib[2]);
  d[1] = make_float4(ib[3], ib[4], ib[5], ib[6]);
  d[2] = make_float4(ib[7], ib[8], 0.f, 0.f);
  if (cache_meta) cache_meta[(size_t)(slot0 + i) * 4 + 2] = 0.f;
}

// Running totals of a closed-loop rollout in one launch: ADMM iterations, problems whose status
// is not "solved", factorisation-cache hits (meta may be nullptr).  acc[3], unsigned 64-bit.
__global__ void __launch_bounds__(256) stats_kernel(const int32_t* __restrict__ iters,
                                                    const int32_t* __restrict__ status,
                                                    const uint8_t* __restrict__ hitflag, int32_t B,
                                                    unsigned long long* __restrict__ acc) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned it = 0, bad = 0, hit = 0;
  if (b < B) {
    it = (unsigned)iters[b];
    bad = status[b] != 1;
    hit = hitflag ? (unsigned)hitflag[b] : 0u;
  }
  it = __reduce_add_sync(0xffffffffu, it);
  bad = __reduce_add_sync(0xffffffffu, bad);
  hit = __reduce_add_sync(0xffffffffu, hit);
  if ((threadIdx.x & 31) == 0) {
    if (it) atomicAdd(acc, (unsigned long long)it);
    if (bad) atomicAdd(acc + 1, (unsigned long long)bad);
    if (hit) atomicAdd(acc + 2, (unsigned long long)hit);
  }
}

// ---------------------------------------------------------------------------------------
// Leg controllers on the output side of the MPC (SURVEY.md section 8f.3): one thread per
// (robot, leg) turns the first-stage force of the solve, the simulator's leg Jacobians /
// inertia / bias forces and the gait tables into joint torques.
//   stance leg:  tau = J' (-f)                                      (reference src/main.py:203-214)
//   swing  leg:  tau = J' (Kp (p_des - p) + Kd (v_des - v))
//                    + J' (J*M*J') (a_des - Jdot dq) + CG          (src/main.py:219-282; J*M*J' is the
//                                                                   ELEMENTWISE product, as in the reference)
// with the swing reference p_des, v_des, a_des of src/foot_trajectory_generator.py:27-96 (cubic
// xy, quartic z over 0.8 ss, z clamp of src/main.py:229-231) and the controller's stance mask
// (planned feet_id while time_in_step <= ss, all-stance afterwards - src/main.py:152-160 with the
// side effect of foot_trajectory_generator.py:53-54).  Streaming, HBM-bound: 57 floats in,
// 6 floats + 1 byte out per leg.
// ---------------------------------------------------------------------------------------
struct LegParams {
  GaitTables gt;
  const int32_t* __restrict__ tick;      // [1] current tick (device)
  const float* __restrict__ U;           // [B,N,12] forces of the solve (stage 0 is applied)
  const float* __restrict__ J;           // [B,4,3,3] linear foot Jacobian, leg columns, world frame
  const float* __restrict__ Jdot;        // [B,4,3,3]
  const float* __restrict__ Mleg;        // [B,4,3,3] rows 3:6 of the mass matrix, leg columns
  const float* __restrict__ cg;          // [B,4,3] Coriolis + gravity of the leg joints
  const float* __restrict__ dq;          // [B,4,3] joint velocities
  const float* __restrict__ foot_pos;    // [B,4,3] measured
  const float* __restrict__ foot_vel;    // [B,4,3]
  float* __restrict__ tau;               // [B,4,3]
  float* __restrict__ p_des;             // [B,4,3] desired foot position (what the reference logs), nullable
  uint8_t* __restrict__ stance;          // [B] stance bits the controller used, nullable
  int32_t B, N;
  float kp[3], kd[3];
};

__global__ void __launch_bounds__(128) leg_torque_kernel(const LegParams p) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.B * 4) return;
  const int b = idx >> 2, l = idx & 3;
  const GaitTables& gt = p.gt;
  const int t = *p.tick;
  const int ss = gt.ss[b], period = ss + gt.ds[b];
  int step = t / period;
  if (step > gt.S - 1) step = gt.S - 1;
  const int tin = t - step * period;
  const int bits = tin <= ss ? (int)gt.feet_id[(size_t)b * gt.S + step] : 0xF;
  const bool is_stance = (bits >> l) & 1;
  const int nxt = step + 1 < gt.S ? step + 1 : step;
  const float* p0 = gt.plan_pos + (((size_t)b * gt.S + step) * 4 + l) * 3;
  const float* p1 = gt.plan_pos + (((size_t)b * gt.S + nxt) * 4 + l) * 3;
  float pd[3] = {p0[0], p0[1], p0[2]}, vd[3] = {0.f, 0.f, 0.f}, ad[3] = {0.f, 0.f, 0.f};
  if (!is_stance && step != 0) {
    const float ts = 0.8f * (float)ss, tt = (float)tin;
    if (tt >= ts) {
      pd[0] = p1[0]; pd[1] = p1[1]; pd[2] = p1[2];
    } else {
      const float u = tt / ts, idt = 1.f / gt.dt;
      const float s0 = u * u * (3.f - 2.f * u);                      // -2u^3 + 3u^2
      const float s1 = 6.f * u * (1.f - u) / ts * idt;               // d/dt, per second
      const float s2 = 6.f * (1.f - 2.f * u) / (ts * ts) * idt * idt;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const float d = p1[k] - p0[k];
        pd[k] = p0[k] + d * s0; vd[k] = d * s1; ad[k] = d * s2;
      }
      const float h16 = 16.f * gt.step_height;
      const float um = u - 1.f;
      pd[2] = p0[2] + h16 * u * u * um * um;                         // 16h (u^4 - 2u^3 + u^2)
      vd[2] = h16 * (4.f * u * u * u - 6.f * u * u + 2.f * u) / ts * idt;
      ad[2] = h16 * (12.f * u * u - 12.f * u + 2.f) / (ts * ts) * idt * idt;
      if (pd[2] < 0.f) { pd[2] = 0.f; vd[2] = 0.f; }
    }
  }
  const size_t o3 = (size_t)idx * 3, o9 = (size_t)idx * 9;
  float Jl[3][3];
#pragma unroll
  for (int i = 0; i < 9; ++i) Jl[i / 3][i % 3] = __ldg(p.J + o9 + i);
  float w[3];                                                        // task-space vector, tau = J' w (+ CG)
  float bias[3] = {0.f, 0.f, 0.f};
  if (is_stance) {
    const float* f = p.U + (size_t)b * p.N * 12 + 3 * l;
    w[0] = -__ldg(f); w[1] = -__ldg(f + 1); w[2] = -__ldg(f + 2);
  } else {
    float e[3];                                                      // a_des - Jdot dq
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      float acc = ad[i];
#pragma unroll
      for (int k = 0; k < 3; ++k) acc -= __ldg(p.Jdot + o9 + 3 * i + k) * __ldg(p.dq + o3 + k);
      e[i] = acc;
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      float acc = p.kp[i] * (pd[i] - __ldg(p.foot_pos + o3 + i)) + p.kd[i] * (vd[i] - __ldg(p.foot_vel + o3 + i));
#pragma unroll
      for (int k = 0; k < 3; ++k) acc += Jl[i][k] * __ldg(p.Mleg + o9 + 3 * i + k) * Jl[k][i] * e[k];
      w[i] = acc;
      bias[i] = __ldg(p.cg + o3 + i);
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k)
    p.tau[o3 + k] = Jl[0][k] * w[0] + Jl[1][k] * w[1] + Jl[2][k] * w[2] + bias[k];
  if (p.p_des) { p.p_des[o3] = pd[0]; p.p_des[o3 + 1] = pd[1]; p.p_des[o3 + 2] = pd[2]; }
  if (p.stance && l == 0) p.stance[b] = (uint8_t)bits;
}


// ---------------------------------------------------------------------------------------
// Lite3 leg kinematics (SURVEY.md section 8f.3): what the reference reads from DART every tick
// (src/main.py:203-214, 236-262, 286-350) in closed form from the joint tree of
// lite3_urdf/urdf/Lite3.urdf (hip offsets :45/:143/:240/:337, roll axis -x :48, thigh offset :73,
// pitch / knee axis -y :76/:103, thigh 0.20 :100, shank 0.21 :122; link masses / centres of mass
// :32-33, :54-55, :82-83, :109).  One thread per (robot, leg): foot position / velocity, the
// world-frame linear Jacobian of the foot w.r.t. the leg's 3 joints and its time derivative, the
// base-translation rows of the joint-space inertia matrix at the leg's columns
// (sum_i m_i J_com_i) and the gravity torques of the leg's joints.  Host mirror: kinematics.py.
// Streaming: 21 floats in, 45 floats out per leg.
// ---------------------------------------------------------------------------------------
struct KinParams {
  const float* __restrict__ base_pos;   // [B,3]
  const float* __restrict__ theta;      // [B,3] torso rotation vector
  const float* __restrict__ v_base;     // [B,3]
  const float* __restrict__ w_base;     // [B,3] world-frame angular velocity
  const float* __restrict__ q;          // [B,4,3] HipX, HipY, Knee
  const float* __restrict__ dq;         // [B,4,3]
  float* __restrict__ foot_pos;         // [B,4,3]
  float* __restrict__ foot_vel;         // [B,4,3]
  float* __restrict__ J;                // [B,4,3,3]
  float* __restrict__ Jdot;             // [B,4,3,3]
  float* __restrict__ Mleg;             // [B,4,3,3] nullable
  float* __restrict__ cg;               // [B,4,3]   nullable
  int32_t B;
  float g;                              // gravity (negative, along z)
};

struct V3 { float x, y, z; };
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 operator*(float s, V3 a) { return {s * a.x, s * a.y, s * a.z}; }
__device__ __forceinline__ V3 cross(V3 a, V3 b) {
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
struct M3 { float m[3][3]; };
__device__ __forceinline__ V3 mul(const M3& R, V3 v) {
  return {R.m[0][0] * v.x + R.m[0][1] * v.y + R.m[0][2] * v.z, R.m[1][0] * v.x + R.m[1][1] * v.y + R.m[1][2] * v.z,
          R.m[2][0] * v.x + R.m[2][1] * v.y + R.m[2][2] * v.z};
}

__global__ void __launch_bounds__(128) leg_kinematics_kernel(const KinParams p) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.B * 4) return;
  const int b = idx >> 2, l = idx & 3;
  const float sx = l < 2 ? 1.f : -1.f, sy = (l & 1) ? -1.f : 1.f;
  // torso rotation exp([theta]x)
  const float tx = p.theta[3 * b], ty = p.theta[3 * b + 1], tz = p.theta[3 * b + 2];
  const float ang2 = tx * tx + ty * ty + tz * tz, ang = sqrtf(ang2);
  float ka, kb;                      // sin(a)/a, (1 - cos a)/a^2
  if (ang < 1e-4f) { ka = 1.f - ang2 * (1.f / 6.f); kb = 0.5f - ang2 * (1.f / 24.f); }
  else { float sn, cs; sincosf(ang, &sn, &cs); ka = sn / ang; kb = (1.f - cs) / ang2; }
  M3 Rb;
  Rb.m[0][0] = 1.f - kb * (ty * ty + tz * tz); Rb.m[0][1] = -ka * tz + kb * tx * ty; Rb.m[0][2] = ka * ty + kb * tx * tz;
  Rb.m[1][0] = ka * tz + kb * tx * ty; Rb.m[1][1] = 1.f - kb * (tx * tx + tz * tz); Rb.m[1][2] = -ka * tx + kb * ty * tz;
  Rb.m[2][0] = -ka * ty + kb * tx * tz; Rb.m[2][1] = ka * tx + kb * ty * tz; Rb.m[2][2] = 1.f - kb * (tx * tx + ty * ty);
  const V3 pb = {p.base_pos[3 * b], p.base_pos[3 * b + 1], p.base_pos[3 * b + 2]};
  const V3 vb = {p.v_base[3 * b], p.v_base[3 * b + 1], p.v_base[3 * b + 2]};
  const V3 wb = {p.w_base[3 * b], p.w_base[3 * b + 1], p.w_base[3 * b + 2]};
  const float q1 = p.q[3 * idx], q2 = p.q[3 * idx + 1], q3 = p.q[3 * idx + 2];
  const float d1 = p.dq[3 * idx], d2 = p.dq[3 * idx + 1], d3 = p.dq[3 * idx + 2];
  float s1, c1, s2, c2, s23, c23;
  sincosf(q1, &s1, &c1);
  sincosf(q2, &s2, &c2);
  sincosf(q2 + q3, &s23, &c23);
  // torso-frame geometry.  R1 = rot(-x, q1) = [[1,0,0],[0,c1,s1],[0,-s1,c1]]; the pitch joints
  // rotate about R1 (0,-1,0), by q2 (thigh) and q2 + q3 (shank): R1 Ry' with Ry'(q) (0,0,z) = (-s z, 0, c z)
  auto r1 = [&](V3 v) -> V3 { return {v.x, c1 * v.y + s1 * v.z, -s1 * v.y + c1 * v.z}; };
  auto leg_plane = [&](float sq, float cq, V3 v) -> V3 {        // R1 Ry'(q) v
    return r1({cq * v.x - sq * v.z, v.y, sq * v.x + cq * v.z});
  };
  const V3 o1b = {sx * 0.1745f, sy * 0.062f, 0.f};
  const V3 o2b = o1b + r1({0.f, sy * 0.0985f, 0.f});
  const V3 o3b = o2b + leg_plane(s2, c2, {0.f, 0.f, -0.20f});
  const V3 fb = o3b + leg_plane(s23, c23, {0.f, 0.f, -0.21f});
  const V3 a1b = {-1.f, 0.f, 0.f};
  const V3 a2b = r1({0.f, -1.f, 0.f});                            // hip pitch and knee axes coincide
  // world frame
  const V3 o[3] = {pb + mul(Rb, o1b), pb + mul(Rb, o2b), pb + mul(Rb, o3b)};
  const V3 a[3] = {mul(Rb, a1b), mul(Rb, a2b), mul(Rb, a2b)};
  const V3 pf = pb + mul(Rb, fb);
  const float dqv[3] = {d1, d2, d3};
  auto point_vel = [&](V3 x, int upto) -> V3 {                    // point fixed in link `upto` (0 = torso)
    V3 v = vb + cross(wb, x - pb);
#pragma unroll
    for (int k = 0; k < 3; ++k)
      if (k < upto) v = v + dqv[k] * cross(a[k], x - o[k]);
    return v;
  };
  const V3 pdot = point_vel(pf, 3);
  V3 wl = wb;                                                     // angular velocity of the link carrying axis k
  float Jm[3][3], Jd[3][3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const V3 arm = pf - o[k];
    const V3 jc = cross(a[k], arm);
    const V3 adot = cross(wl, a[k]);
    const V3 jd = cross(adot, arm) + cross(a[k], pdot - point_vel(o[k], k));
    Jm[0][k] = jc.x; Jm[1][k] = jc.y; Jm[2][k] = jc.z;
    Jd[0][k] = jd.x; Jd[1][k] = jd.y; Jd[2][k] = jd.z;
    wl = wl + dqv[k] * a[k];
  }
  const size_t o3 = (size_t)idx * 3, o9 = (size_t)idx * 9;
  p.foot_pos[o3] = pf.x; p.foot_pos[o3 + 1] = pf.y; p.foot_pos[o3 + 2] = pf.z;
  p.foot_vel[o3] = pdot.x; p.foot_vel[o3 + 1] = pdot.y; p.foot_vel[o3 + 2] = pdot.z;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) { p.J[o9 + 3 * i + k] = Jm[i][k]; p.Jdot[o9 + 3 * i + k] = Jd[i][k]; }
  if (p.Mleg || p.cg) {
    // centres of mass of hip, thigh, shank, foot (torso frame) and their masses
    const V3 cb[4] = {o1b + r1({-sx * 0.0047f, -sy * 0.0091f, -0.0018f}),
                      o2b + leg_plane(s2, c2, {-0.00523f, -sy * 0.0216f, -0.0273f}),
                      o3b + leg_plane(s23, c23, {0.00585f, -8.732e-07f, -0.12f}), fb};
    const float ml[4] = {0.428f, 0.61f, 0.115f, 0.01f};
    float Mr[3][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const V3 c = pb + mul(Rb, cb[i]);
#pragma unroll
      for (int k = 0; k < 3; ++k)
        if (k <= i) {
          const V3 jc = ml[i] * cross(a[k], c - o[k]);
          Mr[0][k] += jc.x; Mr[1][k] += jc.y; Mr[2][k] += jc.z;
        }
    }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int k = 0; k < 3; ++k)
        if (p.Mleg) p.Mleg[o9 + 3 * i + k] = Mr[i][k];
    if (p.cg) {
#pragma unroll
      for (int k = 0; k < 3; ++k) p.cg[o3 + k] = -Mr[2][k] * p.g;       // -Mrow' (0, 0, g)
    }
  }
}

// FP32 FMA micro-benchmark: the denominator of the on-chip roofline (SURVEY.md section 8d).
// 8 independent FMA chains per thread, 256 threads, grid = a multiple of the SM count.
__global__ void __launch_bounds__(256) fma_peak_kernel(float* out, int iters, float a, float b) {
  float v0 = threadIdx.x, v1 = v0 + 1.f, v2 = v0 + 2.f, v3 = v0 + 3.f, v4 = v0 + 4.f, v5 = v0 + 5.f,
        v6 = v0 + 6.f, v7 = v0 + 7.f;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      v0 = fmaf(v0, a, b); v1 = fmaf(v1, a, b); v2 = fmaf(v2, a, b); v3 = fmaf(v3, a, b);
      v4 = fmaf(v4, a, b); v5 = fmaf(v5, a, b); v6 = fmaf(v6, a, b); v7 = fmaf(v7, a, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = ((v0 + v1) + (v2 + v3)) + ((v4 + v5) + (v6 + v7));
}

#endif  // CMPC_SOLVE_KERNELS_ONLY

}  // namespace cmpc
