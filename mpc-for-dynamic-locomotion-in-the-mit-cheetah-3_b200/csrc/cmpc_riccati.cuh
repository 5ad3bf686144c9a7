// cmpc_riccati.cuh - stage-wise (Riccati) variant of the solve kernel for long horizons.
//
// Same ADMM, same iterates as solve_kernel (cmpc_kernels.cuh): only the x-update's linear solve
// changes.  K dlt = b with K = D^-1 + G' M G is an LQ problem: M is the Gram matrix of six decoupled
// double integrators driven by the stage wrenches w_k = G_k u_k,
//     pos_{k+1} = pos_k + dt vel_k,  vel_{k+1} = vel_k + dt w_k,  cost sum_k w_pos pos_k^2 + w_vel vel_k^2,
// so  q = P^-1 s  (s = G D b, then dlt_k = D_k (b_k - G_k' q_k), exactly the quantities of solve_kernel)
// follows from one backward and one forward sweep over the stages with 6x6 / 6x12 matrices instead
// of a dense 6N x 6N inverse:  O(N) work per iteration and per factorisation instead of O(N^2) and
// O(N^3), no horizon Gram matrices (M, M^-1) at all.  fp32 error of q: 1e-6 relative (measured against
// the dense fp64 solve, oracle/riccati_form.py), against ~1e-3 for the dense fp32 Gauss-Jordan sweep.
//
//   factor (once per rho, backward over k = N-1 .. 0, S_N = Q, xi = (pos, vel) in R^12):
//        Shat = dt^2 S_vv,  T_k = d E_k  (E_k = sum over stance legs of Gp Gp', Gp = [Ghat ; I/m]),
//        Phi = (I + T Shat)^-1,  Gam = Phi T,  L = Gam B'SA,  Y = A'S B Phi,  S <- Q + A'S (A - B L)
//   solve (every iteration):
//        p_k  = F_k' p_{k+1} + Y_k s_k          (backward, F_k = A - B L_k)
//        xi_{k+1} = F_k xi_k + B (Phi_k s_k - dt Gam_k p^v_{k+1})     (forward)
//        q_k  = B' mu_{k+1},  mu_k = Q xi_k + A' mu_{k+1}            (adjoint, diagonal)
//
// One CTA per problem: 4N leg threads run the leg phases of solve_kernel unchanged; the two stage
// recursions are sequential and run on 12 lanes of warp 0 (lane i < 6: position-like component of
// axis i, lane 6 + i: velocity-like component), exchanging the 12 state values with warp shuffles.
// All per-stage matrices live in shared memory (288 floats per stage), laid out so that lane l of
// the recursion reads 12 consecutive floats per stage.  Throughput comes from several CTAs per SM
// (shared memory bound): the sequential warps of different problems interleave.
#pragma once
#include "cmpc_kernels.cuh"

namespace cmpc {

// WEIGHTS adds 16 floats after the rest: the slot's weight record, which persists through the ADMM loop.  FORCE adds
// 12 floats per leg after that: the leg maps, which persist because every factorisation rebuilds E_k from them.  STAGE
// adds 12 floats per stage after those: the slot's stage weights, read by every factorisation and adjoint pass.
template <int N, bool WEIGHTS = false, bool FORCE = false, bool STAGE = false>
struct RGeo {
  static constexpr int NLEG = 4 * N;
  static constexpr int TH0 = ((NLEG + 31) / 32) * 32;
  static constexpr int THREADS = TH0 < 64 ? 64 : TH0;
  static constexpr int LWARPS = (NLEG + 31) / 32;
  static constexpr int NW = 6 * N;
  static constexpr int NX = 13 * (N + 1);
  // dynamic shared memory, in floats (every block a multiple of 4 floats)
  static constexpr int R4(int v) { return ((v + 3) / 4) * 4; }
  static constexpr int O_BW = 0;                       // [N][12][12]  lane: L^T row (6) | Y row (6)
  static constexpr int O_FW = O_BW + 144 * N;          // [N][12][12]  lane<6: Gam row | Phi row; lane>=6: Lp row | Lv row
  static constexpr int O_E = O_FW + 144 * N;           // [N][21]  E_k, upper triangle packed
  static constexpr int O_S = O_E + R4(21 * N);         // [6N] wrench-space rhs
  static constexpr int O_XI = O_S + R4(NW);            // [12 (N+1)]
  static constexpr int O_V = O_XI + 12 * (N + 1);      // [6N] refreshed gradient / phi, w0
  static constexpr int O_WK = O_V + R4(NW);            // factorisation scratch
  static constexpr int WK = 144 + 7 * 36;              // S + 7 6x6 temporaries
  static constexpr int O_PRE = O_WK + WK;              // [18 N] g_k, phi_k / prefix sums of the X output / U staging
  static constexpr int O_MISC = O_PRE + R4(18 * N > 12 * (N + 1) ? 18 * N : 12 * (N + 1));   // x0[16], red[2][LWARPS][8], mask[N]
  static constexpr int O_WT = O_MISC + 16 + 2 * LWARPS * 8 + R4(N);   // [4 kWeightF4] (WEIGHTS instantiations)
  static constexpr int O_LEG = O_WT + (WEIGHTS ? 4 * kWeightF4 : 0);   // [NLEG][12] leg maps (FORCE instantiations)
  static constexpr int O_WS = O_LEG + (FORCE ? 12 * NLEG : 0);   // [N][12] stage weights (STAGE instantiations)
  static constexpr int FLOATS = O_WS + (STAGE ? 12 * N : 0);
  static constexpr size_t SMEM_BYTES = (size_t)FLOATS * 4;
  // set-up only arrays, aliased on the matrix area (dead before the first factorisation writes it)
  static constexpr int A_G = O_BW;                     // [NLEG][12] leg maps
  static constexpr int A_XD = A_G + 12 * NLEG;         // [NX + 3]
  static constexpr int A_R = A_XD + R4(NX + 3);        // [12N] lever arms
  static constexpr int A_H = A_R + 12 * N;             // [6N] linear term
  static constexpr int A_BODY = A_H + R4(NW);          // [4 kBodyF4] the slot's body (BODY instantiations)
  static_assert(A_BODY + 4 * kBodyF4 <= O_FW, "set-up arrays must fit in the backward-matrix area");
  static_assert(2 * 2 * NW <= 144 * N, "stage errors (doubles) must fit in the forward-matrix area");
};

// index of element (i, j), i <= j, of a packed upper triangle of a symmetric 6x6 matrix
__device__ __forceinline__ int sym6(int i, int j) {
  const int a = i < j ? i : j, b = i < j ? j : i;
  return a * 6 - (a * (a - 1)) / 2 + (b - a);
}

// Adjoint of the tracking cost over the state trajectory in s_xi: out_{k-1} = B' mu_k,
// mu_k = Q xi_k + A' mu_{k+1}.  Lanes 0-5, one axis each, no communication.
template <int N>
__device__ __forceinline__ void adjoint_pass(const float* __restrict__ s_xi, float* __restrict__ out, float dt,
                                             int n_eff, float qp, float qv, int lane) {
  if (lane < 6) {
    // chunks of CH stages: all loads of a chunk are issued before its (dependent) FMA chain - left to
    // itself the compiler keeps load -> use -> store per stage and the chain pays one LDS latency per stage
    constexpr int CH = 6;
    float mp = 0.f, mv = 0.f;
    for (int k = N; k >= 1; k -= CH) {
      float pos[CH], vel[CH];
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        const int kk = k - u > 1 ? k - u : 1;
        pos[u] = s_xi[12 * kk + lane];
        vel[u] = s_xi[12 * kk + 6 + lane];
      }
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        const int kk = k - u;
        const float cq = (kk >= 1 && kk <= n_eff) ? 1.f : 0.f;           // stages that carry cost
        const float mvn = fmaf(cq * qv, vel[u], fmaf(dt, mp, mv));       // mu^v_k = Qv vel + dt mu^p_{k+1} + mu^v_{k+1}
        mp = fmaf(cq * qp, pos[u], mp);                                  // mu^p_k = Qp pos + mu^p_{k+1}
        mv = mvn;
        if (kk >= 1) out[6 * (kk - 1) + lane] = dt * mv;                 // q_{k-1} = B' mu_k
      }
    }
  }
}

// The stage recursions of q = P^-1 s, one warp.  Kept out of line on purpose: inside the solve kernel
// the leg state of every thread is live across this code and the register allocator then re-derives
// addresses and sinks the prefetches into the dependent chain (measured: 180-200 cycles per stage and
// pass against 75-85 for the same loops compiled on their own).
//  backward: lanes 0-11 carry p (lane i: p^p_i, lane 6+i: p^v_i); lanes 12-17 turn the same six shuffled
//            values into the feed-forward wrench w0_k = phi_k - dt Gam_k p^v_{k+1}.  Every active lane
//            evaluates  g - dt c[0:6] . p^v  with its own row c and its own g (s_g[18 k + lane]).
//  forward:  lane 6+i owns vel_i and a private copy of the six positions; six velocities are exchanged.
template <int N>
__device__ __noinline__ void riccati_sweeps(const float* __restrict__ s_bw, const float* __restrict__ s_fw,
                                            const float* __restrict__ s_g, float* __restrict__ s_w0,
                                            float* __restrict__ s_xi, float* __restrict__ s_q, float dt,
                                            int n_eff, float qp, float qv) {
  const int lane = threadIdx.x & 31;
  const int l12 = lane < 12 ? lane : 0;
  const int l18 = lane < 18 ? lane : 0;
  const int partner = lane < 6 ? lane : (lane < 12 ? lane - 6 : 0);
  {
    const float* base = lane < 12 ? s_bw + 12 * lane : s_fw + 12 * (l18 >= 12 ? l18 - 12 : 0);
    const float cpp = (lane >= 6 && lane < 12) ? dt : 0.f;
    const bool wlane = lane >= 12 && lane < 18;
    float pc = 0.f;
    const float* row = base + 144 * (N - 1);
    float4 c0 = *reinterpret_cast<const float4*>(row);
    float2 c1 = *reinterpret_cast<const float2*>(row + 4);
    float g = s_g[18 * (N - 1) + l18];
#pragma unroll 2
    for (int k = N - 1; k >= 0; --k) {
      const int kn = k > 0 ? k - 1 : 0;
      const float* nrow = base + 144 * kn;
      const float4 n0 = *reinterpret_cast<const float4*>(nrow);          // next stage, while the shuffles fly
      const float2 n1 = *reinterpret_cast<const float2*>(nrow + 4);
      const float gn = s_g[18 * kn + l18];
      const float y0 = __shfl_sync(0xffffffffu, pc, 6), y1 = __shfl_sync(0xffffffffu, pc, 7),
                  y2 = __shfl_sync(0xffffffffu, pc, 8), y3 = __shfl_sync(0xffffffffu, pc, 9),
                  y4 = __shfl_sync(0xffffffffu, pc, 10), y5 = __shfl_sync(0xffffffffu, pc, 11);
      const float pp = __shfl_sync(0xffffffffu, pc, partner);
      const float a0 = fmaf(c0.z, y2, fmaf(c0.y, y1, c0.x * y0));
      const float a1 = fmaf(c1.y, y5, fmaf(c1.x, y4, c0.w * y3));
      const float val = fmaf(-dt, a0 + a1, g);
      if (wlane) s_w0[6 * k + lane - 12] = val;                            // w0_k
      pc = fmaf(cpp, pp, pc) + val;
      c0 = n0; c1 = n1; g = gn;
    }
  }
  __syncwarp();
  {
    const bool vlane = lane >= 6 && lane < 12;
    float xc = 0.f;                                   // lane i<6: pos_i, lane 6+i: vel_i
    float ps[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (lane < 12) s_xi[lane] = 0.f;
    const float* row = s_fw + 12 * l12;
    float4 c0 = *reinterpret_cast<const float4*>(row), c1 = *reinterpret_cast<const float4*>(row + 4),
           c2 = *reinterpret_cast<const float4*>(row + 8);
    float w0 = vlane ? s_w0[lane - 6] : 0.f;
#pragma unroll 2
    for (int k = 0; k < N; ++k) {
      const int kn = k + 1 < N ? k + 1 : k;
      const float* nrow = s_fw + 144 * kn + 12 * l12;
      const float4 n0 = *reinterpret_cast<const float4*>(nrow), n1 = *reinterpret_cast<const float4*>(nrow + 4),
                   n2 = *reinterpret_cast<const float4*>(nrow + 8);
      const float wn = vlane ? s_w0[6 * kn + lane - 6] : 0.f;
      // the position part of the feedback only needs local data: off the critical path
      const float ap = fmaf(c1.y, ps[5], fmaf(c1.x, ps[4], fmaf(c0.w, ps[3], fmaf(c0.z, ps[2], fmaf(c0.y, ps[1], c0.x * ps[0])))));
      const float base_inc = w0 - ap;
      const float v0 = __shfl_sync(0xffffffffu, xc, 6), v1 = __shfl_sync(0xffffffffu, xc, 7),
                  v2 = __shfl_sync(0xffffffffu, xc, 8), v3 = __shfl_sync(0xffffffffu, xc, 9),
                  v4 = __shfl_sync(0xffffffffu, xc, 10), v5 = __shfl_sync(0xffffffffu, xc, 11);
      const float vel = __shfl_sync(0xffffffffu, xc, lane < 6 ? lane + 6 : lane);
      const float a0 = fmaf(c2.x, v2, fmaf(c1.w, v1, c1.z * v0));
      const float a1 = fmaf(c2.w, v5, fmaf(c2.z, v4, c2.y * v3));
      const float inc = vlane ? base_inc - (a0 + a1) : vel;
      xc = fmaf(dt, inc, xc);
      ps[0] = fmaf(dt, v0, ps[0]); ps[1] = fmaf(dt, v1, ps[1]); ps[2] = fmaf(dt, v2, ps[2]);
      ps[3] = fmaf(dt, v3, ps[3]); ps[4] = fmaf(dt, v4, ps[4]); ps[5] = fmaf(dt, v5, ps[5]);
      if (lane < 12) s_xi[12 * (k + 1) + lane] = xc;
      c0 = n0; c1 = n1; c2 = n2; w0 = wn;
    }
  }
  __syncwarp();
  adjoint_pass<N>(s_xi, s_q, dt, n_eff, qp, qv, lane);
}

// v = M w for the wrench sequence in s_s (exact gradient refresh): open-loop double integrators, then
// the same adjoint pass.  One warp, lanes 0-5.
template <int N>
__device__ __noinline__ void gram_sweeps(const float* __restrict__ s_s, float* __restrict__ s_xi,
                                         float* __restrict__ s_v, float dt, int n_eff, float qp, float qv) {
  const int lane = threadIdx.x & 31;
  if (lane < 6) {
    constexpr int CH = 6;
    float pos = 0.f, vel = 0.f;
    s_xi[lane] = 0.f; s_xi[6 + lane] = 0.f;
    for (int k = 0; k < N; k += CH) {
      float w[CH];
#pragma unroll
      for (int u = 0; u < CH; ++u) w[u] = s_s[6 * (k + u < N ? k + u : N - 1) + lane];
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        if (k + u < N) {
          pos = fmaf(dt, vel, pos);
          vel = fmaf(dt, w[u], vel);
          s_xi[12 * (k + u + 1) + lane] = pos;
          s_xi[12 * (k + u + 1) + 6 + lane] = vel;
        }
      }
    }
  }
  __syncwarp();
  adjoint_pass<N>(s_xi, s_v, dt, n_eff, qp, qv, lane);
}

// The adjoint pass with the state weights of every stage (STAGE instantiations): Q of stage k is 2 w_k from the
// slot's stage weights [N][12], found at float WS of the dynamic shared memory (RGeo::O_WS).  Each chunk loads its
// stages' Q with pos and vel, the cost mask folded into the load, so the loads stay off the dependent FMA chain.
template <int N, int WS>
__device__ __forceinline__ void adjoint_pass_stage(const float* __restrict__ s_xi, float* __restrict__ out, float dt,
                                                   int n_eff, int lane) {
  extern __shared__ __align__(16) float smem[];
  const float* s_ws = smem + WS;
  if (lane < 6) {
    constexpr int CH = 6;
    float mp = 0.f, mv = 0.f;
    for (int k = N; k >= 1; k -= CH) {
      float pos[CH], vel[CH], qp[CH], qv[CH];
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        const int kk = k - u > 1 ? k - u : 1;
        const bool cost = k - u >= 1 && k - u <= n_eff;                 // stages that carry cost
        pos[u] = s_xi[12 * kk + lane];
        vel[u] = s_xi[12 * kk + 6 + lane];
        qp[u] = cost ? 2.f * s_ws[12 * (kk - 1) + lane] : 0.f;
        qv[u] = cost ? 2.f * s_ws[12 * (kk - 1) + 6 + lane] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        const int kk = k - u;
        const float mvn = fmaf(qv[u], vel[u], fmaf(dt, mp, mv));        // mu^v_k = Qv_k vel + dt mu^p_{k+1} + mu^v_{k+1}
        mp = fmaf(qp[u], pos[u], mp);                                   // mu^p_k = Qp_k pos + mu^p_{k+1}
        mv = mvn;
        if (kk >= 1) out[6 * (kk - 1) + lane] = dt * mv;                // q_{k-1} = B' mu_k
      }
    }
  }
}

// riccati_sweeps and gram_sweeps with adjoint_pass_stage (STAGE instantiations).  The stage recursions are those of
// riccati_sweeps line for line; they are repeated rather than shared so that riccati_sweeps, which the kernels of the
// other feature sets call, compiles to the same machine code as before.
template <int N, int WS>
__device__ __noinline__ void riccati_sweeps_stage(const float* __restrict__ s_bw, const float* __restrict__ s_fw,
                                                  const float* __restrict__ s_g, float* __restrict__ s_w0,
                                                  float* __restrict__ s_xi, float* __restrict__ s_q, float dt,
                                                  int n_eff) {
  const int lane = threadIdx.x & 31;
  const int l12 = lane < 12 ? lane : 0;
  const int l18 = lane < 18 ? lane : 0;
  const int partner = lane < 6 ? lane : (lane < 12 ? lane - 6 : 0);
  {
    const float* base = lane < 12 ? s_bw + 12 * lane : s_fw + 12 * (l18 >= 12 ? l18 - 12 : 0);
    const float cpp = (lane >= 6 && lane < 12) ? dt : 0.f;
    const bool wlane = lane >= 12 && lane < 18;
    float pc = 0.f;
    const float* row = base + 144 * (N - 1);
    float4 c0 = *reinterpret_cast<const float4*>(row);
    float2 c1 = *reinterpret_cast<const float2*>(row + 4);
    float g = s_g[18 * (N - 1) + l18];
#pragma unroll 2
    for (int k = N - 1; k >= 0; --k) {
      const int kn = k > 0 ? k - 1 : 0;
      const float* nrow = base + 144 * kn;
      const float4 n0 = *reinterpret_cast<const float4*>(nrow);          // next stage, while the shuffles fly
      const float2 n1 = *reinterpret_cast<const float2*>(nrow + 4);
      const float gn = s_g[18 * kn + l18];
      const float y0 = __shfl_sync(0xffffffffu, pc, 6), y1 = __shfl_sync(0xffffffffu, pc, 7),
                  y2 = __shfl_sync(0xffffffffu, pc, 8), y3 = __shfl_sync(0xffffffffu, pc, 9),
                  y4 = __shfl_sync(0xffffffffu, pc, 10), y5 = __shfl_sync(0xffffffffu, pc, 11);
      const float pp = __shfl_sync(0xffffffffu, pc, partner);
      const float a0 = fmaf(c0.z, y2, fmaf(c0.y, y1, c0.x * y0));
      const float a1 = fmaf(c1.y, y5, fmaf(c1.x, y4, c0.w * y3));
      const float val = fmaf(-dt, a0 + a1, g);
      if (wlane) s_w0[6 * k + lane - 12] = val;                            // w0_k
      pc = fmaf(cpp, pp, pc) + val;
      c0 = n0; c1 = n1; g = gn;
    }
  }
  __syncwarp();
  {
    const bool vlane = lane >= 6 && lane < 12;
    float xc = 0.f;                                   // lane i<6: pos_i, lane 6+i: vel_i
    float ps[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (lane < 12) s_xi[lane] = 0.f;
    const float* row = s_fw + 12 * l12;
    float4 c0 = *reinterpret_cast<const float4*>(row), c1 = *reinterpret_cast<const float4*>(row + 4),
           c2 = *reinterpret_cast<const float4*>(row + 8);
    float w0 = vlane ? s_w0[lane - 6] : 0.f;
#pragma unroll 2
    for (int k = 0; k < N; ++k) {
      const int kn = k + 1 < N ? k + 1 : k;
      const float* nrow = s_fw + 144 * kn + 12 * l12;
      const float4 n0 = *reinterpret_cast<const float4*>(nrow), n1 = *reinterpret_cast<const float4*>(nrow + 4),
                   n2 = *reinterpret_cast<const float4*>(nrow + 8);
      const float wn = vlane ? s_w0[6 * kn + lane - 6] : 0.f;
      // the position part of the feedback only needs local data: off the critical path
      const float ap = fmaf(c1.y, ps[5], fmaf(c1.x, ps[4], fmaf(c0.w, ps[3], fmaf(c0.z, ps[2], fmaf(c0.y, ps[1], c0.x * ps[0])))));
      const float base_inc = w0 - ap;
      const float v0 = __shfl_sync(0xffffffffu, xc, 6), v1 = __shfl_sync(0xffffffffu, xc, 7),
                  v2 = __shfl_sync(0xffffffffu, xc, 8), v3 = __shfl_sync(0xffffffffu, xc, 9),
                  v4 = __shfl_sync(0xffffffffu, xc, 10), v5 = __shfl_sync(0xffffffffu, xc, 11);
      const float vel = __shfl_sync(0xffffffffu, xc, lane < 6 ? lane + 6 : lane);
      const float a0 = fmaf(c2.x, v2, fmaf(c1.w, v1, c1.z * v0));
      const float a1 = fmaf(c2.w, v5, fmaf(c2.z, v4, c2.y * v3));
      const float inc = vlane ? base_inc - (a0 + a1) : vel;
      xc = fmaf(dt, inc, xc);
      ps[0] = fmaf(dt, v0, ps[0]); ps[1] = fmaf(dt, v1, ps[1]); ps[2] = fmaf(dt, v2, ps[2]);
      ps[3] = fmaf(dt, v3, ps[3]); ps[4] = fmaf(dt, v4, ps[4]); ps[5] = fmaf(dt, v5, ps[5]);
      if (lane < 12) s_xi[12 * (k + 1) + lane] = xc;
      c0 = n0; c1 = n1; c2 = n2; w0 = wn;
    }
  }
  __syncwarp();
  adjoint_pass_stage<N, WS>(s_xi, s_q, dt, n_eff, lane);
}

template <int N, int WS>
__device__ __noinline__ void gram_sweeps_stage(const float* __restrict__ s_s, float* __restrict__ s_xi,
                                               float* __restrict__ s_v, float dt, int n_eff) {
  const int lane = threadIdx.x & 31;
  if (lane < 6) {
    constexpr int CH = 6;
    float pos = 0.f, vel = 0.f;
    s_xi[lane] = 0.f; s_xi[6 + lane] = 0.f;
    for (int k = 0; k < N; k += CH) {
      float w[CH];
#pragma unroll
      for (int u = 0; u < CH; ++u) w[u] = s_s[6 * (k + u < N ? k + u : N - 1) + lane];
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        if (k + u < N) {
          pos = fmaf(dt, vel, pos);
          vel = fmaf(dt, w[u], vel);
          s_xi[12 * (k + u + 1) + lane] = pos;
          s_xi[12 * (k + u + 1) + 6 + lane] = vel;
        }
      }
    }
  }
  __syncwarp();
  adjoint_pass_stage<N, WS>(s_xi, s_v, dt, n_eff, lane);
}

// BODY reads the problem's rigid body from its slot of p.body instead of p.inv_mass / p.ib.
// CONTACT projects each leg-stage onto its own contact surface from p.contact (LegContact).
// WEIGHTS reads the problem's cost weights from its slot of p.weights instead of p.w / p.r_weight.
// FORCE adds each stance leg-stage's force reference from p.force (see solve_kernel): d becomes a per-leg d_l, and
// every factorisation rebuilds E_k as sum_l (d_l / d) Gp_l Gp_l' so that T_k = d E_k stays sum_l d_l Gp_l Gp_l'.
// STAGE reads the state weights of every stage from p.wstage (S_N, the backward recursion, h, the adjoint pass).
template <int N, int MINB, bool BODY = false, bool CONTACT = false, bool WEIGHTS = false, bool FORCE = false,
          bool STAGE = false>
__global__ void __launch_bounds__((RGeo<N>::THREADS), MINB)
solve_riccati_kernel(const SolveParams p) {
  static_assert(!FORCE || (BODY && WEIGHTS), "force references are compiled with BODY + WEIGHTS only");
  static_assert(!STAGE || FORCE, "stage weights are compiled with BODY + WEIGHTS + FORCE only");
  using G_ = RGeo<N, WEIGHTS, FORCE, STAGE>;
  constexpr int NW = G_::NW, NLEG = G_::NLEG, THREADS = G_::THREADS, LWARPS = G_::LWARPS, NX = G_::NX;
  extern __shared__ __align__(16) float smem[];
  float* s_bw = smem + G_::O_BW;
  float* s_fw = smem + G_::O_FW;
  float* s_E = smem + G_::O_E;
  float* s_s = smem + G_::O_S;
  float* s_xi = smem + G_::O_XI;
  float* s_v = smem + G_::O_V;
  float* s_wk = smem + G_::O_WK;
  float* s_pre = smem + G_::O_PRE;
  float* s_x0 = smem + G_::O_MISC;
  float* s_red = s_x0 + 16;                               // [2][LWARPS][8]
  int* s_mask = reinterpret_cast<int*>(s_red + 2 * LWARPS * 8);
  // set-up only, aliased on the matrix area (first written by factorize)
  float* s_G = smem + (FORCE ? G_::O_LEG : G_::A_G);      // [NLEG][12]; FORCE: persists, d_l / d at 9
  float* s_xd = smem + G_::A_XD;
  float* s_r = smem + G_::A_R;
  float* s_h = smem + G_::A_H;
  float* s_body = smem + G_::A_BODY;
  double* s_e = reinterpret_cast<double*>(s_fw);          // [2][6N]
  float* s_wt = smem + G_::O_WT;                          // WEIGHTS: the slot's {w[0..12], r_weight, 0, 0}, persists
  float* s_ws = smem + G_::O_WS;                          // STAGE: the slot's stage weights [N][12], persist

  if ((int)blockIdx.x >= p.B) return;
  grid_dependency_wait();
  const int b = p.order ? p.order[blockIdx.x] : (int)blockIdx.x;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const bool leg_warp = warp < LWARPS;
  const int slot = p.slot0 + b;
  const int n_eff = p.n_eff > 0 ? p.n_eff : N;
  // The sequential stage recursions run on ONE warp of the CTA.  A warp's scheduler (SM sub-partition)
  // is its index in the CTA modulo 4, and the CTAs resident on one SM are 148 apart in blockIdx (a
  // multiple of 4): always taking warp 0 would queue the sequential warps of all resident CTAs on one
  // scheduler and leave three idle.  Rotate the choice with the CTA's wave on its SM.
  unsigned nsm;
  asm("mov.u32 %0, %%nsmid;" : "=r"(nsm));
  const int seq_warp = (int)((blockIdx.x + blockIdx.x / nsm) % (unsigned)(THREADS / 32));

  // ---- phase 0: stage the per-problem record ------------------------------------------------
  for (int i = tid; i < 13; i += THREADS) s_x0[i] = __ldg(p.x0 + (size_t)b * 13 + i);
  for (int i = tid; i < NX; i += THREADS) s_xd[i] = __ldg(p.x_des + (size_t)b * NX + i);
  for (int i = tid; i < 3 * NLEG; i += THREADS) s_r[i] = __ldg(p.r + (size_t)b * 3 * NLEG + i);
  for (int i = tid; i < N; i += THREADS) s_mask[i] = (int)__ldg(p.mask + (size_t)b * N + i);
  for (int i = tid; i < NW; i += THREADS) { s_s[i] = 0.f; s_v[i] = 0.f; }
  if constexpr (BODY) {
    if (tid < kBodyF4) reinterpret_cast<float4*>(s_body)[tid] = __ldg(p.body + (size_t)slot * kBodyF4 + tid);
  }
  if constexpr (WEIGHTS) {
    if (tid < kWeightF4) reinterpret_cast<float4*>(s_wt)[tid] = __ldg(p.weights + (size_t)slot * kWeightF4 + tid);
  }
  if constexpr (STAGE) {
    for (int i = tid; i < N * kStageF4; i += THREADS)
      reinterpret_cast<float4*>(s_ws)[i] = __ldg(p.wstage + (size_t)slot * N * kStageF4 + i);
  }
  float4 fr_in = make_float4(0.f, 0.f, 0.f, 0.f);   // FORCE: this leg-stage's {f_ref, w_f}
  if constexpr (FORCE) {
    if (tid < NLEG) fr_in = __ldg(p.force + (size_t)slot * NLEG + tid);
    if (tid == 0) s_x0[14] = fr_in.w;                // NaN: the slot was stored invalid (set_force_ref_kernel)
  }
  const float mu = __ldg(p.mu + b);
  const bool is_leg = tid < NLEG;
  float wx_in[3] = {0.f, 0.f, 0.f};
  float wy_in[3] = {0.f, 0.f, 0.f};
  const bool warm = p.warm_mode != 0 && p.warm_valid[slot] != 0;
  if (is_leg && warm) {
    const float* wx = p.warm_x + ((size_t)slot * NLEG + tid) * 3;
    wx_in[0] = wx[0]; wx_in[1] = wx[1]; wx_in[2] = wx[2];
    if (p.warm_mode == 2) {
      const float* wy = p.warm_y + ((size_t)slot * NLEG + tid) * 3;
      wy_in[0] = wy[0]; wy_in[1] = wy[1]; wy_in[2] = wy[2];
    }
  }
  __syncthreads();

  float sn, cs;
  sincosf(s_x0[2], &sn, &cs);
  const float im = BODY ? s_body[0] : p.inv_mass;
  const float alpha = p.alpha;
  const float dt = p.dt;
  float rho = p.rho;
  float rho_inv = 1.f / rho;

  // ---- phase 1: leg geometry, E_k, linear term ----------------------------------------------
  const int lj = tid >> 2, ll = tid & 3;
  bool stance = false;
  float Gh[3][3];
  float dinv = 0.f;
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int k = 0; k < 3; ++k) Gh[a][k] = 0.f;
  if (is_leg) {
    stance = (s_mask[lj] >> ll) & 1;
    if constexpr (BODY) leg_map_full(cs, sn, s_body + 1, s_r[3 * tid], s_r[3 * tid + 1], s_r[3 * tid + 2], Gh);
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
      for (int k = 0; k < 3; ++k) s_G[12 * tid + 3 * a + k] = Gh[a][k];
    s_G[12 * tid + 11] = stance ? 1.f : 0.f;
  }
  // FORCE: 2 w_f and -2 w_f f_ref of this leg, zero on swing legs (which ignore their entries)
  float w2 = 0.f, fl[3] = {0.f, 0.f, 0.f};
  if constexpr (FORCE) {
    if (stance) {
      w2 = 2.f * fr_in.w;
      fl[0] = -w2 * fr_in.x; fl[1] = -w2 * fr_in.y; fl[2] = -w2 * fr_in.z;
    }
  }
  for (int i = tid; i < NW; i += THREADS) {
    double ep = 0.0, ev = 0.0;
    if (i / 6 + 1 <= n_eff) stage_error(i / 6 + 1, i % 6, s_x0, s_xd, cs, sn, dt, ep, ev);
    s_e[i] = ep;
    s_e[NW + i] = ev;
  }
  __syncthreads();
  // E_k[a][a2] = sum over stance legs l, components c of Gp_l[a][c] Gp_l[a2][c]; upper triangle (21
  // entries per stage, 6 / 5 / 5 / 5 per thread of the stage); FORCE builds it in every factorisation instead
  if (!FORCE && is_leg) {
    for (int e = ll; e < 21; e += 4) {
      int a = 0, rem = e;
      while (rem >= 6 - a) { rem -= 6 - a; ++a; }
      const int a2 = a + rem;
      float acc = 0.f;
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        const float* g = s_G + 12 * (4 * lj + l);
        const float st = g[11];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float ga = a < 3 ? g[3 * a + c] : (a - 3 == c ? im * st : 0.f);
          const float gb = a2 < 3 ? g[3 * a2 + c] : (a2 - 3 == c ? im * st : 0.f);
          acc = fmaf(ga, gb, acc);
        }
      }
      s_E[21 * lj + e] = acc;
    }
  }
  if constexpr (STAGE) {
    for (int i = tid; i < NW; i += THREADS) {
      const int j = i / 6, a = i % 6;
      const double dtd = dt;
      double acc = 0.0;
      for (int k = j + 1; k <= N; ++k) {   // stage k's weights: row k - 1
        const double wp = s_ws[12 * (k - 1) + a], wv = s_ws[12 * (k - 1) + 6 + a];
        acc += 2.0 * (wp * dtd * dtd * (double)(k - 1 - j) * s_e[6 * (k - 1) + a] + wv * dtd * s_e[NW + 6 * (k - 1) + a]);
      }
      s_h[i] = (float)acc;
    }
  } else {
    for (int i = tid; i < NW; i += THREADS) {
      const int j = i / 6, a = i % 6;
      const double wp = (WEIGHTS ? s_wt[a] : p.w[a]), wv = (WEIGHTS ? s_wt[6 + a] : p.w[6 + a]), dtd = dt;
      double acc = 0.0;
      for (int k = j + 1; k <= N; ++k)
        acc += 2.0 * (wp * dtd * dtd * (double)(k - 1 - j) * s_e[6 * (k - 1) + a] + wv * dtd * s_e[NW + 6 * (k - 1) + a]);
      s_h[i] = (float)acc;
    }
  }
  __syncthreads();
  float gl[3] = {0.f, 0.f, 0.f};
  float hj[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (is_leg && stance) {
#pragma unroll
    for (int a = 0; a < 6; ++a) hj[a] = s_h[6 * lj + a];
#pragma unroll
    for (int k = 0; k < 3; ++k)
      gl[k] = Gh[0][k] * hj[0] + Gh[1][k] * hj[1] + Gh[2][k] * hj[2] + im * hj[3 + k];
    if constexpr (FORCE) {
#pragma unroll
      for (int k = 0; k < 3; ++k) gl[k] += fl[k];
    }
  }
  __syncthreads();          // the set-up arrays (aliased on the matrix area) are dead from here on

  // ---- factorisation (whole CTA; re-run when rho adapts) ------------------------------------
  // Backward Riccati recursion over the stages.  Every 6x6 product of a stage is one round: one
  // output element per thread (dot product of length 6 out of shared memory), rounds separated by
  // CTA barriers; only the 6x6 inverse runs on 6 lanes of warp 0 (rows in registers, pivot rows by
  // shuffle).  ~9 short rounds per stage instead of one warp walking through all of them.
  float* S = s_wk;                 // 12x12 row-major: [pos | vel] blocks
  float* Mx = s_wk + 144;          // I + T Shat, then Phi
  float* Gm = Mx + 36;             // Gam
  float* Lp = Gm + 36;
  float* Lv = Lp + 36;
  float* Up = Lv + 36;             // dt R Phi
  float* Uv = Up + 36;             // dt V Phi
  auto factorize = [&]() {
    dinv = stance ? 1.f / (p.sigma + 2.f * (WEIGHTS ? s_wt[13] : p.r_weight) + rho) : 0.f;
    const float d = 1.f / (p.sigma + 2.f * (WEIGHTS ? s_wt[13] : p.r_weight) + rho);
    if constexpr (FORCE) {
      // d_l = 1 / (c + 2 w_f) and E_k = sum_l (d_l / d) Gp_l Gp_l', c = 1 / d (cd): the set-up loop of the other
      // instantiations with each leg's terms scaled by c / (c + 2 w_f), exactly 1 at zero weight, so that a zero
      // weight gives their E_k bit for bit
      const float cd = p.sigma + 2.f * s_wt[13] + rho;
      dinv = stance ? 1.f / (cd + w2) : 0.f;
      if (is_leg) s_G[12 * tid + 9] = cd / (cd + w2);
      __syncthreads();
      if (is_leg) {
        for (int e = ll; e < 21; e += 4) {
          int a = 0, rem = e;
          while (rem >= 6 - a) { rem -= 6 - a; ++a; }
          const int a2 = a + rem;
          float acc = 0.f;
#pragma unroll
          for (int l = 0; l < 4; ++l) {
            const float* g = s_G + 12 * (4 * lj + l);
            const float st = g[11], sl = g[9];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              const float ga = a < 3 ? g[3 * a + c] : (a - 3 == c ? im * st : 0.f);
              const float gb = a2 < 3 ? g[3 * a2 + c] : (a2 - 3 == c ? im * st : 0.f);
              acc = fmaf(ga * sl, gb, acc);
            }
          }
          s_E[21 * lj + e] = acc;
        }
      }
      // (the barrier after S_N below orders these stores before round 1 reads them)
    }
    for (int e = tid; e < 144; e += THREADS) {       // S_N = Q (0 beyond the stages that carry cost)
      const int i = e / 12, j = e - 12 * i;
      // w[0:6] position-like, w[6:12] velocity-like; STAGE: stage N's (terminal) weights
      S[e] = (i == j && N <= n_eff) ? 2.f * (STAGE ? s_ws[12 * (N - 1) + i] : (WEIGHTS ? s_wt[i] : p.w[i])) : 0.f;
    }
    __syncthreads();
    for (int k = N - 1; k >= 0; --k) {
      const float* Ek = s_E + 21 * k;
      // round 1: Mx = I + T (dt^2 V),  T = d E_k
      for (int e = tid; e < 36; e += THREADS) {
        const int i = e / 6, j = e - 6 * i;
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int m = 0; m < 6; m += 2) {
          a0 = fmaf(Ek[sym6(i, m)], S[12 * (6 + m) + 6 + j], a0);
          a1 = fmaf(Ek[sym6(i, m + 1)], S[12 * (7 + m) + 6 + j], a1);
        }
        Mx[e] = fmaf(d * dt * dt, a0 + a1, i == j ? 1.f : 0.f);
      }
      __syncthreads();
      // round 2: Phi = Mx^-1, in-place Gauss-Jordan, lane r < 6 of the sequential warp holds row r
      if (warp == seq_warp) {
        float row[6];
        const int r = lane < 6 ? lane : 0;
#pragma unroll
        for (int j = 0; j < 6; ++j) row[j] = Mx[6 * r + j];
#pragma unroll
        for (int kk = 0; kk < 6; ++kk) {
          float pr[6];
#pragma unroll
          for (int j = 0; j < 6; ++j) pr[j] = __shfl_sync(0xffffffffu, row[j], kk);
          const float ip = __fdividef(1.f, pr[kk]);
          const float f = lane == kk ? 1.f - ip : row[kk] * ip;     // row -= f * pivot row; pivot row: scale by ip
#pragma unroll
          for (int j = 0; j < 6; ++j) {
            const float upd = fmaf(-f, pr[j], row[j]);
            row[j] = j == kk ? (lane == kk ? ip : -f) : upd;
          }
        }
        if (lane < 6) {
#pragma unroll
          for (int j = 0; j < 6; ++j) Mx[6 * r + j] = row[j];
        }
      }
      __syncthreads();
      // round 3: Gam = Phi T ; Up = dt R Phi ; Uv = dt V Phi   (108 outputs)
      for (int e = tid; e < 108; e += THREADS) {
        const int blk = e / 36, ee = e - 36 * blk, i = ee / 6, j = ee - 6 * i;
        float a0 = 0.f, a1 = 0.f;
        if (blk == 0) {
#pragma unroll
          for (int m = 0; m < 6; m += 2) {
            a0 = fmaf(Mx[6 * i + m], Ek[sym6(m, j)], a0);
            a1 = fmaf(Mx[6 * i + m + 1], Ek[sym6(m + 1, j)], a1);
          }
          Gm[ee] = d * (a0 + a1);
        } else {
          const float* Sr = S + 12 * (6 * (blk - 1) + i) + 6;      // row i of R (blk 1) or V (blk 2)
#pragma unroll
          for (int m = 0; m < 6; m += 2) {
            a0 = fmaf(Sr[m], Mx[6 * m + j], a0);
            a1 = fmaf(Sr[m + 1], Mx[6 * m + 6 + j], a1);
          }
          (blk == 1 ? Up : Uv)[ee] = dt * (a0 + a1);
        }
      }
      __syncthreads();
      // round 4: Lp = dt Gam R' ; Lv = dt Gam (dt R' + V)      (R'[m][j] = S_vp[m][j])
      for (int e = tid; e < 72; e += THREADS) {
        const int blk = e / 36, ee = e - 36 * blk, i = ee / 6, j = ee - 6 * i;
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int m = 0; m < 6; m += 2) {
          const float r0 = S[12 * (6 + m) + j], r1 = S[12 * (7 + m) + j];
          const float c0 = blk ? fmaf(dt, r0, S[12 * (6 + m) + 6 + j]) : r0;
          const float c1 = blk ? fmaf(dt, r1, S[12 * (7 + m) + 6 + j]) : r1;
          a0 = fmaf(Gm[6 * i + m], c0, a0);
          a1 = fmaf(Gm[6 * i + m + 1], c1, a1);
        }
        (blk ? Lv : Lp)[ee] = dt * (a0 + a1);
      }
      __syncthreads();
      // round 5: publish the stage's matrices in recursion layout, and the new S (registers first)
      {
        float* bw = s_bw + 144 * k;
        float* fw = s_fw + 144 * k;
        for (int e = tid; e < 144; e += THREADS) {
          const int ln = e / 12, c = e - 12 * ln, i = ln < 6 ? ln : ln - 6;
          // backward: lane i<6: [Lp[:,i] | Yp[i,:]], lane 6+i: [Lv[:,i] | Yv[i,:]],  Y = [Up ; dt Up + Uv]
          float vb, vf;
          if (c < 6) vb = (ln < 6 ? Lp : Lv)[6 * c + i];
          else vb = ln < 6 ? Up[6 * i + (c - 6)] : fmaf(dt, Up[6 * i + (c - 6)], Uv[6 * i + (c - 6)]);
          // forward area: lane i<6: [Gam[i,:] | Phi[i,:]] (feed-forward wrench, used by the backward pass),
          //               lane 6+i: [Lp[i,:] | Lv[i,:]] (feedback of the forward pass)
          if (ln < 6) vf = c < 6 ? Gm[6 * i + c] : Mx[6 * i + (c - 6)];
          else vf = c < 6 ? Lp[6 * i + c] : Lv[6 * i + (c - 6)];
          bw[e] = vb;
          fw[e] = vf;
        }
      }
      // S <- Q + A'S(A - B L):  P' = Qp + P - dt R Lp ; R' = dt P + R - dt R Lv ;
      //                         V' = Qv + dt^2 P + dt (R + R') + V - dt (dt R + V) Lv
      // (thread e < 36 owns element (i, j) of the three blocks; S is only rewritten after a barrier)
      float nP = 0.f, nR = 0.f, nV = 0.f;
      {
        const int e = tid < 36 ? tid : 0;
        const int i = e / 6, j = e - 6 * i;
        float rlp = 0.f, rlv = 0.f, wlv = 0.f;
#pragma unroll
        for (int m = 0; m < 6; ++m) {
          const float rim = S[12 * i + 6 + m];                       // R[i][m]
          rlp = fmaf(rim, Lp[6 * m + j], rlp);
          rlv = fmaf(rim, Lv[6 * m + j], rlv);
          wlv = fmaf(fmaf(dt, rim, S[12 * (6 + i) + 6 + m]), Lv[6 * m + j], wlv);
        }
        const float Pij = S[12 * i + j], Rij = S[12 * i + 6 + j], Rji = S[12 * j + 6 + i], Vij = S[12 * (6 + i) + 6 + j];
        const bool cost = k >= 1 && k <= n_eff;                      // stage k carries cost
        const float* wk = s_ws + 12 * (k >= 1 ? k - 1 : 0);         // STAGE: stage k's weights
        nP = Pij - dt * rlp + ((i == j && cost) ? 2.f * (STAGE ? wk[i] : (WEIGHTS ? s_wt[i] : p.w[i])) : 0.f);
        nR = fmaf(dt, Pij, Rij) - dt * rlv;
        nV = dt * dt * Pij + dt * (Rij + Rji) + Vij - dt * wlv +
             ((i == j && cost) ? 2.f * (STAGE ? wk[6 + i] : (WEIGHTS ? s_wt[6 + i] : p.w[6 + i])) : 0.f);
      }
      __syncthreads();
      if (tid < 36) {          // P and V are written from their upper triangle only: exactly symmetric
        const int i = tid / 6, j = tid - 6 * i;
        S[12 * i + 6 + j] = nR;
        S[12 * (6 + j) + i] = nR;
        if (i <= j) {
          S[12 * i + j] = nP; S[12 * j + i] = nP;
          S[12 * (6 + i) + 6 + j] = nV; S[12 * (6 + j) + 6 + i] = nV;
        }
      }
      __syncthreads();
    }
  };
  factorize();

  // ---- q = P^-1 s -----------------------------------------------------------------------------
  // (1) all threads: the rhs-dependent vectors of every stage, g_k = Y_k s_k (12) and phi_k = Phi_k s_k (6);
  // (2) warp 0: the stage recursions (riccati_sweeps, out of line).
  float* s_g = s_pre;              // [N][18]: g_k (lanes 0-11 of the backward pass) | phi_k (lanes 12-17)
  float* s_q = s_pre;              // [6N] q, written by the adjoint pass when g is dead
  float* s_w0 = s_v;               // [6N] w0 (s_v is otherwise only used by the gradient refresh)
  const float qp_l = lane < 6 ? 2.f * (WEIGHTS ? s_wt[lane] : p.w[lane]) : 0.f, qv_l = lane < 6 ? 2.f * (WEIGHTS ? s_wt[6 + lane] : p.w[6 + lane]) : 0.f;
  auto riccati_solve = [&]() {
    if (is_leg) {
      const float2* sp = reinterpret_cast<const float2*>(s_s + 6 * lj);
      const float2 s01 = sp[0], s23 = sp[1], s45 = sp[2];
#pragma unroll
      for (int u = 0; u < 5; ++u) {
        const int o = ll + 4 * u;                      // 18 outputs per stage over the stage's 4 threads
        if (o < 18) {
          const float2* rw = reinterpret_cast<const float2*>((o < 12 ? s_bw + 12 * o : s_fw + 12 * (o - 12)) + 144 * lj + 6);
          const float2 r01 = rw[0], r23 = rw[1], r45 = rw[2];
          s_g[18 * lj + o] = fmaf(r01.y, s01.y, r01.x * s01.x) + fmaf(r23.y, s23.y, r23.x * s23.x) + fmaf(r45.y, s45.y, r45.x * s45.x);
        }
      }
    }
    __syncthreads();
    if (warp == seq_warp) {
      // STAGE: the adjoint pass reads the stage weights at s_ws
      if constexpr (STAGE) riccati_sweeps_stage<N, G_::O_WS>(s_bw, s_fw, s_g, s_w0, s_xi, s_q, dt, n_eff);
      else riccati_sweeps<N>(s_bw, s_fw, s_g, s_w0, s_xi, s_q, dt, n_eff, qp_l, qv_l);
    }
  };
  auto gram_apply = [&]() {
    if (warp == seq_warp) {
      if constexpr (STAGE) gram_sweeps_stage<N, G_::O_WS>(s_s, s_xi, s_v, dt, n_eff);
      else gram_sweeps<N>(s_s, s_xi, s_v, dt, n_eff, qp_l, qv_l);
    }
  };

  // ---- initial iterate ------------------------------------------------------------------------
  const float fmin = p.f_min, fmax = p.f_max;
  const float inv1 = 1.f / (1.f + mu * mu), inv2 = 1.f / (1.f + 2.f * mu * mu);
  LegContact lc{};
  bool bad_contact = false;          // a leg-stage of this slot was stored invalid (mu = NaN, set_contact_kernel)
  if constexpr (CONTACT) {
    if (is_leg) load_contact(p.contact + ((size_t)slot * NLEG + tid) * kContactF4, mu, lc);
    else lc = LegContact{{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}, mu, inv1, inv2, fmin, fmax};
    bad_contact = __syncthreads_or(!(lc.mu == lc.mu)) != 0;
  }
  auto project = [&](float wx, float wy, float wz, float& zx, float& zy, float& zz) {
    if constexpr (CONTACT) {
      project_contact(lc, wx, wy, wz, zx, zy, zz);
    } else {
      const float ax_ = fabsf(wx), ay_ = fabsf(wy);
      const float big = fmaxf(ax_, ay_), small = fminf(ax_, ay_);
      const float f2 = (wz + mu * big) * inv1;
      const float f1 = (wz + mu * (ax_ + ay_)) * inv2;
      float fz = (mu * wz >= big) ? wz : ((mu * f2 >= small) ? f2 : f1);
      fz = fminf(fmaxf(fz, fmin), fmax);
      const float lim = mu * fz;
      zx = fminf(fmaxf(wx, -lim), lim);
      zy = fminf(fmaxf(wy, -lim), lim);
      zz = fz;
    }
  };
  float x[3] = {0.f, 0.f, 0.f}, y[3] = {0.f, 0.f, 0.f}, z[3] = {0.f, 0.f, 0.f};
  float vh[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (is_leg && stance) {
    if (warm) {
      x[0] = wx_in[0]; x[1] = wx_in[1]; x[2] = wx_in[2];
      y[0] = wy_in[0]; y[1] = wy_in[1]; y[2] = wy_in[2];
    }
    project(x[0], x[1], x[2], z[0], z[1], z[2]);
  }
#pragma unroll
  for (int a = 0; a < 6; ++a) vh[a] = hj[a];

  // wrench of a per-leg vector: s_s[6 j + a] = sum over the stage's legs of Gp v  (whole leg warps)
  auto store_wrench = [&](const float v3[3]) {
    if (leg_warp) {
      float wv[6];
#pragma unroll
      for (int a = 0; a < 3; ++a)
        wv[a] = quad_sum(Gh[a][0] * v3[0] + Gh[a][1] * v3[1] + Gh[a][2] * v3[2]);
#pragma unroll
      for (int k = 0; k < 3; ++k) wv[3 + k] = quad_sum(v3[k] * im);
      if (is_leg && ll < 3) *reinterpret_cast<float2*>(s_s + 6 * lj + 2 * ll) = pick_pair(wv, ll);
    }
  };
  auto refresh_gradient = [&]() {
    store_wrench(x);
    __syncthreads();
    gram_apply();
    __syncthreads();
    if (is_leg && stance) {
#pragma unroll
      for (int a = 0; a < 6; ++a) vh[a] = s_v[6 * lj + a] + hj[a];
    }
  };
  if (warm) refresh_gradient();

  float ng = 0.f;
  {
    float m = fmaxf(fabsf(gl[0]), fmaxf(fabsf(gl[1]), fabsf(gl[2])));
    if (leg_warp) {
      m = warp_max_nonneg(m);
      if (lane == 0) s_red[(LWARPS + warp) * 8] = m;
    }
    __syncthreads();
#pragma unroll
    for (int wv = 0; wv < LWARPS; ++wv) ng = fmaxf(ng, s_red[(LWARPS + wv) * 8]);
    __syncthreads();
  }

  // ---- ADMM (same iteration as solve_kernel) -------------------------------------------------
  int it = 0, status = 0;
  float pri = 0.f, dua = 0.f;
  const float two_rw = 2.f * p.r_weight;   // WEIGHTS: 2 s_wt[13], read where it is used
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
    float t[3] = {0.f, 0.f, 0.f};
    if (leg_warp) {
      float gr[3], rp[3];
      float trw = two_rw;
      if constexpr (WEIGHTS) trw = 2.f * s_wt[13];
      if constexpr (FORCE) trw += w2;   // (2 r_weight + 2 w_f) x - 2 w_f f_ref; a zero weight adds exact zeros
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        gr[k] = Gh[0][k] * vh[0] + Gh[1][k] * vh[1] + Gh[2][k] * vh[2] + im * vh[3 + k] + trw * x[k];
        if constexpr (FORCE) gr[k] += fl[k];
        rp[k] = x[k] - z[k];
        t[k] = -dinv * (gr[k] + y[k] + rho * rp[k]);
      }
      store_wrench(t);
      if (chk) {
        float st_[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        float sum = 0.f;
        if (stance) {
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            const float rd = gr[k] + y[k];
            st_[0] = fmaxf(st_[0], fabsf(rp[k]));
            st_[1] = fmaxf(st_[1], fabsf(rd));
            st_[2] = fmaxf(st_[2], fmaxf(fabsf(x[k]), fabsf(z[k])));
            st_[3] = fmaxf(st_[3], fmaxf(fabsf(gr[k] - gl[k]), fabsf(y[k])));
            sum += x[k] + rd;
          }
        }
        st_[4] = fabsf(sum * 0.f);
#pragma unroll
        for (int k = 0; k < 5; ++k) {
          const float m = warp_max_nonneg(st_[k]);
          if (lane == 0) s_red[warp * 8 + k] = m;
        }
      }
    }
    __syncthreads();
    if (chk) {
      float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, m4 = 0.f;
#pragma unroll
      for (int wv = 0; wv < LWARPS; ++wv) {
        m0 = fmaxf(m0, s_red[wv * 8 + 0]);
        m1 = fmaxf(m1, s_red[wv * 8 + 1]);
        m2 = fmaxf(m2, s_red[wv * 8 + 2]);
        m3 = fmaxf(m3, s_red[wv * 8 + 3]);
        m4 += s_red[wv * 8 + 4];
      }
      pri = m0;
      dua = m1;
      const float eps_p = p.eps_abs + p.eps_rel * m2;
      const float eps_d = p.eps_abs + p.eps_rel * fmaxf(m3, ng);
      // an invalid body (1/m = NaN, see set_body_kernel), contact or weight set (r_weight = NaN, see
      // set_weights_kernel) fails the problem also when no stance force carries it
      if (!(m4 == 0.f) || !(m0 == m0) || !(m1 == m1) || (BODY && !(im == im)) || (CONTACT && bad_contact) ||
          (WEIGHTS && !(s_wt[13] == s_wt[13])) || (FORCE && !(s_x0[14] == s_x0[14]))) {
        status = -1;
        break;
      }
      if (pri <= eps_p && dua <= eps_d) { status = 1; break; }
      if (it >= p.max_iter) { status = 0; break; }
      if (adapt_now) {
        const float pr_n = m0 / (m2 + 1e-10f);
        const float du_n = m1 / (fmaxf(m3, ng) + 1e-10f);
        float rn = rho * sqrtf(pr_n / (du_n + 1e-10f));
        rn = fminf(fmaxf(rn, p.rho_min), p.rho_max);
        if (fmaxf(pr_n, du_n) > kRhoAdaptFloor &&
            (rn > rho * p.adaptive_rho_tolerance || rn * p.adaptive_rho_tolerance < rho)) {
          rho = rn;
          rho_inv = 1.f / rho;
          factorize();          // uniform: every thread of the CTA sees the same statistics
          continue;             // redo phase A of this iterate with the new factor
        }
      }
    }
    riccati_solve();            // s_s -> s_q  (warp 0; the other warps wait at the barrier)
    __syncthreads();
    if (leg_warp) {
      const int lq = is_leg ? 6 * lj : 0;
      float qv[6];
#pragma unroll
      for (int a = 0; a < 6; ++a) qv[a] = s_q[lq + a];
#pragma unroll
      for (int a = 0; a < 6; ++a) vh[a] = fmaf(alpha, qv[a], vh[a]);
      float w3[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float dl = t[k] - dinv * (Gh[0][k] * qv[0] + Gh[1][k] * qv[1] + Gh[2][k] * qv[2] + im * qv[3 + k]);
        const float xt = x[k] + dl;
        x[k] = fmaf(alpha, dl, x[k]);
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

  // ---- outputs ------------------------------------------------------------------------------
  __syncthreads();
  if (is_leg) {
    s_pre[3 * tid] = x[0]; s_pre[3 * tid + 1] = x[1]; s_pre[3 * tid + 2] = x[2];
    float* wx = p.warm_x + ((size_t)slot * NLEG + tid) * 3;
    wx[0] = x[0]; wx[1] = x[1]; wx[2] = x[2];
    float* wy = p.warm_y + ((size_t)slot * NLEG + tid) * 3;
    wy[0] = y[0]; wy[1] = y[1]; wy[2] = y[2];
  }
  if (tid == 0) {
    if (p.iters) p.iters[b] = it;
    if (p.pri_res) p.pri_res[b] = pri;
    if (p.dua_res) p.dua_res[b] = dua;
    if (p.status) p.status[b] = status;
    p.warm_valid[slot] = status >= 0 ? 1 : 0;
  }
  __syncthreads();
  for (int i = tid; i < 3 * NLEG; i += THREADS) p.U[(size_t)b * 3 * NLEG + i] = s_pre[i];
  if (p.X) {
    store_wrench(x);
    __syncthreads();
    float* c1 = s_pre;                       // [6][N+1]
    float* c2 = s_pre + 6 * (N + 1);
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
    const float g = s_x0[12];
    for (int o = tid; o < NX; o += THREADS) {
      const int k = o / 13, cidx = o % 13;
      const float kf = (float)k;
      float val;
      if (cidx == 12) {
        val = g;
      } else if (cidx < 3) {
        const float rw0 = cidx == 0 ? (cs * s_x0[6] - sn * s_x0[7])
                                    : (cidx == 1 ? (sn * s_x0[6] + cs * s_x0[7]) : s_x0[8]);
        val = s_x0[cidx] + kf * dt * rw0 + dt * dt * c2[cidx * (N + 1) + k];
      } else if (cidx < 6) {
        const int aa = cidx - 3;
        val = s_x0[cidx] + kf * dt * s_x0[9 + aa] + dt * dt * c2[(3 + aa) * (N + 1) + k];
        if (aa == 2) val += 0.5f * kf * (kf - 1.f) * dt * dt * g;
      } else if (cidx < 9) {
        const float sx = c1[k], sy = c1[(N + 1) + k], sz = c1[2 * (N + 1) + k];
        const int aa = cidx - 6;
        const float rot = aa == 0 ? (cs * sx + sn * sy) : (aa == 1 ? (-sn * sx + cs * sy) : sz);
        val = s_x0[cidx] + dt * rot;
      } else {
        const int aa = cidx - 9;
        val = s_x0[cidx] + dt * c1[(3 + aa) * (N + 1) + k];
        if (aa == 2) val += kf * dt * g;
      }
      p.X[(size_t)b * NX + o] = val;
    }
  }
}

}  // namespace cmpc
