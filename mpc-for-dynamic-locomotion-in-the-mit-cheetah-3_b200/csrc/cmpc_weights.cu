// cmpc_weights.cu - per-robot cost weights (cmpc_set_weights, cmpc_set_stage_weights): the kernels that store them,
// and the BODY + WEIGHTS and
// BODY + CONTACT + WEIGHTS solve kernels (solve_rows<true, false, true> and <true, true, true>).  A translation unit
// of its own so that the kernels of cmpc.cu, cmpc_body.cu and cmpc_contact.cu compile exactly as they do without
// these (see solve_rows in cmpc_launch.cuh).
#define CMPC_SOLVE_KERNELS_ONLY   // the other kernels of cmpc_kernels.cuh are defined in cmpc.cu
#include "cmpc_launch.cuh"

namespace cmpc {

template const SolveRow* solve_rows<true, false, true>();
template const SolveRow* solve_rows<true, true, true>();

// the state before any cmpc_set_weights: every slot holds the handle's record and Gram tables
__global__ void __launch_bounds__(256) init_weights_kernel(float4* __restrict__ weights, float* __restrict__ w_Minv,
                                                           float* __restrict__ w_Mg, float4 r0, float4 r1, float4 r2,
                                                           float4 r3, const float* __restrict__ Minv,
                                                           const float* __restrict__ Mg, int slots, int per_slot) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (long long)slots * kWeightF4) {
    const int q = (int)(i % kWeightF4);
    weights[i] = q == 0 ? r0 : (q == 1 ? r1 : (q == 2 ? r2 : r3));
  }
  if (w_Minv && i < (long long)slots * per_slot) {
    const int e = (int)(i % per_slot);
    w_Minv[i] = Minv[e];
    w_Mg[i] = Mg[e];
  }
}

// Store the weights of slots [slot0, slot0 + B) (cmpc_set_weights, cmpc_set_stage_weights) and invalidate their
// cached factors, which were computed with the previous M^-1 and r_weight.  Stage k's weights are row k - 1 of the
// slot's rows in w, ws floats apart: ws = 0 gives every stage the slot's one row (cmpc_set_weights).  One CTA per
// slot, warp a builds axis a: the Gram matrix M_a of the user horizon N (axis_gram in cmpc.cu, with stage k's
// weights in term k) and its inverse by the Gauss-Jordan loop of cmpc_create, in fp64 with the operations in the
// host's order, each rounded on its own (no contraction into DFMA), so that the configuration's weights give the
// handle's Mg / Minv bit for bit.  Lane i owns row i of the augmented matrix [M | I] in shared memory.  Both are
// rounded to fp32 and embedded as blockdiag(M_N, I) on a padded horizon; without tables (w_Minv = nullptr) only the
// left half is eliminated, for the pivot test.  A handle with stage weights (wstage != nullptr) also receives every
// stage's w[0..11] there (the padding stages keep their zeros); the record keeps stage 1's row.  A slot whose weights
// are invalid (an entry of w on some stage or r_weight non-finite or negative, w[6] != w[7] on some stage, or a pivot
// of some axis not finite and positive, as cmpc_create tests it) is stored with r_weight = NaN, which every solve of
// the slot reports through its non-finite guard.
__global__ void __launch_bounds__(192) set_weights_kernel(const float* __restrict__ w, int32_t ws,
                                                          const float* __restrict__ r_weight,
                                                          float4* __restrict__ weights, float4* __restrict__ wstage,
                                                          float* __restrict__ w_Minv, float* __restrict__ w_Mg,
                                                          float* __restrict__ cache_meta, int32_t slot0, int32_t N,
                                                          int32_t NK, float dt) {
  extern __shared__ double s_aug[];   // [6][N][W]
  const int b = blockIdx.x, slot = slot0 + b;
  const int a = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool tables = w_Minv != nullptr;
  const int W = tables ? 2 * N : N;
  double* A = s_aug + (size_t)a * N * W;
  const float* wb = w + (size_t)b * (ws ? (size_t)ws * N : 13);   // the slot's rows
  float wl[13];
  bool ok = true;
#pragma unroll
  for (int i = 0; i < 13; ++i) {
    wl[i] = __ldg(wb + i);
    ok = ok && isfinite(wl[i]) && wl[i] >= 0.f;
  }
  const float rw = __ldg(r_weight + b);
  ok = ok && wl[6] == wl[7] && isfinite(rw) && rw >= 0.f;
  if (ws) {   // the other stages' rows, then CTA-uniform
    for (int e = threadIdx.x; e < ws * N; e += blockDim.x) {
      const float v = __ldg(wb + e);
      ok = ok && isfinite(v) && v >= 0.f && (e % ws != 6 || v == __ldg(wb + e + 1));
    }
    ok = __syncthreads_and(ok) != 0;
  }
  if (wstage) {
    float* t = reinterpret_cast<float*>(wstage + (size_t)slot * NK * kStageF4);
    for (int e = threadIdx.x; e < 12 * N; e += blockDim.x) t[e] = __ldg(wb + ws * (e / 12) + e % 12);
  }
  bool pd = true;
  if (ok) {   // CTA-uniform
    const double dd = dt;
    const float* wa = wb + a;   // stage k: wa[ws (k - 1)] position-like, wa[ws (k - 1) + 6] velocity-like
    const size_t tab = ((size_t)slot * 6 + a) * NK * NK;
    // M_a[j][j2] = 2 sum_{k > max(j, j2)}^{N} (w_pos,k dt^4 (k-1-j)(k-1-j2) + w_vel,k dt^2)
    for (int i = lane; i < N; i += 32) {
      for (int j2 = 0; j2 < N; ++j2) {
        double acc = 0.0;
        for (int k = (i > j2 ? i : j2) + 1; k <= N; ++k) {
          const double wp = __ldg(wa + ws * (k - 1)), wv = __ldg(wa + ws * (k - 1) + 6);
          const double t1 = __dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn(wp, dd), dd), dd), dd),
                                                (double)(k - 1 - i)), (double)(k - 1 - j2));
          acc = __dadd_rn(acc, __dadd_rn(t1, __dmul_rn(__dmul_rn(wv, dd), dd)));
        }
        const double m = __dmul_rn(2.0, acc);
        A[(size_t)i * W + j2] = m;
        if (tables) w_Mg[tab + (size_t)i * NK + j2] = (float)m;
      }
      if (tables)
        for (int j = 0; j < N; ++j) A[(size_t)i * W + N + j] = i == j ? 1.0 : 0.0;
    }
    __syncwarp();
    for (int k = 0; k < N; ++k) {
      const double piv = A[(size_t)k * W + k];
      if (!(piv > 0.0) || !isfinite(piv)) { pd = false; break; }   // warp-uniform
      __syncwarp();
      for (int j = lane; j < W; j += 32) A[(size_t)k * W + j] = __ddiv_rn(A[(size_t)k * W + j], piv);
      __syncwarp();
      for (int i = lane; i < N; i += 32) {
        if (i == k) continue;
        const double f = A[(size_t)i * W + k];
        if (f == 0.0) continue;
        for (int j = 0; j < W; ++j)
          A[(size_t)i * W + j] = __dsub_rn(A[(size_t)i * W + j], __dmul_rn(f, A[(size_t)k * W + j]));
      }
      __syncwarp();
    }
    if (tables && pd) {
      for (int e = lane; e < NK * NK; e += 32) {
        const int i = e / NK, j = e - i * NK;
        if (i < N && j < N) w_Minv[tab + e] = (float)A[(size_t)i * W + N + j];
        else w_Minv[tab + e] = i == j ? 1.f : 0.f;
      }
      // the padding rows and columns of M (its N x N block was written above)
      for (int e = lane; e < NK * NK; e += 32) {
        const int i = e / NK, j = e - i * NK;
        if (i >= N || j >= N) w_Mg[tab + e] = i == j ? 1.f : 0.f;
      }
    }
  }
  const bool valid = __syncthreads_and(ok && pd) != 0;
  if (threadIdx.x == 0) {
    float4* d = weights + (size_t)slot * kWeightF4;
    d[0] = make_float4(wl[0], wl[1], wl[2], wl[3]);
    d[1] = make_float4(wl[4], wl[5], wl[6], wl[7]);
    d[2] = make_float4(wl[8], wl[9], wl[10], wl[11]);
    d[3] = make_float4(wl[12], valid ? rw : __int_as_float(0x7fc00000), 0.f, 0.f);
    if (cache_meta) cache_meta[(size_t)slot * 4 + 2] = 0.f;
  }
}

cudaError_t init_weights(float4* weights, float* w_Minv, float* w_Mg, const float rec[4 * kWeightF4],
                         const float* Minv, const float* Mg, int slots, int NK, cudaStream_t s) {
  const int per_slot = 6 * NK * NK;
  const long long items = (long long)slots * (w_Minv ? per_slot : kWeightF4);
  init_weights_kernel<<<(unsigned)((items + 255) / 256), 256, 0, s>>>(
      weights, w_Minv, w_Mg, make_float4(rec[0], rec[1], rec[2], rec[3]), make_float4(rec[4], rec[5], rec[6], rec[7]),
      make_float4(rec[8], rec[9], rec[10], rec[11]), make_float4(rec[12], rec[13], rec[14], rec[15]), Minv, Mg, slots,
      per_slot);
  return cudaGetLastError();
}

cudaError_t store_weights(const float* w, int ws, const float* r_weight, float4* weights, float4* wstage,
                          float* w_Minv, float* w_Mg, float* cache_meta, int slot0, int B, int N, int NK, float dt,
                          int dev, cudaStream_t s) {
  // the augmented matrices of the six axes: 6 N 2N doubles (86 KB at N = 30), or 6 N^2 without tables (173 KB at
  // N = 60), above the 48 KB default
  constexpr int kMaxSmem = 6 * 60 * 60 * (int)sizeof(double);
  static PerDevice setup;
  const cudaError_t e = set_up_once(setup, dev, [&](int&, int&) {
    return cudaFuncSetAttribute(set_weights_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
  });
  if (e != cudaSuccess) return e;
  const size_t smem = (size_t)6 * N * (w_Minv ? 2 * N : N) * sizeof(double);
  set_weights_kernel<<<(unsigned)B, 192, smem, s>>>(w, ws, r_weight, weights, wstage, w_Minv, w_Mg, cache_meta, slot0,
                                                     N, NK, dt);
  return cudaGetLastError();
}

// the state before any cmpc_set_stage_weights: every stage of a slot holds its weight record's w[0..11], the padding
// stages of a padded horizon zeros
__global__ void __launch_bounds__(256) init_stage_weights_kernel(float4* __restrict__ wstage,
                                                                 const float4* __restrict__ weights, int slots, int N,
                                                                 int NK) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)slots * NK * kStageF4) return;
  const int q = (int)(i % kStageF4), k = (int)((i / kStageF4) % NK);
  const long long slot = i / ((long long)NK * kStageF4);
  wstage[i] = k < N ? weights[slot * kWeightF4 + q] : make_float4(0.f, 0.f, 0.f, 0.f);
}

cudaError_t init_stage_weights(float4* wstage, const float4* weights, int slots, int N, int NK, cudaStream_t s) {
  const long long items = (long long)slots * NK * kStageF4;
  init_stage_weights_kernel<<<(unsigned)((items + 255) / 256), 256, 0, s>>>(wstage, weights, slots, N, NK);
  return cudaGetLastError();
}

}  // namespace cmpc
