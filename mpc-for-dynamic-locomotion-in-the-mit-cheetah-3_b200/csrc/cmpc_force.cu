// cmpc_force.cu - per-robot force references (cmpc_set_force_ref): the kernel that stores them, and the
// BODY + WEIGHTS + FORCE and BODY + CONTACT + WEIGHTS + FORCE solve kernels (solve_rows<true, false, true, true> and
// <true, true, true, true>).  A translation unit of its own so that the kernels of the other modules compile exactly
// as they do without these (see solve_rows in cmpc_launch.cuh).
#define CMPC_SOLVE_KERNELS_ONLY   // the other kernels of cmpc_kernels.cuh are defined in cmpc.cu
#include "cmpc_launch.cuh"

namespace cmpc {

template const SolveRow* solve_rows<true, false, true, true>();
template const SolveRow* solve_rows<true, true, true, true>();

// Store the force references of slots [slot0, slot0 + B), stages [0, N) at the kernel horizon's stride NK
// (cmpc_set_force_ref), one warp per slot, and invalidate the slots' cached factors, which depend on d_l.  The
// padding stages of a padded horizon keep the zeros of the first call.  A slot with a non-finite f_ref or a
// non-finite or negative weight anywhere is stored with w_f = NaN on every leg-stage, so that every solve of it
// reports CMPC_STATUS_NAN, an all-swing one included (the solve kernels test leg-stage 0).
__global__ void __launch_bounds__(128) set_force_ref_kernel(const float* __restrict__ f_ref,
                                                            const float* __restrict__ weight,
                                                            float4* __restrict__ force, float* __restrict__ cache_meta,
                                                            int32_t slot0, int32_t B, int32_t N, int32_t NK) {
  const int b = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;   // whole warps
  const float* f = f_ref + (size_t)b * 12 * N;
  const float* w = weight + (size_t)b * 4 * N;
  bool bad = false;
  for (int i = lane; i < 4 * N; i += 32)
    bad = bad || !isfinite(f[3 * i]) || !isfinite(f[3 * i + 1]) || !isfinite(f[3 * i + 2]) || !isfinite(w[i]) ||
          !(w[i] >= 0.f);
  bad = __any_sync(0xffffffffu, bad);
  float4* d = force + (size_t)(slot0 + b) * 4 * NK;
  for (int i = lane; i < 4 * N; i += 32)
    d[i] = make_float4(f[3 * i], f[3 * i + 1], f[3 * i + 2], bad ? __int_as_float(0x7fc00000) : w[i]);
  if (cache_meta && lane == 0) cache_meta[(size_t)(slot0 + b) * 4 + 2] = 0.f;
}

cudaError_t store_force_ref(const float* f_ref, const float* weight, float4* force, float* cache_meta, int slot0, int B,
                            int N, int NK, cudaStream_t s) {
  set_force_ref_kernel<<<(unsigned)(((size_t)B * 32 + 127) / 128), 128, 0, s>>>(f_ref, weight, force, cache_meta, slot0,
                                                                                B, N, NK);
  return cudaGetLastError();
}

}  // namespace cmpc
