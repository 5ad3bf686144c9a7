// cmpc_wrench.cu - per-robot external wrench (cmpc_set_wrench): the kernel that stores it, and the pre- and post-pass
// of a solve around the unchanged solve kernels.  A known wrench changes only the free response of x0, by its forced
// response phi (wrench_response), so the QP with the wrench is the QP without it on x_des - phi, and its predicted
// states are that QP's X + phi (DESIGN.md section 4).  A translation unit of its own so that the kernels of the other
// modules compile exactly as they do without these (see solve_rows in cmpc_launch.cuh).
#define CMPC_SOLVE_KERNELS_ONLY   // the other kernels of cmpc_kernels.cuh are defined in cmpc.cu
#include "cmpc_launch.cuh"

namespace cmpc {

namespace {
constexpr int kWrenchThreads = 64;   // one CTA per problem, a thread per stage (horizons up to 60)
constexpr int kWrenchMaxN = 60;
}  // namespace

// store the wrenches of slots [slot0, slot0 + B), N stages each (cmpc_set_wrench): one warp per slot.  A slot with a
// non-finite entry is stored as NaN throughout, so that its shifted x_des is NaN and wrench_finish_kernel reports it.
__global__ void __launch_bounds__(128) set_wrench_kernel(const float* __restrict__ force,
                                                         const float* __restrict__ torque, float* __restrict__ wrench,
                                                         int32_t slot0, int32_t B, int32_t N) {
  const int b = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;   // whole warps
  const float* f = force + (size_t)b * 3 * N;
  const float* t = torque + (size_t)b * 3 * N;
  bool bad = false;
  for (int i = lane; i < 3 * N; i += 32) bad = bad || !isfinite(f[i]) || !isfinite(t[i]);
  bad = __any_sync(0xffffffffu, bad);
  float* d = wrench + (size_t)(slot0 + b) * 6 * N;
  for (int i = lane; i < 6 * N; i += 32) {
    const int j = i / 6, c = i - 6 * j;
    d[i] = bad ? __int_as_float(0x7fc00000) : (c < 3 ? f[3 * j + c] : t[3 * j + c - 3]);
  }
}

// the problem's wrench record, body and yaw in shared memory
__device__ __forceinline__ void load_wrench(const WrenchParams& p, int b, float* s_eps, float* s_bd, float& c,
                                            float& s) {
  const float* e = p.wrench + (size_t)b * 6 * p.N;
  for (int i = threadIdx.x; i < 6 * p.N; i += blockDim.x) s_eps[i] = __ldg(e + i);
  if (threadIdx.x < 4 * kBodyF4) s_bd[threadIdx.x] = __ldg(reinterpret_cast<const float*>(p.body + (size_t)b * kBodyF4) + threadIdx.x);
  sincosf(p.x0[(size_t)b * 13 + 2], &s, &c);
  __syncthreads();
}

// x_des_out = x_des - phi over the kernel horizon's NK + 1 stages.  An entry with phi == 0 is copied, so that a zero
// wrench gives the caller's x_des bit for bit (x - (-0) would turn -0 into +0).  In place on a padded horizon.
__global__ void __launch_bounds__(kWrenchThreads) wrench_shift_kernel(const WrenchParams p) {
  __shared__ float s_eps[6 * kWrenchMaxN];
  __shared__ float s_bd[4 * kBodyF4];
  __shared__ float s_phi[kWrenchMaxN + 1][12];
  const int b = blockIdx.x;
  grid_dependency_wait();   // pad_kernel's output
  float c, s;
  load_wrench(p, b, s_eps, s_bd, c, s);
  for (int k = threadIdx.x; k <= p.NK; k += blockDim.x)
    wrench_response(k, p.N, s_eps, c, s, p.dt, s_bd[0], s_bd + 1, s_phi[k]);
  __syncthreads();
  const int NX = 13 * (p.NK + 1);
  const float* xd = p.x_des + (size_t)b * NX;
  float* out = p.x_des_out + (size_t)b * NX;
  for (int i = threadIdx.x; i < NX; i += blockDim.x) {
    const int k = i / 13, cidx = i - 13 * k;
    float v = xd[i];
    const float ph = cidx < 12 ? s_phi[k][cidx] : 0.f;
    if (ph != 0.f) v -= ph;
    out[i] = v;
  }
}

// After the solve (and unpad_kernel): X += phi over the N + 1 stages of the caller's X (entries with phi == 0 are
// left alone, as above), and CMPC_STATUS_NAN for a slot stored with an invalid wrench.  The solve kernels report its
// NaN x_des themselves when a stance force carries it, but not for an all-swing problem, whose QP has no unknowns.
__global__ void __launch_bounds__(kWrenchThreads) wrench_finish_kernel(const WrenchParams p) {
  __shared__ float s_eps[6 * kWrenchMaxN];
  __shared__ float s_bd[4 * kBodyF4];
  __shared__ float s_phi[kWrenchMaxN + 1][12];
  const int b = blockIdx.x;
  float c, s;
  load_wrench(p, b, s_eps, s_bd, c, s);
  if (p.status && threadIdx.x == 0 && s_eps[0] != s_eps[0]) p.status[b] = -1;   // CMPC_STATUS_NAN
  if (!p.X) return;
  for (int k = threadIdx.x; k <= p.N; k += blockDim.x)
    wrench_response(k, p.N, s_eps, c, s, p.dt, s_bd[0], s_bd + 1, s_phi[k]);
  __syncthreads();
  const int NX = 13 * (p.N + 1);
  float* X = p.X + (size_t)b * NX;
  for (int i = threadIdx.x; i < NX; i += blockDim.x) {
    const int k = i / 13, cidx = i - 13 * k;
    const float ph = cidx < 12 ? s_phi[k][cidx] : 0.f;
    if (ph != 0.f) X[i] += ph;
  }
}

cudaError_t store_wrench(const float* force, const float* torque, float* wrench, int slot0, int B, int N,
                         cudaStream_t s) {
  set_wrench_kernel<<<(unsigned)(((size_t)B * 32 + 127) / 128), 128, 0, s>>>(force, torque, wrench, slot0, B, N);
  return cudaGetLastError();
}

cudaError_t wrench_shift(const WrenchParams& p, cudaStream_t s) {
  return launch_pdl(wrench_shift_kernel, dim3((unsigned)p.B), dim3(kWrenchThreads), 0, s, p);
}

cudaError_t wrench_finish(const WrenchParams& p, cudaStream_t s) {
  wrench_finish_kernel<<<(unsigned)p.B, kWrenchThreads, 0, s>>>(p);
  return cudaGetLastError();
}

}  // namespace cmpc
