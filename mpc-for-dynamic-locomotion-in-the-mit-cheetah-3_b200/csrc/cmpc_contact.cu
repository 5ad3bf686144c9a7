// cmpc_contact.cu - per-foot contact surfaces (cmpc_set_contact): the kernels that store them, and the BODY + CONTACT
// solve kernels (solve_rows<true, true, false>), projecting each leg-stage onto its own contact surface.  A
// translation unit of its own so that the kernels of cmpc.cu and cmpc_body.cu compile exactly as they do without
// these (see solve_rows in cmpc_launch.cuh).
#define CMPC_SOLVE_KERNELS_ONLY   // the other kernels of cmpc_kernels.cuh are defined in cmpc.cu
#include "cmpc_launch.cuh"

namespace cmpc {

template const SolveRow* solve_rows<true, true, false>();

// the contact array's state before any cmpc_set_contact: world axes, mu < 0 (the call's mu), the
// configuration's bounds, for n leg-stages
__global__ void __launch_bounds__(256) init_contact_kernel(float4* __restrict__ contact, float f_min, float f_max,
                                                           size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  contact[i * kContactF4] = make_float4(0.f, 0.f, 1.f, -1.f);
  contact[i * kContactF4 + 1] = make_float4(f_min, f_max, 0.f, 0.f);
}

// store the contacts of slots [slot0, slot0 + B), stages [0, N) at the kernel horizon's stride NK
// (cmpc_set_contact): the unit normal, mu and the bounds.  A leg-stage whose normal is non-finite or shorter
// than 1e-6, whose mu is non-finite or negative, or whose bounds are not finite with 0 <= f_min <= f_max, is
// stored with mu = NaN, which every solve of the slot reports through its non-finite guard.
__global__ void __launch_bounds__(256) set_contact_kernel(const float* __restrict__ normal,
                                                          const float* __restrict__ mu,
                                                          const float* __restrict__ f_min,
                                                          const float* __restrict__ f_max,
                                                          float4* __restrict__ contact, int32_t slot0, int32_t B,
                                                          int32_t N, int32_t NK) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // (b, stage, leg)
  if (i >= (long long)B * N * 4) return;
  const long long b = i / (4 * N), jl = i - b * 4 * N;
  float nx = normal[3 * i], ny = normal[3 * i + 1], nz = normal[3 * i + 2];
  const float m = mu[i], lo = f_min[i], hi = f_max[i];
  // scaled by the largest component first, so that any finite normal normalises without overflow and
  // (0, 0, c > 0) gives (0, 0, 1) exactly
  const float s = fmaxf(fabsf(nx), fmaxf(fabsf(ny), fabsf(nz)));
  bool ok = isfinite(nx) && isfinite(ny) && isfinite(nz) && s > 0.f;
  if (ok) {
    nx /= s; ny /= s; nz /= s;
    const float len = sqrtf(nx * nx + ny * ny + nz * nz);
    ok = s * len >= 1e-6f;
    nx /= len; ny /= len; nz /= len;
  }
  ok = ok && isfinite(m) && m >= 0.f && isfinite(lo) && isfinite(hi) && lo >= 0.f && lo <= hi;
  float4* d = contact + ((size_t)(slot0 + b) * NK * 4 + jl) * kContactF4;
  d[0] = ok ? make_float4(nx, ny, nz, m) : make_float4(0.f, 0.f, 1.f, __int_as_float(0x7fc00000));
  d[1] = make_float4(lo, hi, 0.f, 0.f);
}

cudaError_t init_contact(float4* contact, float f_min, float f_max, size_t n, cudaStream_t s) {
  init_contact_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(contact, f_min, f_max, n);
  return cudaGetLastError();
}

cudaError_t store_contact(const float* normal, const float* mu, const float* f_min, const float* f_max,
                          float4* contact, int slot0, int B, int N, int NK, cudaStream_t s) {
  const long long items = (long long)B * N * 4;
  set_contact_kernel<<<(unsigned)((items + 255) / 256), 256, 0, s>>>(normal, mu, f_min, f_max, contact, slot0, B, N,
                                                                     NK);
  return cudaGetLastError();
}

}  // namespace cmpc
