// SPDX-License-Identifier: MIT
// Blocked symmetric sweep of one problem's Jacobi-scaled matrix A = S P S (6N <= 64 rows) on the
// tensor cores: the factorisation step of solve_kernel<..., TC = true>.
//
// The SIMT sweep of cmpc_kernels.cuh eliminates one pivot per barrier (a rank-1 update of rows
// held in registers, the pivot row broadcast through shared memory).  Here eight pivots are
// eliminated at a time:
//     L = A[:, k] - E_k,   A_kk = Lc Lc',   Y = L Lc^-T,   A <- A - Y Y'            (k = 0 .. 7)
// which is the same sweep operator applied blockwise (A_kk -> 2I - A_kk^-1, A_ik -> A_ik A_kk^-1,
// A_ij -> A_ij - A_ik A_kk^-1 A_kj), so that after the eight steps A = 2I - A^-1.  The rank-8 update is
// `mma.sync.m16n8k8` TF32 with the 3xTF32 split (Y = hi + lo, hi*hi + lo*hi + hi*lo, fp32 accumulate:
// products exact to ~2^-22) on the matrix kept in accumulator fragments: 2 warps x (32 rows x 64
// columns) = 64 registers per thread.  Both operands come from the same 64 x 8 panel Y in shared
// memory through `ldmatrix` (a 32-bit word is two b16 "elements": tile i of an .x4 load gives lane l
// the word (row l/4, col l%4), which is exactly the TF32 A / B fragment).  The 8 x 8 Cholesky and
// the triangular solve of the own row are done redundantly by every thread (no exchange, one
// barrier after the panel is published and one after Y is stored).
//
// tcgen05 / TMEM does not apply (one 64 x 64 matrix per CTA of 64 threads, no operand shared
// between problems, M < 64-row UMMA shapes); the legacy tensor path measured 0.46 HMMA.1688.TF32 per
// SM-cycle on B200 (scripts/micro/mma_sweep.cu) and is 12 % busy over a config-2 launch (ncu).
// Measured inside solve_kernel (clock64 phase stamps, staging included): 11.9 k cycles per sweep alone on
// an SM and 19.6 k on a loaded one, against 20.3 k / 38 k for the SIMT sweep; accuracy 1.5e-4 of
// max|A^-1| at condition numbers 1e3..1e4 (host fp32 Gauss-Jordan: 0.6e-4), absorbed by the
// residual-correction form of the ADMM iteration like the SIMT sweep's own rounding.
#pragma once

#include <cstdint>

namespace cmpc {

constexpr int kTcN = 64;                        // padded matrix size (rows 6N .. 63: identity)
constexpr int kTcPS = 68;                       // row stride (words) of the row <-> fragment staging area
constexpr int kTcYS = 12;                       // row stride of the panel Y: ldmatrix rows on 8 distinct bank groups
// staging rows of one matrix: the identity padding rows are generated in registers, not staged, so that 8 CTAs
// (this area + 7.4 KB of solver state + 1 KB reserved each) fit the 196 KB shared-memory carve-out and leave
// 60 KB of L1 to the register spills of the ADMM loop (measured: with the 228 KB carve-out they go to L2)
template <int NW>
__host__ __device__ constexpr int tc_smem_floats() { return NW * kTcPS > kTcN * (8 + 2 * kTcYS) ? NW * kTcPS : kTcN * (8 + 2 * kTcYS); }

__device__ __forceinline__ float tf32_round(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t* a, const uint32_t* b) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// four 8 x 4 tiles of 32-bit words; lanes 8i .. 8i+7 supply the row addresses of tile i
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const float* p) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}

// Called by all 64 threads of the CTA (two full warps: mma.sync / ldmatrix are warp-collective).
//   in : row[0 .. NW) = row `tid` of A (unit diagonal) for tid < NW; threads NW .. 63 own the identity padding
//   out: row[0 .. NW) = row `tid` of -A^-1
// sP: tc_smem_floats<NW>() floats of shared memory, 16-byte aligned, owned by this call between its barriers.
template <int NW, int NWP>
__device__ __forceinline__ void tc_sweep(float (&row)[NWP], float* __restrict__ sP, const int tid) {
  static_assert(NW <= kTcN && NW % 4 == 0 && NWP >= NW, "one 64 x 64 fragment matrix per CTA");
  const int lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
  // ---- rows -> staging area, negated: the accumulators hold -A, so the update is acc += Y Y' ----
  if (tid < NW) {
    float* mine = sP + tid * kTcPS;
#pragma unroll
    for (int c = 0; c < NW; c += 4)
      *reinterpret_cast<float4*>(mine + c) = make_float4(-row[c], -row[c + 1], -row[c + 2], -row[c + 3]);
#pragma unroll
    for (int c = NW; c < kTcN; c += 4) *reinterpret_cast<float4*>(mine + c) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  float acc[2][8][4];       // rows 32w + 16mt + {g, g+8}, columns 8nt + {2t, 2t+1}
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int r0 = 32 * w + 16 * mt + g, r1 = r0 + 8, c0 = 8 * nt + 2 * t;
      // rows >= NW are the identity padding (-I in the negated matrix)
      const float2 u = r0 < NW ? *reinterpret_cast<const float2*>(sP + r0 * kTcPS + c0)
                               : make_float2(r0 == c0 ? -1.f : 0.f, r0 == c0 + 1 ? -1.f : 0.f);
      const float2 v = r1 < NW ? *reinterpret_cast<const float2*>(sP + r1 * kTcPS + c0)
                               : make_float2(r1 == c0 ? -1.f : 0.f, r1 == c0 + 1 ? -1.f : 0.f);
      acc[mt][nt][0] = u.x; acc[mt][nt][1] = u.y; acc[mt][nt][2] = v.x; acc[mt][nt][3] = v.y;
    }
  __syncthreads();          // the staging area becomes the panels
  float* sL = sP;                               // [64][8]   column block k of -A
  float* sYh = sP + kTcN * 8;                   // [64][12]  tf32(Y)
  float* sYl = sYh + kTcN * kTcYS;              // [64][12]  tf32(Y - tf32(Y))
  // ldmatrix row addresses of this lane.  A operand: tiles (rows 0-7 | 8-15) x (words 0-3 | 4-7) of a
  // 16-row group; B operand: two 8-row groups x (words 0-3 | 4-7) -> (b0, b1) of two column tiles
  const int a_off = (32 * w + (lane & 7) + 8 * ((lane >> 3) & 1)) * kTcYS + 4 * (lane >> 4);
  const int b_off = (8 * (lane >> 4) + (lane & 7)) * kTcYS + 4 * ((lane >> 3) & 1);
#pragma unroll 1
  for (int k = 0; k < 8; ++k) {
    // a. publish column block k (predicated stores: no dynamically indexed register array)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
      if (nt == k) {
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          float* q = sL + (32 * w + 16 * mt + g) * 8 + 2 * t;
          *reinterpret_cast<float2*>(q) = make_float2(acc[mt][nt][0], acc[mt][nt][1]);
          *reinterpret_cast<float2*>(q + 64) = make_float2(acc[mt][nt][2], acc[mt][nt][3]);
        }
      }
    __syncthreads();
    // b. Cholesky A_kk = Lc Lc' (redundantly in every thread), then the own row of Y = L Lc^-T
    float lc[8][8], inv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 lo = *reinterpret_cast<const float4*>(sL + (8 * k + i) * 8);
      const float4 hi = *reinterpret_cast<const float4*>(sL + (8 * k + i) * 8 + 4);
      lc[i][0] = -lo.x; lc[i][1] = -lo.y; lc[i][2] = -lo.z; lc[i][3] = -lo.w;
      lc[i][4] = -hi.x; lc[i][5] = -hi.y; lc[i][6] = -hi.z; lc[i][7] = -hi.w;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float s = lc[j][j];
#pragma unroll
      for (int m = 0; m < j; ++m) s = fmaf(-lc[j][m], lc[j][m], s);
      inv[j] = rsqrtf(s);
#pragma unroll
      for (int i = j + 1; i < 8; ++i) {
        float v = lc[i][j];
#pragma unroll
        for (int m = 0; m < j; ++m) v = fmaf(-lc[i][m], lc[j][m], v);
        lc[i][j] = v * inv[j];
      }
    }
    float y[8];
    {
      const float4 lo = *reinterpret_cast<const float4*>(sL + tid * 8);
      const float4 hi = *reinterpret_cast<const float4*>(sL + tid * 8 + 4);
      y[0] = -lo.x; y[1] = -lo.y; y[2] = -lo.z; y[3] = -lo.w; y[4] = -hi.x; y[5] = -hi.y; y[6] = -hi.z; y[7] = -hi.w;
    }
    const int own = tid - 8 * k;                 // L = A[:, k] - E_k: minus one on the block's own diagonal
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = y[j] - (own == j ? 1.f : 0.f);
#pragma unroll
      for (int m = 0; m < j; ++m) v = fmaf(-y[m], lc[j][m], v);
      y[j] = v * inv[j];
    }
    float yh[8], yl[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      yh[j] = tf32_round(y[j]);
      yl[j] = tf32_round(y[j] - yh[j]);
    }
    *reinterpret_cast<float4*>(sYh + tid * kTcYS) = make_float4(yh[0], yh[1], yh[2], yh[3]);
    *reinterpret_cast<float4*>(sYh + tid * kTcYS + 4) = make_float4(yh[4], yh[5], yh[6], yh[7]);
    *reinterpret_cast<float4*>(sYl + tid * kTcYS) = make_float4(yl[0], yl[1], yl[2], yl[3]);
    *reinterpret_cast<float4*>(sYl + tid * kTcYS + 4) = make_float4(yl[4], yl[5], yl[6], yl[7]);
    __syncthreads();
    // c. rank-8 update (-A) += Y Y'
    uint32_t ah[2][4], al[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      ldmatrix_x4(ah[mt], sYh + a_off + 16 * mt * kTcYS);
      ldmatrix_x4(al[mt], sYl + a_off + 16 * mt * kTcYS);
    }
#pragma unroll
    for (int np = 0; np < 4; ++np) {             // two column tiles per ldmatrix.x4
      uint32_t bh[4], bl[4];
      ldmatrix_x4(bh, sYh + b_off + 16 * np * kTcYS);
      ldmatrix_x4(bl, sYl + b_off + 16 * np * kTcYS);
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          mma_tf32(acc[mt][2 * np + h], al[mt], bh + 2 * h);
          mma_tf32(acc[mt][2 * np + h], ah[mt], bl + 2 * h);
          mma_tf32(acc[mt][2 * np + h], ah[mt], bh + 2 * h);
        }
    }
  }
  // ---- fragments -> staging area -> rows:  acc = A^-1 - 2I ----
  __syncthreads();
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int r0 = 32 * w + 16 * mt + g, r1 = r0 + 8;
      float* q = sP + r0 * kTcPS + 8 * nt + 2 * t;
      if (r0 < NW) *reinterpret_cast<float2*>(q) = make_float2(acc[mt][nt][0], acc[mt][nt][1]);
      if (r1 < NW) *reinterpret_cast<float2*>(q + 8 * kTcPS) = make_float2(acc[mt][nt][2], acc[mt][nt][3]);
    }
  __syncthreads();
  {   // every thread (the padding threads re-read the last row): `row` must be dead across the sweep, it shares
      // the register file with acc
    const float* mine = sP + (tid < NW ? tid : NW - 1) * kTcPS;
#pragma unroll
    for (int c = 0; c < NW; c += 4) {
      const float4 v = *reinterpret_cast<const float4*>(mine + c);
      row[c] = -v.x - (c == tid ? 2.f : 0.f);
      row[c + 1] = -v.y - (c + 1 == tid ? 2.f : 0.f);
      row[c + 2] = -v.z - (c + 2 == tid ? 2.f : 0.f);
      row[c + 3] = -v.w - (c + 3 == tid ? 2.f : 0.f);
    }
  }
}

}  // namespace cmpc
