// Device helpers shared by the K2 kernels (K2p, K2c, SYRK, finalize; see k2_frames.cu for the math).
#pragma once
#include "mcba_internal.h"
#include "mcba_obs.cuh"

namespace mcba {

// Bulk async copies into shared memory, completed on an mbarrier (K2c, SYRK, back-substitution).
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// FP64 tensor path: C (8 x 8, two values per lane) += A (8 x 4) B (4 x 8), one value of each per lane (SYRK, solve).
__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__host__ __device__ constexpr int tri12(int i, int j) { return i * 12 - (i * (i - 1)) / 2 + (j - i); }
__host__ __device__ constexpr int sym12(int i, int j) { return i <= j ? tri12(i, j) : tri12(j, i); }
__host__ __device__ constexpr int tri6(int i, int j) { return i * 6 - (i * (i - 1)) / 2 + (j - i); }
__host__ __device__ constexpr int sym6(int i, int j) { return i <= j ? tri6(i, j) : tri6(j, i); }
// Accumulator layout of the raw 12x12 Gauss-Newton block A_cf and q_cf (kAcc = 128 slots, 4
// blocks of 32 for the lane transpose-reduction); raw column order of mcba_obs.cuh
// [fx fy cx cy k1 k2 | m (3) | G (3)]:
//   block 0: entries only the u rows touch (columns fx, cx):  19 of A + 2 of q
//   block 1: entries only the v rows touch (columns fy, cy):  19 of A + 2 of q
//   blocks 2-3: entries both rows touch (columns k1, k2, ext): 36 of A + 8 of q
// The four products fx.fy, fx.cy, cx.fy, cx.cy are structurally zero and have no slot (-1).
__host__ __device__ constexpr int tri8(int i, int j) { return i * 8 - (i * (i - 1)) / 2 + (j - i); }
__host__ __device__ constexpr int acc_slot_upper(int I, int J) {   // I <= J
  const bool Iu = I == 0 || I == 2, Iv = I == 1 || I == 3;
  const bool Ju = J == 0 || J == 2, Jv = J == 1 || J == 3;
  if ((Iu && Jv) || (Iv && Ju)) return -1;
  if (Iu || Iv) {
    const int base = Iu ? 0 : 32;
    if (Ju || Jv) return base + (I < 2 ? (J < 2 ? 0 : 1) : 2);   // (f,f) (f,c) (c,c)
    return base + (I < 2 ? 3 : 11) + (J - 4);
  }
  return 64 + tri8(I - 4, J - 4);
}
__host__ __device__ constexpr int acc_slot(int I, int J) { return I <= J ? acc_slot_upper(I, J) : acc_slot_upper(J, I); }
__host__ __device__ constexpr int acc_slot_q(int I) {
  return I == 0 ? 19 : I == 2 ? 20 : I == 1 ? 32 + 19 : I == 3 ? 32 + 20 : 64 + 36 + (I - 4);
}

// Hand-off from K2p to K2c, per (camera, frame) pair: 63 doubles, [tile][c][63][lane]
//   0..35  A[i, ext j]  (i = raw intrinsic row 0..5, j = 0..5 over [m | G])
//   36..56 A[ext r, ext s], r <= s, packed upper (tri6)
//   57..62 q[ext r]
constexpr int kHandoff = 63;

// V = P'^T V'' P', g = P'^T g'' with P' = blkdiag(J_l(rho), I); damping lambda * D_f^2 with the
// running Marquardt scaling; 6x6 Cholesky; returns L^-1 (packed lower) and y = L^-1 g.
__device__ __forceinline__ void pose_block_factor(const double (&Vpp)[21], const double (&gpp)[6],
                                                  const double (&Jl)[9], double lambda, double* d2p,
                                                  bool write_d2, double (&Linv)[21], double (&yv)[6],
                                                  double (&gp)[6], double& gmax) {
  double V[36];
  double T1[9];  // V''_ee J
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      T1[3 * i + j] = Vpp[sym6(i, 0)] * Jl[j] + Vpp[sym6(i, 1)] * Jl[3 + j] + Vpp[sym6(i, 2)] * Jl[6 + j];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      V[6 * i + j] = Jl[i] * T1[j] + Jl[3 + i] * T1[3 + j] + Jl[6 + i] * T1[6 + j];
      const double vt = Jl[i] * Vpp[tri6(0, 3 + j)] + Jl[3 + i] * Vpp[tri6(1, 3 + j)] + Jl[6 + i] * Vpp[tri6(2, 3 + j)];
      V[6 * i + 3 + j] = vt;
      V[6 * (3 + j) + i] = vt;
      V[6 * (3 + i) + 3 + j] = Vpp[sym6(3 + i, 3 + j)];
    }
    gp[i] = Jl[i] * gpp[0] + Jl[3 + i] * gpp[1] + Jl[6 + i] * gpp[2];
    gp[3 + i] = gpp[3 + i];
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double d2 = fmax(d2p[i * 32], V[7 * i]);
    if (write_d2) d2p[i * 32] = d2;
    if (d2 == 0.0) d2 = 1.0;
    V[7 * i] = fma(lambda, d2, V[7 * i]);
    gmax = fmax(gmax, fabs(gp[i]));
  }
  // Cholesky factor, 1/L_jj stored on the diagonal; empty frames at lambda = 0 give zeros.
  // Every loop has a constant trip count (the triangular bounds are predicates) so that the
  // whole factorisation unrolls into registers.
  double Lm[21];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double s = V[7 * j];
#pragma unroll
    for (int k = 0; k < 6; ++k)
      if (k < j) s -= Lm[j * (j + 1) / 2 + k] * Lm[j * (j + 1) / 2 + k];
    const double inv = s > 0.0 ? rsqrt(s) : 0.0;
    Lm[j * (j + 1) / 2 + j] = inv;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      if (i > j) {
        double t = V[6 * i + j];
#pragma unroll
        for (int k = 0; k < 6; ++k)
          if (k < j) t -= Lm[i * (i + 1) / 2 + k] * Lm[j * (j + 1) / 2 + k];
        Lm[i * (i + 1) / 2 + j] = t * inv;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    Linv[j * (j + 1) / 2 + j] = Lm[j * (j + 1) / 2 + j];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      if (i > j) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k)
          if (k >= j && k < i) t += Lm[i * (i + 1) / 2 + k] * Linv[k * (k + 1) / 2 + j];
        Linv[i * (i + 1) / 2 + j] = -t * Lm[i * (i + 1) / 2 + i];
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double t = 0.0;
#pragma unroll
    for (int j = 0; j < 6; ++j)
      if (j <= i) t += Linv[i * (i + 1) / 2 + j] * gp[j];
    yv[i] = t;
  }
}

// One row of Z_cf = (W' P') L^-T from one row of W' = A[:,ext] E'.
__device__ __forceinline__ void z_row(const double (&b)[6], const double (&Jl)[9], const double (&Linv)[21],
                                      double (&z)[6]) {
  double w[6];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    w[k] = b[0] * Jl[k] + b[1] * Jl[3 + k] + b[2] * Jl[6 + k];
    w[3 + k] = b[3 + k];
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    double t = 0.0;
#pragma unroll
    for (int j = 0; j < 6; ++j)
      if (j <= k) t += w[j] * Linv[k * (k + 1) / 2 + j];
    z[k] = t;
  }
}

}  // namespace mcba
