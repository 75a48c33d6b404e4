// K3a: the damped reduced camera system  (S + lambda D_c^2) delta_cam = -b  solved by ONE CTA
// (replaces the cuSOLVER potrf + potrs + damping launches of round 1: five library / helper kernels,
// ~90 us of launch and library latency per LM iteration for a 72 x 72 system).
// Math: SURVEY.md Appendix A ("Schur form"), scipy's x_scale='jac' analogue (common.py:598-610).
//
// The lower triangle lives packed in shared memory (12C <= 192: 161 KB), augmented by one more row
// that holds the right-hand side -b: a right-looking blocked Cholesky of the augmented matrix leaves
// y = L^-1 (-b) in that row, so the forward substitution costs nothing extra.  The sequential chain
// of a Cholesky (pivot -> rsqrt -> scale -> update -> next pivot, 12C links) is what bounds a system
// this small, so everything else is taken off it:
//   * panel of 8 columns: ONE thread per row of the block column; every thread factors the 8 x 8
//     diagonal block redundantly in registers (broadcast reads) and solves its own row against it in
//     the same unrolled loop -- no hand-over between a factoring thread and the row threads, and the
//     reciprocal square root is a MUFU seed with two corrections instead of the library call;
//   * trailing matrix: the 8 x 8 tiles are dealt out to the 16 warps ONCE and their accumulators stay
//     in registers for the whole factorisation (FP64 tensor path, DMMA m8n8k4, same fragment mapping
//     as the SYRK in k2_schur.cu); a tile goes back to shared memory only when its block column is
//     the next panel.  Two CTA barriers per panel.
//   * L^T delta = y: one warp, y in registers, 12C steps of (broadcast delta_j, row j of L is
//     contiguous in the packed layout): no CTA barrier at all.
// A non-positive (or NaN) pivot is reported in info[0] like potrf's (the LM loop then rejects the step).
#include <cstdio>
#include <cstdlib>

#include "k2_common.cuh"

namespace mcba {

#ifdef MCBA_SOLVE_TIMING
__device__ long long g_solve_clk[8];
#define MCBA_T0(name) const long long name = clock64()
#define MCBA_ACC(i, t0) do { if (threadIdx.x == 0) g_solve_clk[i] += clock64() - (t0); } while (0)
#define MCBA_STAMP(i) do { if (threadIdx.x == 0) g_solve_clk[i] = clock64(); } while (0)
#else
#define MCBA_STAMP(i) do {} while (0)
#define MCBA_T0(name) do {} while (0)
#define MCBA_ACC(i, t0) do {} while (0)
#endif

constexpr int kSolveThreads = 512;
constexpr int kSolveWarps = kSolveThreads / 32;
constexpr int kSolveMaxN = 192;   // 16 cameras; larger systems take the library path

__host__ __device__ __forceinline__ int pk(int i, int j) { return i * (i + 1) / 2 + j; }   // j <= i

// 1/sqrt(t), t > 0 in the normal range: MUFU.RSQ64H seed (> 20 bits) and ONE third-order correction
// (relative error ~ (5/16) e^3 < 2^-60); four dependent FP64 operations instead of the library's
// slow path on the critical chain of every pivot.  Non-positive or NaN t gives NaN / inf, which the
// pivot test reports.
__device__ __forceinline__ double solve_rsqrt(double t) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(t));
  const double e = fma(-t, y * y, 1.0);
  return fma(y * e, fma(0.375, e, 0.5), y);
}

struct SolveParams {
  const double* red;    // packed reduced system [S | b | g | diag | ...]
  long long offS, offB, offDiag;
  int nc;
  double lambda;
  double* D2cam;        // running max of diag(U) (Marquardt scaling), updated here
  double* dcam;         // out: delta_cam (true basis), nc
  int* info;            // out: 0, or 1 + index of the first non-positive pivot
  const uint8_t* fixed; // [nc] held parameters (mcba_set_fixed): identity row / column, 0 right-hand side; nullptr = none
};

// kT: trailing tiles per warp (3: up to 6 cameras, 8: up to 10, 19: up to 16 -- 24 * 25 / 2 = 300 tiles of the
// 200-row augmented system over 16 warps).  kSmemAcc (the 19-tile variant): 38 accumulators per lane beside the
// panel's 8 x 8 block do not fit in 128 registers (they spilled to local memory: 0.116 ms for 192 x 192), so that
// variant keeps the tiles where they already live -- the packed matrix in shared memory -- and every update is
// load, two DMMAs, store; the 19 tiles of a warp are independent, so their round trips overlap.
template <int kT>
__global__ void __launch_bounds__(kSolveThreads, 1) solve_reduced_kernel(const SolveParams p) {
  constexpr bool kSmemAcc = kT > 8;
  extern __shared__ double A[];                 // packed lower triangle of the augmented matrix, n1p rows
  __shared__ double s_inv[kSolveMaxN + 8];      // 1 / L_jj
  __shared__ int s_info;
  const int nc = p.nc, n1p = (nc + 1 + 7) & ~7, nb = n1p / 8;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_info = 0;
  MCBA_STAMP(0);

  // ---- load: S (lower triangle), row nc = -b, unit diagonal on the padding; 8 independent loads per
  //      thread and pass.  The damping of the diagonal is added after the barrier by one thread per row.
  double damp = 0.0;
  if (tid < nc) {
    double d2 = fmax(p.D2cam[tid], p.red[p.offDiag + tid]);
    p.D2cam[tid] = d2;
    if (d2 == 0.0) d2 = 1.0;
    damp = p.lambda * d2;
  }
  // rows i and n1p-1-i together hold n1p+1 entries: element e of the (n1p/2) x (n1p+1) rectangle of
  // row pairs (no square root, nothing wasted)
  const int n_pk = n1p * (n1p + 1) / 2, pw = n1p + 1;
  for (int base = 0; base < n_pk; base += 8 * kSolveThreads) {
    double v[8];
    int at[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int e = base + u * kSolveThreads + tid;
      v[u] = 0.0;
      at[u] = -1;
      if (e < n_pk) {
        const int pr = e / pw, off = e - pr * pw;
        const int i = off <= pr ? pr : n1p - 1 - pr, j = off <= pr ? off : off - pr - 1;
        at[u] = pk(i, j);
        const bool held_j = p.fixed && j < nc && p.fixed[j];
        if (i < nc) v[u] = held_j || (p.fixed && p.fixed[i]) ? (i == j ? 1.0 : 0.0) : __ldcg(p.red + p.offS + (size_t)i * nc + j);
        else if (i == nc) v[u] = j < nc ? (held_j ? 0.0 : -__ldcg(p.red + p.offB + j)) : 1.0;
        else v[u] = i == j ? 1.0 : 0.0;
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (at[u] >= 0) A[at[u]] = v[u];
  }
  __syncthreads();
  MCBA_STAMP(1);
  if (tid < nc) A[pk(tid, tid)] += damp;

  // ---- this warp's tiles of the trailing matrix: tile (ib, jb), 1 <= jb <= ib < nb, numbered block
  //      column by block column and dealt round-robin (the tiles still active at any panel are then
  //      spread evenly over the warps); accumulators in registers until the tile's column is the panel
  int tij[kT];
  double acc[kT][2];
  const int n_tiles = (nb - 1) * nb / 2;
  const int fr = lane >> 2, fc = 2 * (lane & 3);
  __syncthreads();
#pragma unroll
  for (int s = 0; s < kT; ++s) {
    const int t = warp + s * kSolveWarps;
    tij[s] = -1;
    acc[s][0] = acc[s][1] = 0.0;
    if (t < n_tiles) {
      // column jb holds nb - jb tiles; find it
      int jb = 1, rem = t;
      while (rem >= nb - jb) { rem -= nb - jb; ++jb; }
      const int ib = jb + rem;
      tij[s] = (ib << 8) | jb;
      const int cr = ib * 8 + fr, cc = jb * 8 + fc;
      if (!kSmemAcc && cc <= cr) acc[s][0] = A[pk(cr, cc)];
      if (!kSmemAcc && cc + 1 <= cr) acc[s][1] = A[pk(cr, cc + 1)];
    }
  }
  MCBA_STAMP(2);
#ifdef MCBA_SOLVE_TIMING
  if (tid == 0) { g_solve_clk[5] = 0; g_solve_clk[6] = 0; }
#endif
  // ---- blocked Cholesky of the leading nc columns
  for (int k0 = 0; k0 < nc; k0 += 8) {
    const int w = nc - k0 < 8 ? nc - k0 : 8;   // pivot columns of this panel
    // One thread per row i >= k0 of the block column, straight-line code: every thread factors the
    // 8 x 8 diagonal block in registers and solves ITS row against it (for a row of the block itself
    // that solve reproduces the factor's row, so all rows run the same instructions).  A partial last
    // panel (12C not a multiple of 8) is processed to the full width: its extra columns belong to the
    // right-hand-side / padding rows, whose values nobody reads.
    const int i = k0 + tid;
    double x[8];
    MCBA_T0(tp0);
    if (i < n1p) {
      double a[36];
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int c = 0; c < 8; ++c)
          if (c <= r) a[pk(r, c)] = A[pk(k0 + r, k0 + c)];
      const double* row = A + pk(i, k0);
#pragma unroll
      for (int c = 0; c < 8; ++c) x[c] = (tid >= 8 || c <= tid) ? row[c] : 0.0;
      int bad = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const double d = a[pk(j, j)];
        if (!(d > 0.0) && bad == 0 && j < w) bad = k0 + j + 1;
        const double inv = solve_rsqrt(d);
#pragma unroll
        for (int r = 0; r < 8; ++r)
          if (r > j) a[pk(r, j)] *= inv;
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
          for (int c = 0; c < 8; ++c)
            if (r > j && c > j && c <= r) a[pk(r, c)] = fma(-a[pk(r, j)], a[pk(c, j)], a[pk(r, c)]);
        double t = x[j];           // own row against column j of the factor
#pragma unroll
        for (int c = 0; c < 8; ++c)
          if (c < j) t = fma(-x[c], a[pk(j, c)], t);
        x[j] = t * inv;
        if (tid == 0) s_inv[k0 + j] = inv;
      }
      if (tid == 0 && bad && s_info == 0) s_info = bad;
      if (tid >= 8) {
        double* wrow = A + pk(i, k0);
#pragma unroll
        for (int c = 0; c < 8; ++c) wrow[c] = x[c];
      }
    }
    MCBA_ACC(5, tp0);
    __syncthreads();
    MCBA_T0(tp1);
    // the rows of the diagonal block go back only now: until the barrier the other warps were still
    // reading the unfactored block (nobody reads it during the trailing update)
    if (tid < 8) {
      double* wrow = A + pk(i, k0);
#pragma unroll
      for (int c = 0; c < 8; ++c)
        if (c <= tid) wrow[c] = x[c];
    }
    // trailing update on the FP64 tensor path: C_ij -= L_i L_j^T for this warp's tiles right of the panel
    // (measured: jumping to the first live slot and batching the fragment loads of four tiles were
    // both slower than this plain loop with a warp-uniform test per slot)
    const int kb = k0 >> 3;
    const int fk = k0 + (lane & 3);
    // (a straight-line version of the shared-memory variant -- dead slots computing on a valid row pair and storing
    // nothing, so that the slots' chains can overlap -- was slower: 0.146 ms against 0.094 ms at 192 x 192)
#pragma unroll
    for (int s = 0; s < kT; ++s) {
      const int jb = tij[s] & 0xff, ib = tij[s] >> 8;
      if (tij[s] >= 0 && jb > kb) {     // warp-uniform
        const double a0 = -A[pk(ib * 8 + fr, fk)], a1 = -A[pk(ib * 8 + fr, fk + 4)];
        const double b0 = A[pk(jb * 8 + fr, fk)], b1 = A[pk(jb * 8 + fr, fk + 4)];
        const int cr = ib * 8 + fr, cc = jb * 8 + fc;
        if (kSmemAcc) {                 // the tile lives in shared memory (fragments read the panel's columns only)
          double c0 = cc <= cr ? A[pk(cr, cc)] : 0.0, c1 = cc + 1 <= cr ? A[pk(cr, cc + 1)] : 0.0;
          dmma_m8n8k4(c0, c1, a0, b0);
          dmma_m8n8k4(c0, c1, a1, b1);
          if (cc <= cr) A[pk(cr, cc)] = c0;
          if (cc + 1 <= cr) A[pk(cr, cc + 1)] = c1;
        } else {
          dmma_m8n8k4(acc[s][0], acc[s][1], a0, b0);
          dmma_m8n8k4(acc[s][0], acc[s][1], a1, b1);
          if (jb == kb + 1) {           // the next panel: back to shared memory
            if (cc <= cr) A[pk(cr, cc)] = acc[s][0];
            if (cc + 1 <= cr) A[pk(cr, cc + 1)] = acc[s][1];
          }
        }
      }
    }
    MCBA_ACC(6, tp1);
    __syncthreads();
  }

  MCBA_STAMP(3);
  // ---- backward substitution L^T delta = y (y = row nc of the factor): warp 0, y in registers
  if (warp == 0) {
    constexpr int kSlots = (kSolveMaxN + 31) / 32;
    double y[kSlots];
#pragma unroll
    for (int s = 0; s < kSlots; ++s) y[s] = (lane + 32 * s) < nc ? A[pk(nc, lane + 32 * s)] : 0.0;
    // 32 unknowns per register slot, slots from the last to the first (compile-time slot index: the
    // carried chain of a step is broadcast -> multiply -> fused multiply-add, nothing else)
#pragma unroll
    for (int sj = kSlots - 1; sj >= 0; --sj) {
      const int j_hi = nc - 1 < 32 * sj + 31 ? nc - 1 : 32 * sj + 31;
      for (int j = j_hi; j >= 32 * sj; --j) {
        const double dj = __shfl_sync(0xffffffffu, y[sj], j & 31) * s_inv[j];
        const double* Lj = A + pk(j, 0);
#pragma unroll
        for (int s = 0; s < kSlots; ++s)
          if (s < sj) y[s] = fma(-Lj[lane + 32 * s], dj, y[s]);
        const int i = lane + 32 * sj;
        const double l = i < j ? Lj[i] : 0.0;
        y[sj] = i == j ? dj : fma(-l, dj, y[sj]);
      }
    }
#pragma unroll
    for (int s = 0; s < kSlots; ++s)
      if (lane + 32 * s < nc) p.dcam[lane + 32 * s] = p.fixed && p.fixed[lane + 32 * s] ? 0.0 : y[s];
    if (lane == 0) p.info[0] = s_info;
    MCBA_STAMP(4);
  }
}

// ------------------------------------------------------------------ library path (12C > 192, or MCBA_CUSOLVER=1 for A/B runs)
__global__ void damp_kernel(const double* __restrict__ red, long long offS, long long offB, long long offDiag,
                            int nc, double lambda, double* __restrict__ D2cam, double* __restrict__ Sd,
                            double* __restrict__ rhs, const uint8_t* __restrict__ fixed) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nc * nc) return;
  const int r = i / nc, q = i % nc;
  const bool held = fixed && (fixed[r] || fixed[q]);   // identity row / column, 0 right-hand side: delta = 0 there
  double v = held ? 0.0 : red[offS + i];
  if (r == q) {
    double d2 = fmax(D2cam[r], red[offDiag + r]);
    D2cam[r] = d2;
    if (d2 == 0.0) d2 = 1.0;
    v = held ? 1.0 : fma(lambda, d2, v);
    rhs[r] = held ? 0.0 : -red[offB + r];
  }
  Sd[i] = v;
}

bool solve_uses_library(int nc) {
  static const bool force = getenv("MCBA_CUSOLVER") != nullptr;
  return force || nc > kSolveMaxN;
}

// Which solve runs for a 12C-wide system: kSolveTier* (mcba_plan_info).
int solve_tier(int nc) {
  if (solve_uses_library(nc)) return kSolveTierLibrary;
  const int n1p = (nc + 1 + 7) & ~7;
  const int nb = n1p / 8, per_warp = ((nb - 1) * nb / 2 + kSolveWarps - 1) / kSolveWarps;
  if (per_warp <= 3) return kSolveTierRegs3;
  if (per_warp <= 8) return kSolveTierRegs8;
  return kSolveTierSmem19;
}

// cuSOLVER handle on the handle's stream and the potrf workspace of the 12C-wide solve, created on first use
// (the common sizes never touch the library; the covariance's camera inverse does)
int ensure_solver(mcba_handle* h) {
  if (!h->solver) {
    const int nc = h->L.nc;
    if (cusolverDnCreate(&h->solver) != CUSOLVER_STATUS_SUCCESS) { set_error("cusolverDnCreate failed"); return MCBA_ERR_SOLVER; }
    if (cusolverDnDpotrf_bufferSize(h->solver, CUBLAS_FILL_MODE_LOWER, nc, h->d_Sd, nc, &h->lwork) != CUSOLVER_STATUS_SUCCESS) {
      set_error("cusolverDnDpotrf_bufferSize failed");
      return MCBA_ERR_SOLVER;
    }
    MCBA_CUDA(cudaMalloc((void**)&h->d_work, sizeof(double) * (size_t)(h->lwork > 0 ? h->lwork : 1)));
  }
  cusolverDnSetStream(h->solver, h->stream);
  return MCBA_OK;
}

int solve_reduced(mcba_handle* h, double lambda) {
  const Layout& L = h->L;
  const int nc = L.nc;
  const int tier = solve_tier(nc);
  if (tier != kSolveTierLibrary) {
    SolveParams p;
    p.red = h->d_red; p.offS = L.offS; p.offB = L.offB; p.offDiag = L.offDiag; p.nc = nc; p.lambda = lambda;
    p.D2cam = h->d_D2cam; p.dcam = h->d_dcam; p.info = h->d_info; p.fixed = h->any_fixed ? h->d_fixed : nullptr;
    const int n1p = (nc + 1 + 7) & ~7;
    const size_t smem = sizeof(double) * (size_t)n1p * (n1p + 1) / 2;
#define MCBA_SOLVE(KT)                                                                                                     \
  do {                                                                                                                     \
    MCBA_CUDA(set_dynamic_smem((const void*)solve_reduced_kernel<KT>, smem));                                              \
    solve_reduced_kernel<KT><<<1, kSolveThreads, smem, h->stream>>>(p);                                                    \
  } while (0)
    if (tier == kSolveTierRegs3) MCBA_SOLVE(3);
    else if (tier == kSolveTierRegs8) MCBA_SOLVE(8);
    else MCBA_SOLVE(19);
#undef MCBA_SOLVE
#ifdef MCBA_SOLVE_TIMING
    {
      long long c[8];
      cudaStreamSynchronize(h->stream);
      cudaMemcpyFromSymbol(c, g_solve_clk, sizeof(c));
      fprintf(stderr, "solve phases (cycles): load %lld  setup %lld  panels %lld  backward %lld | factor (warp 0) %lld  update (warp 0) %lld\n", c[1] - c[0], c[2] - c[1], c[3] - c[2], c[4] - c[3], c[5], c[6]);
    }
#endif
    h->launches++;
    MCBA_CUDA(cudaGetLastError());
    return MCBA_OK;
  }
  int rc = ensure_solver(h);
  if (rc) return rc;
  damp_kernel<<<(nc * nc + 255) / 256, 256, 0, h->stream>>>(h->d_red, L.offS, L.offB, L.offDiag, nc, lambda,
                                                            h->d_D2cam, h->d_Sd, h->d_dcam, h->any_fixed ? h->d_fixed : nullptr);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  cusolverStatus_t st = cusolverDnDpotrf(h->solver, CUBLAS_FILL_MODE_LOWER, nc, h->d_Sd, nc, h->d_work, h->lwork, h->d_info);
  if (st != CUSOLVER_STATUS_SUCCESS) { set_error("cusolverDnDpotrf failed"); return MCBA_ERR_SOLVER; }
  st = cusolverDnDpotrs(h->solver, CUBLAS_FILL_MODE_LOWER, nc, 1, h->d_Sd, nc, h->d_dcam, nc, h->d_info + 1);
  if (st != CUSOLVER_STATUS_SUCCESS) { set_error("cusolverDnDpotrs failed"); return MCBA_ERR_SOLVER; }
  h->launches += 4;  // potrf + potrs kernels (library; approximate count)
  return MCBA_OK;
}

}  // namespace mcba
