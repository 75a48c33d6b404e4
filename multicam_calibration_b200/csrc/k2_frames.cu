// K2: fused residual + analytic Jacobian + robust scaling + per-frame Schur elimination
// (replaces scipy's finite-difference Jacobian + LSMR for the path
// bundle_adjustment.py:299-313; math in SURVEY.md Appendix A), as two kernels:
//
//   K2p (k2_producer.cuh)  per (camera, frame) pair: walk the board corners, accumulate the raw
//       12x12 block A_cf / q_cf in registers, add it to the camera partial sums, hand the
//       extrinsic part (63 doubles per pair) to K2c.            FP64-pipe bound.
//   K2c (below)            per frame: map the hand-off to the pose basis (W' = A[:,ext] E',
//       V'' = E'^T A_ee E'), sum over cameras, factor V_f + lambda D_f^2 = L L^T (6x6, per lane),
//       write Z_cf = W_cf L^-T, y_f = L^-1 g_f, L^-1 for the SYRK and the back-substitution,
//       and the per-tile sums Z y.  Every global access is a coalesced 256-byte row
//       (lane = frame is the fastest index of H, Z, y, L^-1).  HBM bound: reads 504 B,
//       writes 576 B per pair.
//
// K2c comes in two builds (k2_consumer_parts): the staged ring for 2-6 cameras and a streamed pair of kernels
// (pose block per tile, Z rows per live unit) for any other count.
// A rejected LM step only changes lambda: K2c is re-run on the same hand-off, K2p is not.
#include "k2_producer.cuh"

namespace mcba {

// ------------------------------------------------------------------ K2c
struct K2CParams {
  int C;
  long long F, nTiles;
  const double* H;       // [tile][c][63][32]
  const int* perm;       // tile slot -> frame index in x (-1 = padding)
  const unsigned int* active;   // [tile] bit c: camera c has observations in the tile
  const int* units;      // [C][nTiles] live tiles per camera, compacted (build_units_kernel)
  const int* unit_count; // [C]
  const double* x;       // 12C + 6F
  const CamConst* cams;
  double lambda;
  double* Z;             // [tile][row 12C][k 6][lane 32]
  double* Linv;          // [tile][21][32]
  double* y;             // [tile][6][32]
  double* JlTau;         // [tile][12][32] J_l(rho_f) | tau_f (streamed path only: pose kernel -> rows kernel)
  double* partZy;        // [tile][12C]  sum over the tile's frames of Z_f y_f
  double* gpose;         // [f][6]
  double* D2pose;        // [tile][6][32] running max of diag(V_f)
  double* partG;         // [tile] max |g_pose|
};

// E' = [[Rc, 0], [K, Rc]],  K = [t_cf]x Rc   (rows: raw [m | G], cols: pose perturbation [eps | tau])
__device__ __forceinline__ void pose_map(const CamConst& cam, const double (&pose)[6], double (&Rc)[9], double (&K)[9]) {
  double tcf[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) Rc[i] = cam.R[i];
  mat3_vec(Rc, pose + 3, tcf);
  tcf[0] += cam.t[0];
  tcf[1] += cam.t[1];
  tcf[2] += cam.t[2];
  cross_mat3(tcf, Rc, K);
}

// Camera c's contribution to the pose block of this lane's frame: V'' += E'^T A_ee E', g'' += E'^T q_e.
// h: this lane's hand-off column of the pair (global or shared memory), entries kTile doubles apart.
__device__ __forceinline__ void pose_block_load(const double* __restrict__ h, double (&Aee)[21], double (&qe)[6]) {
#pragma unroll
  for (int i = 0; i < 21; ++i) Aee[i] = h[(36 + i) * kTile];
#pragma unroll
  for (int i = 0; i < 6; ++i) qe[i] = h[(57 + i) * kTile];
}
__device__ __forceinline__ void pose_block_apply(const double (&Aee)[21], const double (&qe)[6], const double (&Rc)[9],
                                                 const double (&K)[9], double (&Vpp)[21], double (&gpp)[6]);
__device__ __forceinline__ void pose_block_add(const double* __restrict__ h, const double (&Rc)[9], const double (&K)[9],
                                               double (&Vpp)[21], double (&gpp)[6]) {
  double Aee[21], qe[6];
  pose_block_load(h, Aee, qe);
  pose_block_apply(Aee, qe, Rc, K, Vpp, gpp);
}
__device__ __forceinline__ void pose_block_apply(const double (&Aee)[21], const double (&qe)[6], const double (&Rc)[9],
                                                 const double (&K)[9], double (&Vpp)[21], double (&gpp)[6]) {
  double Be[36];
#pragma unroll
  for (int r = 0; r < 6; ++r) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      Be[r * 6 + k] = Aee[sym6(r, 0)] * Rc[k] + Aee[sym6(r, 1)] * Rc[3 + k] + Aee[sym6(r, 2)] * Rc[6 + k] +
                      Aee[sym6(r, 3)] * K[k] + Aee[sym6(r, 4)] * K[3 + k] + Aee[sym6(r, 5)] * K[6 + k];
      Be[r * 6 + 3 + k] = Aee[sym6(r, 3)] * Rc[k] + Aee[sym6(r, 4)] * Rc[3 + k] + Aee[sym6(r, 5)] * Rc[6 + k];
    }
  }
#pragma unroll
  for (int a = 0; a < 6; ++a) {
#pragma unroll
    for (int n = a; n < 6; ++n) {
      double v;
      if (a < 3) {
        v = Rc[a] * Be[n] + Rc[3 + a] * Be[6 + n] + Rc[6 + a] * Be[12 + n] + K[a] * Be[18 + n] +
            K[3 + a] * Be[24 + n] + K[6 + a] * Be[30 + n];
      } else {
        v = Rc[a - 3] * Be[18 + n] + Rc[3 + a - 3] * Be[24 + n] + Rc[6 + a - 3] * Be[30 + n];
      }
      Vpp[tri6(a, n)] += v;
    }
    if (a < 3) {
      gpp[a] += Rc[a] * qe[0] + Rc[3 + a] * qe[1] + Rc[6 + a] * qe[2] + K[a] * qe[3] + K[3 + a] * qe[4] +
                K[6 + a] * qe[5];
    } else {
      gpp[a] += Rc[a - 3] * qe[3] + Rc[3 + a - 3] * qe[4] + Rc[6 + a - 3] * qe[5];
    }
  }
}

// Z_cf = (A[:,ext] E' P') L^-T for one camera, one raw camera row at a time, written as coalesced
// rows of the tile's Z block (z points at [row 12c][k 0][lane]); zy[row] += sum_k Z[row][k] y[k].
template <int kRow0, int kRow1>
__device__ __forceinline__ void z_rows_range(const double* __restrict__ h, const double (&Rc)[9], const double (&K)[9],
                                             const double (&Jl)[9], const double (&Linv)[21], const double (&yv)[6],
                                             double* __restrict__ z, double (&zy)[12]) {
#pragma unroll
  for (int row = kRow0; row < kRow1; ++row) {
    double am[3], ag[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      am[j] = row < 6 ? h[(row * 6 + j) * kTile] : h[(36 + sym6(row - 6, j)) * kTile];
      ag[j] = row < 6 ? h[(row * 6 + 3 + j) * kTile] : h[(36 + sym6(row - 6, 3 + j)) * kTile];
    }
    double b[6], zr[6];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      b[k] = am[0] * Rc[k] + am[1] * Rc[3 + k] + am[2] * Rc[6 + k] + ag[0] * K[k] + ag[1] * K[3 + k] + ag[2] * K[6 + k];
      b[3 + k] = ag[0] * Rc[k] + ag[1] * Rc[3 + k] + ag[2] * Rc[6 + k];
    }
    z_row(b, Jl, Linv, zr);
    double t = zy[row];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      z[(size_t)(row * 6 + k) * kTile] = zr[k];   // padded lanes carry zeros (their hand-off is zero)
      t = fma(zr[k], yv[k], t);
    }
    zy[row] = t;
  }
}
__device__ __forceinline__ void z_rows(const double* __restrict__ h, const double (&Rc)[9], const double (&K)[9],
                                       const double (&Jl)[9], const double (&Linv)[21], const double (&yv)[6],
                                       double* __restrict__ z, double (&zy)[12]) {
  z_rows_range<0, 12>(h, Rc, K, Jl, Linv, yv, z, zy);
}

// lane l < 12 receives the sum over the warp of zy[l]
__device__ __forceinline__ double zy_lane_sum(double (&zy)[12], int lane) {
#pragma unroll
  for (int row = 0; row < 12; ++row) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) zy[row] += __shfl_xor_sync(0xffffffffu, zy[row], off);
  }
  double v = zy[0];
#pragma unroll
  for (int row = 1; row < 12; ++row) v = lane == row ? zy[row] : v;
  return v;
}

__device__ __forceinline__ void store_pose_outputs(const K2CParams& p, long long tile, long long f, bool fvalid, int lane,
                                                   const double (&Linv)[21], const double (&yv)[6], const double (&gp)[6]) {
  double* lo = p.Linv + (size_t)tile * 21 * 32 + lane;
#pragma unroll
  for (int i = 0; i < 21; ++i) lo[i * 32] = Linv[i];
  double* yo = p.y + (size_t)tile * 6 * 32 + lane;
#pragma unroll
  for (int i = 0; i < 6; ++i) yo[i * 32] = yv[i];
  if (fvalid) {
#pragma unroll
    for (int i = 0; i < 6; i += 2)
      *reinterpret_cast<double2*>(p.gpose + (size_t)f * 6 + i) = make_double2(gp[i], gp[i + 1]);
  }
}

// Staged path (kC <= 6 cameras, warp = camera): persistent CTAs, two per SM.  The whole hand-off
// block of a tile (kC x 63 x 32 doubles, contiguous) arrives by ONE bulk async copy into shared
// memory; while one CTA of the SM waits for its copy the other one computes, so no warp waits on
// a global load and each scheduler hosts three warps.  Z, y and L^-1 leave as coalesced 256-byte
// rows.  The cross-camera sum of the pose block goes through a small exchange buffer in two
// rounds (11 + 10 values; g'' travels in the camera's already consumed q_ext slots of the
// stage), which is what lets two CTAs fit in the 228 KB of an SM.  Partial outputs per CTA.
constexpr int kXchg = 11;   // values per exchange round

template <int kC>
__global__ void __launch_bounds__(kC * 32, 2) k2c_ring_kernel(const K2CParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ unsigned long long full_bar;
  constexpr int kStage = kC * kHandoff * kTile;                  // doubles per stage
  double* stage = reinterpret_cast<double*>(smem_raw);           // [kC][63][32]
  double* s_X = stage + kStage;                                  // [kC][kXchg][32]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int nc = 12 * kC;
  const int c = warp;
  const int n_it = p.nTiles > blockIdx.x ? (int)((p.nTiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
  // thread 0 only: one bulk copy per LIVE camera of the tile (frames are sorted by visibility
  // mask, so a dead (tile, camera) unit has an all-zero hand-off that is never read, and its Z rows,
  // zeroed once when the observations were tiled, are never written)
  auto issue = [&](int it) {
    const long long tile = blockIdx.x + (long long)it * gridDim.x;
    const unsigned m = p.active[tile] & ((1u << kC) - 1u);
    constexpr unsigned kUnitBytes = kHandoff * kTile * sizeof(double);
    const unsigned bytes = (unsigned)__popc(m) * kUnitBytes;
    mbar_expect_tx(&full_bar, bytes);
    if (m == (1u << kC) - 1u) {
      tma_load_1d(stage, p.H + (size_t)tile * kStage, bytes, &full_bar);
    } else {
#pragma unroll
      for (int cc = 0; cc < kC; ++cc) {
        if ((m >> cc) & 1u)
          tma_load_1d(stage + (size_t)cc * kHandoff * kTile, p.H + (size_t)tile * kStage + (size_t)cc * kHandoff * kTile,
                      kUnitBytes, &full_bar);
      }
    }
  };
  if (threadIdx.x == 0) {
    mbar_init(&full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (n_it > 0) issue(0);
  }
  __syncthreads();
  const CamConst& cam = p.cams[c];
  double zy[12], gmax = 0.0;
#pragma unroll
  for (int i = 0; i < 12; ++i) zy[i] = 0.0;
  double* h = stage + (size_t)c * kHandoff * kTile + lane;

  for (int it = 0; it < n_it; ++it) {
    const long long tile = blockIdx.x + (long long)it * gridDim.x;
    const long long f = p.perm[tile * kTile + lane];
    const bool fvalid = f >= 0;
    const bool live = (p.active[tile] >> c) & 1u;   // warp-uniform
    double pose[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) pose[i] = fvalid ? p.x[(size_t)nc + f * 6 + i] : 0.0;
    double Jl[9], Rc[9], K[9];
    so3_left_jacobian(pose, Jl);
    pose_map(cam, pose, Rc, K);
    mbar_wait(&full_bar, (unsigned)(it & 1));
    double Vpp[21], gpp[6];
    {
      double Vp[21], gq[6];
#pragma unroll
      for (int i = 0; i < 21; ++i) Vp[i] = 0.0;
#pragma unroll
      for (int i = 0; i < 6; ++i) gq[i] = 0.0;
      if (live) pose_block_add(h, Rc, K, Vp, gq);
      // round 1: V''[0..10] through s_X, g'' through this camera's (consumed) q_ext slots
#pragma unroll
      for (int i = 0; i < kXchg; ++i) s_X[(c * kXchg + i) * kTile + lane] = Vp[i];
#pragma unroll
      for (int i = 0; i < 6; ++i) h[(57 + i) * kTile] = gq[i];
      __syncthreads();
#pragma unroll
      for (int i = 0; i < kXchg; ++i) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kC; ++w) t += s_X[(w * kXchg + i) * kTile + lane];
        Vpp[i] = t;
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kC; ++w) t += stage[((size_t)w * kHandoff + 57 + i) * kTile + lane];
        gpp[i] = t;
      }
      __syncthreads();
      // round 2: V''[11..20]
#pragma unroll
      for (int i = kXchg; i < 21; ++i) s_X[(c * kXchg + i - kXchg) * kTile + lane] = Vp[i];
      __syncthreads();
#pragma unroll
      for (int i = kXchg; i < 21; ++i) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kC; ++w) t += s_X[(w * kXchg + i - kXchg) * kTile + lane];
        Vpp[i] = t;
      }
    }
    double Linv[21], yv[6], gp[6];
    pose_block_factor(Vpp, gpp, Jl, p.lambda, p.D2pose + (size_t)tile * 6 * 32 + lane, warp == 0, Linv, yv, gp, gmax);
    if (warp == 0) store_pose_outputs(p, tile, f, fvalid, lane, Linv, yv, gp);
    if (live) z_rows(h, Rc, K, Jl, Linv, yv, p.Z + ((size_t)(tile * nc + c * 12) * 6) * kTile + lane, zy);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // our generic writes (g'') precede the next bulk copy
    __syncthreads();   // every warp is done with the stage and with s_X
    if (threadIdx.x == 0 && it + 1 < n_it) issue(it + 1);
  }
  const double v = zy_lane_sum(zy, lane);
  if (lane < 12) p.partZy[(size_t)blockIdx.x * nc + c * 12 + lane] = v;
  if (warp == 0) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) gmax = fmax(gmax, __shfl_xor_sync(0xffffffffu, gmax, off));
    if (lane == 0) p.partG[blockIdx.x] = gmax;
  }
}

// Streamed path (any camera count): two kernels of unsynchronised warps, no CTA barrier and no exchange between
// warps in the tile loops.  Every warp pulls what it needs of a pair's hand-off through its OWN two-stage ring of
// bulk async copies (per-warp mbarriers; 18 KB per warp, kW = 12 warps per SM for up to 6 cameras):
//   k2c_pose_kernel   one warp per FRAME TILE: rows 36..62 (A_ee, q_ext) of every live camera ->
//                     V'' += E'^T A_ee E', g'' += E'^T q_e in registers, then the 6x6 factor of V_f + lambda D_f^2
//                     ONCE per frame (the staged path repeats it in every camera's warp); writes L^-1, y, g_pose;
//   k2c_rows_kernel   one warp per LIVE (tile, camera) UNIT (K2p's unit lists): rows 0..35 (A[int, ext]) -> the six
//                     intrinsic rows of Z_cf, rows 36..56 (A_ee again: an L2 hit) -> its six extrinsic rows; Z y.
// The staged kernel spends 14 us on a tile (six warps in step, three CTA barriers, the tile's 97 KB in one copy);
// here a tile's pose block is ~15 us of ONE warp and its rows are spread over as many warps as it has cameras, so
// 50,000 frames (1563 tiles, 7500 units) fill 148 x 12 warps in one round each.  Partial outputs per CTA.
constexpr int kStreamRows = 36;                                  // rows of 32 doubles per stage
constexpr int kStreamStage = kStreamRows * kTile;                // doubles per stage
inline size_t k2c_stream_smem(int C, int warps) {
  return sizeof(double) * ((size_t)warps * 2 * kStreamStage + (size_t)warps * 12 * C + (size_t)C * 12 + warps) +
         sizeof(unsigned long long) * 2 * warps + sizeof(int) * (size_t)(C + 2);
}

struct K2cStreamShared {
  double* ring;                 // this warp's two stages
  double* zy_all;               // [kW][12C]
  double* cam;                  // [C][12]: R | t
  double* gmax;                 // [kW]
  unsigned long long* bar;      // this warp's two mbarriers
  int* ucum;                    // [C + 1] live units before camera c
};
template <int kW>
__device__ __forceinline__ K2cStreamShared k2c_stream_carve(unsigned char* smem_raw, int C, int warp) {
  K2cStreamShared s;
  double* base = reinterpret_cast<double*>(smem_raw);
  s.ring = base + (size_t)warp * 2 * kStreamStage;
  s.zy_all = base + (size_t)kW * 2 * kStreamStage;
  s.cam = s.zy_all + (size_t)kW * 12 * C;
  s.gmax = s.cam + (size_t)C * 12;
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(s.gmax + kW);
  s.bar = bars + 2 * warp;
  s.ucum = reinterpret_cast<int*>(bars + 2 * kW);
  return s;
}
template <int kW>
__device__ __forceinline__ void k2c_stream_init(const K2CParams& p, const K2cStreamShared& s, int lane) {
  if (lane == 0) {
    mbar_init(s.bar, 1);
    mbar_init(s.bar + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = threadIdx.x; i < p.C * 12; i += kW * 32) {
    const CamConst& cam = p.cams[i / 12];
    const int j = i % 12;
    s.cam[i] = j < 9 ? cam.R[j] : cam.t[j - 9];
  }
}
__device__ __forceinline__ void k2c_stream_copy(const K2cStreamShared& s, unsigned k, const double* src, unsigned rows) {
  const unsigned bytes = rows * kTile * (unsigned)sizeof(double);
  mbar_expect_tx(s.bar + (k & 1u), bytes);
  tma_load_1d(s.ring + (size_t)(k & 1u) * kStreamStage, src, bytes, s.bar + (k & 1u));
}
// E' of camera c for this lane's pose from the shared copy of R_c | t_c
__device__ __forceinline__ void k2c_stream_map(const double* s_cam, int c, const double (&pose)[6], double (&Rc)[9],
                                               double (&K)[9]) {
  double tcf[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) Rc[i] = s_cam[c * 12 + i];
  mat3_vec(Rc, pose + 3, tcf);
#pragma unroll
  for (int i = 0; i < 3; ++i) tcf[i] += s_cam[c * 12 + 9 + i];
  cross_mat3(tcf, Rc, K);
}

template <int kW>
__global__ void __launch_bounds__(kW * 32, 1) k2c_pose_kernel(const K2CParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int C = p.C, nc = 12 * C;
  const K2cStreamShared s = k2c_stream_carve<kW>(smem_raw, C, warp);
  k2c_stream_init<kW>(p, s, lane);
  __syncthreads();
  const long long gw = (long long)blockIdx.x * kW + warp, nW = (long long)gridDim.x * kW;
  const int n_it = p.nTiles > gw ? (int)((p.nTiles - gw + nW - 1) / nW) : 0;
  const unsigned cmask = C >= 32 ? 0xffffffffu : (1u << C) - 1u;
  // issue side: rows 36..62 of the live cameras of this warp's tiles, two copies ahead of the consumer
  int it_i = 0;
  unsigned rem_i = 0, k_i = 0;
  bool done_i = n_it == 0;
  if (!done_i) rem_i = p.active[gw] & cmask;
  auto issue_next = [&]() {
    if (done_i) return;
    while (rem_i == 0) {
      ++it_i;
      if (it_i >= n_it) { done_i = true; return; }
      rem_i = p.active[gw + (long long)it_i * nW] & cmask;
    }
    const int c = __ffs(rem_i) - 1;
    rem_i &= rem_i - 1;
    if (lane == 0)
      k2c_stream_copy(s, k_i, p.H + ((size_t)((gw + (long long)it_i * nW) * C + c) * kHandoff + 36) * kTile, 27u);
    ++k_i;
  };
  unsigned k_c = 0;
  issue_next();
  issue_next();
  double gmax = 0.0;
  for (int it = 0; it < n_it; ++it) {
    const long long tile = gw + (long long)it * nW;
    const long long f = p.perm[tile * kTile + lane];
    const bool fvalid = f >= 0;
    const unsigned act = p.active[tile] & cmask;
    double pose[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) pose[i] = fvalid ? p.x[(size_t)nc + f * 6 + i] : 0.0;
    double Jl[9];
    so3_left_jacobian(pose, Jl);
    double Vpp[21], gpp[6];
#pragma unroll
    for (int i = 0; i < 21; ++i) Vpp[i] = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) gpp[i] = 0.0;
    for (unsigned m = act; m; m &= m - 1) {
      const int c = __ffs(m) - 1;
      double Rc[9], K[9];
      k2c_stream_map(s.cam, c, pose, Rc, K);
      mbar_wait(s.bar + (k_c & 1u), (k_c >> 1) & 1u);
      pose_block_add(s.ring + (size_t)(k_c & 1u) * kStreamStage + lane - 36 * kTile, Rc, K, Vpp, gpp);   // stage row 0 = hand-off row 36
      __syncwarp();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      ++k_c;
      issue_next();   // (refilling the stage before the arithmetic, from a register copy, was slower: 23 -> 28 us)
    }
    double Linv[21], yv[6], gp[6];
    pose_block_factor(Vpp, gpp, Jl, p.lambda, p.D2pose + (size_t)tile * 6 * 32 + lane, true, Linv, yv, gp, gmax);
    store_pose_outputs(p, tile, f, fvalid, lane, Linv, yv, gp);
    {   // what the rows kernel needs of the pose, as coalesced rows: J_l(rho_f) and tau_f
      double* jt = p.JlTau + (size_t)tile * 12 * kTile + lane;
#pragma unroll
      for (int i = 0; i < 9; ++i) jt[i * kTile] = Jl[i];
#pragma unroll
      for (int i = 0; i < 3; ++i) jt[(9 + i) * kTile] = pose[3 + i];
    }
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) gmax = fmax(gmax, __shfl_xor_sync(0xffffffffu, gmax, off));
  if (lane == 0) s.gmax[warp] = gmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    double g = 0.0;
    for (int w = 0; w < kW; ++w) g = fmax(g, s.gmax[w]);
    p.partG[blockIdx.x] = g;
  }
}

template <int kW>
__global__ void __launch_bounds__(kW * 32, 1) k2c_rows_kernel(const K2CParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int C = p.C, nc = 12 * C;
  const K2cStreamShared s = k2c_stream_carve<kW>(smem_raw, C, warp);
  k2c_stream_init<kW>(p, s, lane);
  double* s_zy = s.zy_all + (size_t)warp * nc;
  for (int i = lane; i < nc; i += 32) s_zy[i] = 0.0;
  if (threadIdx.x == 0) {
    int a = 0;
    for (int c = 0; c < C; ++c) { s.ucum[c] = a; a += p.unit_count[c]; }
    s.ucum[C] = a;
  }
  __syncthreads();
  const int n_units = s.ucum[C];
  const long long gw = (long long)blockIdx.x * kW + warp, nW = (long long)gridDim.x * kW;
  const int n_it = n_units > gw ? (int)((n_units - gw + nW - 1) / nW) : 0;
  // unit j of the camera-major list -> (camera, tile); j only grows, so the camera cursor only moves forward
  auto unit_of = [&](long long j, int& c) -> long long {
    while (j >= s.ucum[c + 1]) ++c;
    return p.units[(long long)c * p.nTiles + (j - s.ucum[c])];
  };
  // Issue side, three stages per unit, two ahead of the consumer; nothing the consumer needs comes from a
  // dependent global load (the pose kernel left L^-1, y, J_l and tau per tile as coalesced rows):
  //   0: L^-1 (21 rows) | y (6)        1: A_ee (21 rows: hand-off rows 36..56) | J_l, tau (12)        2: A[int, ext] (36)
  int it_i = 0, sub_i = 0, c_i = 0;
  long long tile_i = 0;
  unsigned k_i = 0;
  auto issue_next = [&]() {
    if (it_i >= n_it) return;
    if (sub_i == 0) tile_i = unit_of(gw + (long long)it_i * nW, c_i);
    if (lane == 0) {
      // the barrier's shared address is converted once, ahead of the stage addresses, and serves the expect_tx and
      // every copy of the stage: spelt with mbar_expect_tx / tma_load_1d, the conversion moves into each call and
      // ptxas schedules this issue path differently
      const unsigned b = smem_u32(s.bar + (k_i & 1u));
      double* st = s.ring + (size_t)(k_i & 1u) * kStreamStage;
      const double* hp = p.H + (size_t)(tile_i * C + c_i) * kHandoff * kTile;
      auto copy = [&](double* dst, const double* src, unsigned rows) {
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         smem_u32(dst)),
                     "l"(src), "r"(rows * kTile * (unsigned)sizeof(double)), "r"(b)
                     : "memory");
      };
      const unsigned rows = sub_i == 0 ? 27u : (sub_i == 1 ? 33u : 36u);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(rows * kTile * (unsigned)sizeof(double)) : "memory");
      if (sub_i == 0) {
        copy(st, p.Linv + (size_t)tile_i * 21 * kTile, 21u);
        copy(st + 21 * kTile, p.y + (size_t)tile_i * 6 * kTile, 6u);
      } else if (sub_i == 1) {
        copy(st, hp + 36 * kTile, 21u);
        copy(st + 21 * kTile, p.JlTau + (size_t)tile_i * 12 * kTile, 12u);
      } else {
        copy(st, hp, 36u);
      }
    }
    ++k_i;
    if (++sub_i == 3) { sub_i = 0; ++it_i; }
  };
  unsigned k_c = 0;
  auto acquire = [&]() -> const double* {
    mbar_wait(s.bar + (k_c & 1u), (k_c >> 1) & 1u);
    return s.ring + (size_t)(k_c & 1u) * kStreamStage + lane;
  };
  auto release = [&]() {
    __syncwarp();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    ++k_c;
    issue_next();
  };
  issue_next();
  issue_next();
  int c = 0;
  for (int it = 0; it < n_it; ++it) {
    const long long tile = unit_of(gw + (long long)it * nW, c);
    double Linv[21], yv[6];
    {
      const double* st = acquire();
#pragma unroll
      for (int i = 0; i < 21; ++i) Linv[i] = st[i * kTile];
#pragma unroll
      for (int i = 0; i < 6; ++i) yv[i] = st[(21 + i) * kTile];
      release();
    }
    double zy[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) zy[i] = 0.0;
    double* z = p.Z + ((size_t)(tile * nc + c * 12) * 6) * kTile + lane;
    double Jl[9], Rc[9], K[9];
    {
      const double* st = acquire();
      double pose[6] = {0.0, 0.0, 0.0, st[30 * kTile], st[31 * kTile], st[32 * kTile]};
#pragma unroll
      for (int i = 0; i < 9; ++i) Jl[i] = st[(21 + i) * kTile];
      k2c_stream_map(s.cam, c, pose, Rc, K);
      z_rows_range<6, 12>(st - 36 * kTile, Rc, K, Jl, Linv, yv, z, zy);   // stage row 0 = hand-off row 36
      release();
    }
    {
      const double* st = acquire();
      z_rows_range<0, 6>(st, Rc, K, Jl, Linv, yv, z, zy);
      release();
    }
    const double v = zy_lane_sum(zy, lane);
    if (lane < 12) s_zy[c * 12 + lane] += v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nc; i += kW * 32) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kW; ++w) t += s.zy_all[(size_t)w * nc + i];
    p.partZy[(size_t)blockIdx.x * nc + i] = t;
  }
}

// The evaluation that closes a solve needs neither Z nor the factor: only the pose gradient
// g_f = P'^T sum_c E'^T q_ext (and max |g|, the optimality).  One warp per frame tile reads the six q_ext rows of
// every live camera straight from the hand-off (coalesced 256-byte rows): 10 % of K2c's reads, none of its writes.
__global__ void __launch_bounds__(256) k2c_grad_kernel(const K2CParams p) {
  __shared__ double s_g[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, kW = blockDim.x >> 5;
  const int C = p.C, nc = 12 * C;
  const unsigned cmask = C >= 32 ? 0xffffffffu : (1u << C) - 1u;
  double gmax = 0.0;
  for (long long tile = (long long)blockIdx.x * kW + warp; tile < p.nTiles; tile += (long long)gridDim.x * kW) {
    const long long f = p.perm[tile * kTile + lane];
    const bool fvalid = f >= 0;
    double pose[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) pose[i] = fvalid ? p.x[(size_t)nc + f * 6 + i] : 0.0;
    double Jl[9];
    so3_left_jacobian(pose, Jl);
    double gpp[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (unsigned m = p.active[tile] & cmask; m; m &= m - 1) {
      const int c = __ffs(m) - 1;
      double Rc[9], K[9], qe[6];
      pose_map(p.cams[c], pose, Rc, K);
      const double* h = p.H + ((size_t)(tile * C + c) * kHandoff + 57) * kTile + lane;
#pragma unroll
      for (int i = 0; i < 6; ++i) qe[i] = h[i * kTile];
#pragma unroll
      for (int a = 0; a < 3; ++a) {   // the g'' part of pose_block_apply
        gpp[a] += Rc[a] * qe[0] + Rc[3 + a] * qe[1] + Rc[6 + a] * qe[2] + K[a] * qe[3] + K[3 + a] * qe[4] + K[6 + a] * qe[5];
        gpp[3 + a] += Rc[a] * qe[3] + Rc[3 + a] * qe[4] + Rc[6 + a] * qe[5];
      }
    }
    double gp[6];
#pragma unroll
    for (int i = 0; i < 3; ++i) {     // g = P'^T g'' (pose_block_factor)
      gp[i] = Jl[i] * gpp[0] + Jl[3 + i] * gpp[1] + Jl[6 + i] * gpp[2];
      gp[3 + i] = gpp[3 + i];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) gmax = fmax(gmax, fabs(gp[i]));
    if (fvalid) {
#pragma unroll
      for (int i = 0; i < 6; i += 2)
        *reinterpret_cast<double2*>(p.gpose + (size_t)f * 6 + i) = make_double2(gp[i], gp[i + 1]);
    }
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) gmax = fmax(gmax, __shfl_xor_sync(0xffffffffu, gmax, off));
  if (lane == 0) s_g[warp] = gmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    double g = 0.0;
    for (int w = 0; w < kW; ++w) g = fmax(g, s_g[w]);
    p.partG[blockIdx.x] = g;
  }
}

// ------------------------------------------------------------------ launchers
int k2c_stream_warps(int C) {
  int w = 12;
  while (w > 1 && k2c_stream_smem(C, w) > 227u * 1024u) --w;
  return w >= 12 ? 12 : (w >= 10 ? 10 : (w >= 8 ? 8 : 4));
}
// K2c variant (1 staged ring, 2 streamed pair) and the number of per-CTA partial outputs (Z y, max |g|) it produces.
int k2_consumer_parts(const Layout& L, int n_sm, int* mode) {
  // measured on B200: the staged ring wins where it applies (6 x 50,000: 0.076 ms against 0.023 + 0.050 ms for the
  // streamed pair, and clearly on small shards, where one tile per warp leaves most warps of the pose kernel idle);
  // the streamed pair serves every other camera count (16 x 25,000: 0.114 ms against 0.146 ms for one CTA per tile)
  if (L.C >= 2 && L.C <= 6) {
    *mode = 1;
    return (int)(L.nTiles < 2 * n_sm ? L.nTiles : 2 * n_sm);
  }
  *mode = 2;
  return (int)(L.nTiles < n_sm ? L.nTiles : n_sm);
}

int k2_producer_grid(const Layout& L, int n_sm, int* warps) {
  // 8 warps per CTA (2 per scheduler at 255 registers) once that still fills the GPU,
  // otherwise narrower CTAs so that small problems spread over more SMs.
  int w = 8;
  while (w > 1 && (long long)L.C * ((L.nTiles + w - 1) / w) < n_sm) w >>= 1;
  *warps = w;
  const long long groups = (long long)L.C * ((L.nTiles + w - 1) / w);
  return (int)(groups < n_sm ? groups : n_sm);
}

template <int kLoss, int kWarps>
static int launch_k2p_t(mcba_handle* h, const K2PParams& p) {
  const size_t smem = k2p_smem(p.C, p.N, kWarps);
  MCBA_CUDA(set_dynamic_smem((const void*)k2p_kernel<kLoss, kWarps>, smem));
  k2p_kernel<kLoss, kWarps><<<h->grid_frames, kWarps * 32, smem, h->stream>>>(p);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

template <int kLoss>
static int launch_k2p_w(mcba_handle* h, const K2PParams& p) {
  switch (h->prod_warps) {
    case 8: return launch_k2p_t<kLoss, 8>(h, p);
    case 4: return launch_k2p_t<kLoss, 4>(h, p);
    case 2: return launch_k2p_t<kLoss, 2>(h, p);
    default: return launch_k2p_t<kLoss, 1>(h, p);
  }
}

int launch_k2_producer(mcba_handle* h, const double* x, int loss, double f_scale) {
  const Layout& L = h->L;
  K2PParams p;
  p.C = L.C;
  p.N = L.N;
  p.F = L.F;
  p.nTiles = L.nTiles;
  p.obs = h->d_obs_tiled;
  p.perm = h->d_perm;
  p.units = h->d_units;
  p.unit_count = h->d_unit_count;
  p.gprefix = h->d_unit_count + 32;
  p.obj = h->d_obj;
  p.x = x;
  p.cams = h->d_cams;
  p.inv_c = 1.0 / f_scale;
  p.c2 = f_scale * f_scale;
  p.H = h->d_H;
  p.partU = h->d_partU;
  p.partS = h->d_partS;
  p.n_scalars = reinterpret_cast<const unsigned long long*>(h->d_unit_count + 96);
  if ((loss & 0xff) == kLossLinear) return launch_k2p_w<kLossLinear>(h, p);
  if (loss & kLossIrls) return launch_k2p_w<kLossSoftL1 | kLossIrls>(h, p);
  return launch_k2p_w<kLossSoftL1>(h, p);
}

// pose gradient and max |g| only (the closing evaluation of a solve); same partial-output count as K2c
int launch_k2_gradient(mcba_handle* h, const double* x) {
  const Layout& L = h->L;
  K2CParams p{};
  p.C = L.C;
  p.F = L.F;
  p.nTiles = L.nTiles;
  p.H = h->d_H;
  p.perm = h->d_perm;
  p.active = h->d_active;
  p.x = x;
  p.cams = h->d_cams;
  p.gpose = h->d_gpose;
  p.partG = h->d_partG;
  k2c_grad_kernel<<<h->n_part_c, 256, 0, h->stream>>>(p);   // 8 warps: one tile per warp at 6 x 50,000 (296 CTAs)
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

int launch_k2_consumer(mcba_handle* h, const double* x, double lambda) {
  const Layout& L = h->L;
  K2CParams p;
  p.C = L.C;
  p.F = L.F;
  p.nTiles = L.nTiles;
  p.H = h->d_H;
  p.perm = h->d_perm;
  p.active = h->d_active;
  p.units = h->d_units;
  p.unit_count = h->d_unit_count;
  p.x = x;
  p.cams = h->d_cams;
  p.lambda = lambda;
  p.Z = h->d_Z;
  p.Linv = h->d_Linv;
  p.y = h->d_y;
  p.JlTau = h->d_JlTau;
  p.gpose = h->d_gpose;
  p.D2pose = h->d_D2pose;
  p.partG = h->d_partG;
  p.partZy = h->d_partZy;
  if (h->k2c_mode == 2) {
    const int w = k2c_stream_warps(L.C);
    const size_t smem = k2c_stream_smem(L.C, w);
#define MCBA_K2C_STREAM(WV)                                                                                          \
  do {                                                                                                               \
    MCBA_CUDA(set_dynamic_smem((const void*)k2c_pose_kernel<WV>, smem));    \
    MCBA_CUDA(set_dynamic_smem((const void*)k2c_rows_kernel<WV>, smem));    \
    k2c_pose_kernel<WV><<<h->n_part_c, WV * 32, smem, h->stream>>>(p);                                               \
    k2c_rows_kernel<WV><<<h->n_part_c, WV * 32, smem, h->stream>>>(p);                                               \
    h->launches++;                                                                                                   \
  } while (0)
    switch (w) {
      case 12: MCBA_K2C_STREAM(12); break;
      case 10: MCBA_K2C_STREAM(10); break;
      case 8: MCBA_K2C_STREAM(8); break;
      default: MCBA_K2C_STREAM(4); break;
    }
#undef MCBA_K2C_STREAM
  } else {
    const int C = L.C;
    const size_t smem = sizeof(double) * ((size_t)C * kHandoff * kTile + (size_t)C * kXchg * kTile);
    const int grid = h->n_part_c;
#define MCBA_K2C_RING(CV)                                                                                          \
  do {                                                                                                             \
    MCBA_CUDA(set_dynamic_smem((const void*)k2c_ring_kernel<CV>, smem));  \
    k2c_ring_kernel<CV><<<grid, CV * 32, smem, h->stream>>>(p);                                                     \
  } while (0)
    switch (C) {
      case 2: MCBA_K2C_RING(2); break;
      case 3: MCBA_K2C_RING(3); break;
      case 4: MCBA_K2C_RING(4); break;
      case 5: MCBA_K2C_RING(5); break;
      default: MCBA_K2C_RING(6); break;
    }
#undef MCBA_K2C_RING
  }
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

}  // namespace mcba
