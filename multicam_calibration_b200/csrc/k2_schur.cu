// K2b: S_raw = sum_f Z_f Z_f^T and Z_f y_f (register-tiled SYRK over the frame
// axis), the finalisation of the packed reduced camera system in the true
// parameter basis and K3, the pose back-substitution (the damped Cholesky solve
// between the two is k3_solve.cu).
// Math: SURVEY.md Appendix A ("Schur form for this problem").
#include <cstdlib>

#include <cstring>

#include "k2_common.cuh"
#include "mcba_peer.cuh"

namespace mcba {

__host__ __device__ inline int tile_index(int bi, int bj, int nb) { return bi * nb - (bi * (bi - 1)) / 2 + (bj - bi); }

// ------------------------------------------------------------------ SYRK
// S_raw = sum_f Z_f Z_f^T over this rank's frames, on the FP64 tensor path (DMMA m8n8k4).
// Z is [tile][row][k*32 + lane]: per tile a row-major (nc x 192) matrix whose K axis is
// (pose column, frame).  Persistent CTAs stream (tile, K-chunk) stages into shared memory with
// bulk async copies (one per row, rows padded by 4 doubles so that the 8 x 4 fragment loads are
// bank-conflict free) through a 3-stage mbarrier ring; each of the 8 warps owns up to NT 8x8
// tiles of the upper block triangle and keeps their accumulators in registers for the whole
// kernel.  The A fragment of row block I and the B fragment of row block J are the same
// mapping (lane -> row I*8 + lane/4, k = k0 + lane%4), so one load serves both roles.
// B200: DMMA and DFMA share the FP64 pipe at the same FMA rate (profiles/r01_b_ubench_*), but
// one DMMA replaces 8 DFMA issue slots and all the operand shuffling of a register-tiled SYRK.
constexpr int kSyrkStages = 3;
// consumer (DMMA) warps kW = 8 (<= 96 tiles: 6 cameras) or 15 (up to 300 tiles: 16 cameras without
// re-reading Z; 15 + 1 warps = 4 per scheduler leaves 128 registers per thread); warp kW is the copy producer
constexpr int kZK = 6 * kTile;    // K extent of one tile of Z

struct SyrkParams {
  const double* Z;
  int nc, nc8, nb8, nT;      // rows, rows padded to 8, row blocks, upper-triangle 8x8 tiles
  int nTiles;                // frame tiles
  int KW;                    // K width of one stage (divides 192, multiple of 4)
  double* part;              // [gridDim.x][nc8 * nc8]
};

// this warp's share of the nT tiles handled by CTA column blockIdx.y: [t0, t0 + cnt)
template <int kSyrkWarps>
__device__ __forceinline__ void syrk_tile_range(const SyrkParams& p, int warp, int& t0, int& cnt) {
  const int per_col = (p.nT + (int)gridDim.y - 1) / (int)gridDim.y;
  const int c0 = (int)blockIdx.y * per_col;
  const int n = min(per_col, p.nT - c0) > 0 ? min(per_col, p.nT - c0) : 0;
  const int base = n / kSyrkWarps, extra = n % kSyrkWarps;
  // the last `extra` warps take one more tile (keeps the scheduler that also hosts the producer warp light)
  const int first_big = kSyrkWarps - extra;
  cnt = base + (warp >= first_big ? 1 : 0);
  t0 = c0 + warp * base + (warp > first_big ? warp - first_big : 0);
}

constexpr int kSyrkSlots = 20;   // tiles per warp: 15 warps x 20 = the 300 tiles of 16 cameras
template <int NT>
__device__ __forceinline__ void syrk_stage(const double* __restrict__ st, const int (&offA)[kSyrkSlots],
                                           const int (&offB)[kSyrkSlots], double (&acc)[kSyrkSlots][2], int KW) {
  // K-steps in flight per warp: enough independent fragment loads to cover the shared-memory
  // latency without spilling the accumulators
  constexpr int kUnroll = NT <= 6 ? 4 : (NT <= 12 ? 2 : 1);
#pragma unroll kUnroll
  for (int k0 = 0; k0 < KW; k0 += 4) {
#pragma unroll
    for (int sl = 0; sl < NT; ++sl) {
      const double a = st[offA[sl] + k0];
      const double b = st[offB[sl] + k0];
      dmma_m8n8k4(acc[sl][0], acc[sl][1], a, b);
    }
  }
}

// ---- compile-time tile lists (common camera counts): which 8x8 tiles a warp owns is then known
// to the compiler, so the A fragment of a row block is loaded ONCE per run of tiles that share it
// and a diagonal tile reuses it as its B fragment -- plain straight-line code, no run-time masks
// (those were measured slower, scripts/experiments/README.md).  The fragment loads are what bounds
// the SYRK (shared-memory bandwidth): ~7 instead of 12 per k-step at 6 cameras.
__host__ __device__ constexpr int st_tile_i(int t, int nb8) {
  int I = 0, rem = t;
  while (I < nb8 - 1 && rem >= nb8 - I) { rem -= nb8 - I; ++I; }
  return I;
}
__host__ __device__ constexpr int st_tile_j(int t, int nb8) {
  int I = 0, rem = t;
  while (I < nb8 - 1 && rem >= nb8 - I) { rem -= nb8 - I; ++I; }
  return I + rem;
}
template <int kW, int NB8, int WARP>
struct StaticTiles {   // mirrors syrk_tile_range for gridDim.y == 1
  static constexpr int nT = NB8 * (NB8 + 1) / 2;
  static constexpr int base = nT / kW, extra = nT % kW, first_big = kW - extra;
  static constexpr int cnt = base + (WARP >= first_big ? 1 : 0);
  static constexpr int t0 = WARP * base + (WARP > first_big ? WARP - first_big : 0);
};

template <int kW, int NB8, int WARP, int SL>
struct StaticStep {
  using T = StaticTiles<kW, NB8, WARP>;
  static __device__ __forceinline__ void run(const double* __restrict__ st, int ld8, double& a,
                                             double (&acc)[kSyrkSlots][2]) {
    if constexpr (SL < T::cnt) {
      constexpr int t = T::t0 + SL;
      constexpr int I = st_tile_i(t, NB8), J = st_tile_j(t, NB8);
      constexpr int Iprev = SL > 0 ? st_tile_i(t - 1, NB8) : -1;
      if constexpr (I != Iprev) a = st[I * ld8];
      double b = a;
      if constexpr (I != J) b = st[J * ld8];
      dmma_m8n8k4(acc[SL][0], acc[SL][1], a, b);
      StaticStep<kW, NB8, WARP, SL + 1>::run(st, ld8, a, acc);
    }
  }
  static __device__ __forceinline__ void store(double* __restrict__ out, int nc8, int lane,
                                               const double (&acc)[kSyrkSlots][2]) {
    if constexpr (SL < T::cnt) {
      constexpr int t = T::t0 + SL;
      constexpr int I = st_tile_i(t, NB8), J = st_tile_j(t, NB8);
      *reinterpret_cast<double2*>(out + (size_t)(I * 8 + (lane >> 2)) * nc8 + J * 8 + 2 * (lane & 3)) =
          make_double2(acc[SL][0], acc[SL][1]);
      StaticStep<kW, NB8, WARP, SL + 1>::store(out, nc8, lane, acc);
    }
  }
};

// the whole consumer loop of one warp with a compile-time tile list
template <int kW, int NB8, int WARP>
__device__ __forceinline__ void syrk_consume_static(const SyrkParams& p, const double* stages, size_t stage_doubles,
                                                    int ld, int n_units, unsigned long long* full_bar,
                                                    unsigned long long* empty_bar, int lane) {
  using T = StaticTiles<kW, NB8, WARP>;
  constexpr int kUnroll = T::cnt <= 6 ? 8 : (T::cnt <= 12 ? 2 : 1);
  double acc[kSyrkSlots][2];
#pragma unroll
  for (int s = 0; s < kSyrkSlots; ++s) acc[s][0] = acc[s][1] = 0.0;
  const int lane_off = (lane >> 2) * ld + (lane & 3);
  const int ld8 = 8 * ld;
  for (int unit = 0; unit < n_units; ++unit) {
    const int s = unit % kSyrkStages;
    mbar_wait(&full_bar[s], (unsigned)((unit / kSyrkStages) & 1));
    const double* st = stages + (size_t)s * stage_doubles + lane_off;
#pragma unroll kUnroll
    for (int k0 = 0; k0 < p.KW; k0 += 4) {
      double a = 0.0;
      StaticStep<kW, NB8, WARP, 0>::run(st + k0, ld8, a, acc);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
  }
  StaticStep<kW, NB8, WARP, 0>::store(p.part + (size_t)blockIdx.x * p.nc8 * p.nc8, p.nc8, lane, acc);
}

template <int kW, int NB8, int WARP = 0>
__device__ __forceinline__ void syrk_dispatch_static(int warp, const SyrkParams& p, const double* stages,
                                                     size_t stage_doubles, int ld, int n_units,
                                                     unsigned long long* full_bar, unsigned long long* empty_bar, int lane) {
  if constexpr (WARP < kW) {
    if (warp == WARP) syrk_consume_static<kW, NB8, WARP>(p, stages, stage_doubles, ld, n_units, full_bar, empty_bar, lane);
    else syrk_dispatch_static<kW, NB8, WARP + 1>(warp, p, stages, stage_doubles, ld, n_units, full_bar, empty_bar, lane);
  }
}

template <int kSyrkWarps, int NB8 = 0>
__global__ void __launch_bounds__((kSyrkWarps + 1) * 32, 1) k2_syrk_kernel(const SyrkParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ unsigned long long full_bar[kSyrkStages], empty_bar[kSyrkStages];
  double* stages = reinterpret_cast<double*>(smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ld = p.KW + 4;
  const size_t stage_doubles = (size_t)p.nc8 * ld;
  const int chunks = kZK / p.KW;
  const int my_tiles = p.nTiles > (int)blockIdx.x ? (p.nTiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int n_units = my_tiles * chunks;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kSyrkStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], kSyrkWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // padding rows nc .. nc8-1 are never written by the copies: zero them once
  for (int s = 0; s < kSyrkStages; ++s)
    for (int i = threadIdx.x; i < (p.nc8 - p.nc) * ld; i += blockDim.x) stages[s * stage_doubles + (size_t)p.nc * ld + i] = 0.0;
  __syncthreads();

  if (warp == kSyrkWarps) {
    // ---------------- producer: one bulk copy per row of the (tile, K-chunk) stage ----------------
    int tile = blockIdx.x, ch = 0;
    for (int unit = 0; unit < n_units; ++unit) {
      const int s = unit % kSyrkStages;
      if (unit >= kSyrkStages) mbar_wait(&empty_bar[s], (unsigned)((unit / kSyrkStages - 1) & 1));
      double* dst = stages + (size_t)s * stage_doubles;
      const double* src = p.Z + ((size_t)tile * p.nc) * kZK + (size_t)ch * p.KW;
      if (lane == 0) mbar_expect_tx(&full_bar[s], (unsigned)(p.nc * p.KW * sizeof(double)));
      __syncwarp();
      for (int r = lane; r < p.nc; r += 32)
        tma_load_1d(dst + (size_t)r * ld, src + (size_t)r * kZK, (unsigned)(p.KW * sizeof(double)), &full_bar[s]);
      if (++ch == chunks) { ch = 0; tile += gridDim.x; }
    }
    return;
  }

  if constexpr (NB8 > 0) {   // compile-time tile lists (gridDim.y == 1)
    syrk_dispatch_static<kSyrkWarps, NB8>(warp, p, stages, stage_doubles, ld, n_units, full_bar, empty_bar, lane);
    return;
  }
  // ---------------- consumers: up to 12 tiles of the upper block triangle per warp ----------------
  int t0, cnt;
  syrk_tile_range<kSyrkWarps>(p, warp, t0, cnt);
  int offA[kSyrkSlots], offB[kSyrkSlots];
  {
    int I = 0, rem = t0;
    while (I < p.nb8 - 1 && rem >= p.nb8 - I) { rem -= p.nb8 - I; ++I; }
    int J = I + rem;
    if (J >= p.nb8) { I = 0; J = 0; }   // empty range
#pragma unroll
    for (int s = 0; s < kSyrkSlots; ++s) {
      offA[s] = (I * 8 + (lane >> 2)) * ld + (lane & 3);
      offB[s] = (J * 8 + (lane >> 2)) * ld + (lane & 3);
      if (s + 1 < cnt) { ++J; if (J == p.nb8) { ++I; J = I; } }
    }
  }
  double acc[kSyrkSlots][2];
#pragma unroll
  for (int s = 0; s < kSyrkSlots; ++s) acc[s][0] = acc[s][1] = 0.0;

  for (int unit = 0; unit < n_units; ++unit) {
    const int s = unit % kSyrkStages;
    mbar_wait(&full_bar[s], (unsigned)((unit / kSyrkStages) & 1));
    const double* st = stages + (size_t)s * stage_doubles;
    switch (cnt) {   // warp-uniform: exact trip counts, no predicated DMMA
      case 1: syrk_stage<1>(st, offA, offB, acc, p.KW); break;
      case 2: syrk_stage<2>(st, offA, offB, acc, p.KW); break;
      case 3: syrk_stage<3>(st, offA, offB, acc, p.KW); break;
      case 4: syrk_stage<4>(st, offA, offB, acc, p.KW); break;
      case 5: syrk_stage<5>(st, offA, offB, acc, p.KW); break;
      case 6: syrk_stage<6>(st, offA, offB, acc, p.KW); break;
      case 7: syrk_stage<7>(st, offA, offB, acc, p.KW); break;
      case 8: syrk_stage<8>(st, offA, offB, acc, p.KW); break;
      case 9: syrk_stage<9>(st, offA, offB, acc, p.KW); break;
      case 10: syrk_stage<10>(st, offA, offB, acc, p.KW); break;
      case 11: syrk_stage<11>(st, offA, offB, acc, p.KW); break;
      case 12: syrk_stage<12>(st, offA, offB, acc, p.KW); break;
      case 13: syrk_stage<13>(st, offA, offB, acc, p.KW); break;
      case 14: syrk_stage<14>(st, offA, offB, acc, p.KW); break;
      case 15: syrk_stage<15>(st, offA, offB, acc, p.KW); break;
      case 16: syrk_stage<16>(st, offA, offB, acc, p.KW); break;
      case 17: syrk_stage<17>(st, offA, offB, acc, p.KW); break;
      case 18: syrk_stage<18>(st, offA, offB, acc, p.KW); break;
      case 19: syrk_stage<19>(st, offA, offB, acc, p.KW); break;
      case 20: syrk_stage<20>(st, offA, offB, acc, p.KW); break;
      default: break;
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
  }

  // one partial per CTA column; tiles of different warps / blockIdx.y are disjoint
  double* out = p.part + (size_t)blockIdx.x * p.nc8 * p.nc8;
  {
    int I = 0, rem = t0;
    while (I < p.nb8 - 1 && rem >= p.nb8 - I) { rem -= p.nb8 - I; ++I; }
    int J = I + rem;
#pragma unroll
    for (int s = 0; s < kSyrkSlots; ++s) {
      if (s < cnt) {
        *reinterpret_cast<double2*>(out + (size_t)(I * 8 + (lane >> 2)) * p.nc8 + J * 8 + 2 * (lane & 3)) =
            make_double2(acc[s][0], acc[s][1]);
        ++J;
        if (J == p.nb8) { ++I; J = I; }
      }
    }
  }
}

struct SyrkConfig {
  int warps, gy, KW;
  size_t smem;
};

static SyrkConfig syrk_config(int nc) {
  SyrkConfig c;
  const int nc8 = (nc + 7) / 8 * 8, nb8 = nc8 / 8, nT = nb8 * (nb8 + 1) / 2;
  c.warps = nT <= 8 * 12 ? 8 : 15;
  c.gy = (nT + c.warps * kSyrkSlots - 1) / (c.warps * kSyrkSlots);   // at most kSyrkSlots tiles per warp
  static const int widths[] = {192, 96, 64, 48, 32, 16, 8};
  c.KW = 8;
  for (int w : widths) {
    if ((size_t)kSyrkStages * nc8 * (w + 4) * sizeof(double) <= 220 * 1024) { c.KW = w; break; }
  }
  c.smem = (size_t)kSyrkStages * nc8 * (c.KW + 4) * sizeof(double);
  return c;
}

int syrk_grid(int nc, long long F, int n_sm) {
  (void)nc;
  const long long tiles = (F + kTile - 1) / kTile;
  return (int)(tiles < n_sm ? tiles : n_sm);
}

// Block count of the compiled tile list the SYRK uses for a 12C-wide system, 0 when the tiles are listed at
// run time (more than one CTA row, no compiled list for this width, or MCBA_SYRK_RUNTIME set).
static int syrk_static_nb(const SyrkConfig& c, int nc) {
  static const bool no_static = getenv("MCBA_SYRK_RUNTIME") != nullptr;   // A/B: run-time tile lists
  const int nb8 = (nc + 7) / 8;
  if (c.gy != 1 || no_static) return 0;
  if (c.warps == 8) return (nb8 == 3 || nb8 == 5 || nb8 == 6 || nb8 == 8 || nb8 == 9 || nb8 == 12) ? nb8 : 0;
  return (nb8 == 18 || nb8 == 24) ? nb8 : 0;
}

void syrk_plan(int nc, int* warps, int* gy, int* static_nb) {
  const SyrkConfig c = syrk_config(nc);
  *warps = c.warps;
  *gy = c.gy;
  *static_nb = syrk_static_nb(c, nc);
}

int launch_k2_syrk(mcba_handle* h) {
  const Layout& L = h->L;
  const SyrkConfig c = syrk_config(L.nc);
  SyrkParams p;
  p.Z = h->d_Z;
  p.nc = L.nc; p.nc8 = L.nc8; p.nb8 = L.nc8 / 8; p.nT = p.nb8 * (p.nb8 + 1) / 2;
  p.nTiles = (int)L.nTiles;
  p.KW = c.KW;
  p.part = h->d_partSyrk;
#define MCBA_SYRK(W, NB)                                                                                          \
  do {                                                                                                            \
    MCBA_CUDA(set_dynamic_smem((const void*)k2_syrk_kernel<W, NB>, c.smem)); \
    k2_syrk_kernel<W, NB><<<dim3(h->grid_syrk, c.gy), (W + 1) * 32, c.smem, h->stream>>>(p);                      \
  } while (0)
  const int nb = syrk_static_nb(c, L.nc);
  if (c.warps == 8) {
    switch (nb) {
      case 3: MCBA_SYRK(8, 3); break;    // 2 cameras
      case 5: MCBA_SYRK(8, 5); break;    // 3
      case 6: MCBA_SYRK(8, 6); break;    // 4
      case 8: MCBA_SYRK(8, 8); break;    // 5
      case 9: MCBA_SYRK(8, 9); break;    // 6
      case 12: MCBA_SYRK(8, 12); break;  // 8
      default: MCBA_SYRK(8, 0); break;
    }
  } else {
    switch (nb) {
      case 18: MCBA_SYRK(15, 18); break;  // 12 cameras
      case 24: MCBA_SYRK(15, 24); break;  // 16
      default: MCBA_SYRK(15, 0); break;
    }
  }
#undef MCBA_SYRK
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

// ------------------------------------------------------------------ finalize
// ONE kernel from the per-CTA partial sums of K2p / K2c / SYRK to the packed reduced camera system
// on every rank:
//   reduce    four CTAs per block (c, c'), c <= c', each add a quarter of the partials of the 12x12 block
//             of sum Z Z^T (and, on the diagonal, of U_raw, g_raw and Z y) in a fixed order -- 1024
//             threads, every load of a thread requested before anything waits (one memory round trip);
//             the last of the four to finish adds the quarters in index order and goes on alone;
//   basis     S0_cc' = T_c^T ( [c==c'] U_raw,c - (Z Z^T)_cc' ) T_c'  with
//             T_c = [[I6,0,0],[0,Jl,0],[0,[t]x Jl,I3]]  (rows raw [intr | m | G], cols true [intr | r | t]);
//   exchange  (multi-GPU, peer memory) the block goes straight from shared memory into slot [rank] of
//             every peer, the CTA publishes its flag, waits for the same CTA of the other ranks and
//             adds the slots in rank order (mcba_peer.cuh): no second launch, no round trip through
//             d_red, no grid-wide counter;
//   store     both mirror entries of the symmetric system, b, g_cam, diag(U), the scalars.
// The last CTA handles the scalars (cost, sum f^2, count, max |g_pose| per rank).
constexpr int kFinThreads = 1024;
constexpr int kFinSplit = 4; // CTAs that share the partial sums of one block (the last one to finish goes on)
constexpr int kFinGS = 7;    // partial groups of the 144-element block sum   (7 x 144 = 1008 threads)
constexpr int kFinGU = 8;    // partial groups of the 128-slot U / g sum      (8 x 128 = 1024)
constexpr int kFinGZ = 64;   // partial groups of the 12-element Z y sum      (64 x 12 = 768)
constexpr int kFinVals = 144 + kAcc + 12;   // per block: sum Z Z^T block | U_raw, g_raw slots | Z y

struct FinalizeParams {
  int C, nc, nc8, rank;
  const CamConst* cams;
  const double* partSyrk; int nPartSyrk;   // [nPartSyrk][nc8 * nc8], upper 8x8 block triangle valid
  const double* partU; int nPartU;         // [nPartU][C][kAcc]
  const double* partZy; int nPartZy;       // [nPartZy][nc]
  const double* partS;                     // [nPartU][kRsNum]  (K2p: cost, sum f^2, count)
  const double* partG; long long nPartG;   // [nPartG] max |pose gradient| per K2c partial
  double* scratch;                         // [pairs][kFinSplit][kFinVals]
  unsigned int* counter;                   // [pairs], zero between launches
  double* red;
  long long offS, offB, offG, offDiag, offScal, offRank;
  int exchange;                            // 1: sum over ranks through peer memory (pv valid)
  PeerView pv;
};

__device__ __forceinline__ void build_T(const CamConst& cam, double* T /*[144]*/, int tid) {
  if (tid < 144) {
    const int r = tid / 12, q = tid % 12;
    double v = (r == q) ? 1.0 : 0.0;
    if (r >= 6 && r < 9 && q >= 6 && q < 9) v = cam.Jl[(r - 6) * 3 + (q - 6)];
    if (r >= 9 && q >= 6 && q < 9) v = cam.tJ[(r - 9) * 3 + (q - 6)];
    T[tid] = v;
  }
}

// Partials lo + g, lo + g + G, ... (< hi) of one element: the first eight are REQUESTED here (independent
// loads, nothing waits on them yet) and summed by strided_sum_finish in a fixed order, so that a thread can
// have the loads of several segments in flight at once.
struct StridedLoads {
  double a[8];
  const double* src;
  size_t stride;
  int next, hi, G;
};
__device__ __forceinline__ void strided_sum_start(StridedLoads& L, const double* __restrict__ src, size_t stride, int lo, int hi,
                                                  int g, int G) {
  L.src = src; L.stride = stride; L.hi = hi; L.G = G;
  int p = lo + g;
#pragma unroll
  for (int u = 0; u < 8; ++u) L.a[u] = (p + u * G < hi) ? __ldcg(src + (size_t)(p + u * G) * stride) : 0.0;
  L.next = p + 8 * G;
}
__device__ __forceinline__ double strided_sum_finish(StridedLoads& L) {
  for (int p = L.next; p < L.hi; p += 8 * L.G) {   // more than eight per thread (many K2c partials): further rounds
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (p + u * L.G < L.hi) L.a[u] += __ldcg(L.src + (size_t)(p + u * L.G) * L.stride);
  }
  return ((L.a[0] + L.a[1]) + (L.a[2] + L.a[3])) + ((L.a[4] + L.a[5]) + (L.a[6] + L.a[7]));
}

// vals[i] <- sum over ranks of vals[i], exchanged at offset off[i] of the slots (off < 0: not exchanged;
// no-op without peers); vals/off: this CTA's outputs in shared memory
__device__ __forceinline__ void exchange_values(const FinalizeParams& p, double* vals, const int* off, int n, int cta) {
  if (!p.exchange) return;
  const PeerView& pv = p.pv;
  for (int s = 0; s < pv.nranks; ++s) {
    double* dst = peer_slot_of(pv, (pv.rank + s) % pv.nranks);
    for (int i = threadIdx.x; i < n; i += blockDim.x)
      if (off[i] >= 0) dst[off[i]] = vals[i];
  }
  peer_publish(pv, cta);
  peer_wait(pv, cta);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    if (off[i] < 0) continue;
    double acc = 0.0;
    for (int r = 0; r < pv.nranks; ++r) acc += __ldcg(peer_slot_from(pv, r) + off[i]);
    vals[i] = acc;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kFinThreads, 1) finalize_kernel(const FinalizeParams p) {
  __shared__ double sm_red[kFinGU * kAcc];      // partial-group sums (largest: 8 x 128; Z y: 64 x 12; block: 7 x 144)
  __shared__ double M[144], X[144], Tc[144], Tp[144], Ur[kAcc], vec[24];
  __shared__ double vals[192];                  // this CTA's outputs: 144 block entries | diag 12 | g 12 | b 12
  __shared__ int off[192];
  __shared__ bool s_last;
  const int tid = threadIdx.x;
  const int nPairs = p.C * (p.C + 1) / 2;
  const int blk = blockIdx.x / kFinSplit, part = blockIdx.x % kFinSplit;
  if (blk == nPairs) {  // ---------------- scalars (one CTA)
    if (part != 0) return;
    double a = 0, b = 0, k = 0, g = 0;
    for (int i = tid; i < p.nPartU; i += blockDim.x) {
      const double* s = p.partS + (size_t)i * kRsNum;
      a += s[kRsCost]; b += s[kRsSumSq]; k += s[kRsCount];
    }
    for (long long i = tid; i < p.nPartG; i += blockDim.x) g = fmax(g, p.partG[i]);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
      k += __shfl_xor_sync(0xffffffffu, k, o);
      g = fmax(g, __shfl_xor_sync(0xffffffffu, g, o));
    }
    if ((tid & 31) == 0) { sm_red[(tid >> 5) * 4] = a; sm_red[(tid >> 5) * 4 + 1] = b; sm_red[(tid >> 5) * 4 + 2] = k; sm_red[(tid >> 5) * 4 + 3] = g; }
    __syncthreads();
    const int nv = kRsNum + kMaxRanks;
    if (tid < nv) { vals[tid] = 0.0; off[tid] = (int)(tid < kRsNum ? p.offScal + tid : p.offRank + (tid - kRsNum)); }
    __syncthreads();
    if (tid == 0) {
      a = b = k = g = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += sm_red[w * 4]; b += sm_red[w * 4 + 1]; k += sm_red[w * 4 + 2]; g = fmax(g, sm_red[w * 4 + 3]); }
      vals[kRsCost] = a; vals[kRsSumSq] = b; vals[kRsCount] = k;
      vals[kRsNum + p.rank] = g;
    }
    __syncthreads();
    exchange_values(p, vals, off, nv, nPairs);
    if (tid < nv) p.red[off[tid]] = vals[tid];
    return;
  }
  // ---------------- block (c, cp), c <= cp; this CTA's quarter of the partials
  int c = 0, rem = blk;
  while (rem >= p.C - c) { rem -= p.C - c; ++c; }
  const int cp = c + rem;
  const bool diag = c == cp;
  // request every load of the thread before anything waits: block sum, and on the diagonal U / g and Z y
  StridedLoads lS, lU, lZ;
  const bool hasS = tid < 144 * kFinGS, hasZ = diag && tid < 12 * kFinGZ;
  if (hasS) {
    const int e = tid % 144, g = tid / 144;
    const int r = 12 * c + e / 12, q = 12 * cp + e % 12;
    // r <= q element-wise within a diagonal camera block is not guaranteed: pick the stored 8x8 tile
    const size_t idx = (r / 8 <= q / 8) ? (size_t)r * p.nc8 + q : (size_t)q * p.nc8 + r;
    strided_sum_start(lS, p.partSyrk + idx, (size_t)p.nc8 * p.nc8, p.nPartSyrk * part / kFinSplit,
                      p.nPartSyrk * (part + 1) / kFinSplit, g, kFinGS);
  }
  if (diag) {
    const int e = tid % kAcc, g = tid / kAcc;
    strided_sum_start(lU, p.partU + (size_t)c * kAcc + e, (size_t)p.C * kAcc, p.nPartU * part / kFinSplit,
                      p.nPartU * (part + 1) / kFinSplit, g, kFinGU);
  }
  if (hasZ) {
    const int e = tid % 12, g = tid / 12;
    strided_sum_start(lZ, p.partZy + 12 * c + e, (size_t)p.nc, p.nPartZy * part / kFinSplit,
                      p.nPartZy * (part + 1) / kFinSplit, g, kFinGZ);
  }
  double* mine = p.scratch + ((size_t)blk * kFinSplit + part) * kFinVals;
  if (hasS) sm_red[tid] = strided_sum_finish(lS);
  __syncthreads();
  if (tid < 144) {
    double t = 0.0;
#pragma unroll
    for (int g = 0; g < kFinGS; ++g) t += sm_red[g * 144 + tid];
    mine[tid] = t;
  }
  if (diag) {
    __syncthreads();
    sm_red[tid] = strided_sum_finish(lU);
    __syncthreads();
    if (tid < kAcc) {
      double t = 0.0;
#pragma unroll
      for (int g = 0; g < kFinGU; ++g) t += sm_red[g * kAcc + tid];
      mine[144 + tid] = t;
    }
    __syncthreads();
    if (hasZ) sm_red[tid] = strided_sum_finish(lZ);
    __syncthreads();
    if (tid < 12) {
      double t = 0.0;
      for (int g = 0; g < kFinGZ; ++g) t += sm_red[g * 12 + tid];
      mine[144 + kAcc + tid] = t;
    }
  }
  // the last of the block's kFinSplit CTAs to get here adds the quarters (in index order) and goes on
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(p.counter + blk, 1u) == kFinSplit - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (tid == 0) p.counter[blk] = 0;
  const double* all = p.scratch + (size_t)blk * kFinSplit * kFinVals;
  if (tid < kFinVals && (diag || tid < 144)) {
    double t = 0.0;
#pragma unroll
    for (int r = 0; r < kFinSplit; ++r) t += __ldcg(all + (size_t)r * kFinVals + tid);
    if (tid < 144) M[tid] = -t;
    else if (tid < 144 + kAcc) Ur[tid - 144] = t;
    else vec[12 + (tid - 144 - kAcc)] = t;      // Z y, combined with g_raw below
  }
  build_T(p.cams[c], Tc, tid);
  build_T(p.cams[cp], Tp, tid);
  __syncthreads();
  if (diag) {
    if (tid < 12) {
      const double graw = Ur[acc_slot_q(tid)];
      vec[tid] = graw;
      vec[12 + tid] = graw - vec[12 + tid];
    }
    if (tid < 144) {
      const int slot = acc_slot(tid / 12, tid % 12);   // -1: structurally zero product (fx.fy, fx.cy, cx.fy, cx.cy)
      if (slot >= 0) M[tid] += Ur[slot];
    }
    // diag(T^T U_raw T), b, g_cam: X = U_raw T
    if (tid < 144) {
      const int i = tid / 12, j = tid % 12;
      double s = 0;
#pragma unroll
      for (int k = 0; k < 12; ++k) {
        const int sl = acc_slot(i, k);
        s += (sl >= 0 ? Ur[sl] : 0.0) * Tc[k * 12 + j];
      }
      X[tid] = s;
    }
    __syncthreads();
    if (tid < 12) {
      double d = 0, g = 0, b = 0;
#pragma unroll
      for (int k = 0; k < 12; ++k) {
        d += Tc[k * 12 + tid] * X[k * 12 + tid];
        g += Tc[k * 12 + tid] * vec[k];
        b += Tc[k * 12 + tid] * vec[12 + k];
      }
      vals[144 + tid] = d; off[144 + tid] = (int)(p.offDiag + 12 * c + tid);
      vals[156 + tid] = g; off[156 + tid] = (int)(p.offG + 12 * c + tid);
      vals[168 + tid] = b; off[168 + tid] = (int)(p.offB + 12 * c + tid);
    }
    __syncthreads();
  }
  // S0 = Tc^T M Tp
  if (tid < 144) {
    const int i = tid / 12, j = tid % 12;
    double s = 0;
#pragma unroll
    for (int k = 0; k < 12; ++k) s += M[i * 12 + k] * Tp[k * 12 + j];
    X[tid] = s;
  }
  __syncthreads();
  if (tid < 144) {
    const int i = tid / 12, j = tid % 12;
    double s = 0;
#pragma unroll
    for (int k = 0; k < 12; ++k) s += Tc[k * 12 + i] * X[k * 12 + j];
    // diagonal blocks: only the (i <= j) entry is exchanged, kept and mirrored (exact symmetry)
    vals[tid] = s;
    off[tid] = (diag && i > j) ? -1 : (int)(p.offS + (size_t)(12 * c + i) * p.nc + 12 * cp + j);
  }
  __syncthreads();
  const int nv = diag ? 180 : 144;
  exchange_values(p, vals, off, nv, blk);
  if (tid < 144) {
    const int i = tid / 12, j = tid % 12;
    if (!diag || i <= j) {
      const double s = vals[tid];
      const int r = 12 * c + i, q = 12 * cp + j;
      p.red[p.offS + (size_t)r * p.nc + q] = s;
      p.red[p.offS + (size_t)q * p.nc + r] = s;
    }
  } else if (diag && tid < 180) {
    p.red[off[tid]] = vals[tid];
  }
}

int launch_finalize(mcba_handle* h, bool exchange) {
  const Layout& L = h->L;
  FinalizeParams p;
  p.C = L.C; p.nc = L.nc; p.nc8 = L.nc8; p.rank = h->rank;
  p.cams = h->d_cams;
  p.partSyrk = h->d_partSyrk; p.nPartSyrk = h->grid_syrk;
  p.partU = h->d_partU; p.nPartU = h->grid_frames;
  p.partZy = h->d_partZy; p.nPartZy = h->n_part_c;
  p.partS = h->d_partS; p.partG = h->d_partG; p.nPartG = h->n_part_c;
  p.scratch = h->d_fin_scratch; p.counter = h->d_fin_counter;
  p.red = h->d_red;
  p.offS = L.offS; p.offB = L.offB; p.offG = L.offG; p.offDiag = L.offDiag; p.offScal = L.offScal; p.offRank = L.offRank;
  p.exchange = exchange ? 1 : 0;
  if (exchange) p.pv = peer_next_call(h);
  else memset(&p.pv, 0, sizeof(p.pv));
  finalize_kernel<<<(L.C * (L.C + 1) / 2 + 1) * kFinSplit, kFinThreads, 0, h->stream>>>(p);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

// ------------------------------------------------------------------ K3 back-substitution
// delta_f = -L^-T (y_f + Z_f^T delta_raw),  x_new = x + delta.  HBM bound: the kernel's work is to
// stream Z once (576 B per (camera, frame)).  Persistent CTAs of four warps; every warp owns whole
// frame tiles (lane = frame) and pulls its tile's Z block through its OWN ring of three 18 KB
// shared-memory stages with bulk asynchronous copies (12 rows = one camera per stage, contiguous in
// Z): 220 KB in flight per SM without a single register or a dependent global load, the warp's lane
// 0 re-arms a stage as soon as the warp has consumed it (same warp: no empty barrier).  y, L^-1 and
// the Marquardt scaling of the tile are requested before the stream so their latency hides behind
// it; no CTA barrier in the tile loop.
constexpr int kBackWarps = 4;
constexpr int kBackRows = 12;                        // rows of Z per stage (12C is always a multiple)
constexpr int kBackStages = 3;
constexpr int kBackStageDoubles = kBackRows * 6 * kTile;
struct BackParams {
  int C, nc, rank;
  long long F, nTiles;
  const CamConst* cams;
  const int* perm;      // tile slot -> frame index in x (-1 = padding)
  const unsigned int* active;   // [tile] bit c: camera c has observations in the tile (its Z rows are zero otherwise)
  const double* x;
  double* x_new;
  const double* dcam;   // true-basis camera step (12C)
  const double* Z; const double* Linv; const double* y; const double* gpose; const double* D2pose;
  const double* D2cam; const double* gcam;
  double* part; unsigned int* counter; double* out;  // out[0..3] = |dx|^2, |x|^2, g.dx, dx D2 dx
  const uint8_t* fixed; // [nc] held camera parameters: x copied, left out of the scalars (nullptr = none)
};

__global__ void __launch_bounds__(kBackWarps * 32, 1) backsub_kernel(const BackParams p) {
  extern __shared__ __align__(128) unsigned char bs_smem[];
  __shared__ unsigned long long full_bar[kBackWarps][kBackStages];
  __shared__ double s_part[kBackWarps][4];
  __shared__ bool s_last;
  const int tid = threadIdx.x, nc = p.nc, lane = tid & 31, warp = tid >> 5;
  double* ring = reinterpret_cast<double*>(bs_smem) + (size_t)warp * kBackStages * kBackStageDoubles;
  double* draw = reinterpret_cast<double*>(bs_smem) + (size_t)kBackWarps * kBackStages * kBackStageDoubles;   // [nc] camera step, raw basis
  for (int r = tid; r < nc; r += blockDim.x) {
    const int c = r / 12, i = r % 12;
    const double* d = p.dcam + 12 * c;
    const CamConst& cam = p.cams[c];
    double v;
    if (i < 6) v = d[i];
    else if (i < 9) v = cam.Jl[(i - 6) * 3] * d[6] + cam.Jl[(i - 6) * 3 + 1] * d[7] + cam.Jl[(i - 6) * 3 + 2] * d[8];
    else v = cam.tJ[(i - 9) * 3] * d[6] + cam.tJ[(i - 9) * 3 + 1] * d[7] + cam.tJ[(i - 9) * 3 + 2] * d[8] + d[i];
    draw[r] = v;
  }
  if (lane == 0) {
    for (int s = 0; s < kBackStages; ++s) mbar_init(&full_bar[warp][s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // this warp's tiles: gw, gw + W, ...; its stream of stages: the LIVE (tile, camera) units in order -- the Z rows
  // of a camera that did not see the tile's frames are zero (never written) and are not read either
  const long long gw = (long long)blockIdx.x * kBackWarps + warp, W = (long long)gridDim.x * kBackWarps;
  const int chunks = nc / kBackRows;
  const unsigned cmask = chunks >= 32 ? 0xffffffffu : (1u << chunks) - 1u;
  const long long my_tiles = p.nTiles > gw ? (p.nTiles - gw + W - 1) / W : 0;
  long long it_i = 0, k_i = 0;             // issue cursor (all lanes keep it; lane 0 issues)
  unsigned rem_i = my_tiles > 0 ? (p.active[gw] & cmask) : 0u;
  auto issue_next = [&]() {
    while (rem_i == 0) {
      if (++it_i >= my_tiles) { it_i = my_tiles; return; }
      rem_i = p.active[gw + it_i * W] & cmask;
    }
    const int ch = __ffs(rem_i) - 1;
    rem_i &= rem_i - 1;
    if (lane == 0) {
      const long long tile = gw + it_i * W;
      const int s = (int)(k_i % kBackStages);
      constexpr unsigned bytes = kBackStageDoubles * sizeof(double);
      mbar_expect_tx(&full_bar[warp][s], bytes);
      tma_load_1d(ring + (size_t)s * kBackStageDoubles, p.Z + ((size_t)tile * nc + (size_t)ch * kBackRows) * 6 * kTile, bytes,
                  &full_bar[warp][s]);
    }
    ++k_i;
  };
  for (int s0 = 0; s0 < kBackStages; ++s0)
    if (it_i < my_tiles) issue_next();

  double dd = 0, xx = 0, gd = 0, dDd = 0;
  long long q = 0;
  for (long long it = 0; it < my_tiles; ++it) {
    const long long tile = gw + it * W;
    const long long f = p.perm[tile * kTile + lane];
    double v[6], li[21], d2[6];
    {
      const double* yo = p.y + (size_t)tile * 6 * kTile + lane;
      const double* lo = p.Linv + (size_t)tile * 21 * kTile + lane;
      const double* so = p.D2pose + (size_t)tile * 6 * kTile + lane;
#pragma unroll
      for (int k = 0; k < 6; ++k) { v[k] = yo[k * kTile]; d2[k] = so[k * kTile]; }
#pragma unroll
      for (int k = 0; k < 21; ++k) li[k] = lo[k * kTile];
    }
    double s[6] = {0, 0, 0, 0, 0, 0};
    for (unsigned m = p.active[tile] & cmask; m; m &= m - 1, ++q) {
      const int ch = __ffs(m) - 1;
      const int st = (int)(q % kBackStages);
      mbar_wait(&full_bar[warp][st], (unsigned)((q / kBackStages) & 1));
      const double* z = ring + (size_t)st * kBackStageDoubles + lane;
      const double* dr = draw + ch * kBackRows;
#pragma unroll
      for (int r = 0; r < kBackRows; ++r) {
        const double w = dr[r];
#pragma unroll
        for (int k = 0; k < 6; ++k) s[k] = fma(z[(r * 6 + k) * kTile], w, s[k]);
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // our reads of the stage precede the copy that refills it
      __syncwarp();
      if (it_i < my_tiles) issue_next();
    }
    if (f >= 0) {
#pragma unroll
      for (int k = 0; k < 6; ++k) v[k] += s[k];
      double xo[6], gp[6];
#pragma unroll
      for (int k = 0; k < 6; k += 2) {
        const double2 a = *reinterpret_cast<const double2*>(p.x + (size_t)nc + (size_t)f * 6 + k);
        const double2 g = *reinterpret_cast<const double2*>(p.gpose + (size_t)f * 6 + k);
        xo[k] = a.x; xo[k + 1] = a.y; gp[k] = g.x; gp[k + 1] = g.y;
      }
      double xn[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        double d = 0.0;
#pragma unroll
        for (int j = k; j < 6; ++j) d -= li[j * (j + 1) / 2 + k] * v[j];
        xn[k] = xo[k] + d;
        const double sc = d2[k] == 0.0 ? 1.0 : d2[k];
        dd = fma(d, d, dd);
        xx = fma(xo[k], xo[k], xx);
        gd = fma(gp[k], d, gd);
        dDd = fma(sc * d, d, dDd);
      }
#pragma unroll
      for (int k = 0; k < 6; k += 2)
        *reinterpret_cast<double2*>(p.x_new + (size_t)nc + (size_t)f * 6 + k) = make_double2(xn[k], xn[k + 1]);
    }
  }
  if (blockIdx.x == 0 && warp == 0) {
    for (int r = lane; r < nc; r += 32) {
      const double d = p.dcam[r], xo = p.x[r];
      if (p.fixed && p.fixed[r]) { p.x_new[r] = xo; continue; }   // a copy: -0.0 survives
      p.x_new[r] = xo + d;
      if (p.rank == 0) {  // camera terms are counted once across ranks
        double d2 = p.D2cam[r];
        if (d2 == 0.0) d2 = 1.0;
        dd = fma(d, d, dd);
        xx = fma(xo, xo, xx);
        gd = fma(p.gcam[r], d, gd);
        dDd = fma(d2 * d, d, dDd);
      }
    }
  }
  // step scalars: lanes -> warp -> CTA (fixed order) -> per-CTA partial; the last CTA adds the partials
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    dd += __shfl_xor_sync(0xffffffffu, dd, off);
    xx += __shfl_xor_sync(0xffffffffu, xx, off);
    gd += __shfl_xor_sync(0xffffffffu, gd, off);
    dDd += __shfl_xor_sync(0xffffffffu, dDd, off);
  }
  if (lane == 0) { s_part[warp][0] = dd; s_part[warp][1] = xx; s_part[warp][2] = gd; s_part[warp][3] = dDd; }
  __syncthreads();
  if (tid == 0) {
    double* o = p.part + (size_t)blockIdx.x * 4;
#pragma unroll
    for (int qd = 0; qd < 4; ++qd) {
      double t = 0.0;
#pragma unroll
      for (int w = 0; w < kBackWarps; ++w) t += s_part[w][qd];
      o[qd] = t;
    }
    __threadfence();
    s_last = atomicAdd(p.counter, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last && warp == 0) {
    __threadfence();
    double a = 0, b = 0, c = 0, d = 0;
    for (unsigned i = lane; i < gridDim.x; i += 32) {
      a += __ldcg(p.part + i * 4); b += __ldcg(p.part + i * 4 + 1); c += __ldcg(p.part + i * 4 + 2); d += __ldcg(p.part + i * 4 + 3);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, off);
      b += __shfl_xor_sync(0xffffffffu, b, off);
      c += __shfl_xor_sync(0xffffffffu, c, off);
      d += __shfl_xor_sync(0xffffffffu, d, off);
    }
    if (lane == 0) {
      p.out[0] = a; p.out[1] = b; p.out[2] = c; p.out[3] = d;
      *p.counter = 0;
    }
  }
}

int launch_backsub(mcba_handle* h, const double* x, double* x_new, double lambda) {
  (void)lambda;
  const Layout& L = h->L;
  BackParams p;
  p.C = L.C; p.nc = L.nc; p.rank = h->rank; p.F = L.F; p.nTiles = L.nTiles;
  p.cams = h->d_cams; p.perm = h->d_perm; p.active = h->d_active; p.x = x; p.x_new = x_new; p.dcam = h->d_dcam;
  p.Z = h->d_Z; p.Linv = h->d_Linv; p.y = h->d_y; p.gpose = h->d_gpose; p.D2pose = h->d_D2pose;
  p.D2cam = h->d_D2cam; p.gcam = h->d_red + L.offG;
  p.fixed = h->any_fixed ? h->d_fixed : nullptr;
  p.part = h->d_scal + 64 + 3 * 4096;                                     // [grid_back][4]
  p.counter = reinterpret_cast<unsigned int*>(h->d_scal + 33);
  p.out = h->d_scal + 8;
  const size_t smem = sizeof(double) * ((size_t)kBackWarps * kBackStages * kBackStageDoubles + (size_t)((L.nc + 1) & ~1));
  MCBA_CUDA(set_dynamic_smem((const void*)backsub_kernel, smem));
  backsub_kernel<<<h->grid_back, kBackWarps * 32, smem, h->stream>>>(p);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

}  // namespace mcba
