// Internal (non-ABI) declarations shared by the translation units of libmcba.
#pragma once
#include <cuda_runtime.h>
#include <cusolverDn.h>
#include <stdint.h>

#include <string>

#include "../../include/mcba.h"
#include "mcba_math.cuh"

namespace mcba {

// Scalars that travel with the reduced camera system (appended to the packed
// buffer so that ONE all-reduce per evaluation carries everything).
enum RedScalar : int {
  kRsCost = 0,      // 0.5 * sum rho
  kRsSumSq = 1,     // sum f^2 (for the reprojection RMS)
  kRsCount = 2,     // number of finite scalar residuals
  kRsGmaxPose = 3,  // max |g| over this rank's pose gradients (NOT summed: slot per rank below)
  kRsNum = 8
};

constexpr int kMaxRanks = 64;
constexpr int kProfRing = 2048;
constexpr int kProfEvents = 5;   // CUDA events recorded per profiled evaluation
constexpr int kAcc = 128;  // accumulator slots of the raw 12x12 block + q per camera (layout: k2_common.cuh)

struct Layout {
  int C = 0, N = 0;
  long long F = 0, nTiles = 0, Fpad = 0;
  int nc = 0;   // 12 C
  int nc8 = 0;  // nc rounded up to a multiple of 8 (DMMA tile rows of the SYRK)
  // packed reduced buffer offsets (doubles)
  long long offS = 0, offB = 0, offG = 0, offDiag = 0, offScal = 0, offRank = 0, redLen = 0;
};

}  // namespace mcba

namespace mcba {
// cudaFuncAttributeMaxDynamicSharedMemorySize once per (kernel, device) and size instead of a driver call in front
// of every launch (the attribute is a maximum: it only ever grows).  ~1 us each, five of them per LM iteration on the
// host's critical path between the trial's scalars and the next evaluation.
cudaError_t set_dynamic_smem(const void* kernel, size_t bytes);
}
namespace mcba { struct HostPipe; }

struct mcba_handle {
  mcba::Layout L;
  mcba::HostPipe* pipe = nullptr;   // chunked upload + evaluation of mcba_build_reduced_host (mcba_api.cu), lazily built
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  int n_sm = 148;
  // observations
  double* d_obs_ref = nullptr;   // (C,F,N,2) reference layout
  double2* d_obs_tiled = nullptr;
  double* d_obj = nullptr;
  int* d_perm = nullptr;             // [2 Fpad] tile slot -> frame (-1 padding) | sort scratch
  unsigned int* d_mask = nullptr;    // [2 Fpad] ~visibility mask per frame | sort scratch
  unsigned int* d_active = nullptr;  // [nTiles] cameras with at least one observation in the tile
  int* d_units = nullptr;            // [C][nTiles] live tiles per camera, compacted
  int* d_unit_count = nullptr;       // [0..C) live units per camera | [32..32+C] group prefix for K2p | [96..97] finite scalars (u64, K2p's count)
  void* d_sort_tmp = nullptr;
  size_t sort_tmp_bytes = 0;
  long long* d_row_off = nullptr;  // [C * nBlk + 1] exclusive scan of finite scalars per K1 chunk
  unsigned int* d_chunk_rows = nullptr;   // [C * nBlk] per K1 chunk: rows (camera, frame) with at least one finite scalar (lazy)
  long long m = 0;                 // finite scalar residuals
  long long n_obs = 0;             // (c,f,n) with at least one finite scalar
  bool have_obs = false;
  bool have_rows = false;          // row offsets / m / n_obs computed (lazily, K1 only)
  // state
  double* d_x = nullptr;
  double* d_xtrial = nullptr;
  mcba::CamConst* d_cams = nullptr;
  double* d_H = nullptr;      // K2p -> K2c hand-off [tile][c][63][32]
  // second set of K2p outputs (allocated by the first mcba_lm_run): the LM loop evaluates K2p at
  // the TRIAL point into these and swaps the two sets when the step is accepted
  double* d_H_alt = nullptr;
  double* d_partU_alt = nullptr;
  double* d_partS_alt = nullptr;
  mcba::CamConst* d_cams_alt = nullptr;
  bool alt_stale = true;      // d_H_alt needs zeroing (dead units are never written)
  double* d_partG = nullptr;  // [n_part_c] max |pose gradient| per K2c partial
  double* d_partZy = nullptr; // [n_part_c][12C] partial sums of Z_f y_f
  double* d_Z = nullptr;
  double* d_Linv = nullptr;
  double* d_y = nullptr;
  double* d_JlTau = nullptr;  // [nTiles][12][32] J_l(rho_f) | tau_f (streamed K2c)
  double* d_gpose = nullptr;
  double* d_D2pose = nullptr;
  double* d_D2cam = nullptr;  // running max of diag(U) (true basis), 12C
  double* d_partU = nullptr;
  double* d_partS = nullptr;
  double* d_partSyrk = nullptr;
  double* d_Sraw = nullptr;   // [nc8 x nc8 raw-basis sum Z Z^T (upper 8x8 tiles) | Z y (12C) | U partial sums (C x kAcc)]
  double* d_red = nullptr;    // packed reduced system (see Layout)
  double* d_fin_scratch = nullptr;      // finalize: per block and quarter, the partial sums [pairs][4][144 + kAcc + 12]
  unsigned int* d_fin_counter = nullptr; // finalize: arrivals per block (zero between launches)
  double* d_Sd = nullptr;     // damped copy handed to potrf
  double* d_dcam = nullptr;   // [delta_cam true (12C) | delta_cam raw (12C)]
  double* d_scal = nullptr;   // step scalars (device), partials
  // camera parameters held at their initial values (mcba_set_fixed): 12C bytes, 0 / 1; the kernels get
  // d_fixed only while some entry is held (nullptr: the unmasked path)
  uint8_t h_fixed[12 * 32] = {};
  uint8_t* d_fixed = nullptr;
  bool any_fixed = false;
  double* h_pinned = nullptr; // pinned host mirror for small read-backs
  // mapped pinned block the LM loop polls: [16 doubles | sequence flag]; device aliases of the same memory
  double* h_signal_vals = nullptr;
  unsigned long long* h_signal_flag = nullptr;
  double* d_signal_vals = nullptr;
  unsigned long long* d_signal_flag = nullptr;
  unsigned long long signal_seq = 0;
  cudaEvent_t readback_done = nullptr;
  int n_part_c = 0;           // K2c partial outputs (one per persistent CTA)
  int k2c_mode = 0;           // 1 staged ring (2..6 cameras), 2 streamed pair (any other count; k2_frames.cu)
  int grid_frames = 0, prod_warps = 8, grid_syrk = 0, grid_cost = 0, grid_back = 0;
  // solver
  cusolverDnHandle_t solver = nullptr;
  double* d_work = nullptr;
  int lwork = 0;
  int* d_info = nullptr;
  // multi-GPU
  void* nccl_comm = nullptr;
  int rank = 0, nranks = 1;
  // peer-memory exchange (mcba_peer.cu): exchange block = [flags 2 x nranks x nflag | slots 2 x nranks x cap]
  void* peer_block = nullptr;
  int peer_nflag = 0;
  long long peer_cap = 0;
  double* peer_slots[mcba::kMaxRanks] = {};
  unsigned long long* peer_flags[mcba::kMaxRanks] = {};
  void* peer_mapped[mcba::kMaxRanks] = {};   // IPC mappings to close
  unsigned long long peer_epoch = 0;
  bool peer_ready = false;
  long long launches = 0;  // kernels launched by this handle (bench gpu_launches)
  // optional per-kernel timing (CUDA events on the launching stream; bench.py roofline)
  bool profile = false;
  cudaEvent_t* prof_ev = nullptr;   // ring of kProfEvents events per evaluation
  int prof_n = 0;
};

namespace mcba {

void set_error(const std::string& msg);
#define MCBA_CUDA(expr)                                                                   \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      mcba::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));               \
      return MCBA_ERR_CUDA;                                                               \
    }                                                                                     \
  } while (0)

// Scope guards for the error paths: a stream-ordered work block and CUDA events are released on
// every return.
struct AsyncBlock {
  unsigned char* p = nullptr;
  cudaStream_t st = nullptr;
  explicit AsyncBlock(cudaStream_t s) : st(s) {}
  AsyncBlock(const AsyncBlock&) = delete;
  AsyncBlock& operator=(const AsyncBlock&) = delete;
  ~AsyncBlock() { if (p) cudaFreeAsync(p, st); }
};
struct EventPair {
  cudaEvent_t a = nullptr, b = nullptr;
  EventPair() = default;
  EventPair(const EventPair&) = delete;
  EventPair& operator=(const EventPair&) = delete;
  ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
};

int keep_async_pool(int device);   // k0_frontend.cu
void host_rodrigues(const double r[3], double R[9]);   // k5_points.cu
int peer_allreduce(mcba_handle* h, double* buf, long long n);   // mcba_peer.cu

// kernel launchers (defined in the .cu files)
int launch_prep_cameras(mcba_handle* h, const double* x);
int launch_tile_observations(mcba_handle* h);
int ensure_row_offsets(mcba_handle* h);
int launch_residuals(mcba_handle* h, const double* x, double* r_out);
int launch_predict(mcba_handle* h, const double* x, double* uv_out);
int launch_cost(mcba_handle* h, const double* x, int loss, double f_scale, double* out_scal);
int launch_k2_producer(mcba_handle* h, const double* x, int loss, double f_scale);
int launch_k2_consumer(mcba_handle* h, const double* x, double lambda);
int launch_k2_gradient(mcba_handle* h, const double* x);   // pose gradient only (closing evaluation)
int k2_producer_grid(const mcba::Layout& L, int n_sm, int* warps);
int k2_consumer_parts(const mcba::Layout& L, int n_sm, int* mode);
int k2c_stream_warps(int C);
// SYRK CTA width (warps), CTA rows (gy) and the block count of the compiled tile list (0: run-time list)
void syrk_plan(int nc, int* warps, int* gy, int* static_nb);
// solve of the reduced system: tiles per warp of the one-CTA kernel, or the library
enum SolveTier : int { kSolveTierLibrary = 0, kSolveTierRegs3 = 3, kSolveTierRegs8 = 8, kSolveTierSmem19 = 119 };
int solve_tier(int nc);
// dynamic shared memory of the observation transpose (k1_residual.cu): [32 frames][N + 1] corners
inline size_t tile_observations_smem(int N) { return sizeof(double2) * kTile * ((size_t)N + 1); }
int launch_k2_syrk(mcba_handle* h);
int syrk_grid(int nc, long long F, int n_sm);
int launch_finalize(mcba_handle* h, bool exchange);   // exchange: sum over ranks inside the kernel (peer memory)
int launch_jacobian_blocks(mcba_handle* h, const double* x, double* Jc, double* Jp);
int launch_backsub(mcba_handle* h, const double* x, double* x_new, double lambda);
int allreduce_packed(mcba_handle* h, double* buf, long long n);
int ensure_solver(mcba_handle* h);   // k3_solve.cu

// calibration covariance (k8_covariance.cu, driven by mcba_covariance)
constexpr double kCovPivotTol = 1e-12;   // relative Cholesky pivot s_j / A_jj at or below which a block is singular
// per frame, from the factor K2c left at lambda = 0 (D2pose holding diag V_f): out[0] frames without observations,
// out[1] observed frames with a relative pivot <= kCovPivotTol (u64), out[2] min relative pivot of the observed frames
int launch_cov_frame_check(mcba_handle* h, unsigned long long* d_out);
// gauge-fixed inverse of the reduced camera system in d_red: d_cov (12C x 12C, true basis, unscaled by s^2; 0 on the
// rows / columns of held parameters (held[r], may be null; wins over NaN) and of the reference camera's extrinsics
// (none for reference_camera = -1), NaN on unobserved cameras) and d_sraw = T d_cov T^T (raw basis, 0 for unobserved
// cameras); *min_pivot = smallest relative pivot of the Jacobi-scaled Cholesky (+inf when nothing is left to
// invert), *info = potrf's
int covariance_cameras(mcba_handle* h, int reference_camera, const int* observed, const uint8_t* held, double* d_cov,
                       double* d_sraw, double* min_pivot, int* info);
// per frame: s2 L^-T (I + Z^T Sigma_raw Z) L^-1 into d_pose_cov (F,6,6), caller's frame order; NaN for empty frames
int launch_cov_poses(mcba_handle* h, const double* d_sraw, double s2, double* d_pose_cov);

}  // namespace mcba
