// C-ABI entry points of libmcba (see include/mcba.h), the handle life cycle and
// the Levenberg-Marquardt driver that replaces scipy.optimize.least_squares for
// bundle_adjustment.py:307-313.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "mcba_internal.h"
#include "mcba_peer.cuh"

namespace mcba {

cudaError_t set_dynamic_smem(const void* kernel, size_t bytes) {
  static std::mutex mu;
  static std::unordered_map<unsigned long long, size_t> granted;   // (kernel, device) -> bytes
  int device = 0;
  cudaError_t e = cudaGetDevice(&device);
  if (e != cudaSuccess) return e;
  const unsigned long long key = (unsigned long long)reinterpret_cast<uintptr_t>(kernel) * 64ull + (unsigned)device;
  std::lock_guard<std::mutex> lock(mu);
  auto it = granted.find(key);
  if (it != granted.end() && it->second >= bytes) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) granted[key] = bytes;
  return e;
}

static thread_local std::string g_error;
void set_error(const std::string& msg) { g_error = msg; }
int solve_reduced(mcba_handle* h, double lambda);
static void destroy_pipe(mcba_handle* h);   // chunked host path of mcba_build_reduced_host (below)
static bool pipe_parent_is_stale(mcba_handle* h);
static int refresh_parent_from_pipe(mcba_handle* h);
static void pipe_forget(mcba_handle* h);

// ------------------------------------------------------------------ NCCL (resolved lazily: torch already maps libnccl.so.2)
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int load_nccl() {
  if (g_nccl.lib) return MCBA_OK;
  void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) {
    set_error(std::string("cannot load libnccl: ") + dlerror());
    return MCBA_ERR_NCCL;
  }
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(lib, "ncclCommInitRank");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(lib, "ncclAllReduce");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(lib, "ncclCommDestroy");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(lib, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy) {
    set_error("libnccl is missing required symbols");
    return MCBA_ERR_NCCL;
  }
  g_nccl.lib = lib;
  return MCBA_OK;
}

int allreduce_packed(mcba_handle* h, double* buf, long long n) {
  if (h->nranks <= 1) return MCBA_OK;
  if (h->peer_ready) return peer_allreduce(h, buf, n);   // one kernel over NVLink peer memory
  if (!h->nccl_comm) return MCBA_OK;
  ncclResult_t r = g_nccl.AllReduce(buf, buf, (size_t)n, ncclDouble, ncclSum, (ncclComm_t)h->nccl_comm, h->stream);
  if (r != ncclSuccess) {
    set_error(std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error"));
    return MCBA_ERR_NCCL;
  }
  h->launches++;
  return MCBA_OK;
}

// partial sums -> packed reduced system in d_red, summed over the ranks: inside the finalize kernel
// when the peer buffers are mapped, by ncclAllReduce behind it otherwise
static int finalize_and_sum(mcba_handle* h) {
  const bool peer = h->nranks > 1 && h->peer_ready;
  int rc = launch_finalize(h, peer);
  if (rc || peer) return rc;
  return allreduce_packed(h, h->d_red, h->L.redLen);
}

// ------------------------------------------------------------------ evaluation helpers
struct EvalOut {
  double cost, sumsq, count, gnorm;
};

// residual + Jacobian + Schur at x; the packed system is left (all-reduced) in d_red
// (redamp: x and the loss are those of the previous call, only lambda changed -> K2p is skipped)
static int evaluate(mcba_handle* h, const double* x, double lambda, int loss, double f_scale, bool redamp = false) {
  int rc;
  const bool prof = h->profile && !redamp && h->prof_n < kProfRing;
  cudaEvent_t* ev = prof ? h->prof_ev + kProfEvents * h->prof_n : nullptr;
  if (prof) cudaEventRecord(ev[0], h->stream);
  if (!redamp) {   // K2p also builds and publishes the camera constants of x (d_cams)
    if ((rc = launch_k2_producer(h, x, loss, f_scale))) return rc;
  }
  if (prof) cudaEventRecord(ev[1], h->stream);
  if ((rc = launch_k2_consumer(h, x, lambda))) return rc;
  if (prof) cudaEventRecord(ev[4], h->stream);
  if ((rc = launch_k2_syrk(h))) return rc;
  if (prof) cudaEventRecord(ev[2], h->stream);
  if ((rc = finalize_and_sum(h))) return rc;
  if (prof) { cudaEventRecord(ev[3], h->stream); h->prof_n++; }
  return MCBA_OK;
}

// K2c + SYRK + finalize (+ all-reduce) on the K2p outputs the handle currently points at.
// need_system = false: the evaluation that closes a solve only has to deliver the gradient and the
// scalars at the final point -- K2c and the SYRK are skipped.
static int evaluate_tail(mcba_handle* h, const double* x, double lambda, bool need_system = true) {
  int rc;
  if (!need_system) {
    // gradient and cost only: the pose gradients come from a kernel that reads just the q_ext rows of the hand-off
    // (no Z, no factor: b and S in d_red are left stale, nothing reads them before the next evaluation rebuilds them)
    if ((rc = launch_k2_gradient(h, x))) return rc;
    return finalize_and_sum(h);
  }
  if ((rc = launch_k2_consumer(h, x, lambda))) return rc;
  if ((rc = launch_k2_syrk(h))) return rc;
  return finalize_and_sum(h);
}

// out[0..2] = fixed-order sum over K2p's per-CTA partials {0.5 sum rho, sum f^2, count}; with peers the
// 12 step scalars out[0..11] (3 from here, 4 from the back-substitution) are then summed over the
// ranks in the same launch (mcba_peer.cuh)
// Where the scalars go besides d_scal: a MAPPED pinned host block that the LM loop polls (no D2H copy
// operations and no driver wait between the trial walk and the host's accept / reject decision).
struct HostSignal {
  double* vals;                  // [16]: the 12 step scalars, [12] = pivot info of the solve
  unsigned long long* flag;      // written last, after a system-scope fence
  unsigned long long seq;
  const int* info;               // d_info of the solve kernel
};

__global__ void sum_scalars_kernel(const double* __restrict__ partS, int n, double* __restrict__ out, int exchange,
                                   const PeerView pv, const HostSignal sig) {
  __shared__ double s[3][32];
  const int lane = threadIdx.x;
  double a = 0, b = 0, k = 0;
  for (int i = lane; i < n; i += 32) {
    a += partS[(size_t)i * kRsNum + kRsCost];
    b += partS[(size_t)i * kRsNum + kRsSumSq];
    k += partS[(size_t)i * kRsNum + kRsCount];
  }
  s[0][lane] = a; s[1][lane] = b; s[2][lane] = k;
  __syncwarp();
  double v = 0.0;
  if (lane < 3) {
    for (int i = 0; i < 32; ++i) v += s[lane][i];
    out[lane] = v;
  } else if (lane < 12) {
    v = out[lane];
  }
  if (exchange) {
    if (lane < 12)
      for (int r = 0; r < pv.nranks; ++r) peer_slot_of(pv, (pv.rank + r) % pv.nranks)[lane] = v;
    peer_publish(pv, 0);
    peer_wait(pv, 0);
    if (lane < 12) {
      double acc = 0.0;
      for (int r = 0; r < pv.nranks; ++r) acc += __ldcg(peer_slot_from(pv, r) + lane);
      out[lane] = acc;
      v = acc;
    }
  }
  if (sig.flag) {   // results straight into host memory, then the sequence number
    if (lane < 12) sig.vals[lane] = v;
    if (lane == 12) sig.vals[12] = (double)sig.info[0];
    __threadfence_system();
    __syncwarp();
    if (lane == 0) asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(sig.flag), "l"(sig.seq) : "memory");
  }
}

// trial-point scalars of the LM loop: sum of K2p's partials (+ the sum over ranks)
static int launch_sum_scalars(mcba_handle* h, bool signal_host) {
  const bool peer = h->nranks > 1 && h->peer_ready;
  const bool direct = signal_host && (peer || h->nranks == 1);   // NCCL sums behind the kernel: no direct signal
  PeerView pv;
  if (peer) pv = peer_next_call(h); else std::memset(&pv, 0, sizeof(pv));
  HostSignal sig{nullptr, nullptr, 0, h->d_info};
  if (direct) {
    sig.vals = h->d_signal_vals;
    sig.flag = h->d_signal_flag;
    sig.seq = ++h->signal_seq;
  }
  sum_scalars_kernel<<<1, 32, 0, h->stream>>>(h->d_partS, h->grid_frames, h->d_scal, peer ? 1 : 0, pv, sig);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  if (peer || h->nranks == 1) return MCBA_OK;
  return allreduce_packed(h, h->d_scal, 12);
}

// Spin until the scalar kernel of the current trial has written its sequence number into the mapped
// host block (a few microseconds after the kernel ends, against tens for two D2H copies and a stream
// synchronisation).  A failed launch / trapped kernel shows up in cudaStreamQuery.
static int wait_host_signal(mcba_handle* h) {
  volatile unsigned long long* flag = h->h_signal_flag;
  unsigned spins = 0;
  while (*flag != h->signal_seq) {
    if ((++spins & 0x3fff) == 0) {
      const cudaError_t q = cudaStreamQuery(h->stream);
      if (q == cudaSuccess) { if (*flag == h->signal_seq) break; }
      else if (q != cudaErrorNotReady) { set_error(std::string("LM loop: ") + cudaGetErrorString(q)); return MCBA_ERR_CUDA; }
    }
#if defined(__x86_64__)
    __builtin_ia32_pause();
#endif
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  return MCBA_OK;
}

static void swap_k2p_outputs(mcba_handle* h) {
  std::swap(h->d_H, h->d_H_alt);
  std::swap(h->d_partU, h->d_partU_alt);
  std::swap(h->d_partS, h->d_partS_alt);
  std::swap(h->d_cams, h->d_cams_alt);
}

static int ensure_alt_outputs(mcba_handle* h) {
  const Layout& L = h->L;
  const size_t h_bytes = sizeof(double) * (size_t)L.nTiles * L.C * 63 * kTile;
  if (!h->d_H_alt) {
    MCBA_CUDA(cudaMalloc((void**)&h->d_H_alt, h_bytes));
    MCBA_CUDA(cudaMalloc((void**)&h->d_partU_alt, sizeof(double) * (size_t)h->grid_frames * L.C * kAcc));
    MCBA_CUDA(cudaMalloc((void**)&h->d_partS_alt, sizeof(double) * (size_t)h->grid_frames * kRsNum));
    MCBA_CUDA(cudaMalloc((void**)&h->d_cams_alt, sizeof(CamConst) * L.C));
    h->alt_stale = true;
  }
  if (h->alt_stale) {
    MCBA_CUDA(cudaMemsetAsync(h->d_H_alt, 0, h_bytes, h->stream));
    h->alt_stale = false;
  }
  return MCBA_OK;
}

// The scalars of the last evaluation ([b | g | diag | scalars | rank slots] of d_red) travel to the
// pinned mirror asynchronously; parse_eval reads them after the caller's next synchronisation.
static int enqueue_eval_readback(mcba_handle* h) {
  const Layout& L = h->L;
  const long long tail = L.redLen - L.offB;
  MCBA_CUDA(cudaMemcpyAsync(h->h_pinned, h->d_red + L.offB, sizeof(double) * tail, cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaEventRecord(h->readback_done, h->stream));   // parse_eval's caller waits on this (already complete by then)
  return MCBA_OK;
}

static void parse_eval(mcba_handle* h, EvalOut* out) {
  const Layout& L = h->L;
  const double* t = h->h_pinned;
  const double* g = t + (L.offG - L.offB);
  const double* sc = t + (L.offScal - L.offB);
  const double* rk = t + (L.offRank - L.offB);
  double gn = 0.0;
  for (int i = 0; i < L.nc; ++i)   // gtol / optimality of the free sub-problem: held entries do not count
    if (!h->any_fixed || !h->h_fixed[i]) gn = std::max(gn, std::fabs(g[i]));
  bool bad = false;
  for (int i = 0; i < L.nc; ++i) bad |= !std::isfinite(g[i]);
  for (int i = 0; i < kMaxRanks; ++i) gn = std::max(gn, rk[i]);
  out->cost = sc[kRsCost];
  out->sumsq = sc[kRsSumSq];
  out->count = sc[kRsCount];
  out->gnorm = bad ? NAN : gn;
}

static int read_eval(mcba_handle* h, EvalOut* out) {
  int rc = enqueue_eval_readback(h);
  if (rc) return rc;
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  parse_eval(h, out);
  return MCBA_OK;
}

}  // namespace mcba

using namespace mcba;

extern "C" {

const char* mcba_last_error(void) { return g_error.c_str(); }
int mcba_version(void) { return 100; }

void mcba_default_options(mcba_options* o) {
  std::memset(o, 0, sizeof(*o));
  o->ftol = 1e-4;  // bundle_adjustment.py:302
  o->xtol = 1e-8;
  o->gtol = 1e-8;
  o->max_nfev = 0;
  o->loss = MCBA_LOSS_SOFT_L1;
  o->f_scale = 1.0;
  o->verbose = 2;
  o->hessian = MCBA_HESSIAN_AUTO;
  o->lambda0 = 1e-3;
  o->lambda_min = 1e-12;
  o->lambda_max = 1e12;
}

// allocations and library handles of a new problem; on failure the caller destroys the partly built handle
static int create_impl(mcba_handle* h, int C, int64_t F, int N, int device) {
  MCBA_CUDA(cudaSetDevice(device));
  h->device = device;
  Layout& L = h->L;
  L.C = C; L.N = N; L.F = F;
  L.nTiles = (F + kTile - 1) / kTile;
  L.Fpad = L.nTiles * kTile;
  L.nc = 12 * C;
  L.nc8 = (L.nc + 7) / 8 * 8;
  L.offS = 0;
  L.offB = (long long)L.nc * L.nc;
  L.offG = L.offB + L.nc;
  L.offDiag = L.offG + L.nc;
  L.offScal = L.offDiag + L.nc;
  L.offRank = L.offScal + kRsNum;
  L.redLen = L.offRank + kMaxRanks;
  cudaDeviceProp prop;
  MCBA_CUDA(cudaGetDeviceProperties(&prop, device));
  if (tile_observations_smem(N) > prop.sharedMemPerBlockOptin) {
    set_error("mcba_create: a board of " + std::to_string(N) + " points needs " + std::to_string(tile_observations_smem(N)) +
              " bytes of shared memory to tile its observations; this device allows " +
              std::to_string(prop.sharedMemPerBlockOptin) + " per block (at most " +
              std::to_string(prop.sharedMemPerBlockOptin / (sizeof(double2) * kTile) - 1) + " points)");
    return MCBA_ERR_ARG;
  }
  h->n_sm = prop.multiProcessorCount;
  MCBA_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  h->grid_frames = k2_producer_grid(L, h->n_sm, &h->prod_warps);
  h->n_part_c = k2_consumer_parts(L, h->n_sm, &h->k2c_mode);
  h->grid_syrk = syrk_grid(L.nc, F, h->n_sm);
  h->grid_cost = (int)std::min<long long>((L.nTiles * C + 7) / 8, 8LL * h->n_sm);
  h->grid_back = (int)std::min<long long>((L.nTiles + 3) / 4, (long long)h->n_sm);   // backsub: persistent CTAs of 4 warps, whole tiles per warp
  const long long n = L.nc + 6 * F;
  auto alloc = [&](void** p, size_t bytes) { return cudaMalloc(p, bytes ? bytes : 8); };
#define MCBA_ALLOC(ptr, count) MCBA_CUDA(alloc((void**)&(ptr), sizeof(*(ptr)) * (size_t)(count)))
  MCBA_ALLOC(h->d_obs_ref, (size_t)C * F * N * 2);
  MCBA_ALLOC(h->d_obs_tiled, (size_t)L.nTiles * C * N * kTile);
  MCBA_ALLOC(h->d_obj, 3 * N);
  MCBA_ALLOC(h->d_perm, 2 * L.Fpad);
  MCBA_ALLOC(h->d_mask, 2 * L.Fpad);
  MCBA_ALLOC(h->d_active, L.nTiles);
  MCBA_ALLOC(h->d_units, (size_t)C * L.nTiles);
  MCBA_ALLOC(h->d_unit_count, 128);
  MCBA_ALLOC(h->d_row_off, (size_t)C * ((F + 31) / 32) + 1);
  MCBA_ALLOC(h->d_x, n);
  MCBA_ALLOC(h->d_xtrial, n);
  MCBA_ALLOC(h->d_cams, C);
  MCBA_ALLOC(h->d_Z, (size_t)L.Fpad * 6 * L.nc);
  MCBA_ALLOC(h->d_Linv, (size_t)L.nTiles * 21 * kTile);
  MCBA_ALLOC(h->d_y, (size_t)L.nTiles * 6 * kTile);
  MCBA_ALLOC(h->d_JlTau, (size_t)L.nTiles * 12 * kTile);
  MCBA_ALLOC(h->d_gpose, (size_t)L.Fpad * 6);
  MCBA_ALLOC(h->d_D2pose, (size_t)L.nTiles * 6 * kTile);
  MCBA_ALLOC(h->d_D2cam, L.nc);
  MCBA_ALLOC(h->d_H, (size_t)L.nTiles * C * 63 * kTile);
  MCBA_ALLOC(h->d_partG, L.nTiles);
  MCBA_ALLOC(h->d_partU, (size_t)h->grid_frames * C * kAcc);
  MCBA_ALLOC(h->d_partS, (size_t)h->grid_frames * kRsNum);
  MCBA_ALLOC(h->d_partSyrk, (size_t)h->grid_syrk * L.nc8 * L.nc8);
  MCBA_ALLOC(h->d_partZy, (size_t)L.nTiles * L.nc);
  MCBA_ALLOC(h->d_Sraw, (size_t)L.nc8 * L.nc8 + L.nc + (size_t)C * kAcc);
  MCBA_ALLOC(h->d_red, L.redLen);
  MCBA_ALLOC(h->d_fin_scratch, (size_t)(C * (C + 1) / 2) * 4 * (144 + kAcc + 12));
  MCBA_ALLOC(h->d_fin_counter, C * (C + 1) / 2 + 1);
  MCBA_CUDA(cudaMemset(h->d_fin_counter, 0, sizeof(unsigned int) * (C * (C + 1) / 2 + 1)));
  MCBA_ALLOC(h->d_Sd, (size_t)L.nc * L.nc);
  MCBA_ALLOC(h->d_dcam, 2 * L.nc);
  MCBA_ALLOC(h->d_scal, 64 + 7 * 4096);
  MCBA_ALLOC(h->d_info, 4);
  MCBA_CUDA(cudaMemset(h->d_D2pose, 0, sizeof(double) * L.nTiles * 6 * kTile));
  MCBA_CUDA(cudaMemset(h->d_D2cam, 0, sizeof(double) * L.nc));
  MCBA_CUDA(cudaMemset(h->d_scal, 0, sizeof(double) * (64 + 7 * 4096)));
  MCBA_CUDA(cudaMemset(h->d_info, 0, sizeof(int) * 4));
  MCBA_CUDA(cudaMemset(h->d_gpose, 0, sizeof(double) * L.Fpad * 6));
  MCBA_CUDA(cudaMemset(h->d_partSyrk, 0, sizeof(double) * (size_t)h->grid_syrk * L.nc8 * L.nc8));   // lower block triangle is never written
  MCBA_CUDA(cudaMallocHost((void**)&h->h_pinned, sizeof(double) * (L.redLen + 64)));
  MCBA_CUDA(cudaHostAlloc((void**)&h->h_signal_vals, sizeof(double) * 32, cudaHostAllocMapped));
  std::memset(h->h_signal_vals, 0, sizeof(double) * 32);
  h->h_signal_flag = reinterpret_cast<unsigned long long*>(h->h_signal_vals + 16);
  MCBA_CUDA(cudaHostGetDevicePointer((void**)&h->d_signal_vals, h->h_signal_vals, 0));
  h->d_signal_flag = reinterpret_cast<unsigned long long*>(h->d_signal_vals + 16);
  MCBA_CUDA(cudaEventCreateWithFlags(&h->readback_done, cudaEventDisableTiming));
  // the reduced system is solved by this library's own kernel (k3_solve.cu); a cuSOLVER handle is
  // only created if a system wider than 192 (more than 16 cameras) is ever solved
  return MCBA_OK;
}

int mcba_create(mcba_handle** out, int C, int64_t F, int N, int device) {
  if (!out || C < 1 || F < 1 || N < 1) {
    set_error("mcba_create: n_cameras, n_frames, n_points must be >= 1");
    return MCBA_ERR_ARG;
  }
  if (C > 32) {
    set_error("mcba_create: at most 32 cameras are supported");
    return MCBA_ERR_ARG;
  }
  *out = nullptr;
  mcba_handle* h = new mcba_handle();
  const int rc = create_impl(h, C, F, N, device);
  if (rc) {   // release whatever was allocated before the failure, keep its message
    const std::string why = g_error;
    mcba_destroy(h);
    set_error(why);
    return rc;
  }
  *out = h;
  return MCBA_OK;
}

int mcba_destroy(mcba_handle* h) {
  if (!h) return MCBA_OK;
  cudaSetDevice(h->device);
  destroy_pipe(h);
  if (h->nccl_comm && g_nccl.CommDestroy) g_nccl.CommDestroy((ncclComm_t)h->nccl_comm);
  if (h->solver) cusolverDnDestroy(h->solver);
  for (int s = 0; s < kMaxRanks; ++s) if (h->peer_mapped[s]) cudaIpcCloseMemHandle(h->peer_mapped[s]);
  if (h->peer_block) cudaFree(h->peer_block);
  void* ptrs[] = {h->d_obs_ref, h->d_obs_tiled, h->d_obj, h->d_row_off, h->d_x, h->d_xtrial, h->d_cams, h->d_Z,
                  h->d_Linv, h->d_y, h->d_JlTau, h->d_gpose, h->d_D2pose, h->d_D2cam, h->d_partU, h->d_partS, h->d_partSyrk,
                  h->d_red, h->d_Sd, h->d_dcam, h->d_scal, h->d_info, h->d_work, h->d_Sraw, h->d_H, h->d_H_alt, h->d_partU_alt, h->d_partS_alt, h->d_cams_alt, h->d_partG, h->d_partZy, h->d_perm, h->d_mask, h->d_active, h->d_sort_tmp, h->d_units, h->d_unit_count, h->d_chunk_rows, h->d_fin_scratch, h->d_fin_counter, h->d_fixed};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (h->prof_ev) {
    for (int i = 0; i < kProfEvents * kProfRing; ++i) cudaEventDestroy(h->prof_ev[i]);
    delete[] h->prof_ev;
  }
  if (h->h_pinned) cudaFreeHost(h->h_pinned);
  if (h->h_signal_vals) cudaFreeHost(h->h_signal_vals);
  if (h->readback_done) cudaEventDestroy(h->readback_done);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return MCBA_OK;
}

int mcba_set_stream(mcba_handle* h, void* s) {
  if (!h) return MCBA_ERR_ARG;
  MCBA_CUDA(cudaSetDevice(h->device));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  if (s) {
    if (h->own_stream) cudaStreamDestroy(h->stream);
    h->stream = (cudaStream_t)s;
    h->own_stream = false;
  } else if (!h->own_stream) {
    MCBA_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->own_stream = true;
  }
  if (h->solver) cusolverDnSetStream(h->solver, h->stream);
  return MCBA_OK;
}

int mcba_synchronize(mcba_handle* h) {
  MCBA_CUDA(cudaSetDevice(h->device));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  return MCBA_OK;
}

int mcba_set_observations(mcba_handle* h, const double* uvs, const double* obj, int is_device) {
  if (!h || !uvs || !obj) { set_error("mcba_set_observations: null argument"); return MCBA_ERR_ARG; }
  MCBA_CUDA(cudaSetDevice(h->device));
  pipe_forget(h);   // new observations supersede what a pipelined host call left in its children
  const Layout& L = h->L;
  const size_t uv_bytes = sizeof(double) * (size_t)L.C * L.F * L.N * 2;
  if (is_device) {
    if (uvs != h->d_obs_ref) MCBA_CUDA(cudaMemcpyAsync(h->d_obs_ref, uvs, uv_bytes, cudaMemcpyDeviceToDevice, h->stream));
    if (obj != h->d_obj) MCBA_CUDA(cudaMemcpyAsync(h->d_obj, obj, sizeof(double) * 3 * L.N, cudaMemcpyDeviceToDevice, h->stream));
  } else {
    // caller-owned host memory: pinned buffers take one async copy, pageable ones (a numpy array) are
    // staged through the multi-threaded bounce buffers of mcba_upload instead of the driver's single one
    int rc = mcba_upload(h->device, h->stream, h->d_obs_ref, uvs, uv_bytes);
    if (rc) return rc;
    MCBA_CUDA(cudaMemcpyAsync(h->d_obj, obj, sizeof(double) * 3 * L.N, cudaMemcpyHostToDevice, h->stream));
  }
  int rc = launch_tile_observations(h);
  if (rc) return rc;
  h->have_obs = true;
  h->have_rows = false;
  // a new problem: reset the running Marquardt scaling
  MCBA_CUDA(cudaMemsetAsync(h->d_D2pose, 0, sizeof(double) * L.nTiles * 6 * kTile, h->stream));
  MCBA_CUDA(cudaMemsetAsync(h->d_D2cam, 0, sizeof(double) * L.nc, h->stream));
  return MCBA_OK;
}

static int need_obs(mcba_handle* h) {
  if (!h || !h->have_obs) { set_error("observations not set (call mcba_set_observations first)"); return MCBA_ERR_STATE; }
  MCBA_CUDA(cudaSetDevice(h->device));
  return pipe_parent_is_stale(h) ? refresh_parent_from_pipe(h) : MCBA_OK;
}

int mcba_num_residuals(mcba_handle* h, int64_t* m, int64_t* nobs) {
  int rc = need_obs(h);
  if (rc) return rc;
  if ((rc = ensure_row_offsets(h))) return rc;
  if (m) *m = h->m;
  if (nobs) *nobs = h->n_obs;
  return MCBA_OK;
}

int mcba_residuals(mcba_handle* h, const double* d_x, double* d_r) {
  int rc = need_obs(h);
  if (rc) return rc;
  if ((rc = ensure_row_offsets(h))) return rc;
  return launch_residuals(h, d_x, d_r);
}

int mcba_predict(mcba_handle* h, const double* d_x, double* d_uv) {
  if (!h) return MCBA_ERR_ARG;
  MCBA_CUDA(cudaSetDevice(h->device));
  return launch_predict(h, d_x, d_uv);
}

int mcba_jacobian_blocks(mcba_handle* h, const double* d_x, double* d_Jc, double* d_Jp) {
  if (!h) return MCBA_ERR_ARG;
  MCBA_CUDA(cudaSetDevice(h->device));
  return launch_jacobian_blocks(h, d_x, d_Jc, d_Jp);
}

int mcba_cost(mcba_handle* h, const double* d_x, int loss, double f_scale, double* cost, double* sumsq, int64_t* count) {
  int rc = need_obs(h);
  if (rc) return rc;
  if ((rc = launch_cost(h, d_x, loss, f_scale, h->d_scal))) return rc;
  if ((rc = allreduce_packed(h, h->d_scal, 3))) return rc;
  MCBA_CUDA(cudaMemcpyAsync(h->h_pinned, h->d_scal, sizeof(double) * 3, cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  if (cost) *cost = h->h_pinned[0];
  if (sumsq) *sumsq = h->h_pinned[1];
  if (count) *count = (int64_t)h->h_pinned[2];
  return MCBA_OK;
}

int mcba_build_reduced(mcba_handle* h, const double* d_x, double lambda, int loss, double f_scale, double* h_S,
                       double* h_b, double* h_gcam, double* h_cost) {
  int rc = need_obs(h);
  if (rc) return rc;
  if ((rc = evaluate(h, d_x, lambda, loss, f_scale))) return rc;
  const Layout& L = h->L;
  if (h_S) MCBA_CUDA(cudaMemcpyAsync(h_S, h->d_red + L.offS, sizeof(double) * L.nc * L.nc, cudaMemcpyDeviceToHost, h->stream));
  if (h_b) MCBA_CUDA(cudaMemcpyAsync(h_b, h->d_red + L.offB, sizeof(double) * L.nc, cudaMemcpyDeviceToHost, h->stream));
  if (h_gcam) MCBA_CUDA(cudaMemcpyAsync(h_gcam, h->d_red + L.offG, sizeof(double) * L.nc, cudaMemcpyDeviceToHost, h->stream));
  if (h_cost) MCBA_CUDA(cudaMemcpyAsync(h_cost, h->d_red + L.offScal + kRsCost, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (h_S || h_b || h_gcam || h_cost) MCBA_CUDA(cudaStreamSynchronize(h->stream));   // no outputs: stay asynchronous
  return MCBA_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// mcba_build_reduced_host, pipelined.  The call is bound by PCIe (168 MB of observations at BASELINE
// configs[2] against a 0.36 ms pass), and its dependent tail -- frame masks, sort, tiling, the pass
// itself -- only starts when the last byte has landed.  With page-locked host buffers and enough
// frames the observations instead cross in kHostChunks frame ranges on a copy stream; every range is a
// complete small problem of its own (a child handle: tiled, evaluated and reduced while the next range
// is in flight), and S, b, the camera gradient and the scalars of the ranges, all sums over frames,
// are added at the end (the additivity tests/test_gpu_parity.py checks for shards).  The parent's own
// tiled copy and evaluation are rebuilt from the children when a later call needs them (need_obs), so
// the handle behaves as after mcba_set_observations + mcba_build_reduced.  A range's work is replayed
// from one CUDA graph once the caller's lambda / loss / f_scale have been stable for two calls.
// MCBA_NO_HOST_PIPELINE=1 forces the plain path, MCBA_NO_PIPE_GRAPHS=1 the kernel-by-kernel issue.
namespace mcba {
constexpr int kHostChunks = 8;
constexpr long long kHostPipeMinFrames = 16384;

struct HostPipe {
  std::vector<mcba_handle*> kids;
  std::vector<long long> f0;
  std::vector<cudaEvent_t> landed, done;   // per range: copy finished / evaluation finished (timed: MCBA_PIPE_TRACE)
  cudaEvent_t t0 = nullptr, params = nullptr;
  double* d_x = nullptr;              // staging: [x (12C + 6F) | objpoints (3N)]
  cudaStream_t copy = nullptr;
  cudaEvent_t begin = nullptr;
  const double** d_table = nullptr;   // the children's packed systems (device pointers, fixed)
  // One CUDA graph per range: its ~25 operations (three slice copies, masks, sort, tiling, unit lists, memsets, the
  // four kernels of the evaluation) are captured on the second call with the same lambda / loss / f_scale and replayed with ONE launch afterwards -- the
  // host otherwise spends ~180 driver calls per call of the pipeline, which on a slow or busy host delays the
  // ranges' work behind their transfers (3.4 -> 3.8-3.9 ms observed).  Re-captured when lambda / loss / f_scale change.
  std::vector<cudaGraphExec_t> graphs;
  std::vector<char> warmed;           // the range ran once un-captured (first-use allocations are done)
  double g_lambda = 0.0, g_f_scale = 0.0;
  int g_loss = -1;
  int same_params_calls = 0;          // consecutive calls with these values: a caller that varies lambda never captures
  bool graphs_off = false;            // the stream could not be captured
  bool parent_stale = false;          // the last call's observations are in the children only
  double lambda = 0.0, f_scale = 1.0; // ... and so is its evaluation (re-run on the parent when it is needed)
  int loss = 0;
};

static void destroy_pipe(mcba_handle* h) {
  HostPipe* P = h->pipe;
  if (!P) return;
  for (mcba_handle* k : P->kids) mcba_destroy(k);
  for (cudaGraphExec_t g : P->graphs) if (g) cudaGraphExecDestroy(g);
  for (cudaEvent_t e : P->landed) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : P->done) if (e) cudaEventDestroy(e);
  if (P->t0) cudaEventDestroy(P->t0);
  if (P->params) cudaEventDestroy(P->params);
  if (P->d_x) cudaFree(P->d_x);
  if (P->begin) cudaEventDestroy(P->begin);
  if (P->copy) cudaStreamDestroy(P->copy);
  if (P->d_table) cudaFree(P->d_table);
  delete P;
  h->pipe = nullptr;
}

static bool pipe_parent_is_stale(mcba_handle* h) { return h->pipe && h->pipe->parent_stale; }
static void pipe_forget(mcba_handle* h) { if (h->pipe) h->pipe->parent_stale = false; }

static bool host_pointer_is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

static int ensure_pipe(mcba_handle* h) {
  if (h->pipe) {
    for (mcba_handle* k : h->pipe->kids) k->stream = h->stream;   // the parent's stream may have been replaced
    return MCBA_OK;
  }
  const Layout& L = h->L;
  HostPipe* P = new HostPipe();
  h->pipe = P;
  const long long tiles_per_chunk = (L.nTiles + kHostChunks - 1) / kHostChunks;
  for (int k = 0; k < kHostChunks; ++k) {
    const long long f0 = (long long)k * tiles_per_chunk * kTile;
    if (f0 >= L.F) break;
    const long long fk = std::min<long long>(L.F - f0, tiles_per_chunk * kTile);
    mcba_handle* kid = nullptr;
    int rc = mcba_create(&kid, L.C, fk, L.N, h->device);
    if (rc) return rc;
    if (kid->own_stream && kid->stream) cudaStreamDestroy(kid->stream);
    kid->stream = h->stream;
    kid->own_stream = false;
    P->kids.push_back(kid);
    P->f0.push_back(f0);
    cudaEvent_t e = nullptr;
    MCBA_CUDA(cudaEventCreate(&e));
    P->landed.push_back(e);
    MCBA_CUDA(cudaEventCreate(&e));
    P->done.push_back(e);
    P->graphs.push_back(nullptr);
    P->warmed.push_back(0);
  }
  MCBA_CUDA(cudaStreamCreateWithFlags(&P->copy, cudaStreamNonBlocking));
  MCBA_CUDA(cudaEventCreateWithFlags(&P->begin, cudaEventDisableTiming));
  MCBA_CUDA(cudaEventCreate(&P->t0));
  MCBA_CUDA(cudaEventCreateWithFlags(&P->params, cudaEventDisableTiming));
  MCBA_CUDA(cudaMalloc((void**)&P->d_x, sizeof(double) * (L.nc + 6 * L.F + 3 * L.N)));
  std::vector<const double*> table;
  for (mcba_handle* k : P->kids) table.push_back(k->d_red);
  MCBA_CUDA(cudaMalloc((void**)&P->d_table, sizeof(double*) * table.size()));
  MCBA_CUDA(cudaMemcpy(P->d_table, table.data(), sizeof(double*) * table.size(), cudaMemcpyHostToDevice));
  return MCBA_OK;
}

// out[i] = sum over the children of their packed [S | b | g | diag U | cost, sum f^2, count]
__global__ void sum_children_kernel(const double* const* __restrict__ red, int n_kids, long long n, double* __restrict__ out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int k = 0; k < n_kids; ++k) s += red[k][i];
    out[i] = s;
  }
}

static int new_problem_state(mcba_handle* h) {
  const Layout& L = h->L;
  h->have_obs = true;
  h->have_rows = false;
  // a new problem: reset the running Marquardt scaling
  MCBA_CUDA(cudaMemsetAsync(h->d_D2pose, 0, sizeof(double) * L.nTiles * 6 * kTile, h->stream));
  MCBA_CUDA(cudaMemsetAsync(h->d_D2cam, 0, sizeof(double) * L.nc, h->stream));
  return MCBA_OK;
}

static int build_reduced_host_pipelined(mcba_handle* h, const double* h_uvs, const double* h_obj, const double* h_x,
                                        double lambda, int loss, double f_scale, double* h_S, double* h_b,
                                        double* h_cost) {
  MCBA_CUDA(cudaSetDevice(h->device));
  int rc = ensure_pipe(h);
  if (rc) { const std::string why = g_error; destroy_pipe(h); set_error(why); return rc; }
  HostPipe& P = *h->pipe;
  const Layout& L = h->L;
  const size_t row = sizeof(double) * 2 * (size_t)L.N;           // one (camera, frame) row of corners
  // the copy stream must not overwrite the children's buffers while the previous call's refresh of the
  // parent still reads them (P.begin: recorded behind those copies; a no-op on the first call)
  MCBA_CUDA(cudaStreamWaitEvent(P.copy, P.begin, 0));
  MCBA_CUDA(cudaEventRecord(P.t0, P.copy));
  const int n_kids = (int)P.kids.size();
  // Parameters and board first (2.4 MB, ONE transfer each into the pipeline's own staging block: nothing else
  // reads it, so the copy stream need not wait for the compute stream); the children take their slices from
  // there on the device and the copy engine sees nothing but the eight large transfers afterwards.
  MCBA_CUDA(cudaMemcpyAsync(P.d_x, h_x, sizeof(double) * (L.nc + 6 * L.F), cudaMemcpyHostToDevice, P.copy));
  MCBA_CUDA(cudaMemcpyAsync(P.d_x + L.nc + 6 * L.F, h_obj, sizeof(double) * 3 * L.N, cudaMemcpyHostToDevice, P.copy));
  MCBA_CUDA(cudaEventRecord(P.params, P.copy));
  for (int k = 0; k < n_kids; ++k) {
    mcba_handle* kid = P.kids[k];
    const long long f0 = P.f0[k], fk = kid->L.F;
    MCBA_CUDA(cudaMemcpy2DAsync(kid->d_obs_ref, row * fk, h_uvs + (size_t)f0 * 2 * L.N, row * L.F, row * fk, L.C,
                                cudaMemcpyHostToDevice, P.copy));
    MCBA_CUDA(cudaEventRecord(P.landed[k], P.copy));
  }
  // every range is queued on the copy engine before the first kernel is: nothing on the compute side
  // (launch latency, a host synchronisation in a set-up step) can delay the transfers
  MCBA_CUDA(cudaStreamWaitEvent(h->stream, P.params, 0));
  static const bool no_graphs = getenv("MCBA_NO_PIPE_GRAPHS") != nullptr;
  if (lambda != P.g_lambda || loss != P.g_loss || f_scale != P.g_f_scale) {   // the graphs bake these in
    for (cudaGraphExec_t& g : P.graphs) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
    P.g_lambda = lambda; P.g_loss = loss; P.g_f_scale = f_scale;
    P.same_params_calls = 0;
  } else {
    ++P.same_params_calls;
  }
  // what a range does once its observations have landed (compute stream)
  auto range_work = [&](int k) -> int {
    mcba_handle* kid = P.kids[k];
    const long long f0 = P.f0[k], fk = kid->L.F;
    MCBA_CUDA(cudaMemcpyAsync(kid->d_obj, P.d_x + L.nc + 6 * L.F, sizeof(double) * 3 * L.N, cudaMemcpyDeviceToDevice, h->stream));
    MCBA_CUDA(cudaMemcpyAsync(kid->d_x, P.d_x, sizeof(double) * L.nc, cudaMemcpyDeviceToDevice, h->stream));
    MCBA_CUDA(cudaMemcpyAsync(kid->d_x + L.nc, P.d_x + L.nc + 6 * f0, sizeof(double) * 6 * fk, cudaMemcpyDeviceToDevice, h->stream));
    int r = launch_tile_observations(kid);
    if (r) return r;
    if ((r = new_problem_state(kid))) return r;
    return evaluate(kid, kid->d_x, lambda, loss, f_scale);
  };
  for (int k = 0; k < n_kids; ++k) {
    MCBA_CUDA(cudaStreamWaitEvent(h->stream, P.landed[k], 0));
    if (P.graphs[k]) {
      MCBA_CUDA(cudaGraphLaunch(P.graphs[k], h->stream));
    } else if (P.warmed[k] && !no_graphs && !P.graphs_off && P.same_params_calls >= 1) {
      cudaGraph_t graph = nullptr;
      if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();          // e.g. the legacy default stream cannot be captured: kernel by kernel from now on
        P.graphs_off = true;
        if ((rc = range_work(k))) return rc;
        MCBA_CUDA(cudaEventRecord(P.done[k], h->stream));
        continue;
      }
      rc = range_work(k);
      const cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
      if (rc || ce != cudaSuccess || !graph) {   // not capturable on this driver: run it the plain way from now on
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        P.warmed[k] = 0;
        if ((rc = range_work(k))) return rc;
      } else {
        const cudaError_t ie = cudaGraphInstantiate(&P.graphs[k], graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { P.graphs[k] = nullptr; cudaGetLastError(); P.warmed[k] = 0; if ((rc = range_work(k))) return rc; }
        else MCBA_CUDA(cudaGraphLaunch(P.graphs[k], h->stream));
      }
    } else {
      if ((rc = range_work(k))) return rc;
      P.warmed[k] = no_graphs ? 0 : 1;
    }
    MCBA_CUDA(cudaEventRecord(P.done[k], h->stream));
  }
  // sum of the children's packed systems
  const long long n_sum = L.offScal + 3;
  sum_children_kernel<<<(int)((n_sum + 255) / 256), 256, 0, h->stream>>>(P.d_table, n_kids, n_sum, h->d_red);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  if (h_S) MCBA_CUDA(cudaMemcpyAsync(h_S, h->d_red + L.offS, sizeof(double) * L.nc * L.nc, cudaMemcpyDeviceToHost, h->stream));
  if (h_b) MCBA_CUDA(cudaMemcpyAsync(h_b, h->d_red + L.offB, sizeof(double) * L.nc, cudaMemcpyDeviceToHost, h->stream));
  if (h_cost) MCBA_CUDA(cudaMemcpyAsync(h_cost, h->d_red + L.offScal + kRsCost, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  if (getenv("MCBA_PIPE_TRACE")) {
    for (int k = 0; k < n_kids; ++k) {
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, P.t0, P.landed[k]);
      cudaEventElapsedTime(&b, P.t0, P.done[k]);
      fprintf(stderr, "[mcba pipe] range %d: landed %.3f ms, evaluated %.3f ms\n", k, a, b);
    }
  }
  // The observations now live in the children.  The parent's own tiled copy (what mcba_set_observations would have
  // left) is rebuilt from them when a later call needs it (need_obs): back-to-back host-buffer calls never pay for it.
  P.parent_stale = true;
  P.lambda = lambda; P.loss = loss; P.f_scale = f_scale;
  h->have_obs = true;
  return MCBA_OK;
}

// the parent's observations, parameters and tiling from the children of the last pipelined call
static int refresh_parent_from_pipe(mcba_handle* h) {
  HostPipe& P = *h->pipe;
  const Layout& L = h->L;
  const size_t row = sizeof(double) * 2 * (size_t)L.N;
  for (size_t k = 0; k < P.kids.size(); ++k) {
    mcba_handle* kid = P.kids[k];
    MCBA_CUDA(cudaMemcpy2DAsync(h->d_obs_ref + (size_t)P.f0[k] * 2 * L.N, row * L.F, kid->d_obs_ref, row * kid->L.F,
                                row * kid->L.F, L.C, cudaMemcpyDeviceToDevice, h->stream));
  }
  MCBA_CUDA(cudaMemcpyAsync(h->d_x, P.d_x, sizeof(double) * (L.nc + 6 * L.F), cudaMemcpyDeviceToDevice, h->stream));
  MCBA_CUDA(cudaMemcpyAsync(h->d_obj, P.d_x + L.nc + 6 * L.F, sizeof(double) * 3 * L.N, cudaMemcpyDeviceToDevice, h->stream));
  MCBA_CUDA(cudaEventRecord(P.begin, h->stream));   // the children's buffers and the staging block are free from here on
  P.parent_stale = false;
  int rc = launch_tile_observations(h);
  if (rc) return rc;
  if ((rc = new_problem_state(h))) return rc;
  // ... and the evaluation itself (Z, L^-1, y, pose gradients of the WHOLE problem), so that mcba_solve_step /
  // mcba_gradient find what the plain path would have left
  return evaluate(h, h->d_x, P.lambda, P.loss, P.f_scale);
}
}  // namespace mcba

extern "C" {

int mcba_build_reduced_host(mcba_handle* h, const double* h_uvs, const double* h_obj, const double* h_x,
                            double lambda, int loss, double f_scale, double* h_S, double* h_b, double* h_cost) {
  if (!h) return MCBA_ERR_ARG;
  if (!h_uvs || !h_obj || !h_x) { set_error("mcba_build_reduced_host: null argument"); return MCBA_ERR_ARG; }
  if (h->L.F >= kHostPipeMinFrames && h->nranks <= 1 && !getenv("MCBA_NO_HOST_PIPELINE") && host_pointer_is_pinned(h_uvs) &&
      host_pointer_is_pinned(h_x))
    return build_reduced_host_pipelined(h, h_uvs, h_obj, h_x, lambda, loss, f_scale, h_S, h_b, h_cost);
  int rc = mcba_set_observations(h, h_uvs, h_obj, 0);
  if (rc) return rc;
  const long long n = h->L.nc + 6 * h->L.F;
  MCBA_CUDA(cudaMemcpyAsync(h->d_x, h_x, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
  return mcba_build_reduced(h, h->d_x, lambda, loss, f_scale, h_S, h_b, nullptr, h_cost);
}

int mcba_solve_step(mcba_handle* h, const double* d_x, double lambda, double* d_x_new) {
  int rc = need_obs(h);
  if (rc) return rc;
  if ((rc = solve_reduced(h, lambda))) return rc;
  if ((rc = launch_backsub(h, d_x, d_x_new, lambda))) return rc;
  int info[2] = {0, 0};
  MCBA_CUDA(cudaMemcpyAsync(info, h->d_info, sizeof(int) * 2, cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  if (info[0] != 0) { set_error("reduced camera system is not positive definite (potrf info = " + std::to_string(info[0]) + ")"); return MCBA_ERR_SOLVER; }
  return MCBA_OK;
}

int mcba_gradient(mcba_handle* h, double* d_grad) {
  // gradient of 0.5 sum rho at the last evaluated point: [g_cam | g_pose]
  int rc = need_obs(h);
  if (rc) return rc;
  const Layout& L = h->L;
  MCBA_CUDA(cudaMemcpyAsync(d_grad, h->d_red + L.offG, sizeof(double) * L.nc, cudaMemcpyDeviceToDevice, h->stream));
  MCBA_CUDA(cudaMemcpyAsync(d_grad + L.nc, h->d_gpose, sizeof(double) * 6 * L.F, cudaMemcpyDeviceToDevice, h->stream));
  return MCBA_OK;
}

int mcba_set_fixed(mcba_handle* h, const uint8_t* h_fixed) {
  if (!h) return MCBA_ERR_ARG;
  MCBA_CUDA(cudaSetDevice(h->device));
  const int nc = h->L.nc;
  bool any = false;
  if (h_fixed) {
    for (int i = 0; i < nc; ++i) {
      if (h_fixed[i] > 1) {
        set_error("mcba_set_fixed: entry " + std::to_string(i) + " is " + std::to_string((int)h_fixed[i]) +
                  "; entries must be 0 (free) or 1 (held)");
        return MCBA_ERR_ARG;
      }
      any |= h_fixed[i] != 0;
    }
  }
  // the kernels of work already queued may still read the previous mask
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  h->any_fixed = any;
  if (!any) { std::memset(h->h_fixed, 0, sizeof(h->h_fixed)); return MCBA_OK; }
  std::memcpy(h->h_fixed, h_fixed, nc);
  if (!h->d_fixed) MCBA_CUDA(cudaMalloc((void**)&h->d_fixed, nc));
  MCBA_CUDA(cudaMemcpyAsync(h->d_fixed, h->h_fixed, nc, cudaMemcpyHostToDevice, h->stream));
  return MCBA_OK;
}

int mcba_covariance(mcba_handle* h, const double* d_x, int loss, double f_scale, int ref, double sigma2,
                    double* h_cam_cov, double* d_pose_cov, double* h_stats) {
  int rc = need_obs(h);
  if (rc) return rc;
  const Layout& L = h->L;
  if (!d_x || !h_cam_cov) { set_error("mcba_covariance: null argument"); return MCBA_ERR_ARG; }
  if (loss != MCBA_LOSS_LINEAR && loss != MCBA_LOSS_SOFT_L1) { set_error("mcba_covariance: loss must be linear or soft_l1"); return MCBA_ERR_ARG; }
  if (!(f_scale > 0.0)) { set_error("mcba_covariance: f_scale must be positive"); return MCBA_ERR_ARG; }
  if (ref < -1 || ref >= L.C) {
    set_error("mcba_covariance: reference_camera " + std::to_string(ref) + " is not -1 or in [0, " + std::to_string(L.C) + ")");
    return MCBA_ERR_ARG;
  }
  // the gauge: a camera whose six extrinsics the mask holds pins it; otherwise the reference camera's extrinsics
  const uint8_t* held = h->any_fixed ? h->h_fixed : nullptr;
  auto pinned = [&](int c) {
    if (!held) return false;
    for (int k = 6; k < 12; ++k) if (!held[12 * c + k]) return false;
    return true;
  };
  bool any_pinned = false, any_extrinsic = false;
  for (int c = 0; c < L.C; ++c) {
    any_pinned |= pinned(c);
    for (int k = 6; k < 12; ++k) any_extrinsic |= held && held[12 * c + k];
  }
  int gauge = ref;
  if (any_pinned) {
    if (ref >= 0 && !pinned(ref)) {
      set_error("mcba_covariance: the mask holds all six extrinsics of a camera, which fixes the gauge; reference_camera " +
                std::to_string(ref) + " is not such a camera (give -1 / None, or a pinned camera)");
      return MCBA_ERR_ARG;
    }
    gauge = -1;
  } else if (ref < 0) {
    set_error("mcba_covariance: reference_camera is -1 / None but no camera has all six extrinsics held: the gauge is not fixed");
    return MCBA_ERR_ARG;
  } else if (any_extrinsic) {
    set_error("mcba_covariance: the mask holds some extrinsic parameters but no camera's complete set; with the reference "
              "camera as the gauge that over-constrains the problem (hold all six extrinsics of one camera instead)");
    return MCBA_ERR_ARG;
  }
  if (h->nranks > 1) { set_error("mcba_covariance: frame-sharded handles are not supported"); return MCBA_ERR_STATE; }
  int units[32];
  MCBA_CUDA(cudaMemcpyAsync(units, h->d_unit_count, sizeof(int) * L.C, cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  int observed[32];
  for (int c = 0; c < L.C; ++c) observed[c] = units[c] > 0;
  if (gauge >= 0 && !observed[gauge]) {
    set_error("mcba_covariance: reference camera " + std::to_string(gauge) + " has no observations");
    return MCBA_ERR_ARG;
  }
  EventPair e01, e23;
  MCBA_CUDA(cudaEventCreate(&e01.a)); MCBA_CUDA(cudaEventCreate(&e01.b));
  MCBA_CUDA(cudaEventCreate(&e23.a)); MCBA_CUDA(cudaEventCreate(&e23.b));
  // work block: [D2pose saved | Sigma (nc^2) | Sigma_raw (nc^2) | frame check (3 x u64)]
  const size_t n_d2 = (size_t)L.nTiles * 6 * kTile, n_cc = (size_t)L.nc * L.nc;
  AsyncBlock blk(h->stream);
  MCBA_CUDA(cudaMallocAsync((void**)&blk.p, sizeof(double) * (n_d2 + 2 * n_cc + 3), h->stream));
  double* d2_saved = reinterpret_cast<double*>(blk.p);
  double* d_cov = d2_saved + n_d2;
  double* d_sraw = d_cov + n_cc;
  unsigned long long* d_chk = reinterpret_cast<unsigned long long*>(d_sraw + n_cc);
  MCBA_CUDA(cudaEventRecord(e01.a, h->stream));
  // the evaluation starts from D2 = 0, so that D2pose afterwards holds diag V_f (the pivot test's reference);
  // the caller's running Marquardt scaling is put back behind the check
  MCBA_CUDA(cudaMemcpyAsync(d2_saved, h->d_D2pose, sizeof(double) * n_d2, cudaMemcpyDeviceToDevice, h->stream));
  MCBA_CUDA(cudaMemsetAsync(h->d_D2pose, 0, sizeof(double) * n_d2, h->stream));
  rc = evaluate(h, d_x, 0.0, loss, f_scale);
  if (!rc) rc = launch_cov_frame_check(h, d_chk);
  MCBA_CUDA(cudaMemcpyAsync(h->d_D2pose, d2_saved, sizeof(double) * n_d2, cudaMemcpyDeviceToDevice, h->stream));
  if (rc) return rc;
  MCBA_CUDA(cudaEventRecord(e01.b, h->stream));
  double scal[kRsNum];
  unsigned long long chk[3];
  MCBA_CUDA(cudaMemcpyAsync(scal, h->d_red + L.offScal, sizeof(scal), cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaMemcpyAsync(chk, d_chk, sizeof(chk), cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  const double cost = scal[kRsCost], m = scal[kRsCount];
  double min_pivot;
  std::memcpy(&min_pivot, &chk[2], sizeof(double));
  auto g3 = [](double v) { char b[32]; std::snprintf(b, sizeof(b), "%.3g", v); return std::string(b); };
  if (!std::isfinite(cost)) { set_error("Residuals are not finite at the given parameters."); return MCBA_ERR_NONFINITE; }
  if (chk[1] > 0) {
    set_error(std::to_string(chk[1]) + " frame(s) have a singular pose block (relative Cholesky pivot <= 1e-12, smallest " +
              g3(min_pivot) + "): too few or collinear observed corners");
    return MCBA_ERR_SOLVER;
  }
  long long p_cam = 0;   // free non-gauge parameters of the observed cameras
  for (int r = 0; r < L.nc; ++r)
    p_cam += observed[r / 12] && !(held && held[r]) && !(r / 12 == gauge && r % 12 >= 6);
  const double p = (double)p_cam + 6.0 * ((double)L.F - (double)chk[0]), dof = m - p;
  double s2 = sigma2;
  if (!(sigma2 > 0.0)) {
    if (!(dof > 0.0)) {
      set_error("mcba_covariance: " + std::to_string((long long)m) + " residuals do not exceed the " +
                std::to_string((long long)p) + " free parameters; give sigma2 to use a known noise level");
      return MCBA_ERR_ARG;
    }
    s2 = 2.0 * cost / dof;
  }
  double cam_pivot = 0.0;
  int info = 0;
  if ((rc = covariance_cameras(h, gauge, observed, held, d_cov, d_sraw, &cam_pivot, &info))) return rc;
  if (info != 0 || !(cam_pivot > kCovPivotTol)) {
    set_error("the gauge-fixed camera system is not positive definite after Jacobi scaling (smallest relative pivot " +
              g3(cam_pivot) + ", potrf/potri info " + std::to_string(info) + ")");
    return MCBA_ERR_SOLVER;
  }
  MCBA_CUDA(cudaEventRecord(e23.a, h->stream));
  if (d_pose_cov && (rc = launch_cov_poses(h, d_sraw, s2, d_pose_cov))) return rc;
  MCBA_CUDA(cudaEventRecord(e23.b, h->stream));
  MCBA_CUDA(cudaMemcpyAsync(h_cam_cov, d_cov, sizeof(double) * n_cc, cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  for (size_t i = 0; i < n_cc; ++i) h_cam_cov[i] *= s2;
  if (h_stats) {
    float ms[3] = {0, 0, 0};
    MCBA_CUDA(cudaEventElapsedTime(&ms[0], e01.a, e01.b));
    MCBA_CUDA(cudaEventElapsedTime(&ms[1], e01.b, e23.a));
    MCBA_CUDA(cudaEventElapsedTime(&ms[2], e23.a, e23.b));
    const double st[9] = {s2, dof, m, cost, (double)chk[0], min_pivot, ms[0], ms[1], ms[2]};
    std::memcpy(h_stats, st, sizeof(st));
  }
  return MCBA_OK;
}

int mcba_lm_run(mcba_handle* h, double* d_x, const mcba_options* opt_in, mcba_result* res, double* d_grad) {
  int rc = need_obs(h);
  if (rc) return rc;
  if (!d_x || !res) { set_error("mcba_lm_run: null argument"); return MCBA_ERR_ARG; }
  mcba_options opt;
  if (opt_in) opt = *opt_in; else mcba_default_options(&opt);
  const Layout& L = h->L;
  const long long n_local = L.nc + 6 * L.F;
  if (opt.lambda0 <= 0) opt.lambda0 = 1e-3;
  if (opt.lambda_min <= 0) opt.lambda_min = 1e-12;
  if (opt.lambda_max <= 0) opt.lambda_max = 1e12;
  if (opt.f_scale <= 0) { set_error("f_scale must be positive"); return MCBA_ERR_ARG; }
  std::memset(res, 0, sizeof(*res));
  const long long launches0 = h->launches;

  EventPair timing;   // destroyed on every return
  MCBA_CUDA(cudaEventCreate(&timing.a));
  MCBA_CUDA(cudaEventCreate(&timing.b));
  const cudaEvent_t ev0 = timing.a, ev1 = timing.b;
  MCBA_CUDA(cudaEventRecord(ev0, h->stream));

  double* x = h->d_x;
  double* xt = h->d_xtrial;
  MCBA_CUDA(cudaMemcpyAsync(x, d_x, sizeof(double) * n_local, cudaMemcpyDeviceToDevice, h->stream));
  // fresh Marquardt scaling for this solve
  MCBA_CUDA(cudaMemsetAsync(h->d_D2pose, 0, sizeof(double) * L.nTiles * 6 * kTile, h->stream));
  MCBA_CUDA(cudaMemsetAsync(h->d_D2cam, 0, sizeof(double) * L.nc, h->stream));

  if ((rc = ensure_alt_outputs(h))) return rc;
  double lambda = opt.lambda0, nu = 2.0;
  EvalOut ev;
  // Gauss-Newton weights: IRLS far from the minimum, scipy's Triggs scaling once the cost
  // changes by less than 1 % per step (MCBA_HESSIAN_AUTO); both share gradient and fixed point.
  bool irls = opt.hessian != MCBA_HESSIAN_TRIGGS && (opt.loss & 0xff) != MCBA_LOSS_LINEAR;
  auto loss_code = [&]() { return (opt.loss & 0xff) | (irls ? MCBA_LOSS_IRLS : 0); };
  if ((rc = evaluate(h, x, lambda, loss_code(), opt.f_scale))) return rc;
  if ((rc = read_eval(h, &ev))) return rc;
  int nfev = 1, njev = 1, iter = 0, status = -2;
  if (!std::isfinite(ev.cost) || !std::isfinite(ev.gnorm)) {
    set_error("Residuals are not finite in the initial point.");
    return MCBA_ERR_NONFINITE;
  }
  // The TOTAL parameter count decides the default evaluation budget (scipy: 100 n).  With uneven
  // shards 6 F differs between ranks, and a rank-local budget would let one rank leave the loop --
  // and the collective -- before the others: sum the pose counts over the ranks once.
  // Held camera parameters are not parameters of the sub-problem (every rank holds the same mask).
  long long n_cam_free = L.nc;
  if (h->any_fixed) for (int i = 0; i < L.nc; ++i) n_cam_free -= h->h_fixed[i];
  long long n_total = n_cam_free + 6 * L.F;
  if (h->nranks > 1 && opt.max_nfev <= 0) {
    const double mine = 6.0 * (double)L.F;
    MCBA_CUDA(cudaMemcpyAsync(h->d_scal + 40, &mine, sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if ((rc = allreduce_packed(h, h->d_scal + 40, 1))) return rc;
    MCBA_CUDA(cudaMemcpyAsync(h->h_pinned + L.redLen, h->d_scal + 40, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    MCBA_CUDA(cudaStreamSynchronize(h->stream));
    n_total = n_cam_free + (long long)h->h_pinned[L.redLen];
  }
  int max_nfev = opt.max_nfev > 0 ? opt.max_nfev : (int)std::min<long long>(100 * n_total, 2000000000LL);
  double cost = ev.cost;
  res->cost0 = cost;
  double step_norm = 0.0;
  if (opt.iter_callback) opt.iter_callback(opt.callback_user, 0, nfev, cost, NAN, NAN, ev.gnorm);
  if (ev.gnorm < opt.gtol) status = 1;

  // One host synchronisation per iteration: the scalars of the evaluation at the accepted point
  // are read back together with the NEXT trial's scalars (the trial is enqueued right behind the
  // evaluation, nothing in it depends on the host), so the GPU never idles on a host round trip
  // between the two halves of an iteration.  `pending` = an evaluation whose scalars are still
  // on their way; its iteration line is reported when they arrive.
  const long long trial_off = (L.redLen - L.offB) + 8;   // pinned mirror: [evaluation tail | trial scalars | info]
  bool pending = false;
  double last_rel_reduction = 1.0;
  double pend_reduction = NAN, pend_step = NAN;
  int pend_term = -2;
  auto settle = [&]() {   // the pending evaluation's scalars have arrived
    parse_eval(h, &ev);
    cost = ev.cost;
    if (opt.iter_callback) opt.iter_callback(opt.callback_user, iter, nfev, cost, pend_reduction, pend_step, ev.gnorm);
    pending = false;
    if (pend_term != -2) status = pend_term;
    else if (ev.gnorm < opt.gtol) status = 1;
  };
  while (status == -2) {
    if (nfev >= max_nfev) { status = 0; break; }
    if ((rc = solve_reduced(h, lambda))) return rc;
    if ((rc = launch_backsub(h, x, xt, lambda))) return rc;
    // The trial point is evaluated with the full per-observation kernel K2p into the second set of
    // outputs: its partial sums give the trial cost, and when the step is accepted (the common
    // case) its hand-off is what K2c needs next -- no separate cost pass, no second walk.
    swap_k2p_outputs(h);
    // Which Gauss-Newton weights the trial walk accumulates only matters if the step is accepted.
    // The IRLS -> Triggs switch happens when a step reduces the cost by < 1 %; once the previous
    // step was below 10 % that is the likely outcome, so the trial is walked with Triggs weights
    // already (a wrong guess costs the second walk that a blind trial would always pay).
    const bool guess_switch = irls && opt.hessian == MCBA_HESSIAN_AUTO && last_rel_reduction < 0.1;
    const int trial_loss = guess_switch ? (opt.loss & 0xff) : loss_code();
    if ((rc = launch_k2_producer(h, xt, trial_loss, opt.f_scale))) return rc;
    const bool direct = h->nranks == 1 || h->peer_ready;
    if ((rc = launch_sum_scalars(h, true))) return rc;
    double* hp = h->h_pinned + trial_off;
    if (direct) {
      if ((rc = wait_host_signal(h))) return rc;
      for (int i = 0; i < 12; ++i) hp[i] = h->h_signal_vals[i];
      reinterpret_cast<int*>(hp + 16)[0] = (int)h->h_signal_vals[12];
    } else {   // NCCL fallback: the sum runs behind the kernel, read back the classic way
      MCBA_CUDA(cudaMemcpyAsync(hp, h->d_scal, sizeof(double) * 12, cudaMemcpyDeviceToHost, h->stream));
      MCBA_CUDA(cudaMemcpyAsync(hp + 16, h->d_info, sizeof(int) * 2, cudaMemcpyDeviceToHost, h->stream));
      MCBA_CUDA(cudaStreamSynchronize(h->stream));
    }
    if (pending) {
      MCBA_CUDA(cudaEventSynchronize(h->readback_done));   // enqueued before this trial: complete, returns at once
      settle();
      if (status != -2) { swap_k2p_outputs(h); break; }   // converged at the current point: drop the trial
    }
    ++nfev;
    const double cost_new = hp[0];
    const double dd = hp[8], xx = hp[9], gd = hp[10], dDd = hp[11];
    const int info = reinterpret_cast<const int*>(hp + 16)[0];
    const bool solve_ok = info == 0 && std::isfinite(cost_new) && std::isfinite(dd);
    const double pred = -0.5 * gd + 0.5 * lambda * dDd;
    const double actual = cost - cost_new;
    const double ratio = (solve_ok && pred > 0) ? actual / pred : -1.0;
    const double sn = std::sqrt(dd), xn = std::sqrt(xx);
    bool accepted = solve_ok && actual > 0;
    int term = -2;
    if (solve_ok) {
      const bool f_ok = actual < opt.ftol * cost && ratio > 0.25;   // scipy common.py:705-717
      const bool x_ok = sn < opt.xtol * (opt.xtol + xn);
      if (f_ok && x_ok) term = 4; else if (f_ok) term = 2; else if (x_ok) term = 3;
    }
    if (accepted) {
      std::swap(x, xt);
      step_norm = sn;
      const double t = 2.0 * ratio - 1.0;
      lambda = std::max(opt.lambda_min, lambda * std::max(0.1, 1.0 - t * t * t));
      nu = 2.0;
      ++iter;
      if (irls && opt.hessian == MCBA_HESSIAN_AUTO && actual < 1e-2 * cost) irls = false;
      last_rel_reduction = actual / cost;
      if (loss_code() != trial_loss && term == -2) {   // the Gauss-Newton weights change here (once per solve): walk again
        if ((rc = evaluate(h, x, lambda, loss_code(), opt.f_scale))) return rc;
      } else {
        // (a step that ends the solve needs no new system: gradient and cost do not depend on the weights' variant)
        if ((rc = evaluate_tail(h, x, lambda, term == -2))) return rc;
      }
      if ((rc = enqueue_eval_readback(h))) return rc;
      ++njev;
      pending = true;
      pend_reduction = actual;
      pend_step = sn;
      pend_term = term;
      if (term != -2) {   // the step met ftol / xtol: finish with the evaluation at the new point
        MCBA_CUDA(cudaStreamSynchronize(h->stream));
        settle();
      }
    } else {
      swap_k2p_outputs(h);   // back to the outputs of the current point
      if (term == 3 || term == 4) { status = 3; break; }   // step too small to matter (xtol)
      lambda *= nu;
      nu *= 2.0;
      if (lambda > opt.lambda_max) { status = -1; set_error("damping exceeded lambda_max without finding a descent step"); break; }
      if ((rc = evaluate_tail(h, x, lambda))) return rc;   // pose damping is baked into Z: K2c + SYRK only
      // same point, same cost and gradient: nothing to read back
    }
  }
  if (pending) {   // left the loop on the evaluation budget with the last accepted point's scalars in flight
    // (a step that met ftol / xtol was settled at once, a rejection settles before it is decided): settle them
    // now, so that gtol met at that point reports status 1 rather than 0 -- scipy's trf tests gtol before the
    // budget, and so does every rank, since gnorm is the all-reduced maximum
    MCBA_CUDA(cudaStreamSynchronize(h->stream));
    settle();
  }

  MCBA_CUDA(cudaMemcpyAsync(d_x, x, sizeof(double) * n_local, cudaMemcpyDeviceToDevice, h->stream));
  if (d_grad) { if ((rc = mcba_gradient(h, d_grad))) return rc; }
  MCBA_CUDA(cudaEventRecord(ev1, h->stream));
  MCBA_CUDA(cudaEventSynchronize(ev1));
  float ms = 0;
  MCBA_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
  res->cost = cost;
  res->optimality = ev.gnorm;
  res->rms = ev.count > 0 ? std::sqrt(ev.sumsq / ev.count) : 0.0;
  res->step_norm = step_norm;
  res->lambda = lambda;
  res->solve_ms = ms;
  res->n_residuals = (int64_t)ev.count;
  res->nfev = nfev;
  res->njev = njev;
  res->iterations = iter;
  res->status = status;
  res->kernel_launches = h->launches - launches0;
  return MCBA_OK;
}

int mcba_comm_unique_id(void* id128) {
  int rc = load_nccl();
  if (rc) return rc;
  ncclUniqueId id;
  ncclResult_t r = g_nccl.GetUniqueId(&id);
  if (r != ncclSuccess) { set_error("ncclGetUniqueId failed"); return MCBA_ERR_NCCL; }
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  std::memcpy(id128, &id, 128);
  return MCBA_OK;
}

int mcba_comm_init(mcba_handle* h, const void* id128, int rank, int nranks) {
  if (!h || !id128 || rank < 0 || rank >= nranks || nranks > kMaxRanks) { set_error("mcba_comm_init: bad arguments"); return MCBA_ERR_ARG; }
  int rc = load_nccl();
  if (rc) return rc;
  MCBA_CUDA(cudaSetDevice(h->device));
  ncclUniqueId id;
  std::memcpy(&id, id128, 128);
  ncclComm_t comm;
  ncclResult_t r = g_nccl.CommInitRank(&comm, nranks, id, rank);
  if (r != ncclSuccess) {
    set_error(std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error"));
    return MCBA_ERR_NCCL;
  }
  h->nccl_comm = comm;
  h->rank = rank;
  h->nranks = nranks;
  return MCBA_OK;
}

int64_t mcba_kernel_launches(mcba_handle* h) { return h ? h->launches : 0; }

int mcba_plan_info(mcba_handle* h, int64_t* out, int n) {
  int rc = need_obs(h);
  if (rc) return rc;
  const Layout& L = h->L;
  const int need = MCBA_PLAN_UNITS + L.C;
  if (!out || n < need) {
    set_error("mcba_plan_info: out needs " + std::to_string(need) + " entries");
    return MCBA_ERR_ARG;
  }
  int units[32];
  MCBA_CUDA(cudaMemcpyAsync(units, h->d_unit_count, sizeof(int) * L.C, cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  int sw = 0, gy = 0, nb = 0;
  syrk_plan(L.nc, &sw, &gy, &nb);
  out[MCBA_PLAN_K2P_WARPS] = h->prod_warps;
  out[MCBA_PLAN_K2P_GRID] = h->grid_frames;
  out[MCBA_PLAN_K2C_MODE] = h->k2c_mode;
  out[MCBA_PLAN_K2C_WARPS] = h->k2c_mode == 2 ? k2c_stream_warps(L.C) : 0;
  out[MCBA_PLAN_K2C_PARTS] = h->n_part_c;
  out[MCBA_PLAN_SYRK_WARPS] = sw;
  out[MCBA_PLAN_SYRK_GY] = gy;
  out[MCBA_PLAN_SYRK_STATIC_NB] = nb;
  out[MCBA_PLAN_SOLVE] = solve_tier(L.nc);
  out[MCBA_PLAN_TILES] = L.nTiles;
  out[MCBA_PLAN_BACKSUB_GRID] = h->grid_back;
  out[MCBA_PLAN_CAMERAS] = L.C;
  for (int c = 0; c < L.C; ++c) out[MCBA_PLAN_UNITS + c] = units[c];
  return MCBA_OK;
}

int mcba_profile(mcba_handle* h, int enable, double* ms_out, int* n_out) {
  if (!h) return MCBA_ERR_ARG;
  MCBA_CUDA(cudaSetDevice(h->device));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  if (ms_out) {
    // events of one evaluation: 0 cameras ready, 1 K2p done, 4 K2c done, 2 SYRK done, 3 finalize + all-reduce done
    static const int from[4] = {0, 1, 4, 2}, to[4] = {1, 4, 2, 3};
    double acc[4] = {0, 0, 0, 0};
    for (int i = 0; i < h->prof_n; ++i) {
      for (int k = 0; k < 4; ++k) {
        float ms = 0;
        MCBA_CUDA(cudaEventElapsedTime(&ms, h->prof_ev[kProfEvents * i + from[k]], h->prof_ev[kProfEvents * i + to[k]]));
        acc[k] += ms;
      }
    }
    for (int k = 0; k < 4; ++k) ms_out[k] = acc[k];
  }
  if (n_out) *n_out = h->prof_n;
  h->prof_n = 0;
  if (enable && !h->prof_ev) {
    h->prof_ev = new cudaEvent_t[kProfEvents * kProfRing];
    for (int i = 0; i < kProfEvents * kProfRing; ++i) MCBA_CUDA(cudaEventCreate(&h->prof_ev[i]));
  }
  h->profile = enable != 0;
  return MCBA_OK;
}

}  // extern "C"
