// K1 family: camera constants, observation tiling, the materialised residual
// vector (bundle_adjustment.py:66-98), dense predictions (:33-63), the robust
// cost, and the per-observation analytic Jacobian blocks used by the parity tests.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <type_traits>

#include "mcba_internal.h"
#include "mcba_obs.cuh"

namespace mcba {

// ---------------------------------------------------------------- cameras
__global__ void prep_cameras_kernel(const double* __restrict__ x, int C, CamConst* __restrict__ cams) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double* p = x + 12 * c;
  CamConst k;
  k.fx = p[0]; k.fy = p[1]; k.cx = p[2]; k.cy = p[3]; k.k1 = p[4]; k.k2 = p[5];
  const double r[3] = {p[6], p[7], p[8]};
  k.t[0] = p[9]; k.t[1] = p[10]; k.t[2] = p[11];
  rodrigues(r, k.R);
  so3_left_jacobian(r, k.Jl);
  cross_mat3(k.t, k.Jl, k.tJ);
  cams[c] = k;
}

int launch_prep_cameras(mcba_handle* h, const double* x) {
  prep_cameras_kernel<<<(h->L.C + 31) / 32, 32, 0, h->stream>>>(x, h->L.C, h->d_cams);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

// ---------------------------------------------------------------- observation layouts
// reference (C,F,N,2)  ->  tiled [tile][c][n][lane] (double2), NaN padded to 32 frames.
//
// Frame order.  Tile slot (tile, lane) holds frame perm[tile*32 + lane] (-1 = padding).  When the
// camera count is small the frames are sorted (stably) by their visibility mask - bit c set when
// camera c has at least one finite scalar in the frame - so that the 32 frames of a tile almost
// always share one mask: a (tile, camera) unit then is either fully observed or empty, empty
// units are skipped as a whole and no lane idles through a missing view (20 % of the lanes at
// BASELINE configs[2]).  The order is internal: x, the pose gradient and every C-ABI array stay
// in the caller's frame order; only the pose loads / stores go through perm.

// visibility mask per frame: one warp per (frame), loops cameras
__global__ void frame_mask_kernel(const double* __restrict__ ref, int C, long long F, int N,
                                  unsigned int* __restrict__ mask) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long f = warp; f < F; f += nwarps) {
    unsigned int m = 0;
    for (int c = 0; c < C; ++c) {
      const double* p = ref + ((long long)c * F + f) * 2 * N;
      bool any = false;
      for (int s = lane; s < 2 * N; s += 32) any |= p[s] == p[s];
      if (__any_sync(0xffffffffu, any)) m |= 1u << c;
    }
    if (lane == 0) mask[f] = ~m;   // complement: fully observed frames sort first
  }
}

__global__ void iota_kernel(int* __restrict__ v, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    v[i] = (int)i;
}

// perm padding + per-tile active-camera mask
__global__ void tile_active_kernel(const unsigned int* __restrict__ mask, int* __restrict__ perm, long long F,
                                   long long nTiles, unsigned int* __restrict__ active) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long tile = warp; tile < nTiles; tile += nwarps) {
    const long long slot = tile * kTile + lane;
    unsigned int m = 0;
    if (slot < F) m = ~mask[perm[slot]];
    else perm[slot] = -1;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, off);
    if (lane == 0) active[tile] = m;
  }
}

// Live (tile, camera) units, compacted per camera in tile order: units[c][k] = k-th tile in which
// camera c has observations, count[c] of them.  One CTA per camera.  K2p walks only these.
__global__ void __launch_bounds__(256) build_units_kernel(const unsigned int* __restrict__ active, long long nTiles,
                                                          int* __restrict__ units, int* __restrict__ count) {
  __shared__ int s_warp[8];
  __shared__ int s_base;
  const int c = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (long long t0 = 0; t0 < nTiles; t0 += blockDim.x) {
    const long long t = t0 + threadIdx.x;
    const bool live = t < nTiles && ((active[t] >> c) & 1u);
    const unsigned int b = __ballot_sync(0xffffffffu, live);
    if (lane == 0) s_warp[warp] = __popc(b);
    __syncthreads();
    int off = s_base;
    for (int w = 0; w < warp; ++w) off += s_warp[w];
    if (live) units[(long long)c * nTiles + off + __popc(b & ((1u << lane) - 1u))] = (int)t;
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int w = 0; w < 8; ++w) tot += s_warp[w];
      s_base += tot;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) count[c] = s_base;
}

// gprefix[c] = number of groups of `warps` units before camera c; gprefix[C] = total
__global__ void group_prefix_kernel(const int* __restrict__ count, int C, int warps, int* __restrict__ gprefix) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    int acc = 0;
    for (int c = 0; c < C; ++c) {
      gprefix[c] = acc;
      acc += (count[c] + warps - 1) / warps;
    }
    gprefix[C] = acc;
  }
}

// one CTA per (tile, camera) unit: coalesced row loads -> shared -> coalesced [n][lane] stores
// Also counts the finite scalars it moves (n_scalars, zeroed by the caller): the residual count K2p reports
// with every evaluation without counting again.
__global__ void __launch_bounds__(256) tile_observations_kernel(const double2* __restrict__ ref,
                                                                double2* __restrict__ tiled,
                                                                const int* __restrict__ perm, int C, long long F,
                                                                int N, long long nUnits,
                                                                unsigned long long* __restrict__ n_scalars) {
  extern __shared__ double2 s_rows[];   // [32][N + 1]
  const int ldr = N + 1;
  unsigned int finite = 0;
  for (long long unit = blockIdx.x; unit < nUnits; unit += gridDim.x) {
    const long long tile = unit / C;
    const int c = (int)(unit % C);
    for (int i = threadIdx.x; i < kTile * N; i += blockDim.x) {
      const int r = i / N, n = i % N;
      const int f = perm[tile * kTile + r];
      double2 v = make_double2(nan(""), nan(""));
      if (f >= 0) v = ref[((long long)c * F + f) * N + n];
      finite += (v.x == v.x ? 1u : 0u) + (v.y == v.y ? 1u : 0u);
      s_rows[r * ldr + n] = v;
    }
    __syncthreads();
    double2* out = tiled + (size_t)unit * N * kTile;
    for (int i = threadIdx.x; i < kTile * N; i += blockDim.x) out[i] = s_rows[(i % kTile) * ldr + i / kTile];
    __syncthreads();
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) finite += __shfl_xor_sync(0xffffffffu, finite, off);
  if ((threadIdx.x & 31) == 0 && finite) atomicAdd(n_scalars, (unsigned long long)finite);
}

int launch_tile_observations(mcba_handle* h) {
  const Layout& L = h->L;
  const int blocks = 148 * 8;
  // ---- frame order: sorted by visibility mask.  The 32 frames of a tile share the leading ~log2(nTiles) bits of
  //      the sorted key: all cameras when 2^C <= nTiles, the highest-numbered ones otherwise
  frame_mask_kernel<<<blocks, 256, 0, h->stream>>>(h->d_obs_ref, L.C, L.F, L.N, h->d_mask);
  iota_kernel<<<blocks, 256, 0, h->stream>>>(h->d_perm, L.Fpad);
  size_t bytes = 0;
  unsigned int* keys_out = h->d_mask + L.Fpad;
  int* vals_out = h->d_perm + L.Fpad;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, h->d_mask, keys_out, h->d_perm, vals_out, (int)L.F, 0, L.C, h->stream);
  if (bytes > h->sort_tmp_bytes) {
    if (h->d_sort_tmp) cudaFree(h->d_sort_tmp);
    MCBA_CUDA(cudaMalloc(&h->d_sort_tmp, bytes));
    h->sort_tmp_bytes = bytes;
  }
  MCBA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp, bytes, h->d_mask, keys_out, h->d_perm, vals_out, (int)L.F,
                                            0, L.C, h->stream));
  MCBA_CUDA(cudaMemcpyAsync(h->d_perm, vals_out, sizeof(int) * L.F, cudaMemcpyDeviceToDevice, h->stream));
  h->launches += 4;
  tile_active_kernel<<<blocks, 256, 0, h->stream>>>(h->d_mask, h->d_perm, L.F, L.nTiles, h->d_active);
  const long long units = L.nTiles * L.C;
  const int grid = (int)(units < 148 * 8 ? units : 148 * 8);
  unsigned long long* n_scalars = reinterpret_cast<unsigned long long*>(h->d_unit_count + 96);
  MCBA_CUDA(cudaMemsetAsync(n_scalars, 0, sizeof(unsigned long long), h->stream));
  // 16 * 32 * (N + 1) bytes: above the 48 KB default from 96 corners on (mcba_create rejects boards whose
  // transpose does not fit the device's opt-in limit)
  const size_t tile_smem = tile_observations_smem(L.N);
  MCBA_CUDA(set_dynamic_smem((const void*)tile_observations_kernel, tile_smem));
  tile_observations_kernel<<<grid, 256, tile_smem, h->stream>>>(
      reinterpret_cast<const double2*>(h->d_obs_ref), h->d_obs_tiled, h->d_perm, L.C, L.F, L.N, units, n_scalars);
  build_units_kernel<<<L.C, 256, 0, h->stream>>>(h->d_active, L.nTiles, h->d_units, h->d_unit_count);
  group_prefix_kernel<<<1, 32, 0, h->stream>>>(h->d_unit_count, L.C, h->prod_warps, h->d_unit_count + 32);
  // dead units are never written by K2p: their hand-off stays zero
  MCBA_CUDA(cudaMemsetAsync(h->d_H, 0, sizeof(double) * (size_t)L.nTiles * L.C * 63 * kTile, h->stream));
  h->alt_stale = true;
  // ... and K2c never writes their Z rows
  MCBA_CUDA(cudaMemsetAsync(h->d_Z, 0, sizeof(double) * (size_t)L.Fpad * 6 * L.nc, h->stream));
  h->launches += 4;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

// ---- K1: residuals and predictions by chunks ---------------------------------------------------
// A chunk = one camera's 32 consecutive frames = ONE contiguous block of 32*N double2 in the
// reference layout (C,F,N,2), for the observations as well as for the predictions.
constexpr int kChunkFrames = 32;

// finite scalars of every chunk (one warp per chunk, coalesced) + number of observed corners
__global__ void count_chunks_kernel(const double2* __restrict__ ref, int C, long long F, int N, long long nBlk,
                                    long long* __restrict__ counts, unsigned int* __restrict__ chunk_rows,
                                    unsigned long long* __restrict__ n_obs) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  unsigned long long obs = 0;
  for (long long u = warp; u < (long long)C * nBlk; u += nwarps) {
    const int c = (int)(u / nBlk);
    const long long f0 = (u % nBlk) * kChunkFrames;
    const long long nf = F - f0 < kChunkFrames ? F - f0 : kChunkFrames;
    const double2* p = ref + ((long long)c * F + f0) * N;
    int cnt = 0;
    unsigned rows = 0;   // bit r: (camera, frame f0 + r) has at least one finite scalar
    for (long long i = lane; i < nf * N; i += 32) {
      const double2 o = p[i];
      const bool fu = o.x == o.x, fv = o.y == o.y;
      cnt += (fu ? 1 : 0) + (fv ? 1 : 0);
      obs += (fu | fv) ? 1 : 0;
      if (fu | fv) rows |= 1u << (unsigned)(i / N);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
      cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
      rows |= __shfl_xor_sync(0xffffffffu, rows, off);
    }
    if (lane == 0) { counts[u] = cnt; chunk_rows[u] = rows; }
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) obs += __shfl_xor_sync(0xffffffffu, obs, off);
  if (lane == 0 && obs) atomicAdd(n_obs, obs);
}

// offsets of the NaN compaction (bundle_adjustment.py:97) per chunk; only K1 needs them
int ensure_row_offsets(mcba_handle* h) {
  if (h->have_rows) return MCBA_OK;
  const Layout& L = h->L;
  const long long nBlk = (L.F + kChunkFrames - 1) / kChunkFrames;
  const long long groups = (long long)L.C * nBlk;
  unsigned long long* d_nobs = nullptr;
  MCBA_CUDA(cudaMalloc(&d_nobs, sizeof(unsigned long long)));
  MCBA_CUDA(cudaMemsetAsync(d_nobs, 0, sizeof(unsigned long long), h->stream));
  MCBA_CUDA(cudaMemsetAsync(h->d_row_off, 0, sizeof(long long) * (groups + 1), h->stream));
  int grid = (int)((groups * 32 + 255) / 256 < 148 * 16 ? (groups * 32 + 255) / 256 : 148 * 16);
  if (grid < 1) grid = 1;
  if (!h->d_chunk_rows) MCBA_CUDA(cudaMalloc((void**)&h->d_chunk_rows, sizeof(unsigned int) * (size_t)(groups + 1)));
  count_chunks_kernel<<<grid, 256, 0, h->stream>>>(reinterpret_cast<const double2*>(h->d_obs_ref), L.C, L.F, L.N, nBlk,
                                                  h->d_row_off, h->d_chunk_rows, d_nobs);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  size_t tmp_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, h->d_row_off, h->d_row_off, (int)(groups + 1), h->stream);
  void* d_tmp = nullptr;
  MCBA_CUDA(cudaMalloc(&d_tmp, tmp_bytes));
  MCBA_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, h->d_row_off, h->d_row_off, (int)(groups + 1), h->stream));
  h->launches++;
  long long m = 0;
  unsigned long long nobs = 0;
  MCBA_CUDA(cudaMemcpyAsync(&m, h->d_row_off + groups, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaMemcpyAsync(&nobs, d_nobs, sizeof(nobs), cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  MCBA_CUDA(cudaFree(d_tmp));
  MCBA_CUDA(cudaFree(d_nobs));
  h->m = m;
  h->n_obs = (long long)nobs;
  h->have_rows = true;
  return MCBA_OK;
}

// K1 (chunked): 16 B read + up to 16 B written per (c,f,n) slot, no auxiliary pass.
// Each warp owns chunks (camera c, frames f0..f0+31).
//   phase A  lane = frame: the composed transform X_c = R_c R(rho_f) X_o + (R_c tau_f + t_c) of
//            the chunk's 32 (camera, frame) rows goes to the warp's 3 KB of shared memory
//            (Rodrigues once per row, not once per slot);
//   phase B  lane = slot: the chunk's nf * N slots are walked in their memory order, four groups
//            of 32 in flight per warp: one coalesced 16-byte load per slot, the row's transform
//            from shared memory (at most two distinct rows per group: broadcast reads), one
//            projection for both scalars, then either the ballot-compacted residuals in the
//            reference's order c, f, n, {u, v} (bundle_adjustment.py:97) from a running offset
//            that starts at the chunk's scanned offset, or the coalesced predictions.
// Per group of 32 slots this is ~80 warp instructions (45 of them FP64) against ~160 for a flat
// kernel that indexes every (c,f,n) slot on its own.
#ifndef MCBA_K1_CTAS
#define MCBA_K1_CTAS 4
#endif
template <bool kCompact>
__global__ void __launch_bounds__(256, MCBA_K1_CTAS) residual_chunks_kernel(const double* __restrict__ x, const double2* __restrict__ ref,
                                                              const double* __restrict__ obj,
                                                              const long long* __restrict__ chunk_off,
                                                              const unsigned int* __restrict__ chunk_rows, int C, long long F,
                                                              int N, long long nBlk, double* __restrict__ out) {
  extern __shared__ __align__(16) double k1_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nWarps = blockDim.x >> 5;
  double* s_T = k1_smem + (size_t)warp * kChunkFrames * 12;          // [32 rows][12]
  double* s_cam = k1_smem + (size_t)nWarps * kChunkFrames * 12;       // [C][18]: fx fy cx cy k1 k2 | R (9) | t (3)
  double* s_obj = s_cam + (size_t)C * 18;                             // [3 N]
  int* s_rk = reinterpret_cast<int*>(s_obj + ((3 * N + 1) & ~1)) + warp * kChunkFrames;   // [32] row of the q-th LIVE row of the chunk
  for (int i = threadIdx.x; i < 3 * N; i += blockDim.x) s_obj[i] = obj[i];
  if (threadIdx.x < C) {   // camera constants in the kernel itself: no separate launch in front of it
    const double* p = x + 12 * threadIdx.x;
    double* sc = s_cam + 18 * threadIdx.x;
#pragma unroll
    for (int i = 0; i < 6; ++i) sc[i] = p[i];
    const double r[3] = {p[6], p[7], p[8]};
    double R[9];
    rodrigues(r, R);
#pragma unroll
    for (int i = 0; i < 9; ++i) sc[6 + i] = R[i];
    sc[15] = p[9]; sc[16] = p[10]; sc[17] = p[11];
  }
  __syncthreads();
  const long long nUnits = (long long)C * nBlk;
  const long long gw = (long long)blockIdx.x * nWarps + warp, stride = (long long)gridDim.x * nWarps;
  // slot -> row within the chunk: i / N for i < 32 N <= 2^16 N ... exact for i * N < 2^32 with a 32-bit reciprocal
  // (N = 1: the reciprocal 2^32 does not fit in 32 bits, and the row is the slot itself)
  const unsigned inv_n = (unsigned)((0x100000000ull + (unsigned)N - 1) / (unsigned)N);
  auto row_of = [&](int i) { return N == 1 ? i : (int)__umulhi((unsigned)i, inv_n); };
  const unsigned lt = (1u << lane) - 1u;
  for (long long u = gw; u < nUnits; u += stride) {
    const int c = (int)(u / nBlk);
    const long long f0 = (u % nBlk) * kChunkFrames;
    const int nf = (int)(F - f0 < kChunkFrames ? F - f0 : kChunkFrames);
    const double* sc = s_cam + 18 * c;
    const Intr in{sc[0], sc[1], sc[2], sc[3], sc[4], sc[5]};
    // Rows (camera, frame) without a single detection -- a camera that did not see the board -- are known from
    // the counting pass.  Only the LIVE rows are walked: their transforms and row numbers are stored by rank, and
    // the slot loop runs over rank * N + corner, so a dead row costs neither loads nor instructions.
    const unsigned rows = kCompact ? chunk_rows[u] : (nf >= 32 ? 0xffffffffu : (1u << nf) - 1u);
    const int n_live = __popc(rows);
    const int rank = __popc(rows & lt);
    __syncwarp();   // the previous chunk's readers are done with s_T and s_rk
    if ((rows >> lane) & 1u) {
      s_rk[rank] = lane;
      const double* ps = x + 12 * (long long)C + 6 * (f0 + lane);
      const double rho[3] = {ps[0], ps[1], ps[2]}, tau[3] = {ps[3], ps[4], ps[5]};
      double Rc[9], Rp[9], Rcf[9], tcf[3];
#pragma unroll
      for (int i = 0; i < 9; ++i) Rc[i] = sc[6 + i];
      rodrigues(rho, Rp);
      mat3_mul(Rc, Rp, Rcf);
      mat3_vec(Rc, tau, tcf);
      double2* t = reinterpret_cast<double2*>(s_T + rank * 12);
      t[0] = make_double2(Rcf[0], Rcf[1]);
      t[1] = make_double2(Rcf[2], Rcf[3]);
      t[2] = make_double2(Rcf[4], Rcf[5]);
      t[3] = make_double2(Rcf[6], Rcf[7]);
      t[4] = make_double2(Rcf[8], tcf[0] + sc[15]);
      t[5] = make_double2(tcf[1] + sc[16], tcf[2] + sc[17]);
    }
    __syncwarp();
    const int total = n_live * N;                           // slots of the live rows, in the reference order
    const long long base = ((long long)c * F + f0) * N;     // first slot of the chunk
    // the chunk's residuals start at its scanned offset; positions inside the chunk are 32-bit
    double* out_c = out + (kCompact ? chunk_off[u] : 0);
    int off = 0;
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    constexpr int kU = 4;
    // four groups of 32 slots per step; a step that lies wholly inside the chunk runs without any
    // bounds test (8 of the 9 steps of a full 32-frame x 35-corner chunk), the last one with them
    auto step = [&](int i0, auto checked_tag) {
      constexpr bool kChecked = decltype(checked_tag)::value;
      double2 o[kU];
#pragma unroll
      for (int g = 0; g < kU; ++g) {
        const int i = i0 + g * 32 + lane;
        o[g] = make_double2(qnan, qnan);
        if (kCompact && (!kChecked || i < total)) {
          const int q = row_of(i);
          o[g] = ref[base + (s_rk[q] - q) * N + i];
        }
      }
#pragma unroll
      for (int g = 0; g < kU; ++g) {
        const int i = i0 + g * 32 + lane;
        if (kChecked && i0 + g * 32 >= total) break;   // warp-uniform
        bool fu = false, fv = false;
        double ru = 0.0, rv = 0.0;
        if (!kChecked || i < total) {
          const int q = row_of(i);   // rank of the slot's row among the live rows
          const int n = i - q * N;
          const double2* t = reinterpret_cast<const double2*>(s_T + q * 12);
          const double2 t0 = t[0], t1 = t[1], t2 = t[2], t3 = t[3], t4 = t[4], t5 = t[5];
          const double Rcf[9] = {t0.x, t0.y, t1.x, t1.y, t2.x, t2.y, t3.x, t3.y, t4.x};
          const double tcf[3] = {t4.y, t5.x, t5.y};
          double pu, pv;
          project(in, Rcf, tcf, s_obj[3 * n], s_obj[3 * n + 1], s_obj[3 * n + 2], pu, pv);
          if (kCompact) {
            fu = o[g].x == o[g].x;
            fv = o[g].y == o[g].y;
            ru = o[g].x - pu;
            rv = o[g].y - pv;
          } else {
            reinterpret_cast<double2*>(out)[base + i] = make_double2(pu, pv);   // all rows live here: rank = row
          }
        }
        if (kCompact) {
          const unsigned bu = __ballot_sync(0xffffffffu, fu), bv = __ballot_sync(0xffffffffu, fv);
          const int pos = off + __popc(bu & lt) + __popc(bv & lt);
          double* dst = out_c + pos;
          // both scalars of a detection (the usual case) leave as one 16-byte store when aligned
          if (fu && fv && ((reinterpret_cast<unsigned long long>(dst) & 15ull) == 0)) {
            *reinterpret_cast<double2*>(dst) = make_double2(ru, rv);
          } else {
            if (fu) dst[0] = ru;
            if (fv) dst[fu ? 1 : 0] = rv;
          }
          off += __popc(bu) + __popc(bv);
        }
      }
    };
    int i0 = 0;
    for (; i0 + 32 * kU <= total; i0 += 32 * kU) step(i0, std::false_type{});
    if (i0 < total) step(i0, std::true_type{});
  }
}

static int launch_chunks(mcba_handle* h, const double* x, double* out, bool compact) {
  const Layout& L = h->L;
  const int warps = 8;
  const long long nBlk = (L.F + kChunkFrames - 1) / kChunkFrames;
  const long long units = (long long)L.C * nBlk;
  const size_t smem = sizeof(double) * ((size_t)warps * kChunkFrames * 12 + 18 * (size_t)L.C + ((3 * (size_t)L.N + 1) & ~(size_t)1)) +
                      sizeof(int) * (size_t)warps * kChunkFrames;
  long long grid = (units + warps - 1) / warps;
  if (grid > 8LL * h->n_sm) grid = 8LL * h->n_sm;
  if (smem > 48 * 1024) {
    MCBA_CUDA(set_dynamic_smem((const void*)residual_chunks_kernel<true>, smem));
    MCBA_CUDA(set_dynamic_smem((const void*)residual_chunks_kernel<false>, smem));
  }
  if (compact)
    residual_chunks_kernel<true><<<(int)grid, warps * 32, smem, h->stream>>>(
        x, reinterpret_cast<const double2*>(h->d_obs_ref), h->d_obj, h->d_row_off, h->d_chunk_rows, L.C, L.F, L.N, nBlk, out);
  else
    residual_chunks_kernel<false><<<(int)grid, warps * 32, smem, h->stream>>>(x, nullptr, h->d_obj, nullptr, nullptr, L.C, L.F,
                                                                             L.N, nBlk, out);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

int launch_residuals(mcba_handle* h, const double* x, double* r_out) { return launch_chunks(h, x, r_out, true); }

int launch_predict(mcba_handle* h, const double* x, double* uv_out) { return launch_chunks(h, x, uv_out, false); }

// ---------------------------------------------------------------- robust cost
// warp per (tile, camera), lane = frame, tiled SoA (the walk of K2p without the Jacobian); C ABI mcba_cost
__global__ void __launch_bounds__(256) cost_kernel(const double* __restrict__ x, const double2* __restrict__ obs,
                                                   const double* __restrict__ obj, const CamConst* __restrict__ cams,
                                                   const int* __restrict__ perm, const unsigned int* __restrict__ active,
                                                   int C, long long F, int N, long long nTiles, int loss, double inv_c,
                                                   double c2, double* __restrict__ part, unsigned int* __restrict__ counter,
                                                   double* __restrict__ out) {
  extern __shared__ double s_obj[];
  __shared__ double s_red[8 * 3];
  __shared__ bool s_last;
  for (int i = threadIdx.x; i < 3 * N; i += blockDim.x) s_obj[i] = obj[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long gw = blockIdx.x * (long long)(blockDim.x >> 5) + warp;
  const long long nw = (long long)gridDim.x * (blockDim.x >> 5);
  double cost = 0.0, sumsq = 0.0, cnt = 0.0;
  for (long long job = gw; job < nTiles * C; job += nw) {
    const long long tile = job / C;
    const int c = (int)(job % C);
    if (!((active[tile] >> c) & 1u)) continue;   // no observation of camera c in this tile
    const long long f = perm[tile * kTile + lane];
    if (f >= 0) {
      const CamConst& cam = cams[c];
      const Intr in{cam.fx, cam.fy, cam.cx, cam.cy, cam.k1, cam.k2};
      const double* ps = x + 12 * (long long)C + 6 * f;
      const double rho[3] = {ps[0], ps[1], ps[2]}, tau[3] = {ps[3], ps[4], ps[5]};
      double Rp[9], Rcf[9], tcf[3];
      rodrigues(rho, Rp);
      mat3_mul(cam.R, Rp, Rcf);
      mat3_vec(cam.R, tau, tcf);
      tcf[0] += cam.t[0]; tcf[1] += cam.t[1]; tcf[2] += cam.t[2];
      const double2* ob = obs + (size_t)job * N * kTile + lane;
#pragma unroll 5
      for (int n = 0; n < N; ++n) {
        const double2 o = ob[(size_t)n * kTile];
        const bool hu = o.x == o.x, hv = o.y == o.y;
        if (hu | hv) {
          double pu, pv;
          project(in, Rcf, tcf, s_obj[3 * n], s_obj[3 * n + 1], s_obj[3 * n + 2], pu, pv);
          double rho_, wg, wh;
          if (hu) {
            const double fu = o.x - pu;
            robust_weights(loss, fu, inv_c, c2, rho_, wg, wh);
            cost += rho_; sumsq += fu * fu; cnt += 1.0;
          }
          if (hv) {
            const double fv = o.y - pv;
            robust_weights(loss, fv, inv_c, c2, rho_, wg, wh);
            cost += rho_; sumsq += fv * fv; cnt += 1.0;
          }
        }
      }
    }
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    cost += __shfl_xor_sync(0xffffffffu, cost, off);
    sumsq += __shfl_xor_sync(0xffffffffu, sumsq, off);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
  }
  if (lane == 0) { s_red[warp * 3] = cost; s_red[warp * 3 + 1] = sumsq; s_red[warp * 3 + 2] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0, k = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += s_red[w * 3]; b += s_red[w * 3 + 1]; k += s_red[w * 3 + 2]; }
    part[blockIdx.x * 3] = 0.5 * a;
    part[blockIdx.x * 3 + 1] = b;
    part[blockIdx.x * 3 + 2] = k;
    __threadfence();
    s_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last) {   // deterministic final sum by the last CTA to finish
    __threadfence();
    double a = 0, b = 0, k = 0;
    for (unsigned i = threadIdx.x; i < gridDim.x; i += blockDim.x) {
      a += __ldcg(part + i * 3); b += __ldcg(part + i * 3 + 1); k += __ldcg(part + i * 3 + 2);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, off);
      b += __shfl_xor_sync(0xffffffffu, b, off);
      k += __shfl_xor_sync(0xffffffffu, k, off);
    }
    __syncthreads();
    if (lane == 0) { s_red[warp * 3] = a; s_red[warp * 3 + 1] = b; s_red[warp * 3 + 2] = k; }
    __syncthreads();
    if (threadIdx.x == 0) {
      a = b = k = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += s_red[w * 3]; b += s_red[w * 3 + 1]; k += s_red[w * 3 + 2]; }
      out[0] = a; out[1] = b; out[2] = k;
      *counter = 0;
    }
  }
}

int launch_cost(mcba_handle* h, const double* x, int loss, double f_scale, double* out_scal) {
  const Layout& L = h->L;
  int rc = launch_prep_cameras(h, x);
  if (rc) return rc;
  double* part = h->d_scal + 64;                                  // [grid_cost][3]
  unsigned int* counter = reinterpret_cast<unsigned int*>(h->d_scal + 32);
  cost_kernel<<<h->grid_cost, 256, sizeof(double) * 3 * L.N, h->stream>>>(
      x, h->d_obs_tiled, h->d_obj, h->d_cams, h->d_perm, h->d_active, L.C, L.F, L.N, L.nTiles, loss, 1.0 / f_scale,
      f_scale * f_scale, part, counter, out_scal);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

// ---------------------------------------------------------------- Jacobian blocks (parity path)
// One thread per (c,f,n).  RESIDUAL Jacobian = -(prediction Jacobian).
__global__ void jacobian_blocks_kernel(const double* __restrict__ x, const double* __restrict__ obj,
                                       const CamConst* __restrict__ cams, int C, long long F, int N,
                                       double* __restrict__ Jc, double* __restrict__ Jp) {
  const long long total = (long long)C * F * N;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i % N);
    const long long f = (i / N) % F;
    const int c = (int)(i / ((long long)N * F));
    const CamConst& cam = cams[c];
    const Intr in{cam.fx, cam.fy, cam.cx, cam.cy, cam.k1, cam.k2};
    const double* ps = x + 12 * (long long)C + 6 * f;
    const double rho[3] = {ps[0], ps[1], ps[2]}, tau[3] = {ps[3], ps[4], ps[5]};
    double Rp[9], Jlp[9], Rcf[9], tcf[3], K[9], RJ[9], KJ[9];
    rodrigues(rho, Rp);
    so3_left_jacobian(rho, Jlp);
    mat3_mul(cam.R, Rp, Rcf);
    mat3_vec(cam.R, tau, tcf);
    tcf[0] += cam.t[0]; tcf[1] += cam.t[1]; tcf[2] += cam.t[2];
    cross_mat3(tcf, cam.R, K);
    mat3_mul(cam.R, Jlp, RJ);   // R_c J_l(rho)
    mat3_mul(K, Jlp, KJ);       // [t_cf]x R_c J_l(rho)
    double pu, pv, a[2][10];
    project_jac(in, Rcf, tcf, obj[3 * n], obj[3 * n + 1], obj[3 * n + 2], pu, pv, a[0], a[1]);
    for (int row = 0; row < 2; ++row) {
      const double* ar = a[row];
      double* jc = Jc + (i * 2 + row) * 12;
      double* jp = Jp + (i * 2 + row) * 6;
      for (int k = 0; k < 12; ++k) jc[k] = 0.0;
      jc[row] = -ar[0];            // fx | fy
      jc[2 + row] = -ar[1];        // cx | cy
      jc[4] = -ar[2];
      jc[5] = -ar[3];
      const double* m = ar + 4;
      const double* G = ar + 7;
      for (int k = 0; k < 3; ++k) {
        jc[6 + k] = -(m[0] * cam.Jl[k] + m[1] * cam.Jl[3 + k] + m[2] * cam.Jl[6 + k] +
                      G[0] * cam.tJ[k] + G[1] * cam.tJ[3 + k] + G[2] * cam.tJ[6 + k]);
        jc[9 + k] = -G[k];
        jp[k] = -(m[0] * RJ[k] + m[1] * RJ[3 + k] + m[2] * RJ[6 + k] +
                  G[0] * KJ[k] + G[1] * KJ[3 + k] + G[2] * KJ[6 + k]);
        jp[3 + k] = -(G[0] * cam.R[k] + G[1] * cam.R[3 + k] + G[2] * cam.R[6 + k]);
      }
    }
  }
}

int launch_jacobian_blocks(mcba_handle* h, const double* x, double* Jc, double* Jp) {
  const Layout& L = h->L;
  int rc = launch_prep_cameras(h, x);
  if (rc) return rc;
  const long long total = (long long)L.C * L.F * L.N;
  long long g = (total + 127) / 128;
  if (g > 148 * 8) g = 148 * 8;
  jacobian_blocks_kernel<<<(int)g, 128, 0, h->stream>>>(x, h->d_obj, h->d_cams, L.C, L.F, L.N, Jc, Jp);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

}  // namespace mcba
