// Covariance of the calibration (mcba_covariance): the block inverse of the Gauss-Newton matrix
// H = J~^T J~ of one evaluation at lambda = 0, from what that evaluation already left on the device:
//   cameras  Sigma_cam = S^-1 of the gauge-fixed reduced camera system (true basis), through cuSOLVER
//            potrf / potri on the Jacobi-scaled compacted system (12C <= 384, once per call);
//   frames   Sigma_f = L^-T (I + Z_f^T Sigma_raw Z_f) L^-1, Sigma_raw = T Sigma_cam T^T (raw camera rows,
//            the basis of Z), V_f = L L^T; with Z_f = W_f L^-T this is V^-1 + V^-1 W^T S^-1 W V^-1.
// Pose-block singularity is read off the factor K2c computed: L_jj = 1 / Linv_jj, so the relative pivot is
// s_j / V_jj = 1 / (Linv_jj^2 V_jj), with V_jj = diag V_f left in D2pose by an evaluation that starts from D2 = 0.
#include <cmath>
#include <vector>

#include "k2_common.cuh"

namespace mcba {

// ------------------------------------------------------------------ singular / empty frames
__global__ void cov_frame_check_kernel(const int* __restrict__ perm, const unsigned int* __restrict__ mask,
                                       const double* __restrict__ Linv, const double* __restrict__ D2pose, long long nSlots,
                                       unsigned cmask, unsigned long long* __restrict__ out) {
  unsigned long long n_empty = 0, n_sing = 0;
  double pmin = INFINITY;
  for (long long slot = blockIdx.x * (long long)blockDim.x + threadIdx.x; slot < nSlots;
       slot += (long long)gridDim.x * blockDim.x) {
    const int f = perm[slot];
    if (f < 0) continue;
    if ((~mask[f] & cmask) == 0u) { ++n_empty; continue; }
    const long long tile = slot / kTile;
    const int lane = (int)(slot % kTile);
    double rel = INFINITY;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const double li = Linv[((size_t)tile * 21 + j * (j + 1) / 2 + j) * kTile + lane];
      const double v = D2pose[((size_t)tile * 6 + j) * kTile + lane];
      rel = fmin(rel, li == 0.0 ? 0.0 : 1.0 / (li * li * v));   // Linv_jj = 0: the pivot was <= 0
    }
    if (!(rel > kCovPivotTol)) ++n_sing;
    pmin = fmin(pmin, rel);
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    n_empty += __shfl_xor_sync(0xffffffffu, n_empty, off);
    n_sing += __shfl_xor_sync(0xffffffffu, n_sing, off);
    pmin = fmin(pmin, __shfl_xor_sync(0xffffffffu, pmin, off));
  }
  if ((threadIdx.x & 31) == 0) {
    if (n_empty) atomicAdd(out, n_empty);
    if (n_sing) atomicAdd(out + 1, n_sing);
    // non-negative doubles order like their bit patterns
    atomicMin(out + 2, (unsigned long long)__double_as_longlong(pmin));
  }
}

int launch_cov_frame_check(mcba_handle* h, unsigned long long* d_out) {
  const Layout& L = h->L;
  const unsigned long long init[3] = {0ull, 0ull, 0x7ff0000000000000ull};   // +inf
  MCBA_CUDA(cudaMemcpyAsync(d_out, init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
  const unsigned cmask = L.C >= 32 ? 0xffffffffu : (1u << L.C) - 1u;
  const int grid = (int)std::min<long long>((L.Fpad + 255) / 256, 4LL * h->n_sm);
  cov_frame_check_kernel<<<grid, 256, 0, h->stream>>>(h->d_perm, h->d_mask, h->d_Linv, h->d_D2pose, L.Fpad, cmask, d_out);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

// ------------------------------------------------------------------ camera block
// A = D^-1/2 S[keep, keep] D^-1/2 (column-major, symmetric), rs = D^-1/2 (0 where S_ii <= 0: potrf then fails)
__global__ void cov_compact_kernel(const double* __restrict__ S, int nc, const int* __restrict__ keep, int nk,
                                   double* __restrict__ A, double* __restrict__ rs) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nk * nk; e += gridDim.x * blockDim.x) {
    const int i = e / nk, j = e % nk;
    const double di = S[(size_t)keep[i] * nc + keep[i]], dj = S[(size_t)keep[j] * nc + keep[j]];
    const double si = di > 0.0 ? rsqrt(di) : 0.0, sj = dj > 0.0 ? rsqrt(dj) : 0.0;
    A[e] = S[(size_t)keep[i] * nc + keep[j]] * si * sj;
    if (i == j) rs[i] = si;
  }
}

// smallest squared diagonal entry of the Cholesky factor of the unit-diagonal A: its smallest relative pivot
__global__ void cov_pivot_kernel(const double* __restrict__ A, int nk, double* __restrict__ out) {
  double m = INFINITY;
  for (int j = threadIdx.x; j < nk; j += blockDim.x) {
    const double l = A[(size_t)j * nk + j];
    m = fmin(m, l * l);
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, off));
  __shared__ double s[32];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmin(m, s[w]);
    out[0] = m != m ? 0.0 : m;
  }
}

// Sigma (nc x nc, true basis) from the inverse of A (lower triangle, column-major): pos[r] = row of A, -1 gauge,
// -2 unobserved camera, -3 held parameter (0, also against an unobserved camera)
__global__ void cov_expand_kernel(const double* __restrict__ Ainv, int nk, const double* __restrict__ rs,
                                  const int* __restrict__ pos, int nc, double* __restrict__ cov) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nc * nc; e += gridDim.x * blockDim.x) {
    const int pr = pos[e / nc], pq = pos[e % nc];
    double v;
    if (pr == -3 || pq == -3) v = 0.0;
    else if (pr == -2 || pq == -2) v = NAN;
    else if (pr < 0 || pq < 0) v = 0.0;
    else v = Ainv[(size_t)min(pr, pq) * nk + max(pr, pq)] * rs[pr] * rs[pq];
    cov[e] = v;
  }
}

// row i of T_c = [[I6,0,0],[0,Jl,0],[0,[t]x Jl,I3]] (rows raw [intr | m | G], columns true [intr | r | t])
__device__ __forceinline__ double t_entry(const CamConst& cam, int i, int k) {
  if (i < 6) return i == k ? 1.0 : 0.0;
  if (k < 6) return 0.0;
  if (i < 9) return k < 9 ? cam.Jl[(i - 6) * 3 + (k - 6)] : 0.0;
  return k < 9 ? cam.tJ[(i - 9) * 3 + (k - 6)] : (i == k ? 1.0 : 0.0);
}

// Sigma_raw = T Sigma T^T block by block; unobserved cameras (NaN in Sigma) contribute 0 (their Z rows are 0)
__global__ void cov_raw_kernel(const double* __restrict__ cov, const CamConst* __restrict__ cams, int nc,
                               double* __restrict__ sraw) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nc * nc; e += gridDim.x * blockDim.x) {
    const int r = e / nc, q = e % nc, a = r / 12, b = q / 12, i = r % 12, j = q % 12;
    const CamConst& ca = cams[a];
    const CamConst& cb = cams[b];
    double s = 0.0;
    for (int k = 0; k < 12; ++k) {
      const double tk = t_entry(ca, i, k);
      if (tk == 0.0) continue;
      double t = 0.0;
      for (int l = 0; l < 12; ++l) {
        const double tl = t_entry(cb, j, l);
        if (tl != 0.0) t += cov[(size_t)(12 * a + k) * nc + 12 * b + l] * tl;
      }
      s += tk * t;
    }
    sraw[e] = s == s ? s : 0.0;
  }
}

int covariance_cameras(mcba_handle* h, int ref, const int* observed, const uint8_t* held, double* d_cov, double* d_sraw,
                       double* min_pivot, int* info) {
  const Layout& L = h->L;
  const int nc = L.nc;
  std::vector<int> keep, pos(nc);
  for (int r = 0; r < nc; ++r) {
    const int c = r / 12;
    if (held && held[r]) pos[r] = -3;
    else if (!observed[c]) pos[r] = -2;
    else if (c == ref && r % 12 >= 6) pos[r] = -1;
    else { pos[r] = (int)keep.size(); keep.push_back(r); }
  }
  const int nk = (int)keep.size();
  const int grid = (nc * nc + 255) / 256;
  if (nk == 0) {   // every camera parameter held: nothing to invert, Sigma is 0 / NaN and Sigma_raw 0
    AsyncBlock blk(h->stream);
    MCBA_CUDA(cudaMallocAsync((void**)&blk.p, sizeof(int) * nc, h->stream));
    int* d_pos = reinterpret_cast<int*>(blk.p);
    MCBA_CUDA(cudaMemcpyAsync(d_pos, pos.data(), sizeof(int) * nc, cudaMemcpyHostToDevice, h->stream));
    cov_expand_kernel<<<grid, 256, 0, h->stream>>>(nullptr, 0, nullptr, d_pos, nc, d_cov);
    cov_raw_kernel<<<grid, 256, 0, h->stream>>>(d_cov, h->d_cams, nc, d_sraw);
    h->launches += 2;
    MCBA_CUDA(cudaGetLastError());
    MCBA_CUDA(cudaStreamSynchronize(h->stream));   // pos is a host vector
    *min_pivot = INFINITY;
    *info = 0;
    return MCBA_OK;
  }
  int rc = ensure_solver(h);
  if (rc) return rc;
  int lw_f = 0, lw_i = 0;
  if (cusolverDnDpotrf_bufferSize(h->solver, CUBLAS_FILL_MODE_LOWER, nk, nullptr, nk, &lw_f) != CUSOLVER_STATUS_SUCCESS ||
      cusolverDnDpotri_bufferSize(h->solver, CUBLAS_FILL_MODE_LOWER, nk, nullptr, nk, &lw_i) != CUSOLVER_STATUS_SUCCESS) {
    set_error("cusolverDnDpotrf / potri bufferSize failed");
    return MCBA_ERR_SOLVER;
  }
  const int lwork = std::max(1, std::max(lw_f, lw_i));
  // [A nk^2 | rs nk | work | pivot 1 | info 2 (as doubles) | keep nk, pos nc (ints)]
  const size_t n_dbl = (size_t)nk * nk + nk + lwork + 1 + 2;
  AsyncBlock blk(h->stream);
  MCBA_CUDA(cudaMallocAsync((void**)&blk.p, sizeof(double) * n_dbl + sizeof(int) * (nk + nc), h->stream));
  double* A = reinterpret_cast<double*>(blk.p);
  double* rs = A + (size_t)nk * nk;
  double* work = rs + nk;
  double* d_piv = work + lwork;
  int* d_info = reinterpret_cast<int*>(d_piv + 1);
  int* d_keep = reinterpret_cast<int*>(d_piv + 3);
  int* d_pos = d_keep + nk;
  std::vector<int> idx(keep);
  idx.insert(idx.end(), pos.begin(), pos.end());
  MCBA_CUDA(cudaMemcpyAsync(d_keep, idx.data(), sizeof(int) * idx.size(), cudaMemcpyHostToDevice, h->stream));
  const double* S = h->d_red + L.offS;
  cov_compact_kernel<<<(nk * nk + 255) / 256, 256, 0, h->stream>>>(S, nc, d_keep, nk, A, rs);
  MCBA_CUDA(cudaGetLastError());
  if (cusolverDnDpotrf(h->solver, CUBLAS_FILL_MODE_LOWER, nk, A, nk, work, lwork, d_info) != CUSOLVER_STATUS_SUCCESS) {
    set_error("cusolverDnDpotrf failed");
    return MCBA_ERR_SOLVER;
  }
  cov_pivot_kernel<<<1, 256, 0, h->stream>>>(A, nk, d_piv);
  MCBA_CUDA(cudaGetLastError());
  if (cusolverDnDpotri(h->solver, CUBLAS_FILL_MODE_LOWER, nk, A, nk, work, lwork, d_info + 1) != CUSOLVER_STATUS_SUCCESS) {
    set_error("cusolverDnDpotri failed");
    return MCBA_ERR_SOLVER;
  }
  cov_expand_kernel<<<grid, 256, 0, h->stream>>>(A, nk, rs, d_pos, nc, d_cov);
  cov_raw_kernel<<<grid, 256, 0, h->stream>>>(d_cov, h->d_cams, nc, d_sraw);
  h->launches += 6;   // compact, potrf, pivot, potri, expand, raw (library calls counted once)
  MCBA_CUDA(cudaGetLastError());
  double piv = 0.0;
  int inf[2] = {0, 0};
  MCBA_CUDA(cudaMemcpyAsync(&piv, d_piv, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaMemcpyAsync(inf, d_info, sizeof(inf), cudaMemcpyDeviceToHost, h->stream));
  MCBA_CUDA(cudaStreamSynchronize(h->stream));
  *min_pivot = piv;
  *info = inf[0] != 0 ? inf[0] : inf[1];
  return MCBA_OK;
}

// ------------------------------------------------------------------ pose blocks
// One warp per frame tile (lane = frame), cameras the tile does not see skipped as a whole (their Z rows are 0):
// for every live camera a, Y_a = sum_b Sigma_raw[a, b] Z_b (12 x 6 per lane, in registers; one broadcast read of
// Sigma_raw feeds six FMAs), then G += Z_a^T Y_a (upper triangle).  Sigma_raw sits in shared memory when it fits
// (12C <= 156: 13 cameras), otherwise it is read through the L1 cache from global memory (1.2 MB at 32 cameras,
// L2-resident).  Z rows are coalesced 256-byte loads.  Output: s2 L^-T (I + G) L^-1, 36 doubles per frame.
constexpr int kCovWarps = 4;
constexpr size_t kCovSmemMax = 200 * 1024;

struct CovPoseParams {
  int C, nc;
  long long nTiles;
  const int* perm;
  const unsigned int* mask;
  const unsigned int* active;
  const double* Z;
  const double* Linv;
  const double* sraw;   // global copy
  double s2;
  double* out;          // (F, 6, 6)
  int sraw_in_smem;
};

__global__ void __launch_bounds__(kCovWarps * 32) cov_pose_kernel(const CovPoseParams p) {
  extern __shared__ __align__(16) double cov_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nc = p.nc;
  const double* sig = p.sraw;
  if (p.sraw_in_smem) {
    for (int i = threadIdx.x; i < nc * nc; i += blockDim.x) cov_smem[i] = p.sraw[i];
    __syncthreads();
    sig = cov_smem;
  }
  const unsigned cmask = p.C >= 32 ? 0xffffffffu : (1u << p.C) - 1u;
  for (long long tile = (long long)blockIdx.x * kCovWarps + warp; tile < p.nTiles; tile += (long long)gridDim.x * kCovWarps) {
    const int f = p.perm[tile * kTile + lane];
    const unsigned act = p.active[tile] & cmask;
    const double* zt = p.Z + (size_t)tile * nc * 6 * kTile + lane;   // row r, column k: zt[(r * 6 + k) * kTile]
    double G[21];
#pragma unroll
    for (int i = 0; i < 21; ++i) G[i] = 0.0;
    for (unsigned ma = act; ma; ma &= ma - 1) {
      const int a = __ffs(ma) - 1;
      double Y[12][6];
#pragma unroll
      for (int i = 0; i < 12; ++i)
#pragma unroll
        for (int k = 0; k < 6; ++k) Y[i][k] = 0.0;
      for (unsigned mb = act; mb; mb &= mb - 1) {
        const int b = __ffs(mb) - 1;
        const double* srow = sig + (size_t)(12 * a) * nc + 12 * b;
#pragma unroll 2
        for (int j = 0; j < 12; ++j) {
          double z[6];
#pragma unroll
          for (int k = 0; k < 6; ++k) z[k] = zt[((12 * b + j) * 6 + k) * kTile];
#pragma unroll
          for (int i = 0; i < 12; ++i) {
            const double s = srow[(size_t)i * nc + j];
#pragma unroll
            for (int k = 0; k < 6; ++k) Y[i][k] = fma(s, z[k], Y[i][k]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 12; ++i) {
        double z[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) z[k] = zt[((12 * a + i) * 6 + k) * kTile];
#pragma unroll
        for (int k = 0; k < 6; ++k)
#pragma unroll
          for (int l = k; l < 6; ++l) G[tri6(k, l)] = fma(z[k], Y[i][l], G[tri6(k, l)]);
      }
    }
    if (f < 0) continue;
    double* o = p.out + (size_t)f * 36;
    if ((~p.mask[f] & cmask) == 0u) {   // no observation: the pose is not determined
#pragma unroll
      for (int i = 0; i < 36; i += 2) *reinterpret_cast<double2*>(o + i) = make_double2(NAN, NAN);
      continue;
    }
    double li[21];
    const double* lo = p.Linv + (size_t)tile * 21 * kTile + lane;
#pragma unroll
    for (int i = 0; i < 21; ++i) li[i] = lo[i * kTile];
    // P = (I + G) L^-1  (L^-1 lower: row l, column j <= l), then out = L^-T P
    double P[6][6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        double t = 0.0;
#pragma unroll
        for (int l = 0; l < 6; ++l)
          if (l >= j) t = fma((k == l ? 1.0 : 0.0) + G[sym6(k, l)], li[l * (l + 1) / 2 + j], t);
        P[k][j] = t;
      }
    }
    double res[36];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
#pragma unroll
      for (int j = i; j < 6; ++j) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k)
          if (k >= i) t = fma(li[k * (k + 1) / 2 + i], P[k][j], t);
        res[6 * i + j] = p.s2 * t;
        res[6 * j + i] = p.s2 * t;
      }
    }
#pragma unroll
    for (int i = 0; i < 36; i += 2) *reinterpret_cast<double2*>(o + i) = make_double2(res[i], res[i + 1]);
  }
}

int launch_cov_poses(mcba_handle* h, const double* d_sraw, double s2, double* d_pose_cov) {
  const Layout& L = h->L;
  CovPoseParams p;
  p.C = L.C; p.nc = L.nc; p.nTiles = L.nTiles;
  p.perm = h->d_perm; p.mask = h->d_mask; p.active = h->d_active;
  p.Z = h->d_Z; p.Linv = h->d_Linv; p.sraw = d_sraw; p.s2 = s2; p.out = d_pose_cov;
  const size_t bytes = sizeof(double) * (size_t)L.nc * L.nc;
  p.sraw_in_smem = bytes <= kCovSmemMax ? 1 : 0;
  const size_t smem = p.sraw_in_smem ? bytes : 0;
  MCBA_CUDA(set_dynamic_smem((const void*)cov_pose_kernel, smem));
  const int grid = (int)std::min<long long>((L.nTiles + kCovWarps - 1) / kCovWarps, 16LL * h->n_sm);
  cov_pose_kernel<<<grid, kCovWarps * 32, smem, h->stream>>>(p);
  h->launches++;
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

}  // namespace mcba
