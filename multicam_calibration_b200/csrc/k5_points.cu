// Config 5: batched geometry.project_points (geometry.py:277-325) and
// geometry.triangulate (geometry.py:361-433): undistort (OpenCV's fixed 5-step
// inversion of the 5-coefficient model) -> all-pairs homogeneous DLT (smallest
// right singular vector of the 4x4 system, one-sided Jacobi in fp64) ->
// per-coordinate nanmedian over camera pairs.  One thread per point.
#include "mcba_internal.h"

namespace mcba {

struct ProjCam {
  double R[9], t[3], K[9], k1, k2;
  int has_dist;
};

__global__ void project_points_kernel(const double* __restrict__ pts, long long P, const ProjCam cam,
                                      double* __restrict__ uv) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < P; i += (long long)gridDim.x * blockDim.x) {
    const double p[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    double X[3];
    mat3_vec(cam.R, p, X);
    X[0] += cam.t[0]; X[1] += cam.t[1]; X[2] += cam.t[2];
    if (cam.has_dist) {
      const double xn = X[0] / X[2], yn = X[1] / X[2];
      const double r2 = xn * xn + yn * yn;
      const double d = 1.0 + cam.k1 * r2 + cam.k2 * (r2 * r2);
      X[0] *= d;
      X[1] *= d;
    }
    double h[3];
    mat3_vec(cam.K, X, h);
    reinterpret_cast<double2*>(uv)[i] = make_double2(h[0] / h[2], h[1] / h[2]);
  }
}

// All cameras of a rig in one pass: each point is read once (24 B) and projected into the C
// views (16 B written per view); uv is (C,P,2).  Points are staged through shared memory so that
// the stride-3 reads become coalesced 8-byte rows.
constexpr int kProjByValue = 16;   // cameras passed in the kernel's parameter space (3 KB of the 4 KB limit)
struct ProjCamPack {
  ProjCam c[kProjByValue];
};

__global__ void __launch_bounds__(256) project_points_multi_kernel(const double* __restrict__ pts, long long P, int C,
                                                                   const __grid_constant__ ProjCamPack pack,
                                                                   const ProjCam* __restrict__ cams,
                                                                   double* __restrict__ uv) {
  extern __shared__ unsigned char pm_smem[];
  ProjCam* sc = reinterpret_cast<ProjCam*>(pm_smem);
  double* sp = reinterpret_cast<double*>(pm_smem + sizeof(ProjCam) * C);   // [256][3]
  const double* src = cams ? reinterpret_cast<const double*>(cams) : reinterpret_cast<const double*>(&pack);
  for (int i = threadIdx.x; i < C * (int)(sizeof(ProjCam) / sizeof(double)); i += blockDim.x)
    reinterpret_cast<double*>(sc)[i] = src[i];
  for (long long base = blockIdx.x * 256LL; base < P; base += gridDim.x * 256LL) {
    const long long n_here = P - base < 256 ? P - base : 256;
    __syncthreads();
    for (int i = threadIdx.x; i < 3 * n_here; i += 256) sp[i] = pts[3 * base + i];
    __syncthreads();
    if (threadIdx.x < n_here) {
      const double p[3] = {sp[3 * threadIdx.x], sp[3 * threadIdx.x + 1], sp[3 * threadIdx.x + 2]};
      for (int c = 0; c < C; ++c) {
        const ProjCam& cam = sc[c];
        double X[3];
        mat3_vec(cam.R, p, X);
        X[0] += cam.t[0]; X[1] += cam.t[1]; X[2] += cam.t[2];
        if (cam.has_dist) {
          const double iz = 1.0 / X[2];   // one reciprocal per division pair: the pass is FP64-issue bound
          const double xn = X[0] * iz, yn = X[1] * iz;
          const double r2 = xn * xn + yn * yn;
          const double d = 1.0 + cam.k1 * r2 + cam.k2 * (r2 * r2);
          X[0] *= d;
          X[1] *= d;
        }
        double h[3];
        mat3_vec(cam.K, X, h);
        const double ih = 1.0 / h[2];
        reinterpret_cast<double2*>(uv)[(long long)c * P + base + threadIdx.x] = make_double2(h[0] * ih, h[1] * ih);
      }
    }
  }
}

// X_w[f,n] = R(rho_f) X_o[n] + tau_f   (bundle_adjustment.py:27-29)
__global__ void embed_points_kernel(const double* __restrict__ poses, long long F, const double* __restrict__ obj,
                                    int N, double* __restrict__ world) {
  const long long total = F * N;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long f = i / N;
    const int n = (int)(i % N);
    const double* ps = poses + 6 * f;
    const double r[3] = {ps[0], ps[1], ps[2]};
    double R[9], X[3];
    rodrigues(r, R);
    const double q[3] = {obj[3 * n], obj[3 * n + 1], obj[3 * n + 2]};
    mat3_vec(R, q, X);
    world[3 * i] = X[0] + ps[3];
    world[3 * i + 1] = X[1] + ps[4];
    world[3 * i + 2] = X[2] + ps[5];
  }
}

struct TriCam {
  double P[12];                 // K [R|t]
  double fx, fy, cx, cy, skew;  // K entries used by undistortion
  double k1, k2, p1, p2, k3;
};

// OpenCV undistortPoints(uv, K, dist5, None, K): exactly 5 fixed-point iterations of the
// 5-coefficient model; normalisation ignores skew, re-projection applies the full K.
__device__ __forceinline__ void undistort5(const TriCam& k, double u, double v, double& uo, double& vo) {
  const double x0 = (u - k.cx) / k.fx, y0 = (v - k.cy) / k.fy;
  double x = x0, y = y0;
#pragma unroll
  for (int it = 0; it < 5; ++it) {
    const double r2 = x * x + y * y;
    const double icd = 1.0 / (1.0 + ((k.k3 * r2 + k.k2) * r2 + k.k1) * r2);
    const double dx = 2.0 * k.p1 * x * y + k.p2 * (r2 + 2.0 * x * x);
    const double dy = k.p1 * (r2 + 2.0 * y * y) + 2.0 * k.p2 * x * y;
    x = (x0 - dx) * icd;
    y = (y0 - dy) * icd;
  }
  uo = x * k.fx + y * k.skew + k.cx;
  vo = y * k.fy + k.cy;
}

__global__ void undistort_points_kernel(const double2* __restrict__ in, long long P, const TriCam cam,
                                        double2* __restrict__ out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < P; i += (long long)gridDim.x * blockDim.x) {
    const double2 o = in[i];
    double2 r = make_double2(nan(""), nan(""));
    if (o.x == o.x && o.y == o.y) undistort5(cam, o.x, o.y, r.x, r.y);
    out[i] = r;
  }
}

// Smallest right singular vector of a 4x4 matrix by one-sided (Hestenes) Jacobi.
__device__ __forceinline__ void smallest_right_singular_vector(double A[4][4], double out[4]) {
  double V[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) V[i][j] = (i == j) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 30; ++sweep) {
    bool rotated = false;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
#pragma unroll
      for (int q = p + 1; q < 4; ++q) {
        double a = 0, b = 0, g = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          a = fma(A[i][p], A[i][p], a);
          b = fma(A[i][q], A[i][q], b);
          g = fma(A[i][p], A[i][q], g);
        }
        if (fabs(g) > 1e-16 * sqrt(a * b) && g != 0.0) {
          rotated = true;
          const double zeta = (b - a) / (2.0 * g);
          const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
          const double c = rsqrt(1.0 + t * t), s = c * t;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const double ap = A[i][p], aq = A[i][q];
            A[i][p] = c * ap - s * aq;
            A[i][q] = s * ap + c * aq;
            const double vp = V[i][p], vq = V[i][q];
            V[i][p] = c * vp - s * vq;
            V[i][q] = s * vp + c * vq;
          }
        }
      }
    }
    if (!rotated) break;
  }
  int best = 0;
  double bn = INFINITY;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    double n = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) n = fma(A[i][j], A[i][j], n);
    if (n < bn) { bn = n; best = j; }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) out[i] = best == 0 ? V[i][0] : best == 1 ? V[i][1] : best == 2 ? V[i][2] : V[i][3];
}

// The same vector for the DLT systems of triangulation, ~10x cheaper: A = Q R (Householder), the
// smallest right singular vector of A is that of R.  With one small singular value the null
// direction sits in the last column: start from the back-substitution solution of R[:3,:3] y = -R[:3,3]
// (exact when R33 = 0) and polish with inverse iteration on R^T R (two triangular solves per
// step; error shrinks by (sigma_4 / sigma_3)^2 per step).  Returns false when the iteration has
// not settled to 1e-13 after 8 steps (near-degenerate pair): the caller then runs the Jacobi SVD.
__device__ __forceinline__ bool null_vector_qr(const double (&A0)[4][4], double out[4]) {
  double R[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) R[i][j] = A0[i][j];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    double nrm2 = 0.0;
#pragma unroll
    for (int i = k; i < 4; ++i) nrm2 = fma(R[i][k], R[i][k], nrm2);
    const double alpha = -copysign(sqrt(nrm2), R[k][k]);
    double v[4];
#pragma unroll
    for (int i = k; i < 4; ++i) v[i] = R[i][k];
    v[k] -= alpha;
    double vv = 0.0;
#pragma unroll
    for (int i = k; i < 4; ++i) vv = fma(v[i], v[i], vv);
    if (vv > 0.0) {
      const double beta = 2.0 / vv;
#pragma unroll
      for (int j = k + 1; j < 4; ++j) {
        double d = 0.0;
#pragma unroll
        for (int i = k; i < 4; ++i) d = fma(v[i], R[i][j], d);
        d *= beta;
#pragma unroll
        for (int i = k; i < 4; ++i) R[i][j] = fma(-d, v[i], R[i][j]);
      }
    }
    R[k][k] = alpha;
  }
  const double scale = fabs(R[0][0]) + fabs(R[1][1]) + fabs(R[2][2]);
  if (!(scale > 0.0) || !(scale < INFINITY)) return false;
  if (fabs(R[0][0]) < 1e-12 * scale || fabs(R[1][1]) < 1e-12 * scale || fabs(R[2][2]) < 1e-12 * scale) return false;
  double r33 = R[3][3];
  if (fabs(r33) < 1e-300) r33 = 1e-300;
  const double i0 = 1.0 / R[0][0], i1 = 1.0 / R[1][1], i2 = 1.0 / R[2][2], i3 = 1.0 / r33;
  double y[4];
  y[3] = 1.0;
  y[2] = -(R[2][3]) * i2;
  y[1] = -(R[1][2] * y[2] + R[1][3]) * i1;
  y[0] = -(R[0][1] * y[1] + R[0][2] * y[2] + R[0][3]) * i0;
  {
    const double n = rsqrt(y[0] * y[0] + y[1] * y[1] + y[2] * y[2] + 1.0);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] *= n;
  }
  bool ok = false;
  for (int it = 0; it < 8 && !ok; ++it) {
    double z[4], w[4];
    z[0] = y[0] * i0;                                               // R^T z = y
    z[1] = (y[1] - R[0][1] * z[0]) * i1;
    z[2] = (y[2] - R[0][2] * z[0] - R[1][2] * z[1]) * i2;
    z[3] = (y[3] - R[0][3] * z[0] - R[1][3] * z[1] - R[2][3] * z[2]) * i3;
    w[3] = z[3] * i3;                                               // R w = z
    w[2] = (z[2] - R[2][3] * w[3]) * i2;
    w[1] = (z[1] - R[1][2] * w[2] - R[1][3] * w[3]) * i1;
    w[0] = (z[0] - R[0][1] * w[1] - R[0][2] * w[2] - R[0][3] * w[3]) * i0;
    // scale first: w can be ~1/sigma_4^2
    const double m = fmax(fmax(fabs(w[0]), fabs(w[1])), fmax(fabs(w[2]), fabs(w[3])));
    if (!(m > 0.0) || !(m < INFINITY)) return false;
    const double im = 1.0 / m;
#pragma unroll
    for (int i = 0; i < 4; ++i) w[i] *= im;
    double n = rsqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2] + w[3] * w[3]);
    const double dot = w[0] * y[0] + w[1] * y[1] + w[2] * y[2] + w[3] * y[3];
    if (dot < 0.0) n = -n;
    double diff = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const double wi = w[i] * n;
      diff = fmax(diff, fabs(wi - y[i]));
      y[i] = wi;
    }
    ok = it >= 1 && diff < 1e-13;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) out[i] = y[i];
  return ok;
}

__device__ __forceinline__ double nan_median(double* v, int n) {
  if (n == 0) return nan("");
  for (int i = 1; i < n; ++i) {  // insertion sort
    const double key = v[i];
    int j = i - 1;
    while (j >= 0 && v[j] > key) { v[j + 1] = v[j]; --j; }
    v[j + 1] = key;
  }
  return (n & 1) ? v[n / 2] : 0.5 * (v[n / 2 - 1] + v[n / 2]);
}

template <int kMaxC>
__global__ void __launch_bounds__(128) triangulate_kernel(const double* __restrict__ uvs, int C, long long P,
                                                          const TriCam* __restrict__ cams, double* __restrict__ out) {
  constexpr int kMaxPairs = kMaxC * (kMaxC - 1) / 2;
  extern __shared__ unsigned char s_raw[];
  TriCam* sc = reinterpret_cast<TriCam*>(s_raw);
  for (int i = threadIdx.x; i < C * (int)(sizeof(TriCam) / sizeof(double)); i += blockDim.x)
    reinterpret_cast<double*>(sc)[i] = reinterpret_cast<const double*>(cams)[i];
  __syncthreads();
  for (long long pt = blockIdx.x * (long long)blockDim.x + threadIdx.x; pt < P; pt += (long long)gridDim.x * blockDim.x) {
    double und[kMaxC][2];
    bool seen[kMaxC];
    for (int c = 0; c < C; ++c) {
      const double2 o = reinterpret_cast<const double2*>(uvs)[(long long)c * P + pt];
      undistort5(sc[c], o.x, o.y, und[c][0], und[c][1]);
      // seen from the undistorted pixel, as the reference's triangulate decides it: a NaN input stays
      // NaN, and an infinite or overflowing one (+-inf, 1e300) undistorts to NaN and enters no pair
      seen[c] = (und[c][0] == und[c][0]) && (und[c][1] == und[c][1]);
    }
    double px[kMaxPairs], py[kMaxPairs], pz[kMaxPairs];
    int np = 0;
    for (int i = 0; i < C; ++i) {
      if (!seen[i]) continue;
      for (int j = i + 1; j < C; ++j) {
        if (!seen[j]) continue;
        double A[4][4];
        const double* Pi = sc[i].P;
        const double* Pj = sc[j].P;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          A[0][k] = und[i][0] * Pi[8 + k] - Pi[k];
          A[1][k] = und[i][1] * Pi[8 + k] - Pi[4 + k];
          A[2][k] = und[j][0] * Pj[8 + k] - Pj[k];
          A[3][k] = und[j][1] * Pj[8 + k] - Pj[4 + k];
        }
        double X[4];
        if (!null_vector_qr(A, X)) smallest_right_singular_vector(A, X);
        const double vx = X[0] / X[3], vy = X[1] / X[3], vz = X[2] / X[3];
        // np.nanmedian drops NaN entries per coordinate (geometry.py:432)
        px[np] = vx; py[np] = vy; pz[np] = vz;
        ++np;
      }
    }
    // per-coordinate NaN filtering
    int nx = 0, ny = 0, nz = 0;
    for (int i = 0; i < np; ++i) {
      if (px[i] == px[i]) px[nx++] = px[i];
      if (py[i] == py[i]) py[ny++] = py[i];
      if (pz[i] == pz[i]) pz[nz++] = pz[i];
    }
    double rx = nan(""), ry = nan(""), rz = nan("");
    if (nx + ny + nz > 0) {   // row is NaN only when every pairwise value is NaN (geometry.py:429)
      rx = nan_median(px, nx);
      ry = nan_median(py, ny);
      rz = nan_median(pz, nz);
    }
    out[3 * pt] = rx;
    out[3 * pt + 1] = ry;
    out[3 * pt + 2] = rz;
  }
}

void host_rodrigues(const double r[3], double R[9]) {
  const double th = std::sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
  const double inv = th == 0.0 ? 1.0 : 1.0 / th;
  const double k[3] = {r[0] * inv, r[1] * inv, r[2] * inv};
  const double s = std::sin(th), oc = 1.0 - std::cos(th);
  const double n2 = k[0] * k[0] + k[1] * k[1] + k[2] * k[2];
  R[0] = 1.0 + oc * (k[0] * k[0] - n2); R[1] = -s * k[2] + oc * k[0] * k[1]; R[2] = s * k[1] + oc * k[0] * k[2];
  R[3] = s * k[2] + oc * k[0] * k[1]; R[4] = 1.0 + oc * (k[1] * k[1] - n2); R[5] = -s * k[0] + oc * k[1] * k[2];
  R[6] = -s * k[1] + oc * k[0] * k[2]; R[7] = s * k[0] + oc * k[1] * k[2]; R[8] = 1.0 + oc * (k[2] * k[2] - n2);
}

}  // namespace mcba

using namespace mcba;

extern "C" {

int mcba_project_points(int device, void* stream, const double* d_points, int64_t P, const double* ext,
                        const double* K, const double* dist, double* d_uv) {
  if (!d_points || !ext || !K || !d_uv || P < 0) { set_error("mcba_project_points: bad arguments"); return MCBA_ERR_ARG; }
  MCBA_CUDA(cudaSetDevice(device));
  if (P == 0) return MCBA_OK;
  ProjCam cam;
  host_rodrigues(ext, cam.R);
  for (int i = 0; i < 3; ++i) cam.t[i] = ext[3 + i];
  for (int i = 0; i < 9; ++i) cam.K[i] = K[i];
  cam.has_dist = dist != nullptr;
  cam.k1 = dist ? dist[0] : 0.0;
  cam.k2 = dist ? dist[1] : 0.0;
  const int grid = (int)std::min<long long>((P + 255) / 256, 148 * 16);
  project_points_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_points, P, cam, d_uv);
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

int mcba_project_points_multi(int device, void* stream, const double* d_points, int64_t P, int C, const double* ext,
                              const double* K, const double* dist, double* d_uv) {
  if (!d_points || !ext || !K || !d_uv || P < 0 || C < 1 || C > 64) {
    set_error("mcba_project_points_multi: bad arguments (1 <= n_cameras <= 64)");
    return MCBA_ERR_ARG;
  }
  MCBA_CUDA(cudaSetDevice(device));
  if (P == 0) return MCBA_OK;
  { int rc = keep_async_pool(device); if (rc) return rc; }
  static ProjCamPack pack;     // cameras 0..15 travel by value: no upload, no synchronisation
  ProjCam cams_big[64];
  ProjCam* cams = C <= kProjByValue ? pack.c : cams_big;
  for (int c = 0; c < C; ++c) {
    host_rodrigues(ext + 6 * c, cams[c].R);
    for (int i = 0; i < 3; ++i) cams[c].t[i] = ext[6 * c + 3 + i];
    for (int i = 0; i < 9; ++i) cams[c].K[i] = K[9 * c + i];
    cams[c].has_dist = dist != nullptr;
    cams[c].k1 = dist ? dist[2 * c] : 0.0;
    cams[c].k2 = dist ? dist[2 * c + 1] : 0.0;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int grid = (int)std::min<long long>((P + 255) / 256, 148 * 8);
  const size_t smem = sizeof(ProjCam) * C + sizeof(double) * 3 * 256;
  if (C <= kProjByValue) {
    project_points_multi_kernel<<<grid, 256, smem, s>>>(d_points, P, C, pack, nullptr, d_uv);
    MCBA_CUDA(cudaGetLastError());
    return MCBA_OK;
  }
  ProjCam* d_cams = nullptr;
  MCBA_CUDA(cudaMallocAsync((void**)&d_cams, sizeof(ProjCam) * C, s));
  MCBA_CUDA(cudaMemcpyAsync(d_cams, cams, sizeof(ProjCam) * C, cudaMemcpyHostToDevice, s));
  project_points_multi_kernel<<<grid, 256, smem, s>>>(d_points, P, C, pack, d_cams, d_uv);
  MCBA_CUDA(cudaGetLastError());
  MCBA_CUDA(cudaStreamSynchronize(s));   // cams_big[] is a stack buffer
  MCBA_CUDA(cudaFreeAsync(d_cams, s));
  return MCBA_OK;
}

int mcba_embed_points(int device, void* stream, const double* d_poses, int64_t F, const double* d_obj, int N,
                      double* d_world) {
  if (!d_poses || !d_obj || !d_world || F < 0 || N < 0) { set_error("mcba_embed_points: bad arguments"); return MCBA_ERR_ARG; }
  MCBA_CUDA(cudaSetDevice(device));
  if (F * N == 0) return MCBA_OK;
  const int grid = (int)std::min<long long>((F * N + 255) / 256, 148 * 16);
  embed_points_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_poses, F, d_obj, N, d_world);
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

static void fill_intrinsics(TriCam& cam, const double* Kc, const double* d) {
  cam.fx = Kc[0]; cam.skew = Kc[1]; cam.cx = Kc[2]; cam.fy = Kc[4]; cam.cy = Kc[5];
  cam.k1 = d[0]; cam.k2 = d[1]; cam.p1 = d[2]; cam.p2 = d[3]; cam.k3 = d[4];
}

int mcba_undistort_points(int device, void* stream, const double* d_in, int64_t P, const double* K,
                          const double* dist, double* d_out) {
  if (!d_in || !K || !dist || !d_out || P < 0) { set_error("mcba_undistort_points: bad arguments"); return MCBA_ERR_ARG; }
  MCBA_CUDA(cudaSetDevice(device));
  if (P == 0) return MCBA_OK;
  TriCam cam{};
  fill_intrinsics(cam, K, dist);
  const int grid = (int)std::min<long long>((P + 255) / 256, 148 * 16);
  undistort_points_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const double2*>(d_in), P, cam,
                                                                 reinterpret_cast<double2*>(d_out));
  MCBA_CUDA(cudaGetLastError());
  return MCBA_OK;
}

int mcba_triangulate(int device, void* stream, const double* d_uvs, int C, int64_t P, const double* ext,
                     const double* K, const double* dist, double* d_points) {
  if (!d_uvs || !ext || !K || !dist || !d_points || C < 1 || C > 32 || P < 0) {
    set_error("mcba_triangulate: bad arguments (1 <= n_cameras <= 32)");
    return MCBA_ERR_ARG;
  }
  MCBA_CUDA(cudaSetDevice(device));
  if (P == 0) return MCBA_OK;
  TriCam cams[32];
  for (int c = 0; c < C; ++c) {
    double R[9];
    host_rodrigues(ext + 6 * c, R);
    const double* Kc = K + 9 * c;
    double T[12];
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) T[4 * i + j] = R[3 * i + j];
      T[4 * i + 3] = ext[6 * c + 3 + i];
    }
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 4; ++j)
        cams[c].P[4 * i + j] = Kc[3 * i] * T[j] + Kc[3 * i + 1] * T[4 + j] + Kc[3 * i + 2] * T[8 + j];
    fill_intrinsics(cams[c], Kc, dist + 5 * c);
  }
  TriCam* d_cams = nullptr;
  cudaStream_t s = (cudaStream_t)stream;
  MCBA_CUDA(cudaMallocAsync((void**)&d_cams, sizeof(TriCam) * C, s));
  MCBA_CUDA(cudaMemcpyAsync(d_cams, cams, sizeof(TriCam) * C, cudaMemcpyHostToDevice, s));
  const int grid = (int)std::min<long long>((P + 127) / 128, 148 * 16);
  const size_t smem = sizeof(TriCam) * C;
  if (C <= 8) triangulate_kernel<8><<<grid, 128, smem, s>>>(d_uvs, C, P, d_cams, d_points);
  else triangulate_kernel<32><<<grid, 128, smem, s>>>(d_uvs, C, P, d_cams, d_points);
  MCBA_CUDA(cudaGetLastError());
  MCBA_CUDA(cudaStreamSynchronize(s));   // cams[] is a stack buffer
  MCBA_CUDA(cudaFreeAsync(d_cams, s));
  return MCBA_OK;
}

}  // extern "C"

// ---------------------------------------------------------------- FP64 pipe peak (bench.py roofline denominator)
// Dependent-chain-free DFMA loop, 16 independent accumulators per thread, 16 warps per SM:
// the same measurement as scripts/ubench/fp64_pipes.cu (mode 0), taken live on the device the
// benchmark runs on.  Returns fused multiply-adds per second.
namespace mcba {
__global__ void __launch_bounds__(512) fp64_peak_kernel(double* out, int iters, double seed) {
  double a[16];
  const double x = seed, y = 1.0 - 1e-9;
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = seed + i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = fma(a[i], y, x);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += a[i];
  if (s == 12345.678) *out = s;
}
}  // namespace mcba

extern "C" int mcba_measure_fp64_peak(int device, double* fma_per_s) {
  using namespace mcba;
  if (!fma_per_s) return MCBA_ERR_ARG;
  MCBA_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  MCBA_CUDA(cudaGetDeviceProperties(&prop, device));
  double* d = nullptr;
  MCBA_CUDA(cudaMalloc(&d, 8));
  cudaEvent_t e0, e1;
  MCBA_CUDA(cudaEventCreate(&e0));
  MCBA_CUDA(cudaEventCreate(&e1));
  const int iters = 20000, grid = prop.multiProcessorCount;
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    MCBA_CUDA(cudaEventRecord(e0));
    fp64_peak_kernel<<<grid, 512>>>(d, iters, 0.5);
    MCBA_CUDA(cudaEventRecord(e1));
    MCBA_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    MCBA_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double rate = (double)grid * 512 * 16 * (double)iters / (ms * 1e-3);
    if (rep > 0 && rate > best) best = rate;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *fma_per_s = best;
  return MCBA_OK;
}
