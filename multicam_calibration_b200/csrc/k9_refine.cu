// geometry.refine_points: per-point Levenberg-Marquardt on the reprojection error of a triangulated
// point, with scipy's five robust losses, from the triangulation of k5_points.cu (or a given start).
// One thread per point, persistent grid-stride; the camera constants of the rig in shared memory.
//
// Model (the project_points / bundle-adjustment model, mcba_math.cuh):
//   X_c = R X + t ;  x = X_c/Z_c, y = Y_c/Z_c ;  d = 1 + k1 r^2 + k2 r^4
//   u = fx x d + skew y d + cx ;  v = fy y d + cy ;  residual f = observed - (u, v)
// Jacobian of (u, v) w.r.t. X: G R, G = d(u|v)/dX_c (the BA's d/dtau chain, DESIGN section 2).
// Per scalar residual, z = (f / f_scale)^2, cost 0.5 f_scale^2 rho(z), gradient rho' f.  The iteration's
// Gauss-Newton weight is the IRLS majoriser rho' (every loss here is concave in z, so the weighted model
// bounds the cost from above and a step cannot stall on huber's kink or on the negative curvature of an
// outlier, where scipy's weight collapses to EPS); the covariance uses scipy's weight
// max(rho' + 2 rho'' z, EPS) (common.py:720-731), i.e. J~^T J~ of scipy's result.jac.  The fixed point
// does not depend on the weight.
#include <algorithm>
#include <cmath>
#include <vector>

#include "mcba_internal.h"

namespace mcba {

struct RefineCam {
  double R[9], t[3];
  double fx, fy, cx, cy, skew, k1, k2;   // projection (k1, k2 only)
  double p1, p2, k3;                     // rest of the 5-coefficient model: the triangulation's "seen" rule
};

constexpr double kRefEps = 2.220446049250313e-16;
constexpr double kLambda0 = 1e-4;     // damping relative to diag(H)
constexpr double kLambdaMin = 1e-12;
constexpr double kLambdaMax = 1e16;   // beyond this the step is below any representable change: give up

// scipy least_squares.py:183-219 on z >= 0: rho, rho', rho''
__device__ __forceinline__ void refine_rho(int loss, double z, double& r0, double& r1, double& r2) {
  switch (loss) {
    case MCBA_REFINE_LOSS_SOFT_L1: {
      const double t = 1.0 + z, s = sqrt(t);
      r0 = 2.0 * (s - 1.0);
      r1 = 1.0 / s;
      r2 = -0.5 * r1 / t;
      break;
    }
    case MCBA_REFINE_LOSS_HUBER:
      if (z <= 1.0) { r0 = z; r1 = 1.0; r2 = 0.0; }
      else { const double s = sqrt(z); r0 = 2.0 * s - 1.0; r1 = 1.0 / s; r2 = -0.5 * r1 / z; }
      break;
    case MCBA_REFINE_LOSS_CAUCHY: {
      const double t = 1.0 + z;
      r0 = log1p(z);
      r1 = 1.0 / t;
      r2 = -r1 * r1;
      break;
    }
    case MCBA_REFINE_LOSS_ARCTAN: {
      const double t = 1.0 + z * z;
      r0 = atan(z);
      r1 = 1.0 / t;
      r2 = -2.0 * z * r1 * r1;
      break;
    }
    default: r0 = z; r1 = 1.0; r2 = 0.0;
  }
}

// Projection of X into camera c; residual f = o - uv.  With kJac, P = G R (2x3, row major).
template <bool kJac>
__device__ __forceinline__ void refine_project(const RefineCam& k, const double X[3], double2 o, double& fu, double& fv,
                                               double P[6]) {
  double Xc[3];
  mat3_vec(k.R, X, Xc);
  Xc[0] += k.t[0]; Xc[1] += k.t[1]; Xc[2] += k.t[2];
  const double iz = 1.0 / Xc[2];
  const double xn = Xc[0] * iz, yn = Xc[1] * iz;
  const double r2 = xn * xn + yn * yn;
  const double d = 1.0 + r2 * (k.k1 + k.k2 * r2);
  const double xd = xn * d, yd = yn * d;
  fu = o.x - (k.fx * xd + k.skew * yd + k.cx);
  fv = o.y - (k.fy * yd + k.cy);
  if (kJac) {
    const double dd = 2.0 * (k.k1 + 2.0 * k.k2 * r2);
    const double dxx = d + dd * xn * xn, dxy = dd * xn * yn, dyy = d + dd * yn * yn;
    // A = d(u,v)/d(x,y); G = A [1 0 -x; 0 1 -y] / Z
    const double a11 = (k.fx * dxx + k.skew * dxy) * iz, a12 = (k.fx * dxy + k.skew * dyy) * iz;
    const double a21 = k.fy * dxy * iz, a22 = k.fy * dyy * iz;
    const double G[6] = {a11, a12, -(a11 * xn + a12 * yn), a21, a22, -(a21 * xn + a22 * yn)};
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        P[3 * i + j] = G[3 * i] * k.R[j] + G[3 * i + 1] * k.R[3 + j] + G[3 * i + 2] * k.R[6 + j];
  }
}

struct RefineLoss {
  int loss;
  double inv_fs, fs2;
};

// One scalar residual f with projection-Jacobian row p: cost, gradient of the cost (d f / dX = -p) and
// the weighted normal matrix (upper triangle xx xy xz yy yz zz), weight rho' or, with kTriggs, scipy's.
template <bool kJac, bool kTriggs = false>
__device__ __forceinline__ void refine_scalar(const RefineLoss& L, double f, const double* p, double& cost,
                                              double H[6], double g[3]) {
  double r1 = 1.0, w = 1.0;
  if (L.loss == MCBA_REFINE_LOSS_LINEAR) {
    cost += 0.5 * f * f;
  } else {
    const double fs = f * L.inv_fs, z = fs * fs;
    double r0, r2;
    refine_rho(L.loss, z, r0, r1, r2);
    cost += 0.5 * L.fs2 * r0;
    w = kTriggs ? fmax(r1 + 2.0 * r2 * z, kRefEps) : r1;
  }
  if (kJac) {
    const double gf = -r1 * f;
    g[0] = fma(gf, p[0], g[0]); g[1] = fma(gf, p[1], g[1]); g[2] = fma(gf, p[2], g[2]);
    const double w0 = w * p[0], w1 = w * p[1];
    H[0] = fma(w0, p[0], H[0]); H[1] = fma(w0, p[1], H[1]); H[2] = fma(w0, p[2], H[2]);
    H[3] = fma(w1, p[1], H[3]); H[4] = fma(w1, p[2], H[4]); H[5] = fma(w * p[2], p[2], H[5]);
  }
}

// Cholesky of the 3x3 upper-triangle S (xx xy xz yy yz zz), in place as L (l00 l10 l20 l11 l21 l22).
// False for a non-positive or non-finite pivot.
__device__ __forceinline__ bool chol3(double S[6]) {
  if (!(S[0] > 0.0) || !(S[0] < INFINITY)) return false;
  const double l00 = sqrt(S[0]), l10 = S[1] / l00, l20 = S[2] / l00;
  const double d1 = S[3] - l10 * l10;
  if (!(d1 > 0.0) || !(d1 < INFINITY)) return false;
  const double l11 = sqrt(d1), l21 = (S[4] - l20 * l10) / l11;
  const double d2 = S[5] - l20 * l20 - l21 * l21;
  if (!(d2 > 0.0) || !(d2 < INFINITY)) return false;
  S[0] = l00; S[1] = l10; S[2] = l20; S[3] = l11; S[4] = l21; S[5] = sqrt(d2);
  return true;
}

__device__ __forceinline__ void chol3_solve(const double L[6], const double b[3], double x[3]) {
  const double y0 = b[0] / L[0];
  const double y1 = (b[1] - L[1] * y0) / L[3];
  const double y2 = (b[2] - L[2] * y0 - L[4] * y1) / L[5];
  x[2] = y2 / L[5];
  x[1] = (y1 - L[4] * x[2]) / L[3];
  x[0] = (y0 - L[1] * x[1] - L[2] * x[2]) / L[0];
}

// Observations of a point: registers for up to eight cameras (the loops below unroll over kMaxC), global
// memory (L1 / L2) beyond.
template <int kMaxC>
struct RefineObs {
  static constexpr bool kRegs = kMaxC <= 8;
  double2 r[kRegs ? kMaxC : 1];
  const double2* g;
  long long P, pt;
  __device__ __forceinline__ double2 operator[](int c) const {
    if constexpr (kRegs) return r[c];
    else return g[(long long)c * P + pt];
  }
};

// cost (and with kJac the normal matrix and gradient) of a point over its seen views
template <int kMaxC, bool kJac>
__device__ __forceinline__ double refine_eval(const RefineCam* sc, int C, unsigned seen, const RefineObs<kMaxC>& ob,
                                              const RefineLoss& L, const double X[3], double H[6], double g[3]) {
  double cost = 0.0;
  if (kJac) {
#pragma unroll
    for (int i = 0; i < 6; ++i) H[i] = 0.0;
    g[0] = g[1] = g[2] = 0.0;
  }
#pragma unroll(kMaxC <= 8 ? kMaxC : 1)
  for (int c = 0; c < kMaxC; ++c) {
    if (c >= C || !((seen >> c) & 1u)) continue;
    double fu, fv, P[6];
    refine_project<kJac>(sc[c], X, ob[c], fu, fv, P);
    refine_scalar<kJac>(L, fu, P, cost, H, g);
    refine_scalar<kJac>(L, fv, P + 3, cost, H, g);
  }
  return cost;
}

// (128, 3): without the occupancy hint ptxas holds refine_points_kernel<8> to 128 registers and spills;
// with it, 136 registers and no spills (the observations of eight views stay in registers)
template <int kMaxC>
__global__ void __launch_bounds__(128, 3) refine_points_kernel(const double* __restrict__ uvs, int C, long long P,
                                                            const RefineCam* __restrict__ cams, const double* init,
                                                            mcba_refine_options opt, double* points,
                                                            double* __restrict__ out_cost, double* __restrict__ out_rms,
                                                            int8_t* __restrict__ out_status,
                                                            int16_t* __restrict__ out_iters, double* __restrict__ out_cov,
                                                            double* __restrict__ out_view_err,
                                                            int8_t* __restrict__ out_n_views) {
  extern __shared__ unsigned char rf_smem[];
  RefineCam* sc = reinterpret_cast<RefineCam*>(rf_smem);
  for (int i = threadIdx.x; i < C * (int)(sizeof(RefineCam) / sizeof(double)); i += blockDim.x)
    reinterpret_cast<double*>(sc)[i] = reinterpret_cast<const double*>(cams)[i];
  __syncthreads();
  const RefineLoss L{opt.loss, 1.0 / opt.f_scale, opt.f_scale * opt.f_scale};
  const double nan_ = nan("");
  for (long long pt = blockIdx.x * (long long)blockDim.x + threadIdx.x; pt < P; pt += (long long)gridDim.x * blockDim.x) {
    RefineObs<kMaxC> ob;
    ob.g = reinterpret_cast<const double2*>(uvs);
    ob.P = P;
    ob.pt = pt;
    // seen: the undistorted pixel is finite, as triangulate_kernel decides it (k5_points.cu)
    unsigned seen = 0;
    int n_views = 0;
#pragma unroll(kMaxC <= 8 ? kMaxC : 1)
    for (int c = 0; c < kMaxC; ++c) {
      if (c >= C) continue;
      const double2 o = ob.g[(long long)c * P + pt];
      if constexpr (RefineObs<kMaxC>::kRegs) ob.r[c] = o;
      const RefineCam& k = sc[c];
      const double x0 = (o.x - k.cx) / k.fx, y0 = (o.y - k.cy) / k.fy;
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
      const double uo = x * k.fx + y * k.skew + k.cx, vo = y * k.fy + k.cy;
      if (uo == uo && vo == vo) { seen |= 1u << c; ++n_views; }
    }
    const double X0[3] = {init[3 * pt], init[3 * pt + 1], init[3 * pt + 2]};
    double X[3] = {X0[0], X0[1], X0[2]};
    int status = 0, iters = 0;
    double H[6], g[3];
    if (n_views < 2) {
      status = -1;
      X[0] = X[1] = X[2] = nan_;
    } else {
      double cost = nan_;
      if (isfinite(X0[0]) && isfinite(X0[1]) && isfinite(X0[2]))
        cost = refine_eval<kMaxC, true>(sc, C, seen, ob, L, X, H, g);
      if (!isfinite(cost)) {
        status = -2;
      } else {
        double lambda = kLambda0;
        // scipy trf (trf.py, no bounds) decisions per point: gtol before every step, ftol / xtol after every
        // trial with a finite cost; an accepted step moves x even when it also ends the iteration
        for (;;) {
          if (fmax(fmax(fabs(g[0]), fabs(g[1])), fabs(g[2])) < opt.gtol) { status = 1; break; }
          if (iters >= opt.max_iter) { status = 0; break; }
          ++iters;
          double A[6] = {H[0] * (1.0 + lambda), H[1], H[2], H[3] * (1.0 + lambda), H[4], H[5] * (1.0 + lambda)};
          bool accepted = false;
          int term = 0;
          if (chol3(A)) {
            double dx[3];
            const double mg[3] = {-g[0], -g[1], -g[2]};
            chol3_solve(A, mg, dx);
            const double Xn[3] = {X[0] + dx[0], X[1] + dx[1], X[2] + dx[2]};
            const double cost_new = refine_eval<kMaxC, false>(sc, C, seen, ob, L, Xn, nullptr, nullptr);
            if (isfinite(cost_new)) {
              // predicted reduction -(g.dx + dx^T H dx / 2) of the undamped model
              const double Hd0 = H[0] * dx[0] + H[1] * dx[1] + H[2] * dx[2];
              const double Hd1 = H[1] * dx[0] + H[3] * dx[1] + H[4] * dx[2];
              const double Hd2 = H[2] * dx[0] + H[4] * dx[1] + H[5] * dx[2];
              const double pred = -(g[0] * dx[0] + g[1] * dx[1] + g[2] * dx[2]) -
                                  0.5 * (dx[0] * Hd0 + dx[1] * Hd1 + dx[2] * Hd2);
              const double dF = cost - cost_new;
              const double ratio = pred > 0.0 ? dF / pred : (pred == 0.0 && dF == 0.0 ? 1.0 : 0.0);
              const double dx_norm = sqrt(dx[0] * dx[0] + dx[1] * dx[1] + dx[2] * dx[2]);
              const double x_norm = sqrt(X[0] * X[0] + X[1] * X[1] + X[2] * X[2]);
              const bool ftol_ok = dF < opt.ftol * cost && ratio > 0.25;
              const bool xtol_ok = dx_norm < opt.xtol * (opt.xtol + x_norm);
              term = ftol_ok && xtol_ok ? 4 : ftol_ok ? 2 : xtol_ok ? 3 : 0;
              if (dF > 0.0) {
                accepted = true;
                X[0] = Xn[0]; X[1] = Xn[1]; X[2] = Xn[2];
                cost = cost_new;
              }
            }
          }
          if (term) { status = term; break; }
          if (accepted) {
            lambda = fmax(lambda * 0.1, kLambdaMin);
            cost = refine_eval<kMaxC, true>(sc, C, seen, ob, L, X, H, g);
          } else {
            lambda *= 10.0;
            if (lambda > kLambdaMax) { status = -2; break; }
          }
        }
        if (status == -2) { X[0] = X0[0]; X[1] = X0[1]; X[2] = X0[2]; }
      }
    }
    // closing pass at the returned point: cost, RMS, per-view distances, J~^T J~ for the covariance
    double cost = nan_, sumsq = 0.0;
    const bool have = status != -1 && isfinite(X[0]) && isfinite(X[1]) && isfinite(X[2]);
    if (have) {
      cost = 0.0;
#pragma unroll
      for (int i = 0; i < 6; ++i) H[i] = 0.0;
      g[0] = g[1] = g[2] = 0.0;
    }
#pragma unroll(kMaxC <= 8 ? kMaxC : 1)
    for (int c = 0; c < kMaxC; ++c) {
      if (c >= C) continue;
      double e = nan_;
      if (have && ((seen >> c) & 1u)) {
        double fu, fv, Pj[6];
        refine_project<true>(sc[c], X, ob[c], fu, fv, Pj);
        refine_scalar<true, true>(L, fu, Pj, cost, H, g);
        refine_scalar<true, true>(L, fv, Pj + 3, cost, H, g);
        const double s2 = fu * fu + fv * fv;
        sumsq += s2;
        e = sqrt(s2);
      }
      if (out_view_err) out_view_err[(long long)c * P + pt] = e;
    }
    points[3 * pt] = X[0];
    points[3 * pt + 1] = X[1];
    points[3 * pt + 2] = X[2];
    out_cost[pt] = cost;
    out_rms[pt] = have ? sqrt(sumsq / (2.0 * n_views)) : nan_;
    out_status[pt] = (int8_t)status;
    out_iters[pt] = (int16_t)iters;
    if (out_n_views) out_n_views[pt] = (int8_t)n_views;
    if (out_cov) {
      double cv[6] = {nan_, nan_, nan_, nan_, nan_, nan_};
      if (have && chol3(H)) {
        // inverse of L L^T: columns of L^-T L^-1
        const double s2 = opt.sigma * opt.sigma;
        double e0[3], e1[3], e2[3];
        const double u0[3] = {1.0, 0.0, 0.0}, u1[3] = {0.0, 1.0, 0.0}, u2[3] = {0.0, 0.0, 1.0};
        chol3_solve(H, u0, e0);
        chol3_solve(H, u1, e1);
        chol3_solve(H, u2, e2);
        cv[0] = s2 * e0[0]; cv[1] = s2 * e1[0]; cv[2] = s2 * e2[0];
        cv[3] = s2 * e1[1]; cv[4] = s2 * e2[1]; cv[5] = s2 * e2[2];
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) out_cov[6 * pt + i] = cv[i];
    }
  }
}

// ------------------------------------------------------------------ covariance.point_covariance
// Calibration uncertainty carried into a point X: with J~ scaled as the covariance above (scipy's weight w),
//   H = sum_seen w P^T P,  S_c = -H^-1 sum_{u,v} w P^T J_c  (3 x 12, dX / d theta_c),
//   calibration = sum_{c,d seen} S_c cov[c,d] S_d^T,  measurement = sigma^2 H^-1.
// J_c, the prediction's Jacobian w.r.t. camera c's serialize_params block (fx fy cx cy k1 k2 rvec tvec):
//   d(u,v)/d(fx, fy, cx, cy) = [x d, 0, 1, 0; 0, y d, 0, 1], d/d(k1, k2) = (fx x + skew y, fy y) (r^2, r^4),
//   d/d rvec = G d(R X)/d rvec = -P [X]x Jr, d/d tvec = G = P R^T   (Jr: right Jacobian of the rotation vector).
// A warp takes 32 points: lane i computes point i's H in the order of the closing pass of refine_points_kernel
// (measurement bit-identical to its d_cov), then batches of kPcQ points form S (lane per point and camera) in
// shared memory and the product T = S cov with lanes over cov's columns, kPcQ x 3 rows x kPcCols columns of T per
// lane, and T S^T by a warp reduction.  cov in shared memory up to eight cameras, read through L1 / L2 beyond.
struct PointCovCam {
  RefineCam k;
  double Jr[9];
  double pad_;   // 32 doubles: the per-warp buffers behind the cameras stay 16-byte aligned
};
struct PointCovNan {
  unsigned pair[32];   // bit d of pair[c]: block (c, d) of the camera covariance holds a non-finite entry
};

constexpr int kPcQ = 4;      // points per product batch
constexpr int kPcCols = 3;   // columns of cov per lane per pass: passes of 96 columns
template <int kMaxC>
struct PointCovShape {
  static constexpr bool kSmemCov = kMaxC <= 8;
  static constexpr int kWarps = kMaxC <= 8 ? 8 : 4;
  // per warp: S of a batch (12C rows x kPcQ points x 3), the Cholesky factors of H (32 x 6), seen masks and flags
  __host__ __device__ static size_t warp_doubles(int C) { return (size_t)12 * C * 3 * kPcQ + 32 * 6 + 32; }
  static size_t smem(int C) {
    return sizeof(double) * ((size_t)C * (sizeof(PointCovCam) / sizeof(double)) + (kSmemCov ? (size_t)144 * C * C : 0) +
                             kWarps * warp_doubles(C));
  }
};

// the "seen" rule of refine_points_kernel (the pixel undistorts to a finite point, as k5_points.cu decides it)
__device__ __forceinline__ bool point_cov_seen(const RefineCam& k, double2 o) {
  const double x0 = (o.x - k.cx) / k.fx, y0 = (o.y - k.cy) / k.fy;
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
  const double uo = x * k.fx + y * k.skew + k.cx, vo = y * k.fy + k.cy;
  return uo == uo && vo == vo;
}

// scipy's weight of one scalar residual, as refine_scalar<true, true> applies it
__device__ __forceinline__ double point_cov_weight(const RefineLoss& L, double f) {
  if (L.loss == MCBA_REFINE_LOSS_LINEAR) return 1.0;
  const double fs = f * L.inv_fs, z = fs * fs;
  double r0, r1, r2;
  refine_rho(L.loss, z, r0, r1, r2);
  return fmax(r1 + 2.0 * r2 * z, kRefEps);
}

// Rows of J_c for u and v at X (P = G R from refine_project)
__device__ __forceinline__ void point_cov_camera_rows(const PointCovCam& cam, const double X[3], const double P[6],
                                                      double Ju[12], double Jv[12]) {
  const RefineCam& k = cam.k;
  double Xc[3];
  mat3_vec(k.R, X, Xc);
  Xc[0] += k.t[0]; Xc[1] += k.t[1]; Xc[2] += k.t[2];
  const double iz = 1.0 / Xc[2];
  const double xn = Xc[0] * iz, yn = Xc[1] * iz;
  const double r2 = xn * xn + yn * yn, r4 = r2 * r2;
  const double d = 1.0 + r2 * (k.k1 + k.k2 * r2);
  const double au = k.fx * xn + k.skew * yn, av = k.fy * yn;
  Ju[0] = xn * d; Ju[1] = 0.0; Ju[2] = 1.0; Ju[3] = 0.0; Ju[4] = au * r2; Ju[5] = au * r4;
  Jv[0] = 0.0; Jv[1] = yn * d; Jv[2] = 0.0; Jv[3] = 1.0; Jv[4] = av * r2; Jv[5] = av * r4;
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const double* p = P + 3 * s;
    double* J = s ? Jv : Ju;
    // -p [X]x = (X x p)^T, then times Jr
    const double q0 = X[1] * p[2] - X[2] * p[1], q1 = X[2] * p[0] - X[0] * p[2], q2 = X[0] * p[1] - X[1] * p[0];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      J[6 + j] = q0 * cam.Jr[j] + q1 * cam.Jr[3 + j] + q2 * cam.Jr[6 + j];
      J[9 + j] = p[0] * k.R[3 * j] + p[1] * k.R[3 * j + 1] + p[2] * k.R[3 * j + 2];
    }
  }
}

template <int kMaxC>
__global__ void __launch_bounds__(32 * PointCovShape<kMaxC>::kWarps)
    point_covariance_kernel(const double* __restrict__ uvs, int C, long long P, const PointCovCam* __restrict__ cams,
                            const double* __restrict__ points, const double* __restrict__ cam_cov, PointCovNan nanp,
                            RefineLoss L, double sigma, double* __restrict__ out_meas, double* __restrict__ out_cal,
                            double* __restrict__ out_sens) {
  using Shape = PointCovShape<kMaxC>;
  extern __shared__ __align__(16) double pc_smem[];
  const int n = 12 * C;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  PointCovCam* sc = reinterpret_cast<PointCovCam*>(pc_smem);
  double* scov = pc_smem + C * (sizeof(PointCovCam) / sizeof(double));
  for (int i = threadIdx.x; i < C * (int)(sizeof(PointCovCam) / sizeof(double)); i += blockDim.x)
    pc_smem[i] = reinterpret_cast<const double*>(cams)[i];
  if constexpr (Shape::kSmemCov)
    for (int i = threadIdx.x; i < n * n; i += blockDim.x) scov[i] = cam_cov[i];
  const double* cov = Shape::kSmemCov ? scov : cam_cov;
  double* Sb = scov + (Shape::kSmemCov ? n * n : 0) + warp * Shape::warp_doubles(C);
  double* Lb = Sb + n * 3 * kPcQ;
  unsigned* seen_b = reinterpret_cast<unsigned*>(Lb + 32 * 6);
  unsigned* flag_b = seen_b + 32;   // bit 0: H positive definite (S defined), bit 1: no non-finite covariance block
  __syncthreads();
  const double nan_ = nan("");
  const long long n_groups = (P + 31) / 32;
  for (long long grp = blockIdx.x * (long long)Shape::kWarps + warp; grp < n_groups;
       grp += (long long)gridDim.x * Shape::kWarps) {
    const long long base = grp * 32;
    // lane -> point: seen views, H as the closing pass of refine_points_kernel, the measurement part
    {
      const long long pt = base + lane;
      unsigned seen = 0, flags = 0;
      double H[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      if (pt < P) {
        int n_views = 0;
        const double2* o = reinterpret_cast<const double2*>(uvs);
        for (int c = 0; c < C; ++c)
          if (point_cov_seen(sc[c].k, o[(long long)c * P + pt])) { seen |= 1u << c; ++n_views; }
        const double X[3] = {points[3 * pt], points[3 * pt + 1], points[3 * pt + 2]};
        const bool have = n_views >= 2 && isfinite(X[0]) && isfinite(X[1]) && isfinite(X[2]);
        double cv[6] = {nan_, nan_, nan_, nan_, nan_, nan_};
        if (have) {
          double cost = 0.0, g[3] = {0.0, 0.0, 0.0};
          for (int c = 0; c < C; ++c) {
            if (!((seen >> c) & 1u)) continue;
            double fu, fv, Pj[6];
            refine_project<true>(sc[c].k, X, o[(long long)c * P + pt], fu, fv, Pj);
            refine_scalar<true, true>(L, fu, Pj, cost, H, g);
            refine_scalar<true, true>(L, fv, Pj + 3, cost, H, g);
          }
          if (chol3(H)) {
            const double s2 = sigma * sigma;
            double e0[3], e1[3], e2[3];
            const double u0[3] = {1.0, 0.0, 0.0}, u1[3] = {0.0, 1.0, 0.0}, u2[3] = {0.0, 0.0, 1.0};
            chol3_solve(H, u0, e0);
            chol3_solve(H, u1, e1);
            chol3_solve(H, u2, e2);
            cv[0] = s2 * e0[0]; cv[1] = s2 * e1[0]; cv[2] = s2 * e2[0];
            cv[3] = s2 * e1[1]; cv[4] = s2 * e2[1]; cv[5] = s2 * e2[2];
            flags = 1u;
            bool finite_cov = true;
            for (int c = 0; c < C; ++c)
              if (((seen >> c) & 1u) && (nanp.pair[c] & seen)) finite_cov = false;
            if (finite_cov) flags |= 2u;
          }
        }
        if (out_meas)
#pragma unroll
          for (int i = 0; i < 6; ++i) out_meas[6 * pt + i] = cv[i];
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) Lb[6 * lane + i] = H[i];
      seen_b[lane] = seen;
      flag_b[lane] = flags;
    }
    __syncwarp();
    for (int b = 0; b < 32 / kPcQ; ++b) {
      const long long p0 = base + b * kPcQ;
      if (p0 >= P) break;
      // S of the batch, lane -> (point, camera); zero for an unseen camera or an undefined point
      for (int idx = lane; idx < kPcQ * C; idx += 32) {
        const int p = idx / C, c = idx - p * C, l = b * kPcQ + p;
        double* Sc = Sb + 12 * c * 3 * kPcQ + 3 * p;
        if ((flag_b[l] & 1u) && ((seen_b[l] >> c) & 1u)) {
          const long long pt = p0 + p;
          const double X[3] = {points[3 * pt], points[3 * pt + 1], points[3 * pt + 2]};
          double fu, fv, Pj[6], Ju[12], Jv[12];
          refine_project<true>(sc[c].k, X, reinterpret_cast<const double2*>(uvs)[(long long)c * P + pt], fu, fv, Pj);
          point_cov_camera_rows(sc[c], X, Pj, Ju, Jv);
          const double wu = point_cov_weight(L, fu), wv = point_cov_weight(L, fv);
          const double* Lh = Lb + 6 * l;
#pragma unroll
          for (int j = 0; j < 12; ++j) {
            const double m[3] = {-(wu * Ju[j] * Pj[0] + wv * Jv[j] * Pj[3]), -(wu * Ju[j] * Pj[1] + wv * Jv[j] * Pj[4]),
                                 -(wu * Ju[j] * Pj[2] + wv * Jv[j] * Pj[5])};
            double s[3];
            chol3_solve(Lh, m, s);
            Sc[j * 3 * kPcQ] = s[0]; Sc[j * 3 * kPcQ + 1] = s[1]; Sc[j * 3 * kPcQ + 2] = s[2];
          }
        } else {
#pragma unroll
          for (int j = 0; j < 12; ++j) Sc[j * 3 * kPcQ] = Sc[j * 3 * kPcQ + 1] = Sc[j * 3 * kPcQ + 2] = 0.0;
        }
      }
      __syncwarp();
      unsigned wseen = 0;
#pragma unroll
      for (int p = 0; p < kPcQ; ++p) {
        const int l = b * kPcQ + p;
        if (flag_b[l] & 1u) wseen |= seen_b[l];
        if (out_sens && p0 + p < P) {
          double* dst = out_sens + (p0 + p) * 3 * n;
          const bool ok = flag_b[l] & 1u;
          for (int e = lane; e < 3 * n; e += 32) {
            const int a = e / n, j = e - a * n;
            dst[e] = ok ? Sb[j * 3 * kPcQ + 3 * p + a] : nan_;
          }
        }
      }
      // T = S cov over the seen rows of the batch, then T S^T: upper triangle xx xy xz yy yz zz per point
      double part[kPcQ][6];
#pragma unroll
      for (int p = 0; p < kPcQ; ++p)
#pragma unroll
        for (int e = 0; e < 6; ++e) part[p][e] = 0.0;
      for (int j0 = 0; j0 < n; j0 += 32 * kPcCols) {
        double acc[3 * kPcQ][kPcCols];
#pragma unroll
        for (int r = 0; r < 3 * kPcQ; ++r)
#pragma unroll
          for (int k = 0; k < kPcCols; ++k) acc[r][k] = 0.0;
        for (int c = 0; c < C; ++c) {
          if (!((wseen >> c) & 1u)) continue;
#pragma unroll 4
          for (int q = 0; q < 12; ++q) {
            const int i = 12 * c + q;
            const double2* srow = reinterpret_cast<const double2*>(Sb + i * 3 * kPcQ);
            double s[3 * kPcQ];
#pragma unroll
            for (int h = 0; h < 3 * kPcQ / 2; ++h) {
              const double2 v = srow[h];
              s[2 * h] = v.x; s[2 * h + 1] = v.y;
            }
            double sig[kPcCols];
#pragma unroll
            for (int k = 0; k < kPcCols; ++k) {
              const int j = j0 + lane + 32 * k;
              sig[k] = j < n ? (Shape::kSmemCov ? cov[i * n + j] : __ldg(cov + (size_t)i * n + j)) : 0.0;
            }
#pragma unroll
            for (int r = 0; r < 3 * kPcQ; ++r)
#pragma unroll
              for (int k = 0; k < kPcCols; ++k) acc[r][k] = fma(s[r], sig[k], acc[r][k]);
          }
        }
#pragma unroll
        for (int k = 0; k < kPcCols; ++k) {
          const int j = j0 + lane + 32 * k;
          if (j >= n) continue;
          const double* sj = Sb + j * 3 * kPcQ;
#pragma unroll
          for (int p = 0; p < kPcQ; ++p) {
            const double* t = acc[3 * p] ;
            const double t0 = t[k], t1 = acc[3 * p + 1][k], t2 = acc[3 * p + 2][k];
            const double s0 = sj[3 * p], s1 = sj[3 * p + 1], s2 = sj[3 * p + 2];
            part[p][0] = fma(t0, s0, part[p][0]); part[p][1] = fma(t0, s1, part[p][1]);
            part[p][2] = fma(t0, s2, part[p][2]); part[p][3] = fma(t1, s1, part[p][3]);
            part[p][4] = fma(t1, s2, part[p][4]); part[p][5] = fma(t2, s2, part[p][5]);
          }
        }
      }
#pragma unroll
      for (int p = 0; p < kPcQ; ++p)
#pragma unroll
        for (int e = 0; e < 6; ++e) {
          double v = part[p][e];
#pragma unroll
          for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
          part[p][e] = v;
        }
#pragma unroll
      for (int p = 0; p < kPcQ; ++p)
        if (lane == p && p0 + p < P) {
          const bool ok = (flag_b[b * kPcQ + p] & 3u) == 3u;
#pragma unroll
          for (int e = 0; e < 6; ++e) out_cal[6 * (p0 + p) + e] = ok ? part[p][e] : nan_;
        }
      __syncwarp();
    }
  }
}

}  // namespace mcba

using namespace mcba;

extern "C" int mcba_refine_points(int device, void* stream, const double* d_uvs, int C, int64_t P, const double* ext,
                                  const double* K, const double* dist, const double* d_init,
                                  const mcba_refine_options* opt, double* d_points, double* d_cost, double* d_rms,
                                  int8_t* d_status, int16_t* d_iters, double* d_cov, double* d_view_err,
                                  int8_t* d_n_views) {
  if (!d_uvs || !ext || !K || !dist || !opt || !d_points || !d_cost || !d_rms || !d_status || !d_iters || C < 1 ||
      C > 32 || P < 0) {
    set_error("mcba_refine_points: bad arguments (1 <= n_cameras <= 32)");
    return MCBA_ERR_ARG;
  }
  if (opt->loss < MCBA_REFINE_LOSS_LINEAR || opt->loss > MCBA_REFINE_LOSS_ARCTAN || !(opt->f_scale > 0.0) ||
      !(opt->f_scale < INFINITY) || !(opt->sigma > 0.0) || !(opt->sigma < INFINITY) || !(opt->ftol >= 0.0) ||
      !(opt->xtol >= 0.0) || !(opt->gtol >= 0.0) || opt->max_iter < 1 || opt->max_iter > 32767 || opt->flags != 0) {
    set_error("mcba_refine_points: bad options (loss, f_scale > 0, sigma > 0, tolerances >= 0, "
              "1 <= max_iter <= 32767, flags = 0)");
    return MCBA_ERR_ARG;
  }
  MCBA_CUDA(cudaSetDevice(device));
  if (P == 0) return MCBA_OK;
  { int rc = keep_async_pool(device); if (rc) return rc; }
  cudaStream_t s = (cudaStream_t)stream;
  if (!d_init) {   // the start is triangulate's result, computed into d_points and refined in place
    const int rc = mcba_triangulate(device, stream, d_uvs, C, P, ext, K, dist, d_points);
    if (rc) return rc;
  }
  RefineCam cams[32];
  for (int c = 0; c < C; ++c) {
    host_rodrigues(ext + 6 * c, cams[c].R);
    for (int i = 0; i < 3; ++i) cams[c].t[i] = ext[6 * c + 3 + i];
    const double* Kc = K + 9 * c;
    const double* d = dist + 5 * c;
    cams[c].fx = Kc[0]; cams[c].skew = Kc[1]; cams[c].cx = Kc[2]; cams[c].fy = Kc[4]; cams[c].cy = Kc[5];
    cams[c].k1 = d[0]; cams[c].k2 = d[1]; cams[c].p1 = d[2]; cams[c].p2 = d[3]; cams[c].k3 = d[4];
  }
  RefineCam* d_cams = nullptr;
  MCBA_CUDA(cudaMallocAsync((void**)&d_cams, sizeof(RefineCam) * C, s));
  MCBA_CUDA(cudaMemcpyAsync(d_cams, cams, sizeof(RefineCam) * C, cudaMemcpyHostToDevice, s));
  const int grid = (int)std::min<long long>((P + 127) / 128, 148 * 16);
  const size_t smem = sizeof(RefineCam) * C;
  const double* init = d_init ? d_init : d_points;
  if (C <= 8)
    refine_points_kernel<8><<<grid, 128, smem, s>>>(d_uvs, C, P, d_cams, init, *opt, d_points, d_cost, d_rms, d_status,
                                                    d_iters, d_cov, d_view_err, d_n_views);
  else
    refine_points_kernel<32><<<grid, 128, smem, s>>>(d_uvs, C, P, d_cams, init, *opt, d_points, d_cost, d_rms,
                                                     d_status, d_iters, d_cov, d_view_err, d_n_views);
  const cudaError_t launch = cudaGetLastError();
  const cudaError_t sync = cudaStreamSynchronize(s);   // cams[] is a stack buffer
  cudaFreeAsync(d_cams, s);
  MCBA_CUDA(launch);
  MCBA_CUDA(sync);
  return MCBA_OK;
}

// Right Jacobian of the rotation vector, oracle/np_oracle.py so3_right_jacobian
static void host_so3_right_jacobian(const double r[3], double J[9]) {
  const double th2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2], th = std::sqrt(th2);
  const double a = th < 1e-4 ? 0.5 - th2 / 24.0 : (1.0 - std::cos(th)) / th2;
  const double b = th < 1e-4 ? 1.0 / 6.0 - th2 / 120.0 : (th - std::sin(th)) / (th2 * th);
  const double S[9] = {0.0, -r[2], r[1], r[2], 0.0, -r[0], -r[1], r[0], 0.0};
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double SS = 0.0;
      for (int k = 0; k < 3; ++k) SS += S[3 * i + k] * S[3 * k + j];
      J[3 * i + j] = (i == j ? 1.0 : 0.0) - a * S[3 * i + j] + b * SS;
    }
}

template <int kMaxC>
static int launch_point_covariance(cudaStream_t s, const double* d_uvs, int C, int64_t P, const PointCovCam* d_cams,
                                   const double* d_points, const double* d_cov, const PointCovNan& nanp,
                                   const RefineLoss& L, double sigma, double* d_meas, double* d_cal, double* d_sens) {
  using Shape = PointCovShape<kMaxC>;
  const size_t smem = Shape::smem(C);
  auto kernel = point_covariance_kernel<kMaxC>;
  MCBA_CUDA(set_dynamic_smem(reinterpret_cast<const void*>(kernel), smem));
  int device = 0, sms = 0, per_sm = 0;
  MCBA_CUDA(cudaGetDevice(&device));
  MCBA_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  MCBA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 32 * Shape::kWarps, smem));
  const long long groups = (P + 31) / 32;
  const int grid = (int)std::min<long long>((groups + Shape::kWarps - 1) / Shape::kWarps,
                                            (long long)sms * std::max(per_sm, 1));
  kernel<<<grid, 32 * Shape::kWarps, smem, s>>>(d_uvs, C, P, d_cams, d_points, d_cov, nanp, L, sigma, d_meas, d_cal,
                                                d_sens);
  return MCBA_OK;
}

extern "C" int mcba_point_covariance(int device, void* stream, const double* d_uvs, int C, int64_t P, const double* ext,
                                     const double* K, const double* dist, const double* d_points,
                                     const double* cam_cov, int loss, double f_scale, double sigma, double* d_cov_meas,
                                     double* d_cov_cal, double* d_sens) {
  if (!ext || !K || !dist || !cam_cov || C < 1 || C > 32 || P < 0 ||
      (P > 0 && (!d_uvs || !d_points || !d_cov_cal))) {
    set_error("mcba_point_covariance: bad arguments (1 <= n_cameras <= 32)");
    return MCBA_ERR_ARG;
  }
  if (loss < MCBA_REFINE_LOSS_LINEAR || loss > MCBA_REFINE_LOSS_ARCTAN || !(f_scale > 0.0) || !(f_scale < INFINITY) ||
      !(sigma > 0.0) || !(sigma < INFINITY)) {
    set_error("mcba_point_covariance: bad options (loss, f_scale > 0, sigma > 0)");
    return MCBA_ERR_ARG;
  }
  MCBA_CUDA(cudaSetDevice(device));
  if (P == 0) return MCBA_OK;
  { int rc = keep_async_pool(device); if (rc) return rc; }
  cudaStream_t s = (cudaStream_t)stream;
  PointCovCam cams[32];
  for (int c = 0; c < C; ++c) {
    RefineCam& k = cams[c].k;
    host_rodrigues(ext + 6 * c, k.R);
    for (int i = 0; i < 3; ++i) k.t[i] = ext[6 * c + 3 + i];
    const double* Kc = K + 9 * c;
    const double* d = dist + 5 * c;
    k.fx = Kc[0]; k.skew = Kc[1]; k.cx = Kc[2]; k.fy = Kc[4]; k.cy = Kc[5];
    k.k1 = d[0]; k.k2 = d[1]; k.p1 = d[2]; k.p2 = d[3]; k.k3 = d[4];
    host_so3_right_jacobian(ext + 6 * c, cams[c].Jr);
    cams[c].pad_ = 0.0;
  }
  // non-finite entries mark their (c, d) block and are zeroed: a point that sees both c and d gets NaN, other
  // points never read them
  const int n = 12 * C;
  std::vector<double> cov(cam_cov, cam_cov + (size_t)n * n);
  PointCovNan nanp{};
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j)
      if (!std::isfinite(cov[(size_t)i * n + j])) {
        nanp.pair[i / 12] |= 1u << (j / 12);
        nanp.pair[j / 12] |= 1u << (i / 12);
        cov[(size_t)i * n + j] = 0.0;
      }
  const size_t cam_bytes = sizeof(PointCovCam) * C, cov_bytes = sizeof(double) * n * n;
  unsigned char* d_buf = nullptr;
  MCBA_CUDA(cudaMallocAsync((void**)&d_buf, cam_bytes + cov_bytes, s));
  const PointCovCam* d_cams = reinterpret_cast<const PointCovCam*>(d_buf);
  const double* d_cov = reinterpret_cast<const double*>(d_buf + cam_bytes);
  cudaError_t e = cudaMemcpyAsync(d_buf, cams, cam_bytes, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_buf + cam_bytes, cov.data(), cov_bytes, cudaMemcpyHostToDevice, s);
  int rc = MCBA_OK;
  if (e == cudaSuccess) {
    const RefineLoss L{loss, 1.0 / f_scale, f_scale * f_scale};
    rc = C <= 8 ? launch_point_covariance<8>(s, d_uvs, C, P, d_cams, d_points, d_cov, nanp, L, sigma, d_cov_meas,
                                             d_cov_cal, d_sens)
                : launch_point_covariance<32>(s, d_uvs, C, P, d_cams, d_points, d_cov, nanp, L, sigma, d_cov_meas,
                                              d_cov_cal, d_sens);
  }
  const cudaError_t launch = cudaGetLastError();
  const cudaError_t sync = cudaStreamSynchronize(s);   // cams[] and cov are host stack / heap buffers
  cudaFreeAsync(d_buf, s);
  MCBA_CUDA(e);
  if (rc) return rc;
  MCBA_CUDA(launch);
  MCBA_CUDA(sync);
  return MCBA_OK;
}
