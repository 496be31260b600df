// SURVEY section 8f row 3: the metric loop of test.py on the device.
//   calculate_error   utils/calculate_errors.py:22-28   mean over frames and joints of |est - gt|
//   align_skeleton    utils/calculate_errors.py:60-91   per-frame similarity (Procrustes) alignment
//   umeyama           utils/rigid_transform_with_scale.py:18-43   c, R, t minimising sum |P c R + t - Q|^2
// One thread = one frame, fp64 throughout (the reference runs NumPy float64: ground truth is stored in double).
// The 3x3 SVD of the cross-covariance C = V S W is obtained from the symmetric eigenproblem C^T C = W^T S^2 W
// (cyclic Jacobi, converges to machine precision in a few sweeps); V's first two columns come from C W^T, its third is
// their cross product, so V is orthonormal for planar and collinear poses too.
#include "common.cuh"
#include <math.h>

namespace sceneego {

struct Mat3 { double m[3][3]; };

__device__ inline double det3(const Mat3& a) {
  return a.m[0][0] * (a.m[1][1] * a.m[2][2] - a.m[1][2] * a.m[2][1]) - a.m[0][1] * (a.m[1][0] * a.m[2][2] - a.m[1][2] * a.m[2][0]) +
         a.m[0][2] * (a.m[1][0] * a.m[2][1] - a.m[1][1] * a.m[2][0]);
}

// Eigen-decomposition of a symmetric 3x3 matrix: a = E^T diag(w) E, rows of E are unit eigenvectors, w descending.
__device__ inline void jacobi_eig3(Mat3 a, double (&w)[3], Mat3& e) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) e.m[i][j] = i == j ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 30; ++sweep) {
    const double off = a.m[0][1] * a.m[0][1] + a.m[0][2] * a.m[0][2] + a.m[1][2] * a.m[1][2];
    const double diag = a.m[0][0] * a.m[0][0] + a.m[1][1] * a.m[1][1] + a.m[2][2] * a.m[2][2];
    if (off <= 1e-60 * diag || off == 0.0) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (a.m[p][q] == 0.0) continue;
        const double theta = (a.m[q][q] - a.m[p][p]) / (2.0 * a.m[p][q]);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        // a <- J^T a J with J the rotation in the (p,q) plane
        for (int k = 0; k < 3; ++k) {
          const double akp = a.m[k][p], akq = a.m[k][q];
          a.m[k][p] = c * akp - s * akq;
          a.m[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 3; ++k) {
          const double apk = a.m[p][k], aqk = a.m[q][k];
          a.m[p][k] = c * apk - s * aqk;
          a.m[q][k] = s * apk + c * aqk;
        }
        for (int k = 0; k < 3; ++k) {               // accumulate eigenvectors as rows
          const double epk = e.m[p][k], eqk = e.m[q][k];
          e.m[p][k] = c * epk - s * eqk;
          e.m[q][k] = s * epk + c * eqk;
        }
      }
  }
  for (int i = 0; i < 3; ++i) w[i] = a.m[i][i];
  for (int i = 0; i < 2; ++i)                        // sort descending (3 elements)
    for (int j = 0; j < 2 - i; ++j)
      if (w[j] < w[j + 1]) {
        const double tw = w[j]; w[j] = w[j + 1]; w[j + 1] = tw;
        for (int k = 0; k < 3; ++k) { const double te = e.m[j][k]; e.m[j][k] = e.m[j + 1][k]; e.m[j + 1][k] = te; }
      }
}

template <typename TP>
__global__ void __launch_bounds__(128) pose_errors_kernel(const TP* __restrict__ pred, const double* __restrict__ gt, int B, int J,
                                                         int scale, double* __restrict__ mpjpe, double* __restrict__ pampjpe,
                                                         double* __restrict__ aligned, double* __restrict__ gt_out,
                                                         double* __restrict__ transform) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const TP* P = pred + (size_t)b * J * 3;
  const double* Q = gt + (size_t)b * J * 3;
  const double n = (double)J;
  // calculate_error on the raw poses
  double dist = 0.0, mp[3] = {0, 0, 0}, mq[3] = {0, 0, 0};
  for (int j = 0; j < J; ++j) {
    double d2 = 0.0;
    for (int k = 0; k < 3; ++k) {
      const double pk = (double)P[3 * j + k], qk = Q[3 * j + k];
      d2 += (pk - qk) * (pk - qk);
      mp[k] += pk; mq[k] += qk;
    }
    dist += sqrt(d2);
  }
  if (mpjpe) mpjpe[b] = dist / n;
  for (int k = 0; k < 3; ++k) { mp[k] /= n; mq[k] /= n; }
  // scale = False: both poses are centred first (calculate_errors.py:78-83); umeyama then sees zero means
  const double offp[3] = {scale ? 0.0 : mp[0], scale ? 0.0 : mp[1], scale ? 0.0 : mp[2]};
  const double offq[3] = {scale ? 0.0 : mq[0], scale ? 0.0 : mq[1], scale ? 0.0 : mq[2]};
  const double cp[3] = {mp[0] - offp[0], mp[1] - offp[1], mp[2] - offp[2]};   // means umeyama subtracts
  const double cq[3] = {mq[0] - offq[0], mq[1] - offq[1], mq[2] - offq[2]};
  Mat3 C;
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) C.m[i][k] = 0.0;
  double varp = 0.0;
  for (int j = 0; j < J; ++j) {
    double a[3], q[3];
    for (int k = 0; k < 3; ++k) {
      a[k] = ((double)P[3 * j + k] - offp[k]) - cp[k];
      q[k] = (Q[3 * j + k] - offq[k]) - cq[k];
      varp += a[k] * a[k];
    }
    for (int i = 0; i < 3; ++i)
      for (int k = 0; k < 3; ++k) C.m[i][k] += a[i] * q[k];
  }
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) C.m[i][k] /= n;
  varp /= n;                                                   // np.var(P, axis=0).sum()
  // C = V diag(S) W
  Mat3 CtC, W, V;
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) CtC.m[i][k] = C.m[0][i] * C.m[0][k] + C.m[1][i] * C.m[1][k] + C.m[2][i] * C.m[2][k];
  double ev[3], S[3], U[3][3];
  jacobi_eig3(CtC, ev, W);
  for (int i = 0; i < 3; ++i) S[i] = sqrt(ev[i] > 0.0 ? ev[i] : 0.0);
  const double tiny = 1e-14 * (S[0] > 0.0 ? S[0] : 1.0);
  for (int c = 0; c < 3; ++c)                                  // U[c] = C W[c, :]^T = S[c] V[:, c]
    for (int i = 0; i < 3; ++i) U[c][i] = C.m[i][0] * W.m[c][0] + C.m[i][1] * W.m[c][1] + C.m[i][2] * W.m[c][2];
  // V is made orthonormal from its first two columns.  A singular value below ~1e-8 S[0] is eigenvalue noise of
  // C^T C (absolute error ~eps S[0]^2), so U[c] / S[c] is not a unit vector there: near-planar poses would get a
  // non-orthogonal R.  Column 1 is U[1] orthogonalised against column 0 and normalised, or any unit vector orthogonal
  // to it (rank <= 1: the rotation is not unique); column 2 is col0 x col1, so R = V W needs no third singular vector.
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) V.m[i][k] = i == k ? 1.0 : 0.0;   // rank 0: V = I
  const double n0 = sqrt(U[0][0] * U[0][0] + U[0][1] * U[0][1] + U[0][2] * U[0][2]);
  if (S[0] > tiny && n0 > 0.0) {
    double v0[3], v1[3];
    for (int i = 0; i < 3; ++i) v0[i] = U[0][i] / n0;
    const double p = v0[0] * U[1][0] + v0[1] * U[1][1] + v0[2] * U[1][2];
    for (int i = 0; i < 3; ++i) v1[i] = U[1][i] - p * v0[i];
    double n1 = sqrt(v1[0] * v1[0] + v1[1] * v1[1] + v1[2] * v1[2]);
    if (!(S[1] > tiny && n1 > tiny)) {                         // rank 1: v0 x (the axis least aligned with v0)
      const int k = fabs(v0[0]) <= fabs(v0[1]) ? (fabs(v0[0]) <= fabs(v0[2]) ? 0 : 2) : (fabs(v0[1]) <= fabs(v0[2]) ? 1 : 2);
      const int k1 = (k + 1) % 3, k2 = (k + 2) % 3;
      v1[k] = 0.0; v1[k1] = v0[k2]; v1[k2] = -v0[k1];          // v0 x e_k
      n1 = sqrt(v1[k1] * v1[k1] + v1[k2] * v1[k2]);
    }
    for (int i = 0; i < 3; ++i) { V.m[i][0] = v0[i]; V.m[i][1] = v1[i] / n1; }
    V.m[0][2] = V.m[1][0] * V.m[2][1] - V.m[2][0] * V.m[1][1];
    V.m[1][2] = V.m[2][0] * V.m[0][1] - V.m[0][0] * V.m[2][1];
    V.m[2][2] = V.m[0][0] * V.m[1][1] - V.m[1][0] * V.m[0][1];
  }
  for (int c = 0; c < 3; ++c) S[c] = V.m[0][c] * U[c][0] + V.m[1][c] * U[c][1] + V.m[2][c] * U[c][2];   // trace terms
  if (det3(V) * det3(W) < 0.0) {
    S[2] = -S[2];
    for (int i = 0; i < 3; ++i) V.m[i][2] = -V.m[i][2];
  }
  Mat3 R;
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) R.m[i][k] = V.m[i][0] * W.m[0][k] + V.m[i][1] * W.m[1][k] + V.m[i][2] * W.m[2][k];
  const double c = (S[0] + S[1] + S[2]) / varp;
  double t[3];
  for (int k = 0; k < 3; ++k) t[k] = cq[k] - c * (cp[0] * R.m[0][k] + cp[1] * R.m[1][k] + cp[2] * R.m[2][k]);
  if (transform) {
    double* T = transform + (size_t)b * 13;
    T[0] = c;
    for (int i = 0; i < 3; ++i)
      for (int k = 0; k < 3; ++k) T[1 + 3 * i + k] = R.m[i][k];
    for (int k = 0; k < 3; ++k) T[10 + k] = t[k];
  }
  const double cs = scale ? c : 1.0;                           // scale = False: pose_p.dot(R) + t
  double pa = 0.0;
  for (int j = 0; j < J; ++j) {
    double a[3], d2 = 0.0;
    for (int k = 0; k < 3; ++k) a[k] = (double)P[3 * j + k] - offp[k];
    for (int k = 0; k < 3; ++k) {
      const double v = cs * (a[0] * R.m[0][k] + a[1] * R.m[1][k] + a[2] * R.m[2][k]) + t[k];
      const double g = Q[3 * j + k] - offq[k];
      if (aligned) aligned[((size_t)b * J + j) * 3 + k] = v;
      if (gt_out) gt_out[((size_t)b * J + j) * 3 + k] = g;
      d2 += (v - g) * (v - g);
    }
    pa += sqrt(d2);
  }
  if (pampjpe) pampjpe[b] = pa / n;
}

}  // namespace sceneego

using namespace sceneego;

extern "C" int sceneego_pose_errors_f64(const void* d_pred, int pred_is_f64, const double* d_gt, int batch, int joints,
                                        int scale, double* d_mpjpe, double* d_pampjpe, double* d_aligned,
                                        double* d_gt_out, double* d_transform, void* stream) {
  SE_REQUIRE(d_pred && d_gt && batch > 0 && joints >= 3, "pose_errors: bad argument");
  if (pred_is_f64)
    pose_errors_kernel<double><<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        (const double*)d_pred, d_gt, batch, joints, scale ? 1 : 0, d_mpjpe, d_pampjpe, d_aligned, d_gt_out, d_transform);
  else
    pose_errors_kernel<float><<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        (const float*)d_pred, d_gt, batch, joints, scale ? 1 : 0, d_mpjpe, d_pampjpe, d_aligned, d_gt_out, d_transform);
  SE_CUDA_LAUNCH_CHECK("pose_errors");
  return SCENEEGO_OK;
}
