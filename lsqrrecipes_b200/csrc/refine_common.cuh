// Shared by k_refine.cu (streaming consensus-set + moments pass, moment solves, Levenberg-Marquardt kernels) and k_batch.cu
// (one CTA per small problem): the least-squares moments of every estimator, their accumulation per datum and the
// moments -> parameters solves.  Device code only; every function is inline / static so that both translation units can
// carry their own copy (no relocatable device code).
#pragma once
#include "engine.h"
#include "../../include/lsqr_b200.h"
#include "lm_minpack.cuh"

namespace lsqr {


// number of accumulated doubles per model (index 0 is always the inlier count)
__host__ __device__ constexpr int n_moments(int model, bool lm) {
  const int d = model_dim(model);
  switch (model_family(model)) {
    case FAM_PLANE: case FAM_LINE: return 1 + d + d * (d + 1) / 2;                 // count, sums, upper triangle of the second moments
    case FAM_SPHERE: return lm ? 1 + (d + 1) * (d + 2) / 2 + (d + 1) + 1           // count, J^T J, J^T r, cost
                               : 1 + d + d * (d + 1) / 2 + d + 1;                   // scatter sums, sum |p|^2 p, sum |p|^2
    case FAM_DENSE: return 1 + d * (d + 1) / 2 + d;                                // count, A^T A upper triangle, A^T b
    default: break;
  }
  switch (model) {
    case LINE2D: return 6;
    case ABSOR: return 16;
    case RAY: return 10;
    case PIVOT: return 22;
    case USXW: return lm ? 79 : 91;   // LM: count, J^T J (66), J^T e (11), cost; analytic: count, A^T A (78), A^T b (12)
    case USCP: return lm ? 46 : 55;   // LM: count, 36, 8, cost; analytic: count, 45, 9
  }
  return 0;
}
static_assert(kLmStateDoubles >= LM_SIZE, "engine.h: LM state buffer too small");


// N / NLM = accumulated doubles of the analytic / Levenberg-Marquardt pass, NPLM = parameters of the LM problem
template <int M> struct Mom {
  static constexpr bool kHasLm = model_family(M) == FAM_SPHERE || M == USXW || M == USCP;
  static constexpr int N = n_moments(M, false), NLM = kHasLm ? n_moments(M, true) : 0;
  static constexpr int NPLM = model_family(M) == FAM_SPHERE ? model_dim(M) + 1 : (M == USXW ? 11 : (M == USCP ? 8 : 1));
};
static_assert(Mom<SPHERE8>::NLM <= kMaxMoments && Mom<USXW>::N <= kMaxMoments && Mom<SPHERE8>::NPLM <= kLmMaxP, "engine.h / lm_minpack.cuh capacities");

// q = centred datum.  acc[0] is the inlier count: the callers add it (the streaming pass feeds zeros for data outside the
// consensus set instead of branching, so only the count must know).
template <int DIM> __device__ __forceinline__ void acc_scatter(const double* q, double* acc) {
  int o = 1;
#pragma unroll
  for (int j = 0; j < DIM; j++) acc[o++] += q[j];
#pragma unroll
  for (int j = 0; j < DIM; j++)
#pragma unroll
    for (int k = j; k < DIM; k++) { acc[o] = fma(q[j], q[k], acc[o]); o++; }   // (this TU is built with -fmad=false for agree(); the sums may fuse)
}
template <int DIM> __device__ __forceinline__ void acc_sphere_alg(const double* q, double* acc) {
  double s = 0;
#pragma unroll
  for (int j = 0; j < DIM; j++) s = fma(q[j], q[j], s);
  acc_scatter<DIM>(q, acc);
  int o = 1 + DIM + DIM * (DIM + 1) / 2;
#pragma unroll
  for (int j = 0; j < DIM; j++) { acc[o] = fma(s, q[j], acc[o]); o++; }
  acc[o] += s;
}
// residual / Jacobian of SphereParametersEstimator.hxx:394-431 at x = (centre', r)
template <int DIM> __device__ __forceinline__ void acc_sphere_lm(const double* q, const double* x, double* acc) {
  double J[DIM + 1], s = 0;
#pragma unroll
  for (int j = 0; j < DIM; j++) s += (q[j] - x[j]) * (q[j] - x[j]);
  const double sv = sqrt(s), r = sv - x[DIM];
#pragma unroll
  for (int j = 0; j < DIM; j++) J[j] = (x[j] - q[j]) / sv;
  J[DIM] = -1.0;
  acc[0] += 1.0;
  int o = 1;
#pragma unroll
  for (int a = 0; a <= DIM; a++)
#pragma unroll
    for (int b = a; b <= DIM; b++) { acc[o] = fma(J[a], J[b], acc[o]); o++; }
#pragma unroll
  for (int a = 0; a <= DIM; a++) { acc[o] = fma(J[a], r, acc[o]); o++; }
  acc[o] = fma(r, r, acc[o]);
}

template <int M> __device__ __forceinline__ void accumulate(const double* q, double* acc);
template <> __device__ __forceinline__ void accumulate<PLANE3>(const double* q, double* acc) { acc_scatter<3>(q, acc); }
template <> __device__ __forceinline__ void accumulate<LINE2D>(const double* q, double* acc) { acc_scatter<2>(q, acc); }
#define LSQR_DEF_(ID, DIM) template <> __device__ __forceinline__ void accumulate<ID>(const double* q, double* acc) { acc_scatter<DIM>(q, acc); }
LSQR_PLANE_ND_LIST(LSQR_DEF_)
LSQR_LINE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_
#define LSQR_DEF_(ID, DIM) template <> __device__ __forceinline__ void accumulate<ID>(const double* q, double* acc) { acc_sphere_alg<DIM>(q, acc); }
LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
#undef LSQR_DEF_
// AbsoluteOrientationParametersEstimator.cxx:134-166: sums of both point sets and of p1 p2^T
template <> __device__ __forceinline__ void accumulate<ABSOR>(const double* q, double* acc) {
#pragma unroll
  for (int j = 0; j < 6; j++) acc[1 + j] += q[j];
#pragma unroll
  for (int r = 0; r < 3; r++)
#pragma unroll
    for (int c = 0; c < 3; c++) acc[7 + r * 3 + c] = fma(q[r], q[3 + c], acc[7 + r * 3 + c]);
}
// Weighted Horn (AbsoluteOrientationParametersEstimator.cxx:217-261): pair q (centred) with weight w into sum w, sum w p1,
// sum w p2 and sum w p1 p2^T (acc[0..15])
__device__ __forceinline__ void acc_absor_weighted(const double* q, double w, double* acc) {
  acc[0] += w;
#pragma unroll
  for (int j = 0; j < 6; j++) acc[1 + j] += q[j] * w;
#pragma unroll
  for (int r = 0; r < 3; r++)
#pragma unroll
    for (int c = 0; c < 3; c++) acc[7 + r * 3 + c] += (q[r] * q[3 + c]) * w;
}
// RayIntersectionParametersEstimator.cxx:108-123
template <> __device__ __forceinline__ void accumulate<RAY>(const double* q, double* acc) {
  const double* n = q + 3;
  acc[1] += n[0] * n[0]; acc[2] += n[0] * n[1]; acc[3] += n[0] * n[2];
  acc[4] += n[1] * n[1]; acc[5] += n[1] * n[2]; acc[6] += n[2] * n[2];
  const double s = n[0] * q[0] + n[1] * q[1] + n[2] * q[2];
  acc[7] += q[0] - s * n[0]; acc[8] += q[1] - s * n[1]; acc[9] += q[2] - s * n[2];
}
// Normal equations of the rows [R | -I] x = -t (PivotCalibrationParametersEstimator.cxx:77-83)
template <> __device__ __forceinline__ void accumulate<PIVOT>(const double* q, double* acc) {
  int o = 1;
#pragma unroll
  for (int a = 0; a < 3; a++)
#pragma unroll
    for (int b = a; b < 3; b++) acc[o++] += q[a] * q[b] + q[3 + a] * q[3 + b] + q[6 + a] * q[6 + b];  // (R^T R)_{ab}
#pragma unroll
  for (int j = 0; j < 9; j++) acc[o++] += q[j];                                                          // sum R
#pragma unroll
  for (int a = 0; a < 3; a++) acc[o++] += q[a] * q[9] + q[3 + a] * q[10] + q[6 + a] * q[11];            // R^T t
#pragma unroll
  for (int a = 0; a < 3; a++) acc[o++] += q[9 + a];                                                      // sum t
}

// Normal equations of the rows a.x = b (DenseLinearEquationSystemParametersEstimator.hxx:64-96)
template <int N> __device__ __forceinline__ void acc_dense(const double* q, double* acc) {
  int o = 1;
#pragma unroll
  for (int a = 0; a < N; a++)
#pragma unroll
    for (int b = a; b < N; b++) { acc[o] = fma(q[a], q[b], acc[o]); o++; }
#pragma unroll
  for (int a = 0; a < N; a++) { acc[o] = fma(q[a], q[N], acc[o]); o++; }
}
#define LSQR_DEF_(ID, N) template <> __device__ __forceinline__ void accumulate<ID>(const double* q, double* acc) { acc_dense<N>(q, acc); }
LSQR_DENSE_N_LIST(LSQR_DEF_)
#undef LSQR_DEF_

// Normal equations of the rows [u R2, v R2, R2, -I] x = -t2 (SinglePointTargetUSCalibrationParametersEstimator.cxx:137-189)
template <> __device__ __forceinline__ void accumulate<USXW>(const double* q, double* acc) {
  const double u = q[12], v = q[13];
#pragma unroll
  for (int r = 0; r < 3; r++) {
    double row[12];
#pragma unroll
    for (int c = 0; c < 3; c++) { row[c] = q[3 * r + c] * u; row[3 + c] = q[3 * r + c] * v; row[6 + c] = q[3 * r + c]; row[9 + c] = (c == r) ? -1.0 : 0.0; }
    const double b = -q[9 + r];
    int o = 1;
#pragma unroll
    for (int a = 0; a < 12; a++)
#pragma unroll
      for (int bb = a; bb < 12; bb++) acc[o++] += row[a] * row[bb];
#pragma unroll
    for (int a = 0; a < 12; a++) acc[o++] += row[a] * b;
  }
}
// Levenberg-Marquardt pass of the ultrasound calibrations.  The reference hands MINPACK the SCALAR residuals d_i = |e_i| with
// e_i = R2 (u m_x c1 + v m_y c2 + t3) + t2 - t1 (f, SinglePointTargetUSCalibrationParametersEstimator.cxx:415-507) and the
// Jacobian rows (e_i^T de_i/dx) / d_i (gradf, :510-658); the iteration path depends on that choice (J^T J of the scalar form is
// not the one of the vector form), so the same rows are accumulated here: count, J^T J (upper triangle), J^T d, sum d^2.
// x = [t1 (NT1 = 3, cross-wire only), t3, omega_z, omega_y, omega_x, m_x, m_y]; `tgt` is t1 or the measured pointer tip p.
template <int NT1> __device__ __forceinline__ void acc_us_lm_rows(const double* q, const double* x, const double* tgt, double* acc) {
  constexpr int NP = NT1 + 8;
  const double* y = x + NT1;   // t3, angles, scales
  const double sz = sin(y[3]), cz = cos(y[3]), sy = sin(y[4]), cy = cos(y[4]), sx = sin(y[5]), cx = cos(y[5]);
  const double mx = y[6], my = y[7], u = q[12], v = q[13];
  const double c1[3] = {cz * cy, sz * cy, -sy};
  const double c2[3] = {cz * sy * sx - sz * cx, sz * sy * sx + cz * cx, cy * sx};
  const double dc1[3][3] = {{-sz * cy, cz * cy, 0}, {-cz * sy, -sz * sy, -cy}, {0, 0, 0}};
  const double dc2[3][3] = {{-sz * sy * sx - cz * cx, cz * sy * sx - sz * cx, 0}, {cz * cy * sx, sz * cy * sx, -sy * sx},
                            {cz * sy * cx + sz * sx, sz * sy * cx - cz * sx, cy * cx}};
  double w[3], dw[8][3];   // d w / d (t3 (3), omega (3), m_x, m_y)
#pragma unroll
  for (int k = 0; k < 3; k++) {
    w[k] = u * mx * c1[k] + v * my * c2[k] + y[k];
#pragma unroll
    for (int p = 0; p < 3; p++) { dw[p][k] = (p == k) ? 1.0 : 0.0; dw[3 + p][k] = u * mx * dc1[p][k] + v * my * dc2[p][k]; }
    dw[6][k] = u * c1[k];
    dw[7][k] = v * c2[k];
  }
  double e[3], J[NP];
#pragma unroll
  for (int p = 0; p < NP; p++) J[p] = 0.0;
#pragma unroll
  for (int r = 0; r < 3; r++) {
    const double a = q[3 * r], b = q[3 * r + 1], c = q[3 * r + 2];
    e[r] = a * w[0] + b * w[1] + c * w[2] + q[9 + r] - tgt[r];
    if (NT1) J[r] = -e[r];
#pragma unroll
    for (int p = 0; p < 8; p++) J[NT1 + p] += (a * dw[p][0] + b * dw[p][1] + c * dw[p][2]) * e[r];
  }
  const double d = sqrt(e[0] * e[0] + e[1] * e[1] + e[2] * e[2]);
#pragma unroll
  for (int p = 0; p < NP; p++) J[p] /= d;
  acc[0] += 1.0;
  int o = 1;
#pragma unroll
  for (int i = 0; i < NP; i++)
#pragma unroll
    for (int j = i; j < NP; j++) { acc[o] = fma(J[i], J[j], acc[o]); o++; }
#pragma unroll
  for (int i = 0; i < NP; i++) { acc[o] = fma(J[i], d, acc[o]); o++; }
  acc[o] = fma(d, d, acc[o]);
}
__device__ __forceinline__ void acc_us_lm(const double* q, const double* x, double* acc) { acc_us_lm_rows<3>(q, x, x, acc); }

// Normal equations of the rows [u R2, v R2, R2] x = p - t2 (SinglePointTargetUSCalibrationParametersEstimator.cxx:806-846)
template <> __device__ __forceinline__ void accumulate<USCP>(const double* q, double* acc) {
  const double u = q[12], v = q[13];
#pragma unroll
  for (int r = 0; r < 3; r++) {
    double row[9];
#pragma unroll
    for (int c = 0; c < 3; c++) { row[c] = q[3 * r + c] * u; row[3 + c] = q[3 * r + c] * v; row[6 + c] = q[3 * r + c]; }
    const double b = q[14 + r] - q[9 + r];
    int o = 1;
#pragma unroll
    for (int a = 0; a < 9; a++)
#pragma unroll
      for (int bb = a; bb < 9; bb++) acc[o++] += row[a] * row[bb];
#pragma unroll
    for (int a = 0; a < 9; a++) acc[o++] += row[a] * b;
  }
}
// calibrated pointer: the same rows with the measured tip position p (q[14..16]) in the place of t1 and no unknown for it
__device__ __forceinline__ void acc_uscp_lm(const double* q, const double* x, double* acc) { acc_us_lm_rows<0>(q, x, q + 14, acc); }

// ---------------------------------------------------------------------------------------
// moments -> parameters
// ---------------------------------------------------------------------------------------

// Symmetric positive semi-definite solve through the eigen-decomposition of the diagonally
// scaled matrix; eigenvalues below 1e-13 of the largest are dropped.  Returns the rank.
// Stands in for vnl_matrix_inverse on the normal equations of the reference's tall systems.
template <int N>
__device__ int sym_pinv_solve(const double* A, const double* b, double* x) {
  double S[N * N], V[N * N], ev[N], sc[N], y[N];
  for (int i = 0; i < N; i++) sc[i] = A[i * N + i] > 0 ? 1.0 / sqrt(A[i * N + i]) : 1.0;
  for (int i = 0; i < N; i++) for (int j = 0; j < N; j++) S[i * N + j] = A[i * N + j] * sc[i] * sc[j];
  sym_eig<N>(S, V, ev);
  const double tol = 1e-13 * fabs(ev[N - 1]);
  int rank = 0;
  for (int k = 0; k < N; k++) {
    double d = 0;
    for (int i = 0; i < N; i++) d += V[i * N + k] * (b[i] * sc[i]);
    if (ev[k] > tol) { y[k] = d / ev[k]; rank++; } else y[k] = 0.0;
  }
  for (int i = 0; i < N; i++) { double s = 0; for (int k = 0; k < N; k++) s += V[i * N + k] * y[k]; x[i] = s * sc[i]; }
  return rank;
}

// PlaneParametersEstimator.hxx:141-171 (col 0) / LineParametersEstimator.hxx:80-110 (col DIM-1)
template <int DIM> __device__ int solve_scatter(const double* m, const double* c, int col, double* out) {
  const double n = m[0];
  if (n < 1.0) return 0;
  double C[DIM * DIM], V[DIM * DIM], ev[DIM];
  int o = 1 + DIM;
  for (int j = 0; j < DIM; j++) for (int k = j; k < DIM; k++) { const double v = m[o++] - m[1 + j] * m[1 + k] / n; C[j * DIM + k] = v; C[k * DIM + j] = v; }
  sym_eig<DIM>(C, V, ev);
  for (int j = 0; j < DIM; j++) out[j] = V[j * DIM + col];
  for (int j = 0; j < DIM; j++) out[DIM + j] = m[1 + j] / n + c[j];
  return 2 * DIM;
}
// Line2DParametersEstimator.cxx:50-100
static __device__ int solve_line2d(const double* m, const double* c, double* out) {
  const double n = m[0];
  if (n < 1.0) return 0;
  const double mx = m[1] / n, my = m[2] / n;
  const double c11 = m[3] - n * mx * mx, c12 = m[4] - n * mx * my, c22 = m[5] - n * my * my;
  double nx, ny;
  if (c11 < 1e-12) {
    nx = 1.0; ny = 0.0;
    if (c22 < 1e-12) return 0;
  } else {
    const double lambda1 = (c11 + c22 + sqrt((c11 - c22) * (c11 - c22) + 4 * c12 * c12)) / 2.0;
    nx = -c12; ny = lambda1 - c22;
    const double norm = sqrt(nx * nx + ny * ny);
    nx /= norm; ny /= norm;
  }
  out[0] = nx; out[1] = ny; out[2] = mx + c[0]; out[3] = my + c[1];
  return 4;
}
// SphereParametersEstimator.hxx:267-307 through the normal equations of [-2p, 1] x = -|p|^2.
// Result in centred coordinates: out = (centre', r).
template <int DIM> __device__ int solve_sphere_alg(const double* m, double* out) {
  constexpr int NP = DIM + 1;
  const double n = m[0];
  if (n < (double)NP) return 0;
  double A[NP * NP], b[NP], x[NP];
  int o = 1 + DIM;
  for (int j = 0; j < DIM; j++) for (int k = j; k < DIM; k++) { const double v = 4.0 * m[o++]; A[j * NP + k] = v; A[k * NP + j] = v; }
  for (int j = 0; j < DIM; j++) { A[j * NP + DIM] = -2.0 * m[1 + j]; A[DIM * NP + j] = -2.0 * m[1 + j]; }
  A[DIM * NP + DIM] = n;
  for (int j = 0; j < DIM; j++) b[j] = 2.0 * m[o++];
  b[DIM] = -m[o];
  if (sym_pinv_solve<NP>(A, b, x) < NP) return 0;
  double r2 = -x[DIM];
  for (int j = 0; j < DIM; j++) { out[j] = x[j]; r2 += x[j] * x[j]; }
  if (!(r2 > 0)) return 0;
  out[DIM] = sqrt(r2);
  return NP;
}
// AbsoluteOrientationParametersEstimator.cxx:134-205 (Horn): M = sum p1 p2^T - N mu1 mu2^T, 4x4 N matrix,
// eigenvector of the largest eigenvalue, t = mu2 - R mu1 with the normalised quaternion.
// m[0] is the number of pairs, or the sum of the weights for the weighted variant (:208-297), whose
// size guard is on the number of pairs and is applied by the caller.
static __device__ int solve_absor(const double* m, const double* c, double* out, bool weighted = false) {
  const double n = m[0];
  if (!weighted && n < 3.0) return 0;
  if (weighted && !(n == n && n != 0.0)) return 0;
  double mu1[3], mu2[3], Mm[9], Nm[16], V[16], ev[4], R[9];
  for (int j = 0; j < 3; j++) { mu1[j] = m[1 + j] / n; mu2[j] = m[4 + j] / n; }
  for (int r = 0; r < 3; r++) for (int cc = 0; cc < 3; cc++) Mm[r * 3 + cc] = m[7 + r * 3 + cc] - n * mu1[r] * mu2[cc];
  const double tr = Mm[0] + Mm[4] + Mm[8];
  const double A12 = Mm[5] - Mm[7], A20 = Mm[6] - Mm[2], A01 = Mm[1] - Mm[3];
  for (int i = 0; i < 16; i++) Nm[i] = 0.0;
  Nm[0] = tr; Nm[1] = A12; Nm[2] = A20; Nm[3] = A01; Nm[4] = A12; Nm[8] = A20; Nm[12] = A01;
  for (int r = 0; r < 3; r++) for (int cc = 0; cc < 3; cc++) Nm[(r + 1) * 4 + cc + 1] = ((r == cc) ? -tr : 0.0) + (Mm[r * 3 + cc] + Mm[cc * 3 + r]);
  sym_eig<4>(Nm, V, ev);
  double q[4];
  for (int r = 0; r < 4; r++) { q[r] = V[r * 4 + 3]; out[r] = q[r]; }
  const double norm = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  quat_to_rot(q[0] / norm, q[1] / norm, q[2] / norm, q[3] / norm, R);
  for (int r = 0; r < 3; r++) {
    const double f = R[3 * r] * (mu1[0] + c[0]) + R[3 * r + 1] * (mu1[1] + c[1]) + R[3 * r + 2] * (mu1[2] + c[2]);
    out[4 + r] = (mu2[r] + c[3 + r]) - f;
  }
  return 7;
}
// RayIntersectionParametersEstimator.cxx:124-143
static __device__ int solve_ray(const double* m, const double* c, double* out) {
  const double n = m[0];
  double A[9], x[3];
  A[0] = n - m[1]; A[1] = -m[2]; A[2] = -m[3];
  A[3] = A[1]; A[4] = n - m[4]; A[5] = -m[5];
  A[6] = A[2]; A[7] = A[5]; A[8] = n - m[6];
  if (n < 1.0 || sym_pinv_solve<3>(A, m + 7, x) < 3) return 0;
  for (int j = 0; j < 3; j++) out[j] = x[j] + c[j];
  return 3;
}
// PivotCalibrationParametersEstimator.cxx:63-96 through the 6x6 normal equations
static __device__ int solve_pivot(const double* m, const double* c, double* out) {
  const double n = m[0];
  if (n < 3.0) return 0;
  double A[36], b[6], x[6];
  int o = 1;
  for (int a = 0; a < 3; a++) for (int bb = a; bb < 3; bb++) { const double v = m[o++]; A[a * 6 + bb] = v; A[bb * 6 + a] = v; }
  const double* SR = m + 7;  // sum R, row-major
  for (int a = 0; a < 3; a++) for (int bb = 0; bb < 3; bb++) {
    A[a * 6 + 3 + bb] = -SR[bb * 3 + a];  // -(sum R)^T
    A[(3 + bb) * 6 + a] = -SR[bb * 3 + a];
    A[(3 + a) * 6 + 3 + bb] = (a == bb) ? n : 0.0;
  }
  for (int a = 0; a < 3; a++) { b[a] = -m[16 + a]; b[3 + a] = m[19 + a]; }
  if (sym_pinv_solve<6>(A, b, x) < 6) return 0;
  for (int j = 0; j < 3; j++) { out[j] = x[j]; out[3 + j] = x[3 + j] + c[9 + j]; }
  return 6;
}

// DenseLinearEquationSystemParametersEstimator.hxx:64-96 through the n x n normal equations; rank < n -> no solution
template <int N> __device__ int solve_dense(const double* m, double* out) {
  if (m[0] < (double)N) return 0;
  double A[N * N], b[N];
  int o = 1;
  for (int a = 0; a < N; a++) for (int bb = a; bb < N; bb++) { const double v = m[o++]; A[a * N + bb] = v; A[bb * N + a] = v; }
  for (int a = 0; a < N; a++) b[a] = m[o++];
  return sym_pinv_solve<N>(A, b, out) < N ? 0 : N;
}

// Analytic cross-wire calibration (SinglePointTargetUSCalibrationParametersEstimator.cxx:120-270) through the
// 12 x 12 normal equations; t1 comes back relative to the centre of the t2 components.
static __device__ int solve_us(const double* m, const double* c, double* out) {
  if (m[0] < 4.0) return 0;
  // diagonally scaled Cholesky of the 12 x 12 normal equations; a pivot below 1e-13 of the unit diagonal means
  // rank < 12 (the reference's "points do not yield a solution", .cxx:195-196)
  double S[144], sc[12], y[12], x[12];
  {
    int o = 1;
    for (int a = 0; a < 12; a++) for (int bb = a; bb < 12; bb++) { const double v = m[o++]; S[a * 12 + bb] = v; S[bb * 12 + a] = v; }
    for (int a = 0; a < 12; a++) y[a] = m[o++];
  }
  for (int i = 0; i < 12; i++) { if (!(S[i * 12 + i] > 0)) return 0; sc[i] = 1.0 / sqrt(S[i * 12 + i]); }
  for (int i = 0; i < 12; i++) { for (int j = 0; j < 12; j++) S[i * 12 + j] *= sc[i] * sc[j]; y[i] *= sc[i]; }
  for (int j = 0; j < 12; j++) {
    double d = S[j * 12 + j];
    for (int k = 0; k < j; k++) d -= S[j * 12 + k] * S[j * 12 + k];
    if (!(d > 1e-13)) return 0;
    S[j * 12 + j] = sqrt(d);
    for (int i = j + 1; i < 12; i++) { double t = S[i * 12 + j]; for (int k = 0; k < j; k++) t -= S[i * 12 + k] * S[j * 12 + k]; S[i * 12 + j] = t / S[j * 12 + j]; }
  }
  for (int i = 0; i < 12; i++) { double t = y[i]; for (int k = 0; k < i; k++) t -= S[i * 12 + k] * x[k]; x[i] = t / S[i * 12 + i]; }
  for (int i = 11; i >= 0; i--) { double t = x[i]; for (int k = i + 1; k < 12; k++) t -= S[k * 12 + i] * x[k]; x[i] = t / S[i * 12 + i]; }
  for (int i = 0; i < 12; i++) x[i] *= sc[i];
  if (c) for (int j = 0; j < 3; j++) x[9 + j] += c[9 + j];
  return us_post(x, out) ? 20 : 0;
}

// Analytic calibrated-pointer calibration (.cxx:789-920) through the 9 x 9 normal equations (scaled Cholesky as above)
static __device__ int solve_uscp(const double* m, double* out) {
  if (m[0] < 3.0) return 0;
  double S[81], sc[9], y[9], x[9];
  {
    int o = 1;
    for (int a = 0; a < 9; a++) for (int bb = a; bb < 9; bb++) { const double v = m[o++]; S[a * 9 + bb] = v; S[bb * 9 + a] = v; }
    for (int a = 0; a < 9; a++) y[a] = m[o++];
  }
  for (int i = 0; i < 9; i++) { if (!(S[i * 9 + i] > 0)) return 0; sc[i] = 1.0 / sqrt(S[i * 9 + i]); }
  for (int i = 0; i < 9; i++) { for (int j = 0; j < 9; j++) S[i * 9 + j] *= sc[i] * sc[j]; y[i] *= sc[i]; }
  for (int j = 0; j < 9; j++) {
    double d = S[j * 9 + j];
    for (int k = 0; k < j; k++) d -= S[j * 9 + k] * S[j * 9 + k];
    if (!(d > 1e-13)) return 0;
    S[j * 9 + j] = sqrt(d);
    for (int i = j + 1; i < 9; i++) { double t = S[i * 9 + j]; for (int k = 0; k < j; k++) t -= S[i * 9 + k] * S[j * 9 + k]; S[i * 9 + j] = t / S[j * 9 + j]; }
  }
  for (int i = 0; i < 9; i++) { double t = y[i]; for (int k = 0; k < i; k++) t -= S[i * 9 + k] * x[k]; x[i] = t / S[i * 9 + i]; }
  for (int i = 8; i >= 0; i--) { double t = x[i]; for (int k = i + 1; k < 9; k++) t -= S[k * 9 + i] * x[k]; x[i] = t / S[i * 9 + i]; }
  for (int i = 0; i < 9; i++) x[i] *= sc[i];
  return uscp_post(x, out) ? 17 : 0;
}

// moments -> parameters of any model; returns the number of parameters (0 = the reference's empty vector).
// For the hypersphere family the centre stays in centred coordinates when keep_centred != 0 (LM start).
static __device__ int solve_model(int model, const double* m, const double* c, int keep_centred, double* p) {
  int np = 0;
  switch (model) {
    case PLANE3: np = solve_scatter<3>(m, c, 0, p); break;
    case LINE2D: np = solve_line2d(m, c, p); break;
#define LSQR_DEF_(ID, DIM) case ID: np = solve_scatter<DIM>(m, c, 0, p); break;
    LSQR_PLANE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_
#define LSQR_DEF_(ID, DIM) case ID: np = solve_scatter<DIM>(m, c, DIM - 1, p); break;
    LSQR_LINE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_
#define LSQR_DEF_(ID, DIM) case ID: np = solve_sphere_alg<DIM>(m, p); if (np && !keep_centred) for (int j = 0; j < DIM; j++) p[j] += c[j]; break;
    LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
#undef LSQR_DEF_
#define LSQR_DEF_(ID, N) case ID: np = solve_dense<N>(m, p); break;
    LSQR_DENSE_N_LIST(LSQR_DEF_)
#undef LSQR_DEF_
    case ABSOR: np = solve_absor(m, c, p); break;
    case RAY: np = solve_ray(m, c, p); break;
    case PIVOT: np = solve_pivot(m, c, p); break;
    case USXW: np = solve_us(m, keep_centred ? nullptr : c, p); break;   // LM start: t1 stays relative to the centre
    case USCP: np = solve_uscp(m, p); break;
    default: break;
  }
  return np;
}
// out[0] = number of parameters, out[1..] = parameters.
// ---------------------------------------------------------------------------------------
// Levenberg-Marquardt controller: lm_minpack.cuh (MINPACK's lmder restated on the normal equations, the reference's
// tolerances per estimator).  Result only if MINPACK would report info 1..4 (vnl_levenberg_marquardt::minimize returns
// true), else empty parameters.  One pass of mask_moments_kernel delivers J^T J, J^T f and |f|^2 at the point the state
// asks for.
// ---------------------------------------------------------------------------------------
__host__ __device__ inline void lm_update_model(int model, const double* m, double* st) {
  switch (model) {
#define LSQR_DEF_(ID, DIM) case ID: lm_update<DIM + 1>(m, st, lm_tolerances(0)); break;
    LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
#undef LSQR_DEF_
    case USXW: lm_update<11>(m, st, lm_tolerances(1)); break;
    case USCP: lm_update<8>(m, st, lm_tolerances(2)); break;
    default: break;
  }
}

}  // namespace lsqr
