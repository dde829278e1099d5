// Device-side estimator arithmetic in fp64 "validation" form: the reference's operation order,
// one rounding per operation.  Every translation unit that includes this header is compiled
// with -fmad=false so that nvcc never contracts a*b+c into an FMA; sqrt and / are IEEE
// correctly rounded for double on sm_100a, which makes these bodies round exactly like the
// reference built with g++ -O2 -ffp-contract=off on x86-64 (SURVEY.md section 7 "hard parts").
//
// Hot-path pieces are split in two so the per-hypothesis work is hoisted out of the point
// loop without changing a single rounding: prepare<M>() runs once per hypothesis (e.g. the
// quaternion -> rotation matrix that the reference redoes on every agree() call,
// AbsoluteOrientationParametersEstimator.cxx:318-319), agree<M>() runs per (hypothesis, datum).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace lsqr {

enum : int { PLANE3 = 0, LINE2D = 1, LINE2 = 2, LINE3 = 3, CIRCLE2 = 4, SPHERE3 = 5, ABSOR = 6, RAY = 7, PIVOT = 8, DENSE5 = 9, DENSE6 = 10, USXW = 11, USCP = 12, SPHERE4 = 13, PLANE4 = 14,
              // the rest of the reference's template space (SURVEY 8f-4 / 8f-2): hyperplanes, hyperspheres and lines up to dimension 8, dense systems of 2..8 unknowns
              PLANE2 = 15, PLANE5 = 16, PLANE6 = 17, PLANE7 = 18, PLANE8 = 19, SPHERE5 = 20, SPHERE6 = 21, SPHERE7 = 22, SPHERE8 = 23,
              LINE4 = 24, LINE5 = 25, LINE6 = 26, LINE7 = 27, LINE8 = 28, DENSE2 = 29, DENSE3 = 30, DENSE4 = 31, DENSE7 = 32, DENSE8 = 33, NUM_MODELS = 34 };

// The dimension-templated estimators of the reference as X-macro lists (model id, dimension).  PLANE_ND: the generic branch of
// PlaneParametersEstimator<d> (every d but 3); SPHERE_ND: SphereParametersEstimator<d>::estimateND (every d but 2, 3);
// LINE_ND: LineParametersEstimator<d>; DENSE_N: DenseLinearEquationSystemParametersEstimator<double, n>.
#define LSQR_PLANE_ND_LIST(X) X(PLANE2, 2) X(PLANE4, 4) X(PLANE5, 5) X(PLANE6, 6) X(PLANE7, 7) X(PLANE8, 8)
#define LSQR_SPHERE_ND_LIST(X) X(SPHERE4, 4) X(SPHERE5, 5) X(SPHERE6, 6) X(SPHERE7, 7) X(SPHERE8, 8)
#define LSQR_SPHERE_ALL_LIST(X) X(CIRCLE2, 2) X(SPHERE3, 3) LSQR_SPHERE_ND_LIST(X)
#define LSQR_LINE_ND_LIST(X) X(LINE2, 2) X(LINE3, 3) X(LINE4, 4) X(LINE5, 5) X(LINE6, 6) X(LINE7, 7) X(LINE8, 8)
#define LSQR_DENSE_N_LIST(X) X(DENSE2, 2) X(DENSE3, 3) X(DENSE4, 4) X(DENSE5, 5) X(DENSE6, 6) X(DENSE7, 7) X(DENSE8, 8)
// every model id, for the dispatch switches
#define LSQR_ALL_MODELS(X)                                                                                                    \
  X(PLANE3) X(LINE2D) X(LINE2) X(LINE3) X(CIRCLE2) X(SPHERE3) X(ABSOR) X(RAY) X(PIVOT) X(DENSE5) X(DENSE6) X(USXW) X(USCP) X(SPHERE4) \
  X(PLANE4) X(PLANE2) X(PLANE5) X(PLANE6) X(PLANE7) X(PLANE8) X(SPHERE5) X(SPHERE6) X(SPHERE7) X(SPHERE8) X(LINE4) X(LINE5) X(LINE6)  \
  X(LINE7) X(LINE8) X(DENSE2) X(DENSE3) X(DENSE4) X(DENSE7) X(DENSE8)
#define LSQR_DISPATCH_CASE_(MM) case MM: { CALL(MM); break; }
// switch (model) over every id; the caller defines CALL(MM) around it
#define LSQR_DISPATCH_MODEL(model, CALL_UNUSED) switch (model) { LSQR_ALL_MODELS(LSQR_DISPATCH_CASE_) default: break; }

// family and dimension of a model id (dimension: space dimension, or the number of unknowns of a dense system)
enum : int { FAM_OTHER = 0, FAM_PLANE = 1, FAM_SPHERE = 2, FAM_LINE = 3, FAM_DENSE = 4 };
__host__ __device__ constexpr int model_family(int m) {
  return (m == PLANE3 || m == PLANE4 || m == PLANE2 || (m >= PLANE5 && m <= PLANE8)) ? FAM_PLANE
       : (m == CIRCLE2 || m == SPHERE3 || m == SPHERE4 || (m >= SPHERE5 && m <= SPHERE8)) ? FAM_SPHERE
       : (m == LINE2 || m == LINE3 || (m >= LINE4 && m <= LINE8)) ? FAM_LINE
       : (m == DENSE5 || m == DENSE6 || (m >= DENSE2 && m <= DENSE8)) ? FAM_DENSE : FAM_OTHER;
}
__host__ __device__ constexpr int model_dim(int m) {
  return m == PLANE3 ? 3 : m == PLANE4 ? 4 : m == PLANE2 ? 2 : (m >= PLANE5 && m <= PLANE8) ? m - PLANE5 + 5
       : m == CIRCLE2 ? 2 : m == SPHERE3 ? 3 : m == SPHERE4 ? 4 : (m >= SPHERE5 && m <= SPHERE8) ? m - SPHERE5 + 5
       : m == LINE2 ? 2 : m == LINE3 ? 3 : (m >= LINE4 && m <= LINE8) ? m - LINE4 + 4
       : m == DENSE5 ? 5 : m == DENSE6 ? 6 : (m >= DENSE2 && m <= DENSE4) ? m - DENSE2 + 2 : (m == DENSE7 || m == DENSE8) ? m - DENSE7 + 7 : 0;
}

// dim = doubles per datum, P = parameters, K = minimal subset, HQ = doubles of a prepared
// fp64 hypothesis, Q32 = floats of a hoisted fp32 hypothesis.
struct ModelInfo { int D, P, K, HQ, Q32; };
__host__ __device__ constexpr ModelInfo model_info(int m) {
  const int d = model_dim(m);
  switch (model_family(m)) {
    case FAM_PLANE:  return {d, 2 * d, d, 2 * d, d + 1};
    case FAM_SPHERE: return {d, d + 1, d + 1, d + 5, d + 2};   // prepared: centre, radius and four squared-distance thresholds (prepare_sphere)
    case FAM_LINE:   return {d, 2 * d, 2, 2 * d, d == 2 ? 3 : (d == 3 ? 9 : 2 * d)};   // fp32: 2-D form, Pluecker form, literal form (k_fast.cu)
    // DenseLinearEquationSystemParametersEstimator<double, n>: datum = AugmentedRow (n coefficients, right-hand side)
    case FAM_DENSE:  return {d + 1, d, d, d, d + 2};
    default: break;
  }
  switch (m) {
    case LINE2D:  return {2, 4, 2, 4, 3};
    case ABSOR:   return {6, 7, 3, 12, 12};
    case RAY:     return {6, 3, 2, 3, 3};
    case PIVOT:   return {12, 6, 3, 6, 6};
    // SingleUnknownPointTargetUSCalibrationParametersEstimator (cross-wire phantom): datum = [R2 (9), t2 (3), u, v],
    // parameters [t1, t3, omega_z, omega_y, omega_x, m_x, m_y, m_x R3(:,1), m_y R3(:,2), R3(:,3)]
    case USXW:    return {14, 20, 4, 12, 12};
    // CalibratedPointerTargetUSCalibrationParametersEstimator: datum = [R2 (9), t2 (3), u, v, p (3)],
    // parameters [t3, omega_z, omega_y, omega_x, m_x, m_y, m_x R3(:,1), m_y R3(:,2), R3(:,3)]
    case USCP:    return {17, 17, 3, 9, 9};
  }
  return {0, 0, 0, 0, 0};
}
// Which components are positions (shifted by the centre c at ingest and in the refine moments); directions / rotations are not.
__host__ __device__ inline bool centred_component(int model, int d) {
  switch (model) {
    case RAY: return d < 3;
    case PIVOT: return d >= 9;
    case USXW: return d >= 9 && d < 12;       // t2; rotation entries and pixel coordinates stay
    case USCP: return false;                  // t2 and p enter as p - t2 with no free translation to absorb a shift
    default: return model_family(model) != FAM_DENSE;   // rows of a linear system: a shift would change the solution
  }
}
template <int M> struct Model {
  static constexpr int D = model_info(M).D, P = model_info(M).P, K = model_info(M).K, HQ = model_info(M).HQ, Q32 = model_info(M).Q32;
  static constexpr int FAM = model_family(M), DIM = model_dim(M);
};

// Thresholds of one estimator instance (what the reference keeps in private members).
struct EstCfg {
  double delta;      // SphereParametersEstimator.h / PivotCalibrationParametersEstimator.h: compared against a distance
  double delta2;     // delta*delta, e.g. PlaneParametersEstimator.hxx:17 -- compared against a squared distance
  double cross_eps;  // RayIntersectionParametersEstimator.cxx:14-15: sin(minimalAngularDeviation)^2
  unsigned long long delta2_bits;   // bit pattern of delta2, 0 when delta2 is NaN (below_delta2)
};

constexpr double kEps = 2.220446049250313e-016;      // common/Epsilon.h:19
constexpr double kSphereEps = 1e-9;                  // SphereParametersEstimator.hxx:11
constexpr double kSmallAngle = 0.008726535498373935; // common/Frame.cxx:8
constexpr double kHalfPi = 3.14159265358979323846 / 2.0;  // common/Frame.cxx:10

// ---------------------------------------------------------------------------------------
// Small dense helpers shared by solvers and refine
// ---------------------------------------------------------------------------------------

// Frame(x,y,z,s,qx,qy,qz) rotation entries, common/Frame.cxx:188-198.
__device__ __forceinline__ void quat_to_rot(double s, double qx, double qy, double qz, double* R) {
  R[0] = 1 - 2 * (qy * qy + qz * qz);
  R[1] = 2 * (qx * qy - s * qz);
  R[2] = 2 * (qx * qz + s * qy);
  R[3] = 2 * (qx * qy + s * qz);
  R[4] = 1 - 2 * (qx * qx + qz * qz);
  R[5] = 2 * (qy * qz - s * qx);
  R[6] = 2 * (qx * qz - s * qy);
  R[7] = 2 * (qy * qz + s * qx);
  R[8] = 1 - 2 * (qx * qx + qy * qy);
}

// Frame::getRotationQuaternion, common/Frame.cxx:952-988.
__device__ inline void rot_to_quat(const double* R, double* q) {
  const double lo = kHalfPi - kSmallAngle, hi = kHalfPi + kSmallAngle;
  q[0] = 0.5 * sqrt(R[0] + R[4] + R[8] + 1);
  const double half_theta = acos(q[0]);
  if (!(half_theta > lo && half_theta < hi)) {
    const double denom = 4 * q[0];
    q[1] = (R[7] - R[5]) / denom;
    q[2] = (R[2] - R[6]) / denom;
    q[3] = (R[3] - R[1]) / denom;
  } else {
    int i = 0;
    if (R[4] > R[i * 3 + i]) i = 1;
    if (R[8] > R[i * 3 + i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    const double w = sqrt(R[i * 3 + i] - R[j * 3 + j] - R[k * 3 + k] + 1);
    q[i + 1] = w / 2.0;
    q[j + 1] = (R[i * 3 + j] + R[j * 3 + i]) / (2 * w);
    q[k + 1] = (R[i * 3 + k] + R[k * 3 + i]) / (2 * w);
  }
}

// Cyclic Jacobi, symmetric n x n (row-major a, destroyed); d ascending, eigenvectors in the
// columns of v.  Stands in for vnl_symmetric_eigensystem (PlaneParametersEstimator.hxx:163).
template <int N>
__device__ inline void sym_eig(double* a, double* v, double* d) {
  for (int i = 0; i < N; i++) for (int j = 0; j < N; j++) v[i * N + j] = (i == j) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 100; sweep++) {
    double off = 0.0, diag = 0.0;
    for (int p = 0; p < N; p++) { diag += a[p * N + p] * a[p * N + p]; for (int q = p + 1; q < N; q++) off += a[p * N + q] * a[p * N + q]; }
    if (off <= 1e-34 * diag) break;  // off-diagonal mass below fp64 resolution of the spectrum (also catches off == 0)
    for (int p = 0; p < N; p++) {
      for (int q = p + 1; q < N; q++) {
        const double apq = a[p * N + q];
        if (apq == 0.0) continue;
        const double theta = (a[q * N + q] - a[p * N + p]) / (2.0 * apq);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < N; k++) { const double x = a[k * N + p], y = a[k * N + q]; a[k * N + p] = c * x - s * y; a[k * N + q] = s * x + c * y; }
        for (int k = 0; k < N; k++) { const double x = a[p * N + k], y = a[q * N + k]; a[p * N + k] = c * x - s * y; a[q * N + k] = s * x + c * y; }
        for (int k = 0; k < N; k++) { const double x = v[k * N + p], y = v[k * N + q]; v[k * N + p] = c * x - s * y; v[k * N + q] = s * x + c * y; }
      }
    }
  }
  for (int i = 0; i < N; i++) d[i] = a[i * N + i];
  for (int i = 0; i + 1 < N; i++) {
    int m = i;
    for (int j = i + 1; j < N; j++) if (d[j] < d[m]) m = j;
    if (m != i) {
      double t = d[i]; d[i] = d[m]; d[m] = t;
      for (int k = 0; k < N; k++) { t = v[k * N + i]; v[k * N + i] = v[k * N + m]; v[k * N + m] = t; }
    }
  }
}

// x = pinv(A) b, A (MR x NC, row-major, destroyed), singular values <= tol dropped; returns
// the rank.  One-sided Jacobi.  Stands in for vnl_matrix_inverse + zero_out_absolute + rank
// (PivotCalibrationParametersEstimator.cxx:40-47).
template <int MR, int NC>
__device__ inline int pinv_solve(double* A, const double* b, double tol, double* x) {
  double V[NC * NC], y[NC];
  for (int i = 0; i < NC; i++) for (int j = 0; j < NC; j++) V[i * NC + j] = (i == j) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 60; sweep++) {
    bool rotated = false;
    for (int p = 0; p < NC; p++) {
      for (int q = p + 1; q < NC; q++) {
        double alpha = 0, beta = 0, gamma = 0;
        for (int k = 0; k < MR; k++) { const double ap = A[k * NC + p], aq = A[k * NC + q]; alpha += ap * ap; beta += aq * aq; gamma += ap * aq; }
        if (gamma == 0.0 || fabs(gamma) <= 1e-16 * sqrt(alpha * beta)) continue;
        rotated = true;
        const double zeta = (beta - alpha) / (2.0 * gamma);
        const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
        for (int k = 0; k < MR; k++) { const double xk = A[k * NC + p], yk = A[k * NC + q]; A[k * NC + p] = c * xk - s * yk; A[k * NC + q] = s * xk + c * yk; }
        for (int k = 0; k < NC; k++) { const double xk = V[k * NC + p], yk = V[k * NC + q]; V[k * NC + p] = c * xk - s * yk; V[k * NC + q] = s * xk + c * yk; }
      }
    }
    if (!rotated) break;
  }
  int rank = 0;
  for (int j = 0; j < NC; j++) {
    double s2 = 0, ub = 0;
    for (int k = 0; k < MR; k++) { const double a = A[k * NC + j]; s2 += a * a; ub += a * b[k]; }
    if (sqrt(s2) <= tol) y[j] = 0.0; else { y[j] = ub / s2; rank++; }
  }
  for (int i = 0; i < NC; i++) { double s = 0; for (int j = 0; j < NC; j++) s += V[i * NC + j] * y[j]; x[i] = s; }
  return rank;
}

// Null vector of A (MR x NC, MR < NC, row-major, destroyed) and the number of singular values above tol.  Stands in
// for vnl_svd + zero_out_absolute + rank() + nullvector() (PlaneParametersEstimator.hxx:82-90): vnl_svd keeps NC
// singular values in descending order (the trailing NC-MR are zero) and nullvector() is the last column of V.
template <int MR, int NC>
__device__ inline int null_vector(double* A, double tol, double* x) {
  double V[NC * NC];
  for (int i = 0; i < NC; i++) for (int j = 0; j < NC; j++) V[i * NC + j] = (i == j) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 60; sweep++) {
    bool rotated = false;
    for (int p = 0; p < NC; p++) {
      for (int q = p + 1; q < NC; q++) {
        double alpha = 0, beta = 0, gamma = 0;
        for (int k = 0; k < MR; k++) { const double ap = A[k * NC + p], aq = A[k * NC + q]; alpha += ap * ap; beta += aq * aq; gamma += ap * aq; }
        if (gamma == 0.0 || fabs(gamma) <= 1e-16 * sqrt(alpha * beta)) continue;
        rotated = true;
        const double zeta = (beta - alpha) / (2.0 * gamma);
        const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
        for (int k = 0; k < MR; k++) { const double xk = A[k * NC + p], yk = A[k * NC + q]; A[k * NC + p] = c * xk - s * yk; A[k * NC + q] = s * xk + c * yk; }
        for (int k = 0; k < NC; k++) { const double xk = V[k * NC + p], yk = V[k * NC + q]; V[k * NC + p] = c * xk - s * yk; V[k * NC + q] = s * xk + c * yk; }
      }
    }
    if (!rotated) break;
  }
  int rank = 0, last = 0;
  double wlast = 0.0;
  for (int j = 0; j < NC; j++) {
    double s2 = 0;
    for (int k = 0; k < MR; k++) s2 += A[k * NC + j] * A[k * NC + j];
    const double w = sqrt(s2);
    if (w > tol) rank++;
    if (j == 0 || w <= wlast) { last = j; wlast = w; }
  }
  for (int i = 0; i < NC; i++) x[i] = V[i * NC + last];
  return rank;
}

// ---------------------------------------------------------------------------------------
// estimate(): minimal solvers, one hypothesis per thread.  pts = K data of D doubles in
// subset order.  Returns false for a degenerate subset (reference: empty parameter vector).
// ---------------------------------------------------------------------------------------
template <int M> __device__ bool estimate(const double* pts, const EstCfg& cfg, double* prm);

// PlaneParametersEstimator.hxx:48-69, :107-108
template <> __device__ inline bool estimate<PLANE3>(const double* d, const EstCfg&, double* prm) {
  const double *p0 = d, *p1 = d + 3, *p2 = d + 6;
  const double v10 = p1[0] - p0[0], v11 = p1[1] - p0[1], v12 = p1[2] - p0[2];
  const double v20 = p2[0] - p0[0], v21 = p2[1] - p0[1], v22 = p2[2] - p0[2];
  const double nx = v11 * v22 - v12 * v21;
  const double ny = v12 * v20 - v10 * v22;
  const double nz = v10 * v21 - v11 * v20;
  const double norm = sqrt(nx * nx + ny * ny + nz * nz);
  if (norm < kEps) return false;
  prm[0] = nx / norm; prm[1] = ny / norm; prm[2] = nz / norm;
  prm[3] = p0[0]; prm[4] = p0[1]; prm[5] = p0[2];
  return true;
}

// Line2DParametersEstimator.cxx:11-32
template <> __device__ inline bool estimate<LINE2D>(const double* d, const EstCfg& cfg, double* prm) {
  const double *p0 = d, *p1 = d + 2;
  const double nx = p1[1] - p0[1];
  const double ny = p0[0] - p1[0];
  const double norm_squared = nx * nx + ny * ny;
  if (norm_squared < cfg.delta2) return false;
  const double norm = sqrt(nx * nx + ny * ny);
  prm[0] = nx / norm; prm[1] = ny / norm; prm[2] = p0[0]; prm[3] = p0[1];
  return true;
}

// LineParametersEstimator.hxx:23-48 (separation test through Point::distanceSquared, Point.h:72-74)
template <int DIM> __device__ inline bool estimate_line(const double* d, const EstCfg& cfg, double* prm) {
  const double *p0 = d, *p1 = d + DIM;
  double ds = 0;
  for (int i = 0; i < DIM; i++) { const double t = p0[i] - p1[i]; ds += t * t; }
  if (ds < cfg.delta2) return false;
  double dir_norm = 0.0;
  for (int i = 0; i < DIM; i++) { prm[i] = p0[i] - p1[i]; dir_norm += prm[i] * prm[i]; prm[DIM + i] = p0[i]; }
  dir_norm = sqrt(dir_norm);
  for (int i = 0; i < DIM; i++) prm[i] /= dir_norm;
  return true;
}
#define LSQR_DEF_(ID, DIM) template <> __device__ inline bool estimate<ID>(const double* d, const EstCfg& c, double* prm) { return estimate_line<DIM>(d, c, prm); }
LSQR_LINE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_

// SphereParametersEstimator.hxx:80-109
template <> __device__ inline bool estimate<CIRCLE2>(const double* d, const EstCfg&, double* prm) {
  const double *p0 = d, *p1 = d + 2, *p2 = d + 4;
  const double A00 = p0[0] - p1[0], A01 = p0[1] - p1[1];
  const double A10 = p0[0] - p2[0], A11 = p0[1] - p2[1];
  double detA = (A00 * A11 - A01 * A10);
  if (fabs(detA) < kSphereEps) return false;
  detA *= 2.0;
  const double b0 = A00 * (p0[0] + p1[0]) + A01 * (p0[1] + p1[1]);
  const double b1 = A10 * (p0[0] + p2[0]) + A11 * (p0[1] + p2[1]);
  prm[0] = (A11 * b0 - A01 * b1) / detA;
  prm[1] = (A00 * b1 - A10 * b0) / detA;
  prm[2] = sqrt((p0[0] - prm[0]) * (p0[0] - prm[0]) + (p0[1] - prm[1]) * (p0[1] - prm[1]));
  return true;
}

// SphereParametersEstimator.hxx:115-163
template <> __device__ inline bool estimate<SPHERE3>(const double* d, const EstCfg&, double* prm) {
  const double *p0 = d, *p1 = d + 3, *p2 = d + 6, *p3 = d + 9;
  const double A00 = p0[0] - p1[0], A01 = p0[1] - p1[1], A02 = p0[2] - p1[2];
  const double A10 = p0[0] - p2[0], A11 = p0[1] - p2[1], A12 = p0[2] - p2[2];
  const double A20 = p0[0] - p3[0], A21 = p0[1] - p3[1], A22 = p0[2] - p3[2];
  const double CT00 = A11 * A22 - A12 * A21;
  const double CT10 = A12 * A20 - A10 * A22;
  const double CT20 = A10 * A21 - A11 * A20;
  double detA = A00 * CT00 + A01 * CT10 + A02 * CT20;
  if (fabs(detA) < kSphereEps) return false;
  detA *= 2;
  const double CT01 = A02 * A21 - A01 * A22;
  const double CT11 = A00 * A22 - A02 * A20;
  const double CT21 = A01 * A20 - A00 * A21;
  const double CT02 = A01 * A12 - A02 * A11;
  const double CT12 = A02 * A10 - A00 * A12;
  const double CT22 = A00 * A11 - A01 * A10;
  const double b0 = A00 * (p0[0] + p1[0]) + A01 * (p0[1] + p1[1]) + A02 * (p0[2] + p1[2]);
  const double b1 = A10 * (p0[0] + p2[0]) + A11 * (p0[1] + p2[1]) + A12 * (p0[2] + p2[2]);
  const double b2 = A20 * (p0[0] + p3[0]) + A21 * (p0[1] + p3[1]) + A22 * (p0[2] + p3[2]);
  prm[0] = (CT00 * b0 + CT01 * b1 + CT02 * b2) / detA;
  prm[1] = (CT10 * b0 + CT11 * b1 + CT12 * b2) / detA;
  prm[2] = (CT20 * b0 + CT21 * b1 + CT22 * b2) / detA;
  prm[3] = sqrt(((p0[0] - prm[0]) * (p0[0] - prm[0])) + ((p0[1] - prm[1]) * (p0[1] - prm[1])) + ((p0[2] - prm[2]) * (p0[2] - prm[2])));
  return true;
}

// One side of the orthonormal-triad construction, AbsoluteOrientationParametersEstimator.cxx:24-51 / :53-81.
// VNL helpers as published: normalize() scales by 1/sqrt(sum x^2); dot_product / magnitude sum left to right.
__device__ inline bool triad(const double* P0, const double* P1, const double* P2, double* Rm, double* mean) {
  double x[3], y[3], z[3];
  for (int i = 0; i < 3; i++) mean[i] = (P0[i] + P1[i] + P2[i]) / 3.0;
  for (int i = 0; i < 3; i++) x[i] = P0[i] - mean[i];
  double s = 0.0; for (int i = 0; i < 3; i++) s += x[i] * x[i];
  if (s != 0.0) { const double inv = 1.0 / sqrt(s); for (int i = 0; i < 3; i++) x[i] = inv * x[i]; }
  for (int i = 0; i < 3; i++) y[i] = P1[i] - mean[i];
  double dot = 0.0; for (int i = 0; i < 3; i++) dot += y[i] * x[i];
  for (int i = 0; i < 3; i++) y[i] = y[i] - x[i] * dot;
  s = 0.0; for (int i = 0; i < 3; i++) s += y[i] * y[i];
  if (s != 0.0) { const double inv = 1.0 / sqrt(s); for (int i = 0; i < 3; i++) y[i] = inv * y[i]; }
  z[0] = x[1] * y[2] - x[2] * y[1];
  z[1] = x[2] * y[0] - x[0] * y[2];
  z[2] = x[0] * y[1] - x[1] * y[0];
  s = 0.0; for (int i = 0; i < 3; i++) s += z[i] * z[i];
  if (sqrt(s) < kEps) return false;
  for (int i = 0; i < 3; i++) { Rm[i * 3 + 0] = x[i]; Rm[i * 3 + 1] = y[i]; Rm[i * 3 + 2] = z[i]; }
  return true;
}

// AbsoluteOrientationParametersEstimator.cxx:14-101 (triad construction, NOT Horn -- SURVEY.md 8a-8)
template <> __device__ inline bool estimate<ABSOR>(const double* d, const EstCfg&, double* prm) {
  double R1[9], R2[9], R[9], m1[3], m2[3], q[4];
  if (!triad(d + 0, d + 6, d + 12, R1, m1)) return false;
  if (!triad(d + 3, d + 9, d + 15, R2, m2)) return false;
  for (int i = 0; i < 3; i++)
    for (int k = 0; k < 3; k++) { double s = 0.0; for (int j = 0; j < 3; j++) s += R2[i * 3 + j] * R1[k * 3 + j]; R[i * 3 + k] = s; }
  for (int i = 0; i < 3; i++) { double s = 0.0; for (int j = 0; j < 3; j++) s += R[i * 3 + j] * m1[j]; prm[4 + i] = m2[i] - s; }
  rot_to_quat(R, q);
  prm[0] = q[0]; prm[1] = q[1]; prm[2] = q[2]; prm[3] = q[3];
  return true;
}

// RayIntersectionParametersEstimator.cxx:23-70
template <> __device__ inline bool estimate<RAY>(const double* d, const EstCfg& cfg, double* prm) {
  const double *p1 = d, *n1 = d + 3, *p2 = d + 6, *n2 = d + 9;
  const double p210 = p2[0] - p1[0], p211 = p2[1] - p1[1], p212 = p2[2] - p1[2];
  const double c0 = n1[1] * n2[2] - n1[2] * n2[1];
  const double c1 = n1[2] * n2[0] - n1[0] * n2[2];
  const double c2 = n1[0] * n2[1] - n1[1] * n2[0];
  const double denominator = c0 * c0 + c1 * c1 + c2 * c2;
  if (denominator < cfg.cross_eps) return false;
  const double t1 = (c0 * (p211 * n2[2] - p212 * n2[1]) - c1 * (p210 * n2[2] - p212 * n2[0]) + c2 * (p210 * n2[1] - p211 * n2[0])) / denominator;
  const double t2 = (c0 * (p211 * n1[2] - p212 * n1[1]) - c1 * (p210 * n1[2] - p212 * n1[0]) + c2 * (p210 * n1[1] - p211 * n1[0])) / denominator;
  if (t1 < 0 || t2 < 0) return false;
  prm[0] = (p1[0] + t1 * n1[0] + p2[0] + t2 * n2[0]) / 2.0;
  prm[1] = (p1[1] + t1 * n1[1] + p2[1] + t2 * n2[1]) / 2.0;
  prm[2] = (p1[2] + t1 * n1[2] + p2[2] + t2 * n2[2]) / 2.0;
  return true;
}

// PivotCalibrationParametersEstimator.cxx:9-51: rows [R_i | -I], rhs -t_i, pseudo-inverse, rank < 6 fails.
template <> __device__ inline bool estimate<PIVOT>(const double* d, const EstCfg&, double* prm) {
  double A[9 * 6], b[9];
  for (int i = 0; i < 54; i++) A[i] = 0.0;
  for (int i = 0; i < 3; i++) {
    const double* f = d + 12 * i;
    for (int r = 0; r < 3; r++) {
      for (int c = 0; c < 3; c++) A[(3 * i + r) * 6 + c] = f[3 * r + c];
      A[(3 * i + r) * 6 + 3 + r] = -1.0;
      b[3 * i + r] = -f[9 + r];
    }
  }
  return pinv_solve<9, 6>(A, b, kEps, prm) >= 6;
}

// DenseLinearEquationSystemParametersEstimator.hxx:17-49: n rows -> A x = b through the pseudo-inverse,
// singular values <= EPS zeroed, rank < n fails.
template <int N> __device__ inline bool estimate_dense(const double* d, double* prm) {
  double A[N * N], b[N];
  for (int i = 0; i < N; i++) { for (int j = 0; j < N; j++) A[i * N + j] = d[i * (N + 1) + j]; b[i] = d[i * (N + 1) + N]; }
  return pinv_solve<N, N>(A, b, kEps, prm) >= N;
}
#define LSQR_DEF_(ID, N) template <> __device__ inline bool estimate<ID>(const double* d, const EstCfg&, double* prm) { return estimate_dense<N>(d, prm); }
LSQR_DENSE_N_LIST(LSQR_DEF_)
#undef LSQR_DEF_

// R <- U V^T of its SVD (closest rotation in the Frobenius norm, SinglePointTargetUSCalibrationParametersEstimator
// .cxx:226-229), as the orthogonal polar factor R (R^T R)^(-1/2).
__device__ inline void closest_rotation(double* R) {
  double S[9], V[9], ev[3], W[9], out[9];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { double s = 0; for (int k = 0; k < 3; k++) s += R[k * 3 + i] * R[k * 3 + j]; S[i * 3 + j] = s; }
  sym_eig<3>(S, V, ev);
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { double s = 0; for (int k = 0; k < 3; k++) s += V[i * 3 + k] * V[j * 3 + k] / sqrt(ev[k]); W[i * 3 + j] = s; }
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { double s = 0; for (int k = 0; k < 3; k++) s += R[i * 3 + k] * W[k * 3 + j]; out[i * 3 + j] = s; }
  for (int i = 0; i < 9; i++) R[i] = out[i];
}

// SinglePointTargetUSCalibrationParametersEstimator.cxx:204-250 (and :862-900): scale factors, re-orthonormalised
// rotation and Euler angles from the first six unknowns [m_x R3(:,1), m_y R3(:,2)] of the linear solution;
// out = [omega_z, omega_y, omega_x, m_x, m_y, m_x R3(:,1), m_y R3(:,2), R3(:,3)] (14 values).
__device__ inline void us_rotation_part(const double* x, double* out) {
  const double smallAngle = 0.008726535498373935, halfPI = 1.5707963267948966192313216916398;
  double r1[3], r2[3], r3[3], R3[9];
  for (int i = 0; i < 3; i++) { r1[i] = x[i]; r2[i] = x[3 + i]; }
  const double m_x = sqrt(r1[0] * r1[0] + r1[1] * r1[1] + r1[2] * r1[2]);
  double inv = 1.0 / m_x; for (int i = 0; i < 3; i++) r1[i] = inv * r1[i];
  const double m_y = sqrt(r2[0] * r2[0] + r2[1] * r2[1] + r2[2] * r2[2]);
  inv = 1.0 / m_y; for (int i = 0; i < 3; i++) r2[i] = inv * r2[i];
  r3[0] = r1[1] * r2[2] - r1[2] * r2[1];
  r3[1] = r1[2] * r2[0] - r1[0] * r2[2];
  r3[2] = r1[0] * r2[1] - r1[1] * r2[0];
  for (int i = 0; i < 3; i++) { R3[i * 3 + 0] = r1[i]; R3[i * 3 + 1] = r2[i]; R3[i * 3 + 2] = r3[i]; }
  closest_rotation(R3);
  double omega_z, omega_x;
  const double omega_y = atan2(-R3[6], sqrt(R3[0] * R3[0] + R3[3] * R3[3]));
  if (fabs(omega_y - halfPI) > smallAngle && fabs(omega_y + halfPI) > smallAngle) {
    const double cy = cos(omega_y);
    omega_z = atan2(R3[3] / cy, R3[0] / cy);
    omega_x = atan2(R3[7] / cy, R3[8] / cy);
  } else {
    omega_z = 0;
    omega_x = atan2(R3[1], R3[4]);
  }
  out[0] = omega_z; out[1] = omega_y; out[2] = omega_x; out[3] = m_x; out[4] = m_y;
  out[5] = m_x * R3[0]; out[6] = m_x * R3[3]; out[7] = m_x * R3[6];
  out[8] = m_y * R3[1]; out[9] = m_y * R3[4]; out[10] = m_y * R3[7];
  out[11] = R3[2]; out[12] = R3[5]; out[13] = R3[8];
}
// cross-wire: x = [m_x R3(:,1), m_y R3(:,2), t3, t1] -> the 20 parameters (.cxx:251-268)
__device__ inline bool us_post(const double* x, double* prm) {
  prm[0] = x[9]; prm[1] = x[10]; prm[2] = x[11];
  prm[3] = x[6]; prm[4] = x[7]; prm[5] = x[8];
  us_rotation_part(x, prm + 6);
  bool ok = true;
  for (int i = 0; i < 20; i++) ok = ok && (prm[i] == prm[i]);
  return ok;
}
// calibrated pointer: x = [m_x R3(:,1), m_y R3(:,2), t3] -> the 17 parameters (.cxx:903-920)
__device__ inline bool uscp_post(const double* x, double* prm) {
  prm[0] = x[6]; prm[1] = x[7]; prm[2] = x[8];
  us_rotation_part(x, prm + 3);
  bool ok = true;
  for (int i = 0; i < 17; i++) ok = ok && (prm[i] == prm[i]);
  return ok;
}

// SinglePointTargetUSCalibrationParametersEstimator.cxx:120-270 with four data: rows [u R2, v R2, R2, -I] x = -t2,
// pseudo-inverse with singular values <= FLT_EPSILON zeroed, rank < 12 fails.
template <> __device__ inline bool estimate<USXW>(const double* d, const EstCfg&, double* prm) {
  double A[144], b[12], x[12];
  for (int i = 0; i < 144; i++) A[i] = 0.0;
  for (int i = 0; i < 4; i++) {
    const double* f = d + 14 * i;
    const double ui = f[12], vi = f[13];
    for (int r = 0; r < 3; r++) {
      double* row = A + (3 * i + r) * 12;
      for (int c = 0; c < 3; c++) { row[c] = f[3 * r + c] * ui; row[3 + c] = f[3 * r + c] * vi; row[6 + c] = f[3 * r + c]; }
      row[9 + r] = -1.0;
      b[3 * i + r] = -f[9 + r];
    }
  }
  if (pinv_solve<12, 12>(A, b, 1.192092896e-07, x) < 12) return false;
  return us_post(x, prm);
}

// PlaneParametersEstimator.hxx:70-108 (every dimension other than 3): [n, d] spans the null space of [p_i, -1]
template <int DIM> __device__ inline bool estimate_plane_nd(const double* d, double* prm) {
  double A[DIM * (DIM + 1)], x[DIM + 1];
  for (int i = 0; i < DIM; i++) { for (int j = 0; j < DIM; j++) A[i * (DIM + 1) + j] = d[i * DIM + j]; A[i * (DIM + 1) + DIM] = -1; }
  if (null_vector<DIM, DIM + 1>(A, kEps, x) < DIM) return false;
  double norm = 0;
  for (int i = 0; i < DIM; i++) norm += x[i] * x[i];
  norm = 1.0 / sqrt(norm);
  for (int i = 0; i < DIM; i++) { prm[i] = x[i] * norm; prm[DIM + i] = d[i]; }
  return true;
}
#define LSQR_DEF_(ID, DIM) template <> __device__ inline bool estimate<ID>(const double* d, const EstCfg&, double* prm) { return estimate_plane_nd<DIM>(d, prm); }
LSQR_PLANE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_

// SphereParametersEstimator.hxx:169-202 (estimateND, every dimension other than 2 and 3): rows p0 - p_i, pseudo-inverse
// with singular values <= EPS zeroed; rank < dim means the points lie in a hyperplane.
template <int DIM> __device__ inline bool estimate_sphere_nd(const double* d, double* prm) {
  double A[DIM * DIM], b[DIM], x[DIM];
  for (int i = 0; i < DIM; i++) {
    b[i] = 0.0;
    for (int j = 0; j < DIM; j++) { A[i * DIM + j] = d[j] - d[(i + 1) * DIM + j]; b[i] += A[i * DIM + j] * (d[j] + d[(i + 1) * DIM + j]); }
  }
  if (pinv_solve<DIM, DIM>(A, b, kEps, x) < DIM) return false;   // EPS of common/Epsilon.h here (:189), not the SPHERE_EPS of the 2-D / 3-D determinant tests
  double rSquared = 0.0;
  for (int i = 0; i < DIM; i++) { prm[i] = x[i] * 0.5; rSquared += (d[i] - prm[i]) * (d[i] - prm[i]); }
  prm[DIM] = sqrt(rSquared);
  return true;
}
#define LSQR_DEF_(ID, DIM) template <> __device__ inline bool estimate<ID>(const double* d, const EstCfg&, double* prm) { return estimate_sphere_nd<DIM>(d, prm); }
LSQR_SPHERE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_

// SinglePointTargetUSCalibrationParametersEstimator.cxx:789-920 with three data: rows [u R2, v R2, R2] x = p - t2,
// singular values <= FLT_EPSILON zeroed, rank < 9 fails.
template <> __device__ inline bool estimate<USCP>(const double* d, const EstCfg&, double* prm) {
  double A[81], b[9], x[9];
  for (int i = 0; i < 3; i++) {
    const double* f = d + 17 * i;
    const double ui = f[12], vi = f[13];
    for (int r = 0; r < 3; r++) {
      double* row = A + (3 * i + r) * 9;
      for (int c = 0; c < 3; c++) { row[c] = f[3 * r + c] * ui; row[3 + c] = f[3 * r + c] * vi; row[6 + c] = f[3 * r + c]; }
      b[3 * i + r] = f[14 + r] - f[9 + r];
    }
  }
  if (pinv_solve<9, 9>(A, b, 1.192092896e-07, x) < 9) return false;
  return uscp_post(x, prm);
}

// ---------------------------------------------------------------------------------------
// agree(): prepare once per hypothesis, test once per (hypothesis, datum)
// ---------------------------------------------------------------------------------------
template <int M> __device__ __forceinline__ void prepare(const double* prm, const EstCfg&, double* hq) {
#pragma unroll
  for (int i = 0; i < Model<M>::P; i++) hq[i] = prm[i];
}
template <> __device__ __forceinline__ void prepare<ABSOR>(const double* prm, const EstCfg&, double* hq) {
  quat_to_rot(prm[0], prm[1], prm[2], prm[3], hq);
  hq[9] = prm[4]; hq[10] = prm[5]; hq[11] = prm[6];
}

// cross-wire: the twelve entries agree() reads -- m_x R3(:,1), m_y R3(:,2), t3, t1
template <> __device__ __forceinline__ void prepare<USXW>(const double* prm, const EstCfg&, double* hq) {
#pragma unroll
  for (int i = 0; i < 6; i++) hq[i] = prm[11 + i];
#pragma unroll
  for (int i = 0; i < 3; i++) { hq[6 + i] = prm[3 + i]; hq[9 + i] = prm[i]; }
}

// calibrated pointer: m_x R3(:,1), m_y R3(:,2), t3
template <> __device__ __forceinline__ void prepare<USCP>(const double* prm, const EstCfg&, double* hq) {
#pragma unroll
  for (int i = 0; i < 6; i++) hq[i] = prm[8 + i];
#pragma unroll
  for (int i = 0; i < 3; i++) hq[6 + i] = prm[i];
}

template <int M> __device__ __forceinline__ bool agree(const double* hq, const double* x, const EstCfg& cfg);

// `v < deltaSquared` for a v that is a square or a sum of squares (v >= +0, +inf or NaN), decided on the integer ALU:
// non-negative doubles order like their bit patterns, a NaN (either sign) has a larger pattern than any finite or infinite
// threshold, and a NaN threshold (delta2_bits = 0) admits nothing -- the same truth table as the reference's double compare,
// without a DSETP on the FP64 pipe, which is the pipe that bounds the validation kernel (11 -> 9 FP64 instructions per plane
// evaluation together with the leading `0 +` of the reference's accumulation loops, which cannot change a square: the only
// value it alters is the sign of a zero).
__device__ __forceinline__ bool below_delta2(double v, const EstCfg& cfg) { return (unsigned long long)__double_as_longlong(v) < cfg.delta2_bits; }

// PlaneParametersEstimator.hxx:196-203
template <int DIM> __device__ __forceinline__ bool agree_plane_nd(const double* h, const double* x, const EstCfg& cfg) {
  double sd = h[0] * (x[0] - h[DIM]);
#pragma unroll
  for (int i = 1; i < DIM; i++) sd += h[i] * (x[i] - h[DIM + i]);
  return below_delta2(sd * sd, cfg);
}
template <> __device__ __forceinline__ bool agree<PLANE3>(const double* h, const double* x, const EstCfg& cfg) { return agree_plane_nd<3>(h, x, cfg); }
#define LSQR_DEF_(ID, DIM) template <> __device__ __forceinline__ bool agree<ID>(const double* h, const double* x, const EstCfg& c) { return agree_plane_nd<DIM>(h, x, c); }
LSQR_PLANE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_
// Line2DParametersEstimator.cxx:119-123
template <> __device__ __forceinline__ bool agree<LINE2D>(const double* h, const double* x, const EstCfg& cfg) {
  const double sd = h[0] * (x[0] - h[2]) + h[1] * (x[1] - h[3]);
  return below_delta2(sd * sd, cfg);
}
// LineParametersEstimator.hxx:135-150
template <int DIM> __device__ __forceinline__ bool agree_line(const double* h, const double* x, const EstCfg& cfg) {
  double v[DIM], v_dot_n, ds;
#pragma unroll
  for (int i = 0; i < DIM; i++) { v[i] = x[i] - h[DIM + i]; v_dot_n = i ? v_dot_n + v[i] * h[i] : v[i] * h[i]; }
#pragma unroll
  for (int i = 0; i < DIM; i++) { const double w = v[i] - v_dot_n * h[i]; ds = i ? ds + w * w : w * w; }
  return below_delta2(ds, cfg);
}
#define LSQR_DEF_(ID, DIM) template <> __device__ __forceinline__ bool agree<ID>(const double* h, const double* x, const EstCfg& c) { return agree_line<DIM>(h, x, c); }
LSQR_LINE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_
// SphereParametersEstimator.hxx:255-264 (a distance against delta, not squared): |sqrt(dl) - r| < delta.
// The square root (a ~20-instruction sequence on the FP64 pipe) decides nothing for a datum whose squared distance is clear
// of both (r - delta)^2 and (r + delta)^2 by more than any rounding of the reference's expression could move it (1e-9
// relative on the squared distance = 5e-10 (r +- delta) on the distance, against the few ulp = 4e-16 r the roundings can move
// it); only data inside those two slivers take the reference's expression literally.  The decision is the reference's for
// every datum.  The four thresholds are prepared once per hypothesis (prepare_sphere) as bit patterns: the squared distance is
// a sum of squares (>= +0, +inf or NaN), so it orders like its bits and the tests run on the integer ALU:
//   bits(dl) > OUT_HI or < OUT_LO : surely outside (NaN and +inf included);   IN_LO < bits(dl) < IN_HI : surely inside.
// A threshold that must not fire is all-ones (never exceeded) or zero (nothing below it): delta <= 0 or NaN, r <= 0 or NaN
// disable all four, a radius within 0.1 % of delta (where the margin on r - delta would not cover its own rounding) the
// three that involve r - delta.  hq = [centre (DIM), r, OUT_HI, OUT_LO, IN_HI, IN_LO].
template <int DIM> __device__ __forceinline__ void prepare_sphere(const double* prm, const EstCfg& cfg, double* hq) {
#pragma unroll
  for (int i = 0; i <= DIM; i++) hq[i] = prm[i];
  const double r = prm[DIM], hi = r + cfg.delta, lo = r - cfg.delta;
  constexpr double kUp = 1.0 + 1e-9, kDn = 1.0 - 1e-9;
  long long out_hi = -1LL, out_lo = 0, in_hi = 0, in_lo = -1LL;
  if (cfg.delta > 0.0 && r > 0.0 && hi < 1e150) {
    out_hi = __double_as_longlong(hi * hi * kUp);
    if (lo > 1e-3 * r) {
      out_lo = __double_as_longlong(lo * lo * kDn);
      in_hi = __double_as_longlong(hi * hi * kDn);
      in_lo = __double_as_longlong(lo * lo * kUp);
    }
  }
  hq[DIM + 1] = __longlong_as_double(out_hi); hq[DIM + 2] = __longlong_as_double(out_lo);
  hq[DIM + 3] = __longlong_as_double(in_hi); hq[DIM + 4] = __longlong_as_double(in_lo);
}
#define LSQR_DEF_(ID, DIM) template <> __device__ __forceinline__ void prepare<ID>(const double* prm, const EstCfg& cfg, double* hq) { prepare_sphere<DIM>(prm, cfg, hq); }
LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
#undef LSQR_DEF_
template <int DIM> __device__ __forceinline__ bool agree_sphere(const double* h, const double* x, const EstCfg& cfg) {
  double dl = (x[0] - h[0]) * (x[0] - h[0]);      // (the reference's leading `0 +` cannot change a non-negative term)
#pragma unroll
  for (int i = 1; i < DIM; i++) dl += ((x[i] - h[i]) * (x[i] - h[i]));
  // only the HIGH words are compared (one 32-bit compare per threshold instead of two chained ones: the integer ALU would
  // otherwise bound the kernel): a strictly larger / smaller high word implies the 64-bit relation, equal high words -- a sliver
  // of 2^-20 relative around a threshold -- fall through to the literal expression
  const unsigned b = (unsigned)__double2hiint(dl);
  if (b > (unsigned)__double2hiint(h[DIM + 1]) || b < (unsigned)__double2hiint(h[DIM + 2])) return false;
  if (b < (unsigned)__double2hiint(h[DIM + 3]) && b > (unsigned)__double2hiint(h[DIM + 4])) return true;
  dl = fabs(sqrt(dl) - h[DIM]);
  return dl < cfg.delta;
}
#define LSQR_DEF_(ID, DIM) template <> __device__ __forceinline__ bool agree<ID>(const double* h, const double* x, const EstCfg& c) { return agree_sphere<DIM>(h, x, c); }
LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
#undef LSQR_DEF_
// AbsoluteOrientationParametersEstimator.cxx:316-327 with Frame::apply, common/Frame.cxx:229-248
template <> __device__ __forceinline__ bool agree<ABSOR>(const double* h, const double* x, const EstCfg& cfg) {
  const double qx = h[0] * x[0] + h[1] * x[1] + h[2] * x[2] + h[9];
  const double qy = h[3] * x[0] + h[4] * x[1] + h[5] * x[2] + h[10];
  const double qz = h[6] * x[0] + h[7] * x[1] + h[8] * x[2] + h[11];
  const double dx = qx - x[3], dy = qy - x[4], dz = qz - x[5];
  return below_delta2(dx * dx + dy * dy + dz * dz, cfg);
}
// RayIntersectionParametersEstimator.cxx:164-179
template <> __device__ __forceinline__ bool agree<RAY>(const double* h, const double* x, const EstCfg& cfg) {
  const double* p = x; const double* n = x + 3;
  const double t = n[0] * (h[0] - p[0]) + n[1] * (h[1] - p[1]) + n[2] * (h[2] - p[2]);
  const double dx = h[0] - p[0] - t * n[0];
  const double dy = h[1] - p[1] - t * n[1];
  const double dz = h[2] - p[2] - t * n[2];
  return t >= 0 && below_delta2(dx * dx + dy * dy + dz * dz, cfg);
}
// PivotCalibrationParametersEstimator.cxx:108-123 (Frame::apply then Vector::l2Norm, common/Vector.h:134-139)
template <> __device__ __forceinline__ bool agree<PIVOT>(const double* h, const double* x, const EstCfg& cfg) {
  const double qx = x[0] * h[0] + x[1] * h[1] + x[2] * h[2] + x[9];
  const double qy = x[3] * h[0] + x[4] * h[1] + x[5] * h[2] + x[10];
  const double qz = x[6] * h[0] + x[7] * h[1] + x[8] * h[2] + x[11];
  const double rx = qx - h[3], ry = qy - h[4], rz = qz - h[5];
  double s = 0;
  s += rx * rx; s += ry * ry; s += rz * rz;
  // sqrt(s) < delta is decided by s against delta^2 wherever s is clear of it by more than the roundings of the literal
  // expression can matter (1e-9 relative against a few ulp); the square root is taken only inside that sliver
  if (cfg.delta > 0.0) {
    if (s < cfg.delta2 * (1.0 - 1e-9)) return true;
    if (s > cfg.delta2 * (1.0 + 1e-9)) return false;
  }
  return sqrt(s) < cfg.delta;
}

// SinglePointTargetUSCalibrationParametersEstimator.cxx:71-107: qInT = (T2*T3)*q with VNL's left-to-right
// accumulation; products with the constant 0 / 1 entries of the homogeneous matrices are exact and left out.
template <> __device__ __forceinline__ bool agree<USXW>(const double* h, const double* x, const EstCfg& cfg) {
  const double u = x[12], v = x[13];
  double s = 0;
  double err[3];
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const double a = x[3 * i], b = x[3 * i + 1], c = x[3 * i + 2];
    const double M0 = a * h[0] + b * h[1] + c * h[2];
    const double M1 = a * h[3] + b * h[4] + c * h[5];
    const double M3 = a * h[6] + b * h[7] + c * h[8] + x[9 + i];
    err[i] = (M0 * u + M1 * v + M3) - h[9 + i];
  }
  s = err[0] * err[0] + err[1] * err[1] + err[2] * err[2];
  return below_delta2(s, cfg);
}

// SinglePointTargetUSCalibrationParametersEstimator.cxx:726-761: the same product, compared with the measured pointer tip
template <> __device__ __forceinline__ bool agree<USCP>(const double* h, const double* x, const EstCfg& cfg) {
  const double u = x[12], v = x[13];
  double err[3];
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const double a = x[3 * i], b = x[3 * i + 1], c = x[3 * i + 2];
    const double M0 = a * h[0] + b * h[1] + c * h[2];
    const double M1 = a * h[3] + b * h[4] + c * h[5];
    const double M3 = a * h[6] + b * h[7] + c * h[8] + x[9 + i];
    err[i] = (M0 * u + M1 * v + M3) - x[14 + i];
  }
  const double s = err[0] * err[0] + err[1] * err[1] + err[2] * err[2];
  return below_delta2(s, cfg);
}

// DenseLinearEquationSystemParametersEstimator.hxx:111-119
template <int N> __device__ __forceinline__ bool agree_dense(const double* h, const double* x, const EstCfg& cfg) {
  double sum = 0.0;
#pragma unroll
  for (int i = 0; i < N; i++) sum += x[i] * h[i];
  sum -= x[N];
  return fabs(sum) < cfg.delta;
}
#define LSQR_DEF_(ID, N) template <> __device__ __forceinline__ bool agree<ID>(const double* h, const double* x, const EstCfg& c) { return agree_dense<N>(h, x, c); }
LSQR_DENSE_N_LIST(LSQR_DEF_)
#undef LSQR_DEF_

// ---------------------------------------------------------------------------------------
// Subset generation
// ---------------------------------------------------------------------------------------

// high 32 bits of the 64-bit product a * b
__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

// Philox4x32-10 (Salmon et al., SC'11): counter-based, so hypothesis h's subset depends only
// on (seed, h) -- independent of how hypotheses are split over thread blocks or GPUs, or of
// whether the host draws it (compute() fetches the records of its first round ahead of the upload).
__host__ __device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u; key.y += 0xBB67AE85u;
  }
  return ctr;
}

// K distinct indices in [0, n), in draw order (the reference also hands estimate() its subset
// in draw order, RANSAC.hxx:56-68).  Draw j picks uniformly among the n-j indices not yet taken.
template <int K>
__host__ __device__ __forceinline__ void sample_subset(uint64_t gidx, uint64_t seed, uint32_t n, int32_t* out) {
  constexpr int NB = (K + 3) / 4;   // one counter block per four draws
  uint32_t rnd[4 * NB];
#pragma unroll
  for (int blk = 0; blk < NB; blk++) {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)gidx, (uint32_t)(gidx >> 32), (uint32_t)blk, 0u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    rnd[4 * blk] = r.x; rnd[4 * blk + 1] = r.y; rnd[4 * blk + 2] = r.z; rnd[4 * blk + 3] = r.w;
  }
  uint32_t sorted[K];
#pragma unroll
  for (int j = 0; j < K; j++) {
    uint32_t v = mulhi32(rnd[j], n - j);  // uniform in [0, n-j)
#pragma unroll
    for (int i = 0; i < j; i++) if (v >= sorted[i]) v++;  // skip taken indices, ascending
    out[j] = (int32_t)v;
    int pos = j;
#pragma unroll
    for (int i = j - 1; i >= 0; i--) if (sorted[i] > v) { sorted[i + 1] = sorted[i]; pos = i; }
    sorted[pos] = v;
  }
}

__device__ __forceinline__ uint64_t binom(uint32_t n, int k) {
  if ((uint32_t)k > n) return 0;
  uint64_t r = 1;
  for (int i = 0; i < k; i++) r = r * (n - i) / (i + 1);
  return r;
}

// Subset with lexicographic rank `rank` among ascending K-tuples of {0..n-1}: the enumeration
// order of RANSAC<T,S>::computeAllChoices (RANSAC.hxx:197-213).  Tuples whose j-th element is
// below c (given the earlier elements) number C(n-lo, K-j) - C(n-c, K-j); binary search on c.
template <int K>
__device__ inline void unrank_lex(uint64_t rank, uint32_t n, int32_t* out) {
  uint32_t lo = 0;
#pragma unroll
  for (int j = 0; j < K; j++) {
    const int kk = K - j;
    const uint64_t total = binom(n - lo, kk);
    // largest c in [lo, n-kk] with  total - C(n-c, kk) <= rank
    uint32_t a = lo, b = n - kk;
    while (a < b) {
      const uint32_t mid = a + (b - a + 1) / 2;
      if (total - binom(n - mid, kk) <= rank) a = mid; else b = mid - 1;
    }
    rank -= total - binom(n - a, kk);
    out[j] = (int32_t)a;
    lo = a + 1;
  }
}

}  // namespace lsqr
