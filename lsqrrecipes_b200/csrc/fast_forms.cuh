// fp32 "fast mode" arithmetic shared by the scoring kernels (k_fast.cu) and the batched small-problem kernel (k_batch.cu):
// packed point-pair operations, the hoisted per-hypothesis constants of every estimator (hoist32<M>), its residual form on point
// pairs (Eval<M>) and the counting forms.  See the header comment of k_fast.cu for why each form looks the way it does.
#pragma once
#include "engine.h"

namespace lsqr {

// ---- packed pair arithmetic (sm_100 f32x2) -------------------------------------------------
struct f2 { unsigned long long v; };
__device__ __forceinline__ f2 splat(float a) { f2 r; asm("mov.b64 %0, {%1, %1};" : "=l"(r.v) : "f"(a)); return r; }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { f2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v)); return r; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { f2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
__device__ __forceinline__ f2 sub2(f2 a, f2 b) { f2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
__device__ __forceinline__ void halves(f2 a, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a.v)); }
__device__ __forceinline__ f2 join(float lo, float hi) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi)); return r; }

// ---- hoisted fp32 hypotheses ---------------------------------------------------------------
// Q32 floats per hypothesis, computed once in fp64 from the raw parameters, the data centre c
// (positions are stored as x - c in fp32) and the thresholds:
//   PLANE3   (nx,ny,nz, delta - n.(a-c))      the kernels form s' = s + delta and test 0 <= s' < 2 delta (see count_carry)
//   LINE2D   (nx,ny, -n.(a-c))                 |s| < delta (two FFMA2 per pair leave the ALU pipe as the limit either way; measured: the carry form is 4 % slower here)
//   LINE2    (n_perp, -n_perp.(a-c))            the 2-D line form on the perpendicular of the unit direction
//   LINE3    3 x (n_k, -n_j, -((a-c) x n)_i)    Pluecker form
//   CIRCLE/SPHERE (ctr-c, -(r-delta)^2, 2^32 - bits(4 r delta)): t' = d^2 - (r-delta)^2, inlier <=> 0 <= t' < 4 r delta  (<=> |d - r| < delta)
//   ABSOR    (R[9], R c1 + t - c2)
//   RAY      (x - c)
//   PIVOT    (tDRF, -(tW - c))
//   DENSE n  (x[n], -1, delta): a.x - b + delta as n+1 FMAs over the (uncentred) augmented row
//   USXW     (m_x R3(:,1), m_y R3(:,2), t3, -(t1 - c))
//   USCP     (m_x R3(:,1), m_y R3(:,2), t3)
template <int M> __device__ __forceinline__ void hoist32(const double* p, const double* c, const EstCfg& cfg, float* q);
template <> __device__ __forceinline__ void hoist32<PLANE3>(const double* p, const double* c, const EstCfg& cfg, float* q) {
  q[0] = (float)p[0]; q[1] = (float)p[1]; q[2] = (float)p[2];
  q[3] = (float)(cfg.delta - (p[0] * (p[3] - c[0]) + p[1] * (p[4] - c[1]) + p[2] * (p[5] - c[2])));   // shifted residual s + delta
}
template <int DIM> __device__ __forceinline__ void hoist_plane_nd(const double* p, const double* c, const EstCfg& cfg, float* q) {
  double s = 0;
  for (int i = 0; i < DIM; i++) { q[i] = (float)p[i]; s += p[i] * (p[DIM + i] - c[i]); }
  q[DIM] = (float)(cfg.delta - s);
}
#define LSQR_DEF_(ID, DIM) template <> __device__ __forceinline__ void hoist32<ID>(const double* p, const double* c, const EstCfg& cfg, float* q) { hoist_plane_nd<DIM>(p, c, cfg, q); }
LSQR_PLANE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_
template <> __device__ __forceinline__ void hoist32<LINE2D>(const double* p, const double* c, const EstCfg&, float* q) {
  q[0] = (float)p[0]; q[1] = (float)p[1];
  q[2] = (float)(-(p[0] * (p[2] - c[0]) + p[1] * (p[3] - c[1])));
}
// kD lines (LineParametersEstimator.hxx:135-150: |v - (v.n) n|^2 < delta^2 with v = x - a).  The fast mode takes the direction as
// the unit vector it is for every hypothesis estimate() produces (it is re-normalised here, a no-op then), which makes the
// rejection |v x n| in 3-D and |n_perp . v| in 2-D:
//   d = 2: the 2-D line form, s = n_perp . x - n_perp . (a - c)                                        2 FMA per datum
//   d = 3: Pluecker form, w = x X n - (a - c) X n, every component two FMAs on a hoisted constant:      6 + 3 FMA per datum
// instead of the 9 / 12 operations of the literal form.  The validation mode keeps the literal form (models.cuh).
template <> __device__ __forceinline__ void hoist32<LINE2>(const double* p, const double* c, const EstCfg&, float* q) {
  const double inv = 1.0 / sqrt(p[0] * p[0] + p[1] * p[1]);
  const double px = -p[1] * inv, py = p[0] * inv;
  q[0] = (float)px; q[1] = (float)py;
  q[2] = (float)(-(px * (p[2] - c[0]) + py * (p[3] - c[1])));
}
template <> __device__ __forceinline__ void hoist32<LINE3>(const double* p, const double* c, const EstCfg&, float* q) {
  const double inv = 1.0 / sqrt(p[0] * p[0] + p[1] * p[1] + p[2] * p[2]);
  const double n[3] = {p[0] * inv, p[1] * inv, p[2] * inv}, a[3] = {p[3] - c[0], p[4] - c[1], p[5] - c[2]};
  // w_i = x_j n_k - x_k n_j - (a_j n_k - a_k n_j)   with (i, j, k) cyclic: constants (n_k, -n_j, -m_i) per component
  for (int i = 0; i < 3; i++) {
    const int j = (i + 1) % 3, k = (i + 2) % 3;
    q[3 * i] = (float)n[k]; q[3 * i + 1] = (float)(-n[j]); q[3 * i + 2] = (float)(-(a[j] * n[k] - a[k] * n[j]));
  }
}
// d >= 4: the literal form, constants (n, a - c)
template <int DIM> __device__ __forceinline__ void hoist_line_nd(const double* p, const double* c, float* q) {
  for (int i = 0; i < DIM; i++) { q[i] = (float)p[i]; q[DIM + i] = (float)(p[DIM + i] - c[i]); }
}
#define LSQR_DEF_(ID, DIM) template <> __device__ __forceinline__ void hoist32<ID>(const double* p, const double* c, const EstCfg&, float* q) { hoist_line_nd<DIM>(p, c, q); }
LSQR_DEF_(LINE4, 4) LSQR_DEF_(LINE5, 5) LSQR_DEF_(LINE6, 6) LSQR_DEF_(LINE7, 7) LSQR_DEF_(LINE8, 8)
#undef LSQR_DEF_
// |d - r| < delta  <=>  (r - delta)^2 <= d^2 < (r + delta)^2  <=>  0 <= t' < 4 r delta  with  t' = d^2 - (r - delta)^2: the chain
// starts at -(r - delta)^2 and the datum is an inlier iff bits(t') < bits(4 r delta) as unsigned integers (count_carry; the
// threshold is per hypothesis).  r < delta: no lower bound, t' = d^2 (>= +0) against (r + delta)^2 -- relative, like every other
// form, so the decisions do not depend on the data's scale.  An empty interval (delta not positive -- SphereParametersEstimator.hxx:20
// keeps its sign --, r + delta <= 0, NaN) is stored as window 0: nothing agrees.
template <int DIM> __device__ __forceinline__ void hoist_sphere(const double* p, const double* c, const EstCfg& cfg, float* q) {
  for (int i = 0; i < DIM; i++) q[i] = (float)(p[i] - c[i]);
  const double r = p[DIM], dl = cfg.delta;
  double start = 0.0, width = 0.0;
  if (dl > 0) {
    if (r >= dl) { start = -(r - dl) * (r - dl); width = 4.0 * r * dl; }
    else if (r + dl > 0) width = (r + dl) * (r + dl);
  }
  q[DIM] = (float)start;
  const float wf = (float)width;
  // stored ready for count_carry: 2^32 - bits(window); 0 = nothing agrees (window not positive, or NaN)
  q[DIM + 1] = __uint_as_float((wf > 0.0f) ? 0u - __float_as_uint(wf) : 0u);
}
#define LSQR_DEF_(ID, DIM) template <> __device__ __forceinline__ void hoist32<ID>(const double* p, const double* c, const EstCfg& cfg, float* q) { hoist_sphere<DIM>(p, c, cfg, q); }
LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
#undef LSQR_DEF_
template <> __device__ __forceinline__ void hoist32<ABSOR>(const double* p, const double* c, const EstCfg&, float* q) {
  double R[9];
  quat_to_rot(p[0], p[1], p[2], p[3], R);
  for (int i = 0; i < 9; i++) q[i] = (float)R[i];
  for (int i = 0; i < 3; i++) q[9 + i] = (float)(R[3 * i] * c[0] + R[3 * i + 1] * c[1] + R[3 * i + 2] * c[2] + p[4 + i] - c[3 + i]);
}
template <> __device__ __forceinline__ void hoist32<RAY>(const double* p, const double* c, const EstCfg&, float* q) {
  for (int i = 0; i < 3; i++) q[i] = (float)(p[i] - c[i]);
}
// PivotCalibrationParametersEstimator.cxx:108-123 compares the unsquared distance with delta: a negative one admits nothing, which
// the squared form cannot see -- NaN constants then (every residual NaN: an outlier)
template <> __device__ __forceinline__ void hoist32<PIVOT>(const double* p, const double* c, const EstCfg& cfg, float* q) {
  const bool none = cfg.delta < 0.0;
  for (int i = 0; i < 3; i++) {   // the chain starts at -(tW - c)
    q[i] = none ? __int_as_float(0x7fffffff) : (float)p[i];
    q[3 + i] = none ? __int_as_float(0x7fffffff) : (float)(-(p[3 + i] - c[9 + i]));
  }
}

template <int N> __device__ __forceinline__ void hoist_dense(const double* p, const EstCfg& cfg, float* q) {
  for (int i = 0; i < N; i++) q[i] = (float)p[i];
  q[N] = -1.0f;
  q[N + 1] = (float)cfg.delta;   // the chain starts at +delta: s' = a.x - b + delta, inlier <=> bits(s') < bits(2 delta)
}
#define LSQR_DEF_(ID, N) template <> __device__ __forceinline__ void hoist32<ID>(const double* p, const double*, const EstCfg& cfg, float* q) { hoist_dense<N>(p, cfg, q); }
LSQR_DENSE_N_LIST(LSQR_DEF_)
#undef LSQR_DEF_

template <> __device__ __forceinline__ void hoist32<USXW>(const double* p, const double* c, const EstCfg&, float* q) {
  for (int i = 0; i < 6; i++) q[i] = (float)p[11 + i];
  for (int i = 0; i < 3; i++) { q[6 + i] = (float)p[3 + i]; q[9 + i] = (float)(-(p[i] - c[9 + i])); }   // the chain starts at -(t1 - c)
}

template <> __device__ __forceinline__ void hoist32<USCP>(const double* p, const double*, const EstCfg&, float* q) {
  for (int i = 0; i < 6; i++) q[i] = (float)p[8 + i];
  for (int i = 0; i < 3; i++) q[6 + i] = (float)p[i];
}

// slot of the per-hypothesis counting window among the hoisted constants (-1: the window is 2 delta for every hypothesis)
template <int M> constexpr int thr_slot() { return model_family(M) == FAM_SPHERE ? model_dim(M) + 1 : -1; }

// ---- per-model residual forms on point pairs ----------------------------------------------
struct Thr2 { f2 delta, neg_delta2; float fdelta; };
// The threshold the fp32 kernels compare with |s| and count the shifted forms against (window 2 delta): a delta that is not
// positive admits nothing.  (EstCfg.delta is |delta| where the reference squares it; the dense systems compare |a.x - b| with
// delta itself, and a negative window would have admitted every s' >= 0.)
__host__ __device__ __forceinline__ float fp32_delta(const EstCfg& cfg) { return cfg.delta > 0.0 ? (float)cfg.delta : 0.0f; }

// signed(): g with inlier <=> g < 0.   For PLANE3 / LINE2D, dist(): s with inlier <=> |s| < delta.
template <int M> struct Eval;
template <> struct Eval<PLANE3> {
  static constexpr bool kHasAbsForm = true;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = true;   // dist() is s + delta (the hoisted constant carries the shift)
  __device__ static __forceinline__ f2 dist(const f2* q, const f2* x) { return fma2(q[0], x[0], fma2(q[1], x[1], fma2(q[2], x[2], q[3]))); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) { const f2 s = sub2(dist(q, x), t.delta); return fma2(s, s, t.neg_delta2); }
};
template <int DIM> struct EvalPlaneND {
  static constexpr bool kHasAbsForm = true;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = true;   // dist() is s + delta (the hoisted constant carries the shift)
  __device__ static __forceinline__ f2 dist(const f2* q, const f2* x) {
    f2 s = q[DIM];
#pragma unroll
    for (int i = DIM - 1; i >= 0; i--) s = fma2(q[i], x[i], s);
    return s;
  }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) { const f2 s = sub2(dist(q, x), t.delta); return fma2(s, s, t.neg_delta2); }
};
#define LSQR_DEF_(ID, DIM) template <> struct Eval<ID> : EvalPlaneND<DIM> {};
LSQR_PLANE_ND_LIST(LSQR_DEF_)
#undef LSQR_DEF_
template <> struct Eval<LINE2D> {
  static constexpr bool kHasAbsForm = true;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = false;
  __device__ static __forceinline__ f2 dist(const f2* q, const f2* x) { return fma2(q[0], x[0], fma2(q[1], x[1], q[2])); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) { const f2 s = dist(q, x); return fma2(s, s, t.neg_delta2); }
};
// Every instruction below takes at most ONE datum operand: in the constant-bank kernel the data are uniform registers and an
// FFMA2 / FADD2 encodes a single uniform source -- a second one forces ptxas to fetch the datum with LDC into ordinary
// registers (indexed constant loads, a quarter of the throughput: measured on the pivot estimator, 0.7 -> 2.3 T evals/s).
template <> struct Eval<LINE2> {     // the 2-D line form on the perpendicular (see hoist32<LINE2>)
  static constexpr bool kHasAbsForm = true;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = false;
  __device__ static __forceinline__ f2 dist(const f2* q, const f2* x) { return fma2(q[0], x[0], fma2(q[1], x[1], q[2])); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) { const f2 s = dist(q, x); return fma2(s, s, t.neg_delta2); }
};
template <> struct Eval<LINE3> {     // Pluecker form: |x X n - m|^2 - delta^2 (see hoist32<LINE3>)
  static constexpr bool kHasAbsForm = false;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = false;
  __device__ static __forceinline__ f2 dist(const f2*, const f2*) { return splat(0.f); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) {
    f2 g = t.neg_delta2;
#pragma unroll
    for (int i = 0; i < 3; i++) {
      const f2 w = fma2(x[(i + 1) % 3], q[3 * i], fma2(x[(i + 2) % 3], q[3 * i + 1], q[3 * i + 2]));
      g = fma2(w, w, g);
    }
    return g;
  }
};
// d >= 4: the literal form of LineParametersEstimator.hxx:135-150, v = x - a, w = v - (v.n) n, |w|^2 - delta^2: 4d operations
template <int DIM> struct EvalLineND {
  static constexpr bool kHasAbsForm = false;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = false;
  __device__ static __forceinline__ f2 dist(const f2*, const f2*) { return splat(0.f); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) {
    f2 v[DIM];
#pragma unroll
    for (int i = 0; i < DIM; i++) v[i] = sub2(x[i], q[DIM + i]);
    f2 vn = mul2(v[0], q[0]);
#pragma unroll
    for (int i = 1; i < DIM; i++) vn = fma2(v[i], q[i], vn);
    const f2 nvn = sub2(splat(0.f), vn);
    f2 g = t.neg_delta2;
#pragma unroll
    for (int i = 0; i < DIM; i++) { const f2 w = fma2(nvn, q[i], v[i]); g = fma2(w, w, g); }
    return g;
  }
};
template <> struct Eval<LINE4> : EvalLineND<4> {};
template <> struct Eval<LINE5> : EvalLineND<5> {};
template <> struct Eval<LINE6> : EvalLineND<6> {};
template <> struct Eval<LINE7> : EvalLineND<7> {};
template <> struct Eval<LINE8> : EvalLineND<8> {};
// t' = d^2 - (r - delta)^2 (chain start q[DIM]); per-hypothesis window q[DIM + 1] = 4 r delta (see hoist_sphere)
template <int DIM> __device__ __forceinline__ f2 sphere_t(const f2* q, const f2* x) {
  f2 t = q[DIM];
#pragma unroll
  for (int i = 0; i < DIM; i++) { const f2 w = sub2(x[i], q[i]); t = fma2(w, w, t); }
  return t;
}
template <int DIM> struct EvalSphere {
  static constexpr bool kHasAbsForm = true;
  static constexpr int kThr = DIM + 1;      // per-hypothesis window, stored as 2^32 - bits(window)
  static constexpr bool kShifted = true;    // dist() is already the shifted residual
  __device__ static __forceinline__ f2 dist(const f2* q, const f2* x) { return sphere_t<DIM>(q, x); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2&) { return sphere_t<DIM>(q, x); }
};
#define LSQR_DEF_(ID, DIM) template <> struct Eval<ID> : EvalSphere<DIM> {};
LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
#undef LSQR_DEF_
template <> struct Eval<ABSOR> {
  static constexpr bool kHasAbsForm = false;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = false;
  __device__ static __forceinline__ f2 dist(const f2*, const f2*) { return splat(0.f); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) {
    f2 g = t.neg_delta2;
#pragma unroll
    for (int i = 0; i < 3; i++) {
      const f2 d = sub2(fma2(q[3 * i], x[0], fma2(q[3 * i + 1], x[1], fma2(q[3 * i + 2], x[2], q[9 + i]))), x[3 + i]);
      g = fma2(d, d, g);
    }
    return g;
  }
};
template <> struct Eval<RAY> {
  static constexpr bool kHasAbsForm = false;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = false;
  __device__ static __forceinline__ f2 dist(const f2*, const f2*) { return splat(0.f); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) {
    const f2 vx = sub2(q[0], x[0]), vy = sub2(q[1], x[1]), vz = sub2(q[2], x[2]);
    const f2 tt = fma2(x[3], vx, fma2(x[4], vy, mul2(x[5], vz)));
    const f2 ntt = sub2(splat(0.f), tt);
    const f2 dx = fma2(ntt, x[3], vx), dy = fma2(ntt, x[4], vy), dz = fma2(ntt, x[5], vz);
    const f2 g = fma2(dx, dx, fma2(dy, dy, fma2(dz, dz, t.neg_delta2)));
    // t >= 0 && dist^2 < delta^2  <=>  g < 0 && -t < 0: the sign bit of g AND -t.  A NaN on either side (canonical, positive)
    // is an outlier: an infinite record coordinate makes -t infinite and g NaN, and a select of the larger would keep -inf.
    f2 r;
    asm("and.b64 %0, %1, %2;" : "=l"(r.v) : "l"(g.v), "l"(ntt.v));
    return r;
  }
};
template <> struct Eval<PIVOT> {
  static constexpr bool kHasAbsForm = false;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = false;
  __device__ static __forceinline__ f2 dist(const f2*, const f2*) { return splat(0.f); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) {
    f2 g = t.neg_delta2;
#pragma unroll
    for (int i = 0; i < 3; i++) {
      const f2 d = add2(fma2(q[0], x[3 * i], fma2(q[1], x[3 * i + 1], fma2(q[2], x[3 * i + 2], q[3 + i]))), x[9 + i]);
      g = fma2(d, d, g);
    }
    return g;
  }
};

// |a.x - b| < delta in the shifted form: n+1 FMAs, q[N] = -1 multiplies the right-hand side, the chain starts at q[N+1] = delta
// (DenseLinearEquationSystemParametersEstimator.hxx:111-119)
template <int N> __device__ __forceinline__ f2 dense_dist(const f2* q, const f2* x) {
  f2 s = fma2(q[N], x[N], q[N + 1]);
#pragma unroll
  for (int i = N - 1; i >= 0; i--) s = fma2(q[i], x[i], s);
  return s;
}
template <int N> struct EvalDense {
  static constexpr bool kHasAbsForm = true;
  static constexpr int kThr = -1;   // threshold = delta for every hypothesis
  static constexpr bool kShifted = true;
  __device__ static __forceinline__ f2 dist(const f2* q, const f2* x) { return dense_dist<N>(q, x); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) { const f2 s = sub2(dist(q, x), t.delta); return fma2(s, s, t.neg_delta2); }
};
#define LSQR_DEF_(ID, N) template <> struct Eval<ID> : EvalDense<N> {};
LSQR_DENSE_N_LIST(LSQR_DEF_)
#undef LSQR_DEF_

// cross-wire: e = R2 (u c1 + v c2 + t3) + t2 - t1, |e|^2 - delta^2   (21 FMA-pipe operations)
template <> struct Eval<USXW> {
  static constexpr bool kHasAbsForm = false;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = false;
  __device__ static __forceinline__ f2 dist(const f2*, const f2*) { return splat(0.f); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) {
    f2 w[3];
#pragma unroll
    for (int k = 0; k < 3; k++) w[k] = fma2(x[12], q[k], fma2(x[13], q[3 + k], q[6 + k]));
    f2 g = t.neg_delta2;
#pragma unroll
    for (int r = 0; r < 3; r++) {
      const f2 e = add2(fma2(x[3 * r], w[0], fma2(x[3 * r + 1], w[1], fma2(x[3 * r + 2], w[2], q[9 + r]))), x[9 + r]);
      g = fma2(e, e, g);
    }
    return g;
  }
};

// calibrated pointer: e = R2 (u c1 + v c2 + t3) + (t2 - p); the difference t2 - p is formed in fp64 when the fp32 copy is written
template <> struct Eval<USCP> {
  static constexpr bool kHasAbsForm = false;
  static constexpr int kThr = -1;
  static constexpr bool kShifted = false;
  __device__ static __forceinline__ f2 dist(const f2*, const f2*) { return splat(0.f); }
  __device__ static __forceinline__ f2 signed_(const f2* q, const f2* x, const Thr2& t) {
    f2 w[3];
#pragma unroll
    for (int k = 0; k < 3; k++) w[k] = fma2(x[12], q[k], fma2(x[13], q[3 + k], q[6 + k]));
    f2 g = t.neg_delta2;
#pragma unroll
    for (int r = 0; r < 3; r++) {
      const f2 e = add2(fma2(x[3 * r], w[0], fma2(x[3 * r + 1], w[1], mul2(x[3 * r + 2], w[2]))), x[9 + r]);   // rows 9..11 of the fp32 copy hold t2 - p (ingest_kernel)
      g = fma2(e, e, g);
    }
    return g;
  }
};

template <int M> __device__ __forceinline__ float hyp_thr(const f2* q, float delta) {
  if constexpr (Eval<M>::kThr >= 0) { float lo, hi; halves(q[Eval<M>::kThr], lo, hi); return lo; }
  else return delta;
}
template <int M> __device__ __forceinline__ float hyp_thr(const float* q, float delta) {
  if constexpr (Eval<M>::kThr >= 0) return q[Eval<M>::kThr];
  else return delta;
}
// 2^32 - bits(window) for count_carry: the window is 2 delta for every hypothesis, or the hypothesis' own (hypersphere family)
template <int M, class Q> __device__ __forceinline__ uint32_t hyp_negk(const Q* q, uint32_t negk_delta) {
  if constexpr (Eval<M>::kThr >= 0) return __float_as_uint(hyp_thr<M>(q, 0.f));
  else return negk_delta;
}
// FSETP + predicated IADD on two residuals, written in PTX so that ptxas keeps the 2-instruction form.
__device__ __forceinline__ void count_abs_lt(uint32_t& cnt, f2 s, float delta) {
  float a, b;
  halves(s, a, b);
  asm("{\n\t.reg .pred p0, p1;\n\t"
      "setp.lt.f32 p0, %1, %3;\n\tsetp.lt.f32 p1, %2, %3;\n\t"
      "@p0 add.u32 %0, %0, 1;\n\t@p1 add.u32 %0, %0, 1;\n\t}"
      : "+r"(cnt) : "f"(fabsf(a)), "f"(fabsf(b)), "f"(delta));
}
// Outlier counting through the carry chain, for residuals in the shifted form s' = s + delta (inlier <=> 0 <= s' < 2 delta
// <=> bits(s') < bits(2 delta) as unsigned integers: negative floats, NaN and everything >= 2 delta have larger bit patterns).
// The counter is the HIGH word of a 64-bit value whose low word is replaced by bits(s') before a 64-bit add of
// 2^32 - bits(2 delta): the carry out of the low word is the outlier flag.  ptxas turns two such steps into
//   IADD3 RZ, P0, PT, s0, -K, RZ ;  IADD3 RZ, P1, PT, s1, -K, RZ ;  IADD3.X cnt, PT, PT, RZ, RZ, cnt, P1, P0
// i.e. three ALU instructions per two residuals with ONE register operand each (no value but the counter is written).
__device__ __forceinline__ void count_carry(unsigned long long& acc, f2 s, uint32_t negk) {   // negk = 2^32 - bits(2 delta)
  float a, b;
  halves(s, a, b);
  asm("{\n\t.reg .b64 w, k;\n\t.reg .b32 lo, hi;\n\t"
      "cvt.u64.u32 k, %3;\n\t"
      "mov.b64 {lo, hi}, %0;\n\tmov.b64 w, {%1, hi};\n\tadd.u64 %0, w, k;\n\t"
      "mov.b64 {lo, hi}, %0;\n\tmov.b64 w, {%2, hi};\n\tadd.u64 %0, w, k;\n\t}"
      : "+l"(acc) : "r"(__float_as_uint(a)), "r"(__float_as_uint(b)), "r"(negk));
}
// Three ALU instructions per two residuals: the two FSET.BF results are summed as raw words by one IADD3
// (raw += 0x3F800000 per inlier).  0x3F800000 = 127 << 23, so raw holds (127 k mod 512) << 23 and k is recovered
// by cb_raw_decode() as long as no more than 511 inliers were summed since the last decode.
__device__ __forceinline__ void count_abs_lt4_raw(uint32_t& raw, f2 s01, f2 s23, float delta) {
  float a, b, c, d;
  halves(s01, a, b);
  halves(s23, c, d);
  asm("{\n\t.reg .f32 f0, f1, f2, f3;\n\t.reg .b32 t0, t1, t2, t3;\n\t"
      "set.lt.f32.f32 f0, %1, %5;\n\tset.lt.f32.f32 f1, %2, %5;\n\tset.lt.f32.f32 f2, %3, %5;\n\tset.lt.f32.f32 f3, %4, %5;\n\t"
      "mov.b32 t0, f0;\n\tmov.b32 t1, f1;\n\tmov.b32 t2, f2;\n\tmov.b32 t3, f3;\n\t"
      "add.u32 t0, t0, t1;\n\tadd.u32 %0, %0, t0;\n\tadd.u32 t2, t2, t3;\n\tadd.u32 %0, %0, t2;\n\t}"
      : "+r"(raw) : "f"(fabsf(a)), "f"(fabsf(b)), "f"(fabsf(c)), "f"(fabsf(d)), "f"(delta));
}
__device__ __forceinline__ uint32_t cb_raw_decode(uint32_t raw) { return ((raw >> 23) * 383u) & 511u; }   // 127 * 383 = 1 (mod 512)
__device__ __forceinline__ void count_sign(uint32_t& cnt, f2 g) {
  float a, b;
  halves(g, a, b);
  cnt += __float_as_uint(a) >> 31;
  cnt += __float_as_uint(b) >> 31;
}

}  // namespace lsqr
