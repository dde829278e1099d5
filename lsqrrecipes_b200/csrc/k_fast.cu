// fp32 "fast mode" consensus: the hot kernel of the whole path (RANSAC.hxx:94-99 / :239-244).
//
// Formulation (chosen by measurement: tools/ptx_lab, tools/consensus_lab*.cu, profiles/r01_ptx_lab_rf_model.txt):
//   * An sm_100a SM sub-partition issues one warp instruction per cycle; a packed fma.rn.f32x2 (SASS FFMA2) holds both
//     halves of the FMA pipe for two cycles, an ALU instruction the 16-lane ALU pipe for two, and the register file delivers
//     two 32-bit operands per cycle.  The cost of an evaluation is therefore the FFMA2s of its residual plus whatever the
//     threshold test and the count cost in issue slots, ALU cycles and register reads.
//   * Arithmetic is packed over PAIRS OF POINTS (f32x2); the hypothesis constants are hoisted once per hypothesis in fp64
//     (hoist32_kernel) so that the residual is a bare FMA chain.
//   * Large requests (H >= kCbMinHyps) take the CONSTANT-BANK kernel (consensus_cb_kernel): the points of one launch sit in
//     the 64 KB constant bank, a point pair is a UNIFORM-register operand (LDCU -> `FFMA2 R, R.F32, UR.F32x2, R.F32x2`) and an
//     FFMA2 reads 2-3 registers instead of the 5-6 it reads when the pair comes out of shared memory.
//   * Small requests (adaptive RANSAC rounds, tests) take consensus32_kernel: point tiles staged by TMA bulk copies into a
//     2-deep shared-memory ring (TileRing, bulk_copy.cuh), pairs through LDS.128.
//   * Counting, three ALU instructions per two residuals in the hot kernel:
//       - hyperplanes, dense systems, hypersphere family: CARRY CHAIN (count_carry) -- the residual arrives shifted (the hoisted
//         constant carries +delta; hypersphere: t' = d^2 - (r - delta)^2), inlier <=> bits(s') < bits(window) unsigned (window 2 delta,
//         or the hypothesis' own 4 r delta); two carry-only IADD3 and one IADD3.X with the two predicates as carry-ins, one
//         register operand each;
//       - 2-D lines (Line2D, Line<2>): two FFMA2 per pair leave the ALU pipe as the limit of any 3-ALU count, so of every four
//         point pairs two are tested as |s| < delta (two FSET.BF and one three-input IADD3 on their raw words,
//         count_abs_lt4_raw, decoded by cb_raw_decode) and two through the sign of s^2 - delta^2 (one more FFMA2, LEA.HI):
//         5 + 5 pipe slots per two pairs instead of 4 + 6;
//       - vector residuals (lines of 3 and more dimensions, absolute orientation, ray, pivot, ultrasound): the FMA chain starts
//         at -delta^2, so the SIGN BIT of the sum is the decision and LEA.HI adds it (count_sign).
//     Both kernels evaluate the same predicate per model, so their counts are bit-identical (tested).
// Tensor cores are deliberately unused: contraction depth <= 8 (BASELINE.json north_star: <= 4 for its estimators), and
// TF32 / bf16 operands would destroy a residual of 0.5 on coordinates of 1000.
#include "engine.h"
#include "bulk_copy.cuh"
#include "fast_forms.cuh"

#include <algorithm>
#include <cmath>
#include <mutex>

namespace lsqr {

template <int M>
__global__ void hoist32_kernel(const double* __restrict__ hyp64, size_t hld, uint32_t H, DataView dv, EstCfg cfg, float* __restrict__ hyp32) {
  constexpr int P = Model<M>::P, Q = Model<M>::Q32;
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  double prm[P], c[kMaxDim];
  float q[Q];
#pragma unroll
  for (int j = 0; j < P; j++) prm[j] = hyp64[(size_t)j * hld + h];
#pragma unroll
  for (int j = 0; j < kMaxDim; j++) c[j] = dv.center[j];
  hoist32<M>(prm, c, cfg, q);
  const bool ok = prm[0] == prm[0];
  // layout: groups of four constants, [ceil(Q/4)][hld] float4 -> one 16-byte load per group in the consensus kernels
  float4* out = reinterpret_cast<float4*>(hyp32);
#pragma unroll
  for (int g = 0; g < (Q + 3) / 4; g++) {
    float v[4];
#pragma unroll
    for (int c = 0; c < 4; c++) v[c] = (ok && 4 * g + c < Q) ? q[4 * g + c] : ((4 * g + c == thr_slot<M>()) ? 0.0f : __int_as_float(0x7fc00000));   // degenerate: NaN constants, empty window
    out[(size_t)g * hld + h] = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// Reads the Q hoisted constants of hypothesis h (NaN for h >= H: never agrees).
template <int Q>
__device__ __forceinline__ void load_hyp32(const float* __restrict__ hyp, size_t hld, uint32_t h, uint32_t H, float* q) {
  const float4* in = reinterpret_cast<const float4*>(hyp);
  const float nan = __int_as_float(0x7fc00000);
#pragma unroll
  for (int g = 0; g < (Q + 3) / 4; g++) {
    const float4 v = (h < H) ? __ldg(in + (size_t)g * hld + h) : make_float4(nan, nan, nan, nan);
    const float t[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int c = 0; c < 4; c++) if (4 * g + c < Q) q[4 * g + c] = t[c];
  }
}

void launch_hoist32(int model, const double* hyp64, size_t hld, uint32_t H, const DataView& dv, const EstCfg& cfg, float* hyp32, cudaStream_t s) {
  if (H == 0) return;
  const unsigned blocks = (H + 255) / 256;
#define CALL(MM) hoist32_kernel<MM><<<blocks, 256, 0, s>>>(hyp64, hld, H, dv, cfg, hyp32)
  LSQR_DISPATCH_MODEL(model, CALL)
#undef CALL
}

// PPI = point pairs per inner iteration (2 -> one LDS.128 per component, 1 -> one LDS.64)
template <int M, int R, int THREADS, int TILE, int PPI>
__global__ void __launch_bounds__(THREADS) consensus32_kernel(const float* __restrict__ soa, size_t ld, uint32_t tiles_total, uint32_t tiles_per_chunk,
                                                               const float* __restrict__ hyp, size_t hld, uint32_t H, float delta, float delta2,
                                                               uint32_t* __restrict__ counts) {
  constexpr int D = Model<M>::D, Q = Model<M>::Q32;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bars[2];

  const int tid = threadIdx.x;
  const uint32_t hbase = blockIdx.x * (THREADS * R);
  f2 q[R][Q];
  uint32_t cnt[R];
  unsigned long long out[R];   // kShifted models: outliers in the high word (count_carry)
#pragma unroll
  for (int r = 0; r < R; r++) {
    const uint32_t h = hbase + r * THREADS + tid;
    float qs[Q];
    load_hyp32<Q>(hyp, hld, h, H, qs);
#pragma unroll
    for (int j = 0; j < Q; j++) q[r][j] = splat(qs[j]);
    cnt[r] = 0;
    out[r] = 0ull;
  }
  Thr2 thr;
  thr.delta = splat(delta); thr.neg_delta2 = splat(-delta2); thr.fdelta = delta;
  const uint32_t negk = 0u - __float_as_uint(2.0f * delta);   // 2^32 - bits(2 delta)

  const uint32_t t0 = blockIdx.y * tiles_per_chunk;
  const uint32_t t1 = min(t0 + tiles_per_chunk, tiles_total);
  TileRing<D, TILE, float> ring{soa, ld, t0, t1, reinterpret_cast<float*>(smem_raw), bars, tid};
  ring.start();
  for (uint32_t t = t0; t < t1; t++) {
    const float* tl = ring.wait(t);
#pragma unroll 1
    for (int i = 0; i < TILE; i += 2 * PPI) {
      f2 x[PPI][D];
#pragma unroll
      for (int d = 0; d < D; d++) {
        if constexpr (PPI == 4) {
          const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(tl + d * TILE + i), w = *reinterpret_cast<const ulonglong2*>(tl + d * TILE + i + 4);
          x[0][d].v = v.x; x[1][d].v = v.y; x[2][d].v = w.x; x[3][d].v = w.y;
        } else if constexpr (PPI == 2) {
          const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(tl + d * TILE + i);
          x[0][d].v = v.x; x[1][d].v = v.y;
        } else {
          x[0][d].v = *reinterpret_cast<const unsigned long long*>(tl + d * TILE + i);
        }
      }
#pragma unroll
      for (int r = 0; r < R; r++) {
#pragma unroll
        for (int u = 0; u < PPI; u++) {
          // the predicate must be the constant-bank kernel's for every (hypothesis, datum): shifted models count through the
          // carry chain; the 2-D lines take |s| < delta for the first two point pairs of every group of four and the sign of
          // s^2 - delta^2 for the other two (kMixed, see consensus_cb_kernel); vector residuals the sign of the sum
          if constexpr (Eval<M>::kShifted) count_carry(out[r], Eval<M>::dist(q[r], x[u]), hyp_negk<M>(q[r], negk));
          else if (Eval<M>::kHasAbsForm && (u & 2) == 0) count_abs_lt(cnt[r], Eval<M>::dist(q[r], x[u]), hyp_thr<M>(q[r], thr.fdelta));
          else count_sign(cnt[r], Eval<M>::signed_(q[r], x[u], thr));
        }
      }
    }
    ring.release();
  }
#pragma unroll
  for (int r = 0; r < R; r++) {
    const uint32_t h = hbase + r * THREADS + tid;
    // NaN padding counts as outliers; delta = 0 (bits(2 delta) = 0: no carry ever) admits nothing, like |s| < 0
    if constexpr (Eval<M>::kShifted) cnt[r] = hyp_negk<M>(q[r], negk) ? (t1 - t0) * (uint32_t)TILE - (uint32_t)(out[r] >> 32) : 0u;
    if (h < H && cnt[r]) atomicAdd(&counts[h], cnt[r]);
  }
}

template <int M, int R, int THREADS, int TILE, int PPI>
static int run_consensus32(const DataView& dv, const float* hyp, size_t hld, uint32_t H, const EstCfg& cfg, uint32_t* counts, int num_sms, cudaStream_t s) {
  const uint32_t tiles_total = (uint32_t)(dv.span / TILE);
  const uint32_t hyp_blocks = (H + THREADS * R - 1) / (THREADS * R);
  const TileChunks plan = plan_tile_chunks(tiles_total, hyp_blocks, num_sms);
  const size_t smem = 2 * (size_t)Model<M>::D * TILE * sizeof(float);
  auto kern = consensus32_kernel<M, R, THREADS, TILE, PPI>;
  allow_dynamic_smem(kern, smem);
  kern<<<dim3(hyp_blocks, plan.chunks), THREADS, smem, s>>>(dv.soa32, dv.ld, tiles_total, plan.tiles_per_chunk, hyp, hld, H, fp32_delta(cfg), (float)cfg.delta2,
                                                             counts);
  return 1;
}


// ---- constant-bank variant ---------------------------------------------------------------------
// One launch scores ALL hypotheses of the request against the `cp` points whose components sit in
// the constant bank ([D][cp] floats, cp a multiple of 16, copied there device-to-device before the
// launch).  grid = (hypothesis blocks) x (point sub-chunks of `sub` points); every thread keeps R
// hypotheses as scalars (broadcast .F32 operands), the point pairs are uniform registers.
constexpr int kCbFloats = 16320;              // 65280 B of the 64 KB bank
constexpr uint32_t kCbMinHyps = 98304;        // below this the per-launch overhead outweighs the gain
__constant__ float4 c_tile[kCbFloats / 4];
static std::mutex g_cb_mutex[kMaxDevices];    // the bank is per device, not per context

#ifndef LSQR_CB_MINBLOCKS
#define LSQR_CB_MINBLOCKS 5
#endif
constexpr uint32_t kCbRawMaxSub = 496;       // <= 511 inliers per raw counter, multiple of 16
template <int M> constexpr uint32_t cb_points() { return (uint32_t)(kCbFloats / Model<M>::D / 16 * 16); }   // points per launch

template <int M, int R, int THREADS, int PPI>
__global__ void __launch_bounds__(THREADS, LSQR_CB_MINBLOCKS) consensus_cb_kernel(uint32_t npts, uint32_t sub, const float* __restrict__ hyp, size_t hld, uint32_t H,
                                                                float delta, float delta2, uint32_t* __restrict__ counts) {
  constexpr int D = Model<M>::D, Q = Model<M>::Q32;
  constexpr uint32_t cp = cb_points<M>();
  const int tid = threadIdx.x;
  const uint32_t hbase = blockIdx.x * (THREADS * R);
  float qf[R][Q];
  uint32_t cnt[R], sgn[R];     // sgn: the sign-counted half of the mixed form
  unsigned long long out[R];   // kShifted models: outliers in the high word (count_carry)
#pragma unroll
  for (int r = 0; r < R; r++) {
    load_hyp32<Q>(hyp, hld, hbase + r * THREADS + tid, H, qf[r]);
    cnt[r] = 0; sgn[r] = 0;
    out[r] = 0ull;
  }
  const uint32_t negk = 0u - __float_as_uint(2.0f * delta);   // 2^32 - bits(2 delta)
  Thr2 thr;
  thr.delta = splat(delta); thr.neg_delta2 = splat(-delta2); thr.fdelta = delta;
  // one induction variable in units of 2*PPI points; the component offsets are immediates (cp is a multiple of 16)
  const uint32_t p0 = blockIdx.y * sub, p1 = min(p0 + sub, npts);
  const int g0 = (int)(p0 / (2 * PPI)), g1 = (int)(p1 / (2 * PPI));
  // raw-sum counting (count_abs_lt4_raw) holds 9 bits: the host keeps sub <= kCbRawMaxSub points per CTA
  constexpr bool kCarry = Eval<M>::kShifted;
  constexpr bool kRaw = Eval<M>::kHasAbsForm && !kCarry;
  static_assert(!kRaw || PPI % 4 == 0, "the mixed count alternates in groups of four point pairs");
  // points of group g (2*PPI points) from the constant bank: uniform loads, the values live in uniform registers
  auto load_group = [&](f2 (&x)[PPI][D], int g) {
#pragma unroll
    for (int d = 0; d < D; d++) {
      if constexpr (PPI % 2 == 0) {
#pragma unroll
        for (int j = 0; j < PPI / 2; j++) {
          const float4 v = c_tile[d * (int)(cp / 4) + (PPI / 2) * g + j];
          x[2 * j][d] = join(v.x, v.y); x[2 * j + 1][d] = join(v.z, v.w);
        }
      } else {
        const float2 v = reinterpret_cast<const float2*>(c_tile)[d * (int)(cp / 2) + g];
        x[0][d] = join(v.x, v.y);
      }
    }
  };
  auto score_group = [&](const f2 (&x)[PPI][D]) {
#pragma unroll
    for (int r = 0; r < R; r++) {
      f2 q[Q];
#pragma unroll
      for (int j = 0; j < Q; j++) q[j] = splat(qf[r][j]);
      if constexpr (kCarry) {
        const uint32_t nk = hyp_negk<M>(qf[r], negk);
#pragma unroll
        for (int u = 0; u < PPI; u++) count_carry(out[r], Eval<M>::dist(q, x[u]), nk);
      } else if constexpr (kRaw) {
        // kMixed: of every four point pairs two are tested as |s| < delta (2 FFMA2 + 3 ALU instructions per pair: ALU-bound on
        // its own) and two through the sign of s^2 - delta^2 (3 FFMA2 + 2 ALU: FMA-bound on its own); together 5 + 5 pipe slots
        // per two pairs instead of 4 + 6
        const float th = hyp_thr<M>(qf[r], thr.fdelta);
#pragma unroll
        for (int u = 0; u < PPI; u += 4) {
          count_abs_lt4_raw(cnt[r], Eval<M>::dist(q, x[u]), Eval<M>::dist(q, x[u + 1]), th);
          count_sign(sgn[r], Eval<M>::signed_(q, x[u + 2], thr));
          count_sign(sgn[r], Eval<M>::signed_(q, x[u + 3], thr));
        }
      } else {
#pragma unroll
        for (int u = 0; u < PPI; u++) count_sign(cnt[r], Eval<M>::signed_(q, x[u], thr));
      }
    }
  };
#pragma unroll 1
  for (int g = g0; g < g1; g++) {
    f2 x[PPI][D];
    load_group(x, g);
    score_group(x);
  }
#pragma unroll
  for (int r = 0; r < R; r++) {
    const uint32_t h = hbase + r * THREADS + tid;
    // NaN padding counts as outliers; delta = 0 (bits(2 delta) = 0: no carry ever) admits nothing, like |s| < 0
    if constexpr (kCarry) cnt[r] = hyp_negk<M>(qf[r], negk) ? (uint32_t)(g1 - g0) * (2u * PPI) - (uint32_t)(out[r] >> 32) : 0u;
    if constexpr (kRaw) cnt[r] = cb_raw_decode(cnt[r]) + sgn[r];
    if (h < H && cnt[r]) atomicAdd(&counts[h], cnt[r]);
  }
}

// ---- early exit of the constant-bank path (Prune, engine.h) ------------------------------------
constexpr uint32_t kPruneThreads = 1024;

// The hoisted constants of the hypothesis that holds the arg-max key (index relative to the launch) -> one column (hld 1).
__global__ void prune_seed_kernel(const unsigned long long* __restrict__ key, const float4* __restrict__ hyp, size_t hld, int groups, float4* __restrict__ col) {
  const uint32_t h = 0xFFFFFFFFu - (uint32_t)(*key & 0xFFFFFFFFull);
  if ((int)threadIdx.x < groups) col[threadIdx.x] = hyp[threadIdx.x * hld + h];
}

// Survivors among the live hypotheses [1024 b, 1024 b + 1024): i stays iff cnt[i] + rem >= L (rem: data not scored yet).
__global__ void __launch_bounds__(kPruneThreads) prune_tally_kernel(const uint32_t* __restrict__ cnt, uint32_t H, uint32_t rem, uint32_t L, uint32_t* __restrict__ tally) {
  const uint32_t i = blockIdx.x * kPruneThreads + threadIdx.x;
  const int k = __syncthreads_count(i < H && cnt[i] + rem >= L);
  if (threadIdx.x == 0) tally[blockIdx.x] = (uint32_t)k;
}

// Order-preserving compaction of the live list (constants [groups][hld] float4, running count, index in the launch) with
// the tallies of prune_tally_kernel; a hypothesis that drops out leaves its partial count in counts[id].  id_in == nullptr:
// the list is still the launch's own (counts themselves, identity ids).  The last thread writes the new live count.
__global__ void __launch_bounds__(kPruneThreads) prune_move_kernel(const float4* __restrict__ hyp_in, const uint32_t* __restrict__ cnt_in,
                                                                   const uint32_t* __restrict__ id_in, size_t hld, int groups, uint32_t H, uint32_t rem,
                                                                   uint32_t L, const uint32_t* __restrict__ tally, float4* __restrict__ hyp_out,
                                                                   uint32_t* __restrict__ cnt_out, uint32_t* __restrict__ id_out,
                                                                   uint32_t* __restrict__ counts, uint32_t* __restrict__ live) {
  __shared__ uint32_t warp_base[kPruneThreads / 32];
  __shared__ uint32_t block_base;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t before = 0;   // survivors of the blocks ahead of this one
  for (uint32_t j = threadIdx.x; j < blockIdx.x; j += kPruneThreads) before += tally[j];
  before = __reduce_add_sync(0xffffffffu, before);
  if (lane == 0) warp_base[warp] = before;
  __syncthreads();
  if (warp == 0) {
    const uint32_t v = __reduce_add_sync(0xffffffffu, warp_base[lane]);
    if (lane == 0) block_base = v;
  }
  __syncthreads();
  const uint32_t i = blockIdx.x * kPruneThreads + threadIdx.x;
  const uint32_t c = i < H ? cnt_in[i] : 0u;
  const bool keep = i < H && c + rem >= L;
  const uint32_t ball = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) warp_base[warp] = __popc(ball);
  __syncthreads();
  if (warp == 0) {   // exclusive scan of the 32 warp tallies
    const uint32_t v = warp_base[lane];
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= (uint32_t)o) x += y;
    }
    warp_base[lane] = block_base + x - v;
  }
  __syncthreads();
  const uint32_t pos = warp_base[warp] + __popc(ball & ((1u << lane) - 1u));
  if (keep) {
    for (int g = 0; g < groups; g++) hyp_out[(size_t)g * hld + pos] = hyp_in[(size_t)g * hld + i];
    cnt_out[pos] = c;
    id_out[pos] = id_in ? id_in[i] : i;
  } else if (i < H && id_in) {
    counts[id_in[i]] = c;
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == kPruneThreads - 1) *live = pos + (keep ? 1u : 0u);
}

// The survivors' full counts back to their hypotheses.
__global__ void prune_scatter_kernel(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ id, uint32_t H, uint32_t* __restrict__ counts) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < H) counts[id[i]] = cnt[i];
}

// What a compaction costs, in hypotheses of one plane launch (0.52 ms per 2^20 on a B200, so ~32 us): its two small kernels
// (6.5 us of device time at the bench configuration, profiles/r03_prune_probe.jsonl) and the host round trip for the new
// live count, which leaves the device idle until the next launch arrives.
constexpr double kCompactCostHyps = 65536.0;

// Hypotheses per thread (R) / point pairs per iteration (PPI) of the constant-bank kernel (128 threads), from the sweeps in
// profiles/r01_tune_cb_sweep_models.txt and profiles/r02_tune_cb_blocking.txt (the plane's 12 x 8 -- sixteen points per iteration --
// is 4.6 % faster than the 10 x 4 it replaced: half the loop overhead per point).  Two things decide them:
//   * few hypotheses per thread on a model with few operations per datum make the uniform constant loads (D per point pair)
//     the limit: 3-8x slower, see the plane4 / dense5 columns of the first sweep;
//   * ptxas fetches the data with LDCU into uniform registers only when a loaded pair has enough consumers in the loop body;
//     below that it falls back to indexed LDC.64 into ordinary registers, which an SM sub-partition sustains at about one
//     per 38 cycles (pivot at R = 6, PPI = 1: 12 LDC.64 per 90 FFMA2, 0.70 T evals/s; at R = 8, PPI = 2 the same body
//     uses LDCU).  tests/test_sass_cpu.py pins "no LDC c[0x3] in the loop" for every model.
#ifndef LSQR_CB_THREADS
#define LSQR_CB_THREADS 128
#endif
#ifndef LSQR_CB_R_PLANE
#define LSQR_CB_R_PLANE 12
#endif
#ifndef LSQR_CB_PPI_PLANE
#define LSQR_CB_PPI_PLANE 8
#endif
constexpr int cb_blocking(int m, bool want_r) {
#ifdef LSQR_CB_OVR_MODEL      // R&D builds (tools/build_variants.sh): override one model
  if (m == LSQR_CB_OVR_MODEL) return want_r ? LSQR_CB_OVR_R : LSQR_CB_OVR_PPI;
#endif
  int r = 8, ppi = 2;
  switch (m) {
    case PLANE3: r = LSQR_CB_R_PLANE; ppi = LSQR_CB_PPI_PLANE; break;
    case LINE2D: case LINE2: r = 12; ppi = 8; break;   // two counters per hypothesis (mixed count): 16 x 4 spills, 12 x 8 measured 2.5 % over 14 x 4
    case PLANE2: r = 16; ppi = 4; break;
    case LINE3: r = 8; ppi = 4; break;
    case DENSE2: r = 10; ppi = 8; break;
    case CIRCLE2: r = 12; ppi = 2; break;
    case SPHERE3: r = 10; ppi = 2; break;
    case ABSOR: r = 4; ppi = 4; break;
    case RAY: r = 8; ppi = 4; break;
    case PIVOT: r = 8; ppi = 2; break;
    case DENSE5: case DENSE6: case SPHERE4: case PLANE4: r = 8; ppi = 4; break;
    case USXW: case USCP: r = 4; ppi = 2; break;
    default:   // the wider template space: hypotheses per thread bounded by the registers their constants take
      switch (model_family(m)) {
        case FAM_PLANE: case FAM_DENSE: r = model_dim(m) <= 4 ? 10 : 8; ppi = model_dim(m) <= 6 ? 4 : 2; break;
        case FAM_SPHERE: r = 8; ppi = model_dim(m) <= 6 ? 4 : 2; break;
        case FAM_LINE: r = model_dim(m) <= 5 ? 6 : 4; ppi = 2; break;
        default: break;
      }
      break;
  }
  return want_r ? r : ppi;
}
template <int M> struct BlockCB { static constexpr int R = cb_blocking(M, true), PPI = cb_blocking(M, false); };

template <int M>
static int run_consensus_cb(const DataView& dv, const float* hyp, size_t hld, uint32_t H, const EstCfg& cfg, uint32_t* counts, int num_sms, cudaStream_t s,
                            Prune* pr) {
  constexpr int D = Model<M>::D, R = BlockCB<M>::R, PPI = BlockCB<M>::PPI, THREADS = LSQR_CB_THREADS, G = (Model<M>::Q32 + 3) / 4;
  constexpr uint32_t cp = cb_points<M>();
  auto kern = consensus_cb_kernel<M, R, THREADS, PPI>;
  int dev = 0;
  cudaGetDevice(&dev);
  static int occ[kMaxDevices] = {0};
  if (!occ[dev % kMaxDevices]) {
    int o = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, THREADS, 0) != cudaSuccess || o < 1) o = 4;
    occ[dev % kMaxDevices] = o;
  }
  void* bank = nullptr;
  if (cudaGetSymbolAddress(&bank, c_tile) != cudaSuccess) return -1;
  uint32_t hyp_blocks = 0;   // of the live hypotheses, per launch
  const uint32_t slots = (uint32_t)num_sms * (uint32_t)occ[dev % kMaxDevices];
  // sub-chunks per launch: fill the last wave (the launches of one request serialise on the bank)
  constexpr bool kRaw = Eval<M>::kHasAbsForm && !Eval<M>::kShifted;
  auto pick_sub = [&](uint32_t npts) {
    uint32_t best_sub = kRaw ? std::min(npts, kCbRawMaxSub) : npts; double best_eff = 0.0;
    for (uint32_t nsub = 1; nsub <= 64; nsub++) {
      uint32_t sub = ((npts + nsub - 1) / nsub + 15) / 16 * 16;
      if (kRaw && sub > kCbRawMaxSub) continue;
      if (sub < 128 && nsub > 1) break;
      const uint32_t ny = (npts + sub - 1) / sub;
      const double waves = (double)hyp_blocks * ny / slots;
      const double eff = waves / (double)(uint64_t)(waves + 0.999999);
      if (eff > best_eff + 0.01) { best_eff = eff; best_sub = sub; }
    }
    return best_sub;
  };
  std::lock_guard<std::mutex> lock(g_cb_mutex[dev % kMaxDevices]);
  int launches = 0;
  // The live list: all H hypotheses in place until the first compaction, then alternately in pr->hyp32[0] and [1].
  const float* live_hyp = hyp;
  uint32_t* live_cnt = counts;
  const uint32_t* live_id = nullptr;
  uint32_t live = H, L = 0;   // L = 0: no early exit
  uint64_t evals = 0;
  int flip = 0;
  // the floor L is seeded after the launches that cover ~1 % of the data (at least one)
  const size_t seed_end = pr ? std::max<size_t>(1, (dv.n / 100 + cp - 1) / cp) * cp : 0;
  size_t next_compact = 0, last_compact = SIZE_MAX;
  for (size_t base = 0; base < dv.span && live; base += cp) {
    const uint32_t npts = (uint32_t)((dv.span - base < cp) ? (dv.span - base) : cp);   // span is a multiple of 1024, cp of 16
    if (base >= dv.n) break;                                                        // only NaN padding left
    const uint32_t rem = dv.n - (uint32_t)base;                                     // data not scored yet
    if (pr && base == seed_end) {
      // L: the full count of the hypothesis with the best partial count, through consensus32_kernel (the same fp32 predicate)
      unsigned long long* key = reinterpret_cast<unsigned long long*>(pr->dev + 16);
      if (cudaMemsetAsync(pr->dev + 16, 0, 4 * sizeof(uint32_t), s) != cudaSuccess) return -1;
      launch_argmax(counts, H, 0, key, s);
      prune_seed_kernel<<<1, 32, 0, s>>>(key, reinterpret_cast<const float4*>(hyp), hld, G, reinterpret_cast<float4*>(pr->dev));
      launches += 2 + launch_consensus32(M, dv, reinterpret_cast<const float*>(pr->dev), 1, 1, cfg, pr->dev + 18, num_sms, s);
      if (cudaMemcpyAsync(pr->host, pr->dev + 18, sizeof(uint32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
          cudaMemcpyAsync(pr->host + 2, pr->floor_key, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
          cudaStreamSynchronize(s) != cudaSuccess) return -1;
      L = std::max(pr->host[0], (uint32_t)(*reinterpret_cast<const unsigned long long*>(pr->host + 2) >> 32));
      evals += dv.n;
    }
    if (L > rem && base >= next_compact) {   // some c + rem may now be < L
      const uint32_t blocks = (live + kPruneThreads - 1) / kPruneThreads;
      float* out_hyp = pr->hyp32[flip];
      uint32_t* out_cnt = pr->live_counts[flip];
      uint32_t* out_id = pr->live_ids[flip];
      prune_tally_kernel<<<blocks, kPruneThreads, 0, s>>>(live_cnt, live, rem, L, pr->dev + 20);
      prune_move_kernel<<<blocks, kPruneThreads, 0, s>>>(reinterpret_cast<const float4*>(live_hyp), live_cnt, live_id, hld, G, live, rem, L, pr->dev + 20,
                                                         reinterpret_cast<float4*>(out_hyp), out_cnt, out_id, counts, pr->dev + 19);
      if (cudaMemcpyAsync(pr->host + 1, pr->dev + 19, sizeof(uint32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) return -1;
      launches += 2;
      // next compaction when the hypotheses expected to drop out by then (at the rate seen since the last one) cost more
      // evaluations than a compaction: interval k launches minimises d k / 2 + cost / k at k = sqrt(2 cost / d)
      const double window = last_compact == SIZE_MAX ? 1.0 : (double)((base - last_compact) / cp);
      const double d = std::max(1.0, (double)(live - pr->host[1]) / window);
      next_compact = base + cp * (size_t)std::min(64.0, std::max(1.0, std::sqrt(2.0 * kCompactCostHyps / d)));
      last_compact = base;
      live_hyp = out_hyp; live_cnt = out_cnt; live_id = out_id; live = pr->host[1];
      flip ^= 1;
      if (!live) break;
    }
    hyp_blocks = (live + THREADS * R - 1) / (THREADS * R);
    if (cudaMemcpy2DAsync(bank, sizeof(float) * cp, dv.soa32 + base, sizeof(float) * dv.ld, sizeof(float) * npts, D, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return -1;
    const uint32_t sub = pick_sub(npts);
    kern<<<dim3(hyp_blocks, (npts + sub - 1) / sub), THREADS, 0, s>>>(npts, sub, live_hyp, hld, live, fp32_delta(cfg), (float)cfg.delta2, live_cnt);
    launches += 2;
    evals += (uint64_t)live * std::min(npts, rem);
  }
  if (live_id && live) {
    prune_scatter_kernel<<<(live + 255) / 256, 256, 0, s>>>(live_cnt, live_id, live, counts);
    launches++;
  }
  if (pr) pr->evals = evals;
  // the bank is shared by every context on this device: finish before another request may refill it
  if (cudaStreamSynchronize(s) != cudaSuccess) return -1;
  return launches;
}

// Register blocking per model: R hypotheses per thread sized so that 2*Q32*R duplicated constants
// plus the point pairs stay below ~128 registers at 256 threads.
constexpr int block32_r(int m) {
  switch (m) {
    case PLANE3: case LINE2D: return 9;
    case LINE2: case CIRCLE2: case SPHERE3: case RAY: case PLANE4: return 8;
    case ABSOR: case USXW: case USCP: return 3;
    case PIVOT: return 4;
    default: { const int q = model_info(m).Q32; return q <= 8 ? 6 : (q <= 10 ? 5 : (q <= 12 ? 4 : 3)); }
  }
}
template <int M> struct Block32 { static constexpr int R = block32_r(M), PPI = (M == ABSOR || M == RAY || M == PIVOT || M == USXW || M == USCP) ? 1 : ((M == LINE2D || M == LINE2) ? 4 : 2); };

int launch_consensus32(int model, const DataView& dv, const float* hyp32, size_t hld, uint32_t H, const EstCfg& cfg, uint32_t* counts, int num_sms,
                       cudaStream_t s, Prune* prune) {
  if (H == 0 || dv.n == 0) return 0;
  if (H >= kCbMinHyps) {
#define CALL(MM) return run_consensus_cb<MM>(dv, hyp32, hld, H, cfg, counts, num_sms, s, prune)
    LSQR_DISPATCH_MODEL(model, CALL)
#undef CALL
  }
#define CALL(MM)                                                                                                        \
  if (H <= 8192) return run_consensus32<MM, 1, 128, 512, Block32<MM>::PPI>(dv, hyp32, hld, H, cfg, counts, num_sms, s);  \
  return run_consensus32<MM, Block32<MM>::R, 256, 512, Block32<MM>::PPI>(dv, hyp32, hld, H, cfg, counts, num_sms, s)
  LSQR_DISPATCH_MODEL(model, CALL)
#undef CALL
  return 0;
}

}  // namespace lsqr
