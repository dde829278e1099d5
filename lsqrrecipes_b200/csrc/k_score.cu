// Scoring path: ingest -> (sample + minimal solve) -> hoist -> consensus -> arg-max.
//
// The consensus kernel is the hot path (RANSAC.hxx:94-99 / :239-244 in the reference: N virtual
// agree() calls per hypothesis).  Layout of the work:
//   * grid.x = blocks of THREADS*R hypotheses, grid.y = chunks of the point set.  Each thread
//     keeps R prepared hypotheses in registers for the whole kernel.
//   * The point chunk is streamed through shared memory in SoA tiles of TILE points, staged by
//     TMA bulk copies (cp.async.bulk ... mbarrier::complete_tx) in a 2-deep ring, one copy per
//     component per tile, issued by one elected thread (TileRing, bulk_copy.cuh).
//   * Inside a tile every thread reads the same point (shared-memory broadcast, vector loads of
//     UNR consecutive points) and evaluates agree() for its R hypotheses.
//   * Per-hypothesis counts go to global memory with one atomicAdd per (hypothesis, chunk).
// This TU holds the fp64 validation mode (models.cuh's reference-order agree()); the fp32 fast
// mode lives in k_fast.cu.
// Tensor cores are deliberately unused: the contraction depth is <= 4 (BASELINE.json north_star).
#include "engine.h"
#include "bulk_copy.cuh"
#include "../../include/lsqr_b200.h"

#include <cstdio>

namespace lsqr {

// ---------------------------------------------------------------------------------------
// Ingest: AoS records -> SoA fp64 (reference arithmetic) + SoA fp32 of x - c (fast mode), one pass, chunk by chunk so
// that it overlaps the host-to-device copy (and, with several GPUs, the all-gather) of the chunks behind it.
// ---------------------------------------------------------------------------------------
// The shift c: per-component mean of the first `count` records (count <= kCenterSample), fixed-order tree sum.  c only
// conditions the arithmetic (fp32 copy of x - c, moments of x - c); any point near the data does, and a prefix is known
// as soon as the first chunk has landed.
__global__ void __launch_bounds__(1024) center_sample_kernel(int model, int D, const unsigned char* __restrict__ aos, size_t stride, uint32_t count, double* __restrict__ center) {
  __shared__ double sh[32][kMaxDim];
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double acc[kMaxDim];
#pragma unroll
  for (int d = 0; d < kMaxDim; d++) acc[d] = 0.0;
  // a thread reads whole records (the D doubles of one record share cache lines); 16 records per thread for the full sample
#pragma unroll 4
  for (uint32_t i = tid; i < count; i += blockDim.x) {
    const double* rec = reinterpret_cast<const double*>(aos + (size_t)i * stride);
#pragma unroll
    for (int d = 0; d < kMaxDim; d++) if (d < D) acc[d] += rec[d];
  }
  // fixed-order tree: lanes, then warps
#pragma unroll
  for (int d = 0; d < kMaxDim; d++) {
    double v = acc[d];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) sh[warp][d] = v;
  }
  __syncthreads();
  if (tid < kMaxDim) {
    const int d = (int)tid;
    double m = 0.0;
    if (d < D && centred_component(model, d) && count > 0) {
      for (uint32_t w = 0; w < (blockDim.x >> 5); w++) m += sh[w][d];
      m /= (double)count;
      if (!(m == m) || fabs(m) > 1e300) m = 0.0;
    }
    center[d] = m;
  }
}
void launch_center_sample(int model, const unsigned char* aos_dev, size_t stride, uint32_t count, double* center_dev, cudaStream_t s) {
  center_sample_kernel<<<1, 1024, 0, s>>>(model, model_info(model).D, aos_dev, stride, count, center_dev);
}

// records [first, first + count) of the AoS buffer (record i at aos + i * stride); when pad_to > first + count the columns
// [first + count, pad_to) are filled with NaN (padded data can never agree)
// (calibrated-pointer ultrasound records: rows 9..11 of the fp32 copy hold t2 - p, formed in fp64, rows 14..16 are unused)
__global__ void ingest_kernel(int model, int D, const unsigned char* __restrict__ aos, size_t stride, uint32_t first, uint32_t count, uint32_t pad_to,
                              const double* __restrict__ center, double* __restrict__ soa64, float* __restrict__ soa32, size_t ld) {
  const size_t i = (size_t)first + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (size_t)first + count) {
    const double* rec = reinterpret_cast<const double*>(aos + i * stride);
    for (int d = 0; d < D; d++) {
      const double v = rec[d];
      soa64[(size_t)d * ld + i] = v;
      float f = (float)(v - center[d]);
      if (model == USCP && d >= 9) f = (d < 12) ? (float)(v - rec[d + 5]) : (d >= 14 ? 0.0f : f);
      soa32[(size_t)d * ld + i] = f;
    }
  } else if (i < pad_to) {
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (int d = 0; d < D; d++) { soa64[(size_t)d * ld + i] = nan; soa32[(size_t)d * ld + i] = __int_as_float(0x7fc00000); }
  }
}
void launch_ingest(int model, const unsigned char* aos_dev, size_t stride, uint32_t first, uint32_t count, uint32_t pad_to, const double* center_dev,
                   double* soa64, float* soa32, size_t ld, cudaStream_t s) {
  const size_t span = (size_t)(pad_to > first + count ? pad_to : first + count) - first;
  if (span == 0) return;
  ingest_kernel<<<(unsigned)((span + 255) / 256), 256, 0, s>>>(model, model_info(model).D, aos_dev, stride, first, count, pad_to, center_dev, soa64, soa32, ld);
}

// ---------------------------------------------------------------------------------------
// Sample + minimal solve: one hypothesis per thread
// ---------------------------------------------------------------------------------------
template <int M>
__global__ void __launch_bounds__(128) solve_kernel(SolveArgs a, const double* __restrict__ soa, size_t ld, uint32_t n, EstCfg cfg) {
  constexpr int D = Model<M>::D, P = Model<M>::P, K = Model<M>::K;
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= a.H) return;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  double prm[P];
  bool ok;
  int32_t sub[K];
  if (a.sampler == 3) {  // LSQR_SAMPLE_PARAMS
#pragma unroll
    for (int j = 0; j < P; j++) prm[j] = a.params_in[(size_t)h * P + j];
    ok = (prm[0] == prm[0]);
#pragma unroll
    for (int j = 0; j < K; j++) sub[j] = -1;
  } else {
    const uint64_t g = a.first + h;
    if (a.sampler == 0) sample_subset<K>(g, a.seed, n, sub);
    else if (a.sampler == 1) unrank_lex<K>(g, n, sub);
    else {
#pragma unroll
      for (int j = 0; j < K; j++) sub[j] = a.list[(size_t)h * K + j];
    }
    double pts[K * D];
    bool in_range = true;
#pragma unroll
    for (int j = 0; j < K; j++) {
      in_range = in_range && sub[j] >= 0 && (uint32_t)sub[j] < n;
      const size_t idx = in_range ? (size_t)sub[j] : 0;
      if (a.gathered != nullptr) {   // the subset's records were fetched ahead of the bulk data
        const double* rec = reinterpret_cast<const double*>(a.gathered + ((size_t)h * K + j) * a.gathered_stride);
#pragma unroll
        for (int d = 0; d < D; d++) pts[j * D + d] = rec[d];
      } else {
#pragma unroll
        for (int d = 0; d < D; d++) pts[j * D + d] = soa[(size_t)d * ld + idx];
      }
    }
    ok = in_range && estimate<M>(pts, cfg, prm);
  }
#pragma unroll
  for (int j = 0; j < K; j++) a.subsets[(size_t)j * a.hld + h] = sub[j];
#pragma unroll
  for (int j = 0; j < P; j++) a.hyp64[(size_t)j * a.hld + h] = ok ? prm[j] : nan;
  const unsigned ballot = __ballot_sync(__activemask(), ok);
  if ((threadIdx.x & 31) == (__ffs(__activemask()) - 1) && ballot) atomicAdd(a.n_valid, __popc(ballot));
}

void launch_solve(const SolveArgs& a, const DataView& dv, const EstCfg& cfg, cudaStream_t s) {
  if (a.H == 0) return;
  const unsigned blocks = (a.H + 127) / 128;
#define CALL(MM) solve_kernel<MM><<<blocks, 128, 0, s>>>(a, dv.soa64, dv.ld, dv.n, cfg)
  LSQR_DISPATCH_MODEL(a.model, CALL)
#undef CALL
}

// After the arg-max (and, sharded, its all-reduce): re-derives the winner's subset and parameters from the packed key ON
// THE DEVICE -- every rank holds them whichever shard produced the winner -- and leaves key, valid count, subset and
// parameters in one small record that the host fetches with a single copy.  The parameters also stay on the device for the
// consensus-set pass that follows in compute().
template <int M>
__global__ void winner_kernel(SolveArgs a, const unsigned long long* __restrict__ key, const double* __restrict__ soa, size_t ld, uint32_t n, EstCfg cfg,
                              WinnerRecord* __restrict__ out) {
  constexpr int D = Model<M>::D, P = Model<M>::P, K = Model<M>::K;
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const unsigned long long k = key[0];
  out->key = k;
  out->n_valid = key[1] & 0xFFFFFFFFull;
  for (int j = 0; j < LSQR_MAX_SUBSET; j++) out->subset[j] = -1;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  for (int j = 0; j < LSQR_MAX_PARAMS; j++) out->params[j] = nan;
  if ((k >> 32) == 0) return;
  const uint64_t rel = 0xFFFFFFFFull - (k & 0xFFFFFFFFull);   // index relative to the request's first hypothesis
  double prm[P];
  int32_t sub[K];
  bool ok = true;
  if (a.sampler == 3) {
    for (int j = 0; j < P; j++) prm[j] = a.params_in[(size_t)rel * P + j];
    for (int j = 0; j < K; j++) sub[j] = -1;
  } else {
    if (a.sampler == 0) sample_subset<K>(a.first + rel, a.seed, n, sub);
    else if (a.sampler == 1) unrank_lex<K>(a.first + rel, n, sub);
    else for (int j = 0; j < K; j++) sub[j] = a.list[(size_t)rel * K + j];
    double pts[K * D];
    for (int j = 0; j < K; j++) for (int d = 0; d < D; d++) pts[j * D + d] = soa[(size_t)d * ld + (size_t)sub[j]];
    ok = estimate<M>(pts, cfg, prm);
  }
  for (int j = 0; j < K; j++) out->subset[j] = sub[j];
  if (ok) for (int j = 0; j < P; j++) out->params[j] = prm[j];
}
void launch_winner(const SolveArgs& a, const unsigned long long* key_dev, const DataView& dv, const EstCfg& cfg, WinnerRecord* out, cudaStream_t s) {
#define CALL(MM) winner_kernel<MM><<<1, 32, 0, s>>>(a, key_dev, dv.soa64, dv.ld, dv.n, cfg, out)
  LSQR_DISPATCH_MODEL(a.model, CALL)
#undef CALL
}

// UNR = 2 data per inner iteration: one LDS.128 per component
template <int M, int R, int THREADS, int TILE>
__global__ void __launch_bounds__(THREADS) consensus_kernel(const double* __restrict__ soa, size_t ld, uint32_t tiles_total, uint32_t tiles_per_chunk,
                                                             const double* __restrict__ hyp, size_t hld, uint32_t H, EstCfg thr,
                                                             uint32_t* __restrict__ counts) {
  constexpr int D = Model<M>::D, P = Model<M>::P, HQ = Model<M>::HQ, UNR = 2;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bars[2];

  const int tid = threadIdx.x;
  const uint32_t hbase = blockIdx.x * (THREADS * R);
  double hq[R][HQ];
  uint32_t cnt[R];
#pragma unroll
  for (int r = 0; r < R; r++) {
    const uint32_t h = hbase + r * THREADS + tid;
    double raw[P];
#pragma unroll
    for (int j = 0; j < P; j++) raw[j] = (h < H) ? hyp[(size_t)j * hld + h] : (double)NAN;
    prepare<M>(raw, thr, hq[r]);
    cnt[r] = 0;
  }

  const uint32_t t0 = blockIdx.y * tiles_per_chunk;
  const uint32_t t1 = min(t0 + tiles_per_chunk, tiles_total);
  TileRing<D, TILE, double> ring{soa, ld, t0, t1, reinterpret_cast<double*>(smem_raw), bars, tid};
  ring.start();
  for (uint32_t t = t0; t < t1; t++) {
    const double* tl = ring.wait(t);
#pragma unroll 1
    for (int i = 0; i < TILE; i += UNR) {
      double x[UNR][D];
#pragma unroll
      for (int d = 0; d < D; d++) {
        const double2 v = *reinterpret_cast<const double2*>(tl + d * TILE + i);
        x[0][d] = v.x; x[1][d] = v.y;
      }
#pragma unroll
      for (int r = 0; r < R; r++) {
#pragma unroll
        for (int u = 0; u < UNR; u++) cnt[r] += agree<M>(hq[r], x[u], thr) ? 1u : 0u;
      }
    }
    ring.release();
  }
#pragma unroll
  for (int r = 0; r < R; r++) {
    const uint32_t h = hbase + r * THREADS + tid;
    if (h < H && cnt[r]) atomicAdd(&counts[h], cnt[r]);
  }
}

template <int M, int R, int THREADS, int TILE>
static int run_consensus(const DataView& dv, const double* hyp, size_t hld, uint32_t H, const EstCfg& cfg, uint32_t* counts, int num_sms, cudaStream_t s) {
  const uint32_t tiles_total = (uint32_t)(dv.span / TILE);
  const uint32_t hyp_blocks = (H + THREADS * R - 1) / (THREADS * R);
  const TileChunks plan = plan_tile_chunks(tiles_total, hyp_blocks, num_sms);
  const size_t smem = 2 * (size_t)Model<M>::D * TILE * sizeof(double);
  auto kern = consensus_kernel<M, R, THREADS, TILE>;
  allow_dynamic_smem(kern, smem);
  kern<<<dim3(hyp_blocks, plan.chunks), THREADS, smem, s>>>(dv.soa64, dv.ld, tiles_total, plan.tiles_per_chunk, hyp, hld, H, cfg, counts);
  return 1;
}

// hypotheses per thread of the fp64 validation kernel (models with up to 11 prepared doubles per hypothesis)
#ifndef LSQR_FP64_R
#define LSQR_FP64_R 4
#endif
int launch_consensus(int model, int precision, const DataView& dv, const double* hyp64, const float* hyp32, size_t hld, uint32_t H,
                     const EstCfg& cfg, uint32_t* counts, int num_sms, cudaStream_t s, Prune* prune) {
  if (H == 0 || dv.n == 0) return 0;
  if (precision == 0) {
#define CALL(MM)                                                                                                             \
  if (H <= 4096) return run_consensus<MM, 1, 128, 256>(dv, hyp64, hld, H, cfg, counts, num_sms, s);                                \
  return run_consensus<MM, (Model<MM>::HQ >= 12 ? 2 : LSQR_FP64_R), 128, 256>(dv, hyp64, hld, H, cfg, counts, num_sms, s)
    LSQR_DISPATCH_MODEL(model, CALL)
#undef CALL
  } else {
    return launch_consensus32(model, dv, hyp32, hld, H, cfg, counts, num_sms, s, prune);
  }
  return 0;
}

// ---------------------------------------------------------------------------------------
// Arg-max over a packed (count, index) key: larger count wins, ties go to the SMALLER index
// (strict '>' of RANSAC.hxx:100 and :245 keeps the first maximum).
// ---------------------------------------------------------------------------------------
__global__ void argmax_kernel(const uint32_t* __restrict__ counts, uint32_t H, uint32_t index_base, unsigned long long* __restrict__ key) {
  unsigned long long best = 0ull;
  for (uint32_t h = blockIdx.x * blockDim.x + threadIdx.x; h < H; h += gridDim.x * blockDim.x) {
    const unsigned long long k = ((unsigned long long)counts[h] << 32) | (unsigned long long)(0xFFFFFFFFu - (index_base + h));
    best = k > best ? k : best;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { const unsigned long long v = __shfl_xor_sync(0xffffffffu, best, o); best = v > best ? v : best; }
  __shared__ unsigned long long sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x < 32) {
    best = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0ull;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) { const unsigned long long v = __shfl_xor_sync(0xffffffffu, best, o); best = v > best ? v : best; }
    if (threadIdx.x == 0 && best) atomicMax(key, best);
  }
}
void launch_argmax(const uint32_t* counts, uint32_t H, uint32_t index_base, unsigned long long* key, cudaStream_t s) {
  if (H == 0) return;
  unsigned blocks = (H + 255) / 256;
  if (blocks > 1184) blocks = 1184;
  argmax_kernel<<<blocks, 256, 0, s>>>(counts, H, index_base, key);
}


// ---------------------------------------------------------------------------------------
// The estimator's own estimate() / agree() for callers that use them directly
// (ParametersEstimator.h:41-55); same device functions as the batched path.
// ---------------------------------------------------------------------------------------
template <int M>
__global__ void estimate_one_kernel(const double* __restrict__ packed, EstCfg cfg, double* __restrict__ out) {
  if (threadIdx.x != 0) return;
  constexpr int D = Model<M>::D, P = Model<M>::P, K = Model<M>::K;
  double pts[K * D], prm[P];
  for (int i = 0; i < K * D; i++) pts[i] = packed[i];
  const bool ok = estimate<M>(pts, cfg, prm);
  out[0] = ok ? (double)P : 0.0;
  for (int j = 0; j < P; j++) out[1 + j] = ok ? prm[j] : 0.0;
}
void launch_estimate_one(int model, const double* packed_dev, const EstCfg& cfg, double* out_dev, cudaStream_t s) {
#define CALL(MM) estimate_one_kernel<MM><<<1, 32, 0, s>>>(packed_dev, cfg, out_dev)
  LSQR_DISPATCH_MODEL(model, CALL)
#undef CALL
}
template <int M>
__global__ void agree_many_kernel(const double* __restrict__ params, const double* __restrict__ packed, uint32_t n, EstCfg cfg, uint8_t* __restrict__ out) {
  constexpr int D = Model<M>::D, P = Model<M>::P, HQ = Model<M>::HQ;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double prm[P], hq[HQ], x[D];
#pragma unroll
  for (int j = 0; j < P; j++) prm[j] = params[j];
  prepare<M>(prm, cfg, hq);
#pragma unroll
  for (int d = 0; d < D; d++) x[d] = packed[(size_t)i * D + d];
  out[i] = agree<M>(hq, x, cfg) ? 1 : 0;
}
void launch_agree_many(int model, const double* params_dev, const double* packed_dev, uint32_t n, const EstCfg& cfg, uint8_t* out, cudaStream_t s) {
  if (n == 0) return;
  const unsigned blocks = (n + 255) / 256;
#define CALL(MM) agree_many_kernel<MM><<<blocks, 256, 0, s>>>(params_dev, packed_dev, n, cfg, out)
  LSQR_DISPATCH_MODEL(model, CALL)
#undef CALL
}

}  // namespace lsqr
