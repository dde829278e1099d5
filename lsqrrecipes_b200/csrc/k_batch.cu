// Batched small problems (BASELINE.json configs[4]): one thread block per problem, see the comment above batch_kernel.
#include "bulk_copy.cuh"
#include "refine_common.cuh"
#include "fast_forms.cuh"
#include <cooperative_groups.h>
#include <algorithm>
#include <tuple>

namespace lsqr {

// ---------------------------------------------------------------------------------------
// Batched small problems: one thread block per problem (BASELINE.json config 5; in the
// reference this is a host loop of RANSAC<T,S>::compute calls).  Everything -- subset
// generation, minimal solve, consensus, arg-max, consensus set, least-squares refine -- happens
// inside the block with the problem's points resident in shared memory.  Exhaustive mode enumerates all C(n,k)
// subsets (RANSAC.hxx:150-249) in fp64 reference arithmetic (bit-comparable with the reference's brute-force driver);
// otherwise rounds of Philox hypotheses with the stop rule of RANSAC.hxx:107-110 between rounds, scored in fp64 or -- precision
// LSQR_FP32, what the large-problem path does -- in the fp32 forms of fast_forms.cuh on an fp32 copy of the points relative to the
// problem's first point, two data per packed operation.  Minimal solves, the winner's consensus set, its count and the refine
// are fp64 in every mode, so the returned mask / count / parameters are exact for the chosen hypothesis.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long block_max_u64(unsigned long long v, unsigned long long* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o); v = w > v ? w : v; }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  unsigned long long r = 0;
  for (int w = 0; w < (int)(blockDim.x >> 5); w++) r = sh[w] > r ? sh[w] : r;
  return r;
}

// Hypotheses of one problem, shared by batch_kernel and batch_cluster_kernel.  Record i's component d of a problem is
// x[d * sd + i * si]: SoA rows in shared memory (sd = leading dimension, si = 1) or the packed AoS records in global memory
// (sd = 1, si = D).
template <int M>
__device__ __forceinline__ void gather_subset(const int32_t* sub, const double* x, uint32_t sd, uint32_t si, double* sp) {
#pragma unroll
  for (int j = 0; j < Model<M>::K; j++)
#pragma unroll
    for (int d = 0; d < Model<M>::D; d++) sp[j * Model<M>::D + d] = x[d * sd + sub[j] * si];
}

// fp64 count of hypothesis prm over the SoA rows pts [D][ldp], data first, first + step, ... < n
template <int M>
__device__ __forceinline__ uint32_t count64(const double* prm, const EstCfg& cfg, const double* pts, uint32_t ldp, uint32_t n, uint32_t first, uint32_t step) {
  constexpr int D = Model<M>::D;
  double hq[Model<M>::HQ];
  prepare<M>(prm, cfg, hq);
  uint32_t c = 0;
  for (uint32_t i = first; i < n; i += step) {
    double x[D];
#pragma unroll
    for (int d = 0; d < D; d++) x[d] = pts[d * ldp + i];
    c += agree<M>(hq, x, cfg) ? 1u : 0u;
  }
  return c;
}

// fp32 count of hypothesis prm over the centred fp32 rows ptsf [D][ldf] (x - ctr, NaN past the data), pairs first, first + step, ...
// < n (first and step even); NaN padding counts as an outlier.
template <int M>
__device__ __forceinline__ uint32_t count32(const double* prm, const double* sh_ctr, const EstCfg& cfg, const float* ptsf, uint32_t ldf, uint32_t n,
                                            uint32_t first, uint32_t step) {
  uint32_t c = 0;
  if constexpr (M != USXW && M != USCP) {   // (the ultrasound calibrations have no batched mode)
    constexpr int D = Model<M>::D, Q = Model<M>::Q32;
    double ctr[kMaxDim];
#pragma unroll
    for (int d = 0; d < kMaxDim; d++) ctr[d] = sh_ctr[d];
    float qf[Q];
    hoist32<M>(prm, ctr, cfg, qf);
    f2 q[Q];
#pragma unroll
    for (int j = 0; j < Q; j++) q[j] = splat(qf[j]);
    Thr2 thr;
    const float fdelta = fp32_delta(cfg);
    thr.delta = splat(fdelta); thr.neg_delta2 = splat(-(float)cfg.delta2); thr.fdelta = fdelta;
    const uint32_t negk = hyp_negk<M>(qf, 0u - __float_as_uint(2.0f * fdelta));   // 2^32 - bits(window)
    unsigned long long out = 0ull;
    uint32_t pairs = 0;
    for (uint32_t i = first; i < n; i += step) {
      f2 x[D];
#pragma unroll
      for (int d = 0; d < D; d++) x[d].v = *reinterpret_cast<const unsigned long long*>(ptsf + d * ldf + i);
      if constexpr (Eval<M>::kShifted) count_carry(out, Eval<M>::dist(q, x), negk);
      else if constexpr (Eval<M>::kHasAbsForm) count_abs_lt(c, Eval<M>::dist(q, x), hyp_thr<M>(qf, thr.fdelta));
      else count_sign(c, Eval<M>::signed_(q, x, thr));
      pairs++;
    }
    if constexpr (Eval<M>::kShifted) c = negk ? 2u * pairs - (uint32_t)(out >> 32) : 0u;   // outliers were counted (NaN padding among them)
  }
  return c;
}

// A round's arg-max key into the running best.  When it raised the best, randomized mode lowers the hypothesis budget
// `tries` by the stop rule of RANSAC.hxx:104-110 (stop_rule != 0).
__device__ __forceinline__ void round_update(unsigned long long round_best, unsigned long long& best, bool stop_rule, uint32_t n, int K, double prob,
                                             double log1mp, unsigned long long* tries) {
  if (round_best > best) {
    best = round_best;
    if (stop_rule) {
      const uint32_t c = (uint32_t)(best >> 32);
      unsigned long long cap = *tries;
      if (c == n) cap = 0;
      else if (prob > 0.0 && prob < 1.0) {
        const double den = log(1.0 - pow((double)c / (double)n, (double)K));
        const double t = log1mp / den + 0.5;
        const unsigned long long nt = t >= 4294967295.0 ? 0xFFFFFFFFull : (unsigned long long)(long long)t;
        cap = nt < cap ? nt : cap;
      }
      *tries = cap;
    }
  }
}

// The winner of key `best` solved again from its subset (RANSAC.hxx:129-131), its prepared constants into hq.  False when no
// hypothesis had a consensus set or the solve fails.
template <int M>
__device__ __forceinline__ bool winner_constants(unsigned long long best, int exhaustive, uint64_t gb, uint64_t seed, uint32_t n, const double* x,
                                                 uint32_t sd, uint32_t si, const EstCfg& cfg, double* hq) {
  constexpr int D = Model<M>::D, P = Model<M>::P, K = Model<M>::K;
  if ((uint32_t)(best >> 32) == 0) return false;
  const unsigned long long h = 0xFFFFFFFFull - (best & 0xFFFFFFFFull);
  int32_t sub[K];
  if (exhaustive) unrank_lex<K>(h, n, sub); else sample_subset<K>((gb << 32) | h, seed, n, sub);
  double sp[K * D], prm[P];
  gather_subset<M>(sub, x, sd, si, sp);
  if (!estimate<M>(sp, cfg, prm)) return false;
  prepare<M>(prm, cfg, hq);
  return true;
}

// Consensus set (use_mask) or Levenberg-Marquardt (lm) moments of the block's records into sh_mom.  Record i's component d is
// pts[d * ldp + i * step]; CENTRED accumulates x - ctr (agree() still sees x), otherwise x itself with step 1.
template <int M, bool CENTRED = false>
__device__ void block_moments(const double* pts, uint32_t n, uint32_t ldp, uint32_t step, const double* ctr, const double* hq, const EstCfg& cfg,
                              const double* lmx, bool lm, int use_mask, uint8_t* mask_out, double* sh_part, double* sh_mom) {
  constexpr int D = Model<M>::D;
  constexpr int NMA = Mom<M>::N, NML = Mom<M>::NLM;
  double acc[kMaxMoments];
  const int nm = lm ? NML : NMA;
  const uint32_t si = CENTRED ? step : 1u;
  for (int j = 0; j < kMaxMoments; j++) acc[j] = 0.0;
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    double x[D];
#pragma unroll
    for (int d = 0; d < D; d++) x[d] = pts[d * ldp + i * si];
    const bool in = use_mask ? agree<M>(hq, x, cfg) : true;
    if (mask_out) mask_out[i] = in ? 1 : 0;
    if (in) {
      if constexpr (CENTRED) {
#pragma unroll
        for (int d = 0; d < D; d++) x[d] -= ctr[d];
      }
      if (lm) {
        if constexpr (Model<M>::FAM == FAM_SPHERE) acc_sphere_lm<Model<M>::DIM>(x, lmx, acc);
      } else { acc[0] += 1.0; accumulate<M>(x, acc); }
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  for (int j = 0; j < nm; j++) {
    double v = acc[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) sh_part[warp * kMaxMoments + j] = v;
  }
  __syncthreads();
  if ((int)threadIdx.x < nm) { double v = 0; for (int w = 0; w < nw; w++) v += sh_part[w * kMaxMoments + threadIdx.x]; sh_mom[threadIdx.x] = v; }
  __syncthreads();
}

template <int M>
__global__ void __launch_bounds__(256) batch_kernel(BatchArgs a, EstCfg cfg, int ls_type, uint32_t group) {
  constexpr int D = Model<M>::D, P = Model<M>::P, K = Model<M>::K, HQ = Model<M>::HQ;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* pts = reinterpret_cast<double*>(smem_raw);  // [D][ldp]
  const uint32_t ldp = a.max_n;
  __shared__ unsigned long long sh_key[8];
  __shared__ double sh_part[8 * kMaxMoments];
  __shared__ double sh_mom[kMaxMoments];
  __shared__ double sh_prm[LSQR_MAX_PARAMS + 4];
  __shared__ double sh_state[LM_SIZE];
  __shared__ unsigned long long sh_best;
  __shared__ unsigned long long sh_tries;
  __shared__ int sh_ok;

  const uint32_t b = blockIdx.x;
  const uint64_t off = a.offsets[b] - a.base;                 // record offset inside this launch's data
  const uint32_t n = (uint32_t)(a.offsets[b + 1] - a.offsets[b]);
  if (n > a.max_n) return;                                    // a problem larger than one block: batch_cluster_kernel's
  const uint64_t gb = a.first_problem + b;                    // global problem index: the sampler's counter does not depend on how problems are split over GPUs
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  for (uint32_t i = threadIdx.x; i < n * D; i += blockDim.x) pts[(i % D) * ldp + (i / D)] = a.data[off * D + i];
  // fp32 scoring: the problem's points relative to its first point (centred components only), padded to an even count with NaN
  const bool use32 = a.precision == 1 && !a.exhaustive;
  const uint32_t ldf = (ldp + 1u) & ~1u;
  float* ptsf = reinterpret_cast<float*>(pts + (size_t)D * ldp);   // [D][ldf]
  __shared__ double sh_ctr[kMaxDim];
  if (use32) {
    __syncthreads();
    if (threadIdx.x < (uint32_t)kMaxDim) sh_ctr[threadIdx.x] = (threadIdx.x < (uint32_t)D && n > 0 && centred_component(M, (int)threadIdx.x)) ? pts[threadIdx.x * ldp] : 0.0;
    __syncthreads();
    const uint32_t npad = (n + 1u) & ~1u;
    for (uint32_t i = threadIdx.x; i < npad * D; i += blockDim.x) {
      const uint32_t d = i / npad, j = i % npad;
      ptsf[d * ldf + j] = (j < n) ? (float)(pts[d * ldp + j] - sh_ctr[d]) : __int_as_float(0x7fc00000);
    }
  }
  if (threadIdx.x == 0) {
    sh_best = 0ull;
    unsigned long long all = 0xFFFFFFFFull;  // RANSAC::choose saturates at UINT_MAX (RANSAC.hxx:254-280)
    if (n >= (uint32_t)K) { const uint64_t c = binom(n, K); all = c < all ? c : all; } else all = 0;
    sh_tries = a.exhaustive ? all : (all < a.tries ? all : (unsigned long long)a.tries);
  }
  __syncthreads();

  unsigned long long best = 0ull;
  const double log1mp = log(1.0 - a.prob);
  // G threads share one hypothesis (each counts every G-th datum).  Randomized mode re-evaluates the stop rule after every
  // round and ends in a single-thread refit, so it runs small blocks (many resident per SM) with short rounds; exhaustive
  // mode is throughput-bound and scores one hypothesis per thread (launch_batch picks block size and G).
  const uint32_t G = group;
  const uint32_t per_round = blockDim.x / G, sub_lane = threadIdx.x % G;
  for (unsigned long long done = 0; done < sh_tries; done += per_round) {
    const unsigned long long h = done + threadIdx.x / G;
    unsigned long long key = 0ull;
    if (h < sh_tries) {
      int32_t sub[K];
      if (a.exhaustive) unrank_lex<K>(h, n, sub); else sample_subset<K>((gb << 32) | h, a.seed, n, sub);
      double sp[K * D], prm[P];
      gather_subset<M>(sub, pts, ldp, 1, sp);
      const bool ok = estimate<M>(sp, cfg, prm);   // the same for all G threads of a hypothesis
      uint32_t c = 0;
      if (ok && use32) c = count32<M>(prm, sh_ctr, cfg, ptsf, ldf, n, 2 * sub_lane, 2 * G);
      else if (ok) c = count64<M>(prm, cfg, pts, ldp, n, sub_lane, G);
      if (G > 1) {   // uniform over the block; the G threads of a hypothesis are adjacent lanes of one warp
        const unsigned grp = (0xFFFFFFFFu >> (32u - G)) << ((threadIdx.x & 31u) & ~(G - 1u));
        for (uint32_t o = 1; o < G; o <<= 1) c += __shfl_xor_sync(grp, c, o);
      }
      if (ok) key = ((unsigned long long)c << 32) | (0xFFFFFFFFull - h);
    }
    const unsigned long long round_best = block_max_u64(key, sh_key);
    round_update(round_best, best, !a.exhaustive && threadIdx.x == 0, n, K, a.prob, log1mp, &sh_tries);
    __syncthreads();
  }

  // winner -> consensus set -> least squares (RANSAC.hxx:129-138)
  const uint32_t best_count = (uint32_t)(best >> 32);
  if (threadIdx.x == 0) sh_ok = winner_constants<M>(best, a.exhaustive, gb, a.seed, n, pts, ldp, 1, cfg, sh_prm) ? 1 : 0;
  __syncthreads();
  uint8_t* mask_out = a.out_masks ? a.out_masks + off : nullptr;
  if (threadIdx.x == 0) a.out_counts[b] = best_count;
  if (!sh_ok) {
    for (uint32_t i = threadIdx.x; i < (uint32_t)P; i += blockDim.x) a.out_params[(size_t)b * P + i] = nan;
    if (mask_out) for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) mask_out[i] = 0;
    return;
  }
  double hq[HQ];
#pragma unroll
  for (int j = 0; j < HQ; j++) hq[j] = sh_prm[j];
  block_moments<M>(pts, n, ldp, 1, nullptr, hq, cfg, nullptr, false, 1, mask_out, sh_part, sh_mom);
  if (use32 && threadIdx.x == 0) a.out_counts[b] = (uint32_t)sh_mom[0];   // the fp64 count of the winner's consensus set (the fp32 count chose it)
  double zero_center[kMaxDim];
  for (int j = 0; j < kMaxDim; j++) zero_center[j] = 0.0;
  __shared__ double sh_out[LSQR_MAX_PARAMS + 4];
  if (threadIdx.x == 0) {
    double p[LSQR_MAX_PARAMS];
    int np = 0;
    const double* m = sh_mom;
    const double* c = zero_center;
    if constexpr (M != USXW && M != USCP) np = solve_model(M, m, c, 1, p);   // (the zero centre makes "centred" the caller's frame)
    sh_out[0] = np;
    for (int j = 0; j < np; j++) sh_out[1 + j] = p[j];
  }
  __syncthreads();
  if constexpr (Model<M>::FAM == FAM_SPHERE) {
    if (ls_type == 1) {  // geometric: Levenberg-Marquardt from the algebraic fit
      if (threadIdx.x == 0) {
        for (int i = 0; i < LM_SIZE; i++) sh_state[i] = 0.0;
        const int np = (int)sh_out[0];
        if (np == 0) sh_state[LM_STATUS] = 2.0;
        for (int j = 0; j < np; j++) sh_state[LM_X + j] = sh_out[1 + j];
      }
      __syncthreads();
      // The controller state is touched by thread 0 only; what the block needs per pass (status, evaluation
      // point) goes through sh_bcast, with a barrier on either side of every read.
      constexpr int NPL = Mom<M>::NPLM;
      __shared__ double sh_bcast[1 + NPL];
      for (;;) {
        if (threadIdx.x == 0) {
          sh_bcast[0] = sh_state[LM_STATUS];
          const int o = (sh_state[LM_PHASE] != 0.0) ? LM_TRIAL : LM_X;
          for (int j = 0; j < NPL; j++) sh_bcast[1 + j] = sh_state[o + j];
        }
        __syncthreads();
        double lmx[NPL];
        const double status = sh_bcast[0];
        for (int j = 0; j < NPL; j++) lmx[j] = sh_bcast[1 + j];
        __syncthreads();
        if (status != 0.0) break;
        block_moments<M>(pts, n, ldp, 1, nullptr, hq, cfg, lmx, true, 1, nullptr, sh_part, sh_mom);
        if (threadIdx.x == 0) lm_update_model(M, sh_mom, sh_state);
      }
      if (threadIdx.x == 0) {
        if (sh_state[LM_STATUS] != 1.0) sh_out[0] = 0.0;
        else for (int j = 0; j < P; j++) sh_out[1 + j] = sh_state[LM_X + j];
      }
      __syncthreads();
    }
  }
  const int np = (int)sh_out[0];
  for (uint32_t i = threadIdx.x; i < (uint32_t)P; i += blockDim.x) a.out_params[(size_t)b * P + i] = np ? sh_out[1 + i] : nan;
}

// ---------------------------------------------------------------------------------------
// Batched problems too large for one block: one thread-block cluster of C CTAs (2..16) per problem.  CTA r holds records
// [r S, min((r + 1) S, n)), S = ceil(n / C) rounded up to even, in its shared memory: only the scoring copy (fp64 SoA rows, or
// the fp32 rows of x - first record).  The fp64 records that the minimal solves, the consensus set and the refine need are
// read from the packed batch in global memory.  Every CTA solves the round's 32 hypotheses itself (identical inputs give
// identical bits), eight threads per hypothesis count over its own slice, and after one cluster barrier every CTA reads the
// C x 32 partial counts over distributed shared memory and takes the same decision, so nothing is broadcast.  The
// consensus-set and Levenberg-Marquardt passes reduce their moments the same way, summed in rank order; thread 0 of every
// CTA runs the same solve on the same sums.  Moments are taken relative to the problem's first record.
// ---------------------------------------------------------------------------------------
namespace cg = cooperative_groups;

// the C partial moment vectors of the cluster, in rank order -> tot (every CTA).  `mine` alternates between two buffers:
// a CTA may still be reading a neighbour's previous vector when that neighbour writes its next one.
__device__ __forceinline__ void cluster_sum(const cg::cluster_group& cluster, double* mine, int nm, double* tot) {
  cluster.sync();
  if ((int)threadIdx.x < nm) {
    double v = 0.0;
    for (uint32_t q = 0; q < cluster.num_blocks(); q++) v += cluster.map_shared_rank(mine, q)[threadIdx.x];
    tot[threadIdx.x] = v;
  }
  __syncthreads();
}

constexpr int kClusterThreads = 256;

template <int M>
__global__ void __launch_bounds__(kClusterThreads) batch_cluster_kernel(BatchArgs a, const uint32_t* __restrict__ problems, EstCfg cfg, int ls_type) {
  constexpr int D = Model<M>::D, P = Model<M>::P, K = Model<M>::K, HQ = Model<M>::HQ;
  constexpr uint32_t G = 8, R = kClusterThreads / G;   // threads per hypothesis, hypotheses per round
  const cg::cluster_group cluster = cg::this_cluster();
  const uint32_t C = cluster.num_blocks(), rank = cluster.block_rank(), tid = threadIdx.x;
  extern __shared__ __align__(16) unsigned char cl_smem_raw[];
  double* pts = reinterpret_cast<double*>(cl_smem_raw);   // fp64 scoring: [D][S]
  float* ptsf = reinterpret_cast<float*>(cl_smem_raw);    // fp32 scoring: [D][S], x - first record, NaN padded to even
  __shared__ uint32_t sh_cnt[2][R];                        // partial counts of the round, by round parity (~0u: no hypothesis)
  __shared__ double sh_part[(kClusterThreads / 32) * kMaxMoments];
  __shared__ double sh_mom[2][kMaxMoments];                // this CTA's moments, by pass parity
  __shared__ double sh_tot[kMaxMoments];                   // the cluster's
  __shared__ double sh_prm[LSQR_MAX_PARAMS + 4];
  __shared__ double sh_out[LSQR_MAX_PARAMS + 4];
  __shared__ double sh_state[LM_SIZE];
  __shared__ double sh_ctr[kMaxDim];
  __shared__ unsigned long long sh_best, sh_tries;
  __shared__ int sh_ok;

  const uint32_t b = problems[blockIdx.x / C];
  const uint64_t off = a.offsets[b] - a.base;
  const uint32_t n = (uint32_t)(a.offsets[b + 1] - a.offsets[b]);
  const uint64_t gb = a.first_problem + b;
  const double* rec = a.data + off * D;                    // the problem's records, AoS
  const bool use32 = a.precision == 1;
  const uint32_t S = ((n + C - 1) / C + 1u) & ~1u;
  const uint32_t lo = min(rank * S, n), ns = min(S, n - lo), npad = (ns + 1u) & ~1u;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  if (tid < (uint32_t)kMaxDim) sh_ctr[tid] = (tid < (uint32_t)D && centred_component(M, (int)tid)) ? rec[tid] : 0.0;
  __syncthreads();
  if (use32) {
    for (uint32_t i = tid; i < npad * D; i += kClusterThreads) {
      const uint32_t j = i / D, d = i % D;
      ptsf[d * S + j] = (j < ns) ? (float)(rec[(size_t)lo * D + i] - sh_ctr[d]) : __int_as_float(0x7fc00000);
    }
  } else {
    for (uint32_t i = tid; i < ns * D; i += kClusterThreads) pts[(i % D) * S + i / D] = rec[(size_t)lo * D + i];
  }
  if (tid == 0) {
    unsigned long long all = 0xFFFFFFFFull;
    if (n >= (uint32_t)K) { const uint64_t c = binom(n, K); all = c < all ? c : all; } else all = 0;
    sh_tries = all < a.tries ? all : (unsigned long long)a.tries;
  }
  __syncthreads();

  unsigned long long best = 0ull;   // thread 0's is the problem's
  const double log1mp = log(1.0 - a.prob);
  const uint32_t sub_lane = tid % G, slot = tid / G;
  uint32_t parity = 0;
  for (unsigned long long done = 0; done < sh_tries; done += R, parity ^= 1u) {
    const unsigned long long tries = sh_tries, h = done + slot;
    uint32_t c = ~0u;
    if (h < tries) {
      int32_t sub[K];
      sample_subset<K>((gb << 32) | h, a.seed, n, sub);
      double sp[K * D], prm[P];
      gather_subset<M>(sub, rec, 1, D, sp);
      if (estimate<M>(sp, cfg, prm)) {   // the same in every thread of the hypothesis and every CTA of the cluster
        c = use32 ? count32<M>(prm, sh_ctr, cfg, ptsf, S, npad, 2 * sub_lane, 2 * G) : count64<M>(prm, cfg, pts, S, ns, sub_lane, G);
        const unsigned grp = 0xFFu << ((tid & 31u) & ~(G - 1u));
        for (uint32_t o = 1; o < G; o <<= 1) c += __shfl_xor_sync(grp, c, o);
      }
    }
    if (sub_lane == 0) sh_cnt[parity][slot] = c;
    cluster.sync();
    if (tid < 32) {   // warp 0: the round's keys over the whole problem, the same in every CTA
      const unsigned long long hh = done + tid;
      uint32_t total = 0;
      bool ok = hh < tries;
      for (uint32_t q = 0; q < C; q++) {
        const uint32_t v = cluster.map_shared_rank(&sh_cnt[parity][0], q)[tid];
        ok = ok && v != ~0u;
        total += v;
      }
      unsigned long long key = ok ? ((unsigned long long)total << 32) | (0xFFFFFFFFull - hh) : 0ull;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) { const unsigned long long w = __shfl_xor_sync(0xffffffffu, key, o); key = w > key ? w : key; }
      if (tid == 0) round_update(key, best, true, n, K, a.prob, log1mp, &sh_tries);
    }
    __syncthreads();
  }

  // winner -> consensus set -> least squares, as batch_kernel
  if (tid == 0) {
    sh_best = best;
    sh_ok = winner_constants<M>(best, 0, gb, a.seed, n, rec, 1, D, cfg, sh_prm) ? 1 : 0;
  }
  __syncthreads();
  const uint32_t best_count = (uint32_t)(sh_best >> 32);
  uint8_t* mask_out = a.out_masks ? a.out_masks + off + lo : nullptr;
  if (!sh_ok) {
    if (rank == 0) {
      if (tid == 0) a.out_counts[b] = best_count;
      for (uint32_t i = tid; i < (uint32_t)P; i += kClusterThreads) a.out_params[(size_t)b * P + i] = nan;
    }
    if (mask_out) for (uint32_t i = tid; i < ns; i += kClusterThreads) mask_out[i] = 0;
    cluster.sync();   // no CTA leaves while another may still read its partial counts
    return;
  }
  double hq[HQ];
#pragma unroll
  for (int j = 0; j < HQ; j++) hq[j] = sh_prm[j];
  const double* x64 = use32 ? rec + (size_t)lo * D : pts;   // this CTA's fp64 records
  const uint32_t ld64 = use32 ? 1u : S, st64 = use32 ? (uint32_t)D : 1u;
  uint32_t pass = 0;
  block_moments<M, true>(x64, ns, ld64, st64, sh_ctr, hq, cfg, nullptr, false, 1, mask_out, sh_part, sh_mom[pass & 1]);
  cluster_sum(cluster, sh_mom[pass++ & 1], Mom<M>::N, sh_tot);
  const bool lm = Model<M>::FAM == FAM_SPHERE && ls_type == 1;   // geometric sphere fit: Levenberg-Marquardt from the algebraic fit
  if (tid == 0) {
    double p[LSQR_MAX_PARAMS];
    int np = 0;
    if constexpr (M != USXW && M != USCP) np = solve_model(M, sh_tot, sh_ctr, lm ? 1 : 0, p);   // LM starts in centred coordinates
    sh_out[0] = np;
    for (int j = 0; j < np; j++) sh_out[1 + j] = p[j];
  }
  __syncthreads();
  if constexpr (Model<M>::FAM == FAM_SPHERE) {
    if (lm) {
      constexpr int NPL = Mom<M>::NPLM;
      __shared__ double sh_bcast[1 + NPL];
      if (tid == 0) {
        for (int i = 0; i < LM_SIZE; i++) sh_state[i] = 0.0;
        const int np = (int)sh_out[0];
        if (np == 0) sh_state[LM_STATUS] = 2.0;
        for (int j = 0; j < np; j++) sh_state[LM_X + j] = sh_out[1 + j];
      }
      // every CTA keeps its own copy of the controller state: identical moments give identical updates
      for (;;) {
        __syncthreads();
        if (tid == 0) {
          sh_bcast[0] = sh_state[LM_STATUS];
          const int o = (sh_state[LM_PHASE] != 0.0) ? LM_TRIAL : LM_X;
          for (int j = 0; j < NPL; j++) sh_bcast[1 + j] = sh_state[o + j];
        }
        __syncthreads();
        double lmx[NPL];
        const double status = sh_bcast[0];
        for (int j = 0; j < NPL; j++) lmx[j] = sh_bcast[1 + j];
        if (status != 0.0) break;
        block_moments<M, true>(x64, ns, ld64, st64, sh_ctr, hq, cfg, lmx, true, 1, nullptr, sh_part, sh_mom[pass & 1]);
        cluster_sum(cluster, sh_mom[pass++ & 1], Mom<M>::NLM, sh_tot);
        if (tid == 0) lm_update_model(M, sh_tot, sh_state);
      }
      if (tid == 0) {
        if (sh_state[LM_STATUS] != 1.0) sh_out[0] = 0.0;
        else {
          for (int j = 0; j < Model<M>::DIM; j++) sh_out[1 + j] = sh_state[LM_X + j] + sh_ctr[j];
          sh_out[1 + Model<M>::DIM] = sh_state[LM_X + Model<M>::DIM];
        }
      }
      __syncthreads();
    }
  }
  if (rank == 0) {
    if (tid == 0) a.out_counts[b] = use32 ? (uint32_t)sh_tot[0] : best_count;   // the fp64 count of the winner's consensus set
    const int np = (int)sh_out[0];
    for (uint32_t i = tid; i < (uint32_t)P; i += kClusterThreads) a.out_params[(size_t)b * P + i] = np ? sh_out[1 + i] : nan;
  }
  cluster.sync();   // no CTA leaves while another may still read its moments
}

int launch_batch(const BatchArgs& a, const EstCfg& cfg, int ls_type, cudaStream_t s) {
  if (a.n_problems == 0) return 0;
  const int D = model_info(a.model).D;
  const bool use32 = a.precision == 1 && !a.exhaustive;
  const size_t smem = (size_t)D * a.max_n * sizeof(double) + (use32 ? (size_t)D * ((a.max_n + 1u) & ~1u) * sizeof(float) : 0);
  if (smem > 200 * 1024) return -1;
  const int threads = a.exhaustive ? 256 : 64;
  const uint32_t group = a.exhaustive ? 1u : 2u;
#define CALL(MM)                                                                                  \
  {                                                                                               \
    auto kern = batch_kernel<MM>;                                                                 \
    allow_dynamic_smem(kern, smem);                                                               \
    kern<<<a.n_problems, threads, smem, s>>>(a, cfg, ls_type, group);                            \
  }
#define LSQR_DEF_(ID, DIM) case ID: CALL(ID) break;
  switch (a.model) {
    case PLANE3: CALL(PLANE3) break;
    case LINE2D: CALL(LINE2D) break;
    LSQR_PLANE_ND_LIST(LSQR_DEF_)
    LSQR_LINE_ND_LIST(LSQR_DEF_)
    LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
    LSQR_DENSE_N_LIST(LSQR_DEF_)
    case ABSOR: CALL(ABSOR) break;
    case RAY: CALL(RAY) break;
    case PIVOT: CALL(PIVOT) break;
    default: return -1;
  }
#undef LSQR_DEF_
#undef CALL
  return 1;
}

// ---- the cluster path: limits and launch --------------------------------------------------
namespace {
constexpr size_t kBatchSmem = 200 * 1024;   // dynamic shared memory of one block of either kernel

size_t cluster_smem(int D, bool use32, uint32_t slice) { return (size_t)D * slice * (use32 ? sizeof(float) : sizeof(double)); }

const void* cluster_kernel(int model) {
#define CALL(MM) return reinterpret_cast<const void*>(batch_cluster_kernel<MM>);
#define LSQR_DEF_(ID, DIM) case ID: CALL(ID)
  switch (model) {
    case PLANE3: CALL(PLANE3)
    case LINE2D: CALL(LINE2D)
    LSQR_PLANE_ND_LIST(LSQR_DEF_)
    LSQR_LINE_ND_LIST(LSQR_DEF_)
    LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
    LSQR_DENSE_N_LIST(LSQR_DEF_)
    case ABSOR: CALL(ABSOR)
    case RAY: CALL(RAY)
    case PIVOT: CALL(PIVOT)
    default: return nullptr;
  }
#undef LSQR_DEF_
#undef CALL
}

// Largest cluster the current device schedules for one cluster kernel with `smem` bytes per CTA: 16 CTAs are beyond the
// portable cluster size, so the kernel is allowed them and the occupancy calculator asked whether one such cluster fits;
// otherwise 8.  Once per kernel, size and device.
int cluster_max(const void* kern, size_t smem) {
  static std::mutex mu;
  static std::map<std::tuple<const void*, size_t, int>, int> known;
  int dev = 0;
  cudaGetDevice(&dev);
  {
    std::lock_guard<std::mutex> lock(mu);
    auto it = known.find({kern, smem, dev});
    if (it != known.end()) return it->second;
  }
  allow_dynamic_smem(kern, smem);
  int cmax = 8;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(16); lc.blockDim = dim3(kClusterThreads); lc.dynamicSmemBytes = smem;
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = 16; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
    lc.attrs = &at; lc.numAttrs = 1;
    int clusters = 0;
    if (cudaOccupancyMaxActiveClusters(&clusters, kern, &lc) == cudaSuccess && clusters > 0) cmax = 16;
  }
  cudaGetLastError();   // a refused query is an answer (8), not an error of the next launch
  std::lock_guard<std::mutex> lock(mu);
  known[{kern, smem, dev}] = cmax;
  return cmax;
}
}  // namespace

BatchLimits batch_limits(int model, int precision, int exhaustive) {
  BatchLimits L{};
  const uint64_t D = (uint64_t)model_info(model).D;
  const bool use32 = precision == 1 && !exhaustive;
  // one block: the records and, for fp32 scoring, their fp32 copy padded to even (launch_batch's shared memory)
  uint64_t n = (kBatchSmem - 16) / (D * (sizeof(double) + (use32 ? sizeof(float) : 0)));
  while (n > 0 && D * n * sizeof(double) + (use32 ? D * ((n + 1) & ~1ull) * sizeof(float) : 0) > kBatchSmem) n--;
  L.one_block = L.max_records = n;
  const void* kern = cluster_kernel(model);
  if (exhaustive || !kern) return L;
  L.slice = (uint32_t)(kBatchSmem / (D * (use32 ? sizeof(float) : sizeof(double)))) & ~1u;
  L.max_cluster = cluster_max(kern, cluster_smem((int)D, use32, L.slice));
  L.max_records = std::max<uint64_t>(n, (uint64_t)L.max_cluster * L.slice);
  return L;
}

int launch_batch_cluster(const BatchArgs& a, const uint32_t* problems, uint32_t count, uint32_t cluster, uint32_t slice, const EstCfg& cfg,
                         int ls_type, cudaStream_t s) {
  const void* kern = cluster_kernel(a.model);
  if (!kern) return -1;
  if (count == 0) return 0;
  const size_t smem = cluster_smem(model_info(a.model).D, a.precision == 1, slice);
  allow_dynamic_smem(kern, smem);
  cudaLaunchConfig_t lc{};
  lc.gridDim = dim3(count * cluster); lc.blockDim = dim3(kClusterThreads); lc.dynamicSmemBytes = smem; lc.stream = s;
  cudaLaunchAttribute at{};
  at.id = cudaLaunchAttributeClusterDimension;
  at.val.clusterDim.x = cluster; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
  lc.attrs = &at; lc.numAttrs = 1;
  BatchArgs args = a;
  EstCfg c = cfg;
  void* params[] = {&args, &problems, &c, &ls_type};
  return cudaLaunchKernelExC(&lc, kern, params) == cudaSuccess ? 1 : -1;
}

// ---------------------------------------------------------------------------------------
// Batched least squares (lsqr_least_squares_batch_device): leastSquaresEstimate of every problem of a batch over its selected
// records, one cluster of C CTAs per problem (C from ls_batch_cluster).  CTA r takes records [r S, min((r + 1) S, n)),
// S = ceil(n / C), and streams them from global memory -- nothing stays resident, so a problem has no size limit.  Record j of
// the slice goes to thread j % kLsThreads, in increasing j, whatever the path that brings it in; moments are taken relative to
// the problem's first record and reduced within the block, then over the cluster in rank order, so a problem's result depends
// on its records and the device only.  Thread 0 of every CTA solves the same sums; for the geometric sphere fit every CTA runs
// the same Levenberg-Marquardt controller, one streaming pass per evaluation.
//
// The slice is packed AoS doubles whose start need not be 16-byte aligned.  Tiles of TR records pass through the TileRing as
// one bulk copy each, taken from the first 16-byte boundary of the slice (h = 1 double in when the slice starts off it): a tile
// then lacks the first double of its first record, which that record's thread reads from global memory.  The records after the
// last whole tile are read with plain loads.
// ---------------------------------------------------------------------------------------
constexpr int kLsThreads = 256;
// records per tile: about 12 KB of 2- and 3-D records (two or three per thread), one record per thread above
__host__ __device__ constexpr int ls_tile_records(int D) { return kLsThreads * (D <= 3 ? 6 / D : 1); }
__host__ __device__ constexpr size_t ls_smem(int D) { return 2 * (size_t)ls_tile_records(D) * D * sizeof(double); }

struct LsSlice {
  const double* x;        // the CTA's records
  uint32_t h, tiles, ns;  // 1 when x is not 16-byte aligned; whole tiles; records
  const uint8_t* masks;   // the CTA's mask bytes, or null
  const double* weights;  // the CTA's weights (weighted Horn)
};

// One streaming pass over the CTA's records -> the block's NM moments in `out` (thread tid < NM), read after a block or cluster
// barrier.  LM: the sphere's Levenberg-Marquardt moments at lmx; W: weighted Horn with the number of pairs in [16].
template <int M, bool W, bool LM, int NM, int TD>
__device__ __forceinline__ void ls_pass(TileRing<1, TD, double>& ring, const LsSlice& sl, const double* sh_ctr, const double* lmx, double* sh_part,
                                        double* out) {
  constexpr int D = Model<M>::D, TR = TD / D;
  const uint32_t tid = threadIdx.x;
  double ctr[D];
#pragma unroll
  for (int d = 0; d < D; d++) ctr[d] = sh_ctr[d];
  double acc[NM];
#pragma unroll
  for (int j = 0; j < NM; j++) acc[j] = 0.0;
  auto take = [&](uint32_t j, const double* x) {
    if (sl.masks && !sl.masks[j]) return;
    double q[D];
#pragma unroll
    for (int d = 0; d < D; d++) q[d] = x[d] - ctr[d];
    if constexpr (LM) acc_sphere_lm<Model<M>::DIM>(q, lmx, acc);
    else if constexpr (W) { acc_absor_weighted(q, sl.weights[j], acc); acc[16] += 1.0; }
    else { acc[0] += 1.0; accumulate<M>(q, acc); }
  };
  for (uint32_t t = 0; t < sl.tiles; t++) {
    const double* tile = ring.wait(t);
#pragma unroll
    for (int u = 0; u < TR / kLsThreads; u++) {
      const uint32_t r = u * kLsThreads + tid;
      double x[D];
#pragma unroll
      for (int d = 0; d < D; d++) {
        const int e = (int)(r * D + d) - (int)sl.h;
        x[d] = e >= 0 ? tile[e] : sl.x[(size_t)t * TD];
      }
      take(t * TR + r, x);
    }
    ring.release();
  }
  for (uint32_t j = sl.tiles * TR + tid; j < sl.ns; j += kLsThreads) {
    double x[D];
#pragma unroll
    for (int d = 0; d < D; d++) x[d] = sl.x[(size_t)j * D + d];
    take(j, x);
  }
  const uint32_t lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int j = 0; j < NM; j++) {
    double v = acc[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) sh_part[warp * NM + j] = v;
  }
  __syncthreads();
  if (tid < (uint32_t)NM) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < kLsThreads / 32; w++) v += sh_part[w * NM + tid];
    out[tid] = v;
  }
}

template <int M, bool W>
__global__ void __launch_bounds__(kLsThreads) ls_batch_kernel(LsBatchArgs a, const uint32_t* __restrict__ problems, int ls_type) {
  constexpr int D = Model<M>::D, P = Model<M>::P, K = Model<M>::K;
  constexpr int TD = ls_tile_records(D) * D;
  constexpr bool kSphere = Model<M>::FAM == FAM_SPHERE;
  constexpr int NA = W ? 17 : Mom<M>::N;          // the analytic pass; weighted Horn counts the pairs in [16]
  constexpr int NL = kSphere ? Mom<M>::NLM : 1;   // a Levenberg-Marquardt pass
  constexpr int NMAX = NA > NL ? NA : NL;
  const cg::cluster_group cluster = cg::this_cluster();
  const uint32_t C = cluster.num_blocks(), rank = cluster.block_rank(), tid = threadIdx.x;
  extern __shared__ __align__(16) unsigned char ls_smem_raw[];   // the tile ring: 2 x TD doubles
  __shared__ __align__(8) uint64_t sh_bars[2];
  __shared__ double sh_part[(kLsThreads / 32) * NMAX];
  __shared__ double sh_mom[2][NMAX];   // this CTA's moments, by pass parity
  __shared__ double sh_tot[NMAX];      // the cluster's
  __shared__ double sh_out[LSQR_MAX_PARAMS + 4];
  __shared__ double sh_state[LM_SIZE];
  __shared__ double sh_ctr[kMaxDim];

  const uint32_t b = problems[blockIdx.x / C];
  const uint64_t off = a.offsets[b];
  const uint32_t n = (uint32_t)(a.offsets[b + 1] - off);
  const double* rec = a.data + off * D;
  const uint32_t S = (uint32_t)(((uint64_t)n + C - 1) / C);
  const uint32_t lo = min(rank * S, n), ns = min(S, n - lo);
  LsSlice sl;
  sl.x = rec + (size_t)lo * D;
  sl.h = (uint32_t)((reinterpret_cast<uintptr_t>(sl.x) >> 3) & 1u);
  sl.tiles = (uint64_t)ns * D >= sl.h ? (uint32_t)(((uint64_t)ns * D - sl.h) / TD) : 0u;
  sl.ns = ns;
  sl.masks = a.masks ? a.masks + off + lo : nullptr;
  sl.weights = W ? a.weights + off + lo : nullptr;
  if (tid < (uint32_t)kMaxDim) sh_ctr[tid] = (n > 0 && tid < (uint32_t)D && centred_component(M, (int)tid)) ? rec[tid] : 0.0;
  TileRing<1, TD, double> ring{sl.x + sl.h, 0, 0, sl.tiles, reinterpret_cast<double*>(ls_smem_raw), sh_bars, (int)tid};
  ring.start();   // (its barrier also publishes sh_ctr)

  uint32_t pass = 0;
  ls_pass<M, W, false, NA>(ring, sl, sh_ctr, nullptr, sh_part, sh_mom[pass & 1]);
  cluster_sum(cluster, sh_mom[pass++ & 1], NA, sh_tot);
  const bool lm = kSphere && ls_type == 1;   // geometric sphere fit: Levenberg-Marquardt from the algebraic fit
  if (tid == 0) {
    // the size guards of lsqr_least_squares / lsqr_weighted_least_squares on the selected records
    double p[LSQR_MAX_PARAMS];
    int np = 0;
    if constexpr (W) {
      if (sh_tot[16] >= 3.0) np = solve_absor(sh_tot, sh_ctr, p, true);
    } else if (sh_tot[0] >= (double)K || (M == RAY && sh_tot[0] > 0.0)) {
      np = solve_model(M, sh_tot, sh_ctr, lm ? 1 : 0, p);   // LM starts in centred coordinates
    }
    sh_out[0] = np;
    for (int j = 0; j < np; j++) sh_out[1 + j] = p[j];
  }
  __syncthreads();
  if constexpr (kSphere) {
    if (lm) {   // batch_cluster_kernel's loop, with a streaming pass per evaluation
      constexpr int NPL = Mom<M>::NPLM;
      __shared__ double sh_bcast[1 + NPL];
      if (tid == 0) {
        for (int i = 0; i < LM_SIZE; i++) sh_state[i] = 0.0;
        const int np = (int)sh_out[0];
        if (np == 0) sh_state[LM_STATUS] = 2.0;
        for (int j = 0; j < np; j++) sh_state[LM_X + j] = sh_out[1 + j];
      }
      for (;;) {
        __syncthreads();
        if (tid == 0) {
          sh_bcast[0] = sh_state[LM_STATUS];
          const int o = (sh_state[LM_PHASE] != 0.0) ? LM_TRIAL : LM_X;
          for (int j = 0; j < NPL; j++) sh_bcast[1 + j] = sh_state[o + j];
        }
        __syncthreads();
        double lmx[NPL];
        const double status = sh_bcast[0];
        for (int j = 0; j < NPL; j++) lmx[j] = sh_bcast[1 + j];
        if (status != 0.0) break;
        ring.restart();
        ls_pass<M, W, true, NL>(ring, sl, sh_ctr, lmx, sh_part, sh_mom[pass & 1]);
        cluster_sum(cluster, sh_mom[pass++ & 1], NL, sh_tot);
        if (tid == 0) lm_update_model(M, sh_tot, sh_state);
      }
      if (tid == 0) {
        if (sh_state[LM_STATUS] != 1.0) sh_out[0] = 0.0;
        else {
          for (int j = 0; j < Model<M>::DIM; j++) sh_out[1 + j] = sh_state[LM_X + j] + sh_ctr[j];
          sh_out[1 + Model<M>::DIM] = sh_state[LM_X + Model<M>::DIM];
        }
      }
      __syncthreads();
    }
  }
  if (rank == 0) {
    const int np = (int)sh_out[0];
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (uint32_t i = tid; i < (uint32_t)P; i += kLsThreads) a.out_params[(size_t)b * P + i] = np ? sh_out[1 + i] : nan;
  }
  cluster.sync();   // no CTA leaves while another may still read its moments
}

namespace {
const void* ls_kernel(int model, bool weighted) {
  if (weighted) return model == ABSOR ? reinterpret_cast<const void*>(ls_batch_kernel<ABSOR, true>) : nullptr;
#define CALL(MM) return reinterpret_cast<const void*>(ls_batch_kernel<MM, false>);
#define LSQR_DEF_(ID, DIM) case ID: CALL(ID)
  switch (model) {
    case PLANE3: CALL(PLANE3)
    case LINE2D: CALL(LINE2D)
    LSQR_PLANE_ND_LIST(LSQR_DEF_)
    LSQR_LINE_ND_LIST(LSQR_DEF_)
    LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
    LSQR_DENSE_N_LIST(LSQR_DEF_)
    case ABSOR: CALL(ABSOR)
    case RAY: CALL(RAY)
    case PIVOT: CALL(PIVOT)
    default: return nullptr;
  }
#undef LSQR_DEF_
#undef CALL
}
}  // namespace

int ls_batch_max_cluster(int model, bool weighted) {
  const void* kern = ls_kernel(model, weighted);
  return kern ? cluster_max(kern, ls_smem(model_info(model).D)) : 0;
}

int launch_ls_batch(const LsBatchArgs& a, const uint32_t* problems, uint32_t count, uint32_t cluster, int ls_type, cudaStream_t s) {
  const void* kern = ls_kernel(a.model, a.weights != nullptr);
  if (!kern) return -1;
  if (count == 0) return 0;
  const size_t smem = ls_smem(model_info(a.model).D);
  allow_dynamic_smem(kern, smem);
  cudaLaunchConfig_t lc{};
  lc.gridDim = dim3(count * cluster); lc.blockDim = dim3(kLsThreads); lc.dynamicSmemBytes = smem; lc.stream = s;
  cudaLaunchAttribute at{};
  at.id = cudaLaunchAttributeClusterDimension;
  at.val.clusterDim.x = cluster; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
  if (cluster > 1) { lc.attrs = &at; lc.numAttrs = 1; }   // one CTA per problem: a plain launch
  LsBatchArgs args = a;
  void* params[] = {&args, &problems, &ls_type};
  return cudaLaunchKernelExC(&lc, kern, params) == cudaSuccess ? 1 : -1;
}

}  // namespace lsqr
