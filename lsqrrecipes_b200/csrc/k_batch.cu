// Batched small problems (BASELINE.json configs[4]): one thread block per problem, see the comment above batch_kernel.
#include "refine_common.cuh"
#include "fast_forms.cuh"

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

template <int M>
__device__ void block_moments(const double* pts, uint32_t n, uint32_t ldp, const double* hq, const EstCfg& cfg, const double* lmx, bool lm,
                              int use_mask, uint8_t* mask_out, double* sh_part, double* sh_mom) {
  constexpr int D = Model<M>::D;
  constexpr int NMA = Mom<M>::N, NML = Mom<M>::NLM;
  double acc[kMaxMoments];
  const int nm = lm ? NML : NMA;
  for (int j = 0; j < kMaxMoments; j++) acc[j] = 0.0;
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    double x[D];
#pragma unroll
    for (int d = 0; d < D; d++) x[d] = pts[d * ldp + i];
    const bool in = use_mask ? agree<M>(hq, x, cfg) : true;
    if (mask_out) mask_out[i] = in ? 1 : 0;
    if (in) {
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
      double sp[K * D], prm[P], hq[HQ];
#pragma unroll
      for (int j = 0; j < K; j++)
#pragma unroll
        for (int d = 0; d < D; d++) sp[j * D + d] = pts[d * ldp + sub[j]];
      const bool ok = estimate<M>(sp, cfg, prm);   // the same for all G threads of a hypothesis
      uint32_t c = 0;
      if (ok && use32) {
        if constexpr (M != USXW && M != USCP) {   // (the ultrasound calibrations have no batched mode)
          constexpr int Q = Model<M>::Q32;
          double ctr[kMaxDim];
#pragma unroll
          for (int d = 0; d < kMaxDim; d++) ctr[d] = sh_ctr[d];
          float qf[Q];
          hoist32<M>(prm, ctr, cfg, qf);
          f2 q[Q];
#pragma unroll
          for (int j = 0; j < Q; j++) q[j] = splat(qf[j]);
          Thr2 thr;
          thr.delta = splat((float)cfg.delta); thr.neg_delta2 = splat(-(float)cfg.delta2); thr.fdelta = (float)cfg.delta;
          const uint32_t negk = hyp_negk<M>(qf, 0u - __float_as_uint(2.0f * (float)cfg.delta));   // 2^32 - bits(window)
          unsigned long long out = 0ull;
          uint32_t pairs = 0;
          for (uint32_t i = 2 * sub_lane; i < n; i += 2 * G) {
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
      } else if (ok) {
        prepare<M>(prm, cfg, hq);
        for (uint32_t i = sub_lane; i < n; i += G) {
          double x[D];
#pragma unroll
          for (int d = 0; d < D; d++) x[d] = pts[d * ldp + i];
          c += agree<M>(hq, x, cfg) ? 1u : 0u;
        }
      }
      if (G > 1) {   // uniform over the block; the G threads of a hypothesis are adjacent lanes of one warp
        const unsigned grp = (0xFFFFFFFFu >> (32u - G)) << ((threadIdx.x & 31u) & ~(G - 1u));
        for (uint32_t o = 1; o < G; o <<= 1) c += __shfl_xor_sync(grp, c, o);
      }
      if (ok) key = ((unsigned long long)c << 32) | (0xFFFFFFFFull - h);
    }
    const unsigned long long round_best = block_max_u64(key, sh_key);
    if (round_best > best) {
      best = round_best;
      if (!a.exhaustive && threadIdx.x == 0) {  // stop rule, RANSAC.hxx:104-110
        const uint32_t c = (uint32_t)(best >> 32);
        unsigned long long cap = sh_tries;
        if (c == n) cap = 0;
        else if (a.prob > 0.0 && a.prob < 1.0) {
          const double den = log(1.0 - pow((double)c / (double)n, (double)K));
          const double t = log1mp / den + 0.5;
          const unsigned long long nt = t >= 4294967295.0 ? 0xFFFFFFFFull : (unsigned long long)(long long)t;
          cap = nt < cap ? nt : cap;
        }
        sh_tries = cap;
      }
    }
    __syncthreads();
  }

  // winner -> consensus set -> least squares (RANSAC.hxx:129-138)
  const uint32_t best_count = (uint32_t)(best >> 32);
  if (threadIdx.x == 0) {
    sh_ok = 0;
    if (best_count > 0) {
      const unsigned long long h = 0xFFFFFFFFull - (best & 0xFFFFFFFFull);
      int32_t sub[K];
      if (a.exhaustive) unrank_lex<K>(h, n, sub); else sample_subset<K>((gb << 32) | h, a.seed, n, sub);
      double sp[K * D], prm[P];
      for (int j = 0; j < K; j++) for (int d = 0; d < D; d++) sp[j * D + d] = pts[d * ldp + sub[j]];
      if (estimate<M>(sp, cfg, prm)) { prepare<M>(prm, cfg, sh_prm); sh_ok = 1; }
    }
  }
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
  block_moments<M>(pts, n, ldp, hq, cfg, nullptr, false, 1, mask_out, sh_part, sh_mom);
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
        block_moments<M>(pts, n, ldp, hq, cfg, lmx, true, 1, nullptr, sh_part, sh_mom);
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

}  // namespace lsqr
