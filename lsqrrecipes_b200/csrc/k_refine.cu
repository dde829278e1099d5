// Consensus set + least-squares refine (RANSAC.hxx:129-138 and the estimators'
// leastSquaresEstimate bodies).
//
// One streaming pass per refine: every datum is read once from the fp64 SoA arrays, agree() is
// evaluated in reference arithmetic against the winning hypothesis, the consensus bit is written
// (one 32-bit word per warp via ballot) and -- in the same pass -- the estimator's least-squares
// moments are accumulated over the inliers in fp64.  The kernel is HBM-bound: D*8 bytes read per
// datum, 1 bit written.  Per-block partial sums are combined in a fixed order (reproducible), and a
// single-thread kernel turns the moments into parameters with small Jacobi eigen / pseudo-inverse
// solves.  The sphere's geometric fit runs Levenberg-Marquardt with one such pass per function
// evaluation (J^T J, J^T r and the cost in one sweep) and an on-device controller.
//
// All position components are accumulated relative to dv.center (shift-invariant scatter / normal
// equations), which keeps the fp64 sums well conditioned for coordinates far from the origin.
#include "bulk_copy.cuh"
#include "refine_common.cuh"

namespace lsqr {

int moments_count(int model, bool lm) { return n_moments(model, lm); }

// Blocking of the streaming pass: one persistent CTA per SM walks tiles of TILE data; a tile is D rows of TILE doubles in
// shared memory, filled by D bulk copies (cp.async.bulk, one mbarrier per stage), STAGES tiles deep.  The bytes in flight per
// SM are (STAGES - 1) tiles whatever the compute phase of the warps is -- what the register-staged version lacked
// (profiles/r01_ncu_mask_moments_v2.txt: 25 % warps active, wait + long_scoreboard 60 %, 0.62 of HBM).  Tiles of ~48 KB
// (2048 3-D points: four rows of 32 per thread, interleaved) x 4 stages measured best (profiles/r02_tune_mm.txt).
#ifndef LSQR_MM_SMEM_KB
#define LSQR_MM_SMEM_KB 208
#endif
#ifndef LSQR_MM_TILE_KB
#define LSQR_MM_TILE_KB 48
#endif
#ifndef LSQR_MM_THREADS
#define LSQR_MM_THREADS 512
#endif
template <int M, bool LM> struct MMCfg {
  static constexpr int D = Model<M>::D;
  static constexpr int NM = LM ? Mom<M>::NLM : Mom<M>::N;
  // models with more than 40 accumulators per thread (the two ultrasound calibrations: 46-91 doubles) get the whole register
  // file of an SM for 256 threads; everyone else runs 512 threads
  static constexpr int THREADS = NM > 40 ? 256 : LSQR_MM_THREADS;
  static constexpr int kTileCap = LSQR_MM_TILE_KB * 1024 + 8192;
  static constexpr int TILE = (D * 2048 * 8 <= kTileCap) ? 2048 : (D * 1024 * 8 <= kTileCap) ? 1024 : ((D * 512 * 8 <= kTileCap) ? 512 : 256);
  static_assert(kTilePad % TILE == 0, "a tile must never straddle the end of a row (rows are kTilePad-padded)");
  static constexpr int PPT = (TILE + THREADS - 1) / THREADS;                 // data per thread per tile
  static constexpr int TILE_BYTES = D * TILE * 8;
  static constexpr int kFit = LSQR_MM_SMEM_KB * 1024 / TILE_BYTES;
  static constexpr int STAGES = kFit >= 8 ? 8 : (kFit >= 2 ? kFit : 2);      // stage and phase are carried as counters, no division
  static constexpr size_t SMEM = (size_t)STAGES * TILE_BYTES;
  // light moment sets are accumulated without a branch (zeros for data outside the consensus set): the rows of a tile are
  // then independent straight-line chains that the scheduler interleaves; Levenberg-Marquardt rows (sqrt, division) and the
  // 46-91-term calibration rows stay behind a branch
  static constexpr bool BRANCHLESS = !LM && NM <= 32;
};
int mask_moments_ctas_per_sm() { return 1; }

// MODE 0: every datum counts; 1: evaluate agree() and write the consensus bits (and, when maskbytes != nullptr, the
// std::vector<bool>-shaped byte per datum that the caller of compute() receives); 2: read stored bits.
// HBM-bound: D*8 bytes read per datum, 1 bit (or 1 byte + 1 bit) written.
template <int M, int MODE, bool LM>
__global__ void __launch_bounds__(MMCfg<M, LM>::THREADS, 1) mask_moments_kernel(DataView dv, uint32_t begin, uint32_t end, const double* __restrict__ params_dev,
                                                               const double* __restrict__ lm_state, EstCfg cfg, uint32_t* __restrict__ maskbits,
                                                               uint8_t* __restrict__ maskbytes, double* __restrict__ partials) {
  using C = MMCfg<M, LM>;
  constexpr int D = Model<M>::D, P = Model<M>::P, HQ = Model<M>::HQ;
  constexpr int NM = C::NM, TILE = C::TILE, THREADS = C::THREADS, PPT = C::PPT, STAGES = C::STAGES;
  constexpr bool kFullTile = PPT * THREADS == TILE;
  extern __shared__ __align__(128) unsigned char mm_smem_raw[];
  double* ring = reinterpret_cast<double*>(mm_smem_raw);                     // [STAGES][D][TILE]
  __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES];
  __shared__ double sh[THREADS / 32][NM > 0 ? NM : 1];
  const uint32_t tid = threadIdx.x, lane = tid & 31;

  // LM passes are enqueued a few evaluations ahead of the controller's status word: once the iteration has stopped, the
  // remaining passes are no-ops (the controller ignores the stale moments)
  const bool active = !LM || lm_state[LM_STATUS] == 0.0;
  // tiles [t0, t1) in units of TILE data cover [begin, end); this CTA takes t0 + blockIdx.x, + gridDim.x, ...
  const uint32_t t0 = begin / TILE, t1 = (uint32_t)(((uint64_t)end + TILE - 1) / TILE);
  const uint32_t first = t0 + blockIdx.x;
  const uint32_t n_mine = (active && first < t1) ? (t1 - first + gridDim.x - 1) / gridDim.x : 0;
  auto issue = [&](uint32_t k, uint32_t s) {   // tile number k of this CTA into stage s
    const size_t base = (size_t)(first + k * gridDim.x) * TILE;
    double* dst = ring + (size_t)s * D * TILE;
    mbar_expect_tx(&full_bar[s], (uint32_t)C::TILE_BYTES);
#pragma unroll
    for (int d = 0; d < D; d++) bulk_g2s(dst + d * TILE, dv.soa64 + (size_t)d * dv.ld + base, TILE * 8, &full_bar[s]);
  };
  // the first tiles are on their way before anything else is set up
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; s++) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], THREADS / 32); }
    mbar_fence_init();
    for (uint32_t k = 0; k < (uint32_t)STAGES && k < n_mine; k++) issue(k, k);
  }

  double acc[NM > 0 ? NM : 1];
#pragma unroll
  for (int j = 0; j < NM; j++) acc[j] = 0.0;
  double hq[HQ];
  if (MODE == 1) {
    double prm[P];
#pragma unroll
    for (int j = 0; j < P; j++) prm[j] = params_dev[j];
    prepare<M>(prm, cfg, hq);
  }
  // the shift c of the centred components, once per thread (a load inside the loop would put a global-memory latency on every
  // row's critical path)
  double ctr[D];
#pragma unroll
  for (int d = 0; d < D; d++) ctr[d] = centred_component(M, d) ? dv.center[d] : 0.0;
  double lmx[LM ? Mom<M>::NPLM : 1] = {0};
  if (LM) {
    // the phase selects the evaluation point: x or the trial point
    const int off = (lm_state[LM_PHASE] != 0.0) ? LM_TRIAL : LM_X;
#pragma unroll
    for (int j = 0; j < Mom<M>::NPLM; j++) lmx[j] = lm_state[off + j];
  }
  __syncthreads();   // barriers initialised before anyone waits on them

  // one tile: `checked` tiles straddle begin / end (at most two per launch) and test every row against the range
  auto process = [&](const double (&x)[PPT][D], uint32_t base, bool checked) {
    bool in[PPT], rowok[PPT];
#pragma unroll
    for (int u = 0; u < PPT; u++) {
      const uint32_t p = u * THREADS + tid, i = base + p, row = i - lane;      // rows of 32 data start on multiples of 32
      rowok[u] = (kFullTile || p < (uint32_t)TILE) && (!checked || (row >= begin && row < end));   // warp-uniform
      const bool valid = rowok[u] && (!checked || i < end);
      if (MODE == 0) in[u] = valid;
      else if (MODE == 1) in[u] = valid && agree<M>(hq, x[u], cfg);   // NaN padding beyond n never agrees
      else in[u] = valid && ((maskbits[row >> 5] >> lane) & 1u);
    }
    if (MODE == 1) {
#pragma unroll
      for (int u = 0; u < PPT; u++) {
        const uint32_t p = u * THREADS + tid, i = base + p;
        const unsigned bits = __ballot_sync(0xffffffffu, in[u]);
        if (rowok[u]) {
          if (lane == 0) maskbits[(i - lane) >> 5] = bits;
          if (maskbytes != nullptr && i < end) maskbytes[i] = in[u] ? 1 : 0;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < PPT; u++) {
      if constexpr (C::BRANCHLESS) {
        double q[D];
#pragma unroll
        for (int d = 0; d < D; d++) q[d] = in[u] ? x[u][d] - ctr[d] : 0.0;
        acc[0] += in[u] ? 1.0 : 0.0;
        accumulate<M>(q, acc);
      } else if (in[u]) {
        double q[D];
#pragma unroll
        for (int d = 0; d < D; d++) q[d] = x[u][d] - ctr[d];
        if (LM) {
          if constexpr (Model<M>::FAM == FAM_SPHERE) acc_sphere_lm<Model<M>::DIM>(q, lmx, acc);
          if constexpr (M == USXW) acc_us_lm(q, lmx, acc);
          if constexpr (M == USCP) acc_uscp_lm(q, lmx, acc);
        } else { acc[0] += 1.0; accumulate<M>(q, acc); }
      }
    }
  };

  uint32_t s = 0, parity = 0;
  for (uint32_t k = 0; k < n_mine; k++) {
    const uint32_t base = (first + k * gridDim.x) * (uint32_t)TILE;
    const double* tile = ring + (size_t)s * D * TILE;
    mbar_wait(&full_bar[s], parity);
    double x[PPT][D];
#pragma unroll
    for (int u = 0; u < PPT; u++) {
      const uint32_t p = u * THREADS + tid;
      if (kFullTile || p < (uint32_t)TILE) {
#pragma unroll
        for (int d = 0; d < D; d++) x[u][d] = tile[d * TILE + p];
      }
    }
    // the stage is free as soon as every warp holds its data in registers; thread 0 refills it STAGES tiles ahead
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
    if (tid == 0 && k + STAGES < n_mine) { mbar_wait(&empty_bar[s], parity); issue(k + STAGES, s); }
    const uint32_t s_next = (s + 1 == (uint32_t)STAGES) ? 0u : s + 1;
    parity ^= (s_next == 0u) ? 1u : 0u;
    s = s_next;
    const bool checked = base < begin || (uint64_t)base + TILE > end;   // CTA-uniform
    if (checked) process(x, base, true); else process(x, base, false);
  }
  if (LM && !active) return;   // partials, moments and the controller state keep their values
  // block reduction: shuffle within warps, shared memory across the warps
#pragma unroll
  for (int j = 0; j < NM; j++) {
    double v = acc[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) sh[tid >> 5][j] = v;
  }
  __syncthreads();
  if ((int)tid < NM) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; w++) v += sh[w][tid];
    partials[(size_t)blockIdx.x * kMaxMoments + tid] = v;
  }
}

template <int M, int MODE, bool LM>
static void run_mask_moments(const DataView& dv, uint32_t begin, uint32_t end, const double* params_dev, const double* lm_state, const EstCfg& cfg,
                             const RefineBuffers& rb, cudaStream_t s) {
  using C = MMCfg<M, LM>;
  auto kern = mask_moments_kernel<M, MODE, LM>;
  allow_dynamic_smem(kern, C::SMEM);
  kern<<<rb.blocks, C::THREADS, C::SMEM, s>>>(dv, begin, end, params_dev, lm_state, cfg, rb.maskbits, rb.maskbytes, rb.partials);
}

void launch_mask_moments(int model, const DataView& dv, uint32_t begin, uint32_t end, const double* params_dev, int mask_mode,
                         const double* lm_state, const EstCfg& cfg, const RefineBuffers& rb, cudaStream_t s) {
#define BYMODE(MM, LMV)                                                                           \
  if (mask_mode == 0) run_mask_moments<MM, 0, LMV>(dv, begin, end, params_dev, lm_state, cfg, rb, s);      \
  else if (mask_mode == 1) run_mask_moments<MM, 1, LMV>(dv, begin, end, params_dev, lm_state, cfg, rb, s); \
  else run_mask_moments<MM, 2, LMV>(dv, begin, end, params_dev, lm_state, cfg, rb, s)
  if (lm_state) {
#define LSQR_DEF_(ID, DIM) case ID: { BYMODE(ID, true); break; }
    switch (model) {
      LSQR_SPHERE_ALL_LIST(LSQR_DEF_)
      case USXW: { BYMODE(USXW, true); break; }
      case USCP: { BYMODE(USCP, true); break; }
      default: break;
    }
#undef LSQR_DEF_
    return;
  }
#define CALL(MM) BYMODE(MM, false)
  LSQR_DISPATCH_MODEL(model, CALL)
#undef CALL
#undef BYMODE
}

// Weighted Horn moments (AbsoluteOrientationParametersEstimator.cxx:217-261): sum w, sum w p1, sum w p2,
// sum w p1 p2^T over all n pairs, relative to dv.center.  Same partials layout as mask_moments_kernel.
__global__ void __launch_bounds__(256) weighted_absor_moments_kernel(DataView dv, const double* __restrict__ w, double* __restrict__ partials) {
  constexpr int NM = 16;
  double acc[NM];
#pragma unroll
  for (int j = 0; j < NM; j++) acc[j] = 0.0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < dv.n; i += (size_t)gridDim.x * blockDim.x) {
    double q[6];
#pragma unroll
    for (int d = 0; d < 6; d++) q[d] = dv.soa64[(size_t)d * dv.ld + i] - dv.center[d];
    acc_absor_weighted(q, w[i], acc);
  }
  __shared__ double sh[8][kMaxMoments];
  const uint32_t lane = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < NM; j++) {
    double v = acc[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) sh[threadIdx.x >> 5][j] = v;
  }
  __syncthreads();
  if ((int)threadIdx.x < NM) {
    double v = 0.0;
#pragma unroll
    for (int wp = 0; wp < 8; wp++) v += sh[wp][threadIdx.x];
    partials[(size_t)blockIdx.x * kMaxMoments + threadIdx.x] = v;
  }
}
void launch_weighted_absor_moments(const DataView& dv, const double* weights_dev, const RefineBuffers& rb, cudaStream_t s) {
  weighted_absor_moments_kernel<<<rb.blocks, 256, 0, s>>>(dv, weights_dev, rb.partials);
}

// One warp per moment; lanes stride over the blocks, then a fixed-order shuffle tree: the summation
// order depends only on the launch geometry, so results are reproducible run to run.
__global__ void reduce_partials_kernel(const double* __restrict__ partials, int blocks, int nm, double* __restrict__ moments) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (j >= nm) return;
  double v = 0.0;
  for (int b = lane; b < blocks; b += 32) v += partials[(size_t)b * kMaxMoments + j];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) moments[j] = v;
}
void launch_reduce_partials(const RefineBuffers& rb, int nm, cudaStream_t s) {
  reduce_partials_kernel<<<(nm + 7) / 8, 256, 0, s>>>(rb.partials, rb.blocks, nm, rb.moments);
}

__global__ void solve_moments_kernel(int model, DataView dv, const double* __restrict__ m, int keep_centred, double* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double p[LSQR_MAX_PARAMS];
  const int np = solve_model(model, m, dv.center, keep_centred, p);
  out[0] = (double)np;
  for (int j = 0; j < np; j++) out[1 + j] = p[j];
}
__global__ void solve_weighted_absor_kernel(DataView dv, const double* __restrict__ m, double* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double p[8];
  const int np = solve_absor(m, dv.center, p, true);
  out[0] = (double)np;
  for (int j = 0; j < np; j++) out[1 + j] = p[j];
}
void launch_solve_weighted_absor(const DataView& dv, const double* moments, double* out_dev, cudaStream_t s) {
  solve_weighted_absor_kernel<<<1, 32, 0, s>>>(dv, moments, out_dev);
}
void launch_solve_moments(int model, const DataView& dv, const double* moments, int keep_centred, double* out_dev, cudaStream_t s) {
  solve_moments_kernel<<<1, 32, 0, s>>>(model, dv, moments, keep_centred, out_dev);
}

__global__ void lm_init_kernel(const double* __restrict__ alg_out, double* __restrict__ st) {
  if (threadIdx.x != 0) return;
  for (int i = 0; i < LM_SIZE; i++) st[i] = 0.0;
  const int np = (int)alg_out[0];
  if (np == 0) { st[LM_STATUS] = 2.0; return; }
  for (int j = 0; j < np && j < kLmMaxP; j++) st[LM_X + j] = alg_out[1 + j];   // cross-wire: the first 11 of its 20 parameters
}
__global__ void lm_update_kernel(int model, const double* __restrict__ m, double* __restrict__ st) {
  if (threadIdx.x != 0) return;
  lm_update_model(model, m, st);
}
// .cxx:305-327: entries 11..19 rebuilt from the optimised angles and scales
__device__ void us_expand(const double* x, double* prm) {
  for (int j = 0; j < 11; j++) prm[j] = x[j];
  const double cz = cos(x[6]), sz = sin(x[6]), cy = cos(x[7]), sy = sin(x[7]), cx = cos(x[8]), sx = sin(x[8]);
  prm[11] = x[9] * cz * cy; prm[12] = x[9] * sz * cy; prm[13] = -x[9] * sy;
  prm[14] = x[10] * (cz * sy * sx - sz * cx); prm[15] = x[10] * (sz * sy * sx + cz * cx); prm[16] = x[10] * cy * sx;
  prm[17] = cz * sy * cx + sz * sx; prm[18] = sz * sy * cx - cz * sx; prm[19] = cy * cx;
}
__global__ void lm_finish_kernel(int model, DataView dv, const double* __restrict__ st, double* __restrict__ out) {
  if (threadIdx.x != 0) return;
  if (st[LM_STATUS] != 1.0) { out[0] = 0.0; return; }
  if (model == USXW) {
    double x[11];
    for (int j = 0; j < 11; j++) x[j] = st[LM_X + j];
    for (int j = 0; j < 3; j++) x[j] += dv.center[9 + j];   // t1 was estimated relative to the centre of the t2 components
    out[0] = 20;
    us_expand(x, out + 1);
    return;
  }
  if (model == USCP) {   // .cxx:958-983: entries 8..16 rebuilt from the optimised angles and scales
    double x[11], full[20];
    x[0] = x[1] = x[2] = 0.0;
    for (int j = 0; j < 8; j++) x[3 + j] = st[LM_X + j];
    us_expand(x, full);
    out[0] = 17;
    for (int j = 0; j < 17; j++) out[1 + j] = full[3 + j];
    return;
  }
  const int dim = model_dim(model);
  out[0] = dim + 1;
  for (int j = 0; j < dim; j++) out[1 + j] = st[LM_X + j] + dv.center[j];
  out[1 + dim] = st[LM_X + dim];
}
void launch_lm_init(const double* alg_out_dev, double* state, cudaStream_t s) { lm_init_kernel<<<1, 32, 0, s>>>(alg_out_dev, state); }
void launch_lm_update(int model, const double* moments, double* state, cudaStream_t s) { lm_update_kernel<<<1, 32, 0, s>>>(model, moments, state); }
void launch_lm_finish(int model, const DataView& dv, const double* state, double* out_dev, cudaStream_t s) { lm_finish_kernel<<<1, 32, 0, s>>>(model, dv, state, out_dev); }
int lm_status_offset() { return LM_STATUS; }

// ---------------------------------------------------------------------------------------
__global__ void expand_mask_kernel(const uint32_t* __restrict__ bits, uint32_t first, uint32_t count, uint8_t* __restrict__ bytes) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < count) { const uint32_t i = first + t; bytes[i] = (bits[i >> 5] >> (i & 31)) & 1u; }
}
void launch_expand_mask(const uint32_t* bits, uint32_t first, uint32_t count, uint8_t* bytes, cudaStream_t s) {
  if (count) expand_mask_kernel<<<(count + 255) / 256, 256, 0, s>>>(bits, first, count, bytes);
}


}  // namespace lsqr
