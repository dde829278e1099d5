// Internal interface between the host-side engine (engine.cu) and the kernel translation units.
#pragma once
#include <cstddef>
#include <cstdint>
#include <map>
#include <mutex>
#include <utility>
#include <cuda_runtime.h>

#include "../../include/lsqr_b200.h"
#include "models.cuh"

namespace lsqr {

constexpr int kTilePad = 2048;   // leading dimension of the SoA point arrays is a multiple of this: the largest tile any kernel fetches with one bulk copy per row
                                 // (mask_moments_kernel: 2048 data; with 1024 the last tile of the last row read past the allocation -- found by memcheck)
constexpr int kMaxDim = 20;           // doubles per datum, upper bound (calibrated-pointer US calibration: 17)
constexpr int kLmStateDoubles = 256;  // device scratch reserved for the Levenberg-Marquardt controller state
constexpr int kMaxMoments = 96;  // upper bound on the doubles accumulated per thread by the refine reductions (cross-wire US calibration: 91)

constexpr uint32_t kCenterSample = 16384;   // the shift c is the mean of the first min(n, kCenterSample) records

// Device-resident description of the uploaded data.
struct DataView {
  const double* soa64;  // [D][ld], padded with NaN
  const float* soa32;   // [D][ld], centred (soa64 - center), padded with NaN
  size_t ld;            // leading dimension (stride between components)
  size_t span;          // columns the consensus kernels walk: ld for the whole data set, fewer for a range view (multiple of 1024)
  uint32_t n;           // valid data inside the view
  const double* center; // device, kMaxDim doubles: per-component shift used for soa32 and for the refine moments
};

// What the host reads back after a scoring request: one small record, one copy.
struct WinnerRecord {
  unsigned long long key;      // (count << 32) | (0xFFFFFFFF - index relative to the request's first hypothesis)
  unsigned long long n_valid;
  int32_t subset[LSQR_MAX_SUBSET];
  double params[LSQR_MAX_PARAMS];
};

// ---- launch set-up shared by the kernel translation units -------------------------------
// Point chunks (grid.y) of the tiled consensus kernels: enough (hypothesis block x chunk) work items for ~16 CTAs per SM,
// chunks of at least 4 tiles, at most 65535 chunks, none of them empty.
struct TileChunks { uint32_t chunks, tiles_per_chunk; };
inline TileChunks plan_tile_chunks(uint32_t tiles_total, uint32_t hyp_blocks, int num_sms) {
  uint32_t want = (uint32_t)num_sms * 16;
  uint32_t chunks = (want + hyp_blocks - 1) / hyp_blocks;
  uint32_t max_chunks = (tiles_total + 3) / 4;
  if (max_chunks == 0) max_chunks = 1;
  if (chunks > max_chunks) chunks = max_chunks;
  if (chunks > 65535) chunks = 65535;
  if (chunks == 0) chunks = 1;
  const uint32_t tiles_per_chunk = (tiles_total + chunks - 1) / chunks;
  chunks = (tiles_total + tiles_per_chunk - 1) / tiles_per_chunk;
  return {chunks, tiles_per_chunk};
}

// Per-device tables of the launchers (constant-bank lock, occupancy) hold this many devices; device ids alias beyond it.
constexpr int kMaxDevices = 64;

// Lets `kernel` launch with up to `bytes` of dynamic shared memory on the current device (more than 48 KB needs the limit
// raised).  The limit belongs to one kernel on one device, so the table is keyed by both: instantiations with the same
// signature are different kernels, and a multi-device context launches from one thread per device.
inline void allow_dynamic_smem(const void* kernel, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> raised;
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lock(mu);
  size_t& limit = raised[{kernel, dev}];
  if (bytes <= limit) return;
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess) limit = bytes;
}
template <class Kernel> void allow_dynamic_smem(Kernel* kernel, size_t bytes) { allow_dynamic_smem(reinterpret_cast<const void*>(kernel), bytes); }

// ---- k_score.cu -------------------------------------------------------------------------
// c = mean of the first `count` AoS records (device buffer), per centred component -> center_dev[kMaxDim].
void launch_center_sample(int model, const unsigned char* aos_dev, size_t stride, uint32_t count, double* center_dev, cudaStream_t s);
// AoS records [first, first + count) (stride bytes, D leading doubles each) -> SoA fp64 and SoA fp32 of x - c; columns up to
// pad_to are NaN-filled.
void launch_ingest(int model, const unsigned char* aos_dev, size_t stride, uint32_t first, uint32_t count, uint32_t pad_to, const double* center_dev,
                   double* soa64, float* soa32, size_t ld, cudaStream_t s);

struct SolveArgs {
  int model, sampler;
  uint64_t seed, first;   // global index of hypothesis 0 of this launch
  uint32_t H;             // hypotheses in this launch
  size_t hld;             // leading dimension of the hypothesis arrays
  const int32_t* list;    // LSQR_SAMPLE_LIST: [H][K] on device
  const unsigned char* gathered;  // optional, with `list`: the K records of every subset, AoS [H][K] records of gathered_stride bytes
  size_t gathered_stride; //   (compute(): the minimal subsets are fetched ahead of the bulk upload)
  const double* params_in;// LSQR_SAMPLE_PARAMS: [H][P] on device
  int32_t* subsets;       // out [K][hld]
  double* hyp64;          // out [P][hld]
  uint32_t* n_valid;      // out (atomic)
};
void launch_solve(const SolveArgs& a, const DataView& dv, const EstCfg& cfg, cudaStream_t s);
// key (after arg-max / all-reduce) -> winner's subset and parameters, on the device; a.first = first hypothesis of the REQUEST,
// a.list / a.params_in = the request's device-resident list (samplers 2, 3)
void launch_winner(const SolveArgs& a, const unsigned long long* key_dev, const DataView& dv, const EstCfg& cfg, WinnerRecord* out, cudaStream_t s);
void launch_hoist32(int model, const double* hyp64, size_t hld, uint32_t H, const DataView& dv, const EstCfg& cfg, float* hyp32, cudaStream_t s);

// Early exit of the fp32 constant-bank scoring (k_fast.cu), for requests that want the winner only.  A hypothesis with c
// inliers among the first p data ends with at most c + (n - p); once that is below the full count L of some hypothesis it
// can neither beat nor tie the winner, so it stops being scored and keeps its partial count (< L) in counts[].  The winner,
// its count and the arg-max key are exactly those of the full pass.  Buffers come from ensure_hyp (engine.cu), [hld] each.
struct Prune {
  float* hyp32[2];                // [16][hld] each: the compacted live list's hoisted constants (may alias the request's)
  uint32_t* live_counts[2];       // running counts of the live list
  uint32_t* live_ids[2];          // the live hypotheses' indices in the launch
  uint32_t* dev;                  // scratch: [0, 16) seed hypothesis constants, [16, 18) seed key, [18] L, [19] live count,
                                  // [20, 20 + hld / 1024 + 1) per-block survivor tallies
  uint32_t* host;                 // pinned, 4 words
  const unsigned long long* floor_key;   // arg-max key of the request's earlier batches: its count is a valid L as well
  uint64_t evals;                 // out: hypothesis x datum evaluations launched (real data only), the seed included; left as
                                  // the caller set it (H n) when the request takes the full pass
};
constexpr size_t prune_dev_words(size_t hld) { return 20 + hld / 1024 + 1; }

// counts[h] (+)= |{m : agree(h, datum m)}|.  counts must be zeroed by the caller.  Returns #launches.  With `prune`, fp32
// requests that take the constant-bank kernel exit early (see Prune); the others ignore it.
int launch_consensus(int model, int precision, const DataView& dv, const double* hyp64, const float* hyp32, size_t hld, uint32_t H,
                     const EstCfg& cfg, uint32_t* counts, int num_sms, cudaStream_t s, Prune* prune = nullptr);
// fp32 fast mode (k_fast.cu)
int launch_consensus32(int model, const DataView& dv, const float* hyp32, size_t hld, uint32_t H, const EstCfg& cfg, uint32_t* counts, int num_sms,
                       cudaStream_t s, Prune* prune = nullptr);
// key = max over h of (counts[h] << 32) | (0xFFFFFFFF - (index_base + h)); key must be zeroed first.
void launch_argmax(const uint32_t* counts, uint32_t H, uint32_t index_base, unsigned long long* key, cudaStream_t s);

// ---- k_refine.cu ------------------------------------------------------------------------
struct RefineBuffers {
  uint32_t* maskbits;   // [ld/32]
  uint8_t* maskbytes;   // optional [n]: mask mode 1 also writes one byte per datum (std::vector<bool> order)
  double* partials;     // [blocks][kMaxMoments]
  double* moments;      // [kMaxMoments] reduced (device)
  int blocks;
};
// Fused streaming pass over data [begin,end) (begin a multiple of 32).
// mask_mode 0: every datum counts; 1: evaluate agree(params_dev, datum) in fp64 reference
// arithmetic and write the consensus bits; 2: read the stored bits.  Accumulates the model's
// least-squares moments over the selected data into rb.partials.  lm_state != nullptr selects the
// Levenberg-Marquardt moments (J^T J, J^T r, cost) at the point the controller state asks for.
void launch_mask_moments(int model, const DataView& dv, uint32_t begin, uint32_t end, const double* params_dev, int mask_mode,
                         const double* lm_state, const EstCfg& cfg, const RefineBuffers& rb, cudaStream_t s);
// Sums the per-block partials in a fixed order -> rb.moments.
void launch_reduce_partials(const RefineBuffers& rb, int n_moments, cudaStream_t s);
// moments -> parameters (small eigen / pseudo-inverse solves).  out_dev: [0] = n_params, [1..] params.
void launch_solve_moments(int model, const DataView& dv, const double* moments, int keep_centred, double* out_dev, cudaStream_t s);
// Levenberg-Marquardt controller for the circle / sphere geometric fit (state layout in k_refine.cu).
void launch_lm_init(const double* alg_out_dev, double* state, cudaStream_t s);
void launch_lm_update(int model, const double* moments, double* state, cudaStream_t s);
void launch_lm_finish(int model, const DataView& dv, const double* state, double* out_dev, cudaStream_t s);
// Weighted Horn (AbsoluteOrientationParametersEstimator.cxx:208-297): weighted moments of all n pairs, then the 4x4 eigen solve.
void launch_weighted_absor_moments(const DataView& dv, const double* weights_dev, const RefineBuffers& rb, cudaStream_t s);
void launch_solve_weighted_absor(const DataView& dv, const double* moments, double* out_dev, cudaStream_t s);
int moments_count(int model, bool lm);
int lm_status_offset();   // index of the status word (0 run, 1 converged, 2 failed) in the LM state
int mask_moments_ctas_per_sm();   // grid of launch_mask_moments = this x SMs (one wave)
// bytes[i] = bit i of the consensus set, for i in [first, first + count)
void launch_expand_mask(const uint32_t* bits, uint32_t first, uint32_t count, uint8_t* bytes, cudaStream_t s);

struct BatchArgs {
  int model, exhaustive;
  int precision;             // randomized mode: 0 = fp64 scoring, 1 = fp32 scoring (exhaustive mode is always fp64)
  uint32_t tries;            // cap on hypotheses per problem (randomized mode)
  double prob;               // desiredProbabilityForNoOutliers for the stop rule; <= 0 disables it
  uint64_t seed;
  const double* data;        // packed [total][D] on device
  const uint64_t* offsets;   // [n_problems+1] on device, absolute record offsets (data[0] is record `base`)
  uint64_t base;             // record offset of the first problem of this launch
  uint64_t first_problem;    // global index of the first problem of this launch (the Philox counter of a problem is global)
  uint32_t n_problems;
  uint32_t max_n;            // largest problem (sizes shared memory)
  double* out_params;        // [n_problems][P]
  uint32_t* out_counts;      // [n_problems]
  uint8_t* out_masks;        // [total] or null
};
int launch_batch(const BatchArgs& a, const EstCfg& cfg, int ls_type, cudaStream_t s);
// Problem sizes, in records, of one lsqr_ransac_batch call on the current device.  A problem of up to one_block records takes
// batch_kernel; a larger one takes batch_cluster_kernel on a cluster of C CTAs of `slice` records each (C = 2, 4, .., max_cluster),
// up to max_records.  Exhaustive mode, and a model without the cluster kernel, stop at one_block (max_cluster = 0).
struct BatchLimits { uint64_t one_block, max_records; uint32_t slice; int max_cluster; };
BatchLimits batch_limits(int model, int precision, int exhaustive);
// the smallest cluster whose slices hold n records (0: none)
inline uint32_t batch_cluster_size(const BatchLimits& L, uint64_t n) {
  for (uint32_t c = 2; c <= (uint32_t)L.max_cluster; c *= 2)
    if ((((n + c - 1) / c + 1) & ~1ull) <= L.slice) return c;
  return 0;
}
// The problems a.offsets[problems[i]] (count of them, all of one cluster size) on clusters of `cluster` CTAs whose dynamic
// shared memory holds `slice` records (the largest slice among them).
int launch_batch_cluster(const BatchArgs& a, const uint32_t* problems, uint32_t count, uint32_t cluster, uint32_t slice, const EstCfg& cfg,
                         int ls_type, cudaStream_t s);

// Batched least squares (lsqr_least_squares_batch_device): problem b's records are data[offsets[b] .. offsets[b + 1]) (records of
// D doubles), selected by masks (one byte per record, non-zero = used) when given; weights (one double per record) select the
// weighted Horn fit of the absolute orientation.
struct LsBatchArgs {
  int model;
  const double* data;        // packed records on device, indexed by absolute record offset
  const uint64_t* offsets;   // [n_problems + 1] on device
  const uint8_t* masks;      // optional, indexed like the records
  const double* weights;     // optional (ABSOR only), indexed like the records
  double* out_params;        // [n_problems][P]
};
// A problem of n records takes a cluster of C CTAs (1, 2, 4, .., cmax): the smallest whose CTAs get at most kLsSliceRecords each.
// It depends on n and the device alone, so a problem's result does not depend on the rest of the call.
constexpr uint64_t kLsSliceRecords = 16384;
inline uint32_t ls_batch_cluster(uint64_t n, int cmax) {
  uint32_t c = 1;
  while (c < (uint32_t)cmax && (n + c - 1) / c > kLsSliceRecords) c *= 2;
  return c;
}
// the largest cluster of the model's kernel (weighted: the weighted Horn kernel) the current device schedules: 8 or 16; 0 = no kernel
int ls_batch_max_cluster(int model, bool weighted);
// the problems a.offsets[problems[i]], i < count, each on a cluster of `cluster` CTAs
int launch_ls_batch(const LsBatchArgs& a, const uint32_t* problems, uint32_t count, uint32_t cluster, int ls_type, cudaStream_t s);

// ---- k_score.cu (single-call helpers) ---------------------------------------------------
void launch_estimate_one(int model, const double* packed_dev, const EstCfg& cfg, double* out_dev /* [0]=n_params, [1..P] */, cudaStream_t s);
void launch_agree_many(int model, const double* params_dev, const double* packed_dev, uint32_t n, const EstCfg& cfg, uint8_t* out, cudaStream_t s);

// ---- k_bench.cu -------------------------------------------------------------------------
void launch_fma_bench(int kind, int iters, int blocks, int threads, float* sink, cudaStream_t s);

}  // namespace lsqr
