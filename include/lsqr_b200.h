/* lsqr_b200.h -- C ABI of the B200-native RANSAC / least-squares engine.
 *
 * This is the drop-in boundary for ONE path of zivy/LSQRRecipes: the RANSAC driver
 * (parametersEstimators/RANSAC.h:75-79 randomized compute, :111-113 exhaustive compute,
 * bodies RANSAC.hxx:4-249) together with the estimate / agree / leastSquaresEstimate
 * bodies of the estimators it calls through ParametersEstimator<T,S>
 * (parametersEstimators/ParametersEstimator.h:41-61).  The re-authored C++ headers in
 * include/lsqrRecipes/ keep the reference's class names and signatures and forward here;
 * INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Plain pointers and sizes only; no C++ or torch types.  All entry points return 0 on
 * success or a negative lsqr_status; lsqr_last_error() gives the text.  Nothing throws
 * across this boundary.  One context per host thread; calls are synchronous at return.
 * There is NO CPU fallback: without a CUDA device every call fails with LSQR_ERR_CUDA.
 *
 * Data layouts are the reference's host layouts (SURVEY.md 8a-11): a datum is `dim` doubles
 * at the start of each `stride`-byte record:
 *   Point<double,n>   n doubles                 (common/Point.h:127)       stride 8n
 *   pair<Point3D,Point3D>  first[3], second[3]  (std::pair)                stride 48
 *   Ray3D             p[3], n[3]                (common/Ray3D.h:23-24)     stride 48
 *   Frame             rotation[3][3], translation[3] (common/Frame.h:30-31) stride 104
 */
#ifndef LSQR_B200_H
#define LSQR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lsqr_ctx lsqr_ctx;

/* Estimator behind the context.  Replaces the virtual dispatch of
 * ParametersEstimator<T,S> (ParametersEstimator.h:26-64) for the listed classes. */
typedef enum lsqr_model {
  LSQR_PLANE3 = 0,  /* PlaneParametersEstimator<3>            PlaneParametersEstimator.hxx:36-203 */
  LSQR_LINE2D = 1,  /* Line2DParametersEstimator              Line2DParametersEstimator.cxx:11-123 */
  LSQR_LINE2 = 2,   /* LineParametersEstimator<2>             LineParametersEstimator.hxx:23-150 */
  LSQR_LINE3 = 3,   /* LineParametersEstimator<3> */
  LSQR_CIRCLE2 = 4, /* SphereParametersEstimator<2>           SphereParametersEstimator.hxx:80-109,255-338 */
  LSQR_SPHERE3 = 5, /* SphereParametersEstimator<3>           SphereParametersEstimator.hxx:115-163,255-338 */
  LSQR_ABSOR = 6,   /* AbsoluteOrientationParametersEstimator AbsoluteOrientationParametersEstimator.cxx:14-327 */
  LSQR_RAY = 7,     /* RayIntersectionParametersEstimator     RayIntersectionParametersEstimator.cxx:23-179 */
  LSQR_PIVOT = 8,   /* PivotCalibrationEstimator              PivotCalibrationParametersEstimator.cxx:9-123 */
  LSQR_DENSE5 = 9,  /* DenseLinearEquationSystemParametersEstimator<double,5>   DenseLinearEquationSystemParametersEstimator.hxx:17-119 */
  LSQR_DENSE6 = 10, /* DenseLinearEquationSystemParametersEstimator<double,6>   (datum = AugmentedRow: n coefficients, right-hand side) */
  LSQR_USXW = 11,   /* SingleUnknownPointTargetUSCalibrationParametersEstimator (cross-wire phantom)   SinglePointTargetUSCalibrationParametersEstimator.cxx:10-329
                     * datum = 14 doubles [R2 row-major, t2, u, v]; ls_type 0 = ANALYTIC, 1 = ITERATIVE (Levenberg-Marquardt) */
  LSQR_USCP = 12,   /* CalibratedPointerTargetUSCalibrationParametersEstimator   SinglePointTargetUSCalibrationParametersEstimator.cxx:663-985
                     * datum = 17 doubles [R2 row-major, t2, u, v, p]; ls_type as for LSQR_USXW */
  LSQR_SPHERE4 = 13, /* SphereParametersEstimator<4>: the generic-dimension minimal solver (pseudo-inverse, rank test)   SphereParametersEstimator.hxx:169-202 */
  LSQR_PLANE4 = 14,  /* PlaneParametersEstimator<4>: the generic-dimension minimal solver (null space of [p_i, -1])   PlaneParametersEstimator.hxx:70-108 */
  /* the rest of the reference's template space (SURVEY.md 8f-4, 8f-2): same code paths, one id per instantiation */
  LSQR_PLANE2 = 15,  /* PlaneParametersEstimator<2> (a 2-D line through the generic null-space branch) */
  LSQR_PLANE5 = 16, LSQR_PLANE6 = 17, LSQR_PLANE7 = 18, LSQR_PLANE8 = 19,       /* PlaneParametersEstimator<5..8> */
  LSQR_SPHERE5 = 20, LSQR_SPHERE6 = 21, LSQR_SPHERE7 = 22, LSQR_SPHERE8 = 23,   /* SphereParametersEstimator<5..8> */
  LSQR_LINE4 = 24, LSQR_LINE5 = 25, LSQR_LINE6 = 26, LSQR_LINE7 = 27, LSQR_LINE8 = 28,   /* LineParametersEstimator<4..8> */
  LSQR_DENSE2 = 29, LSQR_DENSE3 = 30, LSQR_DENSE4 = 31, LSQR_DENSE7 = 32, LSQR_DENSE8 = 33,   /* DenseLinearEquationSystemParametersEstimator<double, 2..4, 7, 8> */
  LSQR_NUM_MODELS = 34
} lsqr_model;

typedef enum lsqr_status {
  LSQR_OK = 0,
  LSQR_ERR_ARG = -1,     /* bad argument / unsupported combination */
  LSQR_ERR_CUDA = -2,    /* CUDA runtime failure (including: no device) */
  LSQR_ERR_STATE = -3,   /* call out of order (e.g. score before upload) */
  LSQR_ERR_COMM = -4     /* collective hook failed */
} lsqr_status;

typedef enum lsqr_precision {
  LSQR_FP64 = 0, /* validation mode: the reference's operation order, no FMA contraction; bit-exact counts */
  LSQR_FP32 = 1  /* fast mode: hoisted constants, fused multiply-add.  Decisions differ from LSQR_FP64 only for data within the fp32
                  * rounding band of the threshold.  The kD-line estimators are scored through the perpendicular (d = 2) / the Pluecker
                  * moment (d = 3) of the direction, which is taken as the unit vector estimate() returns (it is re-normalised; imported
                  * parameter vectors with a non-unit direction are scored as their normalised line, where LSQR_FP64 evaluates the
                  * reference's expression literally, LineParametersEstimator.hxx:135-150). */
} lsqr_precision;

typedef enum lsqr_sampler {
  LSQR_SAMPLE_PHILOX = 0,     /* on-device Philox4x32-10, counter = global hypothesis index (replaces RANSAC.hxx:44-79) */
  LSQR_SAMPLE_EXHAUSTIVE = 1, /* lexicographic unranking, the order of RANSAC.hxx:197-213 */
  LSQR_SAMPLE_LIST = 2,       /* caller-supplied ordered subsets, int32 [H][k] */
  LSQR_SAMPLE_PARAMS = 3      /* caller-supplied hypothesis parameters, double [H][P] (agree() only) */
} lsqr_sampler;

/* SphereParametersEstimator::LeastSquaresType (SphereParametersEstimator.h:43) */
typedef enum lsqr_ls_type { LSQR_LS_ALGEBRAIC = 0, LSQR_LS_GEOMETRIC = 1 } lsqr_ls_type;

#define LSQR_MAX_PARAMS 20
#define LSQR_MAX_SUBSET 10

/* ---- model table ------------------------------------------------------------------ */
/* dim = doubles per datum, nparams = length of the parameter vector, k = numForEstimate()
 * (ParametersEstimator.h:61). */
int lsqr_model_info(int model, int* dim, int* nparams, int* k);

/* Model id of a dimension-templated estimator of the reference, or -1 when the engine does not instantiate that dimension:
 * PlaneParametersEstimator<d> (PlaneParametersEstimator.h:24), SphereParametersEstimator<d> (SphereParametersEstimator.h:24) and
 * LineParametersEstimator<d> (LineParametersEstimator.h:35) for d = 2..8, DenseLinearEquationSystemParametersEstimator<double, n>
 * (DenseLinearEquationSystemParametersEstimator.h:149) for n = 2..8.  What a binding of those class templates calls once,
 * in the constructor, in the place of the reference's compile-time `dimension`. */
int lsqr_model_plane(unsigned dimension);
int lsqr_model_sphere(unsigned dimension);
int lsqr_model_line(unsigned dimension);
int lsqr_model_dense(unsigned n);

/* ---- context ---------------------------------------------------------------------- */
int lsqr_ctx_create(lsqr_ctx** out, int device);
/* Number of CUDA devices visible to the process (0 when there is none). */
int lsqr_device_count(void);
/* One context spanning `ngpus` devices of this process (ngpus <= 0: every visible device) -- SURVEY.md 8b's ctx_create(ngpus).
 * The data are replicated on every GPU, the hypotheses of every request are partitioned by global index, the consensus set
 * and the refine are sharded by point range; the exchange steps are native NCCL calls inside the library (one
 * ncclAllReduce(max) on the packed 64-bit key per request, one ncclAllReduce(sum) of <= 91 doubles per refine pass, and the
 * all-gather that replicates the uploaded points over NVLink).  Every entry point below accepts such a context and returns
 * what a single-GPU context returns (lsqr_upload_device, lsqr_set_shard, lsqr_ctx_set_stream and lsqr_ctx_init_nccl excepted:
 * LSQR_ERR_ARG).  The estimator's own methods (estimate / agree / least squares) run on the first device. */
int lsqr_ctx_create_multi(lsqr_ctx** out, int ngpus);
/* Number of GPUs / ranks behind the context (1 for lsqr_ctx_create). */
int lsqr_ctx_world(const lsqr_ctx* ctx);
/* One process per GPU (torchrun, MPI): rank 0 calls lsqr_nccl_unique_id, the launcher broadcasts the 128 bytes, every rank
 * calls lsqr_ctx_init_nccl on its own single-device context.  From then on the context is rank `rank` of `world` and performs
 * its collectives itself with ncclAllReduce / ncclAllGather on its stream; lsqr_upload fetches every world-th chunk of the
 * host buffer (the same buffer content on every rank) and all-gathers the rest. */
int lsqr_nccl_unique_id(void* out_id, size_t bytes /* >= 128 */);
int lsqr_ctx_init_nccl(lsqr_ctx* ctx, const void* id, size_t bytes, int rank, int world);
void lsqr_ctx_destroy(lsqr_ctx* ctx);
const char* lsqr_last_error(const lsqr_ctx* ctx);
/* Run every kernel of this context on an existing CUDA stream (cudaStream_t passed as void*). */
int lsqr_ctx_set_stream(lsqr_ctx* ctx, void* cuda_stream);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t lsqr_kernel_launches(const lsqr_ctx* ctx);

/* Estimator configuration: the constructor arguments of the reference classes
 * (delta: e.g. PlaneParametersEstimator.h:31; aux: RayIntersectionParametersEstimator.h:34-35
 * minimalAngularDeviation, <=0 selects the reference default of 1 degree;
 * ls_type: SphereParametersEstimator.h:37). */
int lsqr_set_estimator(lsqr_ctx* ctx, int model, double delta, double aux, int ls_type);

/* Copy n data records (host memory, reference AoS layout, see top) to the device and build
 * the SoA fp64 / fp32 working layouts.  Replaces the `std::vector<T>& data` argument of
 * RANSAC::compute (RANSAC.h:77).  The input is not retained. */
int lsqr_upload(lsqr_ctx* ctx, const void* aos, size_t n, size_t stride_bytes);
/* Same, for a buffer that already lives in device memory (packed doubles, dim per record). */
int lsqr_upload_device(lsqr_ctx* ctx, const double* dev_packed, size_t n);

/* Multi-GPU sharding with caller-supplied collectives (for launchers that own the communicator; lsqr_ctx_create_multi and
 * lsqr_ctx_init_nccl are the native alternatives): this context scores hypotheses [rank*H/world, (rank+1)*H/world) of every
 * request and refines the points [rank*N/world, (rank+1)*N/world) (boundaries on 32-datum words).  The two exchange steps go
 * through the hooks, which operate IN PLACE on device memory and must be stream-ordered on `cuda_stream`.
 * Counts, fractions and refined parameters are global.  Of the consensus set a rank writes ITS point shard only
 * (lsqr_get_mask, lsqr_get_mask_bits, the mask of lsqr_ransac): bytes outside [begin, end) of the caller's buffer are left
 * untouched; lsqrrecipes_b200/dist.py (full_mask) assembles the ranks' parts.  A multi-GPU group writes all parts itself. */
typedef int (*lsqr_allreduce_max_u64_fn)(void* user, uint64_t* dev_key, void* cuda_stream);
typedef int (*lsqr_allreduce_sum_f64_fn)(void* user, double* dev_vals, int count, void* cuda_stream);
int lsqr_set_shard(lsqr_ctx* ctx, int rank, int world, lsqr_allreduce_max_u64_fn max_fn,
                   lsqr_allreduce_sum_f64_fn sum_fn, void* user);

/* ---- scoring: minimal solve + consensus for a batch of hypotheses ------------------- */
typedef struct lsqr_score_args {
  int sampler;           /* lsqr_sampler */
  int precision;         /* lsqr_precision */
  uint64_t seed;         /* Philox key */
  uint64_t first;        /* global index of the first hypothesis (Philox counter / lexicographic rank) */
  uint64_t count;        /* H: number of hypotheses in this request (global, before sharding) */
  const int32_t* subsets;/* LSQR_SAMPLE_LIST: host int32 [H][k] */
  const double* params;  /* LSQR_SAMPLE_PARAMS: host double [H][P]; NaN row = degenerate */
  uint32_t* out_counts;  /* optional host [H]: full inlier count per hypothesis (no early exit, RANSAC.hxx:239-244).  Without it,
                            fp32 requests of at least 98304 hypotheses exit early (RANSAC.hxx:94): a hypothesis stops being
                            scored once its inliers so far plus the data left cannot reach the full count of one already
                            scored; the result is exactly that of the full pass, with less work on data with many inliers */
  double* out_params;    /* optional host [H][P]: estimate() output per hypothesis, NaN row if degenerate */
} lsqr_score_args;

typedef struct lsqr_score_result {
  uint64_t best_index;   /* global index of the winner; ties -> lowest index (strict '>' of RANSAC.hxx:100,245) */
  uint32_t best_count;   /* its inlier count; 0 = no valid hypothesis */
  uint32_t n_valid;      /* hypotheses whose minimal subset was not degenerate (this rank) */
  int32_t best_subset[LSQR_MAX_SUBSET];
  double best_params[LSQR_MAX_PARAMS];
  double score_ms;       /* device time of solve + consensus + arg-max (CUDA events) */
  double consensus_ms;   /* device time of the consensus kernel(s) alone */
  uint64_t evals;        /* hypothesis x datum evaluations launched (this rank; H x N without the early exit) */
} lsqr_score_result;

/* Scores `count` hypotheses against the uploaded data and returns the winner (most inliers, lowest index on ties).  The
 * winner is the same with and without out_counts; only the per-hypothesis counts need the full pass. */
int lsqr_score(lsqr_ctx* ctx, const lsqr_score_args* args, lsqr_score_result* res);

/* ---- consensus set + least-squares refine ------------------------------------------ */
/* agree() of `params` against every uploaded datum in fp64 reference arithmetic
 * (e.g. PlaneParametersEstimator.hxx:196-203): stores the consensus set on the device,
 * returns its size.  Replaces RANSAC.hxx:129-137. */
int lsqr_consensus(lsqr_ctx* ctx, const double* params, uint32_t* out_count);
/* Copy the stored consensus set to the host, one byte per datum (std::vector<bool> order).  A page-locked
 * destination (cudaHostAlloc / cudaHostRegister) receives the DMA directly; any other is filled through the
 * library's own staging buffer. */
int lsqr_get_mask(lsqr_ctx* ctx, uint8_t* out_bytes);
/* The same set as packed bits: datum i is bit (i & 31) of word i >> 5 (ceil(n / 32) words).  1/8 of the bytes of
 * lsqr_get_mask; include/lsqrRecipes/RANSAC.h fills std::vector<bool> from it. */
int lsqr_get_mask_bits(lsqr_ctx* ctx, uint32_t* out_words);
/* leastSquaresEstimate() over the stored consensus set (RANSAC.hxx:138), or over all data
 * when use_mask == 0.  *n_params = 0 means the reference's "empty parameters" (degenerate). */
int lsqr_refine(lsqr_ctx* ctx, int use_mask, double* out_params, int* n_params);

/* ---- whole calls -------------------------------------------------------------------- */
typedef struct lsqr_compute_result {
  double params[LSQR_MAX_PARAMS];
  int n_params;          /* 0 = empty parameter vector (reference error convention, RANSAC.h:53-63) */
  double fraction;       /* return value of RANSAC::compute: |consensus set| / N */
  uint32_t best_count;
  uint64_t best_index;
  uint64_t tries;        /* hypotheses actually scored */
  double device_ms;      /* sum of device time over all kernels of the call */
} lsqr_compute_result;

/* RANSAC<T,S>::compute(parameters, estimator, data, desiredProbabilityForNoOutliers,
 * consensusSet) -- RANSAC.h:75-79 / RANSAC.hxx:4-145.  Rounds of 256, 1024, 4096 ... Philox-sampled
 * hypotheses; the stop rule of RANSAC.hxx:107-110 is re-evaluated between rounds, so at least as many
 * hypotheses are scored as the reference's loop would try.  Invalid input
 * (N < k, prob outside (0,1)) returns LSQR_OK with fraction = 0, n_params = 0. */
int lsqr_ransac(lsqr_ctx* ctx, double prob, int precision, uint64_t seed, uint8_t* out_mask_bytes,
                lsqr_compute_result* res);
/* The same call with the data still in host memory -- what RANSAC<T,S>::compute receives: lsqr_upload + lsqr_ransac in one
 * pass with identical results (same hypotheses, counts, consensus set and parameters).  The minimal subsets of the first
 * round are drawn on the host with the device's sampler and their records fetched first, so that every chunk of the data is
 * scored against the first 256 hypotheses while the chunks behind it are still crossing PCIe (and, on a multi-GPU context,
 * NVLink).  Invalid input (n < k, prob outside (0,1)) returns LSQR_OK with fraction = 0, n_params = 0 and uploads nothing. */
int lsqr_compute(lsqr_ctx* ctx, const void* aos, size_t n, size_t stride_bytes, double prob, int precision, uint64_t seed,
                 uint8_t* out_mask_bytes, lsqr_compute_result* res);
/* The brute-force overload, RANSAC.h:111-113 / RANSAC.hxx:150-249: all C(N,k) subsets in
 * lexicographic order, first maximum wins. */
int lsqr_ransac_exhaustive(lsqr_ctx* ctx, int precision, uint8_t* out_mask_bytes, lsqr_compute_result* res);

/* Many independent problems (a host loop of RANSAC::compute calls in the reference).  data: host packed doubles, problems
 * back to back; `offsets` [n_problems+1] in records.  exhaustive != 0 enumerates all C(n,k) subsets
 * of each problem (RANSAC.hxx:150-249); otherwise rounds of Philox hypotheses with the stop
 * rule of RANSAC.hxx:107-110 for `prob` (prob <= 0: exactly max_tries hypotheses), capped at
 * max_tries, scored in `precision` (LSQR_FP32: the fast forms on an fp32 copy of the points relative to the problem's
 * first point; exhaustive mode always scores in fp64).  Minimal solves, the winner's consensus set, its count and the
 * refine are fp64 in every mode.  Outputs per problem: params [n_problems][P] (NaN row = empty), counts
 * [n_problems], optional masks (bytes, same indexing as data).
 * A problem of up to `one_block` records (lsqr_batch_capacity) is solved by one thread block with its points in shared
 * memory.  A larger one, in randomized mode, by a thread-block cluster of 2 to 16 blocks that split its points between their
 * shared memories (the smallest cluster that holds it), up to `max_records`; its result depends only on the problem, its
 * index, the seed, prob and max_tries.  Exhaustive mode keeps the one-block limit.  A problem above the limit fails the
 * call with LSQR_ERR_ARG. */
int lsqr_ransac_batch(lsqr_ctx* ctx, const double* data, const uint64_t* offsets, uint64_t n_problems,
                      int exhaustive, double prob, uint32_t max_tries, uint64_t seed, int precision,
                      double* out_params, uint32_t* out_counts, uint8_t* out_masks, double* device_ms);
/* The problem sizes lsqr_ransac_batch takes for the context's model on its device (a group context: its first device), in
 * records: *one_block, the largest one thread block holds, and *max_records, the largest the call takes at all (equal to
 * one_block in exhaustive mode).  LSQR_ERR_ARG for a model without batched mode (the ultrasound calibrations). */
int lsqr_batch_capacity(lsqr_ctx* ctx, int precision, int exhaustive, uint64_t* one_block, uint64_t* max_records);

/* ---- the estimator's own methods, for callers that use them directly ---------------- */
/* estimate() on k (or more) data in host memory; *n_params = 0 when degenerate. */
int lsqr_estimate(lsqr_ctx* ctx, const double* packed, size_t n, double* out_params, int* n_params);
/* agree() of one parameter vector against n packed data; out[n] bytes. */
int lsqr_agree(lsqr_ctx* ctx, const double* params, const double* packed, size_t n, uint8_t* out);
/* leastSquaresEstimate() on n packed data in host memory. */
int lsqr_least_squares(lsqr_ctx* ctx, const double* packed, size_t n, double* out_params, int* n_params);
/* AbsoluteOrientationParametersEstimator::weightedLeastSquaresEstimate (AbsoluteOrientationParametersEstimator.cxx:208-297):
 * Horn's method with one weight per pair; LSQR_ABSOR contexts only; *n_params = 0 for fewer than 3 pairs. */
int lsqr_weighted_least_squares(lsqr_ctx* ctx, const double* packed, size_t n, const double* weights, double* out_params, int* n_params);

/* ---- measurement helpers ------------------------------------------------------------ */
/* Register-resident FMA-chain microbenchmarks: returns lane-FMA/s of the fp32 (kind 0),
 * packed fp32x2 (kind 1) or fp64 (kind 2) pipe on the context's device.  Used by bench.py
 * to state the consensus kernel's roofline against a MEASURED pipe peak. */
int lsqr_microbench_fma(lsqr_ctx* ctx, int kind, int iters, double* out_fma_per_s, double* out_ms);
/* The consensus-set + moments pass (mask_moments_kernel) for `params`, `reps` launches back to back between two CUDA events
 * on the context's stream: average duration of a launch and the bytes one launch has to move (8 dim bytes per datum read,
 * 1 bit written).  bench.py's roofline_refine. */
int lsqr_bench_refine_pass(lsqr_ctx* ctx, const double* params, int reps, double* ms_per_pass, double* algorithmic_bytes);
/* Time of the last refine's streaming moment kernel and the bytes it had to read. */
int lsqr_last_refine_stats(const lsqr_ctx* ctx, double* kernel_ms, double* algorithmic_bytes, int* lm_iterations);

#ifdef __cplusplus
}
#endif
#endif /* LSQR_B200_H */
