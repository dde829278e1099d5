// Host side of the C ABI (include/lsqr_b200.h): context, device buffers, and the orchestration
// that replaces RANSAC<T,S>::compute (parametersEstimators/RANSAC.hxx:4-249).  No arithmetic of
// the path happens on the host: sampling, minimal solves, consensus, arg-max, consensus set and
// least squares (including the small eigen / LM controllers) are all kernels.  The host only
// sequences launches, evaluates the scalar stop rule (RANSAC.hxx:107-110) between rounds and
// moves results.  There is no CPU fallback: every entry point fails with LSQR_ERR_CUDA when no
// device is usable.
//
// Data movement of one compute() call:
//   * upload: the caller's AoS records go to the device in chunks on a copy stream (straight from page-locked memory; from
//     pageable memory -- std::vector<T>, the reference's only input type -- through a ring of pinned buffers filled by a few
//     host threads) while the chunks that have landed are transposed to the SoA fp64 / fp32 working layouts on the compute
//     stream.  With several GPUs each one fetches every world-th chunk over its own PCIe link and an NCCL all-gather over
//     NVLink fans the round out, so the host buffer crosses PCIe once in total.
//   * scoring round -> arg-max -> (all-reduce of the 8-byte key) -> winner re-derived on the device -> ONE small copy back
//     (count for the stop rule, subset, parameters);
//   * consensus set + least-squares moments in one streaming pass that also writes the caller's byte mask -> (all-reduce of
//     the moments) -> on-device solve / Levenberg-Marquardt -> ONE copy back of parameters, count and mask.
// Multi-GPU (SURVEY.md 8e): points replicated, hypotheses partitioned by global index, refine sharded by point range.
// Collectives are native NCCL calls on the context's stream (single-process group: lsqr_ctx_create_multi; one process per
// GPU: lsqr_ctx_init_nccl), or caller-supplied hooks (lsqr_set_shard).
#include "../../include/lsqr_b200.h"

#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <functional>
#include <limits>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "engine.h"

using namespace lsqr;

namespace {
constexpr size_t kAgreeZeroCopy = 16;   // lsqr_agree: up to this many data are read by the kernel straight from page-locked host memory
constexpr int kSmall = 1024, kSmIn = 0, kSmOut = 32, kSmLm = 64, kSmEst = 640, kSmSink = 800;   // layout of lsqr_ctx::small_dev

// ---- NCCL, resolved at first use ---------------------------------------------------------------
// The library is loaded with dlopen instead of a DT_NEEDED entry: a Python process that imports torch carries torch's own
// libnccl.so.2 (2.28), the system has another (2.27), and whichever is mapped first serves the whole process.  Resolving
// at the first multi-GPU call picks up the copy that is already there (RTLD_NOLOAD) and otherwise the system one.
struct Nccl {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};
Nccl& nccl() {
  static Nccl n;
  static std::once_flag once;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
    if (!h) return;
    n.handle = h;
#define SYM(field, name) n.field = reinterpret_cast<decltype(n.field)>(dlsym(h, name))
    SYM(GetUniqueId, "ncclGetUniqueId"); SYM(CommInitRank, "ncclCommInitRank"); SYM(CommInitAll, "ncclCommInitAll"); SYM(CommDestroy, "ncclCommDestroy");
    SYM(AllReduce, "ncclAllReduce"); SYM(AllGather, "ncclAllGather"); SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    n.ok = n.GetUniqueId && n.CommInitRank && n.CommInitAll && n.CommDestroy && n.AllReduce && n.AllGather && n.GetErrorString;
  });
  return n;
}

// ---- a few host threads for pageable -> pinned staging copies ------------------------------------
class HostCopier {
 public:
  explicit HostCopier(int nthreads) : n_(std::max(1, nthreads)) {
    for (int t = 1; t < n_; t++) workers_.emplace_back([this, t] { loop(t); });
  }
  ~HostCopier() {
    { std::lock_guard<std::mutex> lk(m_); stop_ = true; gen_++; }
    cv_.notify_all();
    for (auto& w : workers_) w.join();
  }
  void copy(void* dst, const void* src, size_t bytes) {
    if (n_ == 1 || bytes < (1u << 20)) { memcpy(dst, src, bytes); return; }
    { std::lock_guard<std::mutex> lk(m_); dst_ = (char*)dst; src_ = (const char*)src; bytes_ = bytes; pending_ = n_ - 1; gen_++; }
    cv_.notify_all();
    slice(0);
    std::unique_lock<std::mutex> lk(m_);
    done_.wait(lk, [this] { return pending_ == 0; });
  }

 private:
  void slice(int t) {
    const size_t per = (bytes_ / n_ + 63) & ~(size_t)63, lo = std::min(bytes_, per * t), hi = (t == n_ - 1) ? bytes_ : std::min(bytes_, per * (t + 1));
    if (hi > lo) memcpy(dst_ + lo, src_ + lo, hi - lo);
  }
  void loop(int t) {
    uint64_t seen = 0;
    for (;;) {
      { std::unique_lock<std::mutex> lk(m_); cv_.wait(lk, [&] { return gen_ != seen; }); seen = gen_; if (stop_) return; }
      slice(t);
      { std::lock_guard<std::mutex> lk(m_); pending_--; }
      done_.notify_one();
    }
  }
  int n_;
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cv_, done_;
  char* dst_ = nullptr; const char* src_ = nullptr; size_t bytes_ = 0;
  int pending_ = 0; uint64_t gen_ = 0; bool stop_ = false;
};

// ---- one worker thread per device of a single-process multi-GPU group -----------------------------
class Workers {
 public:
  explicit Workers(int n) : n_(n), rc_(n, 0) {
    for (int t = 0; t < n_; t++) threads_.emplace_back([this, t] { loop(t); });
  }
  ~Workers() {
    { std::lock_guard<std::mutex> lk(m_); stop_ = true; gen_++; }
    cv_.notify_all();
    for (auto& w : threads_) w.join();
  }
  // runs fn(rank) on every worker concurrently; returns the first non-zero status
  int run(const std::function<int(int)>& fn) {
    { std::lock_guard<std::mutex> lk(m_); fn_ = &fn; pending_ = n_; gen_++; }
    cv_.notify_all();
    std::unique_lock<std::mutex> lk(m_);
    done_.wait(lk, [this] { return pending_ == 0; });
    for (int r : rc_) if (r) return r;
    return 0;
  }

 private:
  void loop(int t) {
    uint64_t seen = 0;
    for (;;) {
      const std::function<int(int)>* fn;
      { std::unique_lock<std::mutex> lk(m_); cv_.wait(lk, [&] { return gen_ != seen; }); seen = gen_; if (stop_) return; fn = fn_; }
      const int rc = (*fn)(t);
      { std::lock_guard<std::mutex> lk(m_); rc_[t] = rc; pending_--; }
      done_.notify_one();
    }
  }
  int n_;
  std::vector<int> rc_;
  std::vector<std::thread> threads_;
  std::mutex m_;
  std::condition_variable cv_, done_;
  const std::function<int(int)>* fn_ = nullptr;
  int pending_ = 0; uint64_t gen_ = 0; bool stop_ = false;
};

struct DataSet {
  // the data of lsqr_upload: each rank of a sharded context refines its own point range and the moments are all-reduced.
  // The data of a direct estimator call (least squares) stays whole on one device.
  bool sharded = false;
  double* soa64 = nullptr;
  float* soa32 = nullptr;
  uint32_t* maskbits = nullptr;
  double* center_dev = nullptr;   // kMaxDim doubles
  size_t ld = 0, cap = 0;   // cap = allocated leading dimension
  uint32_t n = 0;
  int D = 0, capD = 0;
  bool moments_valid = false;  // rb.moments holds the LS moments of the stored consensus set
  bool mask_valid = false;
  bool bytes_valid = false;    // ctx->mask_dev holds the consensus set of this data set, one byte per datum (own shard)
  DataView view() const {
    DataView v;
    v.soa64 = soa64; v.soa32 = soa32; v.ld = ld; v.span = ld; v.n = n; v.center = center_dev;
    return v;
  }
  // columns [lo, hi) of the data set (lo a multiple of 1024); `to_end`: the view runs to the NaN-padded end of the arrays
  DataView range(size_t lo, size_t hi, bool to_end) const {
    DataView v = view();
    v.soa64 = soa64 + lo; v.soa32 = soa32 + lo; v.n = (uint32_t)(hi - lo); v.span = to_end ? ld - lo : hi - lo;
    return v;
  }
};

struct Group {
  std::vector<lsqr_ctx*> kids;
  std::unique_ptr<Workers> workers;
};

}  // namespace

struct lsqr_ctx {
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaStream_t copy_stream = nullptr;
  std::string err;
  uint64_t launches = 0;

  int model = -1;
  EstCfg cfg{};
  double delta = 0, aux = 0;
  int ls_type = 1;

  DataSet main{true}, scratch{false};
  unsigned char* staging = nullptr; size_t staging_cap = 0;

  // hypothesis buffers
  size_t hcap = 0;
  int32_t* subsets = nullptr; double* hyp64 = nullptr; float* hyp32 = nullptr; uint32_t* counts = nullptr;
  float* hyp32b = nullptr; uint32_t* live_counts = nullptr; uint32_t* live_ids = nullptr; uint32_t* prune_dev = nullptr;   // early exit (Prune)
  int32_t* list_dev = nullptr; size_t list_cap = 0;
  double* params_in_dev = nullptr; size_t params_in_cap = 0;
  unsigned long long* key_dev = nullptr;  // [0] key, [1] n_valid (as u32 in low half)
  WinnerRecord* winner_dev = nullptr;
  double* small_dev = nullptr;            // kSmall doubles: parameters in @kSmIn, solve out @kSmOut, LM state @kSmLm, estimate() input @kSmEst, sink @kSmSink
  // refine
  RefineBuffers rb{};
  // pinned host scratch
  double* pin = nullptr;                  // 64 doubles, then one WinnerRecord
  WinnerRecord* winner_pin = nullptr;
  double* weights_dev = nullptr; size_t weights_cap = 0;   // lsqr_weighted_least_squares
  double* bt_data = nullptr; size_t bt_data_cap = 0;       // lsqr_ransac_batch: packed problems, offsets, results
  uint64_t* bt_off = nullptr; size_t bt_off_cap = 0;
  double* bt_prm = nullptr; size_t bt_prm_cap = 0;
  uint32_t* bt_cnt = nullptr; size_t bt_cnt_cap = 0;
  uint32_t* bt_cl = nullptr; size_t bt_cl_cap = 0;         //   the problems that take the cluster path, grouped by cluster size
  // lsqr_ransac_batch_device: offsets and cluster lists go up from two page-locked slots used in turn (a copy from pageable
  // memory may wait for the stream); bd_ev[i] is recorded after slot i's copies
  unsigned char* bd_pin[2] = {nullptr, nullptr}; size_t bd_pin_cap[2] = {0, 0};
  cudaEvent_t bd_ev[2]{};
  uint64_t bd_calls = 0;
  cudaEvent_t bd_order[2]{};              // [0]: the caller's stream waits for the context's stream, [1]: the reverse
  unsigned char* gather_dev = nullptr; size_t gather_cap = 0;        // compute(): records of the first round's minimal subsets
  unsigned char* gather_pin = nullptr; size_t gather_pin_cap = 0;
  uint8_t* mask_dev = nullptr; size_t mask_dev_cap = 0;   // consensus set, one byte per datum (device)
  uint8_t* mask_pin = nullptr; size_t mask_pin_cap = 0;   // pinned bounce buffer for its download
  double* agree_pin = nullptr;                            // lsqr_agree on a handful of data: zero-copy parameters, data and answers
  // upload pipeline
  static constexpr int kRing = 4;
  unsigned char* up_pin[kRing] = {nullptr, nullptr, nullptr, nullptr}; size_t up_pin_cap[kRing] = {0, 0, 0, 0};
  cudaEvent_t up_ev[kRing]{};             // chunk in ring slot i has been copied to the device
  cudaEvent_t up_land[8]{};               // chunk copies landed, round-robin
  std::unique_ptr<HostCopier> copier;
  cudaEvent_t ev[6]{};

  // sharding
  int rank = 0, world = 1;
  lsqr_allreduce_max_u64_fn max_fn = nullptr;
  lsqr_allreduce_sum_f64_fn sum_fn = nullptr;
  void* comm_user = nullptr;
  ncclComm_t comm = nullptr;              // native collectives (lsqr_ctx_create_multi / lsqr_ctx_init_nccl)
  Group* group = nullptr;                 // the handle returned by lsqr_ctx_create_multi: no device state of its own

  // stats of the last refine
  double refine_kernel_ms = 0, refine_bytes = 0;
  int lm_iterations = 0;
};

namespace {

int fail(lsqr_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg;
  return code;
}
#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess) return fail(ctx, LSQR_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
  } while (0)
#define CKL()                                                                                            \
  do {                                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                                \
    if (e__ != cudaSuccess) return fail(ctx, LSQR_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e__)); \
  } while (0)
#define CKN(call)                                                                                        \
  do {                                                                                                   \
    ncclResult_t r__ = (call);                                                                           \
    if (r__ != ncclSuccess) return fail(ctx, LSQR_ERR_COMM, std::string(#call) + ": " + nccl().GetErrorString(r__)); \
  } while (0)

template <class T> int ensure(lsqr_ctx* ctx, T** p, size_t* cap, size_t want) {
  if (*cap >= want && *p) return 0;
  if (*p) cudaFree(*p);
  *p = nullptr; *cap = 0;
  CK(cudaMalloc((void**)p, want * sizeof(T)));
  *cap = want;
  return 0;
}
// the same for page-locked host memory
template <class T> int ensure_pinned(lsqr_ctx* ctx, T** p, size_t* cap, size_t want) {
  if (*cap >= want && *p) return 0;
  if (*p) cudaFreeHost(*p);
  *p = nullptr; *cap = 0;
  CK(cudaMallocHost((void**)p, want * sizeof(T)));
  *cap = want;
  return 0;
}

size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }

void free_dataset(DataSet& ds) {
  cudaFree(ds.soa64); cudaFree(ds.soa32); cudaFree(ds.maskbits); cudaFree(ds.center_dev);
  ds = DataSet{ds.sharded};
}

int ensure_dataset(lsqr_ctx* ctx, DataSet& ds, int D, uint32_t n) {
  const size_t ld = round_up(std::max<size_t>(n, 1), kTilePad);
  if (!ds.center_dev) {
    CK(cudaMalloc((void**)&ds.center_dev, sizeof(double) * kMaxDim));
    CK(cudaMemsetAsync(ds.center_dev, 0, sizeof(double) * kMaxDim, ctx->stream));
  }
  if (ds.cap < ld || ds.capD < D) {
    if (ds.soa64) cudaFree(ds.soa64);
    if (ds.soa32) cudaFree(ds.soa32);
    if (ds.maskbits) cudaFree(ds.maskbits);
    ds.soa64 = nullptr; ds.soa32 = nullptr; ds.maskbits = nullptr; ds.cap = 0;
    const int Dc = std::max(D, ds.capD);
    CK(cudaMalloc((void**)&ds.soa64, sizeof(double) * Dc * ld));
    CK(cudaMalloc((void**)&ds.soa32, sizeof(float) * Dc * ld));
    CK(cudaMalloc((void**)&ds.maskbits, sizeof(uint32_t) * (ld / 32)));
    ds.cap = ld; ds.capD = Dc;
  }
  ds.ld = ld; ds.n = n; ds.D = D;
  ds.moments_valid = false; ds.mask_valid = false; ds.bytes_valid = false;
  return 0;
}

int ensure_hyp(lsqr_ctx* ctx, size_t H) {
  const size_t want = round_up(std::max<size_t>(H, 1), 256);
  if (ctx->hcap >= want) return 0;
  if (ctx->subsets) cudaFree(ctx->subsets);
  if (ctx->hyp64) cudaFree(ctx->hyp64);
  if (ctx->hyp32) cudaFree(ctx->hyp32);
  if (ctx->counts) cudaFree(ctx->counts);
  cudaFree(ctx->hyp32b); cudaFree(ctx->live_counts); cudaFree(ctx->live_ids); cudaFree(ctx->prune_dev);
  ctx->subsets = nullptr; ctx->hyp64 = nullptr; ctx->hyp32 = nullptr; ctx->counts = nullptr; ctx->hcap = 0;
  ctx->hyp32b = nullptr; ctx->live_counts = nullptr; ctx->live_ids = nullptr; ctx->prune_dev = nullptr;
  CK(cudaMalloc((void**)&ctx->subsets, sizeof(int32_t) * LSQR_MAX_SUBSET * want));
  CK(cudaMalloc((void**)&ctx->hyp64, sizeof(double) * LSQR_MAX_PARAMS * want));
  CK(cudaMalloc((void**)&ctx->hyp32, sizeof(float) * 16 * want));   // up to four float4 groups per hypothesis (8-D line: 16 constants)
  CK(cudaMalloc((void**)&ctx->counts, sizeof(uint32_t) * want));
  CK(cudaMalloc((void**)&ctx->hyp32b, sizeof(float) * 16 * want));
  CK(cudaMalloc((void**)&ctx->live_counts, sizeof(uint32_t) * 2 * want));
  CK(cudaMalloc((void**)&ctx->live_ids, sizeof(uint32_t) * 2 * want));
  CK(cudaMalloc((void**)&ctx->prune_dev, sizeof(uint32_t) * prune_dev_words(want)));
  ctx->hcap = want;
  return 0;
}

// ---- collectives ---------------------------------------------------------------------------------
int comm_max_u64(lsqr_ctx* ctx, unsigned long long* dev) {
  if (ctx->world <= 1) return 0;
  if (ctx->comm) { CKN(nccl().AllReduce(dev, dev, 1, ncclUint64, ncclMax, ctx->comm, ctx->stream)); return 0; }
  if (!ctx->max_fn) return fail(ctx, LSQR_ERR_COMM, "sharded context without an all-reduce hook");
  if (ctx->max_fn(ctx->comm_user, reinterpret_cast<uint64_t*>(dev), (void*)ctx->stream)) return fail(ctx, LSQR_ERR_COMM, "max all-reduce hook failed");
  return 0;
}
int comm_sum_f64(lsqr_ctx* ctx, double* dev, int count) {
  if (ctx->world <= 1) return 0;
  if (ctx->comm) { CKN(nccl().AllReduce(dev, dev, (size_t)count, ncclDouble, ncclSum, ctx->comm, ctx->stream)); return 0; }
  if (!ctx->sum_fn) return fail(ctx, LSQR_ERR_COMM, "sharded context without a sum all-reduce hook");
  if (ctx->sum_fn(ctx->comm_user, dev, count, (void*)ctx->stream)) return fail(ctx, LSQR_ERR_COMM, "sum all-reduce hook failed");
  return 0;
}

// the threads of the staging copies between pageable and pinned memory, created on first use: most of the cores, shared between
// the devices of a group
HostCopier& copier(lsqr_ctx* ctx) {
  if (!ctx->copier) {
    const int W = ctx->comm && ctx->world > 1 ? ctx->world : 1;
    ctx->copier.reset(new HostCopier(std::min(12, std::max(1, ((int)std::thread::hardware_concurrency() * 3 / 4) / W))));
  }
  return *ctx->copier;
}

// ---- upload ----------------------------------------------------------------------------------------
bool is_pinned(const void* p) {
  cudaPointerAttributes attr{};
  const bool ok = cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  if (!ok) cudaGetLastError();   // an unregistered pointer is not an error here
  return ok;
}

// Host -> device copies on the copy stream, overlapping the work that the compute stream does with what has landed: straight
// from page-locked memory; from pageable memory through the ring of pinned buffers, which the staging threads fill.
struct StagedCopy {
  lsqr_ctx* ctx;
  bool pinned;   // the source is page-locked
  int ring = 0, land = 0;
  // before the first put(): `piece` = the largest put().  The copies must not overtake work already enqueued on the compute
  // stream (it may still read their destination).
  int start(size_t piece) {
    if (!pinned) {
      CK(cudaStreamSynchronize(ctx->copy_stream));   // an earlier upload may still be reading the pinned ring
      for (int i = 0; i < lsqr_ctx::kRing; i++) if (int rc = ensure_pinned(ctx, &ctx->up_pin[i], &ctx->up_pin_cap[i], piece)) return rc;
      copier(ctx);
    }
    CK(cudaEventRecord(ctx->up_land[7], ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->up_land[7], 0));
    return LSQR_OK;
  }
  int put(void* dst, const void* src, size_t bytes) {
    if (pinned) { CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->copy_stream)); return LSQR_OK; }
    const int b = ring % lsqr_ctx::kRing;
    if (ring >= lsqr_ctx::kRing) CK(cudaEventSynchronize(ctx->up_ev[b]));   // the copy that used this buffer has finished
    ring++;
    ctx->copier->copy(ctx->up_pin[b], src, bytes);
    CK(cudaMemcpyAsync(dst, ctx->up_pin[b], bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
    CK(cudaEventRecord(ctx->up_ev[b], ctx->copy_stream));
    return LSQR_OK;
  }
  // the compute stream waits for every copy enqueued so far
  int landed() {
    cudaEvent_t ev = ctx->up_land[land++ % 7];
    CK(cudaEventRecord(ev, ctx->copy_stream));
    CK(cudaStreamWaitEvent(ctx->stream, ev, 0));
    return LSQR_OK;
  }
};

// AoS records, host or device -> SoA fp64 + fp32 on the device, chunk by chunk.
//   * single context: chunk c is copied on the copy stream and transposed on the compute stream as soon as it has landed;
//   * natively sharded context (ctx->comm): rank r copies chunks r, r + W, r + 2W, ... of the host buffer and round j of
//     chunks [jW, (j+1)W) is completed by an in-place all-gather over NVLink before it is transposed.
// after_round(lo, hi, first, last): called after the transposition of records [lo, hi) has been enqueued (compute() scores its
// first round of hypotheses against every range as it lands)
using RoundFn = std::function<int(size_t, size_t, bool, bool)>;
int upload_to(lsqr_ctx* ctx, DataSet& ds, const void* aos, size_t n, size_t stride, bool on_device, const RoundFn* after_round = nullptr) {
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called before uploading data");
  const ModelInfo mi = model_info(ctx->model);
  if (n > 0xFFFFFFF0ull) return fail(ctx, LSQR_ERR_ARG, "too many data records");
  if (stride < sizeof(double) * mi.D || (stride % sizeof(double)) != 0) return fail(ctx, LSQR_ERR_ARG, "stride must be a multiple of 8 and >= 8*dim");
  if (n && !aos) return fail(ctx, LSQR_ERR_ARG, "null data pointer");
  CK(cudaSetDevice(ctx->device));
  if (int rc = ensure_dataset(ctx, ds, mi.D, (uint32_t)n)) return rc;
  cudaStream_t s = ctx->stream;
  CK(cudaMemsetAsync(ds.maskbits, 0, sizeof(uint32_t) * (ds.ld / 32), s));
  const uint32_t N = (uint32_t)n, pad_to = (uint32_t)ds.ld;
  const uint32_t sample = std::min<uint32_t>(N, kCenterSample);
  if (on_device || n == 0) {
    const unsigned char* src = static_cast<const unsigned char*>(aos);
    launch_center_sample(ctx->model, src, stride, sample, ds.center_dev, s);
    launch_ingest(ctx->model, src, stride, 0, N, pad_to, ds.center_dev, ds.soa64, ds.soa32, ds.ld, s);
    ctx->launches += 2;
    CKL();
    return LSQR_OK;
  }
  const bool sharded = ds.sharded && ctx->comm != nullptr && ctx->world > 1;
  const int W = sharded ? ctx->world : 1;
  StagedCopy up{ctx, is_pinned(aos)};
  // chunk: at least the centre sample, ~1/8 of a rank's share, between 256 KB and 16 MB (4 MB from pageable memory: the first
  // copy cannot start before the first chunk has been staged)
  const size_t chunk_cap = up.pinned ? (16u << 20) : (4u << 20);
  size_t chunk_rec = std::max<size_t>(kCenterSample, std::min<size_t>(chunk_cap / stride, std::max<size_t>((256u << 10) / stride, (n / W + 7) / 8)));
  chunk_rec = round_up(chunk_rec, 1024);   // rounds start on tile boundaries of every consensus kernel
  const size_t chunk_bytes = chunk_rec * stride;
  const size_t n_chunks = (n + chunk_rec - 1) / chunk_rec, rounds = (n_chunks + W - 1) / W;
  if (int rc = ensure(ctx, &ctx->staging, &ctx->staging_cap, rounds * W * chunk_bytes)) return rc;
  if (int rc = up.start(chunk_bytes)) return rc;
  const unsigned char* host = static_cast<const unsigned char*>(aos);
  for (size_t j = 0; j < rounds; j++) {
    const size_t g = j * W + (sharded ? ctx->rank : 0);       // the chunk this rank fetches in round j
    const size_t lo = std::min(n, g * chunk_rec), hi = std::min(n, (g + 1) * chunk_rec);
    if (hi > lo) if (int rc = up.put(ctx->staging + g * chunk_bytes, host + lo * stride, (hi - lo) * stride)) return rc;
    if (int rc = up.landed()) return rc;
    if (sharded) CKN(nccl().AllGather(ctx->staging + g * chunk_bytes, ctx->staging + j * W * chunk_bytes, chunk_bytes, ncclUint8, ctx->comm, s));
    if (j == 0) { launch_center_sample(ctx->model, ctx->staging, stride, sample, ds.center_dev, s); ctx->launches++; }
    const size_t r_lo = std::min(n, j * W * chunk_rec), r_hi = std::min(n, (j + 1) * W * chunk_rec);
    const bool last = j + 1 == rounds;
    launch_ingest(ctx->model, ctx->staging, stride, (uint32_t)r_lo, (uint32_t)(r_hi - r_lo), last ? pad_to : (uint32_t)r_hi, ds.center_dev, ds.soa64, ds.soa32, ds.ld, s);
    ctx->launches++;
    if (after_round) if (int rc = (*after_round)(r_lo, r_hi, j == 0, last)) return rc;
  }
  CKL();
  return LSQR_OK;
}

// Number of subsets as the reference counts them (RANSAC::choose, RANSAC.hxx:254-280): the binomial
// coefficient evaluated in double precision as a ratio of two running products, saturating at
// UINT_MAX when either the result or an intermediate does not fit.  The stop rule clamps the
// number of tries with this value (RANSAC.hxx:41,110), so the same saturation must happen here.
unsigned int choose_ref(unsigned int n, unsigned int m) {
  const unsigned int small = std::min(m, n - m);         // multiply the shorter run of factors
  double num = 1.0, den = 1.0;
  for (unsigned int f = n - small + 1; f <= n && f != 0; f++) num *= static_cast<double>(f);
  for (unsigned int f = 1; f <= small; f++) den *= static_cast<double>(f);
  const double c = num / den;
  const double dmax = std::numeric_limits<double>::max(), umax = static_cast<double>(std::numeric_limits<unsigned int>::max());
  if (num > dmax || den > dmax || c > umax) return std::numeric_limits<unsigned int>::max();
  return static_cast<unsigned int>(c);
}

uint64_t choose_exact(uint64_t n, uint64_t k) {
  if (k > n) return 0;
  long double r = 1;
  for (uint64_t i = 0; i < k; i++) r = r * (long double)(n - i) / (long double)(i + 1);
  if (r > 1.8e19L) return ~0ull;
  return (uint64_t)(r + 0.5L);
}

// The stop rule of RANSAC.hxx:104-110 after a new best count.
uint64_t tries_after(uint32_t best_count, uint32_t n, int K, double numerator, unsigned int all_tries) {
  const double denominator = log(1.0 - pow((double)best_count / (double)n, (double)K));  // :107
  const double t = numerator / denominator + 0.5;
  const uint64_t nt = (t >= 4294967295.0 || !(t == t)) ? 0xFFFFFFFFull : (t < 0 ? 0x80000000ull : (uint64_t)t);  // (int) cast semantics of :108
  return std::min<uint64_t>(nt, all_tries);  // :110
}

constexpr size_t kHypBatch = (size_t)1 << 22;

// The winner of a request whose first hypothesis is `first` -> its count, index, parameters and subset.
void decode_winner(const WinnerRecord& w, uint64_t first, const ModelInfo& mi, lsqr_score_result* res) {
  res->n_valid = (uint32_t)w.n_valid;
  res->best_count = (uint32_t)(w.key >> 32);
  for (int j = 0; j < LSQR_MAX_SUBSET; j++) res->best_subset[j] = -1;
  res->best_index = 0;
  if (res->best_count == 0) return;
  res->best_index = first + (0xFFFFFFFFull - (w.key & 0xFFFFFFFFull));
  for (int j = 0; j < mi.P; j++) res->best_params[j] = w.params[j];
  for (int j = 0; j < mi.K; j++) res->best_subset[j] = w.subset[j];
}

// Minimal solve + consensus + arg-max of one request; the winner is re-derived on the device and fetched with one copy.
int score_impl(lsqr_ctx* ctx, const lsqr_score_args* a, lsqr_score_result* res) {
  DataSet& ds = ctx->main;
  if (!ds.soa64) return fail(ctx, LSQR_ERR_STATE, "no data uploaded");
  if (!a || !res) return fail(ctx, LSQR_ERR_ARG, "null argument");
  const ModelInfo mi = model_info(ctx->model);
  if (a->count > 0xFFFFFFFEull) return fail(ctx, LSQR_ERR_ARG, "at most 2^32-2 hypotheses per request");
  if (a->sampler < 0 || a->sampler > 3) return fail(ctx, LSQR_ERR_ARG, "bad sampler");
  if (a->sampler == LSQR_SAMPLE_LIST && !a->subsets) return fail(ctx, LSQR_ERR_ARG, "subset list missing");
  if (a->sampler == LSQR_SAMPLE_PARAMS && !a->params) return fail(ctx, LSQR_ERR_ARG, "parameter list missing");
  CK(cudaSetDevice(ctx->device));
  memset(res, 0, sizeof(*res));   // (res->evals accumulates over the batches below)
  const uint64_t H = a->count;
  const uint64_t lo = H * (uint64_t)ctx->rank / (uint64_t)ctx->world, hi = H * (uint64_t)(ctx->rank + 1) / (uint64_t)ctx->world;
  const bool can_sample = ds.n >= (uint32_t)mi.K || a->sampler == LSQR_SAMPLE_PARAMS;
  const DataView dv = ds.view();
  cudaStream_t s = ctx->stream;
  CK(cudaMemsetAsync(ctx->key_dev, 0, 2 * sizeof(unsigned long long), s));
  CK(cudaEventRecord(ctx->ev[0], s));
  float cons_ms = 0.f;
  const bool listed = a->sampler == LSQR_SAMPLE_LIST || a->sampler == LSQR_SAMPLE_PARAMS;
  const bool one_batch = hi - lo <= kHypBatch;
  bool timed = false;
  if (can_sample) {
    for (uint64_t b0 = lo; b0 < hi; b0 += kHypBatch) {
      const uint32_t B = (uint32_t)std::min<uint64_t>(kHypBatch, hi - b0);
      if (int rc = ensure_hyp(ctx, B)) return rc;
      SolveArgs sa{};
      sa.model = ctx->model; sa.sampler = a->sampler; sa.seed = a->seed; sa.first = a->first + b0; sa.H = B; sa.hld = ctx->hcap;
      sa.subsets = ctx->subsets; sa.hyp64 = ctx->hyp64; sa.n_valid = reinterpret_cast<uint32_t*>(ctx->key_dev + 1);
      if (a->sampler == LSQR_SAMPLE_LIST) {
        if (int rc = ensure(ctx, &ctx->list_dev, &ctx->list_cap, (size_t)B * mi.K)) return rc;
        CK(cudaMemcpyAsync(ctx->list_dev, a->subsets + b0 * mi.K, sizeof(int32_t) * (size_t)B * mi.K, cudaMemcpyHostToDevice, s));
        sa.list = ctx->list_dev;
      } else if (a->sampler == LSQR_SAMPLE_PARAMS) {
        if (int rc = ensure(ctx, &ctx->params_in_dev, &ctx->params_in_cap, (size_t)B * mi.P)) return rc;
        CK(cudaMemcpyAsync(ctx->params_in_dev, a->params + b0 * mi.P, sizeof(double) * (size_t)B * mi.P, cudaMemcpyHostToDevice, s));
        sa.params_in = ctx->params_in_dev;
      }
      launch_solve(sa, dv, ctx->cfg, s); ctx->launches++;
      if (a->precision == LSQR_FP32) { launch_hoist32(ctx->model, ctx->hyp64, ctx->hcap, B, dv, ctx->cfg, ctx->hyp32, s); ctx->launches++; }
      CK(cudaMemsetAsync(ctx->counts, 0, sizeof(uint32_t) * B, s));
      // without per-hypothesis counts only the winner matters: hypotheses that can no longer tie it stop being scored; the
      // request's hoisted constants are not read again once the live list has been compacted out of them
      Prune pr{{ctx->hyp32b, ctx->hyp32}, {ctx->live_counts, ctx->live_counts + ctx->hcap}, {ctx->live_ids, ctx->live_ids + ctx->hcap},
               ctx->prune_dev, reinterpret_cast<uint32_t*>(ctx->pin) /* host scratch */, ctx->key_dev, (uint64_t)B * dv.n};
      CK(cudaEventRecord(ctx->ev[2], s));
      ctx->launches += launch_consensus(ctx->model, a->precision, dv, ctx->hyp64, ctx->hyp32, ctx->hcap, B, ctx->cfg, ctx->counts, ctx->num_sms, s,
                                        a->out_counts ? nullptr : &pr);
      CK(cudaEventRecord(ctx->ev[3], s));
      res->evals += pr.evals;
      timed = true;
      launch_argmax(ctx->counts, B, (uint32_t)b0, ctx->key_dev, s); ctx->launches++;
      CKL();
      if (a->out_counts) CK(cudaMemcpyAsync(a->out_counts + b0, ctx->counts, sizeof(uint32_t) * B, cudaMemcpyDeviceToHost, s));
      if (a->out_params) {
        // device layout is [P][hld]; gather rows on the host side of the copy
        std::vector<double> tmp((size_t)B * mi.P);
        CK(cudaMemcpy2DAsync(tmp.data(), sizeof(double) * B, ctx->hyp64, sizeof(double) * ctx->hcap, sizeof(double) * B, mi.P, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        for (uint32_t h = 0; h < B; h++) for (int j = 0; j < mi.P; j++) a->out_params[(b0 + h) * mi.P + j] = tmp[(size_t)j * B + h];
      }
      if (!one_batch) {   // the event pair is reused by the next batch
        CK(cudaEventSynchronize(ctx->ev[3]));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]));
        cons_ms += ms;
      }
    }
  }
  if (int rc = comm_max_u64(ctx, ctx->key_dev)) return rc;
  // the winner, on the device: index-based samplers always; listed ones when the request's list is still resident (one batch
  // and the whole request on this rank, i.e. unsharded)
  const bool dev_winner = !listed || (one_batch && ctx->world == 1 && can_sample && hi > lo);
  if (dev_winner) {
    SolveArgs wa{};
    wa.model = ctx->model; wa.sampler = a->sampler; wa.seed = a->seed; wa.first = a->first;
    wa.list = ctx->list_dev; wa.params_in = ctx->params_in_dev;
    launch_winner(wa, ctx->key_dev, dv, ctx->cfg, ctx->winner_dev, s); ctx->launches++;
    CK(cudaEventRecord(ctx->ev[1], s));
    CKL();
    CK(cudaMemcpyAsync(ctx->winner_pin, ctx->winner_dev, sizeof(WinnerRecord), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  } else {
    CK(cudaEventRecord(ctx->ev[1], s));
    CK(cudaMemcpyAsync(ctx->winner_pin, ctx->key_dev, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    ctx->winner_pin->n_valid &= 0xFFFFFFFFull;
  }
  float total_ms = 0.f;
  CK(cudaEventElapsedTime(&total_ms, ctx->ev[0], ctx->ev[1]));
  if (one_batch && timed) { float ms = 0.f; CK(cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3])); cons_ms = ms; }
  res->score_ms = total_ms; res->consensus_ms = cons_ms;
  decode_winner(*ctx->winner_pin, a->first, mi, res);   // without dev_winner the record holds the key only: see below
  if (dev_winner || res->best_count == 0) return LSQR_OK;
  // listed sampler whose winner's row is no longer on this device: upload that one row and solve it
  const uint64_t rel = res->best_index - a->first;
  if (int rc = ensure_hyp(ctx, 1)) return rc;
  SolveArgs sa{};
  sa.model = ctx->model; sa.sampler = a->sampler; sa.seed = a->seed; sa.first = res->best_index; sa.H = 1; sa.hld = ctx->hcap;
  sa.subsets = ctx->subsets; sa.hyp64 = ctx->hyp64; sa.n_valid = reinterpret_cast<uint32_t*>(ctx->key_dev + 1);
  if (a->sampler == LSQR_SAMPLE_LIST) {
    if (int rc = ensure(ctx, &ctx->list_dev, &ctx->list_cap, (size_t)mi.K)) return rc;
    CK(cudaMemcpyAsync(ctx->list_dev, a->subsets + rel * mi.K, sizeof(int32_t) * mi.K, cudaMemcpyHostToDevice, s));
    sa.list = ctx->list_dev;
  } else {
    if (int rc = ensure(ctx, &ctx->params_in_dev, &ctx->params_in_cap, (size_t)mi.P)) return rc;
    CK(cudaMemcpyAsync(ctx->params_in_dev, a->params + rel * mi.P, sizeof(double) * mi.P, cudaMemcpyHostToDevice, s));
    sa.params_in = ctx->params_in_dev;
  }
  launch_solve(sa, dv, ctx->cfg, s); ctx->launches++;
  CKL();
  double hp[LSQR_MAX_PARAMS]; int32_t hs[LSQR_MAX_SUBSET];
  CK(cudaMemcpy2DAsync(hp, sizeof(double), ctx->hyp64, sizeof(double) * ctx->hcap, sizeof(double), mi.P, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpy2DAsync(hs, sizeof(int32_t), ctx->subsets, sizeof(int32_t) * ctx->hcap, sizeof(int32_t), mi.K, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  for (int j = 0; j < mi.P; j++) res->best_params[j] = hp[j];
  for (int j = 0; j < mi.K; j++) res->best_subset[j] = hs[j];
  return LSQR_OK;
}

int reduce_moments(lsqr_ctx* ctx, const DataSet& ds, int nm) {
  launch_reduce_partials(ctx->rb, nm, ctx->stream); ctx->launches++;
  return ds.sharded ? comm_sum_f64(ctx, ctx->rb.moments, nm) : LSQR_OK;
}

// this rank's data of the data set, [begin, end)
void shard_range(const lsqr_ctx* ctx, const DataSet& ds, uint32_t* begin, uint32_t* end) {
  const uint32_t n = ds.n;
  if (!ds.sharded || ctx->world <= 1) { *begin = 0; *end = n; return; }
  const uint64_t words = ((uint64_t)n + 31) / 32;
  const uint64_t w0 = words * (uint64_t)ctx->rank / (uint64_t)ctx->world, w1 = words * (uint64_t)(ctx->rank + 1) / (uint64_t)ctx->world;
  *begin = (uint32_t)std::min<uint64_t>(w0 * 32, n);
  *end = (uint32_t)std::min<uint64_t>(w1 * 32, n);
}

// P parameters from the host -> small_dev + kSmIn, through the pinned scratch
int put_params(lsqr_ctx* ctx, const double* params) {
  const int P = model_info(ctx->model).P;
  for (int j = 0; j < P; j++) ctx->pin[32 + j] = params[j];
  CK(cudaMemcpyAsync(ctx->small_dev + kSmIn, ctx->pin + 32, sizeof(double) * P, cudaMemcpyHostToDevice, ctx->stream));
  return LSQR_OK;
}

// Consensus set of the parameters at params_dev (device) over this rank's point shard + the least-squares moments of it,
// enqueued only: no copy back, no synchronisation.  want_bytes: the pass also writes one byte per datum into ctx->mask_dev.
int consensus_enqueue(lsqr_ctx* ctx, DataSet& ds, const double* params_dev, bool want_bytes) {
  const ModelInfo mi = model_info(ctx->model);
  cudaStream_t s = ctx->stream;
  uint32_t b, e;
  shard_range(ctx, ds, &b, &e);
  const int nm = moments_count(ctx->model, false);
  if (want_bytes) if (int rc = ensure(ctx, &ctx->mask_dev, &ctx->mask_dev_cap, (size_t)std::max<uint32_t>(ds.n, 1))) return rc;
  CK(cudaEventRecord(ctx->ev[4], s));
  ctx->rb.maskbits = ds.maskbits;
  ctx->rb.maskbytes = want_bytes ? ctx->mask_dev : nullptr;
  launch_mask_moments(ctx->model, ds.view(), b, e, params_dev, 1, nullptr, ctx->cfg, ctx->rb, s); ctx->launches++;
  ctx->rb.maskbytes = nullptr;
  CK(cudaEventRecord(ctx->ev[5], s));
  if (int rc = reduce_moments(ctx, ds, nm)) return rc;
  CKL();
  ctx->refine_bytes = (double)(e - b) * mi.D * sizeof(double) + (double)(e - b) / 8.0 + (want_bytes ? (double)(e - b) : 0.0);
  ds.moments_valid = true; ds.mask_valid = true; ds.bytes_valid = want_bytes;
  return LSQR_OK;
}

int consensus_impl(lsqr_ctx* ctx, DataSet& ds, const double* params, uint32_t* out_count) {
  if (!ds.soa64) return fail(ctx, LSQR_ERR_STATE, "no data uploaded");
  cudaStream_t s = ctx->stream;
  CK(cudaSetDevice(ctx->device));
  if (int rc = put_params(ctx, params)) return rc;
  if (int rc = consensus_enqueue(ctx, ds, ctx->small_dev + kSmIn, false)) return rc;
  CK(cudaMemcpyAsync(ctx->pin, ctx->rb.moments, sizeof(double), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]));
  ctx->refine_kernel_ms = ms;
  if (out_count) *out_count = (uint32_t)(ctx->pin[0] + 0.5);
  return LSQR_OK;
}

// Least squares over the stored consensus set (or all data), enqueued; the result lands in small_dev + kSmOut
// ([0] = number of parameters, [1..] parameters).  Levenberg-Marquardt refits synchronise once per chunk of evaluations.
int refine_enqueue(lsqr_ctx* ctx, DataSet& ds, int use_mask) {
  cudaStream_t s = ctx->stream;
  const DataView dv = ds.view();
  ctx->rb.maskbits = ds.maskbits;
  ctx->rb.maskbytes = nullptr;
  uint32_t b, e;
  shard_range(ctx, ds, &b, &e);
  const int nm = moments_count(ctx->model, false);
  ctx->lm_iterations = 0;
  if (!(use_mask && ds.moments_valid)) {
    CK(cudaEventRecord(ctx->ev[4], s));
    launch_mask_moments(ctx->model, dv, b, e, nullptr, use_mask ? 2 : 0, nullptr, ctx->cfg, ctx->rb, s); ctx->launches++;
    CK(cudaEventRecord(ctx->ev[5], s));
    if (int rc = reduce_moments(ctx, ds, nm)) return rc;
    ds.moments_valid = false;
  }
  double* out_dev = ctx->small_dev + kSmOut;
  // iterative refinement: geometric circle / sphere fit, iterative ultrasound calibrations (ls_type 1 in both)
  const bool geometric = (model_family(ctx->model) == FAM_SPHERE || ctx->model == USXW || ctx->model == USCP) && ctx->ls_type == LSQR_LS_GEOMETRIC;
  launch_solve_moments(ctx->model, dv, ctx->rb.moments, geometric ? 1 : 0, out_dev, s); ctx->launches++;
  if (geometric) {
    // SphereParametersEstimator.hxx:224-230: algebraic fit as the start, then Levenberg-Marquardt.
    double* st = ctx->small_dev + kSmLm;
    const int nlm = moments_count(ctx->model, true);
    launch_lm_init(out_dev, st, s); ctx->launches++;
    ds.moments_valid = false;
    // The controller stops itself (500 / 5000 evaluations at most).  Passes are enqueued kLmAhead evaluations ahead of the
    // status word, so the host synchronises once per chunk instead of once per evaluation; passes behind a stop are no-ops.
    constexpr int kLmAhead = 8;
    for (int it = 0; it < 5200; it += kLmAhead) {
      for (int k = 0; k < kLmAhead; k++) {
        launch_mask_moments(ctx->model, dv, b, e, nullptr, use_mask ? 2 : 0, st, ctx->cfg, ctx->rb, s); ctx->launches++;
        if (int rc = reduce_moments(ctx, ds, nlm)) return rc;
        launch_lm_update(ctx->model, ctx->rb.moments, st, s); ctx->launches++;
      }
      CK(cudaMemcpyAsync(ctx->pin + 48, st + lm_status_offset(), 3 * sizeof(double), cudaMemcpyDeviceToHost, s));   // status, phase, evaluations
      CK(cudaStreamSynchronize(s));
      ctx->lm_iterations = (int)ctx->pin[50];
      if (ctx->pin[48] != 0.0) break;
    }
    launch_lm_finish(ctx->model, dv, st, out_dev, s); ctx->launches++;
  }
  CKL();
  return LSQR_OK;
}

int refine_impl(lsqr_ctx* ctx, DataSet& ds, int use_mask, double* out_params, int* n_params) {
  if (!ds.soa64) return fail(ctx, LSQR_ERR_STATE, "no data uploaded");
  if (use_mask && !ds.mask_valid) return fail(ctx, LSQR_ERR_STATE, "no consensus set stored; call lsqr_consensus first");
  const ModelInfo mi = model_info(ctx->model);
  cudaStream_t s = ctx->stream;
  CK(cudaSetDevice(ctx->device));
  if (int rc = refine_enqueue(ctx, ds, use_mask)) return rc;
  CK(cudaMemcpyAsync(ctx->pin, ctx->small_dev + kSmOut, sizeof(double) * (1 + LSQR_MAX_PARAMS), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  const int np = (int)ctx->pin[0];
  if (n_params) *n_params = np;
  if (out_params) for (int j = 0; j < np && j < mi.P; j++) out_params[j] = ctx->pin[1 + j];
  return LSQR_OK;
}

// pinned -> pageable copy of a result, by the staging threads when it is large
void host_copy(lsqr_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (bytes >= (1u << 20)) copier(ctx).copy(dst, src, bytes);
  else memcpy(dst, src, bytes);
}

// Enqueues the copy of this rank's part of the consensus set (bytes [b, e) of out_bytes; everything when unsharded) and
// reports whether a bounce through the pinned buffer has to be finished after the synchronisation.
int mask_download_enqueue(lsqr_ctx* ctx, DataSet& ds, uint8_t* out_bytes, bool* bounce, uint32_t* pb, uint32_t* pe) {
  uint32_t b, e;
  shard_range(ctx, ds, &b, &e);
  *pb = b; *pe = e; *bounce = false;
  if (!out_bytes || e <= b) return LSQR_OK;
  if (int rc = ensure(ctx, &ctx->mask_dev, &ctx->mask_dev_cap, (size_t)std::max<uint32_t>(ds.n, 1))) return rc;
  if (!ds.bytes_valid) { launch_expand_mask(ds.maskbits, b, e - b, ctx->mask_dev, ctx->stream); ctx->launches++; ds.bytes_valid = true; }
  // a caller buffer that is itself page-locked takes the DMA directly; any other goes through the library's pinned buffer
  // (persistent: a cudaMalloc/cudaFree pair per call costs up to 0.3 s after the thousands of launches of a large request)
  const bool direct = is_pinned(out_bytes);
  if (!direct) if (int rc = ensure_pinned(ctx, &ctx->mask_pin, &ctx->mask_pin_cap, ds.n)) return rc;
  CK(cudaMemcpyAsync((direct ? out_bytes : ctx->mask_pin) + b, ctx->mask_dev + b, e - b, cudaMemcpyDeviceToHost, ctx->stream));
  *bounce = !direct;
  return LSQR_OK;
}

int get_mask_impl(lsqr_ctx* ctx, DataSet& ds, uint8_t* out_bytes) {
  if (!ds.mask_valid) return fail(ctx, LSQR_ERR_STATE, "no consensus set stored");
  if (!out_bytes || ds.n == 0) return LSQR_OK;
  CK(cudaSetDevice(ctx->device));
  bool bounce; uint32_t b, e;
  if (int rc = mask_download_enqueue(ctx, ds, out_bytes, &bounce, &b, &e)) return rc;
  CK(cudaStreamSynchronize(ctx->stream));
  if (bounce) host_copy(ctx, out_bytes + b, ctx->mask_pin + b, e - b);
  return LSQR_OK;
}

// winner -> consensus set -> least squares: RANSAC.hxx:129-138 / :175-185.  Everything is enqueued behind the scoring; one
// synchronisation brings back count, parameters and the mask.  tries / score_ms: the hypotheses scored and their device time.
int finish_ransac(lsqr_ctx* ctx, const lsqr_score_result& best, uint64_t tries, double score_ms, uint8_t* out_mask, lsqr_compute_result* res) {
  res->tries = tries; res->device_ms = score_ms;
  res->best_count = best.best_count; res->best_index = best.best_index;
  if (best.best_count == 0) { res->n_params = 0; res->fraction = 0.0; return LSQR_OK; }
  const ModelInfo mi = model_info(ctx->model);
  cudaStream_t s = ctx->stream;
  DataSet& ds = ctx->main;
  if (int rc = put_params(ctx, best.best_params)) return rc;
  if (int rc = consensus_enqueue(ctx, ds, ctx->small_dev + kSmIn, out_mask != nullptr)) return rc;
  CK(cudaMemcpyAsync(ctx->pin, ctx->rb.moments, sizeof(double), cudaMemcpyDeviceToHost, s));
  bool bounce = false; uint32_t b = 0, e = 0;
  if (out_mask) if (int rc = mask_download_enqueue(ctx, ds, out_mask, &bounce, &b, &e)) return rc;
  if (int rc = refine_enqueue(ctx, ds, 1)) return rc;
  CK(cudaMemcpyAsync(ctx->pin + 1, ctx->small_dev + kSmOut, sizeof(double) * (1 + LSQR_MAX_PARAMS), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (bounce) host_copy(ctx, out_mask + b, ctx->mask_pin + b, e - b);
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]));
  ctx->refine_kernel_ms = ms;
  res->device_ms += ms;
  const uint32_t cnt = (uint32_t)(ctx->pin[0] + 0.5);
  const int np = (int)ctx->pin[1];
  res->best_count = cnt;
  res->n_params = np;
  for (int j = 0; j < np && j < mi.P; j++) res->params[j] = ctx->pin[2 + j];
  res->fraction = (double)cnt / (double)ds.n;
  return LSQR_OK;
}

// lsqr_ransac's adaptive loop (RANSAC.hxx:100-110): hypotheses [0, done) have been scored, `best` is the first of the best.
struct RansacRounds {
  uint32_t n; int K;
  double numerator;          // log(1 - prob)
  unsigned int all_tries;    // RANSAC.hxx:41
  uint64_t num_tries, done = 0;
  lsqr_score_result best{};
  bool perfect = false;      // a hypothesis agrees with every datum
  double dev_ms = 0;

  RansacRounds(uint32_t n_, int K_, double prob) : n(n_), K(K_), numerator(log(1.0 - prob)), all_tries(choose_ref(n_, (unsigned)K_)), num_tries(all_tries) {}
  // the result of the next `count` hypotheses
  void take(const lsqr_score_result& r, uint64_t count) {
    dev_ms += r.score_ms;
    done += count;
    if (r.best_count > best.best_count) {  // strict '>' : RANSAC.hxx:100
      best = r;
      if (best.best_count == n) perfect = true;   // :104-105
      else num_tries = tries_after(best.best_count, n, K, numerator, all_tries);  // :107-110
    }
  }
};

// Rounds of `round`, 4x, 16x ... (up to 1 Mi) Philox hypotheses until the stop rule or a perfect hypothesis ends the loop; a
// typical problem (inlier ratio ~0.5, k = 3: 65 tries) ends after the first, small round of 256.
int ransac_rounds(lsqr_ctx* ctx, int precision, uint64_t seed, uint64_t round, RansacRounds& st) {
  while (!st.perfect && st.done < st.num_tries) {
    lsqr_score_args a{};
    a.sampler = LSQR_SAMPLE_PHILOX; a.precision = precision; a.seed = seed; a.first = st.done;
    a.count = std::min<uint64_t>(round, st.num_tries - st.done);
    lsqr_score_result r{};
    if (int rc = score_impl(ctx, &a, &r)) return rc;
    st.take(r, a.count);
    round = std::min<uint64_t>(round * 4, (uint64_t)1 << 20);
  }
  return LSQR_OK;
}

int ransac_impl(lsqr_ctx* ctx, double prob, int precision, uint64_t seed, uint8_t* out_mask, lsqr_compute_result* res) {
  if (ctx->model < 0 || !ctx->main.soa64) return fail(ctx, LSQR_ERR_STATE, "set the estimator and upload data first");
  memset(res, 0, sizeof(*res));
  const ModelInfo mi = model_info(ctx->model);
  const uint32_t n = ctx->main.n;
  // RANSAC.hxx:16-19: fewer data than the minimal subset, or probability outside (0,1) -> return 0
  if (n < (uint32_t)mi.K || prob >= 1.0 || prob <= 0.0) return LSQR_OK;
  RansacRounds st(n, mi.K, prob);
  if (int rc = ransac_rounds(ctx, precision, seed, 256, st)) return rc;
  return finish_ransac(ctx, st.best, st.done, st.dev_ms, out_mask, res);
}

int ransac_exhaustive_impl(lsqr_ctx* ctx, int precision, uint8_t* out_mask, lsqr_compute_result* res) {
  if (ctx->model < 0 || !ctx->main.soa64) return fail(ctx, LSQR_ERR_STATE, "set the estimator and upload data first");
  memset(res, 0, sizeof(*res));
  const ModelInfo mi = model_info(ctx->model);
  const uint32_t n = ctx->main.n;
  if (n < (uint32_t)mi.K) return LSQR_OK;  // RANSAC.hxx:168-169
  const uint64_t total = choose_exact(n, mi.K);
  if (total > 0xFFFFFFFEull) return fail(ctx, LSQR_ERR_ARG, "C(N,k) exceeds 2^32-2: the brute-force overload is for small problems (RANSAC.h:107-109)");
  lsqr_score_args a{};
  a.sampler = LSQR_SAMPLE_EXHAUSTIVE; a.precision = precision; a.first = 0; a.count = total;
  lsqr_score_result r{};
  if (int rc = score_impl(ctx, &a, &r)) return rc;
  return finish_ransac(ctx, r, total, r.score_ms, out_mask, res);
}

// RANSAC<T,S>::compute with the data still on the host: lsqr_upload + lsqr_ransac in one pass, same results bit for bit.  The
// minimal subsets of the first round (256 hypotheses, drawn on the host with the device's sampler) are fetched from the caller's
// buffer first, solved at once, and every range of the data is scored against them as soon as it has been transposed, so
// that when the last chunk lands only that chunk is left to score.
int compute_impl(lsqr_ctx* ctx, const void* aos, size_t n, size_t stride, double prob, int precision, uint64_t seed, uint8_t* out_mask, lsqr_compute_result* res) {
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called first");
  memset(res, 0, sizeof(*res));
  const ModelInfo mi = model_info(ctx->model);
  // RANSAC.hxx:16-19: fewer data than the minimal subset, or probability outside (0,1) -> return 0 (nothing is touched)
  if (n < (size_t)mi.K || prob >= 1.0 || prob <= 0.0) return LSQR_OK;
  if (n > 0xFFFFFFF0ull) return fail(ctx, LSQR_ERR_ARG, "too many data records");
  if (!aos) return fail(ctx, LSQR_ERR_ARG, "null data pointer");
  if (stride < sizeof(double) * mi.D || (stride % sizeof(double)) != 0) return fail(ctx, LSQR_ERR_ARG, "stride must be a multiple of 8 and >= 8*dim");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  const uint32_t N = (uint32_t)n;
  RansacRounds st(N, mi.K, prob);
  const uint64_t H0 = std::min<uint64_t>(256, st.all_tries);      // the first round of lsqr_ransac
  const uint64_t lo = H0 * (uint64_t)ctx->rank / (uint64_t)ctx->world, hi = H0 * (uint64_t)(ctx->rank + 1) / (uint64_t)ctx->world;
  const uint32_t B = (uint32_t)(hi - lo);
  // subsets of the whole round (every rank keeps the list: the winner is re-derived from it), records of this rank's share
  std::vector<int32_t> subs((size_t)H0 * mi.K);
#define CALL(MM) for (uint64_t h = 0; h < H0; h++) sample_subset<Model<MM>::K>(h, seed, N, &subs[h * mi.K])
  LSQR_DISPATCH_MODEL(ctx->model, CALL)
#undef CALL
  if (int rc = ensure_hyp(ctx, std::max<uint32_t>(B, 1))) return rc;
  if (int rc = ensure(ctx, &ctx->list_dev, &ctx->list_cap, (size_t)H0 * mi.K)) return rc;
  const size_t gbytes = (size_t)std::max<uint32_t>(B, 1) * mi.K * stride;
  if (int rc = ensure(ctx, &ctx->gather_dev, &ctx->gather_cap, gbytes)) return rc;
  if (int rc = ensure_pinned(ctx, &ctx->gather_pin, &ctx->gather_pin_cap, gbytes + sizeof(int32_t) * H0 * mi.K)) return rc;
  const unsigned char* host = static_cast<const unsigned char*>(aos);
  for (uint32_t h = 0; h < B; h++)
    for (int j = 0; j < mi.K; j++) memcpy(ctx->gather_pin + ((size_t)h * mi.K + j) * stride, host + (size_t)subs[(lo + h) * mi.K + j] * stride, sizeof(double) * mi.D);
  memcpy(ctx->gather_pin + gbytes, subs.data(), sizeof(int32_t) * H0 * mi.K);
  CK(cudaMemsetAsync(ctx->key_dev, 0, 2 * sizeof(unsigned long long), s));
  CK(cudaEventRecord(ctx->ev[0], s));
  CK(cudaMemcpyAsync(ctx->gather_dev, ctx->gather_pin, gbytes, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(ctx->list_dev, ctx->gather_pin + gbytes, sizeof(int32_t) * H0 * mi.K, cudaMemcpyHostToDevice, s));
  SolveArgs sa{};
  sa.model = ctx->model; sa.sampler = LSQR_SAMPLE_LIST; sa.seed = seed; sa.first = lo; sa.H = B; sa.hld = ctx->hcap;
  sa.subsets = ctx->subsets; sa.hyp64 = ctx->hyp64; sa.n_valid = reinterpret_cast<uint32_t*>(ctx->key_dev + 1);
  sa.list = ctx->list_dev + lo * mi.K; sa.gathered = ctx->gather_dev; sa.gathered_stride = stride;
  DataSet& ds = ctx->main;
  const RoundFn score_range = [&](size_t r_lo, size_t r_hi, bool first, bool last) -> int {
    if (B == 0) return 0;
    if (first) {   // the centre is known now: hypotheses (from the fetched records) and their fp32 constants
      DataView dv = ds.view();
      dv.n = N;
      launch_solve(sa, dv, ctx->cfg, s); ctx->launches++;
      if (precision == LSQR_FP32) { launch_hoist32(ctx->model, ctx->hyp64, ctx->hcap, B, dv, ctx->cfg, ctx->hyp32, s); ctx->launches++; }
      CK(cudaMemsetAsync(ctx->counts, 0, sizeof(uint32_t) * B, s));
    }
    if (r_hi > r_lo) ctx->launches += launch_consensus(ctx->model, precision, ds.range(r_lo, r_hi, last), ctx->hyp64, ctx->hyp32, ctx->hcap, B, ctx->cfg, ctx->counts, ctx->num_sms, s);
    return 0;
  };
  if (int rc = upload_to(ctx, ds, aos, n, stride, false, &score_range)) return rc;
  const DataView dv = ds.view();
  if (B) { launch_argmax(ctx->counts, B, (uint32_t)lo, ctx->key_dev, s); ctx->launches++; }
  if (int rc = comm_max_u64(ctx, ctx->key_dev)) return rc;
  SolveArgs wa{};
  wa.model = ctx->model; wa.sampler = LSQR_SAMPLE_LIST; wa.seed = seed; wa.first = 0; wa.list = ctx->list_dev;
  launch_winner(wa, ctx->key_dev, dv, ctx->cfg, ctx->winner_dev, s); ctx->launches++;
  CK(cudaEventRecord(ctx->ev[1], s));
  CKL();
  CK(cudaMemcpyAsync(ctx->winner_pin, ctx->winner_dev, sizeof(WinnerRecord), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  float ms0 = 0.f;
  CK(cudaEventElapsedTime(&ms0, ctx->ev[0], ctx->ev[1]));
  lsqr_score_result r0{};
  decode_winner(*ctx->winner_pin, 0, mi, &r0);
  r0.score_ms = ms0;   // includes the upload it overlaps
  st.take(r0, H0);
  if (int rc = ransac_rounds(ctx, precision, seed, 1024, st)) return rc;
  return finish_ransac(ctx, st.best, st.done, st.dev_ms, out_mask, res);
}

// Routing of problems [p0, p1) of a batch call, from the host offsets alone.  A problem that fits one block takes batch_kernel
// (max_n is taken over those problems only); a larger one a cluster of C CTAs, the smallest that holds it.  cl[k] lists the
// problems (relative to p0) of cluster size 2 << k, cl_slice[k] the largest slice among them; cl_all is cl[0..3] back to back,
// the list the cluster launches read on the device.
struct BatchPlan {
  BatchLimits L;
  bool use32;                // fp32 scoring keeps an fp32 copy of the points next to the fp64 one
  uint32_t max_n = 1;
  std::vector<uint32_t> cl[4];
  uint32_t cl_slice[4] = {0, 0, 0, 0};
  std::vector<uint32_t> cl_all;
};
int plan_batch(lsqr_ctx* ctx, const uint64_t* offsets, uint64_t p0, uint64_t p1, int exhaustive, int precision, BatchPlan* plan) {
  CK(cudaSetDevice(ctx->device));
  BatchPlan& P = *plan;
  P.use32 = precision == LSQR_FP32 && !exhaustive;
  const BatchLimits L = P.L = batch_limits(ctx->model, P.use32 ? 1 : 0, exhaustive);
  for (uint64_t b = p0; b < p1; b++) {
    if (offsets[b + 1] < offsets[b]) return fail(ctx, LSQR_ERR_ARG, "offsets must be non-decreasing");
    const uint64_t nb = offsets[b + 1] - offsets[b];
    if (nb <= L.one_block) { P.max_n = std::max<uint64_t>(P.max_n, nb); continue; }
    if (L.max_cluster == 0) return fail(ctx, LSQR_ERR_ARG, "a problem does not fit in shared memory; use lsqr_ransac for large problems");
    if (nb > L.max_records)
      return fail(ctx, LSQR_ERR_ARG, "a problem of " + std::to_string(nb) + " records exceeds the batch limit of " + std::to_string(L.max_records) +
                                         " records for this model and precision; use lsqr_compute for larger problems");
    const uint32_t c = batch_cluster_size(L, nb);
    const int k = c == 2 ? 0 : c == 4 ? 1 : c == 8 ? 2 : 3;
    P.cl[k].push_back((uint32_t)(b - p0));
    P.cl_slice[k] = std::max<uint32_t>(P.cl_slice[k], (uint32_t)(((nb + c - 1) / c + 1) & ~1ull));
  }
  for (const auto& v : P.cl) P.cl_all.insert(P.cl_all.end(), v.begin(), v.end());
  return LSQR_OK;
}

// The plan's large problems: one cluster launch per cluster size.  `ba` locates the data, offsets and outputs of the whole
// call; cl_dev holds plan.cl_all on the device.  With `tev`, each launch is bracketed by a pair of timing events appended to it
// (all of them destroyed if a launch fails).
int launch_clusters(lsqr_ctx* ctx, const BatchPlan& plan, BatchArgs ba, const uint32_t* cl_dev, cudaStream_t s, std::vector<cudaEvent_t>* tev) {
  size_t first = 0;
  for (int k = 0; k < 4; k++) {
    if (plan.cl[k].empty()) continue;
    ba.n_problems = (uint32_t)plan.cl[k].size();
    cudaEvent_t e0, e1;
    if (tev) {
      CK(cudaEventCreate(&e0)); tev->push_back(e0);
      CK(cudaEventCreate(&e1)); tev->push_back(e1);
      CK(cudaEventRecord(e0, s));
    }
    if (launch_batch_cluster(ba, cl_dev + first, ba.n_problems, 2u << k, plan.cl_slice[k], ctx->cfg, ctx->ls_type, s) < 0) {
      if (tev) for (cudaEvent_t e : *tev) cudaEventDestroy(e);
      return fail(ctx, LSQR_ERR_CUDA, std::string("batch cluster launch: ") + cudaGetErrorString(cudaGetLastError()));
    }
    ctx->launches++;
    if (tev) CK(cudaEventRecord(e1, s));
    first += plan.cl[k].size();
  }
  return LSQR_OK;
}

// problems [p0, p1) of a batch (offsets are absolute record offsets into `data`)
int batch_impl(lsqr_ctx* ctx, const double* data, const uint64_t* offsets, uint64_t p0, uint64_t p1, int exhaustive, double prob, uint32_t max_tries,
               uint64_t seed, int precision, double* out_params, uint32_t* out_counts, uint8_t* out_masks, double* device_ms) {
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called first");
  if (device_ms) *device_ms = 0.0;
  if (p1 <= p0) return LSQR_OK;
  const uint64_t np = p1 - p0;
  if (np > 0x7FFFFFFFull) return fail(ctx, LSQR_ERR_ARG, "too many problems");
  const ModelInfo mi = model_info(ctx->model);
  BatchPlan plan;
  if (int rc = plan_batch(ctx, offsets, p0, p1, exhaustive, precision, &plan)) return rc;
  const uint64_t base = offsets[p0], total = offsets[p1] - base;
  cudaStream_t s = ctx->stream;
  // persistent buffers (a cudaMalloc/cudaFree set per call cost more than the kernel)
  if (int rc = ensure(ctx, &ctx->bt_data, &ctx->bt_data_cap, (size_t)std::max<uint64_t>(total, 1) * mi.D)) return rc;
  if (int rc = ensure(ctx, &ctx->bt_off, &ctx->bt_off_cap, (size_t)np + 1)) return rc;
  if (int rc = ensure(ctx, &ctx->bt_prm, &ctx->bt_prm_cap, (size_t)np * mi.P)) return rc;
  if (int rc = ensure(ctx, &ctx->bt_cnt, &ctx->bt_cnt_cap, (size_t)np)) return rc;
  if (out_masks) if (int rc = ensure(ctx, &ctx->mask_dev, &ctx->mask_dev_cap, (size_t)std::max<uint64_t>(total, 1))) return rc;
  ctx->main.bytes_valid = false;   // mask_dev is shared with the consensus-set bytes
  CK(cudaMemcpyAsync(ctx->bt_off, offsets + p0, sizeof(uint64_t) * (np + 1), cudaMemcpyHostToDevice, s));
  // The problems go up in chunks of whole problems (~16 MB from page-locked memory, ~4 MB through the pinned staging ring from
  // pageable memory, as lsqr_upload does) on the copy stream; each chunk's problems are solved as soon as it has landed, so the
  // kernel hides behind the copy of the chunks that follow (65 536 x 256 3-D points: 403 MB of upload against 2.3 ms of kernel).
  const size_t rec_bytes = (size_t)mi.D * sizeof(double);
  StagedCopy up{ctx, is_pinned(data + base * mi.D)};
  const uint64_t chunk_rec = std::max<uint64_t>((up.pinned ? (16u << 20) : (4u << 20)) / rec_bytes, 1);
  if (int rc = up.start((size_t)chunk_rec * rec_bytes)) return rc;
  std::vector<cudaEvent_t> tev;                      // kernel time = sum over the chunks' launches
  // copies go in pieces of chunk_rec records; a launch covers the problems of ~32 MB of them (several thousand small problems:
  // enough thread blocks to fill the GPU -- launches of one copy piece each, ~650 blocks, tripled the kernel time)
  const uint64_t launch_rec = std::max<uint64_t>(chunk_rec, (32u << 20) / rec_bytes);
  for (uint64_t q0 = p0; q0 < p1;) {
    uint64_t q1 = q0 + 1;
    while (q1 < p1 && offsets[q1 + 1] - offsets[q0] <= launch_rec) q1++;
    const uint64_t rec0 = offsets[q0] - base, nrec = offsets[q1] - offsets[q0];
    for (uint64_t c0 = 0; c0 < nrec; c0 += chunk_rec) {
      const uint64_t cn = std::min<uint64_t>(chunk_rec, nrec - c0);
      if (int rc = up.put(ctx->bt_data + (rec0 + c0) * mi.D, data + (offsets[q0] + c0) * mi.D, cn * rec_bytes)) return rc;
    }
    if (nrec) if (int rc = up.landed()) return rc;
    bool any_small = false;
    for (uint64_t b = q0; b < q1 && !any_small; b++) any_small = offsets[b + 1] - offsets[b] <= plan.L.one_block;
    if (!any_small) { q0 = q1; continue; }   // every problem of this piece takes the cluster path
    BatchArgs ba{};
    ba.model = ctx->model; ba.exhaustive = exhaustive; ba.precision = plan.use32 ? 1 : 0; ba.tries = max_tries; ba.prob = prob; ba.seed = seed;
    ba.data = ctx->bt_data + rec0 * mi.D; ba.offsets = ctx->bt_off + (q0 - p0); ba.n_problems = (uint32_t)(q1 - q0); ba.max_n = plan.max_n;
    ba.base = offsets[q0]; ba.first_problem = q0;
    ba.out_params = ctx->bt_prm + (q0 - p0) * mi.P; ba.out_counts = ctx->bt_cnt + (q0 - p0); ba.out_masks = out_masks ? ctx->mask_dev + rec0 : nullptr;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); tev.push_back(e0);
    CK(cudaEventCreate(&e1)); tev.push_back(e1);
    CK(cudaEventRecord(e0, s));
    if (launch_batch(ba, ctx->cfg, ctx->ls_type, s) < 0) { for (cudaEvent_t e : tev) cudaEventDestroy(e); return fail(ctx, LSQR_ERR_ARG, "batch launch rejected"); }
    ctx->launches++;
    CK(cudaEventRecord(e1, s));
    q0 = q1;
  }
  // the large problems, once every piece has landed
  if (!plan.cl_all.empty()) {
    if (int rc = ensure(ctx, &ctx->bt_cl, &ctx->bt_cl_cap, plan.cl_all.size())) return rc;
    CK(cudaMemcpyAsync(ctx->bt_cl, plan.cl_all.data(), sizeof(uint32_t) * plan.cl_all.size(), cudaMemcpyHostToDevice, s));
    BatchArgs ba{};
    ba.model = ctx->model; ba.precision = plan.use32 ? 1 : 0; ba.tries = max_tries; ba.prob = prob; ba.seed = seed;
    ba.data = ctx->bt_data; ba.offsets = ctx->bt_off; ba.base = base; ba.first_problem = p0;
    ba.out_params = ctx->bt_prm; ba.out_counts = ctx->bt_cnt; ba.out_masks = out_masks ? ctx->mask_dev : nullptr;
    if (int rc = launch_clusters(ctx, plan, ba, ctx->bt_cl, s, &tev)) return rc;
  }
  CKL();
  CK(cudaMemcpyAsync(out_params + p0 * mi.P, ctx->bt_prm, sizeof(double) * np * mi.P, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(out_counts + p0, ctx->bt_cnt, sizeof(uint32_t) * np, cudaMemcpyDeviceToHost, s));
  if (out_masks && total) CK(cudaMemcpyAsync(out_masks + base, ctx->mask_dev, total, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  double total_ms = 0.0;
  for (size_t i = 0; i + 1 < tev.size(); i += 2) { float ms = 0.f; if (cudaEventElapsedTime(&ms, tev[i], tev[i + 1]) == cudaSuccess) total_ms += ms; }
  for (cudaEvent_t e : tev) cudaEventDestroy(e);
  if (device_ms) *device_ms = total_ms;
  return LSQR_OK;
}

// `p` is memory of this context's device (not page-locked or pageable host memory, not managed memory, not another GPU's),
// aligned to `align` bytes
int check_device_ptr(lsqr_ctx* ctx, const void* p, size_t align, const char* name) {
  cudaPointerAttributes attr{};
  const bool ok = p && cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeDevice && attr.device == ctx->device;
  if (!ok) cudaGetLastError();   // a refused query is an answer here, not an error of the next call
  if (!ok) return fail(ctx, LSQR_ERR_ARG, std::string(name) + " is not device memory of device " + std::to_string(ctx->device));
  if (reinterpret_cast<uintptr_t>(p) % align) return fail(ctx, LSQR_ERR_ARG, std::string(name) + " is not aligned to " + std::to_string(align) + " bytes");
  return LSQR_OK;
}

// The device entry points: `enqueue(s)` on the caller's stream (the context's when cuda_stream is null).  bt_off, bt_cl and the
// page-locked slots are shared with every other call on the context: work on another stream is ordered after the context's
// stream at entry, and the context's stream after it at exit (also when enqueueing failed half-way).
template <class Enqueue> int on_caller_stream(lsqr_ctx* ctx, void* cuda_stream, const Enqueue& enqueue) {
  cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
  const bool side = s != ctx->stream;
  if (side) {
    CK(cudaEventRecord(ctx->bd_order[0], ctx->stream));
    CK(cudaStreamWaitEvent(s, ctx->bd_order[0], 0));
  }
  const int rc = enqueue(s);
  if (side) {
    CK(cudaEventRecord(ctx->bd_order[1], s));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->bd_order[1], 0));
  }
  return rc;
}

// The host offsets (np + 1) -> bt_off and the problem list -> bt_cl on stream s, through one of the two page-locked slots (a copy
// from pageable memory may wait for the stream).  The slot's previous copies belong to the call before last: this waits only
// while that call's copies are still queued.  Growing the device buffers may synchronise the device (cudaFree); the sizes of one
// call repeated do not grow them.
int stage_offsets(lsqr_ctx* ctx, const uint64_t* offsets, uint64_t np, const std::vector<uint32_t>& list, cudaStream_t s) {
  if (int rc = ensure(ctx, &ctx->bt_off, &ctx->bt_off_cap, (size_t)np + 1)) return rc;
  if (!list.empty()) if (int rc = ensure(ctx, &ctx->bt_cl, &ctx->bt_cl_cap, list.size())) return rc;
  const int slot = (int)(ctx->bd_calls++ & 1);
  CK(cudaEventSynchronize(ctx->bd_ev[slot]));
  const size_t off_bytes = sizeof(uint64_t) * (np + 1), cl_bytes = sizeof(uint32_t) * list.size();
  if (int rc = ensure_pinned(ctx, &ctx->bd_pin[slot], &ctx->bd_pin_cap[slot], off_bytes + cl_bytes)) return rc;
  memcpy(ctx->bd_pin[slot], offsets, off_bytes);
  if (cl_bytes) memcpy(ctx->bd_pin[slot] + off_bytes, list.data(), cl_bytes);
  CK(cudaMemcpyAsync(ctx->bt_off, ctx->bd_pin[slot], off_bytes, cudaMemcpyHostToDevice, s));
  if (cl_bytes) CK(cudaMemcpyAsync(ctx->bt_cl, ctx->bd_pin[slot] + off_bytes, cl_bytes, cudaMemcpyHostToDevice, s));
  CK(cudaEventRecord(ctx->bd_ev[slot], s));
  return LSQR_OK;
}

// lsqr_ransac_batch_device on stream s, which the caller has ordered after the context's stream.  All one-block problems go in
// one batch_kernel launch: there is no copy for smaller launches to hide behind.
int batch_device_enqueue(lsqr_ctx* ctx, const BatchPlan& plan, const double* dev_data, const uint64_t* offsets, uint64_t np, int exhaustive,
                         double prob, uint32_t max_tries, uint64_t seed, double* dev_params, uint32_t* dev_counts, uint8_t* dev_masks,
                         cudaStream_t s) {
  const ModelInfo mi = model_info(ctx->model);
  if (int rc = stage_offsets(ctx, offsets, np, plan.cl_all, s)) return rc;
  const uint64_t base = offsets[0];
  BatchArgs ba{};
  ba.model = ctx->model; ba.exhaustive = exhaustive; ba.precision = plan.use32 ? 1 : 0; ba.tries = max_tries; ba.prob = prob; ba.seed = seed;
  ba.data = dev_data + base * mi.D; ba.offsets = ctx->bt_off; ba.base = base; ba.first_problem = 0; ba.max_n = plan.max_n;
  ba.out_params = dev_params; ba.out_counts = dev_counts; ba.out_masks = dev_masks ? dev_masks + base : nullptr;
  if (plan.cl_all.size() < np) {   // some problem fits one block (batch_kernel returns at once for the others)
    ba.n_problems = (uint32_t)np;
    if (launch_batch(ba, ctx->cfg, ctx->ls_type, s) < 0) return fail(ctx, LSQR_ERR_ARG, "batch launch rejected");
    ctx->launches++;
  }
  if (int rc = launch_clusters(ctx, plan, ba, ctx->bt_cl, s, nullptr)) return rc;
  CKL();
  return LSQR_OK;
}

int create_single(lsqr_ctx** out, int device) {
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) return LSQR_ERR_CUDA;
  lsqr_ctx* ctx = new lsqr_ctx();
  ctx->device = device;
  auto bail = [&](int code) { lsqr_ctx_destroy(ctx); return code; };
  if (cudaSetDevice(device) != cudaSuccess) return bail(LSQR_ERR_CUDA);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(LSQR_ERR_CUDA);
  if (prop.major < 10) { fprintf(stderr, "lsqr_b200: device %d is sm_%d%d; this library is built for sm_100a only\n", device, prop.major, prop.minor); return bail(LSQR_ERR_CUDA); }
  ctx->num_sms = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(LSQR_ERR_CUDA);
  ctx->own_stream = true;
  if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(LSQR_ERR_CUDA);
  ctx->rb.blocks = ctx->num_sms * mask_moments_ctas_per_sm();   // one wave of resident CTAs
  bool ok = cudaMalloc((void**)&ctx->key_dev, 4 * sizeof(unsigned long long)) == cudaSuccess &&
            cudaMalloc((void**)&ctx->winner_dev, sizeof(WinnerRecord)) == cudaSuccess &&
            cudaMalloc((void**)&ctx->small_dev, kSmall * sizeof(double)) == cudaSuccess &&
            cudaMalloc((void**)&ctx->rb.partials, sizeof(double) * kMaxMoments * ctx->rb.blocks) == cudaSuccess &&
            cudaMalloc((void**)&ctx->rb.moments, sizeof(double) * kMaxMoments) == cudaSuccess &&
            cudaMallocHost((void**)&ctx->pin, 64 * sizeof(double) + sizeof(WinnerRecord)) == cudaSuccess;
  if (ok) ctx->winner_pin = reinterpret_cast<WinnerRecord*>(ctx->pin + 64);
  for (int i = 0; ok && i < 6; i++) ok = cudaEventCreate(&ctx->ev[i]) == cudaSuccess;
  for (int i = 0; ok && i < lsqr_ctx::kRing; i++) ok = cudaEventCreateWithFlags(&ctx->up_ev[i], cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; ok && i < 8; i++) ok = cudaEventCreateWithFlags(&ctx->up_land[i], cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; ok && i < 2; i++) ok = cudaEventCreateWithFlags(&ctx->bd_ev[i], cudaEventDisableTiming) == cudaSuccess &&
                                         cudaEventCreateWithFlags(&ctx->bd_order[i], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) return bail(LSQR_ERR_CUDA);
  *out = ctx;
  return LSQR_OK;
}

// runs fn on every member of a group concurrently (one worker thread per device)
int group_run(lsqr_ctx* g, const std::function<int(lsqr_ctx*, int)>& fn) {
  Group* grp = g->group;
  const int rc = grp->workers->run([&](int r) { return fn(grp->kids[r], r); });
  if (rc) for (lsqr_ctx* k : grp->kids) if (!k->err.empty()) { g->err = k->err; break; }
  return rc;
}

}  // namespace

extern "C" {

int lsqr_model_plane(unsigned d) { return d == 3 ? LSQR_PLANE3 : d == 4 ? LSQR_PLANE4 : d == 2 ? LSQR_PLANE2 : (d >= 5 && d <= 8) ? (int)(LSQR_PLANE5 + d - 5) : -1; }
int lsqr_model_sphere(unsigned d) { return d == 2 ? LSQR_CIRCLE2 : d == 3 ? LSQR_SPHERE3 : d == 4 ? LSQR_SPHERE4 : (d >= 5 && d <= 8) ? (int)(LSQR_SPHERE5 + d - 5) : -1; }
int lsqr_model_line(unsigned d) { return d == 2 ? LSQR_LINE2 : d == 3 ? LSQR_LINE3 : (d >= 4 && d <= 8) ? (int)(LSQR_LINE4 + d - 4) : -1; }
int lsqr_model_dense(unsigned n) { return n == 5 ? LSQR_DENSE5 : n == 6 ? LSQR_DENSE6 : (n >= 2 && n <= 4) ? (int)(LSQR_DENSE2 + n - 2) : (n == 7 || n == 8) ? (int)(LSQR_DENSE7 + n - 7) : -1; }
int lsqr_model_info(int model, int* dim, int* nparams, int* k) {
  if (model < 0 || model >= LSQR_NUM_MODELS) return LSQR_ERR_ARG;
  const ModelInfo mi = model_info(model);
  if (dim) *dim = mi.D;
  if (nparams) *nparams = mi.P;
  if (k) *k = mi.K;
  return LSQR_OK;
}

int lsqr_device_count(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return 0; }
  return count;
}

int lsqr_ctx_create(lsqr_ctx** out, int device) {
  if (!out) return LSQR_ERR_ARG;
  return create_single(out, device);
}

int lsqr_ctx_create_multi(lsqr_ctx** out, int ngpus) {
  if (!out) return LSQR_ERR_ARG;
  *out = nullptr;
  const int count = lsqr_device_count();
  if (count == 0) return LSQR_ERR_CUDA;
  if (ngpus <= 0) ngpus = count;
  if (ngpus > count) return LSQR_ERR_ARG;
  if (ngpus == 1) return create_single(out, 0);
  if (!nccl().ok) return LSQR_ERR_COMM;
  lsqr_ctx* g = new lsqr_ctx();
  g->group = new Group();
  g->world = ngpus;
  auto bail = [&](int code) { lsqr_ctx_destroy(g); return code; };
  std::vector<int> devs(ngpus);
  for (int r = 0; r < ngpus; r++) {
    devs[r] = r;
    lsqr_ctx* k = nullptr;
    if (int rc = create_single(&k, r)) return bail(rc);
    k->rank = r; k->world = ngpus;
    g->group->kids.push_back(k);
  }
  std::vector<ncclComm_t> comms(ngpus);
  if (nccl().CommInitAll(comms.data(), ngpus, devs.data()) != ncclSuccess) return bail(LSQR_ERR_COMM);
  for (int r = 0; r < ngpus; r++) g->group->kids[r]->comm = comms[r];
  g->group->workers.reset(new Workers(ngpus));
  g->group->workers->run([&](int r) { return cudaSetDevice(g->group->kids[r]->device) == cudaSuccess ? 0 : LSQR_ERR_CUDA; });
  *out = g;
  return LSQR_OK;
}

int lsqr_ctx_world(const lsqr_ctx* ctx) { return ctx ? ctx->world : 0; }

int lsqr_nccl_unique_id(void* out_id, size_t bytes) {
  if (!out_id || bytes < sizeof(ncclUniqueId)) return LSQR_ERR_ARG;
  if (!nccl().ok) return LSQR_ERR_COMM;
  ncclUniqueId id;
  if (nccl().GetUniqueId(&id) != ncclSuccess) return LSQR_ERR_COMM;
  memcpy(out_id, &id, sizeof(id));
  return LSQR_OK;
}

int lsqr_ctx_init_nccl(lsqr_ctx* ctx, const void* id_bytes, size_t bytes, int rank, int world) {
  if (!ctx || !id_bytes || bytes < sizeof(ncclUniqueId)) return LSQR_ERR_ARG;
  if (ctx->group) return fail(ctx, LSQR_ERR_ARG, "a multi-GPU group owns its communicators");
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, LSQR_ERR_ARG, "bad rank/world");
  if (!nccl().ok) return fail(ctx, LSQR_ERR_COMM, "libnccl.so.2 not found");
  CK(cudaSetDevice(ctx->device));
  if (ctx->comm) { nccl().CommDestroy(ctx->comm); ctx->comm = nullptr; }
  ncclUniqueId id;
  memcpy(&id, id_bytes, sizeof(id));
  if (world > 1) CKN(nccl().CommInitRank(&ctx->comm, world, id, rank));
  ctx->rank = rank; ctx->world = world; ctx->max_fn = nullptr; ctx->sum_fn = nullptr;
  return LSQR_OK;
}

void lsqr_ctx_destroy(lsqr_ctx* ctx) {
  if (!ctx) return;
  if (ctx->group) {
    ctx->group->workers.reset();
    for (lsqr_ctx* k : ctx->group->kids) lsqr_ctx_destroy(k);
    delete ctx->group;
    delete ctx;
    return;
  }
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
  if (ctx->comm && nccl().ok) nccl().CommDestroy(ctx->comm);
  ctx->copier.reset();
  free_dataset(ctx->main); free_dataset(ctx->scratch);
  cudaFree(ctx->bt_data); cudaFree(ctx->bt_off); cudaFree(ctx->bt_prm); cudaFree(ctx->bt_cnt); cudaFree(ctx->bt_cl);
  cudaFree(ctx->weights_dev); cudaFree(ctx->mask_dev); if (ctx->mask_pin) cudaFreeHost(ctx->mask_pin); if (ctx->agree_pin) cudaFreeHost(ctx->agree_pin);
  cudaFree(ctx->gather_dev); if (ctx->gather_pin) cudaFreeHost(ctx->gather_pin);
  for (int i = 0; i < lsqr_ctx::kRing; i++) if (ctx->up_pin[i]) cudaFreeHost(ctx->up_pin[i]);
  cudaFree(ctx->staging); cudaFree(ctx->subsets); cudaFree(ctx->hyp64); cudaFree(ctx->hyp32); cudaFree(ctx->counts);
  cudaFree(ctx->hyp32b); cudaFree(ctx->live_counts); cudaFree(ctx->live_ids); cudaFree(ctx->prune_dev);
  cudaFree(ctx->list_dev); cudaFree(ctx->params_in_dev); cudaFree(ctx->key_dev); cudaFree(ctx->winner_dev); cudaFree(ctx->small_dev);
  cudaFree(ctx->rb.partials); cudaFree(ctx->rb.moments);
  if (ctx->pin) cudaFreeHost(ctx->pin);
  for (int i = 0; i < 6; i++) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  for (int i = 0; i < lsqr_ctx::kRing; i++) if (ctx->up_ev[i]) cudaEventDestroy(ctx->up_ev[i]);
  for (int i = 0; i < 8; i++) if (ctx->up_land[i]) cudaEventDestroy(ctx->up_land[i]);
  for (int i = 0; i < 2; i++) {
    if (ctx->bd_pin[i]) cudaFreeHost(ctx->bd_pin[i]);
    if (ctx->bd_ev[i]) cudaEventDestroy(ctx->bd_ev[i]);
    if (ctx->bd_order[i]) cudaEventDestroy(ctx->bd_order[i]);
  }
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* lsqr_last_error(const lsqr_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int lsqr_ctx_set_stream(lsqr_ctx* ctx, void* cuda_stream) {
  if (!ctx) return LSQR_ERR_ARG;
  if (ctx->group) return fail(ctx, LSQR_ERR_ARG, "a multi-GPU group runs on its own streams");
  if (ctx->own_stream && ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); }
  ctx->stream = (cudaStream_t)cuda_stream;
  ctx->own_stream = false;
  return LSQR_OK;
}

uint64_t lsqr_kernel_launches(const lsqr_ctx* ctx) {
  if (!ctx) return 0;
  if (ctx->group) { uint64_t t = 0; for (const lsqr_ctx* k : ctx->group->kids) t += k->launches; return t; }
  return ctx->launches;
}

int lsqr_set_estimator(lsqr_ctx* ctx, int model, double delta, double aux, int ls_type) {
  if (!ctx) return LSQR_ERR_ARG;
  if (model < 0 || model >= LSQR_NUM_MODELS) return fail(ctx, LSQR_ERR_ARG, "unknown model");
  if (ls_type != LSQR_LS_ALGEBRAIC && ls_type != LSQR_LS_GEOMETRIC) return fail(ctx, LSQR_ERR_ARG, "bad least-squares type");  // SphereParametersEstimator.hxx:17-18
  if (ctx->group) { ctx->model = model; return group_run(ctx, [&](lsqr_ctx* k, int) { return lsqr_set_estimator(k, model, delta, aux, ls_type); }); }
  if (ctx->model != model) {  // layouts differ between models: the data must be uploaded again
    cudaSetDevice(ctx->device);
    free_dataset(ctx->main); free_dataset(ctx->scratch);
  }
  ctx->model = model; ctx->delta = delta; ctx->aux = aux; ctx->ls_type = ls_type;
  // The reference keeps delta*delta for every estimator but the hypersphere, pivot and dense-system ones (e.g.
  // PlaneParametersEstimator.hxx:16 vs SphereParametersEstimator.hxx:20), so the sign of delta is immaterial there; the device
  // code that compares an unsquared residual (fp32 fast mode) gets |delta|.
  const bool distance_threshold = model_family(model) == FAM_SPHERE || model_family(model) == FAM_DENSE || model == LSQR_PIVOT;
  ctx->cfg.delta = distance_threshold ? delta : fabs(delta);
  ctx->cfg.delta2 = delta * delta;
  { unsigned long long b = 0; const double d2 = ctx->cfg.delta2; if (d2 == d2) memcpy(&b, &d2, sizeof(b)); ctx->cfg.delta2_bits = b; }   // below_delta2 (models.cuh)
  const double ang = aux > 0 ? aux : 0.017453292519943295769236907684886;  // RayIntersectionParametersEstimator.h:35
  double ce = sin(ang);
  ce *= ce;
  ctx->cfg.cross_eps = ce;
  ctx->main.moments_valid = false;
  return LSQR_OK;
}

int lsqr_upload(lsqr_ctx* ctx, const void* aos, size_t n, size_t stride_bytes) {
  if (!ctx) return LSQR_ERR_ARG;
  if (ctx->group) return group_run(ctx, [&](lsqr_ctx* k, int) { return upload_to(k, k->main, aos, n, stride_bytes, false); });
  return upload_to(ctx, ctx->main, aos, n, stride_bytes, false);
}
int lsqr_upload_device(lsqr_ctx* ctx, const double* dev_packed, size_t n) {
  if (!ctx) return LSQR_ERR_ARG;
  if (ctx->group) return fail(ctx, LSQR_ERR_ARG, "a device buffer belongs to one GPU; upload host memory to a multi-GPU group");
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called first");
  return upload_to(ctx, ctx->main, dev_packed, n, sizeof(double) * model_info(ctx->model).D, true);
}

int lsqr_set_shard(lsqr_ctx* ctx, int rank, int world, lsqr_allreduce_max_u64_fn max_fn, lsqr_allreduce_sum_f64_fn sum_fn, void* user) {
  if (!ctx) return LSQR_ERR_ARG;
  if (ctx->group) return fail(ctx, LSQR_ERR_ARG, "a multi-GPU group shards itself");
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, LSQR_ERR_ARG, "bad rank/world");
  if (world > 1 && (!max_fn || !sum_fn)) return fail(ctx, LSQR_ERR_ARG, "hooks required when world > 1");
  if (ctx->comm && nccl().ok) { nccl().CommDestroy(ctx->comm); ctx->comm = nullptr; }
  ctx->rank = rank; ctx->world = world; ctx->max_fn = max_fn; ctx->sum_fn = sum_fn; ctx->comm_user = user;
  return LSQR_OK;
}

int lsqr_score(lsqr_ctx* ctx, const lsqr_score_args* args, lsqr_score_result* res) {
  if (!ctx) return LSQR_ERR_ARG;
  if (ctx->group) {
    if (!args || !res) return fail(ctx, LSQR_ERR_ARG, "null argument");
    std::vector<lsqr_score_result> rs(ctx->world);
    const int rc = group_run(ctx, [&](lsqr_ctx* k, int r) { return score_impl(k, args, &rs[r]); });
    if (rc) return rc;
    *res = rs[0];
    uint32_t nv = 0;
    uint64_t ev = 0;
    for (const auto& r : rs) { nv += r.n_valid; ev += r.evals; res->score_ms = std::max(res->score_ms, r.score_ms); res->consensus_ms = std::max(res->consensus_ms, r.consensus_ms); }
    res->n_valid = nv; res->evals = ev;
    return LSQR_OK;
  }
  return score_impl(ctx, args, res);
}

int lsqr_consensus(lsqr_ctx* ctx, const double* params, uint32_t* out_count) {
  if (!ctx || !params) return LSQR_ERR_ARG;
  if (ctx->group) {
    std::vector<uint32_t> c(ctx->world, 0);
    const int rc = group_run(ctx, [&](lsqr_ctx* k, int r) { return consensus_impl(k, k->main, params, &c[r]); });
    if (!rc && out_count) *out_count = c[0];
    return rc;
  }
  return consensus_impl(ctx, ctx->main, params, out_count);
}
int lsqr_get_mask(lsqr_ctx* ctx, uint8_t* out_bytes) {
  if (!ctx) return LSQR_ERR_ARG;
  if (ctx->group) return group_run(ctx, [&](lsqr_ctx* k, int) { return get_mask_impl(k, k->main, out_bytes); });
  return get_mask_impl(ctx, ctx->main, out_bytes);
}
int lsqr_get_mask_bits(lsqr_ctx* ctx, uint32_t* out_words) {
  if (!ctx || !out_words) return LSQR_ERR_ARG;
  auto one = [&](lsqr_ctx* k) -> int {
    lsqr_ctx* ctx = k;   // for CK
    if (!k->main.mask_valid) return fail(k, LSQR_ERR_STATE, "no consensus set stored");
    uint32_t b, e;
    shard_range(k, k->main, &b, &e);
    if (e <= b) return LSQR_OK;
    CK(cudaSetDevice(k->device));
    const size_t w0 = b / 32, w1 = ((size_t)e + 31) / 32;
    CK(cudaMemcpyAsync(out_words + w0, k->main.maskbits + w0, sizeof(uint32_t) * (w1 - w0), cudaMemcpyDeviceToHost, k->stream));
    CK(cudaStreamSynchronize(k->stream));
    return LSQR_OK;
  };
  if (ctx->group) return group_run(ctx, [&](lsqr_ctx* k, int) { return one(k); });
  return one(ctx);
}
int lsqr_refine(lsqr_ctx* ctx, int use_mask, double* out_params, int* n_params) {
  if (!ctx) return LSQR_ERR_ARG;
  if (ctx->group) {
    std::vector<std::vector<double>> p(ctx->world, std::vector<double>(LSQR_MAX_PARAMS, 0.0));
    std::vector<int> np(ctx->world, 0);
    const int rc = group_run(ctx, [&](lsqr_ctx* k, int r) { return refine_impl(k, k->main, use_mask, p[r].data(), &np[r]); });
    if (rc) return rc;
    if (n_params) *n_params = np[0];
    if (out_params) for (int j = 0; j < np[0]; j++) out_params[j] = p[0][j];
    return LSQR_OK;
  }
  return refine_impl(ctx, ctx->main, use_mask, out_params, n_params);
}

int lsqr_ransac(lsqr_ctx* ctx, double prob, int precision, uint64_t seed, uint8_t* out_mask, lsqr_compute_result* res) {
  if (!ctx || !res) return LSQR_ERR_ARG;
  if (ctx->group) {
    std::vector<lsqr_compute_result> rs(ctx->world);
    const int rc = group_run(ctx, [&](lsqr_ctx* k, int r) { return ransac_impl(k, prob, precision, seed, out_mask, &rs[r]); });
    if (rc) return rc;
    *res = rs[0];
    for (const auto& r : rs) res->device_ms = std::max(res->device_ms, r.device_ms);
    return LSQR_OK;
  }
  return ransac_impl(ctx, prob, precision, seed, out_mask, res);
}

int lsqr_compute(lsqr_ctx* ctx, const void* aos, size_t n, size_t stride_bytes, double prob, int precision, uint64_t seed, uint8_t* out_mask,
                 lsqr_compute_result* res) {
  if (!ctx || !res) return LSQR_ERR_ARG;
  if (ctx->group) {
    std::vector<lsqr_compute_result> rs(ctx->world);
    const int rc = group_run(ctx, [&](lsqr_ctx* k, int r) { return compute_impl(k, aos, n, stride_bytes, prob, precision, seed, out_mask, &rs[r]); });
    if (rc) return rc;
    *res = rs[0];
    for (const auto& r : rs) res->device_ms = std::max(res->device_ms, r.device_ms);
    return LSQR_OK;
  }
  return compute_impl(ctx, aos, n, stride_bytes, prob, precision, seed, out_mask, res);
}

int lsqr_ransac_exhaustive(lsqr_ctx* ctx, int precision, uint8_t* out_mask, lsqr_compute_result* res) {
  if (!ctx || !res) return LSQR_ERR_ARG;
  if (ctx->group) {
    std::vector<lsqr_compute_result> rs(ctx->world);
    const int rc = group_run(ctx, [&](lsqr_ctx* k, int r) { return ransac_exhaustive_impl(k, precision, out_mask, &rs[r]); });
    if (rc) return rc;
    *res = rs[0];
    return LSQR_OK;
  }
  return ransac_exhaustive_impl(ctx, precision, out_mask, res);
}

int lsqr_ransac_batch(lsqr_ctx* ctx, const double* data, const uint64_t* offsets, uint64_t n_problems, int exhaustive, double prob,
                      uint32_t max_tries, uint64_t seed, int precision, double* out_params, uint32_t* out_counts, uint8_t* out_masks, double* device_ms) {
  if (!ctx || !data || !offsets || !out_params || !out_counts) return LSQR_ERR_ARG;
  if (precision != LSQR_FP64 && precision != LSQR_FP32) return fail(ctx, LSQR_ERR_ARG, "bad precision");
  if (n_problems == 0) return LSQR_OK;
  if (ctx->group) {   // independent problems: partitioned across the GPUs, no collective
    const int W = ctx->world;
    std::vector<double> ms(W, 0.0);
    const int rc = group_run(ctx, [&](lsqr_ctx* k, int r) {
      return batch_impl(k, data, offsets, n_problems * r / W, n_problems * (r + 1) / W, exhaustive, prob, max_tries, seed, precision, out_params, out_counts, out_masks, &ms[r]);
    });
    if (device_ms) *device_ms = *std::max_element(ms.begin(), ms.end());
    return rc;
  }
  return batch_impl(ctx, data, offsets, 0, n_problems, exhaustive, prob, max_tries, seed, precision, out_params, out_counts, out_masks, device_ms);
}

int lsqr_ransac_batch_device(lsqr_ctx* ctx, const double* dev_data, const uint64_t* offsets, uint64_t n_problems, int exhaustive, double prob,
                             uint32_t max_tries, uint64_t seed, int precision, double* dev_params, uint32_t* dev_counts, uint8_t* dev_masks,
                             void* cuda_stream) {
  if (!ctx || !offsets) return LSQR_ERR_ARG;
  if (ctx->group) return fail(ctx, LSQR_ERR_ARG, "a device buffer belongs to one GPU; a multi-GPU group takes host batches (lsqr_ransac_batch)");
  if (precision != LSQR_FP64 && precision != LSQR_FP32) return fail(ctx, LSQR_ERR_ARG, "bad precision");
  if (n_problems == 0) return LSQR_OK;
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called first");
  if (n_problems > 0x7FFFFFFFull) return fail(ctx, LSQR_ERR_ARG, "too many problems");
  BatchPlan plan;
  if (int rc = plan_batch(ctx, offsets, 0, n_problems, exhaustive, precision, &plan)) return rc;
  const bool records = offsets[n_problems] > offsets[0];   // data and masks are neither read nor written when every problem is empty
  if (records) if (int rc = check_device_ptr(ctx, dev_data, alignof(double), "dev_data")) return rc;
  if (int rc = check_device_ptr(ctx, dev_params, alignof(double), "dev_params")) return rc;
  if (int rc = check_device_ptr(ctx, dev_counts, alignof(uint32_t), "dev_counts")) return rc;
  if (dev_masks && records) if (int rc = check_device_ptr(ctx, dev_masks, 1, "dev_masks")) return rc;
  return on_caller_stream(ctx, cuda_stream, [&](cudaStream_t s) {
    return batch_device_enqueue(ctx, plan, dev_data, offsets, n_problems, exhaustive, prob, max_tries, seed, dev_params, dev_counts, dev_masks, s);
  });
}

int lsqr_least_squares_batch_device(lsqr_ctx* ctx, const double* dev_data, const uint64_t* offsets, uint64_t n_problems, const uint8_t* dev_masks,
                                    const double* dev_weights, double* dev_params, void* cuda_stream) {
  if (!ctx || !offsets) return LSQR_ERR_ARG;
  if (ctx->group) return fail(ctx, LSQR_ERR_ARG, "a device buffer belongs to one GPU; a multi-GPU group has no batched least squares");
  if (n_problems == 0) return LSQR_OK;
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called first");
  if (ctx->model == USXW || ctx->model == USCP) return fail(ctx, LSQR_ERR_ARG, "the ultrasound calibrations have no batched mode");
  if (dev_weights && ctx->model != ABSOR) return fail(ctx, LSQR_ERR_ARG, "dev_weights: weighted least squares exists for the absolute-orientation estimator only");
  if (n_problems > 0x7FFFFFFFull) return fail(ctx, LSQR_ERR_ARG, "too many problems");
  CK(cudaSetDevice(ctx->device));
  // route by size alone: the problems of cluster size 1 << k in by[k], then all of them back to back in `list`
  const int cmax = ls_batch_max_cluster(ctx->model, dev_weights != nullptr);
  std::vector<uint32_t> by[5], list;
  for (uint64_t b = 0; b < n_problems; b++) {
    if (offsets[b + 1] < offsets[b]) return fail(ctx, LSQR_ERR_ARG, "offsets must be non-decreasing");
    const uint64_t nb = offsets[b + 1] - offsets[b];
    if (nb > 0xFFFFFFFFull) return fail(ctx, LSQR_ERR_ARG, "a problem of " + std::to_string(nb) + " records exceeds the limit of 2^32 - 1 records");
    const uint32_t c = ls_batch_cluster(nb, cmax);
    by[c == 1 ? 0 : c == 2 ? 1 : c == 4 ? 2 : c == 8 ? 3 : 4].push_back((uint32_t)b);
  }
  for (const auto& v : by) list.insert(list.end(), v.begin(), v.end());
  const bool records = offsets[n_problems] > offsets[0];   // data, masks and weights are not read when every problem is empty
  if (records) if (int rc = check_device_ptr(ctx, dev_data, alignof(double), "dev_data")) return rc;
  if (int rc = check_device_ptr(ctx, dev_params, alignof(double), "dev_params")) return rc;
  if (dev_masks && records) if (int rc = check_device_ptr(ctx, dev_masks, 1, "dev_masks")) return rc;
  if (dev_weights && records) if (int rc = check_device_ptr(ctx, dev_weights, alignof(double), "dev_weights")) return rc;
  return on_caller_stream(ctx, cuda_stream, [&](cudaStream_t s) {
    if (int rc = stage_offsets(ctx, offsets, n_problems, list, s)) return rc;
    LsBatchArgs a{};
    a.model = ctx->model; a.data = dev_data; a.offsets = ctx->bt_off; a.masks = dev_masks; a.weights = dev_weights; a.out_params = dev_params;
    size_t first = 0;
    for (int k = 0; k < 5; k++) {
      if (by[k].empty()) continue;
      if (launch_ls_batch(a, ctx->bt_cl + first, (uint32_t)by[k].size(), 1u << k, ctx->ls_type, s) < 0)
        return fail(ctx, LSQR_ERR_CUDA, std::string("batched least-squares launch: ") + cudaGetErrorString(cudaGetLastError()));
      ctx->launches++;
      first += by[k].size();
    }
    CKL();
    return (int)LSQR_OK;
  });
}

int lsqr_batch_capacity(lsqr_ctx* ctx, int precision, int exhaustive, uint64_t* one_block, uint64_t* max_records) {
  if (!ctx || !one_block || !max_records) return LSQR_ERR_ARG;
  if (ctx->group) { lsqr_ctx* k = ctx->group->kids[0]; const int rc = lsqr_batch_capacity(k, precision, exhaustive, one_block, max_records); if (rc) ctx->err = k->err; return rc; }
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called first");
  if (precision != LSQR_FP64 && precision != LSQR_FP32) return fail(ctx, LSQR_ERR_ARG, "bad precision");
  if (ctx->model == USXW || ctx->model == USCP) return fail(ctx, LSQR_ERR_ARG, "the ultrasound calibrations have no batched mode");
  CK(cudaSetDevice(ctx->device));
  const BatchLimits L = batch_limits(ctx->model, precision == LSQR_FP32 ? 1 : 0, exhaustive);
  *one_block = L.one_block;
  *max_records = L.max_records;
  return LSQR_OK;
}

int lsqr_estimate(lsqr_ctx* ctx, const double* packed, size_t n, double* out_params, int* n_params) {
  if (!ctx || !packed || !out_params || !n_params) return LSQR_ERR_ARG;
  if (ctx->group) { lsqr_ctx* k = ctx->group->kids[0]; const int rc = lsqr_estimate(k, packed, n, out_params, n_params); if (rc) ctx->err = k->err; return rc; }
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called first");
  const ModelInfo mi = model_info(ctx->model);
  *n_params = 0;
  if (n < (size_t)mi.K) return LSQR_OK;  // e.g. PlaneParametersEstimator.hxx:45-46
  if ((ctx->model == USXW || ctx->model == USCP) && n != (size_t)mi.K) return LSQR_OK;  // SinglePointTargetUSCalibrationParametersEstimator.cxx:21-22, :674-675: exactly k
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  double* in_dev = ctx->small_dev + kSmEst;  // K*D <= 64 doubles
  CK(cudaMemcpyAsync(in_dev, packed, sizeof(double) * mi.K * mi.D, cudaMemcpyHostToDevice, s));
  launch_estimate_one(ctx->model, in_dev, ctx->cfg, ctx->small_dev + kSmOut, s); ctx->launches++;
  CKL();
  CK(cudaMemcpyAsync(ctx->pin, ctx->small_dev + kSmOut, sizeof(double) * (1 + LSQR_MAX_PARAMS), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  *n_params = (int)ctx->pin[0];
  for (int j = 0; j < *n_params; j++) out_params[j] = ctx->pin[1 + j];
  return LSQR_OK;
}

int lsqr_agree(lsqr_ctx* ctx, const double* params, const double* packed, size_t n, uint8_t* out) {
  if (!ctx || !params || !packed || !out) return LSQR_ERR_ARG;
  if (ctx->group) { lsqr_ctx* k = ctx->group->kids[0]; const int rc = lsqr_agree(k, params, packed, n, out); if (rc) ctx->err = k->err; return rc; }
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called first");
  if (n == 0) return LSQR_OK;
  if (n > 0xFFFFFFF0ull) return fail(ctx, LSQR_ERR_ARG, "too many data records");
  const ModelInfo mi = model_info(ctx->model);
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  if (n <= kAgreeZeroCopy) {
    // a handful of data (the reference's examples call agree() datum by datum): parameters and data go into a small page-locked
    // buffer that the kernel reads in place and answers into (unified addressing) -- one launch and one synchronisation, no copies
    if (!ctx->agree_pin) CK(cudaMallocHost((void**)&ctx->agree_pin, sizeof(double) * (LSQR_MAX_PARAMS + kAgreeZeroCopy * kMaxDim) + kAgreeZeroCopy));
    double* hp = ctx->agree_pin;
    uint8_t* ho = reinterpret_cast<uint8_t*>(hp + LSQR_MAX_PARAMS + kAgreeZeroCopy * kMaxDim);
    memcpy(hp, params, sizeof(double) * mi.P);
    memcpy(hp + LSQR_MAX_PARAMS, packed, sizeof(double) * n * mi.D);
    launch_agree_many(ctx->model, hp, hp + LSQR_MAX_PARAMS, (uint32_t)n, ctx->cfg, ho, s); ctx->launches++;
    CKL();
    CK(cudaStreamSynchronize(s));
    memcpy(out, ho, n);
    return LSQR_OK;
  }
  if (int rc = ensure(ctx, &ctx->staging, &ctx->staging_cap, n * mi.D * sizeof(double) + n)) return rc;
  double* d_in = reinterpret_cast<double*>(ctx->staging);
  uint8_t* d_out = ctx->staging + n * mi.D * sizeof(double);
  CK(cudaMemcpyAsync(d_in, packed, sizeof(double) * n * mi.D, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(ctx->small_dev + kSmIn, params, sizeof(double) * mi.P, cudaMemcpyHostToDevice, s));
  launch_agree_many(ctx->model, ctx->small_dev + kSmIn, d_in, (uint32_t)n, ctx->cfg, d_out, s); ctx->launches++;
  CKL();
  CK(cudaMemcpyAsync(out, d_out, n, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return LSQR_OK;
}

int lsqr_least_squares(lsqr_ctx* ctx, const double* packed, size_t n, double* out_params, int* n_params) {
  if (!ctx || !out_params || !n_params) return LSQR_ERR_ARG;
  if (ctx->group) { lsqr_ctx* k = ctx->group->kids[0]; const int rc = lsqr_least_squares(k, packed, n, out_params, n_params); if (rc) ctx->err = k->err; return rc; }
  if (ctx->model < 0) return fail(ctx, LSQR_ERR_STATE, "lsqr_set_estimator must be called first");
  const ModelInfo mi = model_info(ctx->model);
  *n_params = 0;
  if (n < (size_t)mi.K && ctx->model != RAY) return LSQR_OK;  // size guards, e.g. PlaneParametersEstimator.hxx:133-134
  if (n == 0) return LSQR_OK;
  if (int rc = upload_to(ctx, ctx->scratch, packed, n, sizeof(double) * mi.D, false)) return rc;
  return refine_impl(ctx, ctx->scratch, 0, out_params, n_params);
}

int lsqr_weighted_least_squares(lsqr_ctx* ctx, const double* packed, size_t n, const double* weights, double* out_params, int* n_params) {
  if (!ctx || !out_params || !n_params || !weights) return LSQR_ERR_ARG;
  if (ctx->group) { lsqr_ctx* k = ctx->group->kids[0]; const int rc = lsqr_weighted_least_squares(k, packed, n, weights, out_params, n_params); if (rc) ctx->err = k->err; return rc; }
  if (ctx->model != ABSOR) return fail(ctx, LSQR_ERR_ARG, "weighted least squares exists for the absolute-orientation estimator only");
  *n_params = 0;
  if (n < 3) return LSQR_OK;   // AbsoluteOrientationParametersEstimator.cxx:214-215
  if (int rc = upload_to(ctx, ctx->scratch, packed, n, sizeof(double) * 6, false)) return rc;
  cudaStream_t s = ctx->stream;
  if (int rc = ensure(ctx, &ctx->weights_dev, &ctx->weights_cap, n)) return rc;
  CK(cudaMemcpyAsync(ctx->weights_dev, weights, sizeof(double) * n, cudaMemcpyHostToDevice, s));
  const DataView dv = ctx->scratch.view();
  launch_weighted_absor_moments(dv, ctx->weights_dev, ctx->rb, s);
  launch_reduce_partials(ctx->rb, 16, s);
  launch_solve_weighted_absor(dv, ctx->rb.moments, ctx->small_dev + kSmOut, s); ctx->launches += 3;
  CKL();
  CK(cudaMemcpyAsync(ctx->pin, ctx->small_dev + kSmOut, sizeof(double) * (1 + LSQR_MAX_PARAMS), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  const int np = (int)ctx->pin[0];
  for (int j = 0; j < np; j++) out_params[j] = ctx->pin[1 + j];
  *n_params = np;
  ctx->scratch.moments_valid = false;
  return LSQR_OK;
}

int lsqr_microbench_fma(lsqr_ctx* ctx, int kind, int iters, double* out_fma_per_s, double* out_ms) {
  if (!ctx || kind < 0 || kind > 2 || iters <= 0) return LSQR_ERR_ARG;
  if (ctx->group) return lsqr_microbench_fma(ctx->group->kids[0], kind, iters, out_fma_per_s, out_ms);
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  float* sink = reinterpret_cast<float*>(ctx->small_dev + kSmSink);
  const int blocks = ctx->num_sms * 8, threads = 256;
  launch_fma_bench(kind, 16, blocks, threads, sink, s);  // warm-up
  CK(cudaEventRecord(ctx->ev[0], s));
  launch_fma_bench(kind, iters, blocks, threads, sink, s); ctx->launches += 2;
  CK(cudaEventRecord(ctx->ev[1], s));
  CKL();
  CK(cudaStreamSynchronize(s));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
  const double per_thread = (kind == 0 ? 16.0 : kind == 1 ? 32.0 : 8.0) * 8.0 * (double)iters;
  if (out_ms) *out_ms = ms;
  if (out_fma_per_s) *out_fma_per_s = per_thread * (double)blocks * threads / (ms * 1e-3);
  return LSQR_OK;
}

int lsqr_bench_refine_pass(lsqr_ctx* ctx, const double* params, int reps, double* ms_per_pass, double* algorithmic_bytes) {
  if (!ctx || !params || reps <= 0) return LSQR_ERR_ARG;
  if (ctx->group) return lsqr_bench_refine_pass(ctx->group->kids[0], params, reps, ms_per_pass, algorithmic_bytes);
  DataSet& ds = ctx->main;
  if (ctx->model < 0 || !ds.soa64) return fail(ctx, LSQR_ERR_STATE, "set the estimator and upload data first");
  const ModelInfo mi = model_info(ctx->model);
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  if (int rc = put_params(ctx, params)) return rc;
  uint32_t b, e;
  shard_range(ctx, ds, &b, &e);
  ctx->rb.maskbits = ds.maskbits;
  ctx->rb.maskbytes = nullptr;
  launch_mask_moments(ctx->model, ds.view(), b, e, ctx->small_dev + kSmIn, 1, nullptr, ctx->cfg, ctx->rb, s);   // warm-up
  CK(cudaEventRecord(ctx->ev[4], s));
  for (int i = 0; i < reps; i++) launch_mask_moments(ctx->model, ds.view(), b, e, ctx->small_dev + kSmIn, 1, nullptr, ctx->cfg, ctx->rb, s);
  CK(cudaEventRecord(ctx->ev[5], s));
  ctx->launches += (uint64_t)reps + 1;
  CKL();
  CK(cudaStreamSynchronize(s));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]));
  if (ms_per_pass) *ms_per_pass = (double)ms / reps;
  if (algorithmic_bytes) *algorithmic_bytes = (double)(e - b) * mi.D * sizeof(double) + (double)(e - b) / 8.0;
  ds.moments_valid = false; ds.mask_valid = true; ds.bytes_valid = false;
  return LSQR_OK;
}

int lsqr_last_refine_stats(const lsqr_ctx* ctx, double* kernel_ms, double* algorithmic_bytes, int* lm_iterations) {
  if (!ctx) return LSQR_ERR_ARG;
  if (ctx->group) return lsqr_last_refine_stats(ctx->group->kids[0], kernel_ms, algorithmic_bytes, lm_iterations);
  if (kernel_ms) *kernel_ms = ctx->refine_kernel_ms;
  if (algorithmic_bytes) *algorithmic_bytes = ctx->refine_bytes;
  if (lm_iterations) *lm_iterations = ctx->lm_iterations;
  return LSQR_OK;
}

}  // extern "C"
