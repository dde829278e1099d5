"""ctypes binding of include/lsqr_b200.h (one class, one method per entry point)."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

MODELS = {"plane3": 0, "line2d": 1, "line2": 2, "line3": 3, "circle2": 4, "sphere3": 5, "absor": 6, "ray": 7, "pivot": 8,
          "dense5": 9, "dense6": 10, "usxw": 11, "uscp": 12, "sphere4": 13, "plane4": 14}
# model id -> (dim, n_params, k)  (lsqr_model_info)
MODEL_INFO = {0: (3, 6, 3), 1: (2, 4, 2), 2: (2, 4, 2), 3: (3, 6, 2), 4: (2, 3, 3), 5: (3, 4, 4), 6: (6, 7, 3), 7: (6, 3, 2), 8: (12, 6, 3),
              9: (6, 5, 5), 10: (7, 6, 6), 11: (14, 20, 4), 12: (17, 17, 3), 13: (4, 5, 5), 14: (4, 8, 4)}
# the rest of the reference's template space (include/lsqr_b200.h: LSQR_PLANE2 ... LSQR_DENSE8)
for _d, _id in ((2, 15), (5, 16), (6, 17), (7, 18), (8, 19)):
    MODELS[f"plane{_d}"] = _id
    MODEL_INFO[_id] = (_d, 2 * _d, _d)
for _d in range(5, 9):
    MODELS[f"sphere{_d}"] = 20 + _d - 5
    MODEL_INFO[20 + _d - 5] = (_d, _d + 1, _d + 1)
for _d in range(4, 9):
    MODELS[f"line{_d}"] = 24 + _d - 4
    MODEL_INFO[24 + _d - 4] = (_d, 2 * _d, 2)
for _n, _id in ((2, 29), (3, 30), (4, 31), (7, 32), (8, 33)):
    MODELS[f"dense{_n}"] = _id
    MODEL_INFO[_id] = (_n + 1, _n, _n)
FP64, FP32 = 0, 1
SAMPLE_PHILOX, SAMPLE_EXHAUSTIVE, SAMPLE_LIST, SAMPLE_PARAMS = 0, 1, 2, 3
LS_ALGEBRAIC, LS_GEOMETRIC = 0, 1

_dp = ctypes.POINTER(ctypes.c_double)
_u8p = ctypes.POINTER(ctypes.c_uint8)
_u32p = ctypes.POINTER(ctypes.c_uint32)
_i32p = ctypes.POINTER(ctypes.c_int32)
_u64p = ctypes.POINTER(ctypes.c_uint64)

MAX_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p)
SUM_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p)


class ScoreArgs(ctypes.Structure):
    _fields_ = [("sampler", ctypes.c_int), ("precision", ctypes.c_int), ("seed", ctypes.c_uint64), ("first", ctypes.c_uint64),
                ("count", ctypes.c_uint64), ("subsets", _i32p), ("params", _dp), ("out_counts", _u32p), ("out_params", _dp)]


class ScoreResult(ctypes.Structure):
    _fields_ = [("best_index", ctypes.c_uint64), ("best_count", ctypes.c_uint32), ("n_valid", ctypes.c_uint32),
                ("best_subset", ctypes.c_int32 * 10), ("best_params", ctypes.c_double * 20),
                ("score_ms", ctypes.c_double), ("consensus_ms", ctypes.c_double), ("evals", ctypes.c_uint64)]


class ComputeResult(ctypes.Structure):
    _fields_ = [("params", ctypes.c_double * 20), ("n_params", ctypes.c_int), ("fraction", ctypes.c_double),
                ("best_count", ctypes.c_uint32), ("best_index", ctypes.c_uint64), ("tries", ctypes.c_uint64),
                ("device_ms", ctypes.c_double)]


class LsqrError(RuntimeError):
    pass


def lib_path():
    return os.path.join(_HERE, "liblsqr_b200.so")


_LIB = None


def load_library():
    """Loads liblsqr_b200.so (built in-tree by __graft_entry__.build()).  No fallback."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise LsqrError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
    lib = ctypes.CDLL(path)
    c = ctypes
    sig = {
        "lsqr_model_info": (c.c_int, [c.c_int, c.POINTER(c.c_int), c.POINTER(c.c_int), c.POINTER(c.c_int)]),
        "lsqr_model_plane": (c.c_int, [c.c_uint]), "lsqr_model_sphere": (c.c_int, [c.c_uint]), "lsqr_model_line": (c.c_int, [c.c_uint]),
        "lsqr_model_dense": (c.c_int, [c.c_uint]),
        "lsqr_ctx_create": (c.c_int, [c.POINTER(c.c_void_p), c.c_int]),
        "lsqr_device_count": (c.c_int, []),
        "lsqr_ctx_create_multi": (c.c_int, [c.POINTER(c.c_void_p), c.c_int]),
        "lsqr_ctx_world": (c.c_int, [c.c_void_p]),
        "lsqr_nccl_unique_id": (c.c_int, [c.c_void_p, c.c_size_t]),
        "lsqr_ctx_init_nccl": (c.c_int, [c.c_void_p, c.c_void_p, c.c_size_t, c.c_int, c.c_int]),
        "lsqr_ctx_destroy": (None, [c.c_void_p]),
        "lsqr_last_error": (c.c_char_p, [c.c_void_p]),
        "lsqr_ctx_set_stream": (c.c_int, [c.c_void_p, c.c_void_p]),
        "lsqr_kernel_launches": (c.c_uint64, [c.c_void_p]),
        "lsqr_set_estimator": (c.c_int, [c.c_void_p, c.c_int, c.c_double, c.c_double, c.c_int]),
        "lsqr_upload": (c.c_int, [c.c_void_p, c.c_void_p, c.c_size_t, c.c_size_t]),
        "lsqr_upload_device": (c.c_int, [c.c_void_p, c.c_void_p, c.c_size_t]),
        "lsqr_set_shard": (c.c_int, [c.c_void_p, c.c_int, c.c_int, MAX_FN, SUM_FN, c.c_void_p]),
        "lsqr_score": (c.c_int, [c.c_void_p, c.POINTER(ScoreArgs), c.POINTER(ScoreResult)]),
        "lsqr_consensus": (c.c_int, [c.c_void_p, _dp, _u32p]),
        "lsqr_get_mask": (c.c_int, [c.c_void_p, _u8p]),
        "lsqr_get_mask_bits": (c.c_int, [c.c_void_p, _u32p]),
        "lsqr_refine": (c.c_int, [c.c_void_p, c.c_int, _dp, c.POINTER(c.c_int)]),
        "lsqr_ransac": (c.c_int, [c.c_void_p, c.c_double, c.c_int, c.c_uint64, _u8p, c.POINTER(ComputeResult)]),
        "lsqr_ransac_exhaustive": (c.c_int, [c.c_void_p, c.c_int, _u8p, c.POINTER(ComputeResult)]),
        "lsqr_compute": (c.c_int, [c.c_void_p, c.c_void_p, c.c_size_t, c.c_size_t, c.c_double, c.c_int, c.c_uint64, _u8p, c.POINTER(ComputeResult)]),
        "lsqr_ransac_batch": (c.c_int, [c.c_void_p, _dp, _u64p, c.c_uint64, c.c_int, c.c_double, c.c_uint32, c.c_uint64, c.c_int, _dp, _u32p, _u8p, _dp]),
        "lsqr_batch_capacity": (c.c_int, [c.c_void_p, c.c_int, c.c_int, _u64p, _u64p]),
        "lsqr_estimate": (c.c_int, [c.c_void_p, _dp, c.c_size_t, _dp, c.POINTER(c.c_int)]),
        "lsqr_agree": (c.c_int, [c.c_void_p, _dp, _dp, c.c_size_t, _u8p]),
        "lsqr_least_squares": (c.c_int, [c.c_void_p, _dp, c.c_size_t, _dp, c.POINTER(c.c_int)]),
        "lsqr_weighted_least_squares": (c.c_int, [c.c_void_p, _dp, c.c_size_t, _dp, _dp, c.POINTER(c.c_int)]),
        "lsqr_microbench_fma": (c.c_int, [c.c_void_p, c.c_int, c.c_int, _dp, _dp]),
        "lsqr_last_refine_stats": (c.c_int, [c.c_void_p, _dp, _dp, c.POINTER(c.c_int)]),
        "lsqr_bench_refine_pass": (c.c_int, [c.c_void_p, _dp, c.c_int, _dp, _dp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


EXPORTED_SYMBOLS = [
    "lsqr_model_info", "lsqr_ctx_create", "lsqr_ctx_destroy", "lsqr_last_error", "lsqr_ctx_set_stream", "lsqr_kernel_launches",
    "lsqr_set_estimator", "lsqr_upload", "lsqr_upload_device", "lsqr_set_shard", "lsqr_score", "lsqr_consensus", "lsqr_get_mask",
    "lsqr_refine", "lsqr_ransac", "lsqr_ransac_exhaustive", "lsqr_ransac_batch", "lsqr_estimate", "lsqr_agree", "lsqr_least_squares",
    "lsqr_microbench_fma", "lsqr_last_refine_stats", "lsqr_weighted_least_squares",
    "lsqr_device_count", "lsqr_ctx_create_multi", "lsqr_ctx_world", "lsqr_nccl_unique_id", "lsqr_ctx_init_nccl", "lsqr_get_mask_bits",
    "lsqr_compute", "lsqr_bench_refine_pass", "lsqr_model_plane", "lsqr_model_sphere", "lsqr_model_line", "lsqr_model_dense",
    "lsqr_batch_capacity",
]


def _ptr(a, t):
    return a.ctypes.data_as(t) if a is not None else None


class Engine:
    """One lsqr_ctx.  `model` is a name from MODELS or an id."""

    def __init__(self, model, delta, aux=0.0, ls_type=LS_GEOMETRIC, device=0, gpus=None):
        """gpus: None -> one context on `device`; an int -> lsqr_ctx_create_multi over that many devices of this process
        (0 = all visible), native NCCL inside the library."""
        self.lib = load_library()
        self.model = MODELS[model] if isinstance(model, str) else int(model)
        self.dim, self.n_params, self.k = MODEL_INFO[self.model]
        h = ctypes.c_void_p()
        if gpus is None:
            rc = self.lib.lsqr_ctx_create(ctypes.byref(h), device)
            what = f"lsqr_ctx_create(device={device})"
        else:
            rc = self.lib.lsqr_ctx_create_multi(ctypes.byref(h), int(gpus))
            what = f"lsqr_ctx_create_multi({gpus})"
        if rc != 0:
            raise LsqrError(f"{what} failed with status {rc}: no usable sm_100 CUDA device / NCCL (there is no CPU fallback)")
        self.h = h
        self._hooks = None
        self.n = 0
        self._ck(self.lib.lsqr_set_estimator(self.h, self.model, float(delta), float(aux), int(ls_type)))

    def close(self):
        if getattr(self, "h", None):
            self.lib.lsqr_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise LsqrError(f"status {rc}: {self.lib.lsqr_last_error(self.h).decode()}")

    def set_estimator(self, delta, aux=0.0, ls_type=LS_GEOMETRIC):
        self._ck(self.lib.lsqr_set_estimator(self.h, self.model, float(delta), float(aux), int(ls_type)))

    def set_stream(self, cuda_stream):
        self._ck(self.lib.lsqr_ctx_set_stream(self.h, ctypes.c_void_p(cuda_stream)))

    @property
    def kernel_launches(self):
        return int(self.lib.lsqr_kernel_launches(self.h))

    # -- data -------------------------------------------------------------------------
    def upload(self, data, stride_bytes=None):
        """data: float64 array [n, dim] (or any buffer of n records with the given stride)."""
        d = np.ascontiguousarray(data, dtype=np.float64)
        if stride_bytes is None:
            d = d.reshape(-1, self.dim)
            stride_bytes = self.dim * 8
            n = d.shape[0]
        else:
            n = d.size * 8 // stride_bytes
        self.n = n
        self._ck(self.lib.lsqr_upload(self.h, d.ctypes.data_as(ctypes.c_void_p), n, stride_bytes))

    def upload_ptr(self, host_ptr, n, stride_bytes):
        self.n = n
        self._ck(self.lib.lsqr_upload(self.h, ctypes.c_void_p(host_ptr), n, stride_bytes))

    def upload_device(self, dev_ptr, n):
        self.n = n
        self._ck(self.lib.lsqr_upload_device(self.h, ctypes.c_void_p(dev_ptr), n))

    @property
    def world(self):
        return int(self.lib.lsqr_ctx_world(self.h))

    def nccl_unique_id(self):
        buf = ctypes.create_string_buffer(128)
        self._ck(self.lib.lsqr_nccl_unique_id(buf, 128))
        return buf.raw

    def init_nccl(self, unique_id, rank, world):
        """One process per GPU: the library does its collectives itself (ncclAllReduce / ncclAllGather on its stream)."""
        buf = ctypes.create_string_buffer(bytes(unique_id), 128)
        self._ck(self.lib.lsqr_ctx_init_nccl(self.h, buf, 128, int(rank), int(world)))

    def set_shard(self, rank, world, max_fn=None, sum_fn=None):
        mf = MAX_FN(max_fn) if max_fn else MAX_FN()
        sf = SUM_FN(sum_fn) if sum_fn else SUM_FN()
        self._hooks = (mf, sf)  # keep the trampolines alive
        self._ck(self.lib.lsqr_set_shard(self.h, rank, world, mf, sf, None))

    # -- scoring ----------------------------------------------------------------------
    def score(self, count=None, sampler=SAMPLE_PHILOX, precision=FP32, seed=0, first=0, subsets=None, params=None,
              want_counts=False, want_params=False):
        a = ScoreArgs()
        a.sampler, a.precision, a.seed, a.first = sampler, precision, seed, first
        keep = []
        if subsets is not None:
            s = np.ascontiguousarray(subsets, dtype=np.int32).reshape(-1, self.k)
            keep.append(s)
            a.subsets = _ptr(s, _i32p)
            count = s.shape[0] if count is None else count
        if params is not None:
            p = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, self.n_params)
            keep.append(p)
            a.params = _ptr(p, _dp)
            count = p.shape[0] if count is None else count
        a.count = int(count)
        counts = np.zeros(a.count, dtype=np.uint32) if want_counts else None
        oparams = np.full((a.count, self.n_params), np.nan) if want_params else None
        a.out_counts = _ptr(counts, _u32p)
        a.out_params = _ptr(oparams, _dp)
        r = ScoreResult()
        self._ck(self.lib.lsqr_score(self.h, ctypes.byref(a), ctypes.byref(r)))
        return {
            "best_index": int(r.best_index), "best_count": int(r.best_count), "n_valid": int(r.n_valid),
            "best_subset": np.array(r.best_subset[: self.k]), "best_params": np.array(r.best_params[: self.n_params]),
            "score_ms": r.score_ms, "consensus_ms": r.consensus_ms, "evals": int(r.evals), "counts": counts, "params": oparams,
        }

    def consensus(self, params):
        p = np.ascontiguousarray(params, dtype=np.float64)
        c = ctypes.c_uint32(0)
        self._ck(self.lib.lsqr_consensus(self.h, _ptr(p, _dp), ctypes.byref(c)))
        return int(c.value)

    def get_mask(self):
        m = np.zeros(self.n, dtype=np.uint8)
        self._ck(self.lib.lsqr_get_mask(self.h, _ptr(m, _u8p)))
        return m

    def get_mask_bits(self):
        """The consensus set as packed bits (datum i = bit i & 31 of word i >> 5), unpacked to one bool per datum here."""
        w = np.zeros((self.n + 31) // 32, dtype=np.uint32)
        self._ck(self.lib.lsqr_get_mask_bits(self.h, _ptr(w, _u32p)))
        return np.unpackbits(w.view(np.uint8), bitorder="little")[: self.n]

    def refine(self, use_mask=True):
        out = np.zeros(20)
        n = ctypes.c_int(0)
        self._ck(self.lib.lsqr_refine(self.h, 1 if use_mask else 0, _ptr(out, _dp), ctypes.byref(n)))
        return out[: n.value].copy()

    @staticmethod
    def _result(r, mask):
        return {"params": np.array(r.params[: r.n_params]), "fraction": r.fraction, "best_count": int(r.best_count),
                "best_index": int(r.best_index), "tries": int(r.tries), "device_ms": r.device_ms, "mask": mask}

    def ransac(self, prob, precision=FP32, seed=0, want_mask=True, mask_out=None):
        """mask_out: optional caller-owned uint8[n] (e.g. a view of pinned memory) that receives the consensus set."""
        mask = mask_out if mask_out is not None else (np.zeros(self.n, dtype=np.uint8) if want_mask else None)
        r = ComputeResult()
        self._ck(self.lib.lsqr_ransac(self.h, float(prob), precision, seed, _ptr(mask, _u8p), ctypes.byref(r)))
        return self._result(r, mask)

    def compute(self, data, prob, precision=FP32, seed=0, want_mask=True, mask_out=None, n=None, stride_bytes=None):
        """RANSAC<T,S>::compute with the data still on the host (lsqr_compute): upload and first scoring round overlapped.
        data: float64 array [n, dim], or a raw host pointer (int) together with n and stride_bytes."""
        if isinstance(data, int):
            ptr = ctypes.c_void_p(data)
        else:
            d = np.ascontiguousarray(data, dtype=np.float64).reshape(-1, self.dim)
            n, stride_bytes, ptr = d.shape[0], self.dim * 8, d.ctypes.data_as(ctypes.c_void_p)
        self.n = n
        mask = mask_out if mask_out is not None else (np.zeros(n, dtype=np.uint8) if want_mask else None)
        r = ComputeResult()
        self._ck(self.lib.lsqr_compute(self.h, ptr, n, stride_bytes, float(prob), precision, seed, _ptr(mask, _u8p), ctypes.byref(r)))
        return self._result(r, mask)

    def ransac_exhaustive(self, precision=FP64, want_mask=True):
        mask = np.zeros(self.n, dtype=np.uint8) if want_mask else None
        r = ComputeResult()
        self._ck(self.lib.lsqr_ransac_exhaustive(self.h, precision, _ptr(mask, _u8p), ctypes.byref(r)))
        return self._result(r, mask)

    def ransac_batch(self, data, offsets, exhaustive=False, prob=0.999, max_tries=1024, seed=0, want_masks=False, precision=FP64):
        d = np.ascontiguousarray(data, dtype=np.float64).reshape(-1, self.dim)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        nprob = len(off) - 1
        prm = np.zeros((nprob, self.n_params))
        cnt = np.zeros(nprob, dtype=np.uint32)
        masks = np.zeros(d.shape[0], dtype=np.uint8) if want_masks else None
        ms = ctypes.c_double(0)
        self._ck(self.lib.lsqr_ransac_batch(self.h, _ptr(d, _dp), _ptr(off, _u64p), nprob, 1 if exhaustive else 0, float(prob),
                                            int(max_tries), seed, int(precision), _ptr(prm, _dp), _ptr(cnt, _u32p), _ptr(masks, _u8p), ctypes.byref(ms)))
        return {"params": prm, "counts": cnt, "masks": masks, "device_ms": ms.value}

    def batch_capacity(self, precision=FP64, exhaustive=False):
        """(one_block, max_records): the largest problem, in records, that ransac_batch solves in one thread block, and the
        largest it takes at all (a thread-block cluster per problem; exhaustive mode keeps the one-block limit)."""
        one, most = ctypes.c_uint64(0), ctypes.c_uint64(0)
        self._ck(self.lib.lsqr_batch_capacity(self.h, int(precision), 1 if exhaustive else 0, ctypes.byref(one), ctypes.byref(most)))
        return int(one.value), int(most.value)

    # -- the estimator's own methods ---------------------------------------------------
    def estimate(self, data):
        d = np.ascontiguousarray(data, dtype=np.float64).reshape(-1, self.dim)
        out = np.zeros(20)
        n = ctypes.c_int(0)
        self._ck(self.lib.lsqr_estimate(self.h, _ptr(d, _dp), d.shape[0], _ptr(out, _dp), ctypes.byref(n)))
        return out[: n.value].copy()

    def agree(self, params, data):
        d = np.ascontiguousarray(data, dtype=np.float64).reshape(-1, self.dim)
        p = np.ascontiguousarray(params, dtype=np.float64)
        out = np.zeros(d.shape[0], dtype=np.uint8)
        self._ck(self.lib.lsqr_agree(self.h, _ptr(p, _dp), _ptr(d, _dp), d.shape[0], _ptr(out, _u8p)))
        return out

    def least_squares(self, data):
        d = np.ascontiguousarray(data, dtype=np.float64).reshape(-1, self.dim)
        out = np.zeros(20)
        n = ctypes.c_int(0)
        self._ck(self.lib.lsqr_least_squares(self.h, _ptr(d, _dp), d.shape[0], _ptr(out, _dp), ctypes.byref(n)))
        return out[: n.value].copy()

    def weighted_least_squares(self, data, weights):
        """AbsoluteOrientationParametersEstimator::weightedLeastSquaresEstimate (absolute orientation only)."""
        d = np.ascontiguousarray(data, dtype=np.float64).reshape(-1, self.dim)
        w = np.ascontiguousarray(weights, dtype=np.float64).reshape(-1)
        if len(w) != d.shape[0]:
            raise ValueError("one weight per datum")
        out = np.zeros(20)
        n = ctypes.c_int(0)
        self._ck(self.lib.lsqr_weighted_least_squares(self.h, _ptr(d, _dp), d.shape[0], _ptr(w, _dp), _ptr(out, _dp), ctypes.byref(n)))
        return out[: n.value].copy()

    # -- measurement ------------------------------------------------------------------
    def microbench_fma(self, kind, iters=4096):
        v = ctypes.c_double(0)
        ms = ctypes.c_double(0)
        self._ck(self.lib.lsqr_microbench_fma(self.h, kind, iters, ctypes.byref(v), ctypes.byref(ms)))
        return v.value, ms.value

    def bench_refine_pass(self, params, reps=16):
        """Average duration (ms) of one consensus-set + moments launch over `reps` back-to-back launches, and its bytes."""
        p = np.ascontiguousarray(params, dtype=np.float64)
        ms = ctypes.c_double(0)
        b = ctypes.c_double(0)
        self._ck(self.lib.lsqr_bench_refine_pass(self.h, _ptr(p, _dp), int(reps), ctypes.byref(ms), ctypes.byref(b)))
        return {"ms_per_pass": ms.value, "bytes": b.value}

    def last_refine_stats(self):
        ms = ctypes.c_double(0)
        b = ctypes.c_double(0)
        it = ctypes.c_int(0)
        self._ck(self.lib.lsqr_last_refine_stats(self.h, ctypes.byref(ms), ctypes.byref(b), ctypes.byref(it)))
        return {"kernel_ms": ms.value, "bytes": b.value, "lm_iterations": it.value}
