#!/usr/bin/env python
"""bench.py -- hypothesis x point agree() evaluations per second (BASELINE.json metric).

A "step" is one pass of the hot path over one batch of synthetic input: minimal solve +
consensus scoring + arg-max of H Philox-sampled hypotheses against N points resident in HBM
(workload = BASELINE.json configs[1]: 3D plane, 10 M points, 40 % outliers, 1 M hypotheses per
GPU, fp32 fast mode).  `value` is whole-job evals/s with inputs resident; `e2e` is the same
metric through the C ABI with HOST buffers: upload (H2D) + score + consensus set (D2H mask) +
least-squares refine inside the timed region.  Multi-GPU: points replicated, hypotheses
partitioned (weak scaling: H per GPU fixed), one all-reduce(MAX) on the packed (count,index) key.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy (float64), so that two builds
can be compared output for output: inputs and step seeds depend only on the arguments (with --impl reference the sample is
--cpu-sample-hyps hypotheses, else DUMP_CPU_SAMPLE_HYPS instead of one sized from a timed probe).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY.md 8d accounting: FMA-pipe lane-ops per evaluation in the minimal fused form with per-hypothesis constants hoisted
# (an FFMA, FADD or FMUL each hold one lane of the pipe for one issue), and the same in flop (FFMA = 2).
#   hypersphere: d FADD + 1 FMUL + (d-1) FFMA = 2d.  kD line: SURVEY charges 3d + 1 (d FADD + 2 x (1 FMUL + (d-1) FFMA) + 1 FFMA,
#   the |v|^2 - (v.n)^2 form, which cancels catastrophically in fp32 for coordinates of +-1000); the kernel issues FEWER
#   operations in a form that does not cancel -- d = 2: the 2-D line form on the perpendicular, 2 FFMA; d = 3: the Pluecker form
#   |x X n - m|^2, 9 FFMA -- and the fraction is charged with what it issues.
OPS_PER_EVAL = {"plane3": 3, "plane4": 4, "line2d": 2, "line2": 2, "line3": 9, "circle2": 4, "sphere3": 6, "sphere4": 8, "absor": 15, "ray": 12,
                "pivot": 15, "dense5": 5, "dense6": 6, "usxw": 21, "uscp": 21}
FLOP_PER_EVAL = {"plane3": 6, "plane4": 8, "line2d": 4, "line2": 4, "line3": 18, "circle2": 5, "sphere3": 8, "sphere4": 11, "absor": 26, "ray": 19,
                 "pivot": 26, "dense5": 10, "dense6": 12, "usxw": 39, "uscp": 39}
# the wider template space (SURVEY.md 8f-4 / 8f-2): hyperplane d FFMA, hypersphere 2d, dense system n, kD line in the literal
# form 4d (d FADD + d FFMA + d FFMA + d FFMA; the |v|^2 - (v.n)^2 form SURVEY counts, 3d + 1, cancels in fp32)
for _d in (2, 5, 6, 7, 8):
    OPS_PER_EVAL[f"plane{_d}"], FLOP_PER_EVAL[f"plane{_d}"] = _d, 2 * _d
for _d in (5, 6, 7, 8):
    OPS_PER_EVAL[f"sphere{_d}"], FLOP_PER_EVAL[f"sphere{_d}"] = 2 * _d, 3 * _d - 1
for _d in (4, 5, 6, 7, 8):
    OPS_PER_EVAL[f"line{_d}"], FLOP_PER_EVAL[f"line{_d}"] = 4 * _d, 7 * _d - 1
for _n in (2, 3, 4, 7, 8):
    OPS_PER_EVAL[f"dense{_n}"], FLOP_PER_EVAL[f"dense{_n}"] = _n, 2 * _n
LANEOPS_PER_EVAL = OPS_PER_EVAL


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="plane3", choices=["plane3", "sphere3", "line2d", "absor"])
    ap.add_argument("--points", type=int, default=10_000_000)
    ap.add_argument("--hyps", type=int, default=1_000_000, help="hypotheses per GPU")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp64"])
    ap.add_argument("--cpu-sample-hyps", type=int, default=0, help="hypotheses in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the secondary configurations (BASELINE.json configs[2..4], per-model scoring table)")
    ap.add_argument("--comm", default="native", choices=["native", "hooks"],
                    help="N > 1: collectives issued by the library itself (ncclAllReduce / ncclAllGather, lsqr_ctx_init_nccl) or torch.distributed hooks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64, rank 0)")
    return ap.parse_args()


DUMP_MAX_BYTES = 64 << 20         # all arrays of one dump together
DUMP_CPU_SAMPLE_HYPS = 1024       # reference arm with --dump-outputs and no --cpu-sample-hyps: a fixed sample, not a timed probe


def dump_outputs(out_dir, arrays):
    """One float64 .npy per output of the last timed step, DUMP_MAX_BYTES in all: an array longer than its share is replaced
    by a fixed, seeded sample of its entries, stored with the sampled indices as <name>_index."""
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_MAX_BYTES // 8 // (2 * len(arrays))      # values per array, room left for its index
    for name, a in arrays.items():
        a = np.atleast_1d(np.asarray(a, dtype=np.float64))
        if a.size > cap:
            idx = np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))
            a = a.reshape(-1)[idx]
            np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_traffic():
    """DRAM bytes per launch from the committed ncu --set full captures (profiles/r02_traffic.json)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
    except Exception:
        return {}


def workload_config(model, N, Hper, world, precision, delta):
    """The `config` object both arms print: BASELINE.json configs[1] unless overridden on the command line."""
    return {"workload": f"{model} RANSAC (BASELINE.json configs[1]): {N} synthetic points, 40% outliers, {Hper} Philox hypotheses per GPU, delta={delta}",
            "points": N, "hypotheses_per_gpu": Hper, "hypotheses_total": Hper * world, "precision": precision,
            "parallelism": f"points replicated, hypotheses partitioned x{world}, 1 all-reduce(max) on the packed key",
            "l2": "256 MB flush buffer written between steps"}


def make_data(model, n):
    from lsqrrecipes_b200 import synth
    data, true = synth.GENERATORS[model](n, seed=synth.SEED)
    return data, synth.DELTAS[model]


def host_cores():
    """Cores this process may use.  torch.distributed.run exports OMP_NUM_THREADS=1 when nproc > 1, so the OpenMP default
    is useless there: the CPU legs always pass an explicit thread count."""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def _oracle():
    from oracle import pyoracle
    kind = "ref" if pyoracle.available("ref") else "port"
    if kind == "port" and not pyoracle.available("port"):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"])
    return pyoracle, pyoracle.Oracle(kind), kind


def cpu_reference_run(model, data, delta, n_hyps, threads=0):
    """Times the reference's own estimate()+agree() loop (oracle/_ref when built, else the C port)
    on `threads` host cores over n_hyps random subsets x all points."""
    from lsqrrecipes_b200 import synth
    pyoracle, orc, kind = _oracle()
    threads = threads or host_cores()
    m = pyoracle.MODELS[model]
    k = pyoracle.INFO[m][2]
    subs = synth.random_subsets(data.shape[0], k, n_hyps, seed=123)
    t0 = time.perf_counter()
    counts, _ = orc.score_subsets(m, delta, data, subs, nthreads=threads, want_params=False)
    dt = time.perf_counter() - t0
    return {"kind": "reference" if kind == "ref" else "port", "cores": threads,
            "seconds": dt, "evals": float(n_hyps) * data.shape[0], "best": int(counts.max()), "counts": counts}


def cpu_sample_size(model, data, delta, target_s, threads):
    """Hypotheses per CPU sample so that one sample takes ~target_s: sized from a short probe instead of an assumed rate."""
    probe = max(threads, 4)
    info = cpu_reference_run(model, data, delta, probe, threads)
    rate = probe / max(info["seconds"], 1e-3)
    return max(threads, int(rate * target_s) // threads * threads)


def reference_compute_ms(model, data, delta, prob=0.999, budget_s=60.0):
    """Wall time of the reference's own RANSAC<T,S>::compute (RANSAC.hxx:4-145: srand/rand subsets, estimate, N agree()
    calls per try, least squares over the consensus set) on one host thread, as shipped.  Only oracle/_ref has it."""
    pyoracle, orc, kind = _oracle()
    if kind != "ref":
        return None
    m = pyoracle.MODELS[model]
    n = data.shape[0]
    ms, frac = [], None
    t_all = time.perf_counter()
    for _ in range(3):
        t0 = time.perf_counter()
        prm, mask, frac = orc.ransac_random(m, delta, data, prob)
        ms.append(1e3 * (time.perf_counter() - t0))
        if time.perf_counter() - t_all > budget_s / 3:
            break
    return {"ms": float(np.median(ms)), "runs_ms": [float(x) for x in ms], "points": int(n), "desired_probability": prob, "threads": 1,
            "inlier_fraction": float(frac), "n_params": int(len(prm)),
            "what": "RANSAC<T,S>::compute(parameters, estimator, data, 0.999, &consensusSet) of the reference (oracle/_ref), single-threaded as shipped; "
                    "the number of tries is time-seeded (RANSAC.hxx:44)"}


def reference_compute_configs(budget_s=45.0):
    """SURVEY.md 8d, CPU baseline (i): the reference's own RANSAC<T,S>::compute, one thread as shipped, on BASELINE.json
    configs[2..4] -- sphere + Levenberg-Marquardt, absolute orientation, and a host loop over small problems (the reference's
    analogue of the batched mode) -- with N reduced where the full size would not fit the time box, stated per entry."""
    from lsqrrecipes_b200 import synth
    pyoracle, orc, kind = _oracle()
    if kind != "ref":
        return None
    out, t_all = [], time.perf_counter()

    def one(name, n, what):
        data, _ = synth.GENERATORS[name](n)
        t0 = time.perf_counter()
        prm, mask, frac = orc.ransac_random(pyoracle.MODELS[name], synth.DELTAS[name], data, 0.999)
        return {"config": what, "model": name, "points": n, "ms": 1e3 * (time.perf_counter() - t0), "inlier_fraction": float(frac), "n_params": int(len(prm)), "threads": 1}

    out.append(one("sphere3", 1_000_000, "configs[2] sphere3 + Levenberg-Marquardt, N reduced from 10 M to 1 M points"))
    if time.perf_counter() - t_all < budget_s:
        out.append(one("absor", 1_000_000, "configs[3] absolute orientation, 1M correspondences"))
    for name in ("line2d", "plane3"):
        if time.perf_counter() - t_all > budget_s:
            break
        nprob, npts = 256, 256
        probs = [synth.GENERATORS[name](npts, seed=300 + i)[0] for i in range(64)]
        t0 = time.perf_counter()
        for i in range(nprob):
            orc.ransac_random(pyoracle.MODELS[name], synth.DELTAS[name], probs[i % 64], 0.999)
        dt = time.perf_counter() - t0
        out.append({"config": f"configs[4] host loop of RANSAC::compute over {nprob} of the 65536 x 256-point {name} problems", "model": name, "problems": nprob,
                    "points_per_problem": npts, "ms_per_problem": 1e3 * dt / nprob, "problems_per_s": nprob / dt, "threads": 1})
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    data, delta = make_data(args.model, args.points)
    cores = host_cores()
    # each step is a bounded sample of the workload; the whole run (warm-up + steps + compute()) stays under ~2 minutes
    target_s = min(5.0, max(0.5, 60.0 / max(args.steps + args.warmup / 4.0, 1.0)))
    if args.cpu_sample_hyps:
        n_hyps = args.cpu_sample_hyps
    elif args.dump_outputs:     # the dumped counts must not depend on this host's speed
        n_hyps = DUMP_CPU_SAMPLE_HYPS
    else:
        n_hyps = cpu_sample_size(args.model, data, delta, target_s, cores)
    for _ in range(args.warmup):
        cpu_reference_run(args.model, data, delta, max(n_hyps // 4, cores), cores)
    times, info = [], None
    t_all = time.perf_counter()
    for _ in range(args.steps):
        info = cpu_reference_run(args.model, data, delta, n_hyps, cores)
        times.append(info["seconds"])
    total = time.perf_counter() - t_all
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"counts": info["counts"], "best_count": info["best"]})
    value = info["evals"] * args.steps / sum(times)
    comp = None if args.no_e2e else reference_compute_ms(args.model, data, delta)
    comp_configs = None if (args.no_e2e or args.no_configs) else reference_compute_configs()
    line = {
        "impl": "reference", "metric": "hypothesis x point agree() evals/sec", "value": value, "unit": "evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dict(workload_config(args.model, args.points, args.hyps, args.gpus, args.precision, delta),
                       sample=f"each step times {n_hyps} of the hypotheses x all {args.points} points on {cores} host cores (fp64, the reference's arithmetic)"),
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": info["cores"], "kind": info["kind"],
                         "sample": f"{n_hyps} hypotheses x {args.points} points per step, estimate()+agree() loop of RANSAC.hxx:217-249, OpenMP over hypotheses"},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "compute_e2e": comp, "configs": comp_configs,
        "gpu_launches": 0, "wall_s": total,
    }
    emit_line(line)


def secondary_configs(device, peak_fma_per_s, hbm_peak, budget_s=110.0):
    """BASELINE.json configs[2..4] and a per-model scoring table, time-boxed, single GPU: every number that README.md and
    DESIGN.md quote next to the headline comes from here, i.e. from the driver's own run of this file."""
    import torch
    from lsqrrecipes_b200 import FP32, FP64, Engine, synth
    t_start = time.perf_counter()
    out = []

    def left():
        return budget_s - (time.perf_counter() - t_start)

    def scoring(name, n, H, precision=FP32, reps=2, data=None):
        if data is None:
            data, _ = synth.GENERATORS[name](n)
        eng = Engine(name, synth.DELTAS[name], device=device)
        eng.upload(data)
        eng.score(count=min(H, 131072), precision=precision, seed=1)
        ms = [eng.score(count=H, precision=precision, seed=2 + i)["consensus_ms"] for i in range(reps)]
        eng.close()
        ev = float(H) * n / (min(ms) * 1e-3)
        rec = {"model": name, "points": n, "hypotheses": H, "precision": "fp32" if precision == FP32 else "fp64", "consensus_ms": min(ms), "evals_per_s": ev}
        if precision == FP32:
            rec.update(ops_per_eval=OPS_PER_EVAL[name], frac=ev * OPS_PER_EVAL[name] / peak_fma_per_s,
                       kernel="consensus_cb_kernel" if H >= 98304 else "consensus32_kernel")
        return rec

    def compute(name, n, ls_type=1, data=None):
        """wall time of upload + RANSAC::compute(..., 0.999, &consensusSet), from page-locked and from pageable host memory"""
        if data is None:
            data, _ = synth.GENERATORS[name](n)
        host = torch.from_numpy(data).pin_memory()
        mask_pin = torch.empty(n, dtype=torch.uint8).pin_memory().numpy()
        mask_pag = np.empty(n, dtype=np.uint8)
        eng = Engine(name, synth.DELTAS[name], ls_type=ls_type, device=device)
        res = {}
        for kind, src, mask in (("pinned", host.numpy(), mask_pin), ("pageable", data, mask_pag)):
            ms = []
            for i in range(4):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = eng.compute(src.ctypes.data, 0.999, precision=FP32, seed=50 + i, mask_out=mask, n=n, stride_bytes=data.shape[1] * 8)
                ms.append(1e3 * (time.perf_counter() - t0))
            res[f"compute_ms_{kind}"] = float(np.median(ms[1:]))
        st = eng.last_refine_stats()
        eng.close()
        res.update(model=name, points=n, tries=int(r["tries"]), inlier_fraction=float(r["fraction"]), n_params=int(len(r["params"])),
                   lm_evaluations=int(st["lm_iterations"]), refine_pass_ms=st["kernel_ms"],
                   refine_GBps=(st["bytes"] / (st["kernel_ms"] * 1e-3) / 1e9) if st["kernel_ms"] > 0 else None,
                   refine_frac_of_hbm=(st["bytes"] / (st["kernel_ms"] * 1e-3) / 1e9 / hbm_peak) if st["kernel_ms"] > 0 else None)
        return res

    try:
        # configs[2]: sphere RANSAC (4-point minimal) + Levenberg-Marquardt refine, 10 M points
        data, _ = synth.GENERATORS["sphere3"](10_000_000)
        rec = {"config": "configs[2] sphere3 + Levenberg-Marquardt, 10M points"}
        rec.update(scoring("sphere3", 10_000_000, 262_144, data=data, reps=2))
        rec.update(compute("sphere3", 10_000_000, 1, data=data))
        out.append(rec)
        del data
        # configs[3]: absolute orientation over 1 M correspondences
        data, _ = synth.GENERATORS["absor"](1_000_000)
        rec = {"config": "configs[3] absolute orientation, 1M correspondences"}
        rec.update(scoring("absor", 1_000_000, 1_000_000, data=data, reps=2))
        rec.update(compute("absor", 1_000_000, 1, data=data))
        out.append(rec)
        # configs[1] in fp64 validation mode on a hypothesis slice
        if left() > 20:
            rec = {"config": "configs[1] plane3, fp64 validation mode slice"}
            rec.update(scoring("plane3", 10_000_000, 65_536, precision=FP64, reps=1))
            rec.update(ops_per_eval=9, note="as-written 3 DSUB + 4 DMUL + 2 DADD, no FMA (SURVEY.md 8d)")
            out.append(rec)
        # configs[4]: 65,536 independent small problems of 256 points, one thread block per problem
        for name in ("line2d", "plane3"):
            if left() < 10:
                break
            nprob, npts = 65_536, 256
            rng = np.random.default_rng(17)
            D = synth.GENERATORS[name](8, seed=1)[0].shape[1]
            bases = [synth.GENERATORS[name](npts, seed=300 + i)[0] for i in range(64)]
            data = np.concatenate([bases[i % 64] for i in range(nprob)]) + np.repeat(rng.uniform(-50, 50, (nprob, D)), npts, axis=0)
            offsets = (np.arange(nprob + 1) * npts).astype(np.uint64)
            eng = Engine(name, synth.DELTAS[name], device=device)
            eng.ransac_batch(data[: 1024 * npts], offsets[:1025], prob=0.999, max_tries=2048, seed=1)
            ms, wall, wall_pin = [], [], []
            for i in range(3):
                t0 = time.perf_counter()
                r = eng.ransac_batch(data, offsets, prob=0.999, max_tries=2048, seed=11 + i)
                wall.append(1e3 * (time.perf_counter() - t0))
                ms.append(r["device_ms"])
            ms32 = [eng.ransac_batch(data, offsets, prob=0.999, max_tries=2048, seed=11 + i, precision=FP32)["device_ms"] for i in range(3)]
            pinned = torch.from_numpy(data).pin_memory()
            for i in range(3):
                t0 = time.perf_counter()
                eng.ransac_batch(pinned.numpy(), offsets, prob=0.999, max_tries=2048, seed=11 + i)
                wall_pin.append(1e3 * (time.perf_counter() - t0))
            del pinned
            eng.close()
            out.append({"config": f"configs[4] 65536 x 256-point {name} problems, one CTA each", "model": name, "problems": nprob, "points_per_problem": npts,
                        "kernel_ms": min(ms), "kernel_ms_fp32_scoring": min(ms32), "problems_per_s": nprob / (min(ms) * 1e-3), "wall_ms_pageable": float(np.median(wall)),
                        "wall_ms_pinned": float(np.median(wall_pin)), "host_bytes": int(data.nbytes),
                        "mean_inlier_fraction": float(r["counts"].mean() / npts)})
        # scoring table: every estimator through the constant-bank kernel (131072 hypotheses x 1 M data)
        table = []
        for name in ("line2d", "line2", "line3", "circle2", "sphere4", "plane4", "ray", "pivot", "dense5", "dense6", "usxw", "uscp"):
            if left() < 4:
                break
            table.append(scoring(name, 1_000_000, 1_048_576, reps=1))
        out.append({"config": "scoring table: 1M hypotheses x 1M data per estimator, fp32, frac = evals/s x SURVEY 8d lane-ops / measured FP32 lane rate",
                    "models": table})
        # the dimension-templated estimators at the ends of the instantiated range (2..8)
        table = []
        for name in ("plane2", "plane8", "sphere8", "line4", "line8", "dense2", "dense8"):
            if left() < 4:
                break
            table.append(scoring(name, 1_000_000, 1_048_576, reps=1))
        out.append({"config": "scoring table, template space: PlaneParametersEstimator<2, 8>, SphereParametersEstimator<8>, LineParametersEstimator<4, 8>, "
                              "DenseLinearEquationSystemParametersEstimator<double, 2 / 8>, 1M hypotheses x 1M data, fp32", "models": table})
    except Exception as e:  # a secondary measurement must never take the headline line down
        out.append({"error": repr(e)})
    return out


def multi_gpu_parity(device, rank, world, comm):
    """N > 1, before anything is timed: a sharded request (hypotheses partitioned over the ranks, consensus set and refine
    sharded by point range, collectives by NCCL) must return what an unsharded context on the same GPU returns."""
    import torch
    import torch.distributed as dist
    from lsqrrecipes_b200 import FP32, FP64, Engine, synth
    from lsqrrecipes_b200.dist import full_mask, init_native, install_hooks, upload_replicated
    checks = {}
    for name, n, H in (("plane3", 1_000_003, 65_536), ("sphere3", 300_001, 65_536)):
        data, _ = synth.GENERATORS[name](n, seed=8)
        host = torch.from_numpy(data).pin_memory()
        res = []
        for sharded in (False, True):
            eng = Engine(name, synth.DELTAS[name], device=device)
            if sharded and comm == "native":
                init_native(eng, rank, world)
                eng.upload_ptr(host.data_ptr(), n, data.shape[1] * 8)
            elif sharded:
                eng.set_stream(torch.cuda.current_stream().cuda_stream)
                install_hooks(eng, rank, world)
                upload_replicated(eng, host, rank, world)
            else:
                eng.upload(data)
            r = eng.score(count=H, precision=FP32, seed=11)
            r64 = eng.score(count=4096, precision=FP64, seed=11)
            cnt = eng.consensus(r["best_params"])
            mask = eng.get_mask()
            prm = eng.refine()
            c = eng.ransac(0.999, precision=FP32, seed=12)
            if sharded:
                mask, cmask = full_mask(mask), full_mask(c["mask"])
            else:
                cmask = c["mask"]
            res.append((r["best_index"], r["best_count"], r["best_params"].copy(), r64["best_index"], r64["best_count"], cnt, mask.copy(), prm.copy(),
                        c["best_index"], c["fraction"], cmask.copy(), c["params"].copy()))
            eng.close()
        a, b = res
        checks[name] = bool(a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2]) and a[3] == b[3] and a[4] == b[4] and a[5] == b[5]
                            and np.array_equal(a[6], b[6]) and np.allclose(a[7], b[7], rtol=1e-9, atol=1e-9) and a[8] == b[8] and a[9] == b[9]
                            and np.array_equal(a[10], b[10]) and a[11].shape == b[11].shape and np.allclose(a[11], b[11], rtol=1e-6, atol=1e-6))
    t = torch.tensor([1 if all(checks.values()) else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return {"ok": bool(int(t.item()) == 1), "world": world, "comm": comm, "rank0": checks,
            "what": "sharded == unsharded on every rank: fp32 and fp64 winner (index, count, parameters), consensus count and mask bit-exact, "
                    "refit to 1e-9, compute() index / fraction / mask exact and parameters to 1e-6"}


_JSON_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner) write to file descriptor 1 as
    well, so everything else is pointed at stderr and the line goes to the original descriptor."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit_line(line):
    payload = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(payload.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, payload)


def main():
    args = parse()
    _claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from lsqrrecipes_b200 import FP32, FP64, SAMPLE_PHILOX, Engine
    from lsqrrecipes_b200.dist import init_native, install_hooks, upload_replicated

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    precision = FP32 if args.precision == "fp32" else FP64
    model = args.model
    N, Hper = args.points, args.hyps
    Hglobal = Hper * world

    data, delta = make_data(model, N)
    host = torch.from_numpy(data).pin_memory()                 # host buffer for the e2e leg
    parity = multi_gpu_parity(local, rank, world, args.comm) if world > 1 else None
    eng = Engine(model, delta, device=local)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    if world > 1:
        if args.comm == "native":
            init_native(eng, rank, world)       # ncclAllReduce / ncclAllGather issued by liblsqr_b200.so itself
        else:
            install_hooks(eng, rank, world)
    eng.upload_ptr(host.data_ptr(), N, data.shape[1] * 8)       # untimed: inputs resident in HBM

    # measured pipe peaks for the roofline (same device, same moment)
    ffma, _ = eng.microbench_fma(0, 8192)
    ffma2, _ = eng.microbench_fma(1, 8192)
    dfma, _ = eng.microbench_fma(2, 2048)

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def step(seed):
        flush.zero_()
        return eng.score(count=Hglobal, sampler=SAMPLE_PHILOX, precision=precision, seed=seed)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for w in range(args.warmup):
        step(1000 + w)
    launches0 = eng.kernel_launches
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cons_ms = []
    with ClockSampler(local) as clk:
        ev0.record()
        for s in range(args.steps):
            r = step(s)
            cons_ms.append(r["consensus_ms"])
        ev1.record()
        barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {k: r[k] for k in ("best_index", "best_count", "n_valid", "best_subset", "best_params")})
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = eng.kernel_launches - launches0
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    evals_per_step = float(Hglobal) * float(N)
    value = evals_per_step * args.steps / (elapsed_ms * 1e-3)

    # roofline of the dominant kernel (consensus), from CUDA events on its own stream inside the library
    kern_ms = float(np.mean(cons_ms))
    kern_evals = float(Hper) * float(N)
    if precision == FP32:
        achieved = kern_evals * FLOP_PER_EVAL[model] / (kern_ms * 1e-3) / 1e12
        peak = max(ffma, ffma2) * 2 / 1e12                      # the better of the two measured FP32 chains (scalar FFMA, packed FFMA2)
        bound = "fp32_pipe"
    else:
        achieved = kern_evals * 9 / (kern_ms * 1e-3) / 1e12    # as-written 3 DSUB + 4 DMUL + 2 DADD, no FMA (SURVEY.md 8d)
        peak = dfma / 1e12                                       # one lane-op per cycle per fp64 lane
        bound = "fp64_pipe"
    traffic = load_traffic()
    tr = traffic.get("consensus_cb_kernel", {})
    cb_match = precision == FP32 and tr.get("config") == {"model": model, "points": N, "hyps": Hper}
    n_kernel_launches = -(-N // tr["points_per_launch"]) if cb_match else None
    roofline = {"bound": bound, "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": tr["bytes_per_launch"] if cb_match else None,
                "traffic_note": tr.get("step_level") if cb_match else None,
                "kernel": "consensus_cb_kernel" if (precision == FP32 and Hper >= 98304) else "consensus_kernel", "kernel_ms": kern_ms,
                "launches_per_step": n_kernel_launches,
                "algorithmic_flop_per_launch": (float(Hper) * tr["points_per_launch"] * FLOP_PER_EVAL[model]) if cb_match else None,
                "avg_launch_ms": (kern_ms / n_kernel_launches) if cb_match else None,
                "peak_source": "measured live: the faster of the register-resident FFMA and FFMA2 chains (lsqr_microbench_fma); MEASURED_PEAKS.json has no FP32 figure",
                "ffma_tflops": ffma * 2 / 1e12, "ffma2_tflops": ffma2 * 2 / 1e12, "dfma_tflops": dfma * 2 / 1e12,
                "algorithmic_flop_per_eval": FLOP_PER_EVAL[model] if precision == FP32 else 9}

    # e2e: host buffers in, mask + parameters out, everything inside the timed region
    e2e = None
    if not args.no_e2e:
        def upload_from_host():
            # N > 1: every rank needs all points; 1/world of the bytes per PCIe link, NCCL all-gather over NVLink for the rest
            if world > 1 and args.comm == "hooks":
                upload_replicated(eng, host, rank, world)
            else:       # native: the library fetches every world-th chunk over this rank's PCIe link and all-gathers the round
                eng.upload_ptr(host.data_ptr(), N, data.shape[1] * 8)

        def e2e_step(seed):
            upload_from_host()
            r = eng.score(count=Hglobal, sampler=SAMPLE_PHILOX, precision=precision, seed=seed)
            cnt = eng.consensus(r["best_params"])
            mask = eng.get_mask()
            prm = eng.refine()
            return cnt, mask, prm
        e2e_step(77)
        barrier()
        t0 = time.perf_counter()
        ke = max(1, min(args.steps, 3))
        for s in range(ke):
            cnt, mask, prm = e2e_step(s)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        rs = eng.last_refine_stats()
        # the second half of BASELINE.json's metric: wall time of RANSAC<T,S>::compute(parameters, estimator, data, 0.999,
        # &consensusSet) through the library -- upload from pinned host memory, adaptive rounds, consensus set, refine
        comp_ms, comp = [], None
        mask_host = torch.empty(N, dtype=torch.uint8).pin_memory().numpy()   # the caller's consensus-set buffer
        for s in range(4):
            barrier()
            t0 = time.perf_counter()
            if world > 1 and args.comm == "hooks":
                upload_from_host()
                comp = eng.ransac(0.999, precision=precision, seed=100 + s, mask_out=mask_host)
            else:       # lsqr_compute: upload, first scoring round, consensus set and refine in one pipelined call
                comp = eng.compute(host.data_ptr(), 0.999, precision=precision, seed=100 + s, mask_out=mask_host, n=N, stride_bytes=data.shape[1] * 8)
            comp_ms.append(1e3 * (time.perf_counter() - t0))
        # the same call with the reference's own container types: pageable std::vector-like memory in, pageable mask out
        pag_ms = []
        mask_pag = np.empty(N, dtype=np.uint8)
        for s in range(4):
            barrier()
            t0 = time.perf_counter()
            if world > 1 and args.comm == "hooks":
                upload_replicated(eng, host, rank, world)
                eng.ransac(0.999, precision=precision, seed=200 + s, mask_out=mask_pag)
            else:
                eng.compute(data, 0.999, precision=precision, seed=200 + s, mask_out=mask_pag)
            pag_ms.append(1e3 * (time.perf_counter() - t0))
        tc = torch.tensor([float(np.median(comp_ms[1:])), float(np.median(pag_ms[1:]))], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        compute_e2e = {"ms": float(tc[0].item()), "ms_pageable": float(tc[1].item()), "desired_probability": 0.999, "tries": int(comp["tries"]),
                       "inlier_fraction": float(comp["fraction"]), "device_ms": float(comp["device_ms"]), "n_params": int(len(comp["params"])),
                       "what": "RANSAC<T,S>::compute(parameters, estimator, data, 0.999, &consensusSet) through the C ABI with the data in host memory (lsqr_compute), wall clock, max over ranks; "
                               "ms: page-locked host buffers; ms_pageable: ordinary (std::vector-like) host memory for the data and the consensus set"}
        hbm_peak = None
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        except Exception:
            hbm_peak = 6650.0
        e2e = {"value": evals_per_step * ke / dt, "unit": "evals/s", "h2d_bytes_per_step": int(N * data.shape[1] * 8),
               "d2h_bytes_per_step": int(N + 8 * 16), "ms_per_step": 1e3 * dt / ke, "steps": ke,
               "inlier_fraction": cnt / N, "params": [float(x) for x in prm]}
        trm = traffic.get("mask_moments_kernel", {})
        # the streaming refine pass: average duration of 16 back-to-back launches between two CUDA events on the library's stream
        # (the same launch alone between two events, as compute() issues it, is reported next to it)
        rp = eng.bench_refine_pass(prm if len(prm) else r["best_params"], reps=16)
        roofline_refine = {"bound": "hbm", "achieved": rp["bytes"] / (rp["ms_per_pass"] * 1e-3) / 1e9 if rp["ms_per_pass"] > 0 else None,
                           "peak": hbm_peak, "unit": "GB/s", "kernel": "mask_moments_kernel", "kernel_ms": rp["ms_per_pass"], "launches_timed": 16,
                           "single_launch_ms": rs["kernel_ms"], "algorithmic_bytes": rp["bytes"],
                           "traffic": trm.get("bytes_per_launch") if (world == 1 and trm.get("config") == {"model": model, "points": N}) else None}
        if roofline_refine["achieved"]:
            roofline_refine["frac"] = roofline_refine["achieved"] / hbm_peak
    else:
        roofline_refine = None
        compute_e2e = None

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = host_cores()
        # bounded sample: ~15 s of host work, sized from a short probe
        n_hyps = args.cpu_sample_hyps or cpu_sample_size(model, data, delta, 15.0, cores)
        info = cpu_reference_run(model, data, delta, n_hyps, cores)
        cpu = {"value": info["evals"] / info["seconds"], "unit": "evals/s", "cores": info["cores"], "kind": info["kind"],
               "sample": f"{n_hyps} hypotheses x {N} points, estimate()+agree() loop (RANSAC.hxx:217-249), OpenMP over hypotheses, {info['seconds']:.1f} s"}

    configs = None
    if rank == 0 and world == 1 and not args.no_configs and not args.no_e2e:
        eng.close()
        eng = None
        del flush
        torch.cuda.empty_cache()
        configs = secondary_configs(local, max(ffma, ffma2), hbm_peak)

    if rank == 0:
        line = {
            "metric": "hypothesis x point agree() evals/sec", "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if precision == FP32 else "f64", "data": "synthetic",
            "config": workload_config(model, N, Hper, world, args.precision, delta),
            "roofline": roofline, "roofline_refine": roofline_refine, "cpu_baseline": cpu, "e2e": e2e, "compute_e2e": compute_e2e,
            "gpu_launches": int(launches), "clocks": clk.summary(),
            "best_count": int(r["best_count"]), "multi_gpu_parity": parity, "comm": (args.comm if world > 1 else None), "configs": configs,
        }
        emit_line(line)
    if eng is not None:
        eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
