"""bench.py's output contract, checked where no GPU is needed: the reference arm (the reference's CPU path timed on the
host cores) prints exactly one JSON line on stdout with the keys the driver reads; nothing else reaches stdout."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

REQUIRED = ["impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"]


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--points", "20000", "--hyps", "2000"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "evals/s" and d["vs_baseline"] is None
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port", "ref") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the second half of the metric: the reference's own RANSAC<T,S>::compute, one thread as shipped (only oracle/_ref has it)
    if cb["kind"] == "reference":
        assert d["compute_e2e"]["ms"] > 0 and d["compute_e2e"]["threads"] == 1 and d["compute_e2e"]["points"] == 20000
        kinds = [c["model"] for c in d["configs"]]
        assert kinds == ["sphere3", "absor", "line2d", "plane3"] and all(c["threads"] == 1 for c in d["configs"])
        assert d["configs"][0]["ms"] > 0 and d["configs"][2]["problems_per_s"] > 0


def _bench(args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, cwd=ROOT, timeout=timeout)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def _load_dump(d):
    arrays = {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}
    assert all(a.dtype == np.float64 for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    return arrays


def test_reference_arm_dumps_its_last_step(tmp_path, port):
    """--dump-outputs: the counts of the last timed sample (a fixed DUMP_CPU_SAMPLE_HYPS hypotheses, not the warm-up's quarter),
    identical from run to run and equal to agree() over the same subsets.  Every timed step of this arm scores the same subsets."""
    from lsqrrecipes_b200 import synth
    from oracle.pyoracle import MODELS
    args = ["--impl", "reference", "--steps", "2", "--warmup", "1", "--points", "20000", "--hyps", "2000", "--no-e2e"]
    dumps = []
    for run in ("a", "b"):
        _bench(args + ["--dump-outputs", str(tmp_path / run)])
        dumps.append(_load_dump(tmp_path / run))
    a, b = dumps
    assert sorted(a) == ["best_count", "counts"] and a["counts"].shape == (1024,)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    data, _ = synth.GENERATORS["plane3"](20000, seed=synth.SEED)
    counts, _ = port.score_subsets(MODELS["plane3"], synth.DELTAS["plane3"], data, synth.random_subsets(20000, 3, 1024, seed=123))
    assert np.array_equal(a["counts"], counts.astype(np.float64)) and a["best_count"][0] == counts.max()


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs on the timed path: what score() returned in the last timed step (seed steps - 1; the warm-up steps use
    1000 + w), identical from run to run."""
    from lsqrrecipes_b200 import FP32, SAMPLE_PHILOX, Engine, synth
    steps, N, H = 3, 200_000, 131_072
    args = ["--steps", str(steps), "--warmup", "1", "--points", str(N), "--hyps", str(H), "--no-cpu-baseline", "--no-e2e", "--no-configs"]
    dumps = []
    for run in ("a", "b"):
        line = _bench(args + ["--dump-outputs", str(tmp_path / run)])
        assert line["steps"] == steps
        dumps.append(_load_dump(tmp_path / run))
    a, b = dumps
    assert sorted(a) == ["best_count", "best_index", "best_params", "best_subset", "n_valid"]
    assert all(np.array_equal(a[k], b[k]) for k in a)
    data, _ = synth.GENERATORS["plane3"](N, seed=synth.SEED)
    eng = Engine("plane3", synth.DELTAS["plane3"])
    eng.upload(data)
    want = [eng.score(count=H, sampler=SAMPLE_PHILOX, precision=FP32, seed=s) for s in range(steps)]
    eng.close()
    for k in a:
        assert np.array_equal(a[k], np.atleast_1d(np.asarray(want[-1][k], dtype=np.float64))), k
    assert a["best_count"][0] == line["best_count"]
    assert any(not np.array_equal(a["best_params"], w["best_params"]) for w in want[:-1]), "earlier steps must be told apart"


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
                          "--points", "2000", "--hyps", "100"], capture_output=True, text=True, cwd=ROOT, timeout=600, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
