"""Mints the golden fixtures in this directory from the REFERENCE ITSELF.

Run in the build container (needs /root/reference and oracle/_ref built by oracle/Makefile):

    python tests/golden/make_golden.py [model ...]      (no arguments: every model and the file-based cases)

For every model it stores seeded inputs and what the reference's own classes return for them
through oracle/_ref/libref_oracle.so (reference sources compiled unmodified against the VNL
shim): per-subset estimate() parameters and full agree() counts for an ordered subset list,
the result of RANSAC<T,S>::compute (exhaustive overload) on a small problem, and
leastSquaresEstimate() on the consensus set.  Plus the reference's file-based known-answer
case (testing/Data/pivotCalibrationData.txt).  The fixtures travel to the GPU box; the
reference does not.

    python tests/golden/make_golden.py cases [ref|port]

mints only reference_cases.npz: the inputs of the live comparisons in tests/test_oracle.py and what
the reference returns for them, reduced as those tests read it without oracle/_ref (counts and
rejection patterns in full, parameter matrices as a SHA-256 where compared bit-exact, else a fixed
sample of rows).  `port` mints it from the C restatement instead, for where the reference's sources
are not at hand: the restatement, as it stands, passed all of those comparisons against the
reference live on exactly these inputs.  The file's `source` entry says which of the two it holds.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from lsqrrecipes_b200 import synth  # noqa: E402
from oracle.pyoracle import INFO, MODELS, Oracle  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def mint_reference_cases(kind):
    """tests/golden/reference_cases.npz from Oracle(kind), with the case definitions of tests/test_oracle.py."""
    sys.path.insert(0, os.path.dirname(OUT))
    import test_oracle as t
    orc, fx = Oracle(kind), {}

    def put(prefix, d):
        fx.update({f"{prefix}.{k}": v for k, v in d.items()})
    for name, m in MODELS.items():
        put(f"live.{name}", t.reference_live(orc, name, m, keep=16))
        put(f"degenerate.{name}", t.reference_degenerate(orc, name, m, keep=16))
    for seed in range(4):
        for name, m, data, delta, subs in t.seed_cases(seed):
            put(f"seed{seed}.{name}", t.reference_seed_case(orc, name, m, data, delta, subs, keep=8))
    data, w = t.horn_case()
    put("horn", {"params": orc.weighted_absor(data, w)})
    put("models", t.reference_model_table(orc))
    # one byte blob with an index (name, dtype, shape, offset) instead of ~1300 small .npy members
    names = sorted(fx)
    arrs = [np.ascontiguousarray(fx[k]).reshape(np.shape(fx[k])) for k in names]
    np.savez_compressed(os.path.join(OUT, "reference_cases.npz"), source=np.array("oracle/_ref" if kind == "ref" else "oracle/liboracle.so"),
                        names=np.array(names), dtypes=np.array([a.dtype.str for a in arrs]),
                        shapes=np.array([list(a.shape) + [-1] * (2 - a.ndim) for a in arrs]),
                        offsets=np.cumsum([0] + [a.nbytes for a in arrs]),
                        blob=np.concatenate([a.reshape(-1).view(np.uint8) for a in arrs]))


def main():
    if sys.argv[1:2] == ["cases"]:
        mint_reference_cases(sys.argv[2] if len(sys.argv) > 2 else "ref")
        return
    ref = Oracle("ref")
    only = sys.argv[1:]
    for name, m in MODELS.items():
        if only and name not in only:
            continue
        D, P, k = INFO[m]
        delta = synth.DELTAS[name]
        n = 96
        data, true = synth.GENERATORS[name](n, seed=synth.SEED + m)
        subsets = synth.random_subsets(n, k, 400, seed=synth.SEED + 100 + m)
        counts, params = ref.score_subsets(m, delta, data, subsets)
        # exhaustive RANSAC::compute on a smaller problem (C(28,4) = 20475 subsets at most; the larger minimal subsets of
        # the wider template space get fewer data so that C(ns, k) stays below 20000)
        ns = 28 if (k <= 4 or m <= 14) else {5: 20, 6: 18, 7: 16, 8: 16, 9: 16}[k]
        small, _ = synth.GENERATORS[name](ns, seed=synth.SEED + 200 + m)
        fx = {"data": data, "delta": delta, "subsets": subsets, "counts": counts, "params": params, "true": true, "small": small}
        for ls_type in ([0, 1] if (name.startswith(("circle", "sphere")) or name in ("usxw", "uscp")) else [1]):
            prm, mask, frac, cnt, _ = ref.ransac_exhaustive(m, delta, small, ls_type=ls_type)
            fx[f"ex_params_ls{ls_type}"] = prm
            fx[f"ex_mask_ls{ls_type}"] = mask
            fx[f"ex_fraction_ls{ls_type}"] = frac
            # least squares over the consensus set of the best listed hypothesis
            b = int(np.argmax(counts))
            _, bm = ref.agree(m, delta, params[b], data)
            fx[f"lsq_ls{ls_type}"] = ref.least_squares(m, delta, data[bm.astype(bool)], ls_type)
        np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **fx)
        print(name, "best", counts.max(), "valid", int((~np.isnan(params[:, 0])).sum()), "exhaustive fraction", fx["ex_fraction_ls1"])

    # the reference's second file-based known answer: DenseLinearEquationSystemParametersEstimatorTest.cxx:153-213
    # (least squares over testing/Data/augmentedMatrix.txt against a 17-digit solution, tolerance 0.5)
    if not only or "dense6" in only:
        rows = np.loadtxt("/root/reference/testing/Data/augmentedMatrix.txt")
        ls = ref.least_squares(MODELS["dense6"], 0.5, rows)
        known = np.array([-1.777985584409468e+001, 1.111302171667757e+000, -1.568653413096010e+002, 1.469013927556186e+002,
                          -6.296891425314718e+001, -1.042139650090033e+003])
        np.savez_compressed(os.path.join(OUT, "dense_file.npz"), rows=rows, ls=ls, known_ls=known)
        print("dense file: ls", ls, "max |ls - known|", np.abs(ls - known).max())
    # the reference's own experimental cross-wire data set (testing/SinglePointTargetUSCalibrationParametersEstimatorTest.cxx:
    # 113-166 runs ANALYTIC then ITERATIVE least squares over testing/Data/crossWirePhantomTransformations.txt +
    # crossWirePhantom2DPoints.txt, 54 poses, and only prints the results): what the reference returns for it
    if not only or "usxw" in only:
        T = np.loadtxt("/root/reference/testing/Data/crossWirePhantomTransformations.txt").reshape(-1, 3, 4)
        q = np.loadtxt("/root/reference/testing/Data/crossWirePhantom2DPoints.txt")
        rec = np.concatenate([T[:, :, :3].reshape(len(T), 9), T[:, :, 3], q], axis=1)
        m = MODELS["usxw"]
        np.savez_compressed(os.path.join(OUT, "usxw_file.npz"), data=rec, delta=5.0, ls0=ref.least_squares(m, 5.0, rec, 0),
                            ls1=ref.least_squares(m, 5.0, rec, 1))
        print("cross-wire file: analytic/iterative differ by", np.abs(ref.least_squares(m, 5.0, rec, 0) - ref.least_squares(m, 5.0, rec, 1)).max())
    if only:
        return

    # configs[0] restated (SURVEY.md 8d, config 1a): PlaneParametersEstimatorTest's data shape --
    # 3 exact + 20 noisy points, bounds +-1000, sigma 1, delta 0.5 -- seeded, exhaustive C(23,3)=1771.
    rng = np.random.default_rng(synth.SEED)
    normal = rng.uniform(0, 1, 3)
    normal /= np.linalg.norm(normal)
    a = rng.uniform(-1000, 1000, 3)
    pts = rng.uniform(-1000, 1000, (23, 3))
    pts = pts - ((pts - a) @ normal)[:, None] * normal
    pts[3:] += rng.normal(0, 1.0, (20, 3))
    prm, mask, frac, cnt, _ = ref.ransac_exhaustive(0, 0.5, pts)
    subs = np.array([(i, j, l) for i in range(23) for j in range(i + 1, 23) for l in range(j + 1, 23)], dtype=np.int32)
    counts, params = ref.score_subsets(0, 0.5, pts, subs)
    np.savez_compressed(os.path.join(OUT, "config1_plane23.npz"), data=pts, delta=0.5, params=prm, mask=mask, fraction=frac,
                        all_counts=counts, all_params=params, true=np.concatenate([normal, a]))
    print("config1a plane23: fraction", frac, "best", counts.max(), "first argmax", int(np.argmax(counts)))

    # config 1c: the reference's file-based known-answer test
    path = "/root/reference/testing/Data/pivotCalibrationData.txt"
    frames = synth.frames_from_quat_file(path)
    nfr = len(frames)
    mini = frames[[0, int(nfr / 2.0), nfr - 1]]
    exact = ref.estimate(8, 1.0, mini)
    ls = ref.least_squares(8, 1.0, frames)
    np.savez_compressed(os.path.join(OUT, "pivot_file.npz"), frames=frames, exact=exact, ls=ls,
                        known_exact=np.array([-18.586, 1.98134, -157.439, 146.965, -62.0497, -1042.87]),
                        known_ls=np.array([-17.7799, 1.1113, -156.865, 146.901, -62.9689, -1042.14]))
    print("pivot file: exact", exact, "ls", ls)
    mint_reference_cases("ref")


if __name__ == "__main__":
    main()
