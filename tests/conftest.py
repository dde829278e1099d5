import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")
    # a fresh checkout has no built artefacts (they are git-ignored): build once, in-tree, the way the driver does
    lib = os.path.join(ROOT, "lsqrrecipes_b200", "liblsqr_b200.so")
    if not os.path.exists(lib):
        import shutil
        if shutil.which("nvcc"):
            subprocess.check_call([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=ROOT)


@pytest.fixture(scope="session")
def port():
    """The plain-C restatement (oracle/liboracle.so); built on demand with gcc."""
    from oracle import pyoracle
    if not pyoracle.available("port"):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"])
    return pyoracle.Oracle("port")


@pytest.fixture(scope="session")
def ref():
    """The reference's own sources (oracle/_ref), or None.  They are not part of this repository: point LSQR_REFERENCE at a
    checkout of zivy/LSQRRecipes to build oracle/_ref; without it the comparisons read what the reference returned from
    tests/golden/reference_cases.npz."""
    from oracle import pyoracle
    if not pyoracle.available("ref"):
        src = os.environ.get("LSQR_REFERENCE", "")
        if not (src and os.path.isdir(os.path.join(src, "parametersEstimators"))):
            return None
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref", f"REF={os.path.abspath(src)}"])
    return pyoracle.Oracle("ref")


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def same_up_to_sign(a, b, idx, tol):
    """Eigenvector-derived entries (normals, directions, quaternions) are defined up to sign."""
    a, b = np.array(a, dtype=float), np.array(b, dtype=float)
    if a.shape != b.shape:
        return False
    if len(idx) and np.dot(a[idx], b[idx]) < 0:
        a = a.copy()
        a[idx] = -a[idx]
    scale = np.maximum(np.abs(b), 1.0)
    return bool(np.all(np.abs(a - b) <= tol * scale))


def model_family(name):
    """('plane' | 'sphere' | 'line' | 'dense' | None, dimension) of a dimension-templated estimator name."""
    import re
    if name == "circle2":
        return "sphere", 2
    m = re.fullmatch(r"(plane|sphere|line|dense)(\d)", name)
    return (m.group(1), int(m.group(2))) if m else (None, 0)


class _SignIdx(dict):
    """parameter entries that carry an arbitrary sign after leastSquaresEstimate: hyperplane normals, line directions, quaternions"""

    def __missing__(self, name):
        fam, d = model_family(name)
        return list(range(d)) if fam in ("plane", "line") else []


SIGN_IDX = _SignIdx({"line2d": [0, 1], "absor": [0, 1, 2, 3]})


def is_sphere(name):
    return model_family(name)[0] == "sphere"


def ls_types(name):
    """least-squares variants of an estimator: algebraic / geometric hypersphere, analytic / iterative ultrasound calibration"""
    return [0, 1] if (is_sphere(name) or name in ("usxw", "uscp")) else [1]


def pinv_tol(name):
    """None where estimate() is plain double arithmetic in the reference (bit-exact parity); else the rounding-level tolerance of
    the minimal solvers that go through a pseudo-inverse / null vector (VNL's SVD there, one-sided Jacobi here), which scales
    with the conditioning of the minimal system (the 9x9 / 12x12 calibration systems of random subsets reach 1e7)."""
    fam, d = model_family(name)
    if name == "pivot" or fam == "dense" or (fam == "plane" and d != 3):
        return 1e-9 if d <= 6 else 1e-8
    if name in ("usxw", "uscp") or (fam == "sphere" and d >= 4):
        return 1e-6
    return None


def lm_case_is_clear(port, name, ls_type):
    """The iterative cross-wire fit walks a flat valley: MINPACK needs hundreds to thousands of evaluations and whether its
    1e-15 tests fire before the reference's 5000-evaluation cap (-> empty result) is decided by rounding noise
    (tests/test_lm_cpu.py).  Parity tests on that estimator use cases where the oracle's run ends well inside the cap; call
    this right after port.least_squares()."""
    if name != "usxw" or ls_type != 1:
        return True
    info, nfev = port.last_lm()
    return 1 <= info <= 4 and nfev <= 2500
