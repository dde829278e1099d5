"""Static checks on the built sm_100a code (cuobjdump, no GPU): lsqr_ransac_batch's cluster path has one
batch_cluster_kernel instantiation per batched model, and each of them meets its cluster at the hardware cluster barrier."""
import re
import shutil
import subprocess

import pytest

from lsqrrecipes_b200 import MODELS, api

pytestmark = pytest.mark.skipif(not shutil.which("cuobjdump"), reason="cuobjdump not available")

BATCH_MODELS = [m for n, m in MODELS.items() if n not in ("usxw", "uscp")]   # the ultrasound calibrations have no batched mode


@pytest.fixture(scope="module")
def cluster_kernels():
    out = subprocess.run(["cuobjdump", "-sass", api.lib_path()], capture_output=True, text=True, check=True).stdout
    kernels = {}
    for part in re.split(r"\n\s*Function : ", out)[1:]:
        name, body = part.split("\n", 1)
        m = re.match(r"_ZN4lsqr20batch_cluster_kernelILi(\d+)E", name.strip())
        if m:
            kernels[int(m.group(1))] = body
    return kernels


def test_one_cluster_kernel_per_batched_model(cluster_kernels):
    assert sorted(cluster_kernels) == sorted(BATCH_MODELS)


@pytest.mark.parametrize("model", BATCH_MODELS)
def test_cluster_kernel_meets_at_the_cluster_barrier(cluster_kernels, model):
    body = cluster_kernels[model]
    assert re.search(r"\bUCGABAR_ARV\b", body) and re.search(r"\bUCGABAR_WAIT\b", body)
