"""Static checks on the built sm_100a code (cuobjdump, no GPU): the instruction forms DESIGN.md section 3 relies on are what ptxas
actually emitted.  A compiler change that silently loses one of them would cost throughput, not correctness -- these tests are
the tripwire."""
import collections
import re
import shutil
import subprocess

import pytest

from lsqrrecipes_b200 import api

pytestmark = pytest.mark.skipif(not shutil.which("cuobjdump"), reason="cuobjdump not available")


@pytest.fixture(scope="module")
def sass():
    out = subprocess.run(["cuobjdump", "-sass", api.lib_path()], capture_output=True, text=True, check=True).stdout
    funcs, name = collections.defaultdict(list), None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m and name:
            funcs[name].append(m.group(1).strip())
    return funcs


def _one(funcs, pattern):
    hits = [k for k in funcs if re.search(pattern, k)]
    assert hits, pattern
    return funcs[hits[0]]


def test_plane_kernel_counts_through_the_carry_chain(sass):
    """consensus_cb_kernel<PLANE3, 12, 128, 8>: per pair of residuals 3 FFMA2 with a uniform-register point operand, two IADD3 that
    write only a carry predicate and one IADD3.X that consumes two predicates; no FSET / FSETP / LEA.HI in the loop."""
    ins = _one(sass, r"consensus_cb_kernelILi0ELi12ELi128ELi8E")
    ffma2 = [i for i in ins if i.startswith("FFMA2")]
    assert len(ffma2) >= 288 and sum("UR" in i for i in ffma2) >= 288, "points must come as uniform-register operands"
    cmp_ = [i for i in ins if re.match(r"IADD3 RZ, P\d, PT, R\d+, UR\d+, RZ", i)]
    addx = [i for i in ins if re.match(r"IADD3\.X R\d+, PT, PT, RZ, RZ, R\d+, P\d, P\d", i)]
    assert len(cmp_) >= 192 and len(addx) >= 96, (len(cmp_), len(addx))
    assert not [i for i in ins if i.startswith(("FSET", "FSETP"))]          # no float compare left in this kernel
    assert sum(i.startswith("LEA.HI") for i in ins) <= 2                    # (index arithmetic outside the loop)
    assert sum(i.startswith("LDCU") for i in ins) >= 24, "constant-bank loads"


def test_sphere_kernel_counts_through_the_carry_chain_with_its_own_window(sass):
    """consensus_cb_kernel<SPHERE3, 10, 128, 2>: 3 FADD2 + 3 FFMA2 per pair of residuals; the window 4 r delta is per hypothesis,
    so the two carry-only IADD3 read it from a register (stored pre-negated by the hoist kernel: no negation in the loop)."""
    ins = _one(sass, r"consensus_cb_kernelILi5ELi10ELi128ELi2E")
    assert sum(i.startswith("FFMA2") for i in ins) >= 60 and sum(i.startswith("FADD2") for i in ins) >= 60
    cmp_ = [i for i in ins if re.match(r"IADD3 RZ, P\d, PT, R\d+(\.reuse)?, R\d+(\.reuse)?, RZ", i)]
    addx = [i for i in ins if re.match(r"IADD3\.X R\d+, PT, PT, RZ, RZ, R\d+, P\d, P\d", i)]
    assert len(cmp_) >= 40 and len(addx) >= 20, (len(cmp_), len(addx))
    assert not [i for i in ins if i.startswith(("FSET", "FSETP"))]
    assert sum(i.startswith("IMAD.MOV R") for i in ins) == 0, "the window must not be negated inside the loop"


def test_refine_pass_streams_through_a_tma_ring(sass):
    """mask_moments_kernel<PLANE3, mask mode 1>: tiles arrive by cp.async.bulk (UBLKCP) on mbarriers (SYNCS), are read back
    with LDS.64, and the moments accumulate with DFMA; no global load of the centre inside the loop (two LDG at most, ahead of it)."""
    ins = _one(sass, r"mask_moments_kernelILi0ELi1ELb0E")
    assert any(i.startswith("UBLKCP") for i in ins) and any("SYNCS.PHASECHK" in i for i in ins)
    assert sum(i.startswith("LDS.64") for i in ins) >= 6 and sum(i.startswith("DFMA") for i in ins) >= 12
    first_wait = next(k for k, i in enumerate(ins) if "SYNCS.PHASECHK" in i)
    assert not [i for i in ins[first_wait:] if i.startswith("LDG") and ".64" in i], "per-row global loads inside the streaming loop"


def test_shared_memory_kernel_is_fed_by_tma(sass):
    ins = _one(sass, r"consensus32_kernelILi0ELi9ELi256ELi512ELi2E")
    assert any(i.startswith("UBLKCP") for i in ins), "cp.async.bulk (TMA) must be present"
    assert any("SYNCS" in i for i in ins), "mbarrier wait"


@pytest.mark.parametrize("model", range(34))
def test_constant_bank_kernels_read_their_points_through_uniform_registers(sass, model):
    """Every consensus_cb_kernel<M>: the points of the launch come out of the constant bank with LDCU (uniform registers) and
    never with an indexed LDC into ordinary registers -- ptxas falls back to that when a loaded pair has too few consumers in
    the loop body or an instruction names two data operands, and an SM sub-partition sustains only about one LDC.64 per 38
    cycles (the pivot estimator ran at 0.28 of the FP32 pipe that way, k_fast.cu BlockCB)."""
    ins = _one(sass, rf"consensus_cb_kernelILi{model}ELi\d+ELi128ELi\dE")
    assert not [i for i in ins if re.match(r"LDC(\.\d+)? R\d+, c\[0x3\]", i)], "indexed constant loads of the data"
    assert sum(i.startswith("LDCU.64") or i.startswith("LDCU.128") for i in ins) >= 4
    packed = [i for i in ins if i.startswith(("FFMA2", "FADD2", "FMUL2"))]
    # (the literal kD-line form of d >= 4 touches the datum in one of its four operations per component, everything else in two or more)
    assert sum("UR" in i for i in packed) >= len(packed) // (5 if 24 <= model <= 28 else 2), "packed operations take their datum from a uniform register"


def test_fp64_validation_kernel_compares_on_the_integer_alu(sass):
    """consensus_kernel<PLANE3, 4, 128, 256>: nine FP64-pipe instructions per evaluation (5 DADD + 4 DMUL as the reference
    writes them, minus the leading `0 +`), the threshold test as a 64-bit integer compare (ISETP + ISETP.EX) -- no DSETP."""
    ins = _one(sass, r"consensus_kernelILi0ELi4ELi128ELi256E")
    assert not [i for i in ins if i.startswith("DSETP")], "the squared-distance compare must not occupy the FP64 pipe"
    assert sum(i.startswith("DADD") for i in ins) == 40 and sum(i.startswith("DMUL") for i in ins) == 32   # 8 evaluations per iteration
    assert not [i for i in ins if i.startswith("DFMA")], "validation mode must not contract (the reference is built without FMA)"
    assert sum(".EX" in i and i.startswith("ISETP") for i in ins) >= 8
