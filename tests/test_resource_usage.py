"""Resource usage of the C5 path kernel, read from the built library (no GPU needed).

k_path_sm2 is latency-bound: it hides dependent node loads with resident warps, so it runs at the register cap of its launch
bound, and every spill slot is a local-memory line that competes with the tree nodes for L1.  These tests keep it spill-free
at that cap: its stack frame is the traversal stack alone.
"""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "oclpathtracer_b200", "csrc")

# the instantiation the launcher runs without statistics (capi.cu, launch_mega_t): k_path_sm2<false, MINB = 11, 6 visits per vote>
C5_KERNEL = "_ZN3ptd10k_path_sm2ILb0ELi11ELi6EEEvNS_8SceneDevENS_10RenderArgsEPy"
C5_MIN_CTAS = 11
BLOCK = 128
REGS_PER_SM = 65536
REG_ALLOC_UNIT = 256  # registers are allocated per warp in units of 256


def _cuobjdump():
    found = shutil.which("cuobjdump")
    if found:
        return found
    cuda = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda"
    path = os.path.join(cuda, "bin", "cuobjdump")
    assert os.path.exists(path), "cuobjdump (CUDA toolkit) not found"
    return path


@pytest.fixture(scope="module")
def usage(pt):
    out = subprocess.run([_cuobjdump(), "--dump-resource-usage", pt.LIB_PATH], check=True, capture_output=True, text=True).stdout
    res, fn = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            fn = m.group(1)
        elif fn and "REG:" in line:
            res[fn] = {k: int(v) for k, v in re.findall(r"(\w+):(\d+)", line)}
            fn = None
    return res


def _lstack_bytes():
    with open(os.path.join(CSRC, "pt_device.cuh")) as f:
        entries = int(re.search(r"#define PTD_LSTACK_ENTRIES (\d+)", f.read()).group(1))
    return (entries + 1) * 8  # (ref, entry-t) pairs plus the spare slot below the stack


def test_c5_path_kernel_has_no_spills(usage):
    assert C5_KERNEL in usage, "the C5 path kernel is missing from libptb200.so"
    u = usage[C5_KERNEL]
    assert u["LOCAL"] == 0
    assert u["STACK"] == _lstack_bytes(), f"stack frame {u['STACK']} B: spill slots beyond the {_lstack_bytes()} B traversal stack"


def test_c5_path_kernel_registers_allow_its_launch_bound(usage):
    regs = usage[C5_KERNEL]["REG"]
    per_warp = -(-regs * 32 // REG_ALLOC_UNIT) * REG_ALLOC_UNIT
    ctas = REGS_PER_SM // (per_warp * (BLOCK // 32))
    assert ctas >= C5_MIN_CTAS, f"{regs} registers allow {ctas} CTAs of {BLOCK} threads per SM, the launcher assumes {C5_MIN_CTAS}"
