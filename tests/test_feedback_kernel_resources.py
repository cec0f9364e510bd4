"""CPU-only: the state-feedback kernel (pfc_set_feedback) has no stack frame and no spills in any of its three modes, and the Radau select
and gather kernels, which now also write the feedback rows of the compact slots and packed states, stay spill-free (-Xptxas -v for sm_100a).
Skipped when nvcc is not installed."""
import os
import re
import subprocess
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_small_kernel_resources import CSRC, _nvcc  # noqa: E402


def _resources(tmp_path_factory, source):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    out = tmp_path_factory.mktemp("fb_res") / (source + ".o")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
                        os.path.join(CSRC, source), "-o", str(out)], capture_output=True, text=True, cwd=CSRC)
    assert r.returncode == 0, r.stderr[-4000:]
    res, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            res[cur] = tuple(map(int, m.groups()))
    return res


@pytest.fixture(scope="module")
def state_resources(tmp_path_factory):
    return _resources(tmp_path_factory, "pfc_state.cu")


@pytest.fixture(scope="module")
def radau_resources(tmp_path_factory):
    return _resources(tmp_path_factory, "pfc_radau.cu")


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_feedback_kernel_has_no_local_memory(state_resources, mode):
    found = {k: v for k, v in state_resources.items() if f"state_feedback_kernelILi{mode}E" in k}
    assert len(found) == 1, f"state_feedback_kernel<{mode}> not in the ptxas report"
    for name, (stack, st, ld) in found.items():
        assert stack == 0 and st == 0 and ld == 0, (name, stack, st, ld)


@pytest.mark.parametrize("kernel", ["radau_select_kernel", "radau_gather_kernel"])
def test_select_and_gather_do_not_spill(radau_resources, kernel):
    found = {k: v for k, v in radau_resources.items() if kernel in k}
    assert found, f"{kernel} not in the ptxas report"
    for name, (stack, st, ld) in found.items():
        assert st == 0 and ld == 0, (name, st, ld)
