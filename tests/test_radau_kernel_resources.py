"""CPU-only: the Radau kernels that gather per-environment data into the packed and compact arrays (tau_ext, and the contact-parameter rows
of pfc_set_contact_params) stay free of stack frames and spills (-Xptxas -v of pfc_radau.cu for sm_100a).  Skipped when nvcc is not
installed."""
import os
import re
import subprocess
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_small_kernel_resources import CSRC, _nvcc  # noqa: E402


@pytest.fixture(scope="module")
def radau_resources(tmp_path_factory):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    out = tmp_path_factory.mktemp("radau_res") / "pfc_radau.o"
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
                        os.path.join(CSRC, "pfc_radau.cu"), "-o", str(out)], capture_output=True, text=True, cwd=CSRC)
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


@pytest.mark.parametrize("kernel", ["radau_gather_kernel", "radau_select_kernel", "radau_finish_kernel", "radau_newton_kernel"])
def test_radau_kernels_have_no_local_memory(radau_resources, kernel):
    found = {k: v for k, v in radau_resources.items() if kernel in k}
    assert found, f"{kernel} not in the ptxas report"
    for name, (stack, st, ld) in found.items():
        assert stack == 0 and st == 0 and ld == 0, (name, stack, st, ld)
