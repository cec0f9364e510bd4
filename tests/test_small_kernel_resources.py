"""CPU-only: the small path's kernels keep what they need in registers and shared memory.

pfc_small.cu is compiled for sm_100a with -Xptxas -v and the report is read back:
  * narrow_tile_kernel<4, 4> (the tile kernel every batch runs) fits 128 registers with no stack frame and no spill traffic.  It runs
    at 4 CTAs x 128 threads per SM, so 128 registers is the whole register file, and a spill or a local-memory array silently puts
    L1 / L2 round trips on the critical path of every tile;
  * every broad_tile_kernel variant stays free of spills.
Skipped when nvcc is not installed."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pressurefieldcontact.jl_b200", "csrc")


def _nvcc():
    cand = [shutil.which("nvcc"), os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")]
    return next((c for c in cand if c and os.path.exists(c)), None)


@pytest.fixture(scope="module")
def resources(tmp_path_factory):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    out = tmp_path_factory.mktemp("small_res") / "pfc_small.o"
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
                        os.path.join(CSRC, "pfc_small.cu"), "-o", str(out)], capture_output=True, text=True, cwd=CSRC)
    assert r.returncode == 0, r.stderr[-4000:]
    res, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            res[cur] = dict(zip(("stack", "spill_st", "spill_ld"), map(int, m.groups())))
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and cur in res:
            res[cur]["regs"] = int(m.group(1))
    return res


def _kernels(res, pattern):
    found = {k: v for k, v in res.items() if re.search(pattern, k)}
    assert found, f"no kernel matching {pattern} in the ptxas report"
    return found


def test_narrow_tile_kernel_has_no_local_memory(resources):
    (name, r), = _kernels(resources, r"narrow_tile_kernelILi4ELi4E").items()
    assert r["regs"] <= 128, r
    assert r["stack"] == 0 and r["spill_st"] == 0 and r["spill_ld"] == 0, r


def test_broad_tile_kernels_do_not_spill(resources):
    for name, r in _kernels(resources, r"broad_tile_kernelILi\d+ELi8ELi2E").items():
        assert r["spill_st"] == 0 and r["spill_ld"] == 0, (name, r)
