"""CPU-only: every broad_tile_kernel variant keeps its frontier bookkeeping in registers and shared memory -- no stack frame, no spills
(-Xptxas -v of pfc_small.cu for sm_100a, the same report tests/test_small_kernel_resources.py reads).  The per-problem segment ends
pc[] are read with compile-time indices only; a select chain that the compiler folds back into a run-time index puts the array on the
stack, and every level of every tile then pays local-memory round trips.  Skipped when nvcc is not installed."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_small_kernel_resources import _kernels, resources  # noqa: E402,F401  (the compile-and-parse fixture)


def test_broad_tile_kernels_have_no_local_memory(resources):  # noqa: F811
    found = _kernels(resources, r"broad_tile_kernelILi\d+ELi8ELi2E")
    assert len(found) == 3, sorted(found)
    for name, r in sorted(found.items()):
        print(f"{name}: {r['regs']} registers, {r['stack']} B stack")
        assert r["stack"] == 0 and r["spill_st"] == 0 and r["spill_ld"] == 0, (name, r)
        assert r["regs"] <= 128, (name, r)   # 2 CTAs x 256 threads per SM
