"""CPU-only: the rigid-body kernel of calcXd! (state_dynamics_kernel in pfc_state.cu, -Xptxas -v for sm_100a).

  * state_dynamics_kernel<double>, with and without a per-environment body table (pfc_set_body_params), has no stack frame and no spill
    traffic, at no more than 168 registers;
  * state_dynamics_kernel<Dual<6>> spills by design (255 registers, a stack frame of about 2 KB); its numbers are reported, not pinned,
    and the instantiation without a table must not need more local memory than the one with a table.
The Radau gather kernel, which writes each stage state's table row, is held to the same rule in test_radau_kernel_resources.py.
Skipped when nvcc is not installed."""
import os
import re
import subprocess
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_small_kernel_resources import CSRC, _nvcc  # noqa: E402


@pytest.fixture(scope="module")
def state_resources(tmp_path_factory):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    out = tmp_path_factory.mktemp("state_res") / "pfc_state.o"
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
                        os.path.join(CSRC, "pfc_state.cu"), "-o", str(out)], capture_output=True, text=True, cwd=CSRC)
    assert r.returncode == 0, r.stderr[-4000:]
    res, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            res[cur] = list(map(int, m.groups()))
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and cur in res:
            res[cur].append(int(m.group(1)))
    return {k: v for k, v in res.items() if "state_dynamics_kernel" in k}


def _variants(res, scalar):
    """{with_table: (stack, spill stores, spill loads, registers)} of state_dynamics_kernel<scalar, with_table> (Itanium mangling:
    d = double, NS_4DualILi6EEE = Dual<6>; Lb0E / Lb1E = false / true)."""
    tag = "IdLb" if scalar == "double" else "INS_4DualILi6EEELb"
    out = {}
    for name, v in res.items():
        i = name.find(tag)
        if i >= 0:
            out[name[i + len(tag)] == "1"] = tuple(v)
    return out


def test_double_kernel_has_no_local_memory(state_resources):
    v = _variants(state_resources, "double")
    assert set(v) == {False, True}, state_resources.keys()
    for table, (stack, st, ld, regs) in v.items():
        assert stack == 0 and st == 0 and ld == 0 and regs <= 168, (table, stack, st, ld, regs)


def test_dual6_kernel_reported(state_resources):
    v = _variants(state_resources, "dual6")
    assert set(v) == {False, True}, state_resources.keys()
    for table, (stack, st, ld, regs) in sorted(v.items()):
        print(f"state_dynamics_kernel<Dual<6>, table={table}>: {regs} registers, {stack} B stack, {st} B spill stores, {ld} B spill loads")
    assert v[False][0] <= v[True][0], v
