"""bench.py --dump-outputs: the arrays the timed path returned in its last step, as float64 .npy files.  CPU only: the --impl
reference arm end to end, and the fixed sample written when the outputs exceed the size cap."""
import os
import subprocess
import sys

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_dumps_its_last_step(tmp_path):
    out = tmp_path / "dump"
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--envs", "16", "--steps", "2", "--warmup", "0",
                    "--dump-outputs", str(out)], check=True, capture_output=True)
    from oracle import orc
    from pfc_b200 import scenario as S
    m, X, tw = bench.build_inputs(16)
    S.attach_backend(m, orc.OracleContext())
    ref = m.backend.eval_f64(X, tw)
    assert np.array_equal(np.load(out / "env_index.npy"), np.arange(16.0))
    for name in ("wrench", "n_pairs", "flags"):
        a = np.load(out / f"{name}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, ref[name]), name
    assert (ref["flags"] & 1).sum() > 0


def test_outputs_over_the_cap_are_a_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    n = 1000
    rows = np.arange(n, dtype=np.float64)
    local = {"a": np.repeat(rows, 6).reshape(n, 6), "b": rows.astype(np.int32)}
    for d in ("x", "y"):
        bench.dump_outputs(str(tmp_path / d), local, n)
    idx = np.load(tmp_path / "x" / "env_index.npy")
    assert np.array_equal(idx, np.load(tmp_path / "y" / "env_index.npy"))       # the same sample every run
    assert 0 < len(idx) < n and (np.diff(idx) > 0).all()
    b = np.load(tmp_path / "x" / "b.npy")
    assert b.dtype == np.float64 and np.array_equal(b, idx)
    assert np.array_equal(np.load(tmp_path / "x" / "a.npy"), np.repeat(idx, 6).reshape(-1, 6))
    assert idx.nbytes + b.nbytes + 6 * b.nbytes <= 4000
