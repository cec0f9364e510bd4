#!/usr/bin/env python
"""Kernel-level timing of the small path on the C3 workload (4096 x test/boxes.jl): median per-kernel device times over a few
L2-flushed steps, plus a checksum of the wrenches (to see at a glance that an experiment changed no result)."""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import pfc_b200  # noqa: F401
    from helpers import boxes_env_states, scene_boxes
    from pfc_b200 import capi
    from pfc_b200 import scenario as S
    n_env = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
    m, _ = scene_boxes(None)
    x = boxes_env_states(m, n_env)
    X, tw, _ = S.boundary_arrays(m, x)
    ctx = capi.Context(0)
    S.attach_backend(m, ctx, max_env=n_env)
    dev = torch.device("cuda", 0)
    n_ins = ctx.n_ins
    Xd, twd = torch.from_numpy(np.ascontiguousarray(X)).to(dev), torch.from_numpy(np.ascontiguousarray(tw)).to(dev)
    w = torch.zeros((n_env, n_ins, 6), dtype=torch.float64, device=dev)
    npairs = torch.zeros((n_env, n_ins), dtype=torch.int64, device=dev)
    fl = torch.zeros((n_env, n_ins), dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    step = lambda: ctx.eval_f64_device(n_env, Xd.data_ptr(), twd.data_ptr(), None, w.data_ptr(), None, npairs.data_ptr(), fl.data_ptr())
    for _ in range(5):
        step()
    ctx.sync()
    ctx.set_timing(True)
    split = []
    for _ in range(15):
        with torch.cuda.stream(stream):
            flush.zero_()
        step()
        split.append(ctx.kernel_times())
    ctx.set_timing(False)
    # whole step with events
    e0 = [torch.cuda.Event(enable_timing=True) for _ in range(30)]
    e1 = [torch.cuda.Event(enable_timing=True) for _ in range(30)]
    for k in range(30):
        with torch.cuda.stream(stream):
            flush.zero_()
        e0[k].record(stream); step(); e1[k].record(stream)
    ctx.sync()
    tot = float(np.median([a.elapsed_time(b) for a, b in zip(e0, e1)]))
    wh = w.cpu().numpy()
    print(json.dumps({"n_env": n_env, "broad_us": 1e3 * float(np.median([a for a, _ in split])), "narrow_us": 1e3 * float(np.median([b for _, b in split])), "step_us": 1e3 * tot,
                      "wrench_sha": hashlib.sha256(wh.tobytes()).hexdigest()[:16], "contacts": int((fl.cpu().numpy() & 1).sum())}))


if __name__ == "__main__":
    main()
