#!/usr/bin/env python
"""Cost of continuous affine state feedback (pfc_set_feedback) on test/boxes.jl batches.

  calcXd!           --envs environments through pfc_calcxd_f64_device and pfc_calcxd_jacobian_device in three configurations: no table, a
                    K = 0 table (random x_ref: the same bits as no table), a random table (K ~ U(-50, 50)).  Per call: L2 flushed (a 256 MB
                    memset), then CUDA events around the call on the library's stream; the configurations alternate call by call, --repeat
                    blocks of --calls calls each; median per block.
  roll-out          the workload of scripts/run_radau_rollout.py (--knots knots --dt apart, seeded random tau_ext schedule, h_max 0.05)
                    behind pfc_radau_rollout_device: no table, an n_seg = 1 PD table (w_n = 5 rad/s, zeta = 0.7, every floating body, toward
                    its start state) and an n_seg = --knots table (the same law with w_n from 3 to 8 rad/s over the segments), alternating;
                    wall time around a synchronised call.  A feedback law is other physics: accepted steps per environment are reported
                    beside every time.
  --parent DIR      also runs `bench.py --gpus 1 --steps S --warmup W --no-large --dump-outputs` alternately from DIR (a built checkout of the
                    parent commit) and from this tree, --bench-runs times each, and compares the dumped outputs bit for bit.

Prints one JSON line (and writes it to --out) with the card's name and power limit read in the same run."""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from run_contact_params import _bench, _card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--knots", type=int, default=20)
    ap.add_argument("--dt", type=float, default=0.025)
    ap.add_argument("--rollout-repeat", type=int, default=2)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--parent", default=None)
    ap.add_argument("--bench-runs", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=200)
    ap.add_argument("--bench-warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import pfc_b200  # noqa: F401
    from helpers import boxes_env_states, scene_boxes
    from pfc_b200 import capi
    from test_gpu_state_feedback import _pd_gains, _random_feedback

    out = {"what": "continuous affine state feedback on test/boxes.jl batches", "card": _card(), "n_env": args.envs}
    n_env = args.envs
    m = scene_boxes(capi.Context(0), max_env=n_env)[0]
    c = m.backend
    x = boxes_env_states(m, n_env)
    K, xr = _random_feedback(m, x, 1, args.seed)
    configs = {"no_table": None, "zero_K": (np.zeros_like(K), xr), "random": (K, xr)}
    out["table_bytes"] = {"K": int(K.nbytes), "x_ref": int(xr.nbytes)}

    def use(tab):
        c.set_feedback(*(tab if tab is not None else (None,)))

    # ---- calcXd! and its Jacobian ------------------------------------------------------------------------------------------------
    dev = torch.device("cuda", 0)
    nx, n_ins = x.shape[1], c.n_ins
    xd = torch.as_tensor(x).to(dev)
    xdot = torch.zeros((n_env, nx), dtype=torch.float64, device=dev)
    jac = torch.zeros((n_env, nx, nx), dtype=torch.float64, device=dev)
    npr = torch.zeros((n_env, n_ins), dtype=torch.int64, device=dev)
    fl = torch.zeros((n_env, n_ins), dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.ExternalStream(c.stream, device=dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    entry = {"pfc_calcxd_f64_device": (lambda: c.calcxd_f64_device(n_env, xd.data_ptr(), None, xdot.data_ptr(), npr.data_ptr(), fl.data_ptr()), xdot),
             "pfc_calcxd_jacobian_device": (lambda: c.calcxd_jacobian_device(n_env, xd.data_ptr(), None, jac.data_ptr(), xdot.data_ptr(), npr.data_ptr(),
                                                                             fl.data_ptr()), jac)}
    out["calcxd"] = {}
    for ep, (call, res) in entry.items():
        outputs = {}
        for name, tab in configs.items():   # warm-up of every configuration
            use(tab)
            for _ in range(3):
                call()
            c.sync()
            outputs[name] = res.cpu().numpy().copy()
        results = {k: [] for k in configs}
        for _ in range(args.repeat):
            times = {k: [] for k in configs}
            for _ in range(args.calls):
                for name, tab in configs.items():
                    use(tab)
                    with torch.cuda.stream(stream):
                        flush.zero_()
                        ev0.record(stream)
                        call()
                        ev1.record(stream)
                    ev1.synchronize()
                    times[name].append(ev0.elapsed_time(ev1))
            for name in configs:
                results[name].append(float(np.median(times[name])))
        out["calcxd"][ep] = {"calls_per_block": args.calls, "timing": "CUDA events, L2 flushed before every call", "median_ms_per_block": results,
                             "zero_K_bit_identical_to_no_table": bool(np.array_equal(outputs["no_table"], outputs["zero_K"])),
                             "random_changes_envs": int(sum(not np.array_equal(outputs["no_table"][e], outputs["random"][e]) for e in range(n_env)))}

    # ---- roll-out ----------------------------------------------------------------------------------------------------------------
    nk = args.knots
    knots = args.dt * np.arange(1, nk + 1)
    tau = np.random.default_rng(0).uniform(-1, 1, (nk, n_env, m.nv))
    tau_d = torch.as_tensor(tau).to(dev)
    nc = m.nq + m.nv
    pd1 = (_pd_gains(m, x, 5.0, 0.7)[None], x[None, :, :nc].copy())
    pdk = (np.stack([_pd_gains(m, x, w, 0.7) for w in np.linspace(3.0, 8.0, nk)]), np.repeat(pd1[1], nk, 0))
    ro_configs = {"no_table": None, "pd_n_seg_1": pd1, f"pd_n_seg_{nk}": pdk}

    def rollout(tab):
        use(tab)
        c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
        xs, t = xd.clone(), torch.zeros(n_env, dtype=torch.float64, device=dev)
        x_knot = torch.zeros((nk, n_env, nx), dtype=torch.float64, device=dev)
        stats = torch.zeros((n_env, 4), dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        c.radau_rollout_device(n_env, knots, 100000, xs.data_ptr(), tau_d.data_ptr(), t.data_ptr(), x_knot.data_ptr(), stats.data_ptr())
        c.sync()
        wall = time.perf_counter() - t0
        st = stats.cpu().numpy()
        assert (st[:, 0] == nk).all(), "an environment did not reach every knot"
        _, rounds, syncs = c.radau_step_info()
        return {"ms_per_knot": wall / nk * 1e3, "accepted_steps_per_env": float(st[:, 1].mean()), "rejected_per_env": float(st[:, 2].mean()),
                "rounds": rounds, "host_syncs": syncs}

    rollout(None)   # warm-up: the roll-out's buffers
    ro = {k: [] for k in ro_configs}
    for _ in range(args.rollout_repeat):
        for name, tab in ro_configs.items():
            ro[name].append(rollout(tab))
    out["rollout"] = {"workload": f"{nk} knots {args.dt} s apart, tau_ext uniform(-1, 1) seed 0, h_max 0.05", "runs": ro}
    use(None)

    # ---- parent against this change: bench.py alternately ----------------------------------------------------------------------
    if args.parent:
        runs, dumps = [], {}
        with tempfile.TemporaryDirectory() as tmp:
            for r in range(args.bench_runs):
                for build, tree in (("parent", os.path.abspath(args.parent)), ("this_change", ROOT)):
                    d = os.path.join(tmp, f"{build}_{r}")
                    res = _bench(tree, args, d)
                    runs.append({"build": build, "run": r, "value": res.get("value"), "unit": res.get("unit")})
                    dumps.setdefault(build, d)
            names = sorted(f for f in os.listdir(dumps["parent"]) if f.endswith(".npy"))
            same = all(np.array_equal(np.load(os.path.join(dumps["parent"], f)), np.load(os.path.join(dumps["this_change"], f))) for f in names)
        out["bench_parent_vs_this_change"] = {"command": f"bench.py --gpus 1 --steps {args.bench_steps} --warmup {args.bench_warmup} --no-large",
                                              "runs": runs, "dump_outputs": names, "dump_outputs_bit_identical": bool(same)}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
