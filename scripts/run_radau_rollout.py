#!/usr/bin/env python
"""MPC-style roll-out: n_env test/boxes.jl environments advanced through --knots knot times --dt apart with a seeded, random,
piecewise-constant tau_ext schedule, behind pfc_radau_rollout_device.  The same schedule is also run as --knots one-knot calls, the
way a caller without roll-outs would have to stop at every knot.  Both runs start from the same controller state (pfc_radau_init) on
the same context and alternate --repeat times; prints one JSON line (and writes it to --out) with, per run: ms per knot and per simulated
second, accepted steps per environment, host synchronisations per round of steps, and the mean number of environments per Jacobian call
(every round of steps takes one Jacobian of the environments still under way).  Also: whether the two runs agree bit for bit, the card
and its power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--knots", type=int, default=20)
    ap.add_argument("--dt", type=float, default=0.025)
    ap.add_argument("--h-max", type=float, default=0.05)
    ap.add_argument("--repeat", type=int, default=2)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import pfc_b200  # noqa: F401
    from helpers import boxes_env_states, scene_boxes
    from pfc_b200 import capi
    from pfc_b200.radau_batched import DeviceBatchedRadau

    n_env, K = args.envs, args.knots
    m = scene_boxes(capi.Context(0), max_env=3 * n_env)[0]
    c = m.backend
    x0 = boxes_env_states(m, n_env)
    knots = args.dt * np.arange(1, K + 1)
    tau = np.random.default_rng(args.seed).uniform(-1, 1, (K, n_env, m.nv))
    dr = DeviceBatchedRadau(m, n_env, h_max=args.h_max)

    def run(one_knot_calls):
        c.radau_init(n_env, 2, 1.0e-4, args.h_max, 1.0e-16)
        with torch.cuda.stream(dr.stream):
            dr.t = torch.zeros(n_env, dtype=torch.float64, device=dr.dev)
            x = torch.as_tensor(x0).to(dr.dev)
            tau_d = torch.as_tensor(tau).to(dr.dev)
            c.sync()
            calls = [(k, k + 1) for k in range(K)] if one_knot_calls else [(0, K)]
            stats, syncs, attempt_rounds, x_knot = [], 0, 0, []
            t0 = time.perf_counter()
            for k0, k1 in calls:
                xk, st = dr.rollout(x, knots[k0:k1], tau_d[k0:k1])
                x = xk[-1]
                x_knot.append(xk)
                stats.append(st)
                _, nr, ns = c.radau_step_info()
                syncs += ns
                attempt_rounds += nr
            c.sync()
            wall = time.perf_counter() - t0
        stats = torch.stack(stats).cpu().numpy()            # [call][env][4]
        steps = stats[:, :, 1]
        step_rounds = int(steps.max(axis=1).sum())           # a round of steps per step of the slowest environment of each call
        assert (stats[:, :, 0].sum(axis=0) == K).all(), "an environment did not reach every knot"
        rec = {"ms_per_knot": wall / K * 1e3, "ms_per_simulated_second": wall / (K * args.dt) * 1e3,
               "accepted_steps_per_env": float(steps.sum(axis=0).mean()), "calls": len(calls), "step_rounds": step_rounds,
               "host_synchronisations_per_step_round": syncs / step_rounds, "attempt_rounds_per_step_round": attempt_rounds / step_rounds,
               "mean_active_envs_per_jacobian": float(steps.sum()) / step_rounds}
        return rec, torch.cat(x_knot).cpu().numpy()

    run(False)   # warm-up: module loads, the roll-out's buffers
    results = {"rollout": [], "one_knot_calls": []}
    for _ in range(args.repeat):
        for name, one in (("rollout", False), ("one_knot_calls", True)):
            rec, xk = run(one)
            results[name].append((rec, xk))
    identical = all(np.array_equal(a[1], b[1]) for a, b in zip(results["rollout"], results["one_knot_calls"]))
    out = {"scene": "C3 batch of test/boxes.jl", "n_env": n_env, "h_max": args.h_max, "knots": K, "knot_spacing_s": args.dt,
           "tau_ext": f"uniform(-1, 1) per (knot, env, dof), seed {args.seed}", "repeat": args.repeat, "card": _card(),
           "x_knot_identical_rollout_vs_one_knot_calls": bool(identical)}
    for name, rs in results.items():
        out[name] = rs[-1][0]
        out[name]["ms_per_knot_all_repeats"] = [r[0]["ms_per_knot"] for r in rs]
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
