#!/usr/bin/env python
"""Cost of per-environment contact parameters (pfc_set_contact_params) on test/boxes.jl batches.

  batch evaluation  --envs environments through pfc_eval_f64_device in three configurations: no table, a table of the scene's own values,
                    a random table.  Per call: L2 flushed (a 256 MB memset), then CUDA events around the call on the library's stream; the
                    configurations alternate call by call, --repeat blocks of --calls calls each; median per block.
  roll-out          the workload of scripts/run_radau_rollout.py (--knots knots --dt apart, seeded random tau_ext schedule, h_max 0.05)
                    behind pfc_radau_rollout_device, with no table, the scene's own values and a random table, alternating; wall time
                    around a synchronised call.  A random table is other physics: its accepted steps are reported beside its time.
  --parent DIR      also runs `bench.py --gpus 1 --steps S --warmup W --no-large --dump-outputs` alternately from DIR (a built checkout of the
                    parent commit) and from this tree, --bench-runs times each, and compares the dumped outputs bit for bit.

Prints one JSON line (and writes it to --out) with the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip()


def _tables(m, n_env, seed):
    """(own, random) tables [n_env][n_ins][8]: the scene's constants, and random ones (Ebar x U(0.3, 3) per tetrahedral mesh, chi U(0, 3),
    mu_d U(0.05, 0.6), mu_s = mu_d U(1, 1.6), v_c U(2e-3, 3e-2) per instruction)."""
    rng = np.random.default_rng(seed)
    ins = m.ContactInstructions
    ebar = np.array([mc.c_prop.E_bar if mc.mesh.is_tet else 0.0 for mc in m.MeshCache])
    own = np.zeros((len(ins), 8))
    for k, ci in enumerate(ins):
        q = ci.friction_model.params()
        own[k, :3] = [ci.chi, ebar[ci.id_1], ebar[ci.id_2]]
        own[k, 3:3 + len(q)] = q
    own = np.repeat(own[None], n_env, 0)
    e_rand = ebar[None, :] * rng.uniform(0.3, 3.0, (n_env, len(ebar)))
    rnd = np.zeros_like(own)
    for k, ci in enumerate(ins):
        assert ci.friction_model.model == 0
        mu_d = rng.uniform(0.05, 0.6, n_env)
        rnd[:, k, 0] = rng.uniform(0.0, 3.0, n_env)
        rnd[:, k, 1], rnd[:, k, 2] = e_rand[:, ci.id_1], e_rand[:, ci.id_2]
        rnd[:, k, 3:6] = np.stack([mu_d * rng.uniform(1.0, 1.6, n_env), mu_d, rng.uniform(2e-3, 3e-2, n_env)], 1)
    return own, rnd


def _bench(tree, args, out_dir):
    cmd = [sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", str(args.bench_steps), "--warmup", str(args.bench_warmup),
           "--no-large", "--dump-outputs", out_dir]
    p = subprocess.run(cmd, capture_output=True, text=True, cwd=tree)
    if p.returncode != 0:
        raise RuntimeError(f"bench.py failed in {tree}:\n{p.stderr[-3000:]}")
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1]
    return json.loads(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--calls", type=int, default=50)
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
    from pfc_b200 import scenario as S

    out = {"what": "per-environment contact parameters on test/boxes.jl batches", "card": _card(), "n_env": args.envs}
    n_env = args.envs
    m = scene_boxes(capi.Context(0), max_env=n_env)[0]
    c = m.backend
    own, rnd = _tables(m, n_env, args.seed)
    configs = {"no_table": None, "own_values": own, "random": rnd}

    # ---- batch evaluation --------------------------------------------------------------------------------------------------------
    dev = torch.device("cuda", 0)
    x = boxes_env_states(m, n_env)
    X, tw, _ = S.boundary_arrays(m, x)
    Xd, twd = torch.as_tensor(X).to(dev), torch.as_tensor(tw).to(dev)
    n_ins = c.n_ins
    w = torch.zeros((n_env, n_ins, 6), dtype=torch.float64, device=dev)
    npr = torch.zeros((n_env, n_ins), dtype=torch.int64, device=dev)
    fl = torch.zeros((n_env, n_ins), dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.ExternalStream(c.stream, device=dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def call():
        c.eval_f64_device(n_env, Xd.data_ptr(), twd.data_ptr(), None, w.data_ptr(), None, npr.data_ptr(), fl.data_ptr())

    results = {k: [] for k in configs}
    outputs = {}
    for name, tab in configs.items():   # warm-up of every configuration
        c.set_contact_params(tab)
        for _ in range(3):
            call()
        c.sync()
        outputs[name] = w.cpu().numpy().copy()
    torch.cuda.synchronize()
    for _ in range(args.repeat):
        times = {k: [] for k in configs}
        for _ in range(args.calls):
            for name, tab in configs.items():
                c.set_contact_params(tab)
                with torch.cuda.stream(stream):
                    flush.zero_()
                    ev0.record(stream)
                    call()
                    ev1.record(stream)
                ev1.synchronize()
                times[name].append(ev0.elapsed_time(ev1))
        for name in configs:
            results[name].append(float(np.median(times[name])))
    out["batch_eval"] = {"entry_point": "pfc_eval_f64_device", "calls_per_block": args.calls, "timing": "CUDA events, L2 flushed before every call",
                         "median_ms_per_block": results,
                         "own_values_bit_identical_to_no_table": bool(np.array_equal(outputs["no_table"], outputs["own_values"])),
                         "random_changes_wrenches_of_envs": int(sum(not np.array_equal(outputs["no_table"][e], outputs["random"][e]) for e in range(n_env)))}

    # ---- roll-out ----------------------------------------------------------------------------------------------------------------
    K = args.knots
    knots = args.dt * np.arange(1, K + 1)
    tau = np.random.default_rng(0).uniform(-1, 1, (K, n_env, m.nv))
    tau_d = torch.as_tensor(tau).to(dev)
    x0 = torch.as_tensor(x).to(dev)

    def rollout(tab):
        c.set_contact_params(tab)
        c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
        xs, t = x0.clone(), torch.zeros(n_env, dtype=torch.float64, device=dev)
        x_knot = torch.zeros((K, n_env, x.shape[1]), dtype=torch.float64, device=dev)
        stats = torch.zeros((n_env, 4), dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        c.radau_rollout_device(n_env, knots, 100000, xs.data_ptr(), tau_d.data_ptr(), t.data_ptr(), x_knot.data_ptr(), stats.data_ptr())
        c.sync()
        wall = time.perf_counter() - t0
        st = stats.cpu().numpy()
        assert (st[:, 0] == K).all(), "an environment did not reach every knot"
        return wall, float(st[:, 1].mean()), x_knot.cpu().numpy()

    rollout(None)   # warm-up: the roll-out's buffers
    ro = {k: [] for k in configs}
    knots_out = {}
    for _ in range(args.rollout_repeat):
        for name, tab in configs.items():
            wall, steps, xk = rollout(tab)
            ro[name].append({"ms_per_knot": wall / K * 1e3, "accepted_steps_per_env": steps})
            knots_out[name] = xk
    out["rollout"] = {"workload": f"{K} knots {args.dt} s apart, tau_ext uniform(-1, 1) seed 0, h_max 0.05", "runs": ro,
                      "own_values_x_knot_bit_identical_to_no_table": bool(np.array_equal(knots_out["no_table"], knots_out["own_values"]))}
    c.set_contact_params(None)

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
