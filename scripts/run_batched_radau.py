#!/usr/bin/env python
"""Batched roll-out: n_env independent test/boxes.jl scenes advanced by the reference's adaptive Radau IIA scheme with every array on
the GPU (pfc_b200.radau_batched).  Prints one JSON line.

  --impl torch   (default) BatchedRadau, the Newton loop as torch ops between library calls: environment-steps per second, the split
                 between Jacobian chunks, stage evaluations and the rest, and the CPU oracle's single-scene rate for scale.
  --impl device  DeviceBatchedRadau, the whole step behind pfc_radau_step_device.
  --impl both    both paths on the same seeded states after the same warm-up: per path ms per batched step, env-steps/s, stage states
                 per environment per step, attempt rounds and host synchronisations per step; the device path's time split (CUDA events
                 inside the library, in a separate pass); how far the two paths agree over the timed steps; the card and its power limit."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cpu-steps", type=int, default=10)
    ap.add_argument("--impl", choices=("torch", "device", "both"), default="torch")
    args = ap.parse_args()
    if args.impl != "torch":
        return compare(args)
    import torch
    import pfc_b200  # noqa: F401
    from helpers import boxes_env_states, scene_boxes
    from oracle import orc
    from pfc_b200 import capi
    from pfc_b200 import dynamics as D
    from pfc_b200 import radau as R
    from pfc_b200 import scenario as S
    from pfc_b200.radau_batched import BatchedRadau

    n_env = args.envs
    m = scene_boxes(capi.Context(0), max_env=3 * n_env)[0]
    x0 = boxes_env_states(m, n_env)
    br = BatchedRadau(m, n_env, h_max=0.05)
    with torch.cuda.stream(br.stream):
        x = torch.as_tensor(x0).to(br.dev)
        for _ in range(args.warmup):
            x, _ = br.step(x)
        m.backend.sync()
        c0, j0, a0 = br.n_calcxd_states, br.n_chunk_states, br.n_attempts
        t0 = time.perf_counter()
        for _ in range(args.steps):
            x, _ = br.step(x)
        m.backend.sync()
        wall = time.perf_counter() - t0
        # split: time the two device entry points alone on the same batch
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record(br.stream)
        br._jacobian(x)
        ev[1].record(br.stream)
        br._calcxd(x)
        ev[2].record(br.stream)
        _, negJ = br._jacobian(x)
        ev[2].record(br.stream)
        shift = torch.view_as_real((1.0 / br.h * br.tab[0]["lam"][0]).to(torch.complex128)).contiguous()
        invc = torch.empty((n_env, br.NX, br.NX), dtype=torch.complex128, device=br.dev)
        m.backend.radau_inv_c_device(n_env, br.NX, negJ.data_ptr(), shift.data_ptr(), None, invc.data_ptr(), br.info.data_ptr())
        ev[3].record(br.stream)
        m.backend.sync()
        ev4 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev4[0].record(br.stream)
        br._calcxd(x)
        ev4[1].record(br.stream)
        m.backend.sync()
        jac_ms, f3_ms, inv_ms = ev[0].elapsed_time(ev[1]), ev4[0].elapsed_time(ev4[1]), ev[2].elapsed_time(ev[3])
        chk = torch.bmm(invc, (negJ.to(torch.complex128) + torch.view_as_complex(shift)[:, None, None] * br.eye)) - br.eye
        inv_residual = float(chk.abs().max())
    assert torch.isfinite(x).all()
    out = {"scene": "C3 batch of test/boxes.jl", "n_env": n_env, "radau_steps": args.steps, "wall_s": wall,
           "env_steps_per_sec": n_env * args.steps / wall, "ms_per_batched_step": wall / args.steps * 1e3,
           "stage_states_per_step_per_env": (br.n_calcxd_states - c0) / (n_env * args.steps),
           "jacobian_chunks_per_step_per_env": (br.n_chunk_states - j0) / (n_env * args.steps),
           "newton_attempt_rounds_per_step": (br.n_attempts - a0) / args.steps,
           "device_ms": {"jacobian_8_dual6_chunks": jac_ms, "calcxd_one_stage": f3_ms, "complex_inverse_one_stage": inv_ms}, "inverse_max_residual": inv_residual,
           "sim_time_mean": float(br.t.mean()), "rule_2_fraction": float((br.rule == 2).double().mean())}
    # the same integrator on the CPU oracle, one scene on one thread (what the reference does per environment)
    mc = scene_boxes(orc.OracleContext())[0]
    dyn = D.FloatingBodyDynamics(mc)
    rr = R.makeRadauIntegrator(dyn, S.num_x(mc), 1.0e-16, 2, 6)
    rr.step.h_max = 0.05
    t0 = time.perf_counter()
    R.integrate_radau(rr, x0[0], t_final=1e9, max_steps=args.cpu_steps, after_step=lambda xx: D.principal_value(mc, xx))
    cpu = time.perf_counter() - t0
    out["cpu_python_mirror_env_steps_per_sec"] = args.cpu_steps / cpu
    out["cpu_oracle_contact_only_env_steps_per_sec_estimate"] = 1.0 / ((rr.n_de_float + 7 * rr.n_de_chunk) / args.cpu_steps * 60e-6)
    out["note"] = "the CPU figures are one scene on one thread: the Python mirror (dominated by interpreter overhead) and an estimate from the " \
                  "oracle's measured 60 us per contact evaluation (Dual-6 chunk ~ 7x) ignoring rigid-body and linear-algebra time"
    print(json.dumps(out))


def _card():
    import subprocess
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip()


def compare(args):
    import torch
    import pfc_b200  # noqa: F401
    from helpers import boxes_env_states, scene_boxes
    from pfc_b200 import capi
    from pfc_b200.radau_batched import BatchedRadau, DeviceBatchedRadau

    n_env, K = args.envs, args.steps
    paths = ("torch", "device") if args.impl == "both" else ("device",)
    m = scene_boxes(capi.Context(0), max_env=3 * n_env)[0]
    x0 = boxes_env_states(m, n_env)
    out = {"scene": "C3 batch of test/boxes.jl", "n_env": n_env, "h_max": 0.05, "warmup_steps": args.warmup, "timed_steps": K, "card": _card()}
    runs = {}
    for name in paths:
        r = (BatchedRadau if name == "torch" else DeviceBatchedRadau)(m, n_env, h_max=0.05)
        syncs = [0]
        if name == "torch":   # host synchronisations of the eager loop: bool() of a device tensor, nonzero(), tolist()
            real_bool, real_nonzero, real_tolist = torch.Tensor.__bool__, torch.nonzero, torch.Tensor.tolist

            def counted(f):
                def g(*a, **k):
                    syncs[0] += 1
                    return f(*a, **k)
                return g
        with torch.cuda.stream(r.stream):
            x = torch.as_tensor(x0).to(r.dev)
            for _ in range(args.warmup):
                x, _ = r.step(x)
            m.backend.sync()
            c0, a0 = (r.n_calcxd_states, r.n_attempts) if name == "torch" else (0, 0)
            hs, xs, evals, rounds = [], [], 0, 0
            if name == "torch":
                torch.Tensor.__bool__, torch.nonzero, torch.Tensor.tolist = counted(real_bool), counted(real_nonzero), counted(real_tolist)
            try:
                t0 = time.perf_counter()
                for _ in range(K):
                    x, h = r.step(x)
                    hs.append(h)
                    xs.append(x)
                    if name == "device":
                        evals = evals + r.stats[:, 3].sum(dtype=torch.int64)    # stays on the device: no read-back in the timed loop
                        _, nr, ns = m.backend.radau_step_info()
                        rounds += nr
                        syncs[0] += ns
                m.backend.sync()
                wall = time.perf_counter() - t0
            finally:
                if name == "torch":
                    torch.Tensor.__bool__, torch.nonzero, torch.Tensor.tolist = real_bool, real_nonzero, real_tolist
            rec = {"ms_per_batched_step": wall / K * 1e3, "env_steps_per_sec": n_env * K / wall,
                   "host_synchronisations_per_step": syncs[0] / K}
            if name == "torch":
                rec["stage_states_per_env_per_step"] = (r.n_calcxd_states - c0) / (n_env * K)
                rec["attempt_rounds_per_step"] = (r.n_attempts - a0) / K
            else:
                rec["stage_states_per_env_per_step"] = int(evals) / (n_env * K)
                rec["attempt_rounds_per_step"] = rounds / K
                # the time split: CUDA events between the library's phases, in a separate pass of K steps (timing on)
                m.backend.set_timing(True)
                split = np.zeros(4)
                xt = x.clone()
                for _ in range(K):
                    xt, _ = r.step(xt)
                    split += m.backend.radau_step_info()[0]
                m.backend.set_timing(False)
                rec["device_ms_per_step"] = dict(zip(("jacobian", "stage_evaluations", "inverses", "newton_and_controller"), (split / K).tolist()))
            runs[name] = (torch.stack(hs).cpu().numpy(), torch.stack(xs).cpu().numpy())
        out[name] = rec
    if len(paths) == 2:
        (h_t, x_t), (h_d, x_d) = runs["torch"], runs["device"]
        differ = (np.abs(h_d - h_t) > 1e-6 * h_t).any(axis=0)    # a different decision shows as a factor 0.1 or 2 in h
        ok = ~differ
        v_t, v_d = x_t[:, ok].reshape(K, ok.sum(), -1, 3), x_d[:, ok].reshape(K, ok.sum(), -1, 3)
        den = np.maximum(np.abs(v_t).max(axis=3), 1e-6 * np.abs(v_t).max(axis=(2, 3))[:, :, None])
        out["agreement"] = {"environments_with_different_decisions": int(differ.sum()),
                            "max_relative_state_difference_per_3_vector": float((np.abs(v_d - v_t).max(axis=3) / den).max()),
                            "max_relative_h_difference": float((np.abs(h_d - h_t) / h_t)[:, ok].max())}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
