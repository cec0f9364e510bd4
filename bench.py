#!/usr/bin/env python
"""bench.py -- contact-wrench evaluations per second on the batched-environments workload.

Workload (config C3 of BASELINE.json / SURVEY.md section 8d): 4096 independent copies of the
reference's test/boxes.jl scene (1-tet half-space + 4 boxes alternately rigid/tri and
compliant/tet, 4 regularized-friction contact instructions, quadrature rule 2) at randomized
settled-stack states (tests/helpers.py::boxes_env_states).  One "step" = one pass of the hot
path (forceAllElasticIntersections!, Float64 mode) over the whole batch; one "eval" = one
environment.  The headline at N GPUs is STRONG scaling -- the 4096 environments of BASELINE.json's configs[2] are split into
contiguous ranges of 4096 / N per GPU (pressurefieldcontact.jl_b200/parallel.py::env_range), one process and one context per GPU,
no collective on the path.  Secondary blocks of the same line: `weak` (4096 environments on every GPU) and `large_scenes` (C4 / C5:
one very large scene; at N > 1 its candidate-pair lists are split over the N GPUs and the per-instruction partial sums cross NCCL).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR also writes what the timed path returned in its last step as DIR/<name>.npy (float64; see dump_outputs): the
inputs are seeded, so two builds run with the same arguments can be compared array by array.

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (CUDA events on the
library's stream, L2 flushed between steps); `e2e` = the same metric through pfc_eval_f64 with
pinned HOST buffers (H2D + kernel + D2H inside the timed region); `roofline` = the fused kernel
against the FP64 peak measured in this process; `cpu_baseline` = the CPU oracle (a C++ port of
the reference algorithm, NOT Julia) on this box's host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOAD = "C3: {n} x test/boxes.jl environments (4 regularized-friction contact instructions each, quad rule 2), randomized settled-stack states"


def narrow_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel on this workload, from the committed
    `ncu --set full` capture of this command (profiles/narrow_tile_traffic.json, written by profiles/ncu_summary.py); None when absent."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "narrow_tile_traffic.json")))
        return int(t["dram_bytes_per_launch"]), t.get("source", "profiles/narrow_tile_traffic.json")
    except Exception:
        return None, None

METRIC = "contact_wrench_evals_per_sec"
UNIT = "evals/s"


def build_inputs(n_env, start=0):
    """Scene description (host mirror) + boundary arrays for the environments [start, start + n_env) (seeds are a function of the
    global environment index, so every partition of the batch sees the same states)."""
    import pfc_b200  # noqa: F401
    from helpers import boxes_env_states, scene_boxes, splitmix64  # noqa: F401
    from pfc_b200 import scenario as S
    m, _ = scene_boxes(None)
    x_all = boxes_env_states(m, n_env, start=start)
    X, tw, s = S.boundary_arrays(m, x_all)
    m.x_all = np.ascontiguousarray(x_all)
    return m, np.ascontiguousarray(X), np.ascontiguousarray(tw)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, local, n_total, rank=0, world=1):
    """Writes `local` (name -> this rank's rows, one per environment) as out_dir/<name>.npy in float64, the environments of all
    ranks in global order.  When the rows of all n_total environments exceed DUMP_BYTES, a fixed seeded sample of environments is
    written instead; env_index.npy always lists the environments written."""
    if world > 1:
        import torch.distributed as dist
        parts = [None] * world
        dist.all_gather_object(parts, local)
        local = {k: np.concatenate([p[k] for p in parts]) for k in local}
    if rank != 0:
        return
    per_env = 8 * (1 + sum(a[0].size for a in local.values()))
    n_keep = min(n_total, DUMP_BYTES // per_env)
    rows = np.arange(n_total) if n_keep == n_total else np.sort(np.random.default_rng(0).choice(n_total, n_keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), rows.astype(np.float64))
    for name, a in local.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a[rows], dtype=np.float64))


class ClockSampler:
    """Samples SM clocks / throttle reasons during the timed region: NVML every 2 ms (pynvml ships as nvidia-ml-py), with
    nvidia-smi polling as the fallback."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.sm, self.sm_max, self.reasons, self._stop, self._t, self.source = index, [], None, set(), threading.Event(), None, "nvml"
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._bits = {"hw_slowdown": pynvml.nvmlClocksEventReasonHwSlowdown if hasattr(pynvml, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                          "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        except Exception:
            self._nv, self.source = None, "nvidia-smi"

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nv is not None:
                    self.sm.append(float(self._nv.nvmlDeviceGetClockInfo(self._h, self._nv.NVML_CLOCK_SM)))
                    try:
                        mask = self._nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                    except Exception:
                        mask = self._nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                    for n, b in self._bits.items():
                        if mask & b:
                            self.reasons.add(n)
                    self._stop.wait(0.002)
                else:
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        r = [c.strip() for c in out.split(",")]
                        self.sm.append(float(r[0]))
                        self.sm_max = float(r[1])
                        for i, n in enumerate(self.NAMES):
                            if len(r) > 2 + i and r[2 + i].lower().startswith("active"):
                                self.reasons.add(n)
                    self._stop.wait(0.05)
            except Exception:
                self._stop.wait(0.05)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max, "reasons": [n for n in self.NAMES if n in self.reasons],
                "samples": len(sm), "source": self.source}


class _RawCuda:
    """A device pointer as a __cuda_array_interface__ object (float64 vector)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": "<f8", "data": (int(ptr), False), "version": 3}


def measure_large_scenes(device_index, rank=0, world=1):
    """Secondary numbers (not the headline): the metric's second half, candidate pairs per second, on the two single-large-scene
    configurations -- C4 (sphere on slab, tet-tet, ~2 x 100 k tets) and C5 (64-body pile, ~0.9 M candidate tri-tet pairs per
    evaluation).  Device-resident inputs, CUDA events on the library's stream, one environment, no L2 flush (the static scene is meant
    to be L2-resident).  At world > 1 the scene is SPLIT over the GPUs (pfc_set_shard + the sharded protocol of include/pfc.h): every
    rank runs the shared breadth-first levels, traverses / sorts / evaluates the sub-trees whose hash falls on it, and the per-instruction
    partial sums (8 doubles each) are all-gathered over the library's own NCCL communicator and added in rank order
    (pfc_eval_sharded_f64_device); the time is the max over ranks.  Traversal +
    compaction are reported against the measured HBM peak with SURVEY 8d's algorithmic bytes (272 B per node pair visited, 12 B per pair
    emitted)."""
    import torch
    import torch.distributed as dist
    from pfc_b200 import capi, parallel, scenes
    from pfc_b200 import scenario as S
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0)
    except Exception:
        hbm_peak = 6650.0
    out = {}
    dev = torch.device("cuda", device_index)
    for name, build in (("C4", lambda: scenes.scene_c4_sphere_on_slab(71, 79)), ("C5", lambda: scenes.scene_c5_pile(4, 24))):
        try:
            m, x = build()
            ctx = capi.Context(device_index)
            S.attach_backend(m, ctx)
            if world > 1:   # the library owns the exchange: NCCL communicator from an id handed over by rank 0
                uid = [capi.Context.comm_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(uid, src=0)
                ctx.comm_init_rank(uid[0], rank, world)
            X, tw, _ = S.boundary_arrays(m, x)
            n_ins = ctx.n_ins
            Xd, twd = torch.from_numpy(X).to(dev), torch.from_numpy(tw).to(dev)
            w = torch.zeros((1, n_ins, 6), dtype=torch.float64, device=dev)
            npairs = torch.zeros((1, n_ins), dtype=torch.int64, device=dev)
            fl = torch.zeros((1, n_ins), dtype=torch.int32, device=dev)
            stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
            if world > 1:
                def step():
                    ctx.eval_sharded_f64_device(1, Xd.data_ptr(), twd.data_ptr(), None, w.data_ptr(), None, npairs.data_ptr(), fl.data_ptr())
            else:
                def step():
                    ctx.eval_f64_device(1, Xd.data_ptr(), twd.data_ptr(), None, w.data_ptr(), None, npairs.data_ptr(), fl.data_ptr())
            for _ in range(3):
                step()
            ctx.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0, reps = ctx.launch_count(), 10
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0.record(stream)
            for _ in range(reps):
                step()
            e1.record(stream)
            ctx.sync()
            ms = e0.elapsed_time(e1) / reps
            n_tests, n_listed = ctx.counters()
            counts = torch.tensor([float(ms), float(n_tests), float(n_listed)], dtype=torch.float64, device=dev)
            ms_min = ms
            if world > 1:
                mx = counts.clone()
                dist.all_reduce(mx, op=dist.ReduceOp.MAX)
                mn = counts.clone()
                dist.all_reduce(mn, op=dist.ReduceOp.MIN)
                dist.all_reduce(counts, op=dist.ReduceOp.SUM)
                ms, ms_min = float(mx[0]), float(mn[0])
                n_tests, n_listed = int(counts[1]), int(counts[2])
            n_pairs = int(npairs.sum().item())   # after the exchange every rank holds the full counts
            gbs = (272 * n_tests + 12 * n_listed) / (ms * 1e-3) * 1e-9
            out[name] = {"ms_per_eval": ms, "n_gpus": world, "candidate_pairs": n_pairs, "node_pairs_tested": int(n_tests), "instructions": n_ins,
                         "candidate_pairs_per_sec": n_pairs / (ms * 1e-3), "contacts": int((fl.cpu().numpy() & 1).sum()),
                         "kernel_launches_per_eval": int((ctx.launch_count() - l0) // reps),
                         "broad_phase_roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak * world, "unit": "GB/s", "frac": gbs / (hbm_peak * world),
                                                  "bytes": "272 B per node pair visited + 12 B per pair emitted (SURVEY 8d), summed over the ranks; the scene is L2-resident"}}
            if world > 1:
                out[name].update({"split": "hash-partitioned sub-trees of the dual-tree recursion, disjoint pair lists", "exchanges_per_eval": 1,
                                  "collective": "library-owned NCCL communicator (pfc_comm_init_rank): all-gather of 8 doubles per large instruction + rank-order sum, on the library's stream",
                                  "ms_fastest_rank": ms_min, "timing": "CUDA events on each rank's stream, max over ranks"})
            ctx.close()
        except Exception as exc:   # secondary measurement: never take the headline down with it
            out[name] = {"error": repr(exc)}
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference is Julia
    (not installable here, no Julia in the image), so this arm times the CPU oracle -- a literal C++
    port of the same algorithm -- with all host threads, on the same workload (every step = all environments), metric and unit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import orc
    from pfc_b200 import scenario as S
    n_env = args.envs
    m, X, tw = build_inputs(n_env)
    cores = orc.lib().orc_max_threads()
    ctx = orc.OracleContext(n_threads=cores)
    S.attach_backend(m, ctx)
    for _ in range(args.warmup):
        ctx.eval_f64(X, tw)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = ctx.eval_f64(X, tw)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: out[k] for k in ("wrench", "n_pairs", "flags")}, n_env)
    v = n_env * args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": WORKLOAD.format(n=n_env), "envs": n_env, "instructions_per_env": 4},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"all {n_env} environments per step, {args.steps} steps, {cores} threads; C++ port of the Julia reference (Julia is not in the image; "
                                   "the reference itself is single-threaded)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--envs", type=int, default=4096, help="environments of the whole job (split over the GPUs)")
    ap.add_argument("--impl", default="pfc", choices=["pfc", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-large", action="store_true", help="skip the secondary single-large-scene measurements (C4 / C5)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (bench_outputs/ is git-ignored)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the contact-wrench path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from pfc_b200 import capi, parallel
    from pfc_b200 import scenario as S

    n_total = args.envs
    lo, hi = parallel.env_range(n_total, rank, world)   # strong scaling: this rank's contiguous range of the job's environments
    n_env = hi - lo
    m, X_h, tw_h = build_inputs(n_env, lo)
    ctx = capi.Context(local_rank)
    S.attach_backend(m, ctx, max_env=n_total)
    n_ins = ctx.n_ins
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    # device-resident buffers
    X_d = torch.from_numpy(X_h).to(dev)
    tw_d = torch.from_numpy(tw_h).to(dev)
    w_d = torch.zeros((n_env, n_ins, 6), dtype=torch.float64, device=dev)
    np_d = torch.zeros((n_env, n_ins), dtype=torch.int64, device=dev)
    fl_d = torch.zeros((n_env, n_ins), dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    torch.cuda.synchronize()

    def step_device():
        ctx.eval_f64_device(n_env, X_d.data_ptr(), tw_d.data_ptr(), None, w_d.data_ptr(), None, np_d.data_ptr(), fl_d.data_ptr())

    # pinned host buffers for the end-to-end leg
    X_p = torch.from_numpy(X_h).pin_memory()
    tw_p = torch.from_numpy(tw_h).pin_memory()
    w_p = torch.zeros((n_env, n_ins, 6), dtype=torch.float64).pin_memory()
    np_p = torch.zeros((n_env, n_ins), dtype=torch.int64).pin_memory()
    fl_p = torch.zeros((n_env, n_ins), dtype=torch.int32).pin_memory()

    def step_e2e_boundary():
        ctx.eval_f64_ptr(n_env, X_p.data_ptr(), tw_p.data_ptr(), None, w_p.data_ptr(), None, np_p.data_ptr(), fl_p.data_ptr())

    # state-level entry point: raw states in, generalized forces out (kinematics prologue and J' w epilogue on the device)
    x_p = torch.from_numpy(m.x_all).pin_memory()
    f_p = torch.zeros((n_env, m.nv), dtype=torch.float64).pin_memory()

    def step_e2e():
        # the result a caller of forceAllElasticIntersections! gets back is f_generalized; pair counts / flags are debug outputs (not requested)
        ctx.eval_state_f64_ptr(n_env, x_p.data_ptr(), f_p.data_ptr(), None, None, None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with ClockSampler(local_rank) as peak_clocks:
        fp64_peak = ctx.measure_fp64_peak()
        ctx.sync()
    peak_clock = peak_clocks.summary()["sm_mhz"]

    for _ in range(max(args.warmup, 3)):
        step_device()
        step_e2e()
        step_e2e_boundary()
    ctx.sync()

    # ---- timed region 1: device-resident, CUDA events on the library's stream, L2 flushed between steps ----
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches0 = ctx.launch_count()
    barrier()
    with ClockSampler(local_rank) as clocks:
        for k in range(args.steps):
            with torch.cuda.stream(stream):
                flush.zero_()
            ev0[k].record(stream)
            step_device()
            ev1[k].record(stream)
        barrier()
        launches = ctx.launch_count() - launches0
        dev_ms = sum(a.elapsed_time(b) for a, b in zip(ev0, ev1))
        # the last timed step's results, before the per-kernel split below runs the path again
        last = {"wrench": w_d.cpu().numpy(), "n_pairs": np_d.cpu().numpy(), "flags": fl_d.cpu().numpy()} if args.dump_outputs else None
        # ---- timed region 2: end to end through pfc_eval_f64 with pinned host buffers (wall clock; the call is synchronous) ----
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            step_e2e()
        e2e_s = time.perf_counter() - t0
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            step_e2e_boundary()
        e2e_b_s = time.perf_counter() - t0
        barrier()
    # per-kernel split (outside the timed regions): CUDA events recorded by the library between its two kernels
    ctx.set_timing(True)
    split = []
    for _ in range(5):
        with torch.cuda.stream(stream):
            flush.zero_()
        step_device()
        split.append(ctx.kernel_times())
    ctx.set_timing(False)
    broad_ms = float(np.median([a for a, _ in split]))
    narrow_ms = float(np.median([b for _, b in split]))
    if world > 1:
        t = torch.tensor([dev_ms, e2e_s, e2e_b_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_s, e2e_b_s = float(t[0]), float(t[1]), float(t[2])

    # ---- secondary, N > 1: weak scaling (every GPU its own n_total environments; independent processes, no collective) ----
    weak = None
    if world > 1:
        _, Xw_h, tww_h = build_inputs(n_total, rank * n_total)
        Xw, tww = torch.from_numpy(Xw_h).to(dev), torch.from_numpy(tww_h).to(dev)
        ww = torch.zeros((n_total, n_ins, 6), dtype=torch.float64, device=dev)
        npw = torch.zeros((n_total, n_ins), dtype=torch.int64, device=dev)
        flw = torch.zeros((n_total, n_ins), dtype=torch.int32, device=dev)
        step_w = lambda: ctx.eval_f64_device(n_total, Xw.data_ptr(), tww.data_ptr(), None, ww.data_ptr(), None, npw.data_ptr(), flw.data_ptr())
        for _ in range(3):
            step_w()
        n_w = max(args.steps // 4, 10)
        w0 = [torch.cuda.Event(enable_timing=True) for _ in range(n_w)]
        w1 = [torch.cuda.Event(enable_timing=True) for _ in range(n_w)]
        barrier()
        for k in range(n_w):
            with torch.cuda.stream(stream):
                flush.zero_()
            w0[k].record(stream)
            step_w()
            w1[k].record(stream)
        barrier()
        tw_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in zip(w0, w1))], dtype=torch.float64, device=dev)
        dist.all_reduce(tw_ms, op=dist.ReduceOp.MAX)
        weak = {"value": n_total * world * n_w / (float(tw_ms[0]) * 1e-3), "unit": UNIT, "scaling": "weak", "envs_per_gpu": n_total, "steps": n_w,
                "ms_per_step": float(tw_ms[0]) / n_w, "what": "device-resident, every GPU its own batch of the full size; no collective"}
        del Xw, tww, ww, npw, flw

    # correctness guard: the timed outputs are real (contacts found, finite wrench)
    w_host = w_d.cpu().numpy()
    assert np.isfinite(w_host).all() and int((fl_d.cpu().numpy() & 1).sum()) > n_env, "benchmark produced no contact work"
    assert np.array_equal(w_host, w_p.numpy()), "device-resident and host-pointer entry points disagree"
    f_chk = S.generalized_forces(m, m.x_all[0], w_host[0])
    assert np.abs(f_p.numpy()[0] - f_chk).max() <= 1e-9 * max(np.abs(f_chk).max(), 1e-300), "state-level entry point disagrees with J' w on the host"
    if args.dump_outputs:   # f_p still holds the last step of timed region 2's state-level leg
        dump_outputs(args.dump_outputs, dict(last, f_generalized=f_p.numpy()), n_total, rank, world)

    # secondary: one very large scene (C4 / C5); at N > 1 split over the GPUs with an NCCL exchange of the partial sums (all ranks take part)
    large = None if args.no_large else measure_large_scenes(local_rank, rank, world)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    evals = n_total * args.steps
    value = evals / (dev_ms * 1e-3)
    ms_per_step = dev_ms / args.steps

    # ---- algorithmic work (instrumented oracle, counted on a sample) + CPU baseline ----
    from oracle import orc
    octx = orc.OracleContext(n_threads=1)
    S.attach_backend(m, octx)
    n_count = min(n_env, 512)
    work = octx.count_work(X_h[:n_count], tw_h[:n_count])
    flops_per_eval = (work["flops_broad"] + work["flops_narrow"]) / n_count
    pairs_per_eval = work["candidate_pairs"] / n_count
    node_pairs_per_eval = work["node_pairs"] / n_count
    achieved_tflops = flops_per_eval * n_env / (ms_per_step * 1e-3) * 1e-12
    narrow_tflops = work["flops_narrow"] / n_count * n_env / (narrow_ms * 1e-3) * 1e-12
    broad_tflops = work["flops_broad"] / n_count * n_env / (broad_ms * 1e-3) * 1e-12
    bytes_per_eval = n_ins * (16 + 6 + 6) * 8 + n_ins * 12  # boundary arrays in + wrench, n_pairs, flags out
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)

    cpu_baseline = None
    if world == 1:   # timed on rank 0 at N = 1 only
        cpu_sample = min(n_env, 1024)
        t0 = time.perf_counter()
        cpu_reps = 0
        while True:
            octx.eval_f64(X_h[:cpu_sample], tw_h[:cpu_sample])
            cpu_reps += 1
            if time.perf_counter() - t0 > args.cpu_seconds or cpu_reps >= 200:
                break
        cpu_1 = cpu_sample * cpu_reps / (time.perf_counter() - t0)
        cores = orc.lib().orc_max_threads()
        octx_mt = orc.OracleContext(n_threads=cores)
        S.attach_backend(m, octx_mt)
        octx_mt.eval_f64(X_h, tw_h)
        t0 = time.perf_counter()
        for _ in range(3):
            octx_mt.eval_f64(X_h, tw_h)
        cpu_mt = n_env * 3 / (time.perf_counter() - t0)
        cpu_baseline = {"value": cpu_1, "unit": UNIT, "cores": 1, "kind": "port",
                        "sample": f"{cpu_sample} of the {n_env} environments x {cpu_reps} repetitions, single thread (the reference is single-threaded); "
                                  "C++ port of the Julia reference, not Julia",
                        "all_cores": {"value": cpu_mt, "cores": cores, "sample": f"all {n_env} environments x 3 repetitions"}}

    h2d = int(m.x_all.nbytes)
    d2h = int(f_p.numel() * 8 + 4)   # generalized forces + the 4-byte error status word
    h2d_b = int(X_h.nbytes + tw_h.nbytes)
    d2h_b = int(w_p.numel() * 8 + np_p.numel() * 8 + fl_p.numel() * 4)
    # secondary: the Jacobian mode the integrator needs once per step (SURVEY 8d "Jacobian-chunk evals/s"): the WHOLE Jacobian of calcXd!
    # for the batch through pfc_calcxd_jacobian_device (one broad phase, all ceil(n_x / 6) Dual-6 chunks side by side), device buffers,
    # timed with CUDA events; beside it the same Jacobian as ceil(n_x / 6) calls of pfc_calcxd_dual6_device (what round 1 did)
    jac = None
    try:
        if getattr(m, "device_dynamics", False) and world == 1:
            nx = m.x_all.shape[1]
            n_chunk = int(np.ceil(nx / 6))
            x_d = torch.from_numpy(m.x_all).to(dev)
            jac_d = torch.empty((n_env, nx, nx), dtype=torch.float64, device=dev)
            xd_d = torch.empty((n_env, nx), dtype=torch.float64, device=dev)
            xd7_d = torch.zeros((n_env, nx, 7), dtype=torch.float64, device=dev)
            npj = torch.zeros((n_env, n_ins), dtype=torch.int64, device=dev)
            flj = torch.zeros((n_env, n_ins), dtype=torch.int32, device=dev)
            torch.cuda.synchronize(dev)   # the fills above ran on torch's stream, the library has its own
            whole = lambda: ctx.calcxd_jacobian_device(n_env, x_d.data_ptr(), None, jac_d.data_ptr(), xd_d.data_ptr(), npj.data_ptr(), flj.data_ptr())
            def chunked():
                for k in range(n_chunk):
                    ctx.calcxd_dual6_device(n_env, x_d.data_ptr(), None, 6 * k, xd7_d.data_ptr(), npj.data_ptr(), flj.data_ptr())
            times = {}
            for name, fn in (("whole", whole), ("chunk_calls", chunked)):
                fn(); ctx.sync()
                reps = 5
                t0 = time.perf_counter()
                for _ in range(reps):
                    fn()
                ctx.sync()
                times[name] = (time.perf_counter() - t0) / reps
            jac = {"value": n_env * n_chunk / times["whole"], "unit": "Dual-6 chunk evals/s", "ms_per_jacobian_batch": times["whole"] * 1e3,
                   "api": "pfc_calcxd_jacobian_device: x[env][n_x] -> jac[env][n_x][n_x] + x_dot, device buffers",
                   "chunks_per_jacobian": n_chunk, "n_x": int(nx),
                   "as_chunk_calls_ms": times["chunk_calls"] * 1e3}
    except Exception as exc:
        jac = {"error": repr(exc)}
    # secondary: the reference's own call pattern -- ONE test/boxes.jl scene per call (Radau on a single scene calls
    # forceAllElasticIntersections! once per stage evaluation): latency of pfc_eval_f64 with pageable host arrays, beside the CPU port
    latency = None
    try:
        if world == 1:
            from helpers import boxes_env_states as _bes, scene_boxes as _sb
            from pfc_b200 import scenario as _S
            lat_ctx = capi.Context(local_rank)
            m1 = _sb(lat_ctx)[0]
            X1, tw1, _ = _S.boundary_arrays(m1, _bes(m1, 1)[0])
            lat_ctx.eval_f64(X1, tw1, None)
            reps = 300
            t0 = time.perf_counter()
            for _ in range(reps):
                lat_ctx.eval_f64(X1, tw1, None)
            gpu_us = (time.perf_counter() - t0) / reps * 1e6
            o1 = orc.OracleContext(n_threads=1)
            m1c = _sb(o1)[0]
            o1.eval_f64(X1, tw1, None)
            t0 = time.perf_counter()
            for _ in range(50):
                o1.eval_f64(X1, tw1, None)
            cpu_us = (time.perf_counter() - t0) / 50 * 1e6
            latency = {"workload": "C1: one test/boxes.jl scene (settled stack) per call", "us_per_call": gpu_us, "api": "pfc_eval_f64 (host arrays, synchronous; through ctypes)",
                       "cpu_port_us_per_call": cpu_us, "cpu_port": "C++ port of the Julia reference, 1 thread"}
            del m1c
    except Exception as exc:
        latency = {"error": repr(exc)}
    # secondary: the reference's adaptive Radau IIA integrator for the whole batch with every array on the GPU (radau_batched.py)
    rollout = None
    try:
        if getattr(m, "device_dynamics", False) and not args.no_large and world == 1:
            from pfc_b200.radau_batched import BatchedRadau
            m.backend = ctx     # (the cpu_baseline leg above attached the oracle to the same scene description)
            br = BatchedRadau(m, n_env, device_index=local_rank, h_max=0.05)
            with torch.cuda.stream(br.stream):
                xb = torch.from_numpy(m.x_all).to(dev)
                for _ in range(2):
                    xb, _ = br.step(xb)
                ctx.sync()
                t0 = time.perf_counter()
                n_roll = 5
                for _ in range(n_roll):
                    xb, _ = br.step(xb)
                ctx.sync()
                dtr = (time.perf_counter() - t0) / n_roll
            rollout = {"value": n_env / dtr, "unit": "environment Radau steps/s", "ms_per_batched_step": dtr * 1e3, "envs": n_env,
                       "what": "adaptive Radau IIA (mirror of src/radau): 8 Dual-6 Jacobian chunks, per-environment complex inverses, Newton stage "
                               "evaluations through pfc_calcxd_f64_device; per-environment step-size / order control"}
    except Exception as exc:
        rollout = {"error": repr(exc)}
    traffic, traffic_src = narrow_traffic()
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(n=n_total), "envs": n_total, "instructions_per_env": n_ins, "envs_per_gpu": n_env,
                   "candidate_pairs_per_eval": pairs_per_eval, "node_pairs_per_eval": node_pairs_per_eval,
                   "l2": "256 MiB flush between timed steps",
                   "parallelism": f"contiguous environment ranges of {n_total} / {world} per GPU (one process and one context per GPU), no collective on the path"},
        "candidate_pairs_per_sec": pairs_per_eval * value,
        "e2e": {"value": evals / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s / args.steps * 1e3,
                "api": "pfc_eval_state_f64: pinned host states x[env][48] in, generalized forces f[env][24] (+ a 4-byte error status) out; "
                       "kinematics prologue and J' w epilogue on the device",
                "boundary_level": {"value": evals / e2e_b_s, "unit": UNIT, "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b,
                                   "ms_per_step": e2e_b_s / args.steps * 1e3, "api": "pfc_eval_f64: X_r2_r1 + twist in, wrenches out (host kinematics not timed)"}},
        "gpu_launches": int(launches),
        "roofline": {"bound": "fp64", "achieved": narrow_tflops, "peak": fp64_peak, "unit": "TFLOP/s",
                     "frac": narrow_tflops / fp64_peak if fp64_peak else None, "traffic": traffic if (world == 1 and n_total == 4096) else None,
                     "traffic_source": traffic_src,
                     "kernel": "narrow_tile_kernel (clip + quadrature + friction + fixed-order sums), the dominant kernel of the step",
                     "kernel_ms": narrow_ms, "kernel_share_of_step": narrow_ms / (narrow_ms + broad_ms),
                     "flops_per_launch": work["flops_narrow"] / n_count * n_env,
                     "peak_source": "DFMA micro-benchmark in this process before the timed regions (pfc_measure_fp64_peak: best of 5 bursts of 148 x 8 CTAs x 256 "
                                    "threads x 8 independent FMA chains); MEASURED_PEAKS.json has no FP64 entry", "peak_sm_mhz": peak_clock,
                     "other_kernels": {"broad_small_kernel": {"kernel_ms": broad_ms, "achieved": broad_tflops, "unit": "TFLOP/s",
                                                              "frac": broad_tflops / fp64_peak if fp64_peak else None,
                                                              "flops_per_launch": work["flops_broad"] / n_count * n_env}},
                     "whole_step": {"achieved": achieved_tflops, "frac": achieved_tflops / fp64_peak if fp64_peak else None, "flops_per_eval": flops_per_eval},
                     "hbm": {"achieved": bytes_per_eval * n_env / (ms_per_step * 1e-3) * 1e-9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": bytes_per_eval * n_env / (ms_per_step * 1e-3) * 1e-9 / hbm_peak, "bytes_per_eval": bytes_per_eval,
                             "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback"}},
        "cpu_baseline": cpu_baseline,
        "clocks": clocks.summary(),
    }
    if weak is not None:
        line["weak"] = weak
    if jac is not None:
        line["jacobian"] = jac
    if rollout is not None:
        line["batched_radau"] = rollout
    if latency is not None:
        line["latency"] = latency
    if large is not None:
        line["large_scenes"] = large
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
