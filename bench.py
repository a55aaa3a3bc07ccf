#!/usr/bin/env python
"""Benchmark of the hydrodynamic body-force path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K ...   # reference arm: the reference's CPU path

metric  = body-force updates/s (whole job, all ranks)
step    = one fused pass of the hot path over one resident batch of bodies
workload (N=1) = BASELINE config "1M heterogeneous boxes per GPU" (C3): 2^20 bodies per GPU,
          per-body coefficient records, fp32 mode, all force terms enabled.  The engine cycles
          through several independent resident batches so that consecutive steps never find
          their inputs in the 126 MB L2 (each batch is 176 MB of algorithmic traffic).
timing  = exactly K steps are timed, split into R regions (CUDA graphs, one kernel node per step)
          bracketed by CUDA events on the launch stream, barrier + synchronize around the whole
          train; per region the MAX over ranks is taken, and ``ms_per_step`` is the MEDIAN region's
          time per step (p10 / p90 and the first region are reported beside it).  The timed steps
          follow untimed back-to-back replays of the same regions (half of a >= 200-replay train
          lasting >= 100 ms), so the number is a sustained one under the power cap, not the first
          milliseconds of a cold board.
outputs = ``--dump-outputs DIR`` writes the force and torque the last timed step returned as
          DIR/force.npy and DIR/torque.npy; the inputs are seeded, so two builds run with the same
          arguments can be compared output for output.
One JSON line on stdout (rank 0).  Multi-GPU: one process per GPU under torchrun, env-sharded,
no data-path collective.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "body-force updates/sec"
UNIT = "bodies/s"
BYTES_PER_BODY_F32 = 168  # 19 state reads + 11 coefficient reads + 12 writes, fp32 (SURVEY.md 8(d))
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md
C4_ROBOTS_TOTAL, C4_BLOCK_ROBOTS, HEXAPOD = 8 * 110592, 110592, 19
DUMP_LIMIT_BYTES = 64 << 20
GRAPH_CHUNK = 120  # kernel nodes per captured graph; each graph launch costs a few us of gap on the stream
WORKLOAD = ("C3: 1M heterogeneous boxes per GPU (randomised dimensions/coefficients), per-body coefficient "
            "records, fused behaviour step, all force terms")


_STDOUT_FD = None


def claim_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line on
    stdout.  Keep a private handle on the real stdout and point fd 1 at stderr for everything else."""
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _STDOUT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_STDOUT_FD, data)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps K")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--bodies-per-gpu", type=int, default=1 << 20)
    ap.add_argument("--batches", type=int, default=6, help="independent resident batches cycled through")
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "tile", "direct"])
    ap.add_argument("--regions", type=int, default=0,
                    help="event-bracketed regions R the K timed steps are split into (0 = one per graph launch of <= 120 steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the force / torque of the last timed step (rank 0) as DIR/<name>.npy")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every step eagerly instead of graph replay")
    ap.add_argument("--no-extra", action="store_true", help="skip the C2/C4/C5/fp64 side measurements")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (used for ncu passes)")
    ap.add_argument("--cpu-sample", type=int, default=1 << 20)
    ap.add_argument("--cpu-seconds", type=float, default=8.0, help="time budget of each CPU-baseline leg")
    ap.add_argument("--ref-budget", type=float, default=150.0, help="reference arm: seconds for all its steps")
    ap.add_argument("--ref-kind", default="auto", choices=["auto", "reference", "port"])
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return args


# --------------------------------------------------------------------------------------------
def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """Per-launch DRAM bytes of the dominant kernel from the committed ncu capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the bench runs."""

    def __init__(self, index, period=0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.stop_flag, self.ok = [], False, False
        self.sm_max = None

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            self.names = {
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
            }
            self.ok = True
            while not self.stop_flag:
                t = time.perf_counter()
                clk = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                try:
                    watts = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    watts = None
                self.samples.append((t, clk, mask, watts))
                time.sleep(self.period)
        except Exception as exc:  # NVML unavailable: report that instead of inventing clocks
            self.error = repr(exc)

    def summary(self, t0, t1):
        under = [s for s in self.samples if t0 <= s[0] <= t1]
        if not self.ok or not under:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": [],
                    "note": getattr(self, "error", "no NVML samples inside the window")}
        reasons = sorted({name for s in under for bit, name in self.names.items() if s[2] & bit})
        watts = [s[3] for s in under if s[3] is not None]
        return {"sm_mhz": float(np.median([s[1] for s in under])), "sm_mhz_min": float(min(s[1] for s in under)),
                "sm_max_mhz": self.sm_max, "reasons": reasons, "samples": len(under),
                "power_w_max": max(watts) if watts else None,
                "window": "NVML samples taken while the settle passes and the timed steps ran"}


def bind_to_gpu_numa_node(gpu_index):
    """Pin this rank's CPU threads (and hence its first-touched pinned buffers) to the NUMA node of
    its GPU; with 8 ranks on one box the host side of the e2e path otherwise crosses sockets."""
    try:
        import pynvml as nv

        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(gpu_index)
        words = (os.cpu_count() + 63) // 64
        mask = nv.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def pctl(xs, q):
    return float(np.percentile(np.asarray(xs, dtype=np.float64), q))


# --------------------------------------------------------------------------------------------
# CPU legs (reported baselines, never the product path)
# --------------------------------------------------------------------------------------------
def host_threads():
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1: override it)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def f64_state(wl):
    return (wl.pos.astype(np.float64), wl.quat_xyzw.astype(np.float64), wl.lin_vel.astype(np.float64),
            wl.ang_vel.astype(np.float64), wl.prev_lin.astype(np.float64), wl.prev_ang.astype(np.float64))


def port_leg(wl, seconds, max_reps=200):
    """The oracle port (oracle/hydro_oracle.c, OpenMP over bodies) on the box's host cores."""
    from oracle import hydro_oracle as O

    nthr = host_threads()
    args = (wl.ctor_rows(), wl.masses()) + f64_state(wl) + (wl.dt,)
    O.step(*args, n_threads=nthr)  # warm-up (page faults, OpenMP pool)
    reps, t0 = 0, time.perf_counter()
    while True:
        O.step(*args, n_threads=nthr)
        reps += 1
        el = time.perf_counter() - t0
        if (el >= seconds and reps >= 3) or reps >= max_reps:
            break
    return {"value": wl.n * reps / el, "unit": UNIT, "cores": nthr, "kind": "port",
            "sample": f"{reps} passes over {wl.n} C3 bodies ({el:.1f} s), float64, C restatement of the Numba "
                      f"path + behaviour tail (oracle/hydro_oracle.c), OpenMP"}


def reference_legs(wl, seconds):
    """The UNMODIFIED reference Numba code (oracle/ref_numba.py: /root/reference live, or the bytecode
    staged in oracle/_ref) on the box's host cores, SURVEY.md 8(d):
      (2) @njit(parallel=True) prange driver over the untouched solve_hydrodynamics, all cores, plus the
          NumPy float64 behaviour tail -- the headline CPU figure;
      (1) as shipped: NumbaHydrodynamicsWrapper.calculate_hydrodynamic_forces called once per body from
          Python, 1 core, plus the same tail."""
    from oracle import ref_numba as R

    t_setup = time.perf_counter()
    cores = R.set_threads(host_threads())
    ctor = wl.ctor_rows()
    R.check_geometry(ctor)
    stepper = R.ReferenceStepper(ctor, wl.masses())
    st = f64_state(wl)
    small = min(wl.n, 4096)
    s_small = R.ReferenceStepper(ctor[:small], wl.masses()[:small])
    s_small.step(*[a[:small] for a in st], wl.dt)  # JIT (~15 s, not timed)
    t_setup = time.perf_counter() - t_setup
    reps, t0 = 0, time.perf_counter()
    while True:
        stepper.step(*st, wl.dt)
        reps += 1
        el = time.perf_counter() - t0
        if (el >= seconds and reps >= 2) or reps >= 50:
            break
    prange = {"value": wl.n * reps / el, "unit": UNIT, "cores": cores, "kind": "reference",
              "sample": f"{reps} passes over {wl.n} C3 bodies ({el:.1f} s), float64: prange driver over the untouched "
                        f"reference solve_hydrodynamics + NumPy behaviour tail; reference {R.source()}, "
                        f"JIT + geometry set-up {t_setup:.0f} s not timed"}
    # (1) as shipped: one Python call per body
    Wrapper, _ = R.load()
    m = min(wl.n, 3000)
    wr = [Wrapper(*row) for row in ctor[:m]]
    a = (st[2][:m] - st[4][:m]) / wl.dt
    al = (st[3][:m] - st[5][:m]) / wl.dt
    best = None
    for _ in range(3):
        t = time.perf_counter()
        for i in range(m):
            try:
                wr[i].calculate_hydrodynamic_forces(st[0][i], st[1][i], st[2][i], st[3][i], a[i], al[i])
            except TypeError:
                pass
        el1 = time.perf_counter() - t
        best = el1 if best is None else min(best, el1)
    prange["as_shipped_wrapper_loop"] = {"value": m / best, "unit": UNIT, "cores": 1, "kind": "reference",
                                         "sample": f"best of 3 passes over {m} bodies, one "
                                                   f"NumbaHydrodynamicsWrapper.calculate_hydrodynamic_forces call per body"}
    return prange


def cpu_baseline(sample_bodies, seconds, kind="auto"):
    from silver2_isaacsim_b200 import workloads as W

    wl = W.heterogeneous_boxes(sample_bodies)
    port = port_leg(wl, seconds)
    if kind == "port":
        return port
    try:
        from oracle import ref_numba as R

        if not R.available():
            raise RuntimeError("reference not staged (oracle/_ref) and /root/reference absent")
        ref = reference_legs(wl, seconds)
        ref["port"] = port
        return ref
    except Exception as exc:
        if kind == "reference":
            raise
        port["reference_unavailable"] = repr(exc)
        return port


def bench_config(n):
    """The workload description both arms print (the reference arm runs on this arm's config)."""
    return {"workload": WORKLOAD, "bodies_per_gpu": n,
            "l2": "inputs larger than any cache: independent resident batches cycled (176 MB of algorithmic "
                  "traffic per step each), no flush needed"}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the box's host cores, all
    host threads, on the B200 arm's config (same 2^20 C3 bodies per step).  kind "reference" = the
    unmodified Numba code (prange driver over solve_hydrodynamics + NumPy tail); falls back to the C
    port only when the reference is neither staged nor present."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from silver2_isaacsim_b200 import workloads as W

    n = args.bodies_per_gpu
    kind = args.ref_kind
    R = None
    if kind != "port":
        try:
            from oracle import ref_numba as R_

            if R_.available():
                R, kind = R_, "reference"
            elif kind == "reference":
                raise RuntimeError("reference not staged (oracle/_ref) and /root/reference absent")
        except ImportError:
            if kind == "reference":
                raise
    if R is None:
        kind = "port"
    cores = host_threads()
    # two independent batches alternate so that no step finds its inputs in a CPU cache
    wls = [W.heterogeneous_boxes(n, seed=W.SEED_BASE + 3 + b) for b in range(2)]
    if kind == "reference":
        cores = R.set_threads(cores)
        R.check_geometry(wls[0].ctor_rows())
        small = min(n, 4096)
        R.ReferenceStepper(wls[0].ctor_rows()[:small], wls[0].masses()[:small]).step(
            *[a[:small] for a in f64_state(wls[0])], wls[0].dt)  # JIT, not timed
        how = (f"prange driver over the untouched reference solve_hydrodynamics + NumPy behaviour tail "
               f"(reference {R.source()}; JIT and geometry set-up not timed)")
    else:
        how = "oracle/hydro_oracle.c (C restatement of the Numba path + tail) with OpenMP"

    def make_runner(m):
        """run(i): one behaviour step over the first m bodies of batch i % 2"""
        states = [tuple(a[:m] for a in f64_state(w)) for w in wls]
        if kind == "reference":
            steppers = [R.ReferenceStepper(w.ctor_rows()[:m], w.masses()[:m]) for w in wls]
            return lambda i: steppers[i % 2].step(*states[i % 2], wls[0].dt)
        from oracle import hydro_oracle as O

        consts = [(w.ctor_rows()[:m], w.masses()[:m]) for w in wls]
        return lambda i: O.step(*consts[i % 2], *states[i % 2], wls[0].dt, n_threads=cores)

    # calibrate on one full step, then bound the per-step sample so that W + K steps fit the budget
    run = make_runner(n)
    run(0)
    t0 = time.perf_counter()
    run(1)
    t_full = time.perf_counter() - t0
    warm = max(0, min(args.warmup, 3) - 2)
    sample = n
    if t_full * (warm + args.steps) > args.ref_budget:
        sample = max(4096, int(n * args.ref_budget / (t_full * (warm + args.steps))) // 4096 * 4096)
        run = make_runner(sample)
        run(0)
    for i in range(warm):
        run(i)
    times = []
    for i in range(args.steps):
        t = time.perf_counter()
        run(i)
        times.append(time.perf_counter() - t)
    el = float(sum(times))
    value = sample * args.steps / el
    desc = (f"{args.steps} steps x {sample} C3 bodies" + ("" if sample == n else f" (bounded sample of the {n}-body batch)")
            + f", float64, {how}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(n),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "extra": {"bodies_per_step": sample, "host_threads": cores, "ms_per_step_median": 1e3 * pctl(times, 50),
                  "ms_per_step_p10": 1e3 * pctl(times, 10), "ms_per_step_p90": 1e3 * pctl(times, 90)},
    }
    emit(line)


# --------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------
def make_batches(torch, W, n, n_batches, dtype, dev, seed0):
    """Independent resident batches of the C3 workload (state tensors per batch; one engine each)."""
    from silver2_isaacsim_b200 import HydroEngine

    batches = []
    npdt = np.float32 if dtype == torch.float32 else np.float64
    for b in range(n_batches):
        wl = W.heterogeneous_boxes(n, seed=seed0 + b, dtype=np.float32)
        eng = HydroEngine(n, dtype=dtype, device=dev)
        eng.set_workload_params(wl)
        t = lambda a: torch.as_tensor(np.ascontiguousarray(a.astype(npdt)), device=dev)
        eng.set_prev(t(wl.prev_lin), t(wl.prev_ang))
        F, T = eng.bind(t(wl.pos), t(wl.quat_xyzw), t(wl.lin_vel), t(wl.ang_vel))
        batches.append((eng, wl, F, T))
    return batches


class RegionTimer:
    """Back-to-back regions, an event between consecutive regions, barrier + synchronize on both sides
    of the train; per region the max over ranks.  ``lead`` is launched untimed right before the first
    event, with no gap between it and the timed regions."""

    def __init__(self, torch, sharding, dev):
        self.torch, self.sharding, self.dev = torch, sharding, dev

    def run(self, region_fns, lead=None):
        torch = self.torch
        regions = len(region_fns)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(regions + 1)]
        torch.cuda.synchronize(self.dev)
        self.sharding.barrier()
        torch.cuda.synchronize(self.dev)
        w0 = time.perf_counter()
        if lead is not None:
            lead()
        ev[0].record()
        for r, region_fn in enumerate(region_fns):
            region_fn()
            ev[r + 1].record()
        torch.cuda.synchronize(self.dev)
        w1 = time.perf_counter()
        self.sharding.barrier()
        ms = np.array([ev[r].elapsed_time(ev[r + 1]) for r in range(regions)], dtype=np.float64)
        return self.sharding.max_over_ranks_vec(ms, self.dev), (w0, w1)

    def run_spaced(self, region_fn, regions, idle_s):
        """The same K-step region timed `regions` times with the GPU left idle for `idle_s` before each one (events
        bracket every region on its own): the board stays below its power cap, so this is the kernel at its
        nominal clock -- how it runs inside a simulation step rather than in a back-to-back benchmark loop."""
        torch = self.torch
        ms = []
        for _ in range(regions):
            torch.cuda.synchronize(self.dev)
            time.sleep(idle_s)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            region_fn()
            e1.record()
            torch.cuda.synchronize(self.dev)
            ms.append(e0.elapsed_time(e1))
        self.sharding.barrier()
        return self.sharding.max_over_ranks_vec(np.array(ms, dtype=np.float64), self.dev)


def build_step_regions(torch, step_fns, steps, regions, dev, use_graph=True, chunk=GRAPH_CHUNK):
    """`regions` callables that together launch EXACTLY `steps` steps, step i being step_fns[i % len(step_fns)]:
    region r launches steps bounds[r] .. bounds[r + 1] - 1, replayed from captured CUDA graphs (one kernel
    node per step) unless use_graph is False.  Returns (callables, steps per region, description)."""
    nb = len(step_fns)
    bounds = [steps * r // regions for r in range(regions + 1)]
    counts = np.diff(bounds)
    if not use_graph:
        def eager(a, b):
            def run():
                for i in range(a, b):
                    step_fns[i % nb]()
            return run
        return [eager(bounds[r], bounds[r + 1]) for r in range(regions)], counts, f"{steps} eager launches"
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for fn in step_fns:
            fn()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    chunk = max(nb, chunk // nb * nb)
    graphs = {}
    fns, launches = [], 0
    for r in range(regions):
        plan, done = [], bounds[r]
        while done < bounds[r + 1]:
            cnt = min(chunk, bounds[r + 1] - done)
            key = (done % nb, cnt)
            if key not in graphs:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):
                    for i in range(cnt):
                        step_fns[(done + i) % nb]()
                graphs[key] = g
            plan.append(graphs[key])
            done += cnt
        launches += len(plan)

        def replay(plan=plan):
            for g in plan:
                g.replay()
        fns.append(replay)
    for fn in fns:  # one untimed pass
        fn()
    torch.cuda.synchronize(dev)
    return fns, counts, (f"CUDA graph replay ({launches} graph launch(es) of <= {chunk} kernel nodes for {steps} steps "
                         f"in {regions} region(s))")


def build_step_region(torch, step_fns, steps, dev, use_graph=True, chunk=GRAPH_CHUNK):
    """A callable that launches EXACTLY `steps` steps (cycling through step_fns): build_step_regions with one region."""
    fns, _, mode = build_step_regions(torch, step_fns, steps, 1, dev, use_graph, chunk)
    return fns[0], mode


def settle_lead(region_fns, steps, est_ms_per_step):
    """(callable, passes): untimed passes over all regions, launched right before the timed steps.  A train of
    >= 200 passes (>= 20 when K > 200, <= 2000) lasting >= 100 ms by the estimate brings the board to its power
    cap; the timed steps take the place of its middle pass, so the number is a sustained one and comparable with
    the medians of such trains in the bench lines under profiles/."""
    train = int(np.ceil(100.0 / max(1e-6, steps * est_ms_per_step)))
    passes = int(min(2000, max(200 if steps <= 200 else 20, train))) // 2

    def lead():
        for _ in range(passes):
            for fn in region_fns:
                fn()
    return lead, passes


def dump_outputs(out_dir, arrays, limit_bytes=DUMP_LIMIT_BYTES, seed=0):
    """Write each (n, ...) array as out_dir/<name>.npy (float32 / float64 as computed).  When all of them
    together exceed limit_bytes, the same fixed, seeded sample of rows is written from each."""
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    rows = None
    if n * row_bytes > limit_bytes:
        rows = np.sort(np.random.default_rng(seed).choice(n, limit_bytes // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a if rows is None else a[rows])
    return {"dir": out_dir, "files": sorted(k + ".npy" for k in arrays), "bodies": n,
            "rows": "all" if rows is None else f"{len(rows)} rows sampled with numpy default_rng({seed})"}


def parity_sample(torch, oracle_mod, scoring, eng_factory, wl, dev, sample=1 << 16):
    """Score a sample of this rank's own shard against the float64 oracle (outside any timed region)."""
    ns = min(sample, wl.n)
    sl = slice(0, ns)
    eng = eng_factory(ns)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a[sl], dtype=np.float32), device=dev)
    eng.set_params_per_body(wl.coeff_per_body()[sl])
    eng.set_prev(t(wl.prev_lin), t(wl.prev_ang))
    eng.set_kernel("tile")
    F, T = eng.step(t(wl.pos), t(wl.quat_xyzw), t(wl.lin_vel), t(wl.ang_vel), wl.dt)
    torch.cuda.synchronize(dev)
    ref = oracle_mod.step(wl.ctor_rows()[sl], wl.masses()[sl], wl.pos[sl], wl.quat_xyzw[sl], wl.lin_vel[sl],
                          wl.ang_vel[sl], wl.prev_lin[sl], wl.prev_ang[sl], wl.dt)
    out = {}
    worst = 0.0
    for name, x, y in (("F", F, ref.force), ("T", T, ref.torque)):
        err, den = scoring.vec_err(x.double().cpu().numpy(), y)
        tol = np.maximum(scoring.FP32_REL * den, scoring.FP32_ABS)
        out["pass_" + name] = float((err <= tol).mean())
        worst = max(worst, float((err / tol).max()))
    out["worst_x_tol"] = worst
    out["bodies"] = ns
    out["kernel"] = eng.last_kernel
    return out


def c4_strong_leg(torch, sharding, W, dev, rank, world, timer, steps):
    """BASELINE config 4 on ALL ranks: 884 736 hexapods x 19 = 16 809 984 bodies in total, robot-contiguous
    shards (strong scaling: the total is fixed), per-body records with +-20 % per-robot jitter, per-robot
    wrench.  Each rank's shard is built on the device from one 110 592-robot host block repeated with
    shifted xy positions (the values do not change the traffic); the first block is scored against the oracle."""
    from oracle import hydro_oracle as O
    from silver2_isaacsim_b200 import HydroEngine
    from tests import scoring

    sh = sharding.shard_robots(C4_ROBOTS_TOTAL, HEXAPOD, world, rank)
    block = W.sharded_robots(C4_BLOCK_ROBOTS, seed=W.SEED_BASE + 40 + rank)
    reps = -(-sh.n_robots // C4_BLOCK_ROBOTS)
    n = sh.n_bodies

    def tile(a, shift=False):
        t = torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32), device=dev)
        if reps > 1:
            parts = []
            for k in range(reps):
                p = t.clone()
                if shift and k:
                    p[:, 0] += 3.0 * k
                parts.append(p)
            t = torch.cat(parts)
        return t[:n].contiguous()

    eng = HydroEngine(n, device=dev)
    eng.set_globals(block.rho, block.g)
    eng.set_params_per_body(tile(block.coeff_per_body()))
    eng.set_articulation(HEXAPOD)
    eng.set_prev(tile(block.prev_lin), tile(block.prev_ang))
    F, T, Wr = eng.bind(tile(block.pos, True), tile(block.quat_xyzw), tile(block.lin_vel), tile(block.ang_vel),
                        robot_wrench=True)
    dt = block.dt
    eng.step_bound(dt)  # first step: v_prev as generated -> the scored one
    torch.cuda.synchronize(dev)
    ns = min(1 << 16, C4_BLOCK_ROBOTS, sh.n_robots) * HEXAPOD
    ref = O.step(block.ctor_rows()[:ns], block.masses()[:ns], block.pos[:ns], block.quat_xyzw[:ns], block.lin_vel[:ns],
                 block.ang_vel[:ns], block.prev_lin[:ns].copy(), block.prev_ang[:ns].copy(), dt,
                 n_threads=max(1, host_threads() // world))
    okF = scoring.fp32_ok(F[:ns].double().cpu().numpy(), ref.force)
    okT = scoring.fp32_ok(T[:ns].double().cpu().numpy(), ref.torque)
    refw = O.robot_wrench(block.pos[:ns].astype(np.float64), ref.force, ref.torque, HEXAPOD)
    magw = O.robot_wrench(block.pos[:ns].astype(np.float64), np.abs(ref.force), np.abs(ref.torque), HEXAPOD)
    w = Wr[:ns // HEXAPOD].double().cpu().numpy()
    okW = np.abs(w - refw).max(axis=1) <= 1e-5 * np.abs(magw).max(axis=1) + 1e-6
    kernel = eng.last_kernel
    region, mode = build_step_region(torch, [lambda: eng.step_bound(dt)], steps, dev)
    est = n * (BYTES_PER_BODY_F32 + 24.0 / HEXAPOD) / 6.0e12 * 1e3
    regions = int(min(200, max(10, np.ceil(100.0 / (steps * est)))))
    ms, _ = timer.run([region] * regions)
    total = sharding.sum_over_ranks(float(n), dev)
    frac = lambda ok: sharding.sum_over_ranks(float(ok.sum()), dev) / sharding.sum_over_ranks(float(ok.size), dev)
    pF, pT, pW = frac(okF), frac(okT), frac(okW)
    med = pctl(ms, 50) / steps
    bpb = BYTES_PER_BODY_F32 + 24.0 / HEXAPOD
    del eng, F, T, Wr
    torch.cuda.empty_cache()
    return {"config": "C4 strong scaling: 884 736 hexapods (16 809 984 bodies) sharded over the ranks, per-body "
                      "records, per-robot wrench", "n_gpus": world, "bodies_total": int(total), "bodies_per_gpu": n,
            "us_per_step": 1e3 * med, "us_per_step_p10": 1e3 * pctl(ms, 10) / steps,
            "us_per_step_p90": 1e3 * pctl(ms, 90) / steps, "updates_per_s": total / (med * 1e-3),
            "achieved_gbs_per_gpu": n * bpb / (med * 1e-3) / 1e9, "regions": regions, "steps_per_region": steps,
            "kernel": kernel, "launch": mode,
            "parity_sample": {"robots_per_gpu": ns // HEXAPOD, "pass_F": pF, "pass_T": pT, "pass_robot_wrench": pW}}


def platform_ceiling(torch, sharding, n, esz, dev, steps=10, regions=8):
    """What this box's host link gives the e2e pattern with NO engine in the way: per step one plain
    pinned cudaMemcpyAsync of 13 scalars/body host->device and one of 6 scalars/body device->host, on two
    streams concurrently, all ranks at once.  The e2e figure can at best equal it."""
    hin = torch.empty(n * 13 * esz, dtype=torch.uint8).pin_memory()
    hout = torch.empty(n * 6 * esz, dtype=torch.uint8).pin_memory()
    din = torch.empty(n * 13 * esz, dtype=torch.uint8, device=dev)
    dout = torch.empty(n * 6 * esz, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def one():
        with torch.cuda.stream(s1):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s2):
            hout.copy_(dout, non_blocking=True)
    for _ in range(3):
        one()
    torch.cuda.synchronize(dev)
    sharding.barrier()
    times = []
    for _ in range(regions):
        t0 = time.perf_counter()
        for _ in range(steps):
            one()
        torch.cuda.synchronize(dev)
        times.append(time.perf_counter() - t0)
    sharding.barrier()
    t = sharding.max_over_ranks(pctl(times, 50), dev)
    total = sharding.sum_over_ranks(float(n), dev)
    return {"value": total * steps / t, "unit": UNIT, "h2d_gbs_per_gpu": n * 13 * esz * steps / t / 1e9,
            "d2h_gbs_per_gpu": n * 6 * esz * steps / t / 1e9,
            "how": "median of %d x %d steps: concurrent pinned cudaMemcpyAsync H2D (13 scalars/body) + D2H (6 scalars/body), "
                   "all ranks at once, no kernel" % (regions, steps)}


def side_measurements(torch, W, dev, dtype_main):
    """Rank 0 only: C2 (hexapod x 4096, table + robot wrench; eager and graph replay), C5 (per-step
    launch vs graph vs persistent rollout), C4 8-GPU shard, C3 at 4x, fp64 C3."""
    from silver2_isaacsim_b200 import HydroEngine

    out = {}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def bound_engine(wl, dtype, robot):
        npdt = np.float32 if dtype == torch.float32 else np.float64
        e = HydroEngine(wl.n, dtype=dtype, device=dev)
        e.set_workload_params(wl)
        t = lambda a: torch.as_tensor(np.ascontiguousarray(a.astype(npdt)), device=dev)
        e.set_prev(t(wl.prev_lin), t(wl.prev_ang))
        e.bind(t(wl.pos), t(wl.quat_xyzw), t(wl.lin_vel), t(wl.ang_vel), robot_wrench=robot)
        return e

    def timeit(fn, reps, rounds=5):
        """median over `rounds` of the mean time of `reps` calls (ms)"""
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(rounds):
            ev0.record()
            for _ in range(reps):
                fn()
            ev1.record()
            torch.cuda.synchronize(dev)
            ts.append(ev0.elapsed_time(ev1) / reps)
        return pctl(ts, 50)

    # C2: 4096 envs x 19 bodies, part-type table in shared memory, per-robot wrench
    wl = W.hexapod_envs(4096)
    e = bound_engine(wl, torch.float32, True)
    ms = timeit(lambda: e.step_bound(wl.dt), 200)
    bytes2 = (124.0 + 24.0 / HEXAPOD) * wl.n
    c2 = {"bodies": wl.n, "us_per_step_eager": 1e3 * ms, "kernel": e.last_kernel,
          "note": "L2-resident (9.7 MB of traffic per step): latency-bound, not HBM-bound"}
    e.capture_rollout(200, wl.dt)
    msg = timeit(e.launch_rollout, 1, rounds=9) / 200
    c2.update({"us_per_step_graph": 1e3 * msg, "updates_per_s": wl.n / (msg * 1e-3),
               "achieved_gbs": bytes2 / (msg * 1e-3) / 1e9, "algorithmic_bytes_per_body": 124.0 + 24.0 / HEXAPOD})
    out["c2_hexapod_4096_envs"] = c2
    del e
    # C4 per-GPU shard at 8 GPUs: 110 592 robots x 19 bodies, per-body records, per-robot wrench
    wl4 = W.sharded_robots(C4_BLOCK_ROBOTS)
    e4a = bound_engine(wl4, torch.float32, True)
    e4b = bound_engine(W.sharded_robots(C4_BLOCK_ROBOTS, seed=W.SEED_BASE + 44), torch.float32, True)
    k4s = [0]

    def f4s():
        (e4a if k4s[0] % 2 == 0 else e4b).step_bound(wl4.dt)
        k4s[0] += 1
    ms = timeit(f4s, 100)
    bytes4 = (BYTES_PER_BODY_F32 + 24.0 / HEXAPOD) * wl4.n
    out["c4_shard_110592_robots"] = {"bodies": wl4.n, "us_per_step": 1e3 * ms, "updates_per_s": wl4.n / (ms * 1e-3),
                                     "achieved_gbs": bytes4 / (ms * 1e-3) / 1e9, "kernel": e4a.last_kernel,
                                     "note": "2 batches alternated, eager launches"}
    del e4a, e4b
    # C5: 1024 bodies, 1000-step rollout: per-step launches vs one captured CUDA graph vs one persistent kernel
    wl5 = W.uniform_small_batch(1024)
    e5 = bound_engine(wl5, torch.float32, False)
    ms_eager = timeit(lambda: [e5.step_bound(wl5.dt) for _ in range(1000)], 1, rounds=3)
    e5.capture_rollout(1000, wl5.dt)
    ms_graph = timeit(e5.launch_rollout, 1, rounds=5)
    c5 = {"us_per_step_launch": ms_eager, "us_per_step_graph": ms_graph, "ratio": ms_eager / ms_graph,
          "state": "static (force-only rollout)"}
    if hasattr(e5, "rollout_persistent"):
        try:
            e5.set_rollout_mode(free_bodies=True, gravity=wl5.g)
            ms_eager_fb = timeit(lambda: e5_free_eager(e5, wl5, 1000), 1, rounds=3)
            e5.capture_rollout(1000, wl5.dt)
            ms_graph_fb = timeit(e5.launch_rollout, 1, rounds=5)
            ms_pers = timeit(lambda: e5.rollout_persistent(1000, wl5.dt, gravity=wl5.g), 1, rounds=5)
            c5["free_bodies"] = {"us_per_step_launch": ms_eager_fb, "us_per_step_graph": ms_graph_fb,
                                 "us_per_step_persistent_kernel": ms_pers,
                                 "note": "force step + semi-implicit Euler per step; persistent = one launch for all 1000 steps"}
        except Exception as exc:
            c5["free_bodies"] = {"error": repr(exc)}
    out["c5_small_batch_1024x1000"] = c5
    del e5
    if dtype_main == torch.float32:
        # the headline workload with strict mode off (flagged bodies keep their fp32 result): what the
        # float64 re-evaluation costs, and what it buys (parity of the same sample, both ways)
        from oracle import hydro_oracle as O
        from tests import scoring
        n = 1 << 20
        bs = make_batches(torch, W, n, 6, torch.float32, dev, W.SEED_BASE + 3)
        res = {}
        for strict in (True, False):
            for b in bs:
                b[0].set_strict(strict)
            region, _ = build_step_region(torch, [(lambda b=b: b[0].step_bound(b[1].dt)) for b in bs], 24, dev)
            ms = timeit(region, 1, rounds=41) / 24
            eng_p = lambda m, strict=strict: _with(HydroEngine(m, dtype=torch.float32, device=dev), lambda e: e.set_strict(strict))
            par = parity_sample(torch, O, scoring, eng_p, bs[0][1], dev, sample=1 << 20)
            res["strict" if strict else "fast"] = {"us_per_step": 1e3 * ms, "achieved_gbs": BYTES_PER_BODY_F32 * n / (ms * 1e-3) / 1e9,
                                                   "parity_1M_bodies": {k: par[k] for k in ("pass_F", "pass_T", "worst_x_tol")}}
        out["c3_strict_vs_fast"] = res
        del bs
        # C3 at 4x the bodies: the per-launch ramp-up / drain amortises
        n4 = 1 << 22
        bs = make_batches(torch, W, n4, 2, torch.float32, dev, W.SEED_BASE + 400)
        k4 = [0]

        def f4():
            bs[k4[0] % 2][0].step_bound(bs[0][1].dt)
            k4[0] += 1
        ms4 = timeit(f4, 60)
        out["c3_4M_bodies"] = {"bodies": n4, "us_per_step": 1e3 * ms4, "updates_per_s": n4 / (ms4 * 1e-3),
                               "achieved_gbs": BYTES_PER_BODY_F32 * n4 / (ms4 * 1e-3) / 1e9}
        del bs
        # mid-size batch, graph replay over independent batches (L2-cold)
        n18 = 1 << 18
        bs = make_batches(torch, W, n18, 24, torch.float32, dev, W.SEED_BASE + 600)
        region, _ = build_step_region(torch, [(lambda b=b: b[0].step_bound(b[1].dt)) for b in bs], 240, dev)
        ms18 = timeit(region, 1, rounds=9) / 240
        out["c3_256k_bodies"] = {"bodies": n18, "us_per_step": 1e3 * ms18, "updates_per_s": n18 / (ms18 * 1e-3),
                                 "achieved_gbs": BYTES_PER_BODY_F32 * n18 / (ms18 * 1e-3) / 1e9,
                                 "kernel": bs[0][0].last_kernel, "note": "24 batches cycled, graph replay"}
        del bs
        # fp64 mode on the C3 workload (336 B/body)
        n = 1 << 20
        bs = make_batches(torch, W, n, 3, torch.float64, dev, W.SEED_BASE + 300)
        k = [0]

        def f():
            bs[k[0] % 3][0].step_bound(bs[0][1].dt)
            k[0] += 1
        ms64 = timeit(f, 60)
        out["c3_fp64_mode"] = {"bodies": n, "us_per_step": 1e3 * ms64, "updates_per_s": n / (ms64 * 1e-3),
                               "achieved_gbs": 2 * BYTES_PER_BODY_F32 * n / (ms64 * 1e-3) / 1e9}
        del bs
    return out


def _with(obj, fn):
    fn(obj)
    return obj


def e5_free_eager(e, wl, steps):
    pos, quat, v, w, F, T = e._bound[0], e._bound[1], e._bound[2], e._bound[3], e._bound[4], e._bound[5]
    for _ in range(steps):
        e.step_bound(wl.dt)
        e.integrate_free_bodies(pos, quat, v, w, F, T, wl.dt, wl.g)


def run_b200(args):
    import torch

    from silver2_isaacsim_b200 import HydroEngine, sharding
    from silver2_isaacsim_b200 import workloads as W

    rank, world, local = sharding.init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (b200 arm) needs a GPU: the engine has no CPU path")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        bind_to_gpu_numa_node(physical_gpu_index(local))
    dtype = torch.float32 if args.dtype == "f32" else torch.float64
    n = args.bodies_per_gpu
    bpb = BYTES_PER_BODY_F32 * (1 if dtype == torch.float32 else 2)

    batches = make_batches(torch, W, n, args.batches, dtype, dev, W.SEED_BASE + 3 + 1000 * rank)
    for b in batches:
        b[0].set_kernel(args.kernel)
    dt = batches[0][1].dt
    timer = RegionTimer(torch, sharding, dev)

    sampler = ClockSampler(physical_gpu_index(local)) if rank == 0 else None
    if sampler:
        sampler.start()

    warm = max(3, args.warmup)
    for i in range(warm):
        batches[i % len(batches)][0].step_bound(dt)
    torch.cuda.synchronize(dev)
    step_fns = [(lambda b=b: b[0].step_bound(dt)) for b in batches]
    # by default a region is one graph launch: more, shorter regions would add launch gaps to the timed steps
    regions = min(args.steps, args.regions or -(-args.steps // GRAPH_CHUNK))
    region_fns, counts, launch_mode = build_step_regions(torch, step_fns, args.steps, regions, dev,
                                                         use_graph=not args.no_graph)
    est_ms_per_step = bpb * n / 6.0e12 * 1e3
    lead, settle_passes = settle_lead(region_fns, args.steps, est_ms_per_step)
    ms_regions, (w0, w1) = timer.run(region_fns, lead=lead)
    dumped = None
    if args.dump_outputs and rank == 0:
        _, _, F_last, T_last = batches[(args.steps - 1) % len(batches)]
        dumped = dump_outputs(args.dump_outputs, {"force": F_last, "torque": T_last})
    ms_step = ms_regions / counts  # per region: ms per step
    ms_med = pctl(ms_step, 50)
    total_bodies = sharding.sum_over_ranks(float(n), dev)
    value = total_bodies / (ms_med * 1e-3)

    # roofline of the dominant (only) kernel: algorithmic bytes per launch / average launch time of the
    # median region (CUDA events on the launch stream)
    per_launch_s = ms_med * 1e-3
    achieved = bpb * n / per_launch_s / 1e9
    peak, peak_src = measured_peak()
    traffic = ncu_traffic()
    clocks = None
    if sampler:
        clocks = sampler.summary(w0, w1)

    # the same region with idle gaps (the board below its power cap): reported next to the sustained median
    spaced = None
    if not args.no_extra:
        try:
            region_ms_est = ms_med * args.steps

            def region():
                for fn in region_fns:
                    fn()
            ms_sp = timer.run_spaced(region, 30, max(0.004, 2.0 * region_ms_est * 1e-3))
            spaced = {"ms_per_step_median": pctl(ms_sp, 50) / args.steps, "ms_per_step_p10": pctl(ms_sp, 10) / args.steps,
                      "ms_per_step_p90": pctl(ms_sp, 90) / args.steps, "regions": int(len(ms_sp)),
                      "achieved_gbs": bpb * n / (pctl(ms_sp, 50) * 1e-3 / args.steps) / 1e9,
                      "what": "the same K-step graph, each replay preceded by an idle gap of twice its own length (>= 4 ms): "
                              "the board never reaches its power cap; max over ranks per replay"}
        except Exception as exc:
            spaced = {"error": repr(exc)}

    # context for the roofline: the SAME launch geometry and TMA traffic with the arithmetic removed (tile config 10),
    # sustained the same way -- what the memory system gives this access pattern on this box in this run
    copy_only = None
    if dtype == torch.float32 and not args.no_extra and args.kernel in ("auto", "tile"):
        try:
            for b in batches:
                b[0].set_tile_config(10)
            for i in range(warm):
                batches[i % len(batches)][0].step_bound(dt)
            torch.cuda.synchronize(dev)
            region_c, counts_c, _ = build_step_regions(torch, step_fns, args.steps, regions, dev,
                                                       use_graph=not args.no_graph)
            lead_c, _ = settle_lead(region_c, args.steps, est_ms_per_step)
            ms_c, _ = timer.run(region_c, lead=lead_c)
            us_c = pctl(ms_c / counts_c, 50) * 1e3
            copy_only = {"us_per_step": us_c, "gbs": bpb * n / us_c / 1e3, "regions": int(len(ms_c)),
                         "what": "tile kernel with the arithmetic removed (h2o_set_tile_config 10): same grid, same bulk "
                                 "loads / stores, timed like the headline steps, max over ranks"}
            del region_c
        except Exception as exc:
            copy_only = {"error": repr(exc)}
        finally:
            for b in batches:
                b[0].set_tile_config(0)

    # per-rank parity sample of this rank's own shard against the float64 oracle (not timed)
    parity = None
    if dtype == torch.float32:
        from oracle import hydro_oracle as O
        from tests import scoring

        p = parity_sample(torch, O, scoring, lambda m: HydroEngine(m, dtype=dtype, device=dev), batches[0][1], dev)
        parity = {"pass_F": sharding.min_over_ranks(p["pass_F"], dev), "pass_T": sharding.min_over_ranks(p["pass_T"], dev),
                  "worst_x_tol": sharding.max_over_ranks(p["worst_x_tol"], dev), "bodies_per_rank": p["bodies"],
                  "ranks": world, "kernel": p["kernel"],
                  "criterion": "fp32 mode per vector: |x-y|_inf <= max(1e-5 |y|_inf, 1e-6) vs the float64 oracle "
                               "(min pass fraction / max error over ranks)"}

    # e2e: public API with HOST buffers (pinned), H2D + kernel + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        eng, wl, _, _ = batches[0]
        npdt = np.float32 if dtype == torch.float32 else np.float64
        pin = [torch.as_tensor(np.ascontiguousarray(a.astype(npdt))).pin_memory()
               for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
        oF = torch.empty(n, 3, dtype=dtype).pin_memory()
        oT = torch.empty(n, 3, dtype=dtype).pin_memory()
        e2e_steps = max(2, min(args.steps, 10))
        e2e_regions = 12
        for _ in range(3):
            eng.step_host(*pin, dt, out_force=oF, out_torque=oT)
        walls = []

        def e2e_region():
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                eng.step_host(*pin, dt, out_force=oF, out_torque=oT)  # returns when the results are in host memory
            walls.append(time.perf_counter() - t0)
        ms_e2e, _ = timer.run([e2e_region] * e2e_regions)
        e2e_s = pctl(ms_e2e, 50) * 1e-3  # device clock (events bracketing the synchronous calls), max over ranks
        e2e_wall = sharding.max_over_ranks(pctl(walls, 50), dev)
        esz = 4 if dtype == torch.float32 else 8
        e2e = {"value": total_bodies * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(n * 13 * esz * world),
               "d2h_bytes_per_step": int(n * 6 * esz * world), "steps": e2e_steps, "regions": e2e_regions,
               "value_p10": total_bodies * e2e_steps / (pctl(ms_e2e, 90) * 1e-3),
               "value_p90": total_bodies * e2e_steps / (pctl(ms_e2e, 10) * 1e-3),
               "host_clock_value": total_bodies * e2e_steps / e2e_wall,
               "api": "HydroEngine.step_host (h2o_step_host), pinned host buffers in and out",
               "path": eng.last_host_path,
               "note": "zero-copy: the fused tile kernel runs on the pinned host buffers (TMA bulk loads pull the 13 input "
                       "scalars per body over PCIe, bulk stores push the 6 output scalars back); one kernel per step, "
                       "transfers and arithmetic overlap tile by tile" if eng.last_host_path == "zero-copy" else
                       "staged: chunked H2D -> kernel -> D2H pipeline on three streams"}
        try:
            e2e["platform_ceiling"] = platform_ceiling(torch, sharding, n, esz, dev)
            e2e["frac_of_ceiling"] = e2e["value"] / e2e["platform_ceiling"]["value"]
        except Exception as exc:
            e2e["platform_ceiling"] = {"error": repr(exc)}
        del pin, oF, oT

    # optional global statistics: the only collective (outside the timed region)
    eng = batches[0][0]
    eng.enable_stats(True)
    eng.step_bound(dt)
    gstats = sharding.allreduce_stats(eng.stats_tensor())
    eng.enable_stats(False)
    kernel_used = eng.last_kernel
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)

    extra = {"timing": {"regions": regions, "timed_steps": args.steps,
                        "steps_per_region": [int(c) for c in counts],
                        "settle": {"passes": settle_passes, "steps": settle_passes * args.steps,
                                   "what": "untimed passes over the same regions launched back to back before the "
                                           "timed steps: half of a >= 200-pass, >= 100 ms train"},
                        "timed_total_ms": float(ms_regions.sum()),
                        "ms_per_step_median": ms_med,
                        "ms_per_step_p10": pctl(ms_step, 10),
                        "ms_per_step_p90": pctl(ms_step, 90),
                        "ms_per_step_first_region": float(ms_step[0]),
                        "ms_per_step_mean": float(ms_regions.sum()) / args.steps,
                        "us_per_step_by_region": [round(1e3 * float(x), 2) for x in ms_step],
                        "note": "ms_per_step / value / roofline use the MEDIAN region (max over ranks per region)",
                        "with_idle_gaps": spaced},
             "dump_outputs": dumped}
    # all ranks: BASELINE config 4, strong scaling with the per-robot wrench
    if not args.no_extra and dtype == torch.float32:
        del batches[1:]
        torch.cuda.empty_cache()
        try:
            extra["c4_strong_scaling"] = c4_strong_leg(torch, sharding, W, dev, rank, world, timer, min(args.steps, 10))
        except Exception as exc:  # side numbers must never lose the headline line
            extra["c4_strong_scaling"] = {"error": repr(exc)}
            sharding.barrier()
    if rank == 0 and not args.no_extra:
        try:
            extra.update(side_measurements(torch, W, dev, dtype))
        except Exception as exc:
            extra["side_error"] = repr(exc)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu = cpu_baseline(args.cpu_sample, args.cpu_seconds, args.ref_kind)
        except Exception as exc:  # the CPU leg must never lose the headline line
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed", "error": repr(exc)}

    if rank == 0:
        cfg = bench_config(n)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_med, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": cfg,
            "impl_config": {"resident_batches": args.batches, "kernel": kernel_used, "launch": launch_mode,
                            "precision": "fp32 storage/traffic; fp32 arithmetic with the waterline, submersion ratio, "
                                         "buoyancy and buoyancy arm carried in fp64 (DESIGN.md section 4)"
                                         if args.dtype == "f32" else "fp64 storage and arithmetic",
                            "parallelism": f"env-sharded x{world}, no data-path collective",
                            "l2": f"{args.batches} independent batches x {bpb * n / 1e6:.0f} MB cycled (> 126 MB L2)"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (traffic or {}).get("dram_bytes_per_launch"), "peak_source": peak_src,
                         "algorithmic_bytes_per_body": bpb, "bodies_per_launch": n,
                         "frac_of_nominal_8TBs": achieved / 8000.0,
                         "regime": "sustained: median of %d regions over the %d timed steps (%.1f ms), launched right after "
                                   "%d untimed steps of the same graphs; the board sits at its power cap after ~40 ms "
                                   "(clocks.reasons)" % (regions, args.steps, float(ms_regions.sum()),
                                                         settle_passes * args.steps),
                         "same_traffic_no_arithmetic": copy_only},
            "e2e": e2e, "gpu_launches": int(args.steps * world), "clocks": clocks,
            "parity_sample": parity, "cpu_baseline": cpu, "global_stats": gstats, "extra": extra,
        }
        emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
