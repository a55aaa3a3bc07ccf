"""Launch overlap of consecutive captured tile kernels: two builds of the library compared on the workloads whose
kernel boundaries it changes, in alternating runs (profiles/r07_launch_overlap.md).

    python tools/overlap_probe.py --lib base=PATH_A --lib new=PATH_B [--rounds 5] [--out DIR]

Each run is a child process with H2O_LIB_PATH set to one build; the builds alternate run by run, round by round, so
that slow drift of the board (clock, power, neighbours) falls on both.  Cases, all sustained (the board at its power
cap) unless said otherwise:
  c3      the headline: 6 resident batches of 2^20 boxes, graph replay of 120-step graphs, median over regions
  sweep   tools/n_sweep.py at MIN_MS=400 for 2^18 .. 2^22 (fixed cost = t(2^20) - t(2^21) / 2)
  c3_256k 2^18 boxes, 24 batches, graph replay (bench.py's c3_256k_bodies leg)
  c2      4096 hexapods, part table + robot wrench, one engine, captured 200-step rollout
  fp64    2^20 boxes in fp64 mode, 3 batches, eager launches (bench.py's c3_fp64_mode leg)
  c4      110 592 hexapods with per-body records and robot wrench, 2 batches, eager (bench.py's c4 shard leg)
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child(cases):
    import torch

    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from silver2_isaacsim_b200 import HydroEngine, workloads as W

    dev = torch.device("cuda:0")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = {}

    def engines(wls, dtype=torch.float32, robot=False):
        npdt = np.float32 if dtype == torch.float32 else np.float64
        es = []
        for wl in wls:
            e = HydroEngine(wl.n, dtype=dtype, device=dev)
            e.set_workload_params(wl)
            t = lambda a: torch.as_tensor(np.ascontiguousarray(a.astype(npdt)), device=dev)
            e.set_prev(t(wl.prev_lin), t(wl.prev_ang))
            e.bind(t(wl.pos), t(wl.quat_xyzw), t(wl.lin_vel), t(wl.ang_vel), robot_wrench=robot)
            e.dt = wl.dt
            es.append(e)
        return es

    def graph(fns, steps):
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for f in fns:
                f()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for i in range(steps):
                fns[i % len(fns)]()
        return g

    def sustained(fn, steps_per_call, settle_ms=1500.0, regions=41):
        """us per step: median over `regions` timed calls, after back-to-back untimed calls for settle_ms."""
        fn(); torch.cuda.synchronize()
        ev0.record(); fn(); ev1.record(); torch.cuda.synchronize()
        settle = max(1, int(settle_ms / max(ev0.elapsed_time(ev1), 1e-3)))
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(regions + 1)]
        for _ in range(settle):
            fn()
        evs[0].record()
        for r in range(regions):
            fn()
            evs[r + 1].record()
        torch.cuda.synchronize()
        per = [1e3 * evs[r].elapsed_time(evs[r + 1]) / steps_per_call for r in range(regions)]
        return float(np.median(per))

    if "c3" in cases:
        es = engines([W.heterogeneous_boxes(1 << 20, seed=W.SEED_BASE + 3 + b) for b in range(6)])
        g = graph([(lambda e=e: e.step_bound(e.dt)) for e in es], 120)
        out["c3_us"] = sustained(g.replay, 120)
        del es, g
    if "sweep" in cases:
        from n_sweep import sweep
        out["sweep_us"] = {str(n): us for n, _, us, _ in sweep((18, 19, 20, 21, 22), min_ms=400.0, dev=dev)}
        s = out["sweep_us"]
        out["fixed_cost_us"] = s[str(1 << 20)] - s[str(1 << 21)] / 2
    if "c3_256k" in cases:
        es = engines([W.heterogeneous_boxes(1 << 18, seed=W.SEED_BASE + 600 + b) for b in range(24)])
        g = graph([(lambda e=e: e.step_bound(e.dt)) for e in es], 240)
        out["c3_256k_us"] = sustained(g.replay, 240)
        del es, g
    if "c2" in cases:
        wl = W.hexapod_envs(4096)
        (e,) = engines([wl], robot=True)
        e.capture_rollout(200, wl.dt)
        out["c2_graph_us"] = sustained(e.launch_rollout, 200, settle_ms=500.0, regions=21)
        del e
    if "fp64" in cases:
        es = engines([W.heterogeneous_boxes(1 << 20, seed=W.SEED_BASE + 300 + b) for b in range(3)], torch.float64)
        k = [0]

        def f():
            for _ in range(60):
                es[k[0] % 3].step_bound(es[0].dt)
                k[0] += 1
        out["fp64_us"] = sustained(f, 60, settle_ms=500.0, regions=21)
        del es
    if "c4" in cases:
        es = engines([W.sharded_robots(110592), W.sharded_robots(110592, seed=W.SEED_BASE + 44)], robot=True)
        k = [0]

        def f():
            for _ in range(100):
                es[k[0] % 2].step_bound(es[0].dt)
                k[0] += 1
        out["c4_us"] = sustained(f, 100, settle_ms=500.0, regions=21)
        del es
    print("RESULT " + json.dumps(out), flush=True)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="NAME=PATH of a build (two or more)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cases", default="c3,sweep,c3_256k,c2,fp64,c4")
    ap.add_argument("--out", default=None, help="write the per-run results as JSON here")
    ap.add_argument("--child", action="store_true")
    args = ap.parse_args()
    cases = args.cases.split(",")
    if args.child:
        return child(cases)
    libs = [tuple(x.split("=", 1)) for x in args.lib]
    runs = []
    print(f"# {gpu_info()}", flush=True)
    for r in range(args.rounds):
        for name, path in (libs if r % 2 == 0 else libs[::-1]):
            env = dict(os.environ, H2O_LIB_PATH=os.path.abspath(path))
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--cases", args.cases],
                               env=env, capture_output=True, text=True)
            line = [l for l in p.stdout.splitlines() if l.startswith("RESULT ")]
            if p.returncode or not line:
                print(p.stdout[-2000:], p.stderr[-4000:], file=sys.stderr)
                raise SystemExit(f"run {r} of {name} failed")
            res = json.loads(line[0][7:])
            runs.append({"round": r, "lib": name, **res})
            print(json.dumps(runs[-1]), flush=True)
    keys = [k for k in runs[0] if k not in ("round", "lib") and not isinstance(runs[0][k], dict)]
    keys += [f"sweep_us.{n}" for n in runs[0].get("sweep_us", {})]
    get = lambda run, k: run[k] if "." not in k else run[k.split(".")[0]][k.split(".")[1]]
    print("| case | " + " | ".join(f"{n} median (min .. max)" for n, _ in libs) + " |")
    print("|---|" + "---|" * len(libs))
    for k in keys:
        cells = []
        for n, _ in libs:
            v = [get(run, k) for run in runs if run["lib"] == n]
            cells.append(f"{np.median(v):.2f} ({min(v):.2f} .. {max(v):.2f})")
        print(f"| {k} | " + " | ".join(cells) + " |")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"gpu": gpu_info(), "runs": runs}, f, indent=1)


if __name__ == "__main__":
    main()
