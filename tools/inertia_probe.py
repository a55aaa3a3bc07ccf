"""Cost of the fluid-acceleration loads (h2o_set_fluid_inertia) on the per-body kernel.

Times, in fp32 and fp64, a graph-replayed fused step of 2^20 heterogeneous boxes (C3 distribution, split layout) and of
the C2 hexapod fleet (per-robot wrench), each in an 8-component JONSWAP sea without and with a two-frame current grid,
with the mode off and on; and the persistent free-body rollout of 1024 bodies in the same sea with the mode off and on.  Both arms of a pair are built first, then timed alternately ROUNDS times (CUDA events
over REPS replays of a STEPS-step graph; PERSIST_STEPS steps per rollout); the median per arm is reported.  Prints one
JSON object with the card's name and power limit; OUT=path also writes it there.

    python tools/inertia_probe.py            # STEPS=20 REPS=50 ROUNDS=5 PERSIST_STEPS=2000
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from silver2_isaacsim_b200 import HydroEngine, waves, workloads as W  # noqa: E402

STEPS = int(os.environ.get("STEPS", 20))
REPS = int(os.environ.get("REPS", 50))
ROUNDS = int(os.environ.get("ROUNDS", 5))
PERSIST_STEPS = int(os.environ.get("PERSIST_STEPS", 2000))
dev = torch.device("cuda:0")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / reps  # us per call


def _tensors(wl, dtype):
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dtype).contiguous()
    return t, [t(a) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]


def step_arm(wl, dtype, inertia, grid):
    """A captured STEPS-step graph on its own handle; returns a callable giving us per step."""
    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    e.set_kernel("direct")
    t, ten = _tensors(wl, dtype)
    e.set_prev(t(wl.prev_lin), t(wl.prev_ang))
    e.set_wave_field(waves.jonswap(2.0, 7.0, n_components=8, seed=1))
    e.set_wave_time(1000.0)
    keep = None
    if grid:  # two frames 600 s apart around the clock, 8 x 8 x 4 nodes over the fleet
        vals = np.random.default_rng(3).uniform(-0.5, 0.5, (2, 4, 8, 8, 3))
        keep = torch.as_tensor(vals, device=dev)
        e.set_current_grid(keep, origin=(-200.0, -200.0, -20.0), spacing=(400 / 7, 400 / 7, 20 / 3), t0=700.0,
                           frame_dt=600.0)
    e.set_fluid_inertia(inertia)
    e.bind(*ten)
    e.capture_rollout(STEPS, wl.dt)
    return e, (ten, keep), lambda: timed(e.launch_rollout, REPS) / STEPS


def persistent_arm(dtype, inertia):
    wl = W.uniform_small_batch(1024)
    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    _, ten = _tensors(wl, dtype)
    e.set_wave_field(waves.jonswap(1.0, 5.0, n_components=8, seed=2))
    e.set_fluid_inertia(inertia)
    e.bind(*ten)
    snap = [x.clone() for x in ten]

    def run():
        for x, s in zip(ten, snap):
            x.copy_(s)
        e.reset()
        e.set_wave_time(0.0)
        e.rollout_persistent(PERSIST_STEPS, wl.dt, gravity=wl.g)

    return e, ten, lambda: timed(run, 5) / PERSIST_STEPS


def alternate(arms):
    """Time the arms alternately ROUNDS times; median us per arm."""
    samples = {k: [] for k in arms}
    for _ in range(ROUNDS):
        for k, (_, _, fn) in arms.items():
            samples[k].append(fn())
    return {k: round(float(np.median(v)), 3) for k, v in samples.items()}


def main():
    res = {"card": card(), "components": 8, "steps_per_graph": STEPS, "replays": REPS, "rounds": ROUNDS,
           "step_us": {}, "persistent_1024_us_per_step": {}}
    loads = {"c3_2^20": W.heterogeneous_boxes(1 << 20), "c2_hexapod": W.hexapod_envs()}
    for dtype, name in ((torch.float32, "fp32"), (torch.float64, "fp64")):
        for lname, wl in loads.items():
            for grid in (False, True):
                arms = {"off": step_arm(wl, dtype, False, grid), "on": step_arm(wl, dtype, True, grid)}
                res["step_us"][f"{name} {lname} sea{' + grid' if grid else ''}"] = alternate(arms)
                for e, _, _ in arms.values():
                    e.close()
                del arms
        arms = {"off": persistent_arm(dtype, False), "on": persistent_arm(dtype, True)}
        res["persistent_1024_us_per_step"][name] = alternate(arms)
        for e, _, _ in arms.values():
            e.close()
        del arms
    line = json.dumps(res)
    print(line)
    if os.environ.get("OUT"):
        os.makedirs(os.path.dirname(os.environ["OUT"]) or ".", exist_ok=True)
        with open(os.environ["OUT"], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
