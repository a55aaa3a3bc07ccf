"""Cost of per-env water conditions (h2o_set_env_conditions) on the per-body kernel.

Times a graph-replayed fused step for two fleets, in fp32 and fp64:
  C2: 4096 hexapods of 19 bodies (77 824 bodies, split layout, per-robot wrench), one env per robot;
  2^20 heterogeneous boxes (C3 distribution) as 4-body envs;
each with: no conditions on the tile kernel, no conditions on the per-body kernel, identity conditions, random
conditions, and random conditions plus an 8-component JONSWAP sea.  Then the persistent free-body rollout of 1024
bodies (4-body envs) with and without random conditions.  Every configuration is warmed up, then timed with CUDA
events over REPS replays of a STEPS-step graph (the 2^20-body working set, ~180 MB in fp32, is larger than the
126 MB L2; the C2 one, ~16 MB, is not).  Prints one JSON object with the card's name and power limit, read in the
same run; OUT=path also writes it there.

    python tools/env_probe.py            # STEPS=20 REPS=50 PERSIST_STEPS=2000
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
PERSIST_STEPS = int(os.environ.get("PERSIST_STEPS", 2000))
dev = torch.device("cuda:0")
CASES = ("tile", "direct", "identity", "random", "random_waves_8")


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


def random_cond(n_envs, seed=0):
    rng = np.random.default_rng(seed)
    c = waves.env_conditions(n_envs, current=rng.uniform(-0.5, 0.5, (n_envs, 3)), surface_dz=rng.uniform(-0.5, 0.5, n_envs),
                             wave_scale=rng.uniform(0.0, 2.0, n_envs), time_offset=rng.uniform(0.0, 1e4, n_envs),
                             origin=rng.uniform(-200.0, 200.0, (n_envs, 2)))
    return torch.as_tensor(c, device=dev)


def step_case(wl, dtype, bodies_per_env, case):
    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    e.set_kernel("tile" if case == "tile" else "direct")
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dtype).contiguous()
    ten = [t(a) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    e.set_prev(t(wl.prev_lin), t(wl.prev_ang))
    n_envs = wl.n // bodies_per_env
    if case == "identity":
        e.set_env_conditions(torch.as_tensor(waves.env_conditions(n_envs), device=dev), bodies_per_env)
    elif case.startswith("random"):
        e.set_env_conditions(random_cond(n_envs), bodies_per_env)
    if case == "random_waves_8":
        e.set_wave_field(waves.jonswap(2.0, 7.0, n_components=8, seed=1))
        e.set_wave_time(1000.0)
    e.bind(*ten, robot_wrench=wl.bodies_per_robot > 0)
    e.capture_rollout(STEPS, wl.dt)
    us = timed(e.launch_rollout, REPS) / STEPS
    assert e.last_kernel == ("tile" if case == "tile" else "direct"), (case, e.last_kernel)
    e.close()
    return us


def persistent_case(dtype, with_cond):
    wl = W.uniform_small_batch(1024)
    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dtype).contiguous()
    ten = [t(a) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    if with_cond:
        e.set_env_conditions(random_cond(wl.n // 4), 4)
    e.bind(*ten)
    snap = [x.clone() for x in ten]

    def run():
        for x, s in zip(ten, snap):
            x.copy_(s)
        e.reset()
        e.rollout_persistent(PERSIST_STEPS, wl.dt, gravity=wl.g)

    us = timed(run, 5) / PERSIST_STEPS
    e.close()
    return us


def main():
    res = {"card": card(), "steps_per_graph": STEPS, "replays": REPS, "step_us": {},
           "persistent_1024_us_per_step": {}}
    fleets = (("c2_hexapods_4096x19", W.hexapod_envs(4096), 19), ("boxes_2^20_envs_of_4", W.heterogeneous_boxes(1 << 20), 4))
    for dtype, name in ((torch.float32, "fp32"), (torch.float64, "fp64")):
        for fleet, wl, bpe in fleets:
            res["step_us"].setdefault(fleet, {})[name] = {c: round(step_case(wl, dtype, bpe, c), 2) for c in CASES}
        res["persistent_1024_us_per_step"][name] = {"no_conditions": round(persistent_case(dtype, False), 3),
                                                   "random_conditions": round(persistent_case(dtype, True), 3)}
    line = json.dumps(res)
    print(line)
    if os.environ.get("OUT"):
        os.makedirs(os.path.dirname(os.environ["OUT"]) or ".", exist_ok=True)
        with open(os.environ["OUT"], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
