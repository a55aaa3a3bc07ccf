"""Cost of the built-in wave field (h2o_set_wave_field) on the per-body kernel.

Times a graph-replayed fused step of 2^20 heterogeneous boxes (C3 distribution, split layout) in fp32 and fp64 for:
flat water on the per-body kernel, a caller height array (h2o_set_surface_heights), and a JONSWAP field of 1, 8, 32
and 64 components; then the persistent free-body rollout of 1024 bodies with and without 8 components.  Every
configuration is warmed up, then timed with CUDA events over REPS replays of a STEPS-step graph (the 2^20-body
working set, ~180 MB in fp32, is larger than the 126 MB L2).  Prints one JSON object with the card's name
and power limit; OUT=path also writes it there.

    python tools/wave_probe.py            # STEPS=20 REPS=50 PERSIST_STEPS=2000
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


def step_case(wl, dtype, case):
    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    e.set_kernel("direct")
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dtype).contiguous()
    ten = [t(a) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    e.set_prev(t(wl.prev_lin), t(wl.prev_ang))
    keep = None
    if case == "eta":
        keep = 0.3 * torch.cos(0.7 * ten[0][:, 0]).contiguous()
        e.set_surface_heights(keep)
    elif case != "flat":
        e.set_wave_field(waves.jonswap(2.0, 7.0, n_components=int(case), seed=1))
        e.set_wave_time(1000.0)
    e.bind(*ten)
    e.capture_rollout(STEPS, wl.dt)
    us = timed(e.launch_rollout, REPS) / STEPS
    assert e.last_kernel == "direct"
    e.close()
    return us


def persistent_case(dtype, n_waves):
    wl = W.uniform_small_batch(1024)
    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dtype).contiguous()
    ten = [t(a) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    if n_waves:
        e.set_wave_field(waves.jonswap(1.0, 5.0, n_components=n_waves, seed=2))
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
    res = {"card": card(), "n_bodies": 1 << 20, "steps_per_graph": STEPS, "replays": REPS, "step_us": {},
           "persistent_1024_us_per_step": {}}
    wl = W.heterogeneous_boxes(1 << 20)
    for dtype, name in ((torch.float32, "fp32"), (torch.float64, "fp64")):
        row = {}
        for case in ("flat", "eta", "1", "8", "32", "64"):
            row[case if case in ("flat", "eta") else f"waves_{case}"] = round(step_case(wl, dtype, case), 2)
        res["step_us"][name] = row
        res["persistent_1024_us_per_step"][name] = {"flat": round(persistent_case(dtype, 0), 3),
                                                   "waves_8": round(persistent_case(dtype, 8), 3)}
    line = json.dumps(res)
    print(line)
    if os.environ.get("OUT"):
        os.makedirs(os.path.dirname(os.environ["OUT"]) or ".", exist_ok=True)
        with open(os.environ["OUT"], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
