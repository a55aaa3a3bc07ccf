"""Cost of the current grid (h2o_set_current_grid) on the per-body kernel and in the persistent rollout.

Times a graph-replayed fused step for two fleets, in fp32 and fp64:
  C2: 4096 hexapods of 19 bodies (77 824 bodies, split layout, per-robot wrench);
  2^20 heterogeneous boxes (C3 distribution);
each on the per-body kernel with: no grid, a depth profile (1x32x1x1), a 3-D grid 1x32x256x256 (~50 MB) spanning the
fleet, two frames of it, and two frames plus an 8-component JONSWAP sea.  Then the persistent free-body rollout of
1024 bodies with no grid, a profile and a time-varying two-frame 3-D grid.  Every configuration is warmed up, then
timed with CUDA events over REPS replays of a STEPS-step graph.  Prints one JSON object with the card's name and
power limit, read in the same run; OUT=path also writes it there.

    python tools/current_probe.py            # STEPS=20 REPS=50 PERSIST_STEPS=2000
"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from silver2_isaacsim_b200 import HydroEngine, currents, waves, workloads as W  # noqa: E402
from tools.env_probe import card, timed  # noqa: E402

STEPS = int(os.environ.get("STEPS", 20))
REPS = int(os.environ.get("REPS", 50))
PERSIST_STEPS = int(os.environ.get("PERSIST_STEPS", 2000))
dev = torch.device("cuda:0")
CASES = ("direct", "profile_1x32x1x1", "grid_1x32x256x256", "grid_2x32x256x256", "grid_2x32x256x256_waves_8")


def make_grid(case, pos):
    """The case's grid over the fleet's bounding box (x, y) and p_z in [-4, 4] m, or None."""
    rng = np.random.default_rng(1)
    if case.startswith("profile"):
        return currents.power_law_profile(0.8, 0.3, seabed_z=-18.4)
    if not case.startswith("grid"):
        return None
    nt = int(case.split("_")[1][0])
    lo, hi = pos[:, :2].min(axis=0), pos[:, :2].max(axis=0)
    return currents.CurrentGrid(rng.uniform(-0.5, 0.5, (nt, 32, 256, 256, 3)), origin=(lo[0], lo[1], -4.0),
                                spacing=((hi[0] - lo[0]) / 255, (hi[1] - lo[1]) / 255, 8.0 / 31), t0=0.0,
                                frame_dt=1.0 if nt > 1 else 0.0)


def set_grid(e, g):
    vals = torch.as_tensor(g.values, device=dev)
    e.set_current_grid(vals, g.origin, g.spacing, g.t0, g.frame_dt)
    return vals


def step_case(wl, dtype, case):
    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    e.set_kernel("direct")
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dtype).contiguous()
    ten = [t(a) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    e.set_prev(t(wl.prev_lin), t(wl.prev_ang))
    g = make_grid(case, wl.pos)
    keep = set_grid(e, g) if g is not None else None
    if case.endswith("waves_8"):
        e.set_wave_field(waves.jonswap(2.0, 7.0, n_components=8, seed=1))
    e.set_wave_time(0.5)
    e.bind(*ten, robot_wrench=wl.bodies_per_robot > 0)
    e.capture_rollout(STEPS, wl.dt)
    us = timed(e.launch_rollout, REPS) / STEPS
    assert e.last_kernel == "direct", (case, e.last_kernel)
    e.close()
    del keep
    return us


def persistent_case(dtype, case):
    wl = W.uniform_small_batch(1024)
    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dtype).contiguous()
    ten = [t(a) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    g = make_grid(case, wl.pos)
    keep = set_grid(e, g) if g is not None else None
    e.bind(*ten)
    snap = [x.clone() for x in ten]

    def run():
        for x, s in zip(ten, snap):
            x.copy_(s)
        e.reset()
        e.set_wave_time(0.0)
        e.rollout_persistent(PERSIST_STEPS, wl.dt, gravity=wl.g)

    us = timed(run, 5) / PERSIST_STEPS
    e.close()
    del keep
    return us


def main():
    res = {"card": card(), "steps_per_graph": STEPS, "replays": REPS, "step_us": {},
           "persistent_1024_us_per_step": {}}
    fleets = (("c2_hexapods_4096x19", W.hexapod_envs(4096)), ("boxes_2^20", W.heterogeneous_boxes(1 << 20)))
    for dtype, name in ((torch.float32, "fp32"), (torch.float64, "fp64")):
        for fleet, wl in fleets:
            res["step_us"].setdefault(fleet, {})[name] = {c: round(step_case(wl, dtype, c), 2) for c in CASES}
        res["persistent_1024_us_per_step"][name] = {
            c: round(persistent_case(dtype, c), 3) for c in ("direct", "profile_1x32x1x1", "grid_2x32x256x256")}
    line = json.dumps(res)
    print(line)
    if os.environ.get("OUT"):
        os.makedirs(os.path.dirname(os.environ["OUT"]) or ".", exist_ok=True)
        with open(os.environ["OUT"], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
