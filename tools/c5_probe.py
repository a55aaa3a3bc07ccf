"""C5: 1024 bodies, 1000-step rollout: eager launches vs CUDA graph (static state / free bodies)."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from silver2_isaacsim_b200 import HydroEngine, workloads as W
dev = torch.device("cuda:0")
wl = W.uniform_small_batch(int(os.environ.get("N", 1024)))
ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
def timeit(fn, reps=5):
    fn(); torch.cuda.synchronize(); ev0.record()
    for _ in range(reps): fn()
    ev1.record(); torch.cuda.synchronize(); return ev0.elapsed_time(ev1) / reps
for free in (False, True):
    e = HydroEngine(wl.n, device=dev); e.set_workload_params(wl)
    t = lambda a: torch.as_tensor(a, device=dev).clone()
    e.bind(t(wl.pos), t(wl.quat_xyzw), t(wl.lin_vel), t(wl.ang_vel))
    e.set_rollout_mode(free_bodies=free)
    ms_e = timeit(lambda: [e.step_bound(wl.dt) for _ in range(1000)]) if not free else float("nan")
    e.capture_rollout(1000, wl.dt)
    ms_g = timeit(e.launch_rollout)
    print(f"N={wl.n} free_bodies={free}: eager {ms_e:.2f} us/step, graph {ms_g:.2f} us/step, kernel {e.last_kernel}")
