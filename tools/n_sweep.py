"""Fused step (C3 distribution, fp32, per-body records): time per step vs bodies per launch.
Every size cycles through enough independent batches to exceed L2 several times; graph replay.
MIN_MS=500 keeps every size running for at least that long (the board's power-capped regime)."""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from silver2_isaacsim_b200 import HydroEngine, workloads as W

LOGNS = (14, 16, 18, 19, 20, 21, 22, 24)


def sweep(logns=LOGNS, min_ms=0.0, dev=torch.device("cuda:0")):
    """Yields (bodies, batches, us per step, kernel) per size."""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    base = W.heterogeneous_boxes(1 << 22, seed=7)
    for logn in logns:
        n = 1 << logn
        nb = max(2, min(64, (1 << 30) // (168 * n)))           # ~1 GB of distinct data
        es = []
        for b in range(nb):
            sl = slice((b * n) % (1 << 22), (b * n) % (1 << 22) + min(n, 1 << 22))
            rep = max(1, n >> 22)
            t = lambda a: torch.as_tensor(np.tile(a[sl], (rep, 1)), device=dev)
            e = HydroEngine(n, device=dev)
            e.set_params_per_body(np.tile(base.coeff[sl], (rep, 1)))
            e.set_prev(t(base.prev_lin), t(base.prev_ang))
            e.bind(t(base.pos), t(base.quat_xyzw), t(base.lin_vel), t(base.ang_vel))
            es.append(e)
        reps = max(240, min(2000, int(2e9 // (168 * n))))
        if min_ms > 0:  # sustained regime: at least min_ms of back-to-back replays per size
            reps = max(reps, int(min_ms * 1e3 / max(3.0, 168 * n / 6.0e6)))
        per = nb * max(1, min(10, reps // nb)); reps = (reps // per) * per or per
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            for e in es: e.step_bound(base.dt)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for i in range(per): es[i % nb].step_bound(base.dt)
        g.replay(); torch.cuda.synchronize(); ev0.record()
        for _ in range(reps // per): g.replay()
        ev1.record(); torch.cuda.synchronize()
        yield n, nb, ev0.elapsed_time(ev1) * 1e3 / reps, es[0].last_kernel
        del es, g


if __name__ == "__main__":
    print("| bodies per launch | batches | us/step | G updates/s | GB/s (168 B/body) | of 6540 GB/s | kernel |")
    print("|---|---|---|---|---|---|---|")
    for n, nb, us, kernel in sweep(min_ms=float(os.environ.get("MIN_MS", "0"))):
        print(f"| 2^{n.bit_length() - 1} = {n} | {nb} | {us:.2f} | {n / us / 1e3:.2f} | {168 * n / us / 1e3:.0f} | {100 * 168 * n / us / 1e3 / 6540.2:.1f} % | {kernel} |")
