"""The reference README's buoy validation, stand-alone on the GPU (SURVEY.md 8(f2), config C1).

A 1 m cube of half the water's density is released from z = 1 m with a small tilt and left to bob
until it floats half submerged.  Forces come from the fused step kernel, the motion from the
device-side free-body stepper (semi-implicit Euler + gravity; inside Isaac Sim PhysX does this part),
both replayed from one captured CUDA graph of 100 steps.  After every replay one CSV row is written in the
column order of the reference's LogVelocity behaviour (log_velocity.py:17-20), and the real-time
factor is reported like its BenchmarkRtf (benchmark_rtf.py:37-71).

With --wave-amplitude > 0 the buoy floats in a regular deep-water wave of that amplitude and --wave-period,
evaluated by the engine at the buoy on every step; the CSV then has one more column, the surface
elevation at the buoy.  --wave-slope also tests the buoy against the wave surface's local tangent plane
(h2o_set_wave_slope), so that the waves roll and pitch it; the CSV then also logs the buoy's roll and pitch angles
(degrees, xyz Euler angles of its orientation).

    python examples/buoy_validation.py [--steps 6000] [--n 1] [--csv /tmp/buoy.csv] [--wave-amplitude 0.2 --wave-period 8]
                                       [--wave-slope]
"""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from silver2_isaacsim_b200 import HydroEngine, waves, workloads as W  # noqa: E402
from silver2_isaacsim_b200.trace import RtfMeter, VelocityTrace    # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=6000)
ap.add_argument("--n", type=int, default=1, help="identical buoys stepped side by side")
ap.add_argument("--csv", default="/tmp/buoy_velocity_log.csv")
ap.add_argument("--wave-amplitude", type=float, default=0.0, help="regular deep-water wave amplitude (m); 0 = still water")
ap.add_argument("--wave-period", type=float, default=8.0, help="wave period (s)")
ap.add_argument("--wave-slope", action="store_true", help="test the buoy against the waves' local tangent plane")
args = ap.parse_args()
if args.wave_slope and not args.wave_amplitude > 0:
    ap.error("--wave-slope needs --wave-amplitude > 0")


def roll_pitch(q):
    """Roll and pitch (degrees) of an xyzw quaternion: the x and y angles of its xyz Euler decomposition."""
    x, y, z, s = (float(c) for c in q)
    roll = np.degrees(np.arctan2(2 * (s * x + y * z), 1 - 2 * (x * x + y * y)))
    pitch = np.degrees(np.arcsin(np.clip(2 * (s * y - z * x), -1.0, 1.0)))
    return roll, pitch


dev = torch.device("cuda:0")
wl = W.readme_buoy()
eng = HydroEngine(args.n, dtype=torch.float64, device=dev)
eng.set_globals(wl.rho, wl.g)
eng.set_part_table(wl.table, wl.slot_type)
rep = lambda a: torch.as_tensor(np.repeat(np.asarray(a, dtype=np.float64), args.n, axis=0), device=dev).contiguous()
pos, quat, v, w = rep(wl.pos), rep(wl.quat_xyzw), rep(wl.lin_vel), rep(wl.ang_vel)
F, T = eng.bind(pos, quat, v, w)
eng.set_rollout_mode(free_bodies=True, gravity=wl.g)   # every captured step: forces, then the stepper
in_waves = args.wave_amplitude > 0
if in_waves:
    eng.set_wave_field(waves.regular(args.wave_amplitude, args.wave_period))
    eng.set_wave_slope(args.wave_slope)

GRAPH = 100
eng.capture_rollout(GRAPH, wl.dt)
columns = (("surface_elevation",) if in_waves else ()) + (("roll_deg", "pitch_deg") if args.wave_slope else ())
trace = VelocityTrace(args.csv, extra_columns=columns)
max_tilt = 0.0
rtf = RtfMeter(report_every=1000)
for k in range(args.steps // GRAPH):
    eng.launch_rollout()
    torch.cuda.synchronize()
    rtf.on_physics_step(wl.dt, GRAPH)
    extra = (float(eng.sample_waves(pos[:1])[0, 0]),) if in_waves else ()   # elevation at the buoy, current clock
    if args.wave_slope:
        extra += roll_pitch(quat[0].cpu())
        max_tilt = max(max_tilt, abs(extra[1]), abs(extra[2]))
    trace.sample(pos.cpu(), v.cpu(), w.cpu(), extra=extra)  # one row per replayed graph
r = rtf.report()
z = float(pos[0, 2])
print(f"{args.n} buoy(s), {r['steps']} steps of {wl.dt * 1e3:.2f} ms: RTF {r['rtf']:.1f}x, {r['steps_per_s']:.0f} steps/s; "
      f"final height of the centre {z:+.4f} m (half submerged = 0), |v| {float(v[0].norm()):.2e} m/s; trace: {args.csv}")
if args.wave_slope:
    print(f"largest logged roll / pitch angle: {max_tilt:.2f} deg")
