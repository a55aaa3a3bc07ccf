"""Harness-side twins of two small reference utilities, for stand-alone rollouts (SURVEY.md 8(f2)).

``VelocityTrace``  writes the CSV of the reference's ``LogVelocity`` behaviour
                   (/root/reference/src/scripts/physics/log_velocity.py:17-53): same header, same
                   z / x / y column order, one row per sample of one body (optional extra columns after them).
``RtfMeter``       accumulates simulated vs wall time like ``BenchmarkRtf``
                   (/root/reference/src/scripts/physics/benchmark_rtf.py:37-71): real-time factor and
                   steps per second, with a live line every ``report_every`` steps.
"""
from __future__ import annotations

import csv
import datetime
import time
from typing import Optional, Sequence

LOG_HEADER = ["timestamp",
              "z_position", "linear_velocity_z", "angular_velocity_z",
              "x_position", "linear_velocity_x", "angular_velocity_x",
              "y_position", "linear_velocity_y", "angular_velocity_y"]  # log_velocity.py:17-20


class VelocityTrace:
    def __init__(self, path: str, body: int = 0, extra_columns: Sequence[str] = ()):
        self.path, self.body, self.n_extra = path, body, len(extra_columns)
        with open(path, "w", newline="") as f:
            csv.writer(f).writerow(LOG_HEADER + list(extra_columns))

    def sample(self, position, linear_vel, angular_vel, timestamp: Optional[str] = None, extra: Sequence[float] = ()):
        """Append one row for body ``self.body`` (tensors or arrays of shape (N,3)), then the ``extra`` values."""
        if len(extra) != self.n_extra:
            raise ValueError(f"expected {self.n_extra} extra values, got {len(extra)}")
        p, v, w = (x[self.body].tolist() for x in (position, linear_vel, angular_vel))
        row = [timestamp or datetime.datetime.now().isoformat(),
               p[2], v[2], w[2], p[0], v[0], w[0], p[1], v[1], w[1]] + [float(x) for x in extra]  # log_velocity.py:38-49
        with open(self.path, "a", newline="") as f:
            csv.writer(f).writerow(row)


class RtfMeter:
    def __init__(self, report_every: int = 600, printer=print):
        self.report_every, self.printer = report_every, printer
        self.reset()

    def reset(self):
        self._t0 = time.time()
        self.total_sim_time = 0.0
        self.steps = 0

    def on_physics_step(self, delta_time: float, n_steps: int = 1):
        self.total_sim_time += delta_time * n_steps
        before = self.steps
        self.steps += n_steps
        if self.report_every and before // self.report_every != self.steps // self.report_every:
            r = self.report()
            self.printer(f"[RTF Benchmark] Live: RTF {r['rtf']:.4f}x | steps/s {r['steps_per_s']:.2f}")

    def report(self) -> dict:
        wall = max(time.time() - self._t0, 1e-9)
        return {"wall_time_s": wall, "sim_time_s": self.total_sim_time, "steps": self.steps,
                "rtf": self.total_sim_time / wall, "steps_per_s": self.steps / wall}
