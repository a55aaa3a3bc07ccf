"""Float64 NumPy free-body rollout around the oracle forces (TEST INFRASTRUCTURE ONLY).

The reference has no integrator (PhysX integrates); BASELINE config 1 asks for a stand-alone
harness: semi-implicit Euler + gravity around the reference force functions.  This mirrors
``free_body_kernel`` in csrc/h2o_kernels.cuh step by step so that a free-running CUDA rollout
can be compared with a float64 one, and records the state sequence for teacher-forced scoring.
"""
from __future__ import annotations

import numpy as np

from . import hydro_oracle as O


def _rot(q):
    """Rotation matrix (..., 3, 3) of xyzw quaternions (..., 4), not normalised."""
    x, y, z, w = np.moveaxis(np.asarray(q, dtype=np.float64), -1, 0)
    x2, y2, z2 = x + x, y + y, z + z
    rows = [[1 - (y * y2 + z * z2), x * y2 - w * z2, x * z2 + w * y2],
            [x * y2 + w * z2, 1 - (x * x2 + z * z2), y * z2 - w * x2],
            [x * z2 - w * y2, y * z2 + w * x2, 1 - (x * x2 + y * y2)]]
    return np.stack([np.stack(r, axis=-1) for r in rows], axis=-2)


def integrate(p, q, v, w, F, T, mass, dims, dt, gravity):
    """One semi-implicit Euler step of a free box (xyzw quaternion); returns new (p,q,v,w).

    One body, or a batch: vectors (..., 3), quaternions (..., 4), mass (...) and dims (..., 3)."""
    p, q, v, w, F, T, dims = (np.asarray(a, dtype=np.float64) for a in (p, q, v, w, F, T, dims))
    mass = np.asarray(mass, dtype=np.float64)[..., None]
    v = v + dt * (F / mass + np.array([0.0, 0.0, -gravity]))
    R = _rot(q)
    dx, dy, dz = np.moveaxis(dims, -1, 0)
    I = mass * np.stack([dy * dy + dz * dz, dx * dx + dz * dz, dx * dx + dy * dy], axis=-1) / 12.0
    tb, wb = np.einsum("...ji,...j->...i", R, T), np.einsum("...ji,...j->...i", R, w)
    gyro = np.cross(wb, I * wb)
    wb = wb + dt * (tb - gyro) / I
    w = np.einsum("...ij,...j->...i", R, wb)
    p = p + dt * v
    x, y, z, s = np.moveaxis(q, -1, 0)
    wx, wy, wz = np.moveaxis(w, -1, 0)
    h = 0.5 * dt
    nq = np.stack([x + h * (wx * s + wy * z - wz * y),
                   y + h * (wy * s + wz * x - wx * z),
                   z + h * (wz * s + wx * y - wy * x),
                   s - h * (wx * x + wy * y + wz * z)], axis=-1)
    return p, nq / np.linalg.norm(nq, axis=-1, keepdims=True), v, w


def rollout(ctor, mass, p, q, v, w, dt, steps, gravity=9.81):
    """Free-running float64 rollout; returns the per-step record (state BEFORE each step, the
    previous velocities the behaviour would hold, and the oracle wrench of that step)."""
    ctor = np.asarray(ctor, dtype=np.float64)
    dims = ctor[0:3]
    p, q, v, w = (np.array(a, dtype=np.float64) for a in (p, q, v, w))
    pv, pw = np.zeros(3), np.zeros(3)  # hydrodynamics_behavior.py:196-198
    rec = {k: np.zeros((steps, n)) for k, n in (("pos", 3), ("quat", 4), ("v", 3), ("w", 3), ("prev_v", 3),
                                                ("prev_w", 3), ("F", 3), ("T", 3))}
    raised = np.zeros(steps, dtype=bool)
    for k in range(steps):
        r = O.step(ctor, [mass], p[None], q[None], v[None], w[None], pv[None], pw[None], dt, n_threads=1)
        for name, val in (("pos", p), ("quat", q), ("v", v), ("w", w), ("prev_v", pv), ("prev_w", pw),
                          ("F", r.force[0]), ("T", r.torque[0])):
            rec[name][k] = val
        raised[k] = bool(r.flags[0] & 1)
        pv, pw = v.copy(), w.copy()
        p, q, v, w = integrate(p, q, v, w, r.force[0], r.torque[0], mass, dims, dt, gravity)
    rec["raised"] = raised
    rec["final"] = (p, q, v, w)
    return rec
