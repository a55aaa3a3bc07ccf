"""Float64 NumPy reference of the behaviour step with fluid-acceleration loads.  TEST TOOL ONLY.

``step`` is ``tests/slope_reference.py``'s restatement of the C oracle's step (optional waterline slope included) with
one addition, a per-body fluid acceleration ``a_f`` (include/h2o.h, ``h2o_set_fluid_inertia``):

* the added mass sees ``a_b - a_f`` in place of ``a_b`` (``M [R^T (a_b - a_f); R^T alpha_b]``, diagonal or dense);
* the Froude-Krylov force ``rho (r V) a_f`` is applied at the centre of buoyancy;

both before the safety clamp.  Without ``fluid_accel`` it is ``slope_reference.step``, bit for bit.
"""
from __future__ import annotations

import numpy as np

from tests import slope_reference as SR


def step(ctor, mass, pos, quat_xyzw, lin_vel, ang_vel, prev_lin, prev_ang, dt, slope=None, fluid_accel=None,
         dense=None, dense_slot=None) -> SR.StepResult:
    """``slope_reference.step`` (Numba semantics) with the optional per-body fluid acceleration ``fluid_accel`` (n,3)."""
    if fluid_accel is None:
        return SR.step(ctor, mass, pos, quat_xyzw, lin_vel, ang_vel, prev_lin, prev_ang, dt, slope=slope, dense=dense,
                       dense_slot=dense_slot)
    f = lambda x, k: np.ascontiguousarray(np.asarray(x, dtype=np.float64)).reshape(-1, k)
    pos, q, v, w = f(pos, 3), f(quat_xyzw, 4), f(lin_vel, 3), f(ang_vel, 3)
    n = len(pos)
    ctor = np.broadcast_to(np.asarray(ctor, dtype=np.float64), (n, 12))
    mass = np.broadcast_to(np.asarray(mass, dtype=np.float64).reshape(-1), (n,))
    sl = None if slope is None else f(slope, 2)
    af = f(fluid_accel, 3)
    a = (v - f(prev_lin, 3)) / dt
    al = (w - f(prev_ang, 3)) / dt
    wd, dp, ht, rho = ctor[:, 0], ctor[:, 1], ctor[:, 2], ctor[:, 7]
    vol = (wd * dp) * ht
    if dense is None:  # numba_hydrodynamics_wrapper.py:101-112
        lin_c, ang_c = ctor[:, 9], ctor[:, 10]
        M = np.zeros((n, 6, 6))
        for k in range(3):
            M[:, k, k] = (vol * lin_c) * rho
        M[:, 3, 3] = ((vol * (dp * dp + ht * ht)) * ang_c) * rho
        M[:, 4, 4] = ((vol * (wd * wd + ht * ht)) * ang_c) * rho
        M[:, 5, 5] = ((vol * (wd * wd + dp * dp)) * ang_c) * rho
    else:
        st = np.asarray(dense_slot, dtype=np.int64).reshape(-1)
        M = np.asarray(dense, dtype=np.float64).reshape(-1, 6, 6)[st[np.arange(n) % len(st)]]
    # the added mass on the fluid-relative acceleration: a enters _solve only there
    fb, fd, fl, td, fam, tam, cob, cop, ratio = SR._solve(ctor, pos, q, v, w, a - af, al, sl, False, M)
    ffk = (rho * (ratio * vol))[:, None] * af  # Froude-Krylov, zero for a dry body (ratio 0)

    tb = SR._cross(cob - pos, fb)
    tdrag = SR._cross(cop - pos, fd)
    tl = SR._cross(cop - pos, fl)
    tfk = SR._cross(cob - pos, ffk)
    F = (((fb + fd) + fl) + fam) + ffk
    T = ((((tb + tdrag) + tl) + td) + tam) + tfk
    scale = np.minimum((mass * 500.0) / (SR._norm(F) + 1e-6), 1.0)
    return SR.StepResult(F * scale[:, None], T * scale[:, None], ratio)


def inertia_magnitude(ctor, sub_ratio, fluid_accel, dense=None, dense_slot=None):
    """|F_FK| + |added-mass force on a_f| per body (the new group's size, for checks that it is not vacuous)."""
    ctor = np.asarray(ctor, dtype=np.float64)
    af = np.asarray(fluid_accel, dtype=np.float64).reshape(-1, 3)
    ctor = np.broadcast_to(ctor, (len(af), 12))
    vol = (ctor[:, 0] * ctor[:, 1]) * ctor[:, 2]
    k = ctor[:, 7] * sub_ratio * vol
    c_am = ctor[:, 9] if dense is None else 0.0
    return k * (1.0 + c_am) * np.linalg.norm(af, axis=1)
