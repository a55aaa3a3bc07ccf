"""Float64 NumPy restatement of the C oracle's behaviour step with a sloped waterline plane.  TEST TOOL ONLY.

``step`` follows ``oracle/hydro_oracle.c`` (``oracle_step_batch`` -> ``oracle_solve`` -> ``oracle_net_wrench``, itself
a restatement of numba_hydrodynamics.py:8-314 and hydrodynamics_behavior.py:194-226) operation by operation, in the
same association order, vectorised over bodies: 27 explicit keypoints, 6 explicit faces, a dense 6x6 added-mass
matvec and world-space lever arms.  It adds one thing: an optional per-body slope ``(sx, sy)`` of the waterline plane
(include/h2o.h, ``h2o_set_wave_slope``).  With it, a world point ``w`` of a body at ``p`` (z measured from the body's
waterline) is under water iff ``(w_z - sx (w_x - p_x)) - sy (w_y - p_y) < 0``.  That test replaces ``w_z < 0`` in the
keypoint wet test, ``z_min`` / ``z_max`` and the face-centre wet test, and nowhere else.

Without a slope it is the oracle; tests/test_wave_slope.py checks it against the unmodified C oracle there (Numba and
Warp-twin semantics, diagonal and dense added mass).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np


@dataclass
class StepResult:
    force: np.ndarray      # (n,3) net force after the clamp
    torque: np.ndarray     # (n,3) net torque after the clamp
    sub_ratio: np.ndarray  # (n,) submersion ratio


def _rot(q, warp_compat):
    """quaternion_to_matrix (numba_hydrodynamics.py:8-51), xyzw, not normalised; the Warp twin adds 2 dq I (C7)."""
    x, y, z, w = (q[:, k] for k in range(4))
    x2, y2, z2 = x + x, y + y, z + z
    xx, xy, xz = x * x2, x * y2, x * z2
    yy, yz, zz = y * y2, y * z2, z * z2
    wx, wy, wz = w * x2, w * y2, w * z2
    m = np.empty((len(q), 3, 3))
    m[:, 0, 0] = 1.0 - (yy + zz); m[:, 0, 1] = xy - wz; m[:, 0, 2] = xz + wy
    m[:, 1, 0] = xy + wz; m[:, 1, 1] = 1.0 - (xx + zz); m[:, 1, 2] = yz - wx
    m[:, 2, 0] = xz - wy; m[:, 2, 1] = yz + wx; m[:, 2, 2] = 1.0 - (xx + yy)
    if warp_compat:
        d2 = 2.0 * (((x * x + y * y) + (z * z + w * w)) - 1.0)
        for k in range(3):
            m[:, k, k] = m[:, k, k] + d2
    return m


def _matvec(m, v):
    """matvec3: acc = m[r][0] v0; acc += m[r][1] v1; acc += m[r][2] v2 (v (n,3) or (3,))."""
    v = np.broadcast_to(v, (m.shape[0], 3))
    return np.stack([(m[:, r, 0] * v[:, 0] + m[:, r, 1] * v[:, 1]) + m[:, r, 2] * v[:, 2] for r in range(3)], axis=1)


def _matTvec(m, v):
    return np.stack([(m[:, 0, r] * v[:, 0] + m[:, 1, r] * v[:, 1]) + m[:, 2, r] * v[:, 2] for r in range(3)], axis=1)


def _norm(v):
    return np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])


def _cross(a, b):
    return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1],
                     a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                     a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1)


def _height(wp, pos, slope):
    """Height of world points wp (n,3) above the waterline plane of bodies at pos (z from the waterline)."""
    if slope is None:
        return wp[:, 2]
    return (wp[:, 2] - slope[:, 0] * (wp[:, 0] - pos[:, 0])) - slope[:, 1] * (wp[:, 1] - pos[:, 1])


def _solve(ctor, pos, q, v, w, a, al, slope, warp_compat, M):
    n = len(pos)
    wd, dp, ht = ctor[:, 0], ctor[:, 1], ctor[:, 2]
    cd, cda, kd, kda = ctor[:, 3], ctor[:, 4], ctor[:, 5], ctor[:, 6]
    rho, g, cl_param = ctor[:, 7], ctor[:, 8], ctor[:, 11]
    vol = (wd * dp) * ht
    rot = _rot(q, warp_compat)
    hx, hy, hz = wd / 2.0, dp / 2.0, ht / 2.0

    # ---- analyze_submersion_and_cob (numba_hydrodynamics.py:53-105), keypoints in the wrapper's order
    z_min = np.full(n, np.inf)
    z_max = np.full(n, -np.inf)
    sums = np.zeros((n, 3))
    count = np.zeros(n)
    zero = np.zeros(n)
    for zs in (hz, zero, -hz):
        for ys in (hy, zero, -hy):
            for xs in (-hx, zero, hx):
                wk = _matvec(rot, np.stack([xs, ys, zs], axis=1)) + pos
                h = _height(wk, pos, slope)
                z_min = np.where(h < z_min, h, z_min)
                z_max = np.where(h > z_max, h, z_max)
                wet = h < 0
                sums = sums + np.where(wet[:, None], wk, 0.0)
                count = count + wet
    inv_c = 1.0 / np.maximum(count, 1.0)
    mean = sums * inv_c[:, None]
    dry = z_min >= 0
    full = ~dry & (z_max <= 0)
    partial = ~dry & ~full
    total = z_max - z_min
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio_p = np.where(total < 1e-6, np.where(z_min < 0, 1.0, 0.0), np.minimum(-z_min / total, 1.0))
    ratio = np.where(dry, 0.0, np.where(full, 1.0, ratio_p))
    use_mean = (count > 0) & (partial | (full & warp_compat))
    cob = np.where(use_mean[:, None], mean, pos)
    wetb = ratio > 1e-9  # numba_hydrodynamics.py:277-279: every output zero otherwise

    fb = rho * (ratio * vol) * g
    speed = _norm(v)
    moving = speed > 1e-6
    with np.errstate(divide="ignore", invalid="ignore"):
        vd = np.where(moving[:, None], v / speed[:, None], 0.0)

    # ---- calculate_pressure_and_area (numba_hydrodynamics.py:107-143)
    tot = np.zeros(n)
    cws = np.zeros((n, 3))
    faces = ((hx, zero, zero, (1, 0, 0), dp * ht), (-hx, zero, zero, (-1, 0, 0), dp * ht),
             (zero, hy, zero, (0, 1, 0), wd * ht), (zero, -hy, zero, (0, -1, 0), wd * ht),
             (zero, zero, hz, (0, 0, 1), wd * dp), (zero, zero, -hz, (0, 0, -1), wd * dp))
    for cx, cy, cz, nrm, farea in faces:
        wn = _matvec(rot, np.array(nrm, dtype=np.float64))
        wc = _matvec(rot, np.stack([cx, cy, cz], axis=1)) + pos
        dotp = (wn[:, 0] * vd[:, 0] + wn[:, 1] * vd[:, 1]) + wn[:, 2] * vd[:, 2]
        align = -dotp
        take = moving & (align > 0) & (_height(wc, pos, slope) < 0)
        av = np.where(take, align * farea, 0.0)
        tot = tot + av
        cws = cws + np.where(take[:, None], wc * av[:, None], 0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        cop = np.where((moving & (tot > 1e-6))[:, None], cws / tot[:, None], cob)
    area = np.where(moving, tot, 0.0)

    # ---- calculate_hybrid_drag (numba_hydrodynamics.py:145-182)
    drag_mag = ((0.5 * rho) * (speed * speed)) * cd * area
    quad = np.where(moving[:, None], -drag_mag[:, None] * vd, 0.0)
    lds = np.where(speed < 0.2, speed / 0.2, 1.0)
    fd = (quad + ((-kd)[:, None] * v) * lds[:, None]) * ratio[:, None]
    aspeed = _norm(w)
    amov = aspeed > 1e-6
    ang_mag = ((0.5 * rho) * (aspeed * aspeed)) * cda * vol
    with np.errstate(divide="ignore", invalid="ignore"):
        quad_t = np.where(amov[:, None], -ang_mag[:, None] * (w / aspeed[:, None]), 0.0)
    ads = np.where(aspeed < 0.2, aspeed / 0.2, 1.0)
    td = (quad_t + ((-kda)[:, None] * w) * ads[:, None]) * ratio[:, None]

    # ---- calculate_lift (numba_hydrodynamics.py:184-217)
    up = rot[:, :, 2]
    dotp = -((up[:, 0] * vd[:, 0] + up[:, 1] * vd[:, 1]) + up[:, 2] * vd[:, 2])
    dotp = np.clip(dotp, -1.0, 1.0)
    clift = np.sin(2 * np.arcsin(dotp))
    lmag = (((0.5 * rho) * (speed * speed)) * clift * area) * cl_param
    axis = _cross(vd, up)
    an = _norm(axis)
    ok = ~(speed < 1e-6) & (ratio > 1e-9) & ~(an < 1e-6)
    with np.errstate(divide="ignore", invalid="ignore"):
        axis = axis / an[:, None]
    ldir = _cross(axis, vd)
    fl = np.where(ok[:, None], (lmag[:, None] * ldir) * ratio[:, None], 0.0)

    # ---- calculate_added_mass (numba_hydrodynamics.py:219-253)
    acc6 = np.concatenate([_matvec(rot, a), _matvec(rot, al)] if warp_compat else [_matTvec(rot, a), _matTvec(rot, al)],
                          axis=1)
    ft = np.zeros((n, 6))
    for i in range(6):
        acc = np.zeros(n)
        for j in range(6):
            acc = acc + M[:, i, j] * acc6[:, j]
        ft[:, i] = -1.0 * acc
    fam = np.where(wetb[:, None], _matvec(rot, ft[:, 0:3]) * ratio[:, None], 0.0)
    tam = np.where(wetb[:, None], _matvec(rot, ft[:, 3:6]) * ratio[:, None], 0.0)

    z3 = np.zeros((n, 3))
    fbv = np.stack([zero, zero, fb], axis=1)
    keep = wetb[:, None]
    cob_out = np.where(keep, cob, pos if warp_compat else z3)
    cop_out = np.where(keep, cop, pos if warp_compat else z3)
    return (np.where(keep, fbv, z3), np.where(keep, fd, z3), np.where(keep, fl, z3), np.where(keep, td, z3), fam, tam,
            cob_out, cop_out, np.where(wetb, ratio, 0.0))


def step(ctor, mass, pos, quat_xyzw, lin_vel, ang_vel, prev_lin, prev_ang, dt, slope=None, warp_compat=False,
         dense=None, dense_slot=None) -> StepResult:
    """One behaviour step for n bodies in float64, as ``oracle.step`` (xyzw quaternions), with the optional per-body
    waterline slope ``slope`` (n,2) [sx, sy].  ``ctor``: (n,12) wrapper-ctor rows; ``warp_compat``: the Warp twin's
    deviations C1, C3, C7, C9; ``dense``: (n_types,6,6) added-mass matrices, body i using ``dense[dense_slot[i %
    len(dense_slot)]]`` instead of the wrapper's diagonal."""
    f = lambda x, k: np.ascontiguousarray(np.asarray(x, dtype=np.float64)).reshape(-1, k)
    pos, q, v, w = f(pos, 3), f(quat_xyzw, 4), f(lin_vel, 3), f(ang_vel, 3)
    n = len(pos)
    ctor = np.broadcast_to(np.asarray(ctor, dtype=np.float64), (n, 12))
    mass = np.broadcast_to(np.asarray(mass, dtype=np.float64).reshape(-1), (n,))
    sl = None if slope is None else f(slope, 2)
    a = (v - f(prev_lin, 3)) / dt
    al = (w - f(prev_ang, 3)) / dt
    if dense is None:  # numba_hydrodynamics_wrapper.py:101-112
        wd, dp, ht, lin_c, ang_c, rho = ctor[:, 0], ctor[:, 1], ctor[:, 2], ctor[:, 9], ctor[:, 10], ctor[:, 7]
        vol = (wd * dp) * ht
        M = np.zeros((n, 6, 6))
        for k in range(3):
            M[:, k, k] = (vol * lin_c) * rho
        M[:, 3, 3] = ((vol * (dp * dp + ht * ht)) * ang_c) * rho
        M[:, 4, 4] = ((vol * (wd * wd + ht * ht)) * ang_c) * rho
        M[:, 5, 5] = ((vol * (wd * wd + dp * dp)) * ang_c) * rho
    else:
        st = np.asarray(dense_slot, dtype=np.int64).reshape(-1)
        M = np.asarray(dense, dtype=np.float64).reshape(-1, 6, 6)[st[np.arange(n) % len(st)]]
    fb, fd, fl, td, fam, tam, cob, cop, ratio = _solve(ctor, pos, q, v, w, a, al, sl, warp_compat, M)

    # ---- hydrodynamics_behavior.py:212-226 (oracle_net_wrench)
    tb = _cross(cob - pos, fb)
    tdrag = _cross(cop - pos, fd)
    tl = _cross(cop - pos, fl)
    F = ((fb + fd) + fl) + fam
    T = (((tb + tdrag) + tl) + td) + tam
    scale = np.minimum((mass * 500.0) / (_norm(F) + 1e-6), 1.0)
    return StepResult(F * scale[:, None], T * scale[:, None], ratio)
