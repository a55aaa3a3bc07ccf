"""Gridded water currents for the engine's current grid (``HydroEngine.set_current_grid``).

A current grid is a space-time lattice of velocity vectors, float64 ``(nt, nz, ny, nx, 3)``; node ``(f, k, j, i)``
sits at ``origin + (i, j, k) * spacing`` and at time ``t0 + f * frame_dt``.  ``include/h2o.h``
(``h2o_set_current_grid``) pins the interpolation.  This module builds grids (``CurrentGrid``, ``profile``,
``power_law_profile``) and evaluates one in float64 with the operations of the GPU evaluator, in the same order
(``evaluate``, the reference the engine is tested against bit for bit).  NumPy only.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np


def _vec3(x, name: str) -> tuple:
    a = np.asarray(x, dtype=np.float64)
    if a.shape != (3,) or not np.isfinite(a).all():
        raise ValueError(f"{name} must be 3 finite values, got {x!r}")
    return tuple(float(v) for v in a)


@dataclass(frozen=True)
class CurrentGrid:
    """``values``: (nt, nz, ny, nx, 3) or (nz, ny, nx, 3) float64 velocities (a private, read-only copy, always
    5-D); ``origin``: (gx, gy, gz); ``spacing``: (hx, hy, hz) > 0; ``t0``: time of frame 0; ``frame_dt``: time
    between frames (> 0 when there is more than one).  z is measured from the mean water level."""

    values: np.ndarray
    origin: tuple = (0.0, 0.0, 0.0)
    spacing: tuple = (1.0, 1.0, 1.0)
    t0: float = 0.0
    frame_dt: float = 0.0

    def __post_init__(self):
        v = np.array(self.values, dtype=np.float64, order="C")
        if v.ndim == 4:
            v = v[None]
        if v.ndim != 5 or v.shape[-1] != 3 or 0 in v.shape:
            raise ValueError(f"values must be (nt, nz, ny, nx, 3) or (nz, ny, nx, 3), got {np.shape(self.values)}")
        if not np.isfinite(v).all():
            raise ValueError("values must be finite")
        v.setflags(write=False)
        spacing = _vec3(self.spacing, "spacing")
        if min(spacing) <= 0.0:
            raise ValueError(f"spacing must be > 0, got {spacing}")
        t0, frame_dt = float(self.t0), float(self.frame_dt)
        if not (math.isfinite(t0) and math.isfinite(frame_dt)):
            raise ValueError("t0 and frame_dt must be finite")
        if v.shape[0] > 1 and frame_dt <= 0.0:
            raise ValueError(f"frame_dt must be > 0 with {v.shape[0]} frames, got {frame_dt}")
        object.__setattr__(self, "values", v)
        object.__setattr__(self, "origin", _vec3(self.origin, "origin"))
        object.__setattr__(self, "spacing", spacing)
        object.__setattr__(self, "t0", t0)
        object.__setattr__(self, "frame_dt", frame_dt)

    @property
    def dims(self) -> tuple:
        """``(nt, nz, ny, nx)``."""
        return tuple(self.values.shape[:4])

    @property
    def geometry(self) -> np.ndarray:
        """``[gx, gy, gz, hx, hy, hz, t0, ht]``, the geometry ``h2o_set_current_grid`` takes."""
        return np.array([*self.origin, *self.spacing, self.t0, self.frame_dt])


def profile(z, velocity) -> CurrentGrid:
    """A depth profile: ``velocity`` (nz, 3) at the evenly spaced, increasing levels ``z`` (nz,) (measured from the
    mean water level), the same at every x and y (``nx = ny = 1``), constant in time."""
    z = np.asarray(z, dtype=np.float64).reshape(-1)
    vel = np.asarray(velocity, dtype=np.float64)
    if vel.shape != (len(z), 3) or len(z) == 0:
        raise ValueError(f"velocity must be (nz, 3) for nz = len(z) = {len(z)} levels, got {vel.shape}")
    if not np.isfinite(z).all():
        raise ValueError("levels must be finite")
    hz = 1.0
    if len(z) > 1:
        hz = (z[-1] - z[0]) / (len(z) - 1)
        if not hz > 0 or not np.allclose(np.diff(z), hz, rtol=1e-9, atol=0.0):
            raise ValueError("levels must be evenly spaced and increasing")
    return CurrentGrid(vel.reshape(1, len(z), 1, 1, 3), origin=(0.0, 0.0, z[0]), spacing=(1.0, 1.0, hz))


def power_law_profile(speed: float, direction: float, seabed_z: float, top_z: float = 0.0, alpha: float = 1.0 / 7.0,
                      nz: int = 32) -> CurrentGrid:
    """The classical seabed boundary layer: a horizontal current towards ``direction`` (radians from +x) of speed
    ``speed * ((z - seabed_z) / (top_z - seabed_z)) ** alpha`` at ``nz`` levels from ``seabed_z`` (zero) to
    ``top_z`` (``speed``); held above ``top_z`` and below the seabed (z from the mean water level)."""
    speed, direction, seabed_z, top_z, alpha = (float(x) for x in (speed, direction, seabed_z, top_z, alpha))
    if not all(math.isfinite(x) for x in (speed, direction, seabed_z, top_z, alpha)):
        raise ValueError("arguments must be finite")
    if not top_z > seabed_z:
        raise ValueError(f"top_z ({top_z}) must be above seabed_z ({seabed_z})")
    if not alpha > 0 or int(nz) < 2:
        raise ValueError("need alpha > 0 and nz >= 2")
    z = np.linspace(seabed_z, top_z, int(nz))
    u = speed * ((z - seabed_z) / (top_z - seabed_z)) ** alpha
    vel = np.stack([u * math.cos(direction), u * math.sin(direction), np.zeros_like(u)], axis=1)
    return profile(z, vel)


def _axis(q, n: int, o: float, h: float):
    """Lower node and weight on one axis, as grid_axis in csrc/h2o_waves.cuh (q without NaN)."""
    if n == 1:
        return np.zeros(q.shape, np.int64), np.zeros(q.shape)
    top = float(n - 1)
    u = (q - o) / h
    u = np.where(u > 0.0, np.where(u < top, u, top), 0.0)
    i = np.minimum(np.floor(u).astype(np.int64), n - 2)
    return i, u - i


def _lerp(a, b, w):
    return a + w[:, None] * (b - a)


def evaluate(grid: CurrentGrid, x, y, z, t) -> np.ndarray:
    """Float64 reference of the grid at grid-frame points ``x, y, z`` and times ``t`` (scalars or one value per
    point): (m, 3) velocities, interpolated along x, then y, then z, then t with ``a + w (b - a)``, held at the
    boundary; NaN rows where a coordinate is NaN."""
    x, y, z, t = np.broadcast_arrays(*(np.asarray(q, dtype=np.float64).reshape(-1) for q in (x, y, z, t)))
    nan = np.isnan(x) | np.isnan(y) | np.isnan(z) | np.isnan(t)
    x, y, z, t = (np.where(nan, 0.0, q) for q in (x, y, z, t))
    it, wt = _axis(t, grid.dims[0], grid.t0, grid.frame_dt)
    along_z = _spatial(grid, x, y, z)
    out = along_z(it)
    if grid.dims[0] > 1:
        out = _lerp(out, along_z(it + 1), wt)
    out = np.array(out, dtype=np.float64)
    out[nan] = np.nan
    return out


def _spatial(grid: CurrentGrid, x, y, z):
    """The spatial interpolation at points x, y, z (without NaN): f -> (m, 3) values of frames f, along x, then y,
    then z."""
    v = grid.values
    _, nz, ny, nx = grid.dims
    (gx, gy, gz), (hx, hy, hz) = grid.origin, grid.spacing
    ix, wx = _axis(x, nx, gx, hx)
    iy, wy = _axis(y, ny, gy, hy)
    iz, wz = _axis(z, nz, gz, hz)

    def along_x(f, k, j):
        a = v[f, k, j, ix]
        return _lerp(a, v[f, k, j, ix + 1], wx) if nx > 1 else a

    def along_y(f, k):
        a = along_x(f, k, iy)
        return _lerp(a, along_x(f, k, iy + 1), wy) if ny > 1 else a

    def along_z(f):
        a = along_y(f, iz)
        return _lerp(a, along_y(f, iz + 1), wz) if nz > 1 else a

    return along_z


def time_derivative(grid: CurrentGrid, x, y, z, t) -> np.ndarray:
    """Float64 reference of the grid's time derivative at grid-frame points ``x, y, z`` and times ``t`` (scalars or one
    value per point): (m, 3) rows ``(G_{f+1} - G_f) / frame_dt``, with ``G_f``, ``G_{f+1}`` the spatial interpolations
    of the two frames ``evaluate`` blends at ``t``, for ``nt > 1`` and ``t`` inside ``[t0, t0 + (nt - 1) frame_dt]``;
    zero rows where the grid is held in time and for one frame; NaN rows where a coordinate is NaN (include/h2o.h,
    h2o_set_fluid_inertia)."""
    x, y, z, t = np.broadcast_arrays(*(np.asarray(q, dtype=np.float64).reshape(-1) for q in (x, y, z, t)))
    nan = np.isnan(x) | np.isnan(y) | np.isnan(z) | np.isnan(t)
    x, y, z, t = (np.where(nan, 0.0, q) for q in (x, y, z, t))
    out = np.zeros((len(x), 3))
    nt = grid.dims[0]
    if nt > 1:
        it, _ = _axis(t, nt, grid.t0, grid.frame_dt)
        u = (t - grid.t0) / grid.frame_dt
        inside = (u >= 0.0) & (u <= float(nt - 1))
        along_z = _spatial(grid, x, y, z)
        out = np.where(inside[:, None], (along_z(it + 1) - along_z(it)) / grid.frame_dt, 0.0)
    out[nan] = np.nan
    return out

