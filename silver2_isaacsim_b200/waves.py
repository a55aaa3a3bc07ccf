"""Linear (Airy) wave fields for the engine's built-in wave evaluator (``HydroEngine.set_wave_field``).

A field is a sum of components ``(a, kx, ky, omega, phase)`` over water of depth ``h`` (``inf`` = deep
water); ``include/h2o.h`` (``h2o_set_wave_field``) pins the formulas.  This module builds fields
(``regular``, ``jonswap``), solves the dispersion relation and evaluates a field in float64
(``evaluate``, the reference the GPU evaluator is tested against).  NumPy only.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

MAX_COMPONENTS = 64  # h2o_set_wave_field


def _check_depth(depth) -> float:
    depth = float(depth)
    if not depth > 0.0:  # also NaN and -inf
        raise ValueError(f"depth must be > 0 (inf = deep water), got {depth}")
    return depth


@dataclass(frozen=True)
class WaveField:
    """``components``: (n, 5) float64 rows ``a, kx, ky, omega, phase``; ``depth``: water depth (``inf`` = deep)."""

    components: np.ndarray
    depth: float = math.inf

    def __post_init__(self):
        c = np.array(self.components, dtype=np.float64)  # a private copy
        if c.ndim != 2 or c.shape[1] != 5:
            raise ValueError("components must be an (n, 5) array of a, kx, ky, omega, phase")
        if len(c) > MAX_COMPONENTS:
            raise ValueError(f"at most {MAX_COMPONENTS} components, got {len(c)}")
        if not np.isfinite(c).all():
            raise ValueError("components must be finite")
        if (c[:, 0] < 0).any():
            raise ValueError("amplitudes must be >= 0")
        if ((c[:, 1] == 0) & (c[:, 2] == 0)).any():
            raise ValueError("every wave vector (kx, ky) must be non-zero")
        if not (c[:, 3] > 0).all():
            raise ValueError("angular frequencies must be > 0")
        c.setflags(write=False)
        object.__setattr__(self, "components", c)
        object.__setattr__(self, "depth", _check_depth(self.depth))

    @property
    def n_components(self) -> int:
        return len(self.components)


def wavenumber(omega, depth=math.inf, g: float = 9.81):
    """Wavenumber k of the linear dispersion relation ``omega^2 = g k tanh(k h)`` (Newton's method on
    ``x tanh x = omega^2 h / g``, x = k h; deep water: ``omega^2 / g``).  ``omega`` may be an array."""
    w = np.asarray(omega, dtype=np.float64)
    if not (np.isfinite(w).all() and (w > 0).all()):
        raise ValueError("omega must be finite and > 0")
    if not g > 0:
        raise ValueError("g must be > 0")
    h = _check_depth(depth)
    k_deep = w * w / g
    if math.isinf(h):
        return k_deep if k_deep.ndim else float(k_deep)
    y = k_deep * h
    x = y / np.sqrt(np.tanh(y ** 0.75)) ** (4.0 / 3.0)  # Fenton & McKee (1990): within ~1 % everywhere
    for _ in range(50):
        th = np.tanh(x)
        dx = (x * th - y) / (th + x * (1.0 - th * th))
        x = x - dx
        if (np.abs(dx) <= 4e-16 * x).all():
            break
    k = x / h
    return k if k.ndim else float(k)


def regular(amplitude: float, period: float, direction: float = 0.0, phase: float = 0.0, depth=math.inf,
            g: float = 9.81) -> WaveField:
    """One regular wave of amplitude ``amplitude`` (m) and period ``period`` (s) travelling towards
    ``direction`` (radians from +x)."""
    if not period > 0:
        raise ValueError("period must be > 0")
    omega = 2.0 * math.pi / period
    k = wavenumber(omega, depth, g)
    return WaveField(np.array([[amplitude, k * math.cos(direction), k * math.sin(direction), omega, phase]]), depth)


def jonswap(hs: float, tp: float, gamma: float = 3.3, n_components: int = 32, direction: float = 0.0, seed: int = 0,
            depth=math.inf, g: float = 9.81) -> WaveField:
    """Unidirectional JONSWAP sea: ``n_components`` equal-width frequency bins over [0.5, 3] x the peak
    frequency ``1 / tp``, amplitude ``sqrt(2 S(f) df)`` at each bin centre, seeded uniform random phases.
    The spectrum is scaled so that the components carry exactly the variance ``(hs / 4)^2``."""
    if not (hs > 0 and tp > 0 and gamma >= 1):
        raise ValueError("need hs > 0, tp > 0 and gamma >= 1")
    if not 1 <= int(n_components) <= MAX_COMPONENTS:
        raise ValueError(f"n_components must be in [1, {MAX_COMPONENTS}]")
    n = int(n_components)
    fp = 1.0 / tp
    f_lo, f_hi = 0.5 * fp, 3.0 * fp
    df = (f_hi - f_lo) / n
    f = f_lo + (np.arange(n) + 0.5) * df
    sigma = np.where(f <= fp, 0.07, 0.09)
    shape = f ** -5.0 * np.exp(-1.25 * (fp / f) ** 4) * gamma ** np.exp(-((f - fp) ** 2) / (2.0 * sigma ** 2 * fp ** 2))
    var = shape * df
    a = np.sqrt(2.0 * var * (hs / 4.0) ** 2 / var.sum())
    omega = 2.0 * math.pi * f
    k = wavenumber(omega, depth, g)
    phase = np.random.default_rng(seed).uniform(0.0, 2.0 * math.pi, n)
    comps = np.stack([a, k * math.cos(direction), k * math.sin(direction), omega, phase], axis=1)
    return WaveField(comps, depth)


def _per_point(x, m: int):
    """A scalar stays a Python float; an array becomes an (m, 1) float64 column."""
    if np.ndim(x) == 0:
        return float(x)
    x = np.asarray(x, dtype=np.float64).reshape(-1)
    if x.shape != (m,):
        raise ValueError(f"expected a scalar or {m} values, got {x.shape[0]}")
    return x[:, None]


def evaluate(field: WaveField, points, t, surface_z=0.0) -> np.ndarray:
    """Float64 reference of the field at ``points`` (m, 3) and clock ``t``: (m, 4) rows ``eta, ux, uy, uz``.
    The phase is formed in the order the GPU evaluator forms it, ``((kx px + ky py) - omega t) + phase``.
    ``t`` and ``surface_z`` are scalars or one value per point."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    t, surface_z = _per_point(t, len(p)), _per_point(surface_z, len(p))
    c = field.components
    a, kx, ky, w, ph = (c[:, j][None, :] for j in range(5))
    k = np.hypot(kx, ky)
    h = field.depth
    z = np.minimum(p[:, 2:3] - surface_z, 0.0)
    if math.isinf(h):
        C = S = np.exp(k * z)
    else:
        z = np.maximum(z, -h)
        inv = -1.0 / np.expm1(-2.0 * k * h)
        e0, e1 = np.exp(k * z), np.exp(-k * (z + 2.0 * h))
        C, S = (e0 + e1) * inv, (e0 - e1) * inv   # cosh(k(z+h)) / sinh(kh), sinh(k(z+h)) / sinh(kh)
    th = ((kx * p[:, 0:1] + ky * p[:, 1:2]) - w * t) + ph
    cs, sn = np.cos(th), np.sin(th)
    uh = a * w * C * cs
    out = np.empty((len(p), 4))
    out[:, 0] = (a * cs).sum(axis=1)
    out[:, 1] = (uh * (kx / k)).sum(axis=1)
    out[:, 2] = (uh * (ky / k)).sum(axis=1)
    out[:, 3] = (a * w * S * sn).sum(axis=1)
    return out


def slope(field: WaveField, points, t) -> np.ndarray:
    """Float64 reference of the surface slope at ``points`` (m, 3) (only x, y matter) and clock ``t`` (scalar or one
    per point): (m, 2) rows ``sx, sy`` = the gradient of ``eta``, ``sum_j -a_j (kx_j, ky_j) sin theta_j`` with the
    ``theta_j`` of ``evaluate`` (include/h2o.h, h2o_set_wave_slope)."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    t = _per_point(t, len(p))
    c = field.components
    a, kx, ky, w, ph = (c[:, j][None, :] for j in range(5))
    th = ((kx * p[:, 0:1] + ky * p[:, 1:2]) - w * t) + ph
    asn = a * np.sin(th)
    out = np.empty((len(p), 2))
    out[:, 0] = -(asn * kx).sum(axis=1)
    out[:, 1] = -(asn * ky).sum(axis=1)
    return out


def acceleration(field: WaveField, points, t, surface_z=0.0) -> np.ndarray:
    """Float64 reference of the water's acceleration at ``points`` (m, 3) and clock ``t``: (m, 3) rows ``ax, ay, az``,
    the time derivative of ``evaluate``'s orbital velocity, ``sum_j a_j omega_j^2 (C_j sin theta_j khat_j,
    -S_j cos theta_j)`` with the ``theta_j``, ``C_j``, ``S_j`` and depth clamp of ``evaluate`` (include/h2o.h,
    h2o_set_fluid_inertia).  ``t`` and ``surface_z`` are scalars or one value per point."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    t, surface_z = _per_point(t, len(p)), _per_point(surface_z, len(p))
    c = field.components
    a, kx, ky, w, ph = (c[:, j][None, :] for j in range(5))
    k = np.hypot(kx, ky)
    h = field.depth
    z = np.minimum(p[:, 2:3] - surface_z, 0.0)
    if math.isinf(h):
        C = S = np.exp(k * z)
    else:
        z = np.maximum(z, -h)
        inv = -1.0 / np.expm1(-2.0 * k * h)
        e0, e1 = np.exp(k * z), np.exp(-k * (z + 2.0 * h))
        C, S = (e0 + e1) * inv, (e0 - e1) * inv
    th = ((kx * p[:, 0:1] + ky * p[:, 1:2]) - w * t) + ph
    aw2 = (a * w) * w
    ah = aw2 * C * np.sin(th)
    out = np.empty((len(p), 3))
    out[:, 0] = (ah * (kx / k)).sum(axis=1)
    out[:, 1] = (ah * (ky / k)).sum(axis=1)
    out[:, 2] = -(aw2 * S * np.cos(th)).sum(axis=1)
    return out


# Columns of a per-env conditions row (HydroEngine.set_env_conditions, h2o_set_env_conditions)
COND_CX, COND_CY, COND_CZ, COND_DZ, COND_SCALE, COND_TAU, COND_X0, COND_Y0 = range(8)
COND_COLS = 8


def _cond_column(x, n: int, width: int, name: str) -> np.ndarray:
    a = np.asarray(x, dtype=np.float64)
    if a.ndim == 0 or a.shape == (width,):
        a = np.broadcast_to(a, (n, width))
    elif width == 1 and a.shape == (n,):
        a = a[:, None]
    if a.shape != (n, width):
        shapes = "a scalar or (E,)" if width == 1 else f"a scalar, ({width},) or (E, {width})"
        raise ValueError(f"{name} must be {shapes} with E = {n}, got {np.shape(x)}")
    if not np.isfinite(a).all():
        raise ValueError(f"{name} must be finite")
    return a


def env_conditions(n_envs: int, current=0.0, surface_dz=0.0, wave_scale=1.0, time_offset=0.0, origin=0.0) -> np.ndarray:
    """Per-env conditions, an (E, 8) float64 array of rows ``cx, cy, cz, dz, s, tau, x0, y0``: the current added to
    the global one, the water-level offset, the wave scale, the wave time offset (s) and the env origin.  Each
    argument is a scalar, one value for every env (``current`` (3,), ``origin`` (2,)) or one per env; the
    defaults make identity rows ``[0, 0, 0, 0, 1, 0, 0, 0]``, which leave every result unchanged."""
    n = int(n_envs)
    if n < 1:
        raise ValueError(f"n_envs must be >= 1, got {n_envs}")
    cond = np.empty((n, COND_COLS))
    cond[:, COND_CX:COND_CZ + 1] = _cond_column(current, n, 3, "current")
    cond[:, COND_DZ] = _cond_column(surface_dz, n, 1, "surface_dz")[:, 0]
    cond[:, COND_SCALE] = _cond_column(wave_scale, n, 1, "wave_scale")[:, 0]
    cond[:, COND_TAU] = _cond_column(time_offset, n, 1, "time_offset")[:, 0]
    cond[:, COND_X0:COND_Y0 + 1] = _cond_column(origin, n, 2, "origin")
    return cond


def evaluate_env(field: WaveField, points, t: float, cond, env_index, surface_z: float = 0.0) -> np.ndarray:
    """Float64 reference of what env ``env_index[k]`` sees of the field at ``points[k]`` and clock ``t``:
    ``s * evaluate(field, p - origin, t + tau, surface_z + dz)`` with the env's row of ``cond`` (E, 8), as rows
    ``s eta, s ux, s uy, s uz`` (the field alone, as ``HydroEngine.sample_waves(points, env)`` returns it)."""
    p = np.array(points, dtype=np.float64).reshape(-1, 3)
    cond = np.asarray(cond, dtype=np.float64)
    if cond.ndim != 2 or cond.shape[1] != COND_COLS:
        raise ValueError(f"cond must be (E, {COND_COLS}), got {cond.shape}")
    r = cond[np.asarray(env_index, dtype=np.int64).reshape(-1)]
    if len(r) != len(p):
        raise ValueError("need one env index per point")
    p[:, 0] = p[:, 0] - r[:, COND_X0]
    p[:, 1] = p[:, 1] - r[:, COND_Y0]
    out = evaluate(field, p, t + r[:, COND_TAU], surface_z + r[:, COND_DZ])
    return r[:, COND_SCALE:COND_SCALE + 1] * out


def slope_env(field: WaveField, points, t: float, cond, env_index) -> np.ndarray:
    """Float64 reference of the slope env ``env_index[k]`` sees at ``points[k]`` and clock ``t``:
    ``s * slope(field, p - origin, t + tau)`` with the env's row of ``cond`` (E, 8), as ``evaluate_env`` forms it
    (``HydroEngine.sample_surface_slope(points, env)`` with the mode on)."""
    p = np.array(points, dtype=np.float64).reshape(-1, 3)
    cond = np.asarray(cond, dtype=np.float64)
    if cond.ndim != 2 or cond.shape[1] != COND_COLS:
        raise ValueError(f"cond must be (E, {COND_COLS}), got {cond.shape}")
    r = cond[np.asarray(env_index, dtype=np.int64).reshape(-1)]
    if len(r) != len(p):
        raise ValueError("need one env index per point")
    p[:, 0] = p[:, 0] - r[:, COND_X0]
    p[:, 1] = p[:, 1] - r[:, COND_Y0]
    return r[:, COND_SCALE:COND_SCALE + 1] * slope(field, p, t + r[:, COND_TAU])


def acceleration_env(field: WaveField, points, t: float, cond, env_index, surface_z: float = 0.0) -> np.ndarray:
    """Float64 reference of the water's acceleration env ``env_index[k]`` sees at ``points[k]`` and clock ``t``:
    ``s * acceleration(field, p - origin, t + tau, surface_z + dz)`` with the env's row of ``cond`` (E, 8), as
    ``evaluate_env`` forms it."""
    p = np.array(points, dtype=np.float64).reshape(-1, 3)
    cond = np.asarray(cond, dtype=np.float64)
    if cond.ndim != 2 or cond.shape[1] != COND_COLS:
        raise ValueError(f"cond must be (E, {COND_COLS}), got {cond.shape}")
    r = cond[np.asarray(env_index, dtype=np.int64).reshape(-1)]
    if len(r) != len(p):
        raise ValueError("need one env index per point")
    p[:, 0] = p[:, 0] - r[:, COND_X0]
    p[:, 1] = p[:, 1] - r[:, COND_Y0]
    out = acceleration(field, p, t + r[:, COND_TAU], surface_z + r[:, COND_DZ])
    return r[:, COND_SCALE:COND_SCALE + 1] * out
