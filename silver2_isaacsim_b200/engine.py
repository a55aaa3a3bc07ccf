"""Batched hydrodynamics force engine: PyTorch host side over the C ABI.

One ``HydroEngine`` replaces N instances of the reference's per-prim stack

    HydrodynamicsBehavior._apply_behavior        hydrodynamics_behavior.py:176-238
    -> WarpHydrodynamicsWrapper.calculate_...    warp_hydrodynamics_wrapper.py:79-132
    -> solve_hydrodynamics_kernel<<<dim=1>>>     warp_hydrodynamics.py:234

with one fused sm_100a kernel launch for all bodies.  PyTorch is used for device
memory, streams and (elsewhere) ``torch.distributed``; tensors cross the boundary
zero-copy as DLPack descriptors; the arithmetic lives in ``csrc/``.
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Sequence, Tuple

import numpy as np
import torch
from torch.utils import dlpack as _dlpack

from . import _lib as L
from . import params as P
from . import waves as W

_TORCH_DTYPES = {torch.float32: L.H2O_F32, torch.float64: L.H2O_F64}
_NP_DTYPES = {L.H2O_F32: np.float32, L.H2O_F64: np.float64}


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class _DL:
    """Keeps DLPack capsules alive for the duration of one C call."""

    def __init__(self):
        self.keep = []

    def __call__(self, t: Optional[torch.Tensor]):
        if t is None:
            return None
        cap = _dlpack.to_dlpack(t)
        self.keep.append(cap)
        return L.capsule_pointer(cap)


class HydroEngine:
    """Hydrodynamic force/torque engine for ``n_bodies`` rigid boxes on one GPU.

    Parameters mirror the reference surface: ``water_density`` / ``gravity`` are the
    ``waterDensity`` / ``gravity`` exposed variables (hydrodynamics_behavior.py:30-31).
    Coefficients are set with one of ``set_params_uniform`` (the reference wrapper ctor),
    ``set_part_table`` (hydrodynamics_config.json parts) or ``set_params_per_body``.
    """

    def __init__(self, n_bodies: int, dtype: torch.dtype = torch.float32, device="cuda:0",
                 water_density: float = 1025.0, gravity: float = 9.81,
                 quat_order: str = "xyzw"):
        if dtype not in _TORCH_DTYPES:
            raise TypeError(f"dtype must be torch.float32 or torch.float64, got {dtype}")
        self._lib = L.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("HydroEngine runs on CUDA devices only (there is no CPU path)")
        self.dtype = dtype
        self.n_bodies = int(n_bodies)
        self.bodies_per_robot = 0
        self._h = ctypes.c_void_p()
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", index)
        L.check(self._lib.h2o_create(ctypes.byref(self._h), self.n_bodies, _TORCH_DTYPES[dtype], index))
        L.check(self._lib.h2o_set_globals(self._h, float(water_density), float(gravity)))
        self.water_density, self.gravity = float(water_density), float(gravity)
        self.quat_order = quat_order
        self._bound = None
        self._wave_slope = False
        self._fluid_inertia = False

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.h2o_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------ parameters
    @property
    def quat_order(self) -> str:
        return self._quat_order

    @quat_order.setter
    def quat_order(self, order: str):
        if order not in ("xyzw", "wxyz"):
            raise ValueError("quat_order must be 'xyzw' or 'wxyz'")
        L.check(self._lib.h2o_set_quat_order(self._h, L.H2O_QUAT_WXYZ if order == "wxyz" else L.H2O_QUAT_XYZW))
        self._quat_order = order

    def set_environment(self, current=(0.0, 0.0, 0.0), surface_z: float = 0.0):
        """Uniform water current (world frame) and height of the flat water surface; the defaults are
        the reference's still water with its surface at z = 0."""
        arr = (ctypes.c_double * 3)(*[float(x) for x in current])
        L.check(self._lib.h2o_set_environment(self._h, arr, float(surface_z)))

    def set_surface_heights(self, eta: Optional[torch.Tensor]):
        """Non-flat water surface: ``eta`` (n,) on the engine's device / dtype holds the surface elevation
        above ``surface_z`` at each body's position; it is read (not copied) by every later step, so the
        caller may update it in place between steps.  ``None`` = flat.  Steps then run on the per-body
        kernel."""
        if eta is None:
            L.check(self._lib.h2o_set_surface_heights(self._h, None))
            self._eta = None
            return
        if eta.device != self.device or eta.dtype != self.dtype or tuple(eta.shape) != (self.n_bodies,) or not eta.is_contiguous():
            raise ValueError(f"eta must be a contiguous ({self.n_bodies},) {self.dtype} tensor on {self.device}")
        L.check(self._lib.h2o_set_surface_heights(self._h, ctypes.c_void_p(eta.data_ptr())))
        self._eta = eta  # keep the borrowed memory alive

    def set_wave_field(self, field: Optional["W.WaveField"]):
        """Built-in linear wave field (``waves.regular`` / ``waves.jonswap`` / ``waves.WaveField``), evaluated on the
        GPU at every body's centre on every step at the engine's wave clock, which then advances by ``dt``.  The
        waterline becomes ``surface_z + eta`` and drag, damping and lift see ``v - (current + u)`` (semantics in
        include/h2o.h).  ``None`` removes the field.  Steps then run on the per-body kernel; ``rollout_persistent``
        and captured rollouts follow the field; ``components`` ignores it."""
        if field is None:
            L.check(self._lib.h2o_set_wave_field(self._h, 0, None, math.inf))
            return
        if not isinstance(field, W.WaveField):
            raise TypeError("field must be a waves.WaveField (waves.regular, waves.jonswap) or None")
        comps = np.ascontiguousarray(field.components, dtype=np.float64)
        L.check(self._lib.h2o_set_wave_field(self._h, int(comps.shape[0]),
                                             comps.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), float(field.depth)))

    def set_wave_slope(self, enable: bool = True):
        """Wave-slope submersion: with a wave field, test each body's keypoints and face centres against the wave
        surface's local tangent plane (slope ``-sum a k sin theta``, scaled per env) instead of the horizontal plane
        through its waterline, so that buoyancy and drag see a body tilted against the wave flank (semantics in
        include/h2o.h, h2o_set_wave_slope).  Off by default; without a wave field it changes nothing.  Drops a
        captured rollout; ``components`` ignores it."""
        L.check(self._lib.h2o_set_wave_slope(self._h, int(bool(enable))))
        self._wave_slope = bool(enable)

    @property
    def wave_slope(self) -> bool:
        """Whether wave-slope submersion is on (``set_wave_slope``)."""
        return self._wave_slope

    def sample_surface_slope(self, points, env=None) -> torch.Tensor:
        """The surface slope a step uses at ``points`` (m,3) world positions and the current clock: a (m,2) float64
        CUDA tensor of rows ``sx, sy`` (``waves.slope`` / ``waves.slope_env``), zeros with the mode off or without a
        wave field.  ``env`` as for ``sample_water``: an index outside ``[0, E)`` gives a NaN row."""
        pts = self._as_dev(points)
        if pts.ndim != 2 or pts.shape[1] != 3:
            raise ValueError(f"points must be (m,3), got {tuple(pts.shape)}")
        out = torch.empty(pts.shape[0], 2, dtype=torch.float64, device=self.device)
        idx = None if env is None else self._env_index(env, pts.shape[0])
        L.check(self._lib.h2o_water_slope_sample(self._h, ctypes.c_void_p(pts.data_ptr()),
                                                 None if idx is None else ctypes.c_void_p(idx.data_ptr()),
                                                 int(pts.shape[0]), ctypes.c_void_p(out.data_ptr()),
                                                 _stream_ptr(self.device)))
        return out

    def set_fluid_inertia(self, enable: bool = True):
        """Fluid-acceleration loads: the Froude-Krylov force ``rho r V a_f`` at the centre of buoyancy, and the added
        mass on the fluid-relative acceleration ``a_b - a_f``, with ``a_f`` the water's acceleration at each body's
        centre (waves, and a current grid with more than one frame; semantics in include/h2o.h,
        h2o_set_fluid_inertia).  Off by default; with still water it changes nothing.  Refused with Warp
        compatibility on (and ``set_warp_compat(True)`` is refused while it is on).  Drops a captured rollout;
        ``components`` ignores it."""
        L.check(self._lib.h2o_set_fluid_inertia(self._h, int(bool(enable))))
        self._fluid_inertia = bool(enable)

    @property
    def fluid_inertia(self) -> bool:
        """Whether fluid-acceleration loads are on (``set_fluid_inertia``)."""
        return self._fluid_inertia

    def sample_fluid_accel(self, points, env=None) -> torch.Tensor:
        """The fluid acceleration a step uses at ``points`` (m,3) world positions and the current clock: a (m,3)
        float64 CUDA tensor of rows ``ax, ay, az`` (``waves.acceleration`` plus ``currents.time_derivative``), zeros
        with the mode off or when nothing accelerates the water.  ``env`` as for ``sample_water``: an index outside
        ``[0, E)`` gives a NaN row."""
        pts = self._as_dev(points)
        if pts.ndim != 2 or pts.shape[1] != 3:
            raise ValueError(f"points must be (m,3), got {tuple(pts.shape)}")
        out = torch.empty(pts.shape[0], 3, dtype=torch.float64, device=self.device)
        idx = None if env is None else self._env_index(env, pts.shape[0])
        L.check(self._lib.h2o_fluid_accel_sample(self._h, ctypes.c_void_p(pts.data_ptr()),
                                                 None if idx is None else ctypes.c_void_p(idx.data_ptr()),
                                                 int(pts.shape[0]), ctypes.c_void_p(out.data_ptr()),
                                                 _stream_ptr(self.device)))
        return out

    @property
    def wave_time(self) -> float:
        """The wave clock (s): read after the work queued so far on the current stream (synchronises it)."""
        t = ctypes.c_double()
        L.check(self._lib.h2o_wave_time_read(self._h, ctypes.byref(t), _stream_ptr(self.device)))
        return t.value

    def set_wave_time(self, t: float):
        """Set the wave clock, in stream order.  A captured rollout is kept: it reads the clock from device memory."""
        t = float(t)
        if not math.isfinite(t):
            raise ValueError("wave time must be finite")
        L.check(self._lib.h2o_wave_time_write(self._h, t, _stream_ptr(self.device)))

    def sample_waves(self, points, env=None) -> torch.Tensor:
        """Wave field at ``points`` (m,3) world positions and the current clock, with the step's evaluator and
        precision: a (m,4) float64 CUDA tensor of rows ``eta, ux, uy, uz`` (zeros without a field).  With ``env``
        (one env index per point, or one for all), each point is seen from that env: rows ``s eta, s u`` at
        ``p - origin`` and ``clock + tau`` (``waves.evaluate_env``); an index outside ``[0, E)`` gives a NaN row."""
        pts, out = self._sample_buffers(points)
        if env is None:
            L.check(self._lib.h2o_wave_sample(self._h, ctypes.c_void_p(pts.data_ptr()), int(pts.shape[0]),
                                              ctypes.c_void_p(out.data_ptr()), _stream_ptr(self.device)))
            return out
        idx = self._env_index(env, pts.shape[0])
        L.check(self._lib.h2o_wave_sample_env(self._h, ctypes.c_void_p(pts.data_ptr()), ctypes.c_void_p(idx.data_ptr()),
                                              int(pts.shape[0]), ctypes.c_void_p(out.data_ptr()),
                                              _stream_ptr(self.device)))
        return out

    def sample_water(self, points, env=None) -> torch.Tensor:
        """What a step sees at ``points`` (m,3) world positions and the current clock: a (m,4) float64 CUDA tensor
        of rows ``waterline, flow_x, flow_y, flow_z``, the full composition of global environment, env row, current
        grid and wave field (include/h2o.h, h2o_water_sample), before a caller height array and before the fp32
        rounding.  ``env`` (one env index per point, or one for all) applies that env's conditions; ``None`` applies
        none; an index outside ``[0, E)`` gives a NaN row."""
        pts, out = self._sample_buffers(points)
        idx = None if env is None else self._env_index(env, pts.shape[0])
        L.check(self._lib.h2o_water_sample(self._h, ctypes.c_void_p(pts.data_ptr()),
                                           None if idx is None else ctypes.c_void_p(idx.data_ptr()), int(pts.shape[0]),
                                           ctypes.c_void_p(out.data_ptr()), _stream_ptr(self.device)))
        return out

    def _sample_buffers(self, points):
        pts = self._as_dev(points)
        if pts.ndim != 2 or pts.shape[1] != 3:
            raise ValueError(f"points must be (m,3), got {tuple(pts.shape)}")
        return pts, torch.empty(pts.shape[0], 4, dtype=torch.float64, device=self.device)

    def _env_index(self, env, m: int) -> torch.Tensor:
        idx = torch.as_tensor(env, device=self.device)
        if idx.dtype.is_floating_point or idx.dtype == torch.bool:
            raise ValueError("env must hold integer env indices")
        idx = idx.reshape(-1).long().clamp(-1, 2 ** 31 - 1).to(torch.int32)  # no wrap-around into [0, E)
        if idx.numel() == 1:
            idx = idx.expand(m)
        idx = idx.contiguous()
        if tuple(idx.shape) != (m,):
            raise ValueError(f"env must be one index or one per point ({m}), got {tuple(idx.shape)}")
        return idx

    def set_current_grid(self, values: Optional[torch.Tensor], origin=(0.0, 0.0, 0.0), spacing=(1.0, 1.0, 1.0),
                         t0: float = 0.0, frame_dt: float = 0.0):
        """Gridded water current: ``values`` is a contiguous float64 tensor on the engine's device, (nt,nz,ny,nx,3)
        or (nz,ny,nx,3) (one frame), of velocities at the nodes ``origin + (i, j, k) * spacing`` and times
        ``t0 + f * frame_dt`` (``currents.CurrentGrid`` builds them).  Every step interpolates it at each body's
        env-local position, depth below the env's mean level and env time, and adds it to the current
        (include/h2o.h).  The tensor is borrowed, not copied: in-place edits reach the next step and the next replay
        of a captured rollout.  ``None`` removes the grid.  Steps then run on the per-body kernel;
        ``rollout_persistent`` follows it; ``components`` ignores it."""
        if values is None:
            L.check(self._lib.h2o_set_current_grid(self._h, None, None, None))
            self._grid = None
            return
        if not isinstance(values, torch.Tensor):
            raise ValueError("values must be a torch tensor (currents.CurrentGrid gives the NumPy values)")
        if (values.dtype != torch.float64 or values.device != self.device or values.ndim not in (4, 5)
                or values.shape[-1] != 3 or not values.is_contiguous()):
            raise ValueError(f"values must be a contiguous (nt,nz,ny,nx,3) or (nz,ny,nx,3) torch.float64 tensor on "
                             f"{self.device}, got {tuple(values.shape)} {values.dtype} on {values.device}")
        if values.numel() == 0:
            raise ValueError("values must not be empty")
        if len(origin) != 3 or len(spacing) != 3:
            raise ValueError("origin and spacing must have 3 values")
        dims = (ctypes.c_int64 * 4)(*([1] * (5 - values.ndim) + list(values.shape[:-1])))
        geom = (ctypes.c_double * 8)(*[float(x) for x in (*origin, *spacing)], float(t0), float(frame_dt))
        L.check(self._lib.h2o_set_current_grid(self._h, ctypes.c_void_p(values.data_ptr()), dims, geom))
        self._grid = values  # keep the borrowed memory alive

    @property
    def current_grid(self) -> Optional[torch.Tensor]:
        """The borrowed current-grid tensor, or ``None``."""
        return getattr(self, "_grid", None)

    def set_env_conditions(self, cond: Optional[torch.Tensor], bodies_per_env: int = 0):
        """Per-env water conditions: ``cond`` is a contiguous (E,8) float64 tensor on the engine's device
        (``waves.env_conditions`` builds one), rows ``cx, cy, cz, dz, s, tau, x0, y0`` for envs of
        ``bodies_per_env`` contiguous bodies (E = n_bodies / bodies_per_env).  The env's current adds to the global
        one, its level to ``surface_z``; its sea is the wave field scaled by ``s`` at ``p - origin`` and
        ``clock + tau`` (include/h2o.h).  The tensor is borrowed, not copied: in-place edits reach the next step and
        the next replay of a captured rollout.  ``None`` removes the conditions.  Steps then run on the per-body
        kernel; ``rollout_persistent`` follows them; ``components`` ignores them."""
        if cond is None:
            L.check(self._lib.h2o_set_env_conditions(self._h, 0, None))
            self._cond = None
            return
        bpe = int(bodies_per_env)
        if not isinstance(cond, torch.Tensor):
            raise ValueError("cond must be a torch tensor (waves.env_conditions gives the NumPy rows)")
        if bpe < 1:
            raise ValueError(f"bodies_per_env must be >= 1, got {bodies_per_env}")
        if self.n_bodies % bpe:  # the library reports BAD_SHAPE
            L.check(self._lib.h2o_set_env_conditions(self._h, bpe, ctypes.c_void_p(cond.data_ptr())))
        n_envs = self.n_bodies // bpe
        if (cond.dtype != torch.float64 or cond.device != self.device or tuple(cond.shape) != (n_envs, W.COND_COLS)
                or not cond.is_contiguous()):
            raise ValueError(f"cond must be a contiguous ({n_envs},{W.COND_COLS}) torch.float64 tensor on {self.device}, "
                             f"got {tuple(cond.shape)} {cond.dtype} on {cond.device}")
        L.check(self._lib.h2o_set_env_conditions(self._h, bpe, ctypes.c_void_p(cond.data_ptr())))
        self._cond = cond  # keep the borrowed memory alive

    @property
    def env_conditions(self) -> Optional[torch.Tensor]:
        """The borrowed (E,8) conditions tensor, or ``None``."""
        return getattr(self, "_cond", None)

    def reset_envs(self, envs, restart_waves: bool = False):
        """Forget the previous-step velocities of the bodies of some envs (the per-env ``_reset``,
        hydrodynamics_behavior.py:240-245): ``envs`` is a bool mask (E,) or env ids.  With ``restart_waves`` those
        envs' ``tau`` becomes ``-clock``, so that their next step sees their sea at env time 0.  Stream-ordered, no
        host synchronisation (except to range-check env ids held on the device); a captured rollout is kept."""
        cond = self.env_conditions
        if cond is None:  # the library reports NOT_CONFIGURED
            L.check(self._lib.h2o_reset_envs(self._h, None, int(bool(restart_waves)), _stream_ptr(self.device)))
        n_envs = cond.shape[0]
        envs = torch.as_tensor(envs)
        if envs.dtype == torch.bool:
            if tuple(envs.shape) != (n_envs,):
                raise ValueError(f"a mask must be ({n_envs},), got {tuple(envs.shape)}")
            mask = envs.to(device=self.device, dtype=torch.uint8).contiguous()
        elif not envs.dtype.is_floating_point:
            ids = envs.reshape(-1).long()
            if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= n_envs):
                raise ValueError(f"env ids must be in [0, {n_envs})")
            mask = torch.zeros(n_envs, dtype=torch.uint8, device=self.device)
            mask[ids.to(self.device)] = 1
        else:
            raise ValueError("envs must be a bool mask or integer env ids")
        L.check(self._lib.h2o_reset_envs(self._h, ctypes.c_void_p(mask.data_ptr()), int(bool(restart_waves)),
                                         _stream_ptr(self.device)))

    def set_added_mass_dense(self, matrices=None, slot_type=None):
        """Dense 6x6 body-frame added-mass matrices (the argument ``calculate_added_mass`` takes,
        numba_hydrodynamics.py:220) instead of the wrapper's diagonal: ``matrices`` is (6,6) or
        (n_types,6,6), body ``i`` uses ``matrices[slot_type[i % len(slot_type)]]``.  ``None`` restores
        the diagonal.  Steps then run on the per-body kernel."""
        if matrices is None:
            L.check(self._lib.h2o_set_added_mass_dense(self._h, 0, None, 0, None))
            return
        m = np.ascontiguousarray(np.asarray(matrices, dtype=np.float64))
        if m.ndim == 2:
            m = m[None]
        if m.ndim != 3 or m.shape[1:] != (6, 6):
            raise ValueError("matrices must be (6,6) or (n_types,6,6)")
        mp = m.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        if slot_type is None:
            if m.shape[0] != 1:
                raise ValueError("slot_type is required with more than one matrix")
            L.check(self._lib.h2o_set_added_mass_dense(self._h, 1, mp, 1, None))
            return
        st = np.ascontiguousarray(np.asarray(slot_type, dtype=np.int32))
        L.check(self._lib.h2o_set_added_mass_dense(self._h, int(m.shape[0]), mp, int(st.size),
                                                   st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))

    def set_params_uniform(self, ctor12: Sequence[float], mass: float):
        """Same twelve scalars, same order, as the reference wrapper ctor
        (numba_hydrodynamics_wrapper.py:9-10) + the body mass used by the clamp."""
        if isinstance(ctor12, P.HydroParams):
            ctor12 = ctor12.ctor_row()
        arr = (ctypes.c_double * 12)(*[float(x) for x in ctor12])
        L.check(self._lib.h2o_set_params_uniform(self._h, arr, float(mass)))
        self.water_density, self.gravity = float(ctor12[7]), float(ctor12[8])

    def set_part_table(self, table, slot_type):
        """Part-type table (n_types,11) in ``params.COEFF_FIELDS`` order + slot->type map."""
        table = np.ascontiguousarray(np.asarray(table, dtype=np.float64))
        slot_type = np.ascontiguousarray(np.asarray(slot_type, dtype=np.int32))
        if table.ndim != 2 or table.shape[1] != L.N_COEFF:
            raise ValueError(f"table must be (n_types,{L.N_COEFF})")
        L.check(self._lib.h2o_set_part_table(
            self._h, table.shape[0], table.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
            slot_type.shape[0], slot_type.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))

    def set_params_per_body(self, coeff):
        """Heterogeneous records (n_bodies,11): torch tensor (any device) or NumPy array."""
        if isinstance(coeff, torch.Tensor) and coeff.is_cuda:
            dl = _DL()
            L.check(self._lib.h2o_set_params_per_body_dl(self._h, dl(coeff.contiguous()), _stream_ptr(self.device)))
            return
        arr = coeff.detach().cpu().numpy() if isinstance(coeff, torch.Tensor) else np.asarray(coeff)
        if arr.dtype not in (np.float32, np.float64):
            arr = arr.astype(np.float64)
        arr = np.ascontiguousarray(arr)
        if arr.shape != (self.n_bodies, L.N_COEFF):
            raise ValueError(f"coeff must be ({self.n_bodies},{L.N_COEFF}), got {arr.shape}")
        L.check(self._lib.h2o_set_params_per_body(
            self._h, arr.ctypes.data_as(ctypes.c_void_p), L.H2O_F32 if arr.dtype == np.float32 else L.H2O_F64,
            _stream_ptr(self.device)))

    def set_params_soa(self, columns: Sequence[torch.Tensor]):
        """Per-body parameters as eleven (n,) CUDA tensors in ``params.COEFF_FIELDS`` order (float32 or
        float64, all the same dtype), e.g. one tensor per exposed USD attribute + the view's masses."""
        if len(columns) != L.N_COEFF:
            raise ValueError(f"expected {L.N_COEFF} columns ({', '.join(P.COEFF_FIELDS)})")
        dt = columns[0].dtype
        if dt not in _TORCH_DTYPES:
            raise ValueError("columns must be float32 or float64")
        cols = []
        for k, c in enumerate(columns):
            if c.dtype != dt or c.device != self.device or tuple(c.shape) != (self.n_bodies,) or not c.is_contiguous():
                raise ValueError(f"column {k} ({P.COEFF_FIELDS[k]}): need a contiguous ({self.n_bodies},) {dt} tensor "
                                 f"on {self.device}")
            cols.append(c)
        arr = (ctypes.c_void_p * L.N_COEFF)(*[c.data_ptr() for c in cols])
        L.check(self._lib.h2o_set_params_soa(self._h, arr, _TORCH_DTYPES[dt], _stream_ptr(self.device)))

    def set_globals(self, water_density: float, gravity: float):
        """waterDensity / gravity (hydrodynamics_behavior.py:30-31)."""
        L.check(self._lib.h2o_set_globals(self._h, float(water_density), float(gravity)))
        self.water_density, self.gravity = float(water_density), float(gravity)

    def set_workload_params(self, wl):
        """Configure from a ``workloads.Workload`` (globals, coefficients, articulation)."""
        self.set_globals(wl.rho, wl.g)
        if wl.coeff is not None:
            self.set_params_per_body(wl.coeff)
        else:
            self.set_part_table(wl.table, wl.slot_type)
        self.set_articulation(wl.bodies_per_robot)

    def set_articulation(self, bodies_per_robot: int):
        L.check(self._lib.h2o_set_articulation(self._h, int(bodies_per_robot)))
        self.bodies_per_robot = int(bodies_per_robot)
        self._n_robots_var = 0

    def set_articulation_offsets(self, offsets):
        """Robots of unequal size: robot ``r`` owns bodies ``[offsets[r], offsets[r+1])`` (``offsets[0] == 0``,
        ``offsets[-1] == n_bodies``); the robot wrench output is then ``(len(offsets) - 1, 6)``."""
        off = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64))
        if off.ndim != 1 or off.size < 2:
            raise ValueError("offsets must be a 1-d array of n_robots + 1 entries")
        L.check(self._lib.h2o_set_articulation_offsets(self._h, int(off.size - 1),
                                                       off.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
        self.bodies_per_robot = 0
        self._n_robots_var = int(off.size - 1)

    @property
    def n_robots(self) -> int:
        """Rows of the per-robot wrench output (0 without an articulation)."""
        if getattr(self, "_n_robots_var", 0) > 0:
            return self._n_robots_var
        return self.n_bodies // self.bodies_per_robot if self.bodies_per_robot > 0 else 0

    def set_kernel(self, choice: str = "auto"):
        code = {"auto": L.H2O_KERNEL_AUTO, "tile": L.H2O_KERNEL_TILE, "direct": L.H2O_KERNEL_DIRECT}[choice]
        L.check(self._lib.h2o_set_kernel(self._h, code))

    def set_warp_compat(self, enable: bool = True):
        """``components`` and the fused step follow the reference's Warp twin (SURVEY.md App. C) instead of the
        Numba path; the step then runs on the per-body kernel in float64 (compatibility mode)."""
        L.check(self._lib.h2o_set_warp_compat(self._h, int(bool(enable))))

    def set_strict(self, enable: bool = True):
        """fp32 mode: ``True`` (default) guarantees the parity bound for every body (bodies whose force / torque
        groups cancel are re-evaluated in float64); ``False`` keeps the plain fp32 result for them."""
        L.check(self._lib.h2o_set_strict(self._h, int(bool(enable))))

    def set_tile_config(self, cfg: int = 0):
        """Tuning knob: tile-kernel variant (0 = default)."""
        L.check(self._lib.h2o_set_tile_config(self._h, int(cfg)))

    @property
    def ctas_per_sm(self) -> int:
        return int(self._lib.h2o_last_ctas_per_sm(self._h))

    def enable_stats(self, enable: bool = True):
        L.check(self._lib.h2o_enable_stats(self._h, int(bool(enable))))

    # ------------------------------------------------------------------ carried state
    def reset(self):
        """Forget the previous-step velocities (``_reset``, hydrodynamics_behavior.py:240-245)."""
        L.check(self._lib.h2o_reset(self._h, _stream_ptr(self.device)))

    def set_prev(self, prev_lin: torch.Tensor, prev_ang: torch.Tensor):
        dl = _DL()
        L.check(self._lib.h2o_set_prev_dl(self._h, dl(self._as_dev(prev_lin)), dl(self._as_dev(prev_ang)),
                                          _stream_ptr(self.device)))

    def prev_velocities(self) -> torch.Tensor:
        """Zero-copy (n,6) view of the engine-owned previous [v, omega] buffer (DLPack export)."""
        out = ctypes.c_void_p()
        L.check(self._lib.h2o_export_prev_dl(self._h, ctypes.byref(out)))
        t = _dlpack.from_dlpack(L.capsule_from_managed(out.value))
        t._h2o_owner = self  # the memory lives as long as the handle
        return t

    # ------------------------------------------------------------------ helpers
    def _as_dev(self, x) -> torch.Tensor:
        if not isinstance(x, torch.Tensor):
            x = torch.as_tensor(np.asarray(x))
        return x.to(device=self.device, dtype=self.dtype).contiguous()

    def _empty(self, *shape) -> torch.Tensor:
        return torch.empty(*shape, dtype=self.dtype, device=self.device)

    def _outputs(self, out_force, out_torque, out_robot_wrench, want_wrench):
        if out_force is None:
            out_force = self._empty(self.n_bodies, 3)
        if out_torque is None:
            out_torque = self._empty(self.n_bodies, 3)
        if want_wrench and out_robot_wrench is None:
            if self.n_robots <= 0:
                raise ValueError("robot wrench requested but set_articulation() was not called")
            out_robot_wrench = self._empty(self.n_robots, 6)
        return out_force, out_torque, out_robot_wrench

    # ------------------------------------------------------------------ fused step
    def step(self, position, orientation_quat, linear_vel, angular_vel, dt: float, out_force=None,
             out_torque=None, out_robot_wrench=None, robot_wrench: bool = False):
        """One physics step for every body (hydrodynamics_behavior.py:194-238, batched).

        Tensors are (N,3)/(N,4) CUDA tensors of the engine dtype; the engine keeps the
        previous-step velocities itself.  Returns ``(force, torque)`` or
        ``(force, torque, robot_wrench)``.
        """
        F, T, W = self._outputs(out_force, out_torque, out_robot_wrench, robot_wrench)
        dl = _DL()
        L.check(self._lib.h2o_step_dl(self._h, dl(position), dl(orientation_quat), dl(linear_vel),
                                      dl(angular_vel), float(dt), dl(F), dl(T), dl(W),
                                      _stream_ptr(self.device)))
        return (F, T) if W is None else (F, T, W)

    def step_physx(self, transforms, velocities, dt: float, out_force=None, out_torque=None,
                   out_robot_wrench=None, robot_wrench: bool = False):
        """Same, PhysX tensor-API layout: transforms (N,7) = [p, q], velocities (N,6) = [v, w]."""
        F, T, W = self._outputs(out_force, out_torque, out_robot_wrench, robot_wrench)
        dl = _DL()
        L.check(self._lib.h2o_step_physx_dl(self._h, dl(transforms), dl(velocities), float(dt), dl(F), dl(T),
                                            dl(W), _stream_ptr(self.device)))
        return (F, T) if W is None else (F, T, W)

    def step_view(self, position, orientation_quat, velocities, dt: float, out_force=None, out_torque=None,
                  out_robot_wrench=None, robot_wrench: bool = False):
        """Same, RigidPrimView layout: ``get_world_poses()`` -> (N,3), (N,4) and ``get_velocities()`` ->
        (N,6) = [v, w] (hydrodynamics_behavior.py:178-189), consumed as they are (no slicing copies)."""
        F, T, W = self._outputs(out_force, out_torque, out_robot_wrench, robot_wrench)
        dl = _DL()
        L.check(self._lib.h2o_step_view_dl(self._h, dl(position), dl(orientation_quat), dl(velocities), float(dt),
                                           dl(F), dl(T), dl(W), _stream_ptr(self.device)))
        return (F, T) if W is None else (F, T, W)

    def bind(self, position=None, orientation_quat=None, linear_vel=None, angular_vel=None, *,
             transforms=None, velocities=None, out_force=None, out_torque=None, out_robot_wrench=None,
             robot_wrench: bool = False):
        """Validate and remember the tensors once; ``step_bound`` is then a single cheap call."""
        F, T, W = self._outputs(out_force, out_torque, out_robot_wrench, robot_wrench)
        dl = _DL()
        if transforms is not None:
            L.check(self._lib.h2o_bind_dl(self._h, L.LAYOUT_PHYSX, dl(transforms), None, dl(velocities), None,
                                          dl(F), dl(T), dl(W)))
            self._bound = (transforms, velocities, F, T, W)
        elif velocities is not None:
            L.check(self._lib.h2o_bind_dl(self._h, L.LAYOUT_VIEW, dl(position), dl(orientation_quat), dl(velocities),
                                          None, dl(F), dl(T), dl(W)))
            self._bound = (position, orientation_quat, velocities, F, T, W)
        else:
            L.check(self._lib.h2o_bind_dl(self._h, L.LAYOUT_SPLIT, dl(position), dl(orientation_quat),
                                          dl(linear_vel), dl(angular_vel), dl(F), dl(T), dl(W)))
            self._bound = (position, orientation_quat, linear_vel, angular_vel, F, T, W)
        return (F, T) if W is None else (F, T, W)

    def step_bound(self, dt: float):
        L.check(self._lib.h2o_step_bound(self._h, float(dt), _stream_ptr(self.device)))

    def set_rollout_mode(self, free_bodies: bool = False, gravity: float = 9.81):
        """Rollouts over the bound tensors: static state (force-only) or free bodies integrated in place."""
        L.check(self._lib.h2o_set_rollout_mode(self._h, int(bool(free_bodies)), float(gravity)))

    def integrate_free_bodies(self, position, orientation_quat, linear_vel, angular_vel, force, torque,
                              dt: float, gravity: float = 9.81):
        """Harness stepper (semi-implicit Euler, box inertia); updates the four state tensors in place."""
        for t in (position, orientation_quat, linear_vel, angular_vel, force, torque):
            if not (t.is_cuda and t.dtype == self.dtype and t.is_contiguous()):
                raise ValueError("integrate_free_bodies takes contiguous CUDA tensors of the engine dtype")
        L.check(self._lib.h2o_integrate_free_bodies(
            self._h, position.data_ptr(), orientation_quat.data_ptr(), linear_vel.data_ptr(), angular_vel.data_ptr(),
            force.data_ptr(), torque.data_ptr(), float(dt), float(gravity), _stream_ptr(self.device)))

    def capture_rollout(self, n_steps: int, dt: float):
        """Capture ``n_steps`` back-to-back steps over the bound tensors into one CUDA graph.  Nothing is
        launched while capturing (state and carried velocities stay as they are); any later ``set_*`` /
        ``enable_stats`` / ``bind`` call drops the graph and ``launch_rollout`` raises until re-captured."""
        L.check(self._lib.h2o_capture_rollout(self._h, int(n_steps), float(dt), _stream_ptr(self.device)))

    def launch_rollout(self):
        L.check(self._lib.h2o_launch_rollout(self._h, _stream_ptr(self.device)))

    def rollout_persistent(self, n_steps: int, dt: float, gravity: float = 9.81, trace_every: int = 0):
        """``n_steps`` x (fused force step -> free-body stepper) over the bound split-layout tensors in ONE
        kernel launch (state in registers across the steps).  Returns the trace tensor
        ``(n_steps // trace_every, n_bodies, 9)`` = [p, v, w] rows when ``trace_every > 0``, else ``None``; a
        ``trace_every`` above ``n_steps`` would write no row and raises ``ValueError``.  The rollout follows the
        Numba semantics and writes no robot wrench: with ``set_warp_compat(True)`` or a bound robot-wrench output
        it raises (use ``capture_rollout`` in free-body mode there)."""
        trace = None
        if trace_every > n_steps:
            raise ValueError(f"trace_every ({trace_every}) > n_steps ({n_steps}) would write no trace row")
        if trace_every > 0:
            trace = self._empty(n_steps // trace_every, self.n_bodies, 9)
        L.check(self._lib.h2o_rollout_persistent(self._h, int(n_steps), float(dt), float(gravity), int(trace_every),
                                                 ctypes.c_void_p(trace.data_ptr()) if trace is not None else None,
                                                 _stream_ptr(self.device)))
        return trace

    # ------------------------------------------------------------------ components
    def components(self, position, orientation_quat, linear_vel, angular_vel, linear_accel, angular_accel,
                   return_flags: bool = False):
        """Batched ``calculate_hydrodynamic_forces`` (numba_hydrodynamics.py:314 order):
        (buoyancy_force, drag_force, lift_force, drag_torque, added_mass_force,
        added_mass_torque, center_of_buoyancy, center_of_pressure, sub_ratio)."""
        outs = [self._empty(self.n_bodies, 3) for _ in range(8)]
        ratio = self._empty(self.n_bodies)
        flags = torch.empty(self.n_bodies, dtype=torch.int32, device=self.device) if return_flags else None
        dl = _DL()
        arr = (ctypes.c_void_p * 8)(*[dl(o) for o in outs])
        L.check(self._lib.h2o_components_dl(self._h, dl(position), dl(orientation_quat), dl(linear_vel),
                                            dl(angular_vel), dl(linear_accel), dl(angular_accel), arr, dl(ratio),
                                            dl(flags), _stream_ptr(self.device)))
        res = tuple(outs) + (ratio,)
        return res + (flags,) if return_flags else res

    # ------------------------------------------------------------------ host arrays
    def _host_in(self, x, cols):
        npdt = _NP_DTYPES[_TORCH_DTYPES[self.dtype]]
        if isinstance(x, torch.Tensor):
            if x.is_cuda or x.dtype != self.dtype or not x.is_contiguous():
                raise ValueError("step_host takes contiguous CPU tensors of the engine dtype")
            assert tuple(x.shape) == (self.n_bodies, cols)
            return x, x.data_ptr()
        a = np.ascontiguousarray(x, dtype=npdt)
        assert a.shape == (self.n_bodies, cols), (a.shape, cols)
        return a, a.ctypes.data

    def _host_out(self, x, rows, cols):
        npdt = _NP_DTYPES[_TORCH_DTYPES[self.dtype]]
        if x is None:
            x = np.empty((rows, cols), dtype=npdt)
        if isinstance(x, torch.Tensor):
            return x, x.data_ptr()
        assert x.dtype == npdt and x.flags.c_contiguous and x.shape == (rows, cols)
        return x, x.ctypes.data

    def step_host(self, position, orientation_quat, linear_vel, angular_vel, dt: float, out_force=None,
                  out_torque=None, out_robot_wrench=None, robot_wrench: bool = False):
        """NumPy / CPU-tensor in, same out.  Pinned (page-locked) buffers take the zero-copy path: the fused
        kernel reads and writes them over PCIe directly (TMA bulk copies), no staging; pageable buffers go
        through a chunked H2D -> kernel -> D2H pipeline.  ``last_host_path`` tells which."""
        keep = [self._host_in(position, 3), self._host_in(orientation_quat, 4), self._host_in(linear_vel, 3),
                self._host_in(angular_vel, 3)]
        F, pf = self._host_out(out_force, self.n_bodies, 3)
        T, pt = self._host_out(out_torque, self.n_bodies, 3)
        W, pw = (None, None)
        if robot_wrench or out_robot_wrench is not None:
            W, pw = self._host_out(out_robot_wrench, self.n_bodies // self.bodies_per_robot, 6)
        L.check(self._lib.h2o_step_host(self._h, keep[0][1], keep[1][1], keep[2][1], keep[3][1], float(dt),
                                        pf, pt, pw))
        return (F, T) if W is None else (F, T, W)

    def step_host_physx(self, transforms, velocities, dt: float, out_force=None, out_torque=None,
                        out_robot_wrench=None, robot_wrench: bool = False):
        """Same with the PhysX layout on the host: transforms (N,7) = [p, q], velocities (N,6) = [v, w]."""
        keep = [self._host_in(transforms, 7), self._host_in(velocities, 6)]
        F, pf = self._host_out(out_force, self.n_bodies, 3)
        T, pt = self._host_out(out_torque, self.n_bodies, 3)
        W, pw = (None, None)
        if robot_wrench or out_robot_wrench is not None:
            W, pw = self._host_out(out_robot_wrench, self.n_bodies // self.bodies_per_robot, 6)
        L.check(self._lib.h2o_step_host_physx(self._h, keep[0][1], keep[1][1], float(dt), pf, pt, pw))
        return (F, T) if W is None else (F, T, W)

    @property
    def last_host_path(self) -> str:
        return {1: "zero-copy", 2: "staged"}.get(int(self._lib.h2o_last_host_path(self._h)), "none")

    # ------------------------------------------------------------------ introspection
    def stats(self, reset: bool = False) -> dict:
        out = (ctypes.c_double * L.N_STATS)()
        L.check(self._lib.h2o_read_stats(self._h, out, int(reset), _stream_ptr(self.device)))
        return dict(zip(L.STATS_FIELDS, list(out)))

    def stats_tensor(self) -> torch.Tensor:
        """Device-resident (8,) float64 statistics vector (for an NCCL all-reduce)."""
        ptr = ctypes.c_void_p()
        L.check(self._lib.h2o_stats_device_ptr(self._h, ctypes.byref(ptr)))
        return _tensor_from_ptr(ptr.value, (L.N_STATS,), torch.float64, self.device, self)

    @property
    def launch_count(self) -> int:
        return int(self._lib.h2o_launch_count(self._h))

    @property
    def last_kernel(self) -> str:
        return {L.H2O_KERNEL_TILE: "tile", L.H2O_KERNEL_DIRECT: "direct"}.get(
            int(self._lib.h2o_last_kernel(self._h)), "none")


class _CudaArrayView:
    """Minimal ``__cuda_array_interface__`` carrier for an engine-owned device buffer."""

    def __init__(self, ptr, shape, typestr, owner):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}
        self._owner = owner


def _tensor_from_ptr(ptr, shape, dtype, device, owner) -> torch.Tensor:
    typestr = {torch.float32: "<f4", torch.float64: "<f8", torch.int32: "<i4"}[dtype]
    t = torch.as_tensor(_CudaArrayView(ptr, shape, typestr, owner), device=device)
    t._h2o_owner = owner
    return t
