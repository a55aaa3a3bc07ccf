"""Batched twin of the reference's ``HydrodynamicsBehavior`` (SURVEY.md 8(f1)).

The reference attaches one ``HydrodynamicsBehavior`` to each scripted prim (20 in the main
scene), each with its own 1-body ``RigidPrimView``, wrapper, graph and ~35 micro-launches
per physics step (hydrodynamics_behavior.py:143-238).  This class keeps that script's
life cycle and parameter surface --

    on_init   exposed variables with the reference defaults (:28-46), then the JSON overlay
              by prim name (:72-112)
    on_play   ``_setup``: read the parameters back, build the force engine, cache masses (:143-174)
    physics   ``_on_physics_step(dt)``: skip if dt <= 1e-6 or the view is invalid (:138-141),
              read poses / velocities, compute, ``apply_forces_and_torques_at_pos`` (:176-234)
    on_stop   ``_reset`` (:240-245)

-- but for ALL scripted prims through ONE view and ONE fused kernel launch.  It is written
against the three ``RigidPrimView`` methods the reference uses (``get_world_poses``,
``get_velocities``, ``apply_forces_and_torques_at_pos`` + ``get_masses`` / ``is_valid``), so it
runs unchanged inside Isaac Sim and, in tests, against a stand-in view.

Deliberate deviation: the reference script evaluates forces through its Warp wrapper
(hydrodynamics_behavior.py:19, :155), whose kernel rotates the accelerations FORWARD into the
"body" frame (warp_hydrodynamics.py:216-217) where the Numba path uses R^T
(numba_hydrodynamics.py:229-230), so its linear added-mass force is -m R^2 a instead of -m a.
BASELINE.json's north star pins this engine to the NUMBA semantics, which the fused fast path
implements; for rotated bodies with a non-zero added-mass coefficient (Body: 0.2 / 0.1) the forces
therefore differ from the Warp production path by that term (SURVEY.md Appendix C1).
``warp_compat=True`` switches the whole step (and ``HydroEngine.components``) to the Warp twin's
semantics -- scored against the reference's own Warp kernel source, tests/golden/reference_warp_golden.npz --
at the price of the per-body float64 kernel instead of the TMA tile kernel.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import params as P
from .engine import HydroEngine
from .waves import WaveField


class BatchedHydrodynamicsBehavior:
    BEHAVIOR_NS = "hydrodynamicsBehavior"                      # hydrodynamics_behavior.py:26
    VARIABLES_TO_EXPOSE = [                                      # names/defaults of :28-46
        {"attr_name": k, "default_value": v} for k, v in P.EXPOSED_VARIABLES
    ]

    def __init__(self, prim_names: Sequence[str], view, device: str = "cuda:0",
                 config_path: Optional[str] = None, dtype: torch.dtype = torch.float32,
                 bodies_per_robot: int = 0, robot_offsets: Optional[Sequence[int]] = None,
                 warp_compat: bool = False, waves: Optional[WaveField] = None, wave_slope: bool = False,
                 fluid_inertia: bool = False):
        self.prim_names = list(prim_names)
        self._view = view
        self._device = device
        self._dtype = dtype
        self._config_path = config_path
        self._bodies_per_robot = int(bodies_per_robot)
        self._warp_compat = bool(warp_compat)
        self._waves = waves  # built-in wave field, installed by _setup with its clock at 0
        self._wave_slope = bool(wave_slope)  # test the prims against the wave surface's tangent plane (needs waves)
        self._fluid_inertia = bool(fluid_inertia)  # Froude-Krylov + added mass on the fluid-relative acceleration
        # robots of unequal size, e.g. [0, 19, 20] for one SILVER2 + the Obsea buoy (the main scene)
        self._robot_offsets = None if robot_offsets is None else [int(o) for o in robot_offsets]
        self._engine: Optional[HydroEngine] = None
        self._F = self._T = None
        self.robot_wrench = None
        self.part_of: List[Optional[str]] = []
        self.on_init()

    # ------------------------------------------------------------------ life cycle
    def on_init(self):
        """Defaults -> JSON ``globals`` -> first matching ``parts`` entry, per prim (:48-112)."""
        try:
            config = P.load_config(self._config_path)
        except (OSError, ValueError):  # "[Hydro] Config missing" / "JSON Error": keep the defaults
            config = {}
        self.exposed: Dict[str, P.HydroParams] = {}
        self.part_of = []
        for name in self.prim_names:
            p, part = P.params_for_prim(name, config)
            self.exposed[name] = p.as_float32()  # USD stores the exposed variables as fp32 Floats
            self.part_of.append(part)
        self._config = config

    def set_exposed_variable(self, prim_name: str, attr_name: str, value: float) -> bool:
        """Edit one exposed variable before play (the property-window path of the reference)."""
        return self.exposed[prim_name].set(attr_name, np.float32(value))

    def on_play(self):
        self._setup()

    def on_stop(self):
        self._reset()

    def on_destroy(self):
        self._reset()

    # ------------------------------------------------------------------ _setup (:143-174)
    def _setup(self):
        n = len(self.prim_names)
        masses = self._view.get_masses(clone=False)
        masses = masses.detach().cpu().numpy() if isinstance(masses, torch.Tensor) else np.asarray(masses)
        first = self.exposed[self.prim_names[0]]
        rows = []
        for i, name in enumerate(self.prim_names):
            p = self.exposed[name]
            if (p.waterDensity, p.gravity) != (first.waterDensity, first.gravity):
                raise ValueError("waterDensity / gravity must be the same for every prim of one engine")
            rows.append(p.coeff_record(float(masses[i])))
        # Isaac core hands quaternions as wxyz; the reference permutes them at :194
        self._engine = HydroEngine(n, dtype=self._dtype, device=self._device,
                                   water_density=first.waterDensity, gravity=first.gravity, quat_order="wxyz")
        self._engine.set_params_per_body(np.asarray(rows, dtype=np.float64))
        if self._warp_compat:
            self._engine.set_warp_compat(True)
        if self._waves is not None:
            self._engine.set_wave_field(self._waves)
            self._engine.set_wave_time(0.0)
            if self._wave_slope:
                self._engine.set_wave_slope(True)
            if self._fluid_inertia:
                self._engine.set_fluid_inertia(True)
        if self._robot_offsets is not None:
            self._engine.set_articulation_offsets(self._robot_offsets)
        else:
            self._engine.set_articulation(self._bodies_per_robot)
        dev = self._engine.device
        self._F = torch.empty(n, 3, dtype=self._dtype, device=dev)
        self._T = torch.empty(n, 3, dtype=self._dtype, device=dev)
        self.robot_wrench = (torch.empty(self._engine.n_robots, 6, dtype=self._dtype, device=dev)
                             if self._engine.n_robots > 0 else None)

    # ------------------------------------------------------------------ physics step (:138-238)
    def _on_physics_step(self, delta_time: float):
        if delta_time <= 1e-6 or self._engine is None or self._view is None or not self._view.is_valid():
            return
        self._apply_behavior(delta_time)

    def _apply_behavior(self, delta_time: float):
        try:
            positions, orientations = self._view.get_world_poses(clone=False)
            full_velocities = self._view.get_velocities(clone=False)
            if full_velocities is None or full_velocities.shape[0] == 0:
                return
            dev, dt_ = self._engine.device, self._dtype
            positions = positions.to(device=dev, dtype=dt_).contiguous()
            orientations = orientations.to(device=dev, dtype=dt_).contiguous()
            full_velocities = full_velocities.to(device=dev, dtype=dt_).contiguous()
        except (UnboundLocalError, IndexError, RuntimeError, AttributeError):
            return  # the reference silently skips the step (:191-192)
        # the (N,6) velocity tensor is consumed as it is: no [:, 0:3] / [:, 3:6] slicing copies (:188-189)
        self._engine.step_view(positions, orientations, full_velocities, delta_time,
                               out_force=self._F, out_torque=self._T, out_robot_wrench=self.robot_wrench)
        self._view.apply_forces_and_torques_at_pos(forces=self._F, torques=self._T, positions=positions,
                                                   is_global=True)

    def _reset(self):
        if self._engine is not None:
            self._engine.close()
        self._engine = None
        self._F = self._T = self.robot_wrench = None
