"""Generate tests/golden/reference_numba_golden.npz (the c3 group: ..._c3.npz) from the UNMODIFIED reference.

Run in the build container only (needs /root/reference + numba):

    python -m oracle.make_golden

For every case it calls the reference's own
``NumbaHydrodynamicsWrapper.calculate_hydrodynamic_forces``
(/root/reference/src/scripts/physics/numba_hydrodynamics_wrapper.py:34) once per
body -- exactly how the reference is used -- and stores inputs + the nine
outputs.  Bodies for which the reference raises ``TypeError`` (wet and at rest,
SURVEY.md A.8) are stored with ``raised=True`` and zero outputs.

Case groups (all float64 arrays; the fp32-representable groups are exact up-casts):
  c3      2048 heterogeneous boxes, fp32-representable inputs (C3 distribution)
  c3f64   1024 heterogeneous boxes drawn directly in float64
  c2      64 hexapod envs (1216 bodies), fp32-representable, part-table parameters
  near    512 boxes within 1 m of the origin (strict fp64 torque set)
  edge    hand-written edge cases: dry, fully wet, identity quaternion with faces
          exactly on the waterline, at-rest (defect), slow (<0.2 m/s), flow along
          body z (lift axis degenerate), non-normalised quaternion, tiny box
"""
from __future__ import annotations

import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import ref_numba  # noqa: E402
from oracle.hydro_oracle import COMPONENT_NAMES  # noqa: E402
from silver2_isaacsim_b200 import params as P  # noqa: E402
from silver2_isaacsim_b200 import workloads as W  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                   "reference_numba_golden.npz")

README_CTOR = [1, 1, 1, 1.2, 0.8, 300, 150, 1025, 9.81, 0.05, 0.02, 1.0]


def _accel(wl):
    a = (wl.lin_vel.astype(np.float64) - wl.prev_lin.astype(np.float64)) / wl.dt
    al = (wl.ang_vel.astype(np.float64) - wl.prev_ang.astype(np.float64)) / wl.dt
    return a, al


def _from_workload(wl):
    a, al = _accel(wl)
    return dict(ctor=wl.ctor_rows(), mass=wl.masses(), pos=wl.pos.astype(np.float64),
                quat=wl.quat_xyzw.astype(np.float64), v=wl.lin_vel.astype(np.float64),
                w=wl.ang_vel.astype(np.float64), a=a, al=al)


def edge_cases():
    rows = []

    def add(ctor, mass, p, q, v, w, a=(0, 0, 0), al=(0, 0, 0)):
        rows.append((ctor, mass, p, q, v, w, a, al))

    I = (0, 0, 0, 1)
    body = [0.26, 0.26, 0.30, 1.2, 0.8, 300, 150, 1025, 9.81, 0.2, 0.1, 0.5]
    tibia = [0.06, 0.09, 0.06, 1.0, 0.1, 20, 2, 1025, 9.81, 0, 0, 0.1]
    # SURVEY.md Appendix B GV1..GV5
    add(README_CTOR, 512.5, (0, 0, -0.2), I, (0.1, 0, -0.3), (0.01, 0.02, 0.03))
    add(body, 18, (2, 10.7, -18.4),
        (0.10259783520851541, -0.20519567041703082, 0.3077935056255462, 0.9233805168766387),
        (0.25, -0.1, 0.05), (0.3, -0.2, 0.1), (1.5, -0.5, 0.25), (-2, 1, 0.5))
    add(tibia, 0.8, (0.3, -0.4, 0.01),
        (0.502518907629606, 0.10050378152592121, -0.30151134457776363, 0.8040302522073697),
        (1, -2, 0.5), (3, 1, -2), (10, 0, -5), (0, 4, 0))
    add(README_CTOR, 512.5, (0, 0, 0.75), I, (0.1, 0, -0.3), (0.01, 0.02, 0.03), (1, 1, 1), (1, 1, 1))
    add(README_CTOR, 512.5, (0, 0, -0.2), I, (0, 0, 0), (0.01, 0.02, 0.03))          # GV5 defect
    # waterline exactly through the middle layer / top face / bottom face (strict < tests)
    add(README_CTOR, 512.5, (0, 0, 0.0), I, (0.3, 0.1, -0.2), (0.1, 0, 0), (1, 2, 3), (0.5, 0, 0))
    add(README_CTOR, 512.5, (0, 0, -0.5), I, (0.3, 0.1, 0.2), (0.1, 0, 0), (1, 2, 3), (0.5, 0, 0))
    add(README_CTOR, 512.5, (0, 0, 0.5), I, (0.3, 0.1, -0.2), (0.1, 0, 0), (1, 2, 3), (0.5, 0, 0))
    add(README_CTOR, 512.5, (0, 0, 0.5 - 1e-12), I, (0.3, 0.1, -0.2), (0.1, 0, 0))     # ratio ~1e-12 <= 1e-9
    add(README_CTOR, 512.5, (0, 0, 0.5 - 1e-8), I, (0.3, 0.1, -0.2), (0.1, 0, 0))      # ratio 1e-8 > 1e-9
    # slow regimes (damping scale), speed thresholds
    add(README_CTOR, 512.5, (1, 2, -3), I, (0.05, 0.01, -0.02), (0.05, 0.0, 0.01), (0.1, 0, 0), (0, 0.1, 0))
    add(README_CTOR, 512.5, (1, 2, -3), I, (5e-7, 0, 0), (0, 0, 0))                    # at rest -> defect
    add(README_CTOR, 512.5, (1, 2, -3), I, (2e-6, 0, 0), (5e-7, 0, 0))
    add(README_CTOR, 512.5, (1, 2, -3), I, (0.2, 0, 0), (0.2, 0, 0))
    # flow along +-body z: lift axis degenerate -> zeros (numba_hydrodynamics.py:210-211)
    add(README_CTOR, 512.5, (0, 0, -2), I, (0, 0, 1.5), (0, 0, 0.3))
    add(README_CTOR, 512.5, (0, 0, -2), I, (0, 0, -1.5), (0, 0, 0.3))
    # flow exactly in a face plane, rotated 90 deg about x
    s = np.sqrt(0.5)
    add(body, 18, (0, 0, -0.05), (s, 0, 0, s), (0.7, 0, 0), (0, 1, 0), (3, 0, 0), (0, 0, 2))
    # non-normalised quaternions (no normalisation in numba_hydrodynamics.py:14-49)
    add(body, 18, (0.2, 0.1, -0.02), (0.2, -0.4, 0.6, 1.1), (0.4, -0.3, 0.2), (1, 1, -1), (2, -2, 1), (1, 0, -3))
    add(tibia, 0.8, (0, 0, 0.0), (0.05, 0.02, 0.0, 0.9), (1, 1, 1), (0.1, 0.1, 0.1), (0, 0, 9), (3, 0, 0))
    # clamp active: tiny mass
    add(README_CTOR, 1.0, (0, 0, -2), I, (2, -1, 0.5), (1, 0, 0), (10, 0, 0), (0, 5, 0))
    # tiny box, total_height < 1e-6 branch
    tiny = [1e-7, 1e-7, 1e-7, 1.2, 0.8, 300, 150, 1025, 9.81, 0.05, 0.02, 1.0]
    add(tiny, 1e-3, (0, 0, 1e-9), I, (0.5, 0, 0), (0, 0, 0))
    add(tiny, 1e-3, (0, 0, -1e-9), I, (0.5, 0, 0), (0, 0, 0))
    arr = lambda k: np.asarray([r[k] for r in rows], dtype=np.float64)
    return dict(ctor=arr(0), mass=arr(1), pos=arr(2), quat=arr(3), v=arr(4), w=arr(5), a=arr(6),
                al=arr(7))


def main():
    groups = {
        "c3": _from_workload(W.heterogeneous_boxes(2048, seed=W.SEED_BASE + 103)),
        "c3f64": _from_workload(W.heterogeneous_boxes(1024, seed=W.SEED_BASE + 203, dtype=np.float64)),
        "c2": _from_workload(W.hexapod_envs(64, seed=W.SEED_BASE + 102)),
        "near": _from_workload(W.heterogeneous_boxes(512, seed=W.SEED_BASE + 303, dtype=np.float64,
                                                     xy_range=1.0)),
        "edge": edge_cases(),
    }
    blob = {}
    for g, d in groups.items():
        out, raised = ref_numba.components_via_wrapper(d["ctor"], d["pos"], d["quat"], d["v"],
                                                       d["w"], d["a"], d["al"])
        for k, v in d.items():
            blob[f"{g}/{k}"] = v
        for name in COMPONENT_NAMES:
            blob[f"{g}/{name}"] = out[name]
        blob[f"{g}/sub_ratio"] = out["sub_ratio"]
        blob[f"{g}/raised"] = raised
        print(f"{g}: n={len(raised)} raised={int(raised.sum())} wet={int((out['sub_ratio'] > 0).sum())} "
              f"partial={int(((out['sub_ratio'] > 0) & (out['sub_ratio'] < 1)).sum())}")
    import numba

    blob["meta/versions"] = np.array([f"numba {numba.__version__}", f"numpy {np.__version__}"])
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    # the c3 group goes to a file of its own: every file stays under 1 MB
    out_c3 = OUT.replace(".npz", "_c3.npz")
    np.savez_compressed(out_c3, **{k: v for k, v in blob.items() if k.startswith("c3/")})
    np.savez_compressed(OUT, **{k: v for k, v in blob.items() if not k.startswith("c3/")})
    for path in (OUT, out_c3):
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
