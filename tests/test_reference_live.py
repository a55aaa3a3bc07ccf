"""The outputs of the UNMODIFIED reference Numba code, stored in ``tests/golden`` by ``oracle/make_golden.py``,
as the checker of a whole behaviour step.  The golden ``c3`` group was computed on
``W.heterogeneous_boxes(2048, seed=W.SEED_BASE + 103)``: the workload is regenerated here, and the fixture
checks that its inputs (previous velocities and step included, through the stored accelerations) are the
stored ones bit for bit.  The reference's force and torque are its stored components through the behaviour
tail (``hydro_oracle.numpy_tail``, hydrodynamics_behavior.py:212-224).

  * CPU: the C restatement ``oracle/hydro_oracle.c`` stepped on that workload against them;
  * GPU (``-m gpu``): the CUDA path through the C ABI against them, both precisions.
"""
import numpy as np
import pytest

from silver2_isaacsim_b200 import workloads as W
from tests import scoring


@pytest.fixture(scope="module")
def ref_step(golden):
    """(workload, force, torque, components, raised) of one behaviour step of the reference."""
    from oracle.hydro_oracle import COMPONENT_NAMES, numpy_tail

    d = golden["c3"]
    wl = W.heterogeneous_boxes(len(d["pos"]), seed=W.SEED_BASE + 103)
    f8 = lambda a: a.astype(np.float64)
    inputs = {"ctor": wl.ctor_rows(), "mass": wl.masses(), "pos": f8(wl.pos), "quat": f8(wl.quat_xyzw),
              "v": f8(wl.lin_vel), "w": f8(wl.ang_vel), "a": (f8(wl.lin_vel) - f8(wl.prev_lin)) / wl.dt,
              "al": (f8(wl.ang_vel) - f8(wl.prev_ang)) / wl.dt}
    for k, x in inputs.items():
        assert np.array_equal(x, d[k]), f"the regenerated workload's {k} is not what the golden c3 group stores"
    comp = {name: d[name] for name in COMPONENT_NAMES + ("sub_ratio",)}
    F, T, _ = numpy_tail(comp, d["pos"], d["mass"])
    raised = d["raised"].copy()
    # a few wet bodies at rest: the reference raises there (SURVEY.md A.8; golden edge case GV5 records it)
    assert golden["edge"]["raised"][4] and not golden["edge"]["v"][4].any()
    wl.lin_vel[:3] = 0.0
    wl.pos[:3, 2] = -5.0
    raised[:3] = True
    return wl, F, T, comp, raised


def test_c_oracle_against_the_live_reference(oracle, ref_step):
    wl, F, T, comp, raised = ref_step
    ref = oracle.step(wl.ctor_rows(), wl.masses(), wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel, wl.prev_lin,
                      wl.prev_ang, wl.dt)
    assert raised[:3].all() and raised.sum() == 3                    # exactly the at-rest wet bodies raise ...
    assert ((ref.flags & 1) != 0).tolist() == raised.tolist()        # ... and the oracle flags exactly those
    ok = ~raised
    scale = scoring.force_scale(wl.coeff_per_body(), wl.rho, wl.g)
    # fastmath reassociation of the reference moves results by ~1e-13 relative (SURVEY.md 8(c))
    assert scoring.fp64_ok(F[ok], ref.force[ok], scale[ok], rel=1e-11).all()
    pn = np.abs(wl.pos).max(axis=1).astype(float) * np.abs(ref.force).max(axis=1)
    assert scoring.fp64_ok(T[ok], ref.torque[ok], scale[ok], extra=pn[ok], rel=1e-11).all()
    for name in ("buoyancy_force", "drag_force", "lift_force", "drag_torque", "added_mass_force", "added_mass_torque"):
        assert scoring.fp64_ok(comp[name][ok], ref.components[name][ok], scale[ok], rel=1e-11).all(), name
    assert np.abs(comp["sub_ratio"][ok] - ref.components["sub_ratio"][ok]).max() < 1e-12


# --------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "fp64"])
def test_cuda_path_against_the_live_reference(ref_step, mode):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from silver2_isaacsim_b200 import HydroEngine

    wl, F_ref, T_ref, comp, raised = ref_step
    dev = torch.device("cuda:0")
    dtype = torch.float32 if mode == "fp32" else torch.float64
    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    e.set_kernel("tile")
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dtype).contiguous()
    e.set_prev(t(wl.prev_lin), t(wl.prev_ang))
    F, T = e.step(t(wl.pos), t(wl.quat_xyzw), t(wl.lin_vel), t(wl.ang_vel), wl.dt)
    torch.cuda.synchronize()
    assert e.last_kernel == "tile"
    F, T = F.double().cpu().numpy(), T.double().cpu().numpy()
    ok = ~raised
    if mode == "fp32":
        scoring.assert_fp32(F[ok], F_ref[ok], "force vs the reference")
        scoring.assert_fp32(T[ok], T_ref[ok], "torque vs the reference")
    else:
        scale = scoring.force_scale(wl.coeff_per_body(), wl.rho, wl.g)
        # 1e-11: the reference's own fastmath noise floor sits at ~1e-13 .. 2e-12 on barely wet bodies
        assert scoring.fp64_ok(F[ok], F_ref[ok], scale[ok], rel=1e-11).all()
        pn = np.abs(wl.pos).max(axis=1).astype(float) * np.abs(F_ref).max(axis=1)
        assert scoring.fp64_ok(T[ok], T_ref[ok], scale[ok], extra=pn[ok], rel=1e-11).all()
    # the bodies for which the reference raises: the engine returns the evident intent (cop = cob, area 0)
    assert np.isfinite(F[raised]).all() and (F[raised][:, 2] > 0).all()
