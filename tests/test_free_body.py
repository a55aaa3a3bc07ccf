"""The free-body stepper (free_body_update, csrc/h2o_model.cuh) against the float64 reference oracle/free_body.py, with
tumbling anisotropic boxes: on the host through tests/host_emul/free_body_emul.cpp; physics checks that do not lean
on the reference; on the GPU through h2o_integrate_free_bodies, the persistent rollout (one step against the oracle,
K steps against K single steps, the trace) and the graph rollout; and what the persistent rollout refuses."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import free_body
from silver2_isaacsim_b200 import params as P
from silver2_isaacsim_b200 import workloads as W
from tests import scoring

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 2.0 ** -52
# Allowed float64 error, in ulps of the magnitude of the terms that form an output (_magnitudes).  Two evaluations of
# the same formulas differ by their roundings only (FMA contraction on one side, matmul or einsum order on the other).
ULPS = 8


@pytest.fixture(scope="session")
def free_body_emul(tmp_path_factory):
    """tests/host_emul/free_body_emul.cpp (free_body_update instantiated for the host), built into a temporary
    directory with the flags of the other emulators."""
    so = str(tmp_path_factory.mktemp("free_body_emul") / "libh2o_free_body_emul.so")
    subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-shared", "-mfma", "-ffp-contract=fast", "-fvisibility=hidden",
                    "-o", so, os.path.join(ROOT, "tests", "host_emul", "free_body_emul.cpp")], check=True)
    lib = ctypes.CDLL(so)
    lib.emul_free_body_step.restype = ctypes.c_int
    return lib


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _host_step(lib):
    def step(p, q, v, w, F, T, mass, dims, dt, gravity):
        p, q, v, w = (np.array(a, dtype=np.float64, order="C") for a in (p, q, v, w))
        F, T, m, d = (np.ascontiguousarray(a, dtype=np.float64) for a in (F, T, mass, dims))
        assert lib.emul_free_body_step(ctypes.c_int64(len(m)), _ptr(p), _ptr(q), _ptr(v), _ptr(w), _ptr(F), _ptr(T),
                                       _ptr(m), _ptr(d), ctypes.c_double(dt), ctypes.c_double(gravity)) == 0
        return p, q, v, w
    return step


def _rot_mag(q):
    """The terms of oracle.free_body._rot summed in absolute value."""
    x, y, z, w = np.moveaxis(np.abs(q), -1, 0)
    x2, y2, z2 = x + x, y + y, z + z
    rows = [[1 + (y * y2 + z * z2), x * y2 + w * z2, x * z2 + w * y2],
            [x * y2 + w * z2, 1 + (x * x2 + z * z2), y * z2 + w * x2],
            [x * z2 + w * y2, y * z2 + w * x2, 1 + (x * x2 + y * y2)]]
    return np.stack([np.stack(r, axis=-1) for r in rows], axis=-2)


def _magnitudes(p, q, v, w, F, T, mass, dims, dt, gravity):
    """Per output of one step, the magnitude of the terms that form it: the step's arithmetic on absolute values,
    every difference taken as a sum.  To first order, every rounding of the step is at most EPS times it."""
    a = np.abs
    m = np.asarray(mass, dtype=np.float64)[:, None]
    dx, dy, dz = np.moveaxis(dims, -1, 0)
    I = m * np.stack([dy * dy + dz * dz, dx * dx + dz * dz, dx * dx + dy * dy], axis=-1) / 12.0
    Mv = a(v) + dt * (a(F) / m + np.array([0.0, 0.0, abs(gravity)]))
    Mr = _rot_mag(q)
    Mtb, Mwb = np.einsum("...ji,...j->...i", Mr, a(T)), np.einsum("...ji,...j->...i", Mr, a(w))
    bx, by, bz = np.moveaxis(Mwb, -1, 0)
    Ix, Iy, Iz = np.moveaxis(I, -1, 0)
    Mg = np.stack([by * (Iz * bz) + bz * (Iy * by), bz * (Ix * bx) + bx * (Iz * bz), bx * (Iy * by) + by * (Ix * bx)],
                  axis=-1)
    Mw = np.einsum("...ij,...j->...i", Mr, Mwb + dt * (Mtb + Mg) / I)
    Mp = a(p) + dt * Mv
    x, y, z, s = np.moveaxis(a(q), -1, 0)
    wx, wy, wz = np.moveaxis(Mw, -1, 0)
    h = 0.5 * dt
    Mnq = np.stack([x + h * (wx * s + wy * z + wz * y), y + h * (wy * s + wz * x + wx * z),
                    z + h * (wz * s + wx * y + wy * x), s + h * (wx * x + wy * y + wz * z)], axis=-1)
    # |q + h (0, w) q| = |q| sqrt(1 + h^2 |w|^2) >= |q|: dividing by |q| bounds the normalised components
    Mq = Mnq / np.linalg.norm(q, axis=-1, keepdims=True)
    return Mp, Mq, Mv, Mw


def _assert_state(got, want, mag, what, f32=False):
    """fp64: within ULPS of the magnitudes.  fp32 (the kernel computes in double from float inputs and rounds
    once): at most one float32 ulp from the float64 reference rounded to float32."""
    for name, g, r, m in zip(("p", "q", "v", "w"), got, want, mag):
        g = np.asarray(g, dtype=np.float64)
        if f32:
            r32 = np.asarray(r, dtype=np.float64).astype(np.float32)
            err = np.abs(g - r32.astype(np.float64))
            tol = np.spacing(np.abs(r32)).astype(np.float64)
        else:
            err = np.abs(g - r)
            tol = ULPS * EPS * m
        bad = ~(err <= tol)
        assert not bad.any(), (what, name, int(bad.sum()), float((err / tol).max()))


def _random_boxes(rng, n, gravity=9.81):
    """Boxes of 0.05 - 3 m sides (a third of them plates or needles), unit and slightly non-unit quaternions,
    |w| up to 10 rad/s, forces up to ~30 g and torques up to ~30 rad/s^2 about the largest axis."""
    dims = np.exp(rng.uniform(np.log(0.05), np.log(3.0), (n, 3)))
    kind = rng.integers(0, 3, n)
    big = rng.uniform(1.0, 3.0, n)
    thin = rng.uniform(0.05, 0.1, n)
    dims[kind == 1] = np.stack([big, big, thin], axis=1)[kind == 1]       # plates
    dims[kind == 2] = np.stack([big, thin, thin], axis=1)[kind == 2]      # needles
    dims = np.take_along_axis(dims, rng.permuted(np.tile(np.arange(3), (n, 1)), axis=1), axis=1)
    mass = rng.uniform(100.0, 3000.0, n) * dims.prod(axis=1)
    q = rng.standard_normal((n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q[::3] *= 1.0 + rng.uniform(-1e-3, 1e-3, (len(q[::3]), 1))
    u = rng.standard_normal((n, 3))
    w = u / np.linalg.norm(u, axis=1, keepdims=True) * rng.uniform(0.0, 10.0, (n, 1))
    Imax = mass * (dims ** 2).sum(axis=1) / 12.0
    return dict(p=rng.uniform(-100.0, 100.0, (n, 3)), q=q, v=rng.standard_normal((n, 3)) * 3.0, w=w,
                F=rng.standard_normal((n, 3)) * (10.0 * gravity * mass)[:, None],
                T=rng.standard_normal((n, 3)) * (10.0 * Imax)[:, None], mass=mass, dims=dims)


def _args(b, keys=("p", "q", "v", "w", "F", "T", "mass", "dims")):
    return [b[k] for k in keys]


DTS = [1 / 60, 1 / 120, 1e-3]


# --------------------------------------------------------------------------- CPU: host stepper vs reference
@pytest.mark.parametrize("dt", DTS, ids=["dt60", "dt120", "dt1e-3"])
def test_host_stepper_matches_reference(free_body_emul, dt):
    b = _random_boxes(np.random.default_rng(int(1 / dt)), 10_000)
    args = _args(b) + [dt, 9.81]
    _assert_state(_host_step(free_body_emul)(*args), free_body.integrate(*args), _magnitudes(*args), "host stepper")


@pytest.fixture(params=["reference", "host"])
def stepper(request):
    if request.param == "reference":
        return free_body.integrate
    return _host_step(request.getfixturevalue("free_body_emul"))


def _inertia(mass, dims):
    dx, dy, dz = np.moveaxis(dims, -1, 0)
    return mass[:, None] * np.stack([dy * dy + dz * dz, dx * dx + dz * dz, dx * dx + dy * dy], axis=-1) / 12.0


def _momentum(q, w, mass, dims):
    """World angular momentum R I R^T w."""
    R = free_body._rot(q)
    wb = np.einsum("...ji,...j->...i", R, w)
    return np.einsum("...ij,...j->...i", R, _inertia(mass, dims) * wb)


def _tumbling_boxes(seed=1, n=20):
    rng = np.random.default_rng(seed)
    dims = rng.uniform(0.2, 2.0, (n, 3))
    q = rng.standard_normal((n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return q, rng.standard_normal((n, 3)), 500.0 * dims.prod(axis=1), dims


def _momentum_drift(step, dt, seconds=10.0):
    """Worst relative drift of the world angular momentum of 20 torque-free tumbling boxes, no gravity."""
    q, w, mass, dims = _tumbling_boxes()
    n = len(mass)
    z = np.zeros((n, 3))
    L0 = _momentum(q, w, mass, dims)
    p, v = z, z
    for _ in range(int(round(seconds / dt))):
        p, q, v, w = step(p, q, v, w, z, z, mass, dims, dt, 0.0)
    return float((np.linalg.norm(_momentum(q, w, mass, dims) - L0, axis=1) / np.linalg.norm(L0, axis=1)).max())


def _check_drift(coarse, fine):
    # the reference measures 3.1e-2 and 2.8e-3; a wrong gyroscopic sign or permuted inertia drifts O(1) at any dt
    assert coarse < 0.05 and coarse / fine >= 8.0, (coarse, fine)


def test_constant_force_closed_form(stepper):
    """No torque, constant force: semi-implicit Euler has v_n = v0 + n dt a, p_n = p0 + n dt v0 + dt^2 a n(n+1)/2."""
    rng = np.random.default_rng(5)
    n, dt, g, steps = 20, 1 / 120, 9.81, 1200
    b = _random_boxes(rng, n)
    p0, q, v0, w, F, mass, dims = b["p"], b["q"], b["v"], b["w"], b["F"], b["mass"], b["dims"]
    a = F / mass[:, None] + [0.0, 0.0, -g]
    p, v = p0, v0
    for _ in range(steps):
        p, q, v, w = stepper(p, q, v, w, F, np.zeros((n, 3)), mass, dims, dt, g)
    k = float(steps)
    vk, pk = v0 + k * dt * a, p0 + k * dt * v0 + dt * dt * a * (k * (k + 1) / 2)
    mv = np.abs(v0) + k * dt * np.abs(a)
    mp = np.abs(p0) + k * dt * np.abs(v0) + dt * dt * np.abs(a) * (k * (k + 1) / 2)
    assert (np.abs(v - vk) <= 4 * k * EPS * mv).all() and (np.abs(p - pk) <= 4 * k * EPS * mp).all()


def test_torque_free_momentum_drift(stepper):
    """Torque-free tumbling: the world angular momentum drifts only to first order in dt."""
    _check_drift(_momentum_drift(stepper, 1 / 120), _momentum_drift(stepper, 1 / 1200))


def _spin(step, axis, rate, dt, seconds, perturb=0.0, dims=(3.0, 2.0, 1.0), mass=100.0):
    """Spin a box about a body axis from the identity; returns the worst off-axis body rate and the final state."""
    q = np.array([[0.0, 0.0, 0.0, 1.0]])
    w = np.full((1, 3), perturb)
    w[0, axis] = rate
    z = np.zeros((1, 3))
    p, v, worst = z, z, 0.0
    m, d = np.array([mass]), np.array([dims], dtype=np.float64)
    for _ in range(int(round(seconds / dt))):
        p, q, v, w = step(p, q, v, w, z, z, m, d, dt, 0.0)
        wb = np.einsum("ji,j->i", free_body._rot(q[0]), w[0])
        worst = max(worst, float(np.abs(np.delete(wb, axis)).max()))
    return worst, q[0], w[0]


@pytest.mark.parametrize("axis", [0, 1, 2], ids=["x", "y", "z"])
def test_intermediate_axis_theorem(stepper, axis):
    """Box 3 x 2 x 1: spin about the largest (z) and smallest (x) inertia axes is stable, about the intermediate
    (y) axis a 1e-3 perturbation grows until the box flips (reference: 1.8e-3, 1.6e-3, 1.43)."""
    worst, _, _ = _spin(stepper, axis, 2.0, 1 / 240, 10.0, perturb=1e-3)
    if axis == 1:
        assert worst > 1.0, worst
    else:
        assert worst < 5e-3, worst


@pytest.mark.parametrize("axis", [0, 1, 2], ids=["x", "y", "z"])
def test_principal_axis_spin(stepper, axis):
    """Spin about a principal axis stays on it; the angle after 1 s is |w| t (reference error 4.6e-5)."""
    worst, q, w = _spin(stepper, axis, 2.0, 1 / 120, 1.0)
    assert worst < 1e-12 and abs(w[axis] - 2.0) < 1e-12
    assert abs(2.0 * math.atan2(q[axis], q[3]) - 2.0) < 1e-4


# --------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu
DTYPES = pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
ORDERS = pytest.mark.parametrize("order", ["xyzw", "wxyz"])


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda:0")


def _npdt(dtype):
    return np.float32 if dtype == torch.float32 else np.float64


def _stored(a, dtype):
    """What the engine holds: a rounded to the engine dtype, as float64."""
    return np.asarray(a, dtype=np.float64).astype(_npdt(dtype)).astype(np.float64)


def _to_dev(a, dtype, dev, order="xyzw"):
    a = np.asarray(a)
    if order == "wxyz" and a.shape[-1] == 4:
        a = a[:, [3, 0, 1, 2]]
    return torch.as_tensor(np.ascontiguousarray(a, dtype=_npdt(dtype)), device=dev)


def _from_dev(t, order="xyzw"):
    a = t.double().cpu().numpy()
    return a[:, [1, 2, 3, 0]] if order == "wxyz" and a.shape[-1] == 4 else a


def _engine(n, dtype, dev, order, params, coeff=None, rho=1025.0, g=9.81):
    """params 'table': the 19-slot hexapod part table (body i is slot i % 19); 'per_body': the (n,11) records coeff.
    Returns the engine and the (n,11) float64 records as the engine stores them."""
    from silver2_isaacsim_b200 import HydroEngine

    e = HydroEngine(n, dtype=dtype, device=dev, quat_order=order)
    e.set_globals(rho, g)
    if params == "table":
        table, slot_type, _, _ = P.hexapod_table()
        table = _stored(table, dtype)
        e.set_part_table(table, slot_type)
        return e, table[slot_type[np.arange(n) % len(slot_type)]]
    coeff = _stored(coeff, dtype)
    e.set_params_per_body(coeff.astype(_npdt(dtype)))
    return e, coeff


def _box_records(b):
    """(n,11) records of _random_boxes: their dimensions and masses, README coefficients otherwise."""
    rec = np.tile(np.asarray(P.HydroParams().coeff_record(1.0), dtype=np.float64), (len(b["mass"]), 1))
    rec[:, 0:3], rec[:, 10] = b["dims"], b["mass"]
    return rec


@gpu
@DTYPES
@ORDERS
@pytest.mark.parametrize("params", ["table", "per_body"])
@pytest.mark.parametrize("n", [1, 255, 257, 100_003])
def test_integrate_free_bodies_matches_reference(dev, dtype, order, params, n):
    """h2o_integrate_free_bodies against free_body.integrate, of the same stored inputs."""
    b = _random_boxes(np.random.default_rng(n), n)
    e, rec = _engine(n, dtype, dev, order, params, _box_records(b))
    b["dims"], b["mass"] = rec[:, 0:3], rec[:, 10]
    for k in ("p", "q", "v", "w", "F", "T"):
        b[k] = _stored(b[k], dtype)
    ten = [_to_dev(b[k], dtype, dev, order) for k in ("p", "q", "v", "w", "F", "T")]
    dt, g = 1 / 120, 9.81
    e.integrate_free_bodies(*ten, dt, g)
    got = [_from_dev(t, order) for t in ten[:4]]
    args = _args(b) + [dt, g]
    _assert_state(got, free_body.integrate(*args), _magnitudes(*args), "h2o_integrate_free_bodies",
                  f32=dtype == torch.float32)
    assert np.array_equal(_from_dev(ten[4]), b["F"]) and np.array_equal(_from_dev(ten[5]), b["T"])


def _hydro_state(kind, n, dtype, strict_quats):
    """Hydrodynamic bodies for the fused step: 'per_body' C3 boxes, or 'table' hexapod bodies (any n).  With
    strict_quats a few quaternions are 1e-6 - 1e-3 off unit, which the fp32 step re-evaluates in float64."""
    if kind == "per_body":
        wl = W.heterogeneous_boxes(n, seed=n)
    else:
        wl = W.hexapod_envs(-(-n // 19), seed=n)
    st = {k: _stored(getattr(wl, a)[:n], dtype) for k, a in (("p", "pos"), ("q", "quat_xyzw"), ("v", "lin_vel"),
                                                              ("w", "ang_vel"), ("pv", "prev_lin"), ("pw", "prev_ang"))}
    if strict_quats:
        rng = np.random.default_rng(n + 1)
        sel = np.arange(0, n, 17)
        f = 1.0 + rng.choice([-1.0, 1.0], len(sel)) * rng.uniform(2e-6, 1e-3, len(sel))
        st["q"][sel] = _stored(st["q"][sel] * f[:, None], dtype)
        assert (np.abs((st["q"][sel] ** 2).sum(axis=1) - 1.0) > 1e-6).all()
    return wl, st


def _bind(e, st, dtype, dev, order):
    ten = [_to_dev(st[k], dtype, dev, order) for k in ("p", "q", "v", "w")]
    e.set_prev(_to_dev(st["pv"], dtype, dev), _to_dev(st["pw"], dtype, dev))
    F, T = e.bind(*ten)
    return ten, F, T


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


PRECISION = pytest.mark.parametrize("dtype,strict", [(torch.float32, True), (torch.float32, False),
                                                     (torch.float64, True)], ids=["fp32", "fp32_lax", "fp64"])


@gpu
@PRECISION
@ORDERS
@pytest.mark.parametrize("params", ["table", "per_body"])
@pytest.mark.parametrize("side", [-1, 1], ids=["warp_ctas", "128_ctas"])
def test_persistent_one_step_matches_oracle(oracle, dev, dtype, strict, order, params, side):
    """A one-step persistent rollout = oracle.step, then free_body.integrate of the GPU's own wrench; the carried
    velocities are the input velocities.  n = 128 sm_count +- 1: both CTA sizes of the kernel."""
    n = 128 * _sm_count() + side
    wl, st = _hydro_state(params, n, dtype, strict_quats=strict)
    coeff = wl.coeff_per_body()[:n] if params == "per_body" else None
    e, rec = _engine(n, dtype, dev, order, params, coeff, wl.rho, wl.g)
    e.set_strict(strict)
    ten, F, T = _bind(e, st, dtype, dev, order)
    e.rollout_persistent(1, wl.dt, gravity=wl.g)
    torch.cuda.synchronize()
    Fg, Tg = _from_dev(F), _from_dev(T)
    ref = oracle.step(P.coeff_to_ctor_rows(rec, wl.rho, wl.g), rec[:, 10], st["p"], st["q"], st["v"], st["w"],
                      st["pv"], st["pw"], wl.dt)
    if dtype == torch.float32:
        # without strict mode about one body per million misses the bound by up to 3x (include/h2o.h)
        lax = dict(min_pass=1.0 - 1e-4, hard_factor=3.0) if not strict else {}
        scoring.assert_fp32(Fg, ref.force, "one-step force", **lax)
        scoring.assert_fp32(Tg, ref.torque, "one-step torque", **lax)
    else:
        scale = scoring.force_scale(rec, wl.rho, wl.g)
        assert scoring.fp64_ok(Fg, ref.force, scale).all()
        pn = np.abs(st["p"]).max(axis=1) * np.abs(ref.force).max(axis=1)
        assert scoring.fp64_ok(Tg, ref.torque, scale, extra=pn).all()
    prev = e.prev_velocities().double().cpu().numpy()
    assert np.array_equal(prev[:, :3], st["v"]) and np.array_equal(prev[:, 3:], st["w"])
    args = [st["p"], st["q"], st["v"], st["w"], Fg, Tg, rec[:, 10], rec[:, 0:3], wl.dt, wl.g]
    _assert_state([_from_dev(t, order) for t in ten], free_body.integrate(*args), _magnitudes(*args),
                  "one-step persistent rollout", f32=dtype == torch.float32)


def _sea(e, wl, dev, rng):
    """A wave field, per-env conditions (envs of 4 bodies) and a time-varying current grid; returns what the engine
    borrows."""
    from silver2_isaacsim_b200 import currents, waves

    e.set_wave_field(waves.jonswap(1.5, 7.0, n_components=16, direction=0.4, seed=3))
    cond = torch.as_tensor(waves.env_conditions(wl.n // 4, current=rng.uniform(-0.5, 0.5, (wl.n // 4, 3)),
                                                surface_dz=rng.uniform(-0.3, 0.3, wl.n // 4),
                                                wave_scale=rng.uniform(0.0, 2.0, wl.n // 4),
                                                time_offset=rng.uniform(0.0, 100.0, wl.n // 4)), device=dev)
    e.set_env_conditions(cond, 4)
    g = currents.CurrentGrid(rng.uniform(-0.8, 0.8, (3, 4, 5, 6, 3)), origin=(-60.0, -60.0, -3.0),
                             spacing=(25.0, 30.0, 1.5), t0=0.0, frame_dt=0.2)
    vals = torch.as_tensor(np.array(g.values), device=dev)
    e.set_current_grid(vals, g.origin, g.spacing, g.t0, g.frame_dt)
    return cond, vals


def _persistent_runs(dev, dtype, sea, K, plans):
    """Run the same start state through each plan: a list of (n_steps, trace_every) persistent calls.  Returns per
    plan the final tensors and the traces."""
    wl = W.heterogeneous_boxes(4000, seed=12, xy_range=50.0)
    wl.pos[:, 2] = np.random.default_rng(13).uniform(-2.5, 1.0, wl.n).astype(np.float32)
    out = []
    for plan in plans:
        e, rec = _engine(wl.n, dtype, dev, "xyzw", "per_body", wl.coeff, wl.rho, wl.g)
        keep = _sea(e, wl, dev, np.random.default_rng(14)) if sea else None
        st = {k: _stored(getattr(wl, a), dtype) for k, a in (("p", "pos"), ("q", "quat_xyzw"), ("v", "lin_vel"),
                                                             ("w", "ang_vel"), ("pv", "prev_lin"), ("pw", "prev_ang"))}
        ten, F, T = _bind(e, st, dtype, dev, "xyzw")
        traces = []
        for steps, te in plan:
            tr = e.rollout_persistent(steps, wl.dt, gravity=wl.g, trace_every=te)
            traces.append(None if tr is None else tr.cpu())
        torch.cuda.synchronize()
        out.append(([t.cpu() for t in ten + [F, T, e.prev_velocities()]], traces, e.wave_time))
        del keep
    return out


def _bits(t):
    return t.contiguous().view(torch.int32 if t.dtype == torch.float32 else torch.int64)


@gpu
@DTYPES
@pytest.mark.parametrize("sea", [False, True], ids=["still", "sea"])
def test_persistent_k_steps_equal_k_single_steps(dev, dtype, sea):
    """K = 50 steps in one launch == 50 one-step launches, bit for bit (state, carried velocities, last wrench,
    clock): the same instantiation with the same per-step roundings and the same clock additions."""
    K = 50
    (a, _, ta), (b, _, tb) = _persistent_runs(dev, dtype, sea, K, [[(K, 0)], [(1, 0)] * K])
    for name, x, y in zip(("pos", "quat", "lin_vel", "ang_vel", "force", "torque", "prev"), a, b):
        assert torch.equal(_bits(x), _bits(y)), name
    assert ta == tb


@gpu
@DTYPES
def test_persistent_trace(dev, dtype):
    """Trace row j of a K = 10 rollout is the state [p, v, w] after step (j + 1) trace_every of single steps, bit for
    bit, for trace_every 1, 3 and K; trace_every > K is refused."""
    K = 10
    plans = [[(1, 1)] * K, [(K, 1)], [(K, 3)], [(K, K)]]
    runs = _persistent_runs(dev, dtype, False, K, plans)
    single = torch.stack([tr[0] for tr in runs[0][1]])                 # (K, n, 9): after steps 1 .. K
    for (_, traces, _), te in zip(runs[1:], (1, 3, K)):
        tr = traces[0]
        assert tuple(tr.shape) == (K // te, single.shape[1], 9)
        assert torch.equal(_bits(tr), _bits(single[te - 1::te][:K // te])), te
    from silver2_isaacsim_b200 import HydroEngine

    e = HydroEngine(19, dtype=dtype, device=dev)
    table, slot_type, _, _ = P.hexapod_table()
    e.set_part_table(table, slot_type)
    z = torch.zeros(19, 3, dtype=dtype, device=dev)
    q = torch.zeros(19, 4, dtype=dtype, device=dev)
    q[:, 3] = 1.0
    e.bind(z.clone(), q, z.clone(), z.clone())
    with pytest.raises(ValueError):
        e.rollout_persistent(K, 1 / 60, trace_every=K + 1)
    buf = torch.zeros(1, 19, 9, dtype=dtype, device=dev)
    assert e._lib.h2o_rollout_persistent(e._h, K, 1 / 60, 9.81, K + 1, ctypes.c_void_p(buf.data_ptr()), None) == 2
    assert e.launch_count == 0 and not buf.any()                       # H2O_ERR_BAD_ARGUMENT, nothing launched


@gpu
@DTYPES
@ORDERS
def test_graph_rollout_equals_eager_steps(dev, dtype, order):
    """Graph rollout in free-body mode == eager step_bound + integrate_free_bodies, bit for bit, on tumbling
    anisotropic boxes (per-body records)."""
    wl, st = _hydro_state("per_body", 3001, dtype, strict_quats=True)
    st["w"] = _stored(st["w"] * 3.0, dtype)
    K, res = 6, []
    for mode in ("eager", "graph"):
        e, _ = _engine(wl.n, dtype, dev, order, "per_body", wl.coeff_per_body(), wl.rho, wl.g)
        ten, F, T = _bind(e, st, dtype, dev, order)
        if mode == "eager":
            for _ in range(2 * K):
                e.step_bound(wl.dt)
                e.integrate_free_bodies(*ten, F, T, wl.dt, wl.g)
        else:
            e.set_rollout_mode(free_bodies=True, gravity=wl.g)
            e.capture_rollout(K, wl.dt)
            e.launch_rollout()
            e.launch_rollout()
        torch.cuda.synchronize()
        res.append([t.cpu() for t in ten + [F, T, e.prev_velocities()]])
    assert not torch.equal(res[0][3], _to_dev(st["w"], dtype, dev).cpu())    # the boxes did tumble
    for name, x, y in zip(("pos", "quat", "lin_vel", "ang_vel", "force", "torque", "prev"), *res):
        assert torch.equal(_bits(x), _bits(y)), name


@gpu
def test_torque_free_tumbling_on_device(dev):
    """h2o_integrate_free_bodies (fp64) with F = T = 0 and no gravity: the momentum drift bounds of the CPU test."""
    from silver2_isaacsim_b200 import HydroEngine

    drift = []
    for dt in (1 / 120, 1 / 1200):
        q, w, mass, dims = _tumbling_boxes()
        n = len(mass)
        rec = np.tile(np.asarray(P.HydroParams().coeff_record(1.0), dtype=np.float64), (n, 1))
        rec[:, 0:3], rec[:, 10] = dims, mass
        e = HydroEngine(n, dtype=torch.float64, device=dev)
        e.set_params_per_body(rec)
        z = np.zeros((n, 3))
        ten = [_to_dev(a, torch.float64, dev) for a in (z, q, z, w, z, z)]
        for _ in range(int(round(10.0 / dt))):
            e.integrate_free_bodies(*ten, dt, 0.0)
        qf, wf = _from_dev(ten[1]), _from_dev(ten[3])
        L0, L1 = _momentum(q, w, mass, dims), _momentum(qf, wf, mass, dims)
        drift.append(float((np.linalg.norm(L1 - L0, axis=1) / np.linalg.norm(L0, axis=1)).max()))
        assert not _from_dev(ten[0]).any() and not _from_dev(ten[2]).any()
    _check_drift(*drift)


def _small_hexapod(dev, dtype, robots=8):
    wl = W.hexapod_envs(robots, seed=77)
    e, rec = _engine(wl.n, dtype, dev, "xyzw", "table", rho=wl.rho, g=wl.g)
    st = {k: _stored(getattr(wl, a), dtype) for k, a in (("p", "pos"), ("q", "quat_xyzw"), ("v", "lin_vel"),
                                                         ("w", "ang_vel"), ("pv", "prev_lin"), ("pw", "prev_ang"))}
    return wl, e, st, rec


@gpu
@DTYPES
def test_persistent_refuses_warp_compat(oracle, dev, dtype):
    """The persistent rollout computes the Numba semantics only: with Warp compatibility on it refuses and leaves
    the state alone; the graph rollout honours the switch and matches the oracle in Warp mode."""
    from silver2_isaacsim_b200 import _lib as L

    wl, e, st, rec = _small_hexapod(dev, dtype)
    e.set_warp_compat(True)
    ten, F, T = _bind(e, st, dtype, dev, "xyzw")
    before = [t.clone() for t in ten]
    with pytest.raises(L.H2OError) as exc:
        e.rollout_persistent(3, wl.dt, gravity=wl.g)
    assert exc.value.status == 8                                       # H2O_ERR_NOT_CONFIGURED
    assert all(torch.equal(a, b) for a, b in zip(before, ten)) and e.launch_count == 0
    e.set_rollout_mode(free_bodies=True, gravity=wl.g)
    e.capture_rollout(1, wl.dt)
    e.launch_rollout()
    torch.cuda.synchronize()
    try:
        oracle.set_warp_compat(True)
        ref = oracle.step(P.coeff_to_ctor_rows(rec, wl.rho, wl.g), rec[:, 10], st["p"], st["q"], st["v"], st["w"],
                          st["pv"], st["pw"], wl.dt)
    finally:
        oracle.set_warp_compat(False)
    Fg, Tg = _from_dev(F), _from_dev(T)
    if dtype == torch.float32:
        scoring.assert_fp32(Fg, ref.force, "warp-compat graph force")
        scoring.assert_fp32(Tg, ref.torque, "warp-compat graph torque")
    else:
        scale = scoring.force_scale(rec, wl.rho, wl.g)
        pn = np.abs(st["p"]).max(axis=1) * np.abs(ref.force).max(axis=1)
        assert scoring.fp64_ok(Fg, ref.force, scale).all() and scoring.fp64_ok(Tg, ref.torque, scale, extra=pn).all()
    args = [st["p"], st["q"], st["v"], st["w"], Fg, Tg, rec[:, 10], rec[:, 0:3], wl.dt, wl.g]
    _assert_state([_from_dev(t) for t in ten], free_body.integrate(*args), _magnitudes(*args), "warp-compat graph",
                  f32=dtype == torch.float32)


@gpu
def test_persistent_refuses_robot_wrench_output(dev):
    """The persistent rollout writes no robot wrench: bound with a robot-wrench output it refuses."""
    from silver2_isaacsim_b200 import _lib as L

    wl, e, st, _ = _small_hexapod(dev, torch.float32)
    e.set_articulation(19)
    ten = [_to_dev(st[k], torch.float32, dev) for k in ("p", "q", "v", "w")]
    e.bind(*ten, robot_wrench=True)
    with pytest.raises(L.H2OError) as exc:
        e.rollout_persistent(3, wl.dt, gravity=wl.g)
    assert exc.value.status == 8 and e.launch_count == 0
    e.bind(*ten)                                                      # without the wrench output it runs
    e.rollout_persistent(3, wl.dt, gravity=wl.g)
    torch.cuda.synchronize()
    assert e.launch_count == 1
