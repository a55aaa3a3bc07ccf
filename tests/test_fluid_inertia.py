"""Fluid-acceleration loads (include/h2o.h, h2o_set_fluid_inertia): the NumPy references of the water's acceleration,
the acceleration evaluator and the model with the inertia group on the host (tests/host_emul/inertia_emul.cpp) against
NumPy and the float64 reference (tests/inertia_reference.py), and on the GPU the sampler, strict step parity, the
opt-in, the step paths, rollouts and a particle-orbit check."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from silver2_isaacsim_b200 import currents
from silver2_isaacsim_b200 import params as P
from silver2_isaacsim_b200 import waves
from silver2_isaacsim_b200 import workloads as W
from tests import inertia_reference as IR
from tests import scoring

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = np.finfo(np.float64).eps


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="session")
def inertia_emul(tmp_path_factory):
    """tests/host_emul/inertia_emul.cpp built into a temporary directory, without multiply-add contraction (so that
    the instantiations with and without the mode are comparable bit for bit)."""
    so = str(tmp_path_factory.mktemp("inertia_emul") / "libh2o_inertia_emul.so")
    subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-shared", "-mfma", "-ffp-contract=off", "-fvisibility=hidden",
                    "-o", so, os.path.join(ROOT, "tests", "host_emul", "inertia_emul.cpp")], check=True)
    lib = ctypes.CDLL(so)
    lib.emul_accel_sample.restype = ctypes.c_int
    lib.emul_inertia_step.restype = ctypes.c_int
    return lib


def _emul_accel(lib, field, points, t, f32, grid=None, env_index=None, cond=None):
    p = np.ascontiguousarray(points, dtype=np.float64)
    c = np.zeros((0, 5)) if field is None else np.ascontiguousarray(field.components, dtype=np.float64)
    depth = math.inf if field is None else field.depth
    out = np.zeros((len(p), 3))
    idx = None if env_index is None else np.ascontiguousarray(env_index, dtype=np.int32)
    cd = np.zeros((1, 8)) if cond is None else np.ascontiguousarray(cond, dtype=np.float64)
    gv = dims = geom = None
    if grid is not None:
        gv = np.ascontiguousarray(grid.values)
        dims = np.array(grid.dims, dtype=np.int64)
        geom = np.ascontiguousarray(grid.geometry)
    rc = lib.emul_accel_sample(int(f32), len(c), _ptr(c), ctypes.c_double(depth), None if gv is None else _ptr(gv),
                               None if dims is None else _ptr(dims), None if geom is None else _ptr(geom),
                               ctypes.c_int64(len(p)), _ptr(p), None if idx is None else _ptr(idx),
                               ctypes.c_int64(len(cd)), _ptr(cd), ctypes.c_double(t), ctypes.c_double(0.0), _ptr(out))
    assert rc == 0
    return out


def _emul_step(lib, mode, inertia_on, slope_on, pos, quat, v, w, a, b, coeff, rho, g, slope, af, dense=None):
    d = lambda x: np.ascontiguousarray(x, dtype=np.float64)
    n = len(pos)
    arrs = [d(x) for x in (pos, quat, v, w, a, b, coeff)]
    sl, afa = d(slope), d(af)
    dn = None if dense is None else d(dense).reshape(n, 36)
    F, T, comp = np.zeros((n, 3)), np.zeros((n, 3)), np.zeros((n, 4))
    rc = lib.emul_inertia_step(mode, int(inertia_on), int(slope_on), ctypes.c_int64(n), *[_ptr(x) for x in arrs],
                               ctypes.c_double(rho), ctypes.c_double(g), _ptr(sl), _ptr(afa),
                               None if dn is None else _ptr(dn), _ptr(F), _ptr(T), _ptr(comp))
    assert rc == 0
    return F, T, comp


FIELDS = {
    "regular_deep": lambda: waves.regular(0.4, 6.0, direction=0.7, phase=0.3),
    "jonswap16_deep": lambda: waves.jonswap(2.0, 7.0, n_components=16, direction=0.4, seed=3),
    "jonswap64_h12": lambda: waves.jonswap(1.5, 9.0, n_components=64, direction=-1.0, seed=5, depth=12.0),
}


def _aw2(field):
    c = field.components
    return float((c[:, 0] * c[:, 3] ** 2).sum())


def _cond(rng, n_envs, tau=100.0):
    return waves.env_conditions(n_envs, current=rng.uniform(-0.5, 0.5, (n_envs, 3)),
                                surface_dz=rng.uniform(-0.3, 0.3, n_envs), wave_scale=rng.uniform(0.0, 2.0, n_envs),
                                time_offset=rng.uniform(0.0, tau, n_envs), origin=rng.uniform(-80, 80, (n_envs, 2)))


def _grid(rng, nt=2, t0=1230.0, ht=10.0):
    """A smooth (nt, 3, 4, 5) current grid over x, y in [-160, 160], z in [-4, 0], frames t0 + f ht."""
    vals = rng.uniform(-0.6, 0.6, (nt, 3, 4, 5, 3))
    return currents.CurrentGrid(vals, origin=(-160.0, -160.0, -4.0), spacing=(80.0, 320.0 / 3, 2.0), t0=t0,
                                frame_dt=ht)


# --------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", sorted(FIELDS))
def test_acceleration_is_the_time_derivative(name):
    """waves.acceleration against the central time difference of waves.evaluate's orbital velocity, below and above
    the surface (clamped), env twin included; one component against its analytic value."""
    field = FIELDS[name]()
    rng = np.random.default_rng(1)
    m, h, t = 2000, 1e-4, 321.25
    p = np.stack([rng.uniform(-300, 300, m), rng.uniform(-300, 300, m), rng.uniform(-6, 2, m)], axis=1)
    fd = (waves.evaluate(field, p, t + h)[:, 1:] - waves.evaluate(field, p, t - h)[:, 1:]) / (2 * h)
    got = waves.acceleration(field, p, t)
    assert got.shape == (m, 3)
    assert np.abs(got - fd).max() <= 1e-6 * _aw2(field)
    above = p[:, 2] > 0
    assert above.any() and np.array_equal(got[above], waves.acceleration(field, p[above] * [1, 1, 0], t))
    cond = _cond(rng, 7)
    env = rng.integers(0, 7, m)
    fd_env = (waves.evaluate_env(field, p, t + h, cond, env)[:, 1:] -
              waves.evaluate_env(field, p, t - h, cond, env)[:, 1:]) / (2 * h)
    assert np.abs(waves.acceleration_env(field, p, t, cond, env) - fd_env).max() <= 2e-6 * _aw2(field)
    if name == "regular_deep":  # a omega^2 e^{kz} (sin theta khat, -cos theta)
        a, kx, ky, om, ph = field.components[0]
        k = math.hypot(kx, ky)
        th = (kx * p[:, 0] + ky * p[:, 1]) - om * t + ph
        e = a * om * om * np.exp(k * np.minimum(p[:, 2], 0.0))
        want = np.stack([e * np.sin(th) * kx / k, e * np.sin(th) * ky / k, -e * np.cos(th)], axis=1)
        assert np.abs(got - want).max() <= 1e-12 * a * om * om


def test_grid_time_derivative():
    """currents.time_derivative is exact for a grid linear in time, and zero for one frame and outside the frames."""
    rng = np.random.default_rng(2)
    base, slope_t = rng.uniform(-1, 1, (3, 4, 5, 3)), rng.uniform(-0.1, 0.1, (3, 4, 5, 3))
    t0, ht, nt = 10.0, 0.5, 5
    g = currents.CurrentGrid(np.stack([base + slope_t * (t0 + f * ht) for f in range(nt)]), origin=(-2.0, -3.0, -4.0),
                             spacing=(1.0, 2.0, 2.0), t0=t0, frame_dt=ht)
    m = 3000
    x, y, z = rng.uniform(-3, 3, m), rng.uniform(-4, 4, m), rng.uniform(-5, 1, m)
    t = rng.uniform(t0, t0 + (nt - 1) * ht, m)
    got = currents.time_derivative(g, x, y, z, t)
    want = currents.time_derivative(currents.CurrentGrid(slope_t[None], origin=g.origin, spacing=g.spacing), x, y, z, 0)
    assert not want.any()                                                  # one frame: zero
    want = currents.evaluate(currents.CurrentGrid(slope_t[None], origin=g.origin, spacing=g.spacing), x, y, z, 0.0)
    assert np.abs(got - want).max() <= 1e-12
    fd = (currents.evaluate(g, x, y, z, t + 1e-3) - currents.evaluate(g, x, y, z, t - 1e-3)) / 2e-3
    inner = (t > t0 + 1e-3) & (t < t0 + (nt - 1) * ht - 1e-3) & (np.abs(((t - t0) / ht) % 1 - 0.5) < 0.49)
    assert np.abs(got[inner] - fd[inner]).max() <= 1e-9
    outside = np.concatenate([rng.uniform(t0 - 5, t0 - 1e-9, 50), rng.uniform(t0 + (nt - 1) * ht + 1e-9, 100, 50)])
    assert not currents.time_derivative(g, x[:100], y[:100], z[:100], outside).any()
    edge = currents.time_derivative(g, x[:2], y[:2], z[:2], [t0, t0 + (nt - 1) * ht])
    assert np.abs(edge - want[:2]).max() <= 1e-12                          # the frame range is closed
    assert np.isnan(currents.time_derivative(g, [np.nan], [0.0], [0.0], [t0 + 0.1])).all()


@pytest.mark.parametrize("f32", [False, True], ids=["fp64", "fp32"])
@pytest.mark.parametrize("name", sorted(FIELDS))
def test_host_accel_evaluator_matches_reference(inertia_emul, name, f32):
    """The evaluator the kernels inline (water_at with a_f) against waves.acceleration(_env) + currents.time_derivative:
    env rows, a two-frame grid, waves plus the grid; fp64 to rounding, fp32 within 2e-6 of sum a_j omega_j^2 (the
    velocity's bound, scaled); a NaN row for an env index outside [0, E)."""
    field = FIELDS[name]()
    rng = np.random.default_rng(3)
    m = 20000
    p = np.stack([rng.uniform(-150, 150, m), rng.uniform(-150, 150, m), rng.uniform(-5, 2, m)], axis=1)
    if f32:
        p = p.astype(np.float32).astype(np.float64)
    tol = (2e-6 if f32 else 64 * EPS) * _aw2(field)
    grid = _grid(rng)
    for t in (1231.0, 1234.5, 99999.37):
        got = _emul_accel(inertia_emul, field, p, t, f32)
        assert np.abs(got - waves.acceleration(field, p, t)).max() <= tol, t
        z = np.minimum(p[:, 2], np.inf)
        dg = currents.time_derivative(grid, p[:, 0], p[:, 1], z, t)
        got = _emul_accel(inertia_emul, None, p, t, f32, grid=grid)
        assert np.abs(got - dg).max() <= 64 * EPS, t                       # float64 in both policies
        got = _emul_accel(inertia_emul, field, p, t, f32, grid=grid)
        assert np.abs(got - (dg + waves.acceleration(field, p, t))).max() <= tol + 64 * EPS, t
        cond = _cond(rng, 5, tau=8.0)
        env = rng.integers(-1, 6, m)
        got = _emul_accel(inertia_emul, field, p, t, f32, grid=grid, env_index=env, cond=cond)
        bad = (env < 0) | (env >= 5)
        assert np.isnan(got[bad]).all() and np.isfinite(got[~bad]).all()
        r = cond[env[~bad]]
        q = p[~bad]
        dge = currents.time_derivative(grid, q[:, 0] - r[:, 6], q[:, 1] - r[:, 7], q[:, 2] - r[:, 3], t + r[:, 5])
        want = dge + waves.acceleration_env(field, q, t, cond, env[~bad])
        assert np.abs(got[~bad] - want).max() <= 2.0 * tol + 64 * EPS, t


def _random_bodies(rng, n, f32=False):
    dims = rng.uniform(0.1, 2.0, (n, 3))
    coeff = np.empty((n, 11))
    coeff[:, 0:3] = dims
    coeff[:, 3] = rng.uniform(0.5, 1.5, n)
    coeff[:, 4] = rng.uniform(0.05, 1.0, n)
    coeff[:, 5] = rng.uniform(5.0, 400.0, n)
    coeff[:, 6] = rng.uniform(1.0, 200.0, n)
    coeff[:, 7] = rng.uniform(0.0, 0.3, n)
    coeff[:, 8] = rng.uniform(0.0, 0.2, n)
    coeff[:, 9] = rng.uniform(0.0, 1.0, n)
    coeff[:, 10] = rng.uniform(0.3, 1.5, n) * 1025.0 * dims.prod(axis=1)
    v, w = rng.uniform(-1.5, 1.5, (n, 3)), rng.uniform(-1.0, 1.0, (n, 3))
    a, b = rng.uniform(-3, 3, (n, 3)), rng.uniform(-3, 3, (n, 3))
    if f32:
        coeff, v, w, a, b = (x.astype(np.float32).astype(np.float64) for x in (coeff, v, w, a, b))
    return coeff, v, w, a, b


def _dense(rng):
    return rng.uniform(-20.0, 20.0, (3, 6, 6)) + np.eye(6)[None] * 200.0, np.array([0, 2, 1, 1], dtype=np.int32)


@pytest.mark.parametrize("dense", [False, True], ids=["diag", "dense"])
@pytest.mark.parametrize("mode", [0, 1], ids=["fp64", "fp32_fast"])
def test_zero_acceleration_equals_mode_off(inertia_emul, mode, dense):
    """The inertia instantiation with a_f = 0 gives the values of the one without (every nonzero bit for bit; a zero
    may change sign, which is why the engine decides inertness in its dispatch), and the same flagged bodies."""
    wl = W.heterogeneous_boxes(30000, seed=21)
    rng = np.random.default_rng(4)
    coeff, v, w, a, b = _random_bodies(rng, wl.n, f32=mode == 1)
    D = None
    if dense:
        M, slots = _dense(rng)
        D = M[slots[np.arange(wl.n) % len(slots)]]
    pos = wl.pos.astype(np.float64)
    z2, z3 = np.zeros((wl.n, 2)), np.zeros((wl.n, 3))
    on = _emul_step(inertia_emul, mode, True, False, pos, wl.quat_xyzw, v, w, a, b, coeff, 1025.0, 9.81, z2, z3, D)
    off = _emul_step(inertia_emul, mode, False, False, pos, wl.quat_xyzw, v, w, a, b, coeff, 1025.0, 9.81, z2, z3, D)
    for x, y in zip(on[:2], off[:2]):
        assert np.array_equal(x, y)
        nz = y != 0
        assert np.array_equal(x[nz].view(np.int64), y[nz].view(np.int64))
    assert np.array_equal(on[2][:, :2], off[2][:, :2])


def _wet_random(wl, rng):
    pos = wl.pos.astype(np.float64)
    pos[:, 2] = rng.uniform(-1.5, 0.8, wl.n)
    return pos


@pytest.mark.parametrize("slope", [False, True], ids=["flat", "slope"])
@pytest.mark.parametrize("mode", [0, 1], ids=["fp64", "fp32_fast"])
def test_host_model_with_inertia_matches_reference(inertia_emul, mode, slope):
    """The host model with the inertia group against the float64 reference fed the same a_f (and slope), under the
    strict bounds; fp32 flagged bodies are re-evaluated in float64; the group is a material share of |F|."""
    wl = W.heterogeneous_boxes(100000, seed=22, xy_range=150.0)
    rng = np.random.default_rng(5)
    pos = _wet_random(wl, rng)
    pos[:, 0:2] = 0.0
    sl = rng.uniform(-0.3, 0.3, (wl.n, 2)) if slope else np.zeros((wl.n, 2))
    af = rng.uniform(-3.0, 3.0, (wl.n, 3))
    vel, ang = wl.lin_vel.astype(np.float64), wl.ang_vel.astype(np.float64)
    pl, pa = wl.prev_lin.astype(np.float64), wl.prev_ang.astype(np.float64)
    acc, aacc = (vel - pl) / wl.dt, (ang - pa) / wl.dt
    F, T, comp = _emul_step(inertia_emul, mode, True, slope, pos, wl.quat_xyzw, vel, ang, acc, aacc,
                            wl.coeff_per_body(), wl.rho, wl.g, sl, af)
    ref = IR.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vel, ang, pl, pa, wl.dt,
                  slope=sl if slope else None, fluid_accel=af)
    share = IR.inertia_magnitude(wl.ctor_rows(), ref.sub_ratio, af) / np.maximum(np.linalg.norm(ref.force, axis=1), 1e-9)
    assert (share > 0.1).mean() > 0.2
    if mode == 1:
        assert comp[:, 1].sum() > 0
        scoring.assert_fp32(F, ref.force, "inertia fp32 force")
        scoring.assert_fp32(T, ref.torque, "inertia fp32 torque")
    else:
        scale = scoring.force_scale(wl.coeff_per_body(), wl.rho, wl.g)
        assert scoring.fp64_ok(F, ref.force, scale).all()
        assert scoring.fp64_ok(T, ref.torque, scale).all()


@pytest.mark.parametrize("mode", [0, 1], ids=["fp64", "fp32_fast"])
def test_host_model_with_inertia_dense_matches_reference(inertia_emul, mode):
    """Dense added mass on the relative acceleration: M [R^T (a - a_f); R^T alpha]."""
    wl = W.heterogeneous_boxes(40000, seed=24, xy_range=150.0)
    rng = np.random.default_rng(6)
    pos = _wet_random(wl, rng)
    pos[:, 0:2] = 0.0
    M, slots = _dense(rng)
    D = M[slots[np.arange(wl.n) % len(slots)]]
    af = rng.uniform(-3.0, 3.0, (wl.n, 3))
    vel, ang = wl.lin_vel.astype(np.float64), wl.ang_vel.astype(np.float64)
    pl, pa = wl.prev_lin.astype(np.float64), wl.prev_ang.astype(np.float64)
    acc, aacc = (vel - pl) / wl.dt, (ang - pa) / wl.dt
    F, T, comp = _emul_step(inertia_emul, mode, True, False, pos, wl.quat_xyzw, vel, ang, acc, aacc,
                            wl.coeff_per_body(), wl.rho, wl.g, np.zeros((wl.n, 2)), af, D)
    ref = IR.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vel, ang, pl, pa, wl.dt, fluid_accel=af, dense=M,
                  dense_slot=slots)
    if mode == 1:
        scoring.assert_fp32(F, ref.force, "inertia dense fp32 force")
        scoring.assert_fp32(T, ref.torque, "inertia dense fp32 torque")
    else:
        scale = scoring.force_scale(wl.coeff_per_body(), wl.rho, wl.g)
        assert scoring.fp64_ok(F, ref.force, scale).all()
        assert scoring.fp64_ok(T, ref.torque, scale).all()


def test_flag_margin_with_inertia(inertia_emul):
    """The conditioning check with the inertia group counted (tests/harness/flag_study.py's criterion): no unflagged
    fp32 body comes closer than 0.65x to the fp32 bound, with a_f up to 2 g and drag-cancelling a_f included."""
    wl = W.heterogeneous_boxes(200000, seed=25, xy_range=150.0)
    rng = np.random.default_rng(7)
    pos = _wet_random(wl, rng)
    pos[:, 0:2] = 0.0
    coeff, v, w, a, b = _random_bodies(rng, wl.n, f32=True)
    af = rng.uniform(-20.0, 20.0, (wl.n, 3)) * rng.uniform(0, 1, (wl.n, 1)) ** 2
    F, T, comp = _emul_step(inertia_emul, 1, True, False, pos, wl.quat_xyzw, v, w, a, b, coeff, 1025.0, 9.81,
                            np.zeros((wl.n, 2)), af)
    ctor = np.concatenate([coeff[:, 0:7], np.full((wl.n, 1), 1025.0), np.full((wl.n, 1), 9.81), coeff[:, 7:10]], axis=1)
    ctor = ctor[:, [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11]]
    ref = IR.step(ctor, coeff[:, 10], pos, wl.quat_xyzw, v, w, v - a * wl.dt, w - b * wl.dt, wl.dt, fluid_accel=af)
    ok = comp[:, 1] == 0
    for x, y in ((F, ref.force), (T, ref.torque)):
        err, den = scoring.vec_err(x[ok], y[ok])
        worst = float((err / np.maximum(scoring.FP32_REL * den, scoring.FP32_ABS)).max())
        assert worst < 0.65, worst
    assert 0 < comp[:, 1].mean() < 0.02


@pytest.mark.parametrize("mode", [0, 1], ids=["fp64", "fp32_fast"])
def test_morison_identity(inertia_emul, mode):
    """A fully submerged body moving with the water (v = u, a_b = a_f, no rotation): drag and lift vanish and the
    added-mass terms cancel, so the net force is buoyancy plus rho V a_f, and the torque is zero."""
    rng = np.random.default_rng(8)
    n = 5000
    coeff, _, _, _, _ = _random_bodies(rng, n, f32=mode == 1)
    coeff[:, 10] = 1e9  # no clamp
    dims = coeff[:, 0:3]
    pos = np.zeros((n, 3))
    pos[:, 2] = -2.0 * dims.max(axis=1) - 0.1
    q = np.tile([0.0, 0.0, 0.0, 1.0], (n, 1)) if mode == 1 else W._unit_quats(rng, n, np.float64)
    af = rng.uniform(-3.0, 3.0, (n, 3))
    if mode == 1:
        af = af.astype(np.float32).astype(np.float64)
    z = np.zeros((n, 3))
    F, T, _ = _emul_step(inertia_emul, mode, True, False, pos, q, z, z, af, z, coeff, 1025.0, 9.81,
                         np.zeros((n, 2)), af)
    vol = dims.prod(axis=1)
    want = 1025.0 * vol[:, None] * af
    want[:, 2] += 1025.0 * vol * 9.81
    rel = 1e-6 if mode == 1 else 1e-13
    assert np.abs(F - want).max(axis=1).max() <= rel * np.abs(want).max()
    assert np.abs(T).max() <= rel * np.abs(want).max() * dims.max()


def test_bad_handle_is_refused():
    """h2o_set_fluid_inertia / h2o_fluid_accel_sample on a NULL handle (no device needed)."""
    from silver2_isaacsim_b200 import _lib as L

    lib = L.load()
    assert lib.h2o_set_fluid_inertia(None, 1) == 1
    assert lib.h2o_fluid_accel_sample(None, None, None, 0, None, None) == 1


# --------------------------------------------------------------------------- GPU
torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu
DTYPES = pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda:0")


def _t(a, dtype, dev):
    return torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dtype).contiguous()


def _bits(t):
    t = t.contiguous()
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int64)


def _engine(wl, dtype, dev, kernel="auto", stats=False):
    from silver2_isaacsim_b200 import HydroEngine

    e = HydroEngine(wl.n, dtype=dtype, device=dev)
    e.set_workload_params(wl)
    e.set_kernel(kernel)
    e.enable_stats(stats)
    return e


@gpu
@DTYPES
def test_sampler_matches_reference(dev, dtype):
    """sample_fluid_accel: zeros with the mode off or still water; waves, grid and env rows against NumPy; NaN rows
    for bad env indices; argument errors as the other samplers."""
    from silver2_isaacsim_b200 import HydroEngine
    from silver2_isaacsim_b200 import _lib as L

    field = FIELDS["jonswap64_h12"]()
    f32 = dtype == torch.float32
    rng = np.random.default_rng(9)
    m = 100_000
    e = HydroEngine(40, dtype=dtype, device=dev)
    p = np.stack([rng.uniform(-150, 150, m), rng.uniform(-150, 150, m), rng.uniform(-5, 2, m)], axis=1)
    p = p.astype(np.float32 if f32 else np.float64).astype(np.float64)
    pt = _t(p, dtype, dev)
    e.set_fluid_inertia(True)
    assert e.fluid_inertia
    assert not e.sample_fluid_accel(pt).any()                              # still water
    e.set_wave_field(field)
    grid = _grid(rng)
    gt = torch.as_tensor(grid.values, device=dev)
    e.set_current_grid(gt, origin=grid.origin, spacing=grid.spacing, t0=grid.t0, frame_dt=grid.frame_dt)
    e.set_fluid_inertia(False)
    assert not e.sample_fluid_accel(pt).any()                              # mode off
    e.set_fluid_inertia(True)
    tol = (2e-6 if f32 else 64 * EPS) * _aw2(field) + 64 * EPS
    cond = _cond(rng, 10, tau=8.0)
    ct = torch.as_tensor(cond, device=dev)
    for t in (1231.0, 1234.5, 99999.37):
        e.set_wave_time(t)
        got = e.sample_fluid_accel(pt)
        assert got.dtype == torch.float64 and tuple(got.shape) == (m, 3)
        want = waves.acceleration(field, p, t) + currents.time_derivative(grid, p[:, 0], p[:, 1], p[:, 2], t)
        assert np.abs(got.cpu().numpy() - want).max() <= tol, t
        with pytest.raises(L.H2OError):
            e.sample_fluid_accel(pt, env=0)                                # env rows without conditions
        e.set_env_conditions(ct, 4)
        env = rng.integers(-2, 12, m)
        got = e.sample_fluid_accel(pt, env=env).cpu().numpy()
        bad = (env < 0) | (env >= 10)
        assert np.isnan(got[bad]).all() and np.isfinite(got[~bad]).all()
        r, q = cond[env[~bad]], p[~bad]
        want = (currents.time_derivative(grid, q[:, 0] - r[:, 6], q[:, 1] - r[:, 7], q[:, 2] - r[:, 3], t + r[:, 5]) +
                waves.acceleration_env(field, q, t, cond, env[~bad]))
        assert np.abs(got[~bad] - want).max() <= 2.0 * tol, t
        e.set_env_conditions(None)
    with pytest.raises(ValueError):
        e.sample_fluid_accel(np.zeros((4, 2)))
    out = torch.empty(4, 3, dtype=torch.float64, device=dev)
    assert e._lib.h2o_fluid_accel_sample(e._h, None, None, 4, ctypes.c_void_p(out.data_ptr()), None) == 2
    assert e._lib.h2o_fluid_accel_sample(e._h, None, None, -1, None, None) == 2
    assert e._lib.h2o_fluid_accel_sample(e._h, None, None, 0, None, None) == 0


@gpu
def test_warp_compat_is_refused_in_either_order(dev):
    from silver2_isaacsim_b200 import _lib as L

    wl = W.uniform_small_batch(256)
    e = _engine(wl, torch.float32, dev)
    e.set_fluid_inertia(True)
    with pytest.raises(L.H2OError, match="Warp"):
        e.set_warp_compat(True)
    e.set_fluid_inertia(False)
    e.set_warp_compat(True)
    with pytest.raises(L.H2OError, match="Warp"):
        e.set_fluid_inertia(True)
    assert not e.fluid_inertia
    e.set_warp_compat(False)
    e.set_fluid_inertia(True)


def _wave_workload(n=200_000, seed=2026):
    wl = W.heterogeneous_boxes(n, seed=seed, xy_range=150.0)
    rng = np.random.default_rng(seed + 1)
    wl.pos[:, 2] = rng.uniform(-3.0, 2.0, n).astype(np.float32)
    wl.bodies_per_robot = 4
    return wl


def _centred(pos):
    p = np.array(pos, dtype=np.float64)
    p[:, 0:2] = 0.0
    return p


def _oracle_inputs(wl, dtype, water):
    pos = _centred(wl.pos)
    pos[:, 2] = pos[:, 2] - water[:, 0]
    flow = water[:, 1:]
    if dtype == torch.float32:
        vrel = (wl.lin_vel - flow.astype(np.float32)).astype(np.float64)
        prel = (wl.prev_lin.astype(np.float64) - wl.lin_vel.astype(np.float64)) + vrel
    else:
        vrel = wl.lin_vel.astype(np.float64) - flow
        prel = wl.prev_lin.astype(np.float64) - flow
    return pos, vrel, prel


def _check(wl, pos_ref, dtype, ref, F, T, what):
    if dtype == torch.float32:
        scoring.assert_fp32(F, ref.force, what + " force")
        scoring.assert_fp32(T, ref.torque, what + " torque")
    else:
        scale = scoring.force_scale(wl.coeff_per_body(), wl.rho, wl.g)
        assert scoring.fp64_ok(F, ref.force, scale).all(), what
        pn = np.abs(pos_ref).max(axis=1) * np.abs(ref.force).max(axis=1)
        assert scoring.fp64_ok(T, ref.torque, scale, extra=pn).all(), what


def _sea_engine(wl, dtype, dev, slope, envs=True, keep=None):
    """A finite-depth JONSWAP sea with a current, env rows and a two-frame grid, the mode on; returns the engine and
    what a step forms (waterline + flow, slope, a_f) at each body."""
    rng = np.random.default_rng(10)
    field = waves.jonswap(2.0, 6.0, n_components=16, direction=0.5, seed=9, depth=40.0)
    cur = np.array([0.3, -0.2, 0.05]).astype(np.float32).astype(np.float64)
    e = _engine(wl, dtype, dev, "auto", stats=True)
    e.set_environment(current=cur, surface_z=0.15)
    e.set_wave_field(field)
    e.set_wave_time(1234.5)
    e.set_wave_slope(slope)
    e.set_fluid_inertia(True)
    keep = [] if keep is None else keep
    grid = _grid(rng)
    keep.append(torch.as_tensor(grid.values, device=dev))
    e.set_current_grid(keep[-1], origin=grid.origin, spacing=grid.spacing, t0=grid.t0, frame_dt=grid.frame_dt)
    env = None
    if envs:
        n_envs = wl.n // 4
        keep.append(torch.as_tensor(_cond(rng, n_envs, tau=4.0), device=dev))
        e.set_env_conditions(keep[-1], 4)
        env = torch.arange(wl.n, device=dev) // 4
    pts = _t(wl.pos, dtype, dev)
    water = e.sample_water(pts, env).cpu().numpy()
    sl = e.sample_surface_slope(pts, env).cpu().numpy()
    af = e.sample_fluid_accel(pts, env).cpu().numpy()
    return e, water, sl, af, keep


@gpu
@DTYPES
@pytest.mark.parametrize("slope", [False, True], ids=["flat", "slope"])
@pytest.mark.parametrize("layout", ["split", "view"])
def test_step_with_inertia_matches_reference(dev, dtype, layout, slope):
    """Strict parity: 2e5 boxes in a finite-depth JONSWAP sea with a current, env rows and a two-frame grid, the
    float64 reference fed the waterline, flow, slope and a_f the kernel forms (sample_water, sample_surface_slope,
    sample_fluid_accel at the same clock); per-robot wrench; the new group is a material share of |F|."""
    wl = _wave_workload()
    e, water, sl, af, keep = _sea_engine(wl, dtype, dev, slope)
    assert np.abs(af).max() > 0.5
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    if layout == "split":
        F, T, Wr = e.step(_t(wl.pos, dtype, dev), _t(wl.quat_xyzw, dtype, dev), _t(wl.lin_vel, dtype, dev),
                          _t(wl.ang_vel, dtype, dev), wl.dt, robot_wrench=True)
    else:
        F, T, Wr = e.step_view(_t(wl.pos, dtype, dev), _t(wl.quat_xyzw, dtype, dev), _t(wl.velocities(), dtype, dev),
                               wl.dt, robot_wrench=True)
    F, T, Wr = (x.double().cpu().numpy() for x in (F, T, Wr))
    assert e.last_kernel == "direct"
    if dtype == torch.float32:
        assert e.stats()["reevaluated_bodies"] > 0
    pos, vrel, prel = _oracle_inputs(wl, dtype, water)
    ref = IR.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vrel, wl.ang_vel, prel, wl.prev_ang, wl.dt,
                  slope=sl if slope else None, fluid_accel=af)
    _check(wl, pos, dtype, ref, F, T, f"inertia {layout}")
    wet = ref.sub_ratio > 0
    share = IR.inertia_magnitude(wl.ctor_rows(), ref.sub_ratio, af) / np.maximum(np.linalg.norm(ref.force, axis=1), 1e-9)
    assert (share[wet] > 0.03).mean() > 0.2
    from oracle import hydro_oracle as O

    want = O.robot_wrench(wl.pos.astype(np.float64), ref.force, ref.torque, 4)
    F4 = np.abs(ref.force).reshape(-1, 4, 3).sum(axis=(1, 2)) + np.abs(ref.torque).reshape(-1, 4, 3).sum(axis=(1, 2))
    lever = np.abs(wl.pos.astype(np.float64)).reshape(-1, 12).max(axis=1) * np.abs(ref.force).reshape(-1, 12).max(axis=1)
    rel = 2e-4 if dtype == torch.float32 else 1e-10
    assert (np.abs(Wr - want).max(axis=1) <= rel * (F4 + lever) + 1e-6).all()


@gpu
@DTYPES
def test_step_with_inertia_dense_matches_reference(dev, dtype):
    wl = _wave_workload(40_000, seed=31)
    wl.bodies_per_robot = 0
    e, water, sl, af, keep = _sea_engine(wl, dtype, dev, False, envs=False)
    rng = np.random.default_rng(8)
    M, slots = _dense(rng)
    e.set_added_mass_dense(M, slots)
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    F, T = e.step(_t(wl.pos, dtype, dev), _t(wl.quat_xyzw, dtype, dev), _t(wl.lin_vel, dtype, dev),
                  _t(wl.ang_vel, dtype, dev), wl.dt)
    F, T = F.double().cpu().numpy(), T.double().cpu().numpy()
    pos, vrel, prel = _oracle_inputs(wl, dtype, water)
    ref = IR.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vrel, wl.ang_vel, prel, wl.prev_ang, wl.dt,
                  fluid_accel=af, dense=M, dense_slot=slots)
    _check(wl, pos, dtype, ref, F, T, "inertia dense")


def _run_paths(dev, dtype, setup, paths=("eager", "bound", "graph", "host", "persistent")):
    wl = W.heterogeneous_boxes(6000, seed=41, xy_range=60.0)
    wl.pos[:, 2] = np.random.default_rng(42).uniform(-2.0, 1.0, wl.n).astype(np.float32)
    S = np.float32 if dtype == torch.float32 else np.float64
    out = {}
    for path in paths:
        e = _engine(wl, dtype, dev)
        keep = setup(e)
        e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
        ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
        if path == "eager":
            res = list(e.step(*ten, wl.dt)) + [e.step(*ten, wl.dt)[0]]
        elif path == "host":
            host = [np.ascontiguousarray(a, dtype=S) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
            F, T = e.step_host(*host, wl.dt)
            F2, _ = e.step_host(*host, wl.dt)
            res = [torch.as_tensor(F), torch.as_tensor(T), torch.as_tensor(F2)]
        elif path in ("bound", "graph"):
            F, T = e.bind(*ten)
            if path == "bound":
                e.step_bound(wl.dt)
                res = [F.clone(), T.clone()]
                e.step_bound(wl.dt)
            else:
                e.capture_rollout(1, wl.dt)
                e.launch_rollout()
                torch.cuda.synchronize()
                res = [F.clone(), T.clone()]
                e.launch_rollout()
            res.append(F.clone())
        else:
            F, T = e.bind(*ten)
            e.rollout_persistent(3, wl.dt, gravity=wl.g)
            res = ten + [F, T]
        torch.cuda.synchronize()
        out[path] = [r.cpu() for r in res] + [e.prev_velocities().cpu()]
        del keep
    return out


@gpu
@DTYPES
def test_opt_in_is_inert(dev, dtype):
    """Mode on with still water (a constant current, a one-frame grid) is bit-identical to mode off on every path,
    signed zeros included; with waves the mode changes the wrench."""
    rng = np.random.default_rng(12)
    grid1 = _grid(rng, nt=1)

    def setup(inertia, field=None):
        def s(e):
            e.set_environment(current=(0.2, -0.1, 0.0))
            g = torch.as_tensor(grid1.values, device=e.device)
            e.set_current_grid(g, origin=grid1.origin, spacing=grid1.spacing)
            if field is not None:
                e.set_wave_field(field)
            if inertia is not None:
                e.set_fluid_inertia(inertia)
            return g
        return s

    ra, rb = _run_paths(dev, dtype, setup(None)), _run_paths(dev, dtype, setup(True))
    for path in ra:
        for x, y in zip(ra[path], rb[path]):
            assert torch.equal(_bits(x), _bits(y)), path
    field = waves.regular(0.5, 5.0)
    ra = _run_paths(dev, dtype, setup(False, field), paths=("eager",))
    rb = _run_paths(dev, dtype, setup(True, field), paths=("eager",))
    assert not torch.equal(ra["eager"][0], rb["eager"][0])


@gpu
@DTYPES
def test_paths_agree(dev, dtype):
    """Eager, bound, captured graph and host-buffer steps with the mode on agree bit for bit (one kernel)."""
    rng = np.random.default_rng(13)
    grid = _grid(rng, t0=-5.0, ht=20.0)

    def setup(e):
        e.set_environment(current=(0.2, -0.1, 0.0))
        e.set_wave_field(waves.jonswap(1.5, 7.0, n_components=16, direction=0.4, seed=3))
        g = torch.as_tensor(grid.values, device=e.device)
        e.set_current_grid(g, origin=grid.origin, spacing=grid.spacing, t0=grid.t0, frame_dt=grid.frame_dt)
        e.set_fluid_inertia(True)
        return g

    r = _run_paths(dev, dtype, setup, paths=("eager", "bound", "graph", "host"))
    for path in ("bound", "graph", "host"):
        for x, y in zip(r["eager"][:3], r[path][:3]):
            assert torch.equal(_bits(x), _bits(y)), path
        assert torch.equal(_bits(r["eager"][-1]), _bits(r[path][-1])), path


def _inertia_rollout_engine(wl, dtype, dev, envs, keep):
    e = _engine(wl, dtype, dev)
    e.set_wave_field(waves.jonswap(1.5, 7.0, n_components=16, direction=0.4, seed=3))
    e.set_fluid_inertia(True)
    rng = np.random.default_rng(14)
    grid = _grid(rng, t0=-1.0, ht=2.0)
    keep.append(torch.as_tensor(grid.values, device=dev))
    e.set_current_grid(keep[-1], origin=grid.origin, spacing=grid.spacing, t0=grid.t0, frame_dt=grid.frame_dt)
    if envs:
        keep.append(torch.as_tensor(_cond(rng, wl.n // 4, tau=0.5), device=dev))
        e.set_env_conditions(keep[-1], 4)
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    F, T = e.bind(*ten)
    return e, ten, F, T


@gpu
@DTYPES
@pytest.mark.parametrize("envs", [False, True], ids=["global", "envs"])
def test_persistent_rollout_k_steps_equal_single_steps(dev, dtype, envs):
    """K inertia steps in one launch == K one-step launches, bit for bit, trace rows and clock included; an env reset
    with restart_waves restarts the env's sea (and its a_f) without breaking that."""
    wl = W.heterogeneous_boxes(3000, seed=51, xy_range=60.0)
    wl.pos[:, 2] = np.random.default_rng(52).uniform(-2.0, 1.0, wl.n).astype(np.float32)
    K, res = 20, []
    for plan in ([(K, 1)], [(1, 1)] * K):
        keep = []
        e, ten, F, T = _inertia_rollout_engine(wl, dtype, dev, envs, keep)
        traces = [e.rollout_persistent(s, wl.dt, gravity=wl.g, trace_every=te) for s, te in plan]
        if envs:
            e.reset_envs(torch.arange(wl.n // 4, device=dev) % 3 == 0, restart_waves=True)
            traces += [e.rollout_persistent(s, wl.dt, gravity=wl.g, trace_every=te) for s, te in plan[:2]]
        torch.cuda.synchronize()
        res.append(([t.cpu() for t in ten + [F, T, e.prev_velocities()]], torch.cat([t.cpu() for t in traces]),
                    e.wave_time))
    (a, ta, ca), (b, tb, cb) = res
    if envs:  # after the reset: one K-launch against two 1-step launches; compare the first K steps only
        ta, tb = ta[:K], tb[:K]
    else:
        for name, x, y in zip(("pos", "quat", "lin_vel", "ang_vel", "force", "torque", "prev"), a, b):
            assert torch.equal(_bits(x), _bits(y)), name
        assert ca == cb
    assert torch.equal(_bits(ta), _bits(tb))


@gpu
@DTYPES
def test_graph_rollout_equals_eager(dev, dtype):
    """Graph rollout in free-body mode with the mode on == eager step_bound + integrate_free_bodies, bit for bit."""
    wl = W.heterogeneous_boxes(3000, seed=61, xy_range=60.0)
    wl.pos[:, 2] = np.random.default_rng(62).uniform(-2.0, 1.0, wl.n).astype(np.float32)
    K, res = 5, []
    for mode in ("eager", "graph"):
        keep = []
        e, ten, F, T = _inertia_rollout_engine(wl, dtype, dev, True, keep)
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
        res.append([t.cpu() for t in ten + [F, T, e.prev_velocities()]] + [torch.tensor(e.wave_time)])
    for name, x, y in zip(("pos", "quat", "lin_vel", "ang_vel", "force", "torque", "prev", "clock"), *res):
        assert torch.equal(_bits(x), _bits(y)), name


@gpu
def test_persistent_rollout_tracks_float64_reference(dev):
    """The README buoy in a regular wave, 200 persistent fp64 steps with the mode on, against a float64 rollout of the
    reference step with a_f (waves.evaluate / waves.acceleration at each step) and free_body.integrate: the C1 bounds
    (1e-11 after 100 steps, 1e-9 after 200)."""
    from oracle import free_body
    from silver2_isaacsim_b200 import HydroEngine

    wl = W.readme_buoy()
    ctor = P.HydroParams().ctor_row()
    mass = float(wl.table[0, 10])
    field = waves.regular(0.25, 4.0, direction=0.3, phase=0.4)
    dt, steps, t0 = wl.dt, 200, 3.0
    p, q, v, w = (np.array(a[0], dtype=np.float64) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel))
    p[2] = 0.1
    pv, pw = np.zeros(3), np.zeros(3)
    t = t0
    ref_pos = []
    for k in range(steps):
        smp = waves.evaluate(field, p[None], t)[0]
        rel = p.copy()
        rel[2] = p[2] - smp[0]
        flow = smp[1:]
        r = IR.step(ctor, [mass], rel[None], q[None], (v - flow)[None], w[None], (pv - flow)[None], pw[None], dt,
                    fluid_accel=waves.acceleration(field, p[None], t))
        pv, pw = v.copy(), w.copy()
        p, q, v, w = free_body.integrate(p, q, v, w, r.force[0], r.torque[0], mass, ctor[0:3], dt, wl.g)
        t = t + dt
        ref_pos.append(p.copy())
    e = HydroEngine(1, dtype=torch.float64, device=dev)
    e.set_params_uniform(ctor, mass)
    e.set_wave_field(field)
    e.set_wave_time(t0)
    e.set_fluid_inertia(True)
    d = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64), device=dev).contiguous()
    start = wl.pos.astype(np.float64).copy()
    start[0, 2] = 0.1
    e.bind(d(start), d(wl.quat_xyzw), d(wl.lin_vel), d(wl.ang_vel))
    trace = e.rollout_persistent(steps, dt, gravity=wl.g, trace_every=100).cpu().numpy()[:, 0]
    drift = {n: float(np.abs(trace[n // 100 - 1, :3] - ref_pos[n - 1]).max()) for n in (100, 200)}
    assert drift[100] < 1e-11 and drift[200] < 1e-9, drift


# The particle-orbit check: a neutrally buoyant 0.2 m cube, 1 m deep, in a deep-water regular wave of steepness
# ka = 0.02 (T = 4 s), started on the water's velocity with the previous velocity the flow one step earlier, no
# linear / angular damping.  The float64 reference rollout (tests/inertia_reference.py + oracle/free_body.py) gives a
# horizontal displacement amplitude of 0.964 a e^{k z0} with the mode on and 0.22 with it off, over four periods.
ORBIT_T, ORBIT_KA, ORBIT_Z0, ORBIT_PERIODS = 4.0, 0.02, -1.0, 4


def _orbit_setup():
    om = 2 * math.pi / ORBIT_T
    k = waves.wavenumber(om)
    field = waves.regular(ORBIT_KA / k, ORBIT_T)
    ctor = P.HydroParams(xDimension=0.2, yDimension=0.2, zDimension=0.2, linearDamping=0.0,
                         angularDamping=0.0).ctor_row()
    return field, ctor, 1025.0 * 0.2 ** 3, om, k


def _amplitude(x, dt, om):
    t = np.arange(1, len(x) + 1) * dt
    A = np.stack([np.ones(len(t)), t, np.cos(om * t), np.sin(om * t)], axis=1)
    c = np.linalg.lstsq(A, x, rcond=None)[0]
    return math.hypot(c[2], c[3])


@gpu
def test_particle_orbit(dev):
    from silver2_isaacsim_b200 import HydroEngine

    field, ctor, mass, om, k = _orbit_setup()
    dt = 1.0 / 60.0
    steps = int(ORBIT_PERIODS * ORBIT_T / dt)
    orbit = ORBIT_KA / k * math.exp(k * ORBIT_Z0)
    p0 = np.array([[0.0, 0.0, ORBIT_Z0]])
    u0 = waves.evaluate(field, p0, 0.0)[:, 1:]
    u_prev = waves.evaluate(field, p0, -dt)[:, 1:]
    amp = {}
    for inertia in (True, False):
        e = HydroEngine(1, dtype=torch.float64, device=dev)
        e.set_params_uniform(ctor, mass)
        e.set_wave_field(field)
        e.set_fluid_inertia(inertia)
        d = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64), device=dev).contiguous()
        e.bind(d(p0), d([[0.0, 0.0, 0.0, 1.0]]), d(u0), d(np.zeros((1, 3))))
        e.set_prev(d(u_prev), d(np.zeros((1, 3))))
        tr = e.rollout_persistent(steps, dt, gravity=9.81, trace_every=1).cpu().numpy()[:, 0]
        amp[inertia] = _amplitude(tr[:, 0], dt, om) / orbit
    assert 0.93 < amp[True] < 1.0, amp
    assert amp[False] < 0.4, amp


@gpu
def test_setter_drops_a_captured_rollout(dev):
    """set_fluid_inertia drops a captured rollout; a refused call leaves it intact."""
    from silver2_isaacsim_b200 import _lib as L

    wl = W.uniform_small_batch(2048)
    e = _engine(wl, torch.float64, dev)
    e.set_wave_field(waves.regular(0.2, 5.0))
    e.bind(*[_t(a, torch.float64, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)])
    e.capture_rollout(2, wl.dt)
    e.launch_rollout()
    e.set_fluid_inertia(True)
    with pytest.raises(L.H2OError):
        e.launch_rollout()
    e.capture_rollout(2, wl.dt)
    with pytest.raises(L.H2OError):
        e.set_warp_compat(True)                                            # refused: the graph stays
    pts = _t(wl.pos, torch.float64, dev)
    out = torch.empty(wl.n, 3, dtype=torch.float64, device=dev)
    idx = torch.zeros(wl.n, dtype=torch.int32, device=dev)
    rc = e._lib.h2o_fluid_accel_sample(e._h, ctypes.c_void_p(pts.data_ptr()), ctypes.c_void_p(idx.data_ptr()), wl.n,
                                       ctypes.c_void_p(out.data_ptr()), None)
    assert rc == 8                                                         # H2O_ERR_NOT_CONFIGURED: no env conditions
    e.launch_rollout()                                                     # still captured
    torch.cuda.synchronize()
