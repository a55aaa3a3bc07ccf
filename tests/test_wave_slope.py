"""Wave-slope submersion (include/h2o.h, h2o_set_wave_slope): the NumPy reference, the slope evaluator and the model
with the tangent-plane waterline on the host (tests/host_emul/slope_emul.cpp) against NumPy and a float64 reference with
a sloped waterline plane (tests/slope_reference.py, itself checked against the C oracle without slope), and on the GPU
the sampler, the steps, the rollouts and the opt-in."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from silver2_isaacsim_b200 import waves
from silver2_isaacsim_b200 import workloads as W
from tests import scoring
from tests import slope_reference as SR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = np.finfo(np.float64).eps


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="session")
def slope_emul(tmp_path_factory):
    """tests/host_emul/slope_emul.cpp built into a temporary directory, without multiply-add contraction: g++ contracts
    the instantiations with and without the slope differently, which would hide what the zero-slope test checks."""
    so = str(tmp_path_factory.mktemp("slope_emul") / "libh2o_slope_emul.so")
    subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-shared", "-mfma", "-ffp-contract=off", "-fvisibility=hidden",
                    "-o", so, os.path.join(ROOT, "tests", "host_emul", "slope_emul.cpp")], check=True)
    lib = ctypes.CDLL(so)
    lib.emul_slope_sample.restype = ctypes.c_int
    lib.emul_slope_step.restype = ctypes.c_int
    return lib


def _emul_slope(lib, field, points, t, f32, env_index=None, cond=None):
    p = np.ascontiguousarray(points, dtype=np.float64)
    c = np.ascontiguousarray(field.components, dtype=np.float64)
    out = np.zeros((len(p), 2))
    idx = None if env_index is None else np.ascontiguousarray(env_index, dtype=np.int32)
    cd = np.zeros((1, 8)) if cond is None else np.ascontiguousarray(cond, dtype=np.float64)
    rc = lib.emul_slope_sample(int(f32), len(c), _ptr(c), ctypes.c_double(field.depth), ctypes.c_int64(len(p)), _ptr(p),
                               None if idx is None else _ptr(idx), ctypes.c_int64(len(cd)), _ptr(cd), ctypes.c_double(t),
                               ctypes.c_double(0.0), _ptr(out))
    assert rc == 0
    return out


def _emul_step(lib, mode, slope_on, pos, quat, v, w, a, b, coeff, rho, g, slope, warp_compat=False):
    d = lambda x: np.ascontiguousarray(x, dtype=np.float64)
    n = len(pos)
    arrs = [d(x) for x in (pos, quat, v, w, a, b, coeff)]
    sl = d(slope)
    F, T, comp = np.zeros((n, 3)), np.zeros((n, 3)), np.zeros((n, 13))
    rc = lib.emul_slope_step(mode, int(slope_on), int(warp_compat), ctypes.c_int64(n), *[_ptr(x) for x in arrs],
                             ctypes.c_double(rho), ctypes.c_double(g), _ptr(sl), _ptr(F), _ptr(T), _ptr(comp))
    assert rc == 0
    return F, T, comp


FIELDS = {
    "jonswap16_deep": lambda: waves.jonswap(2.0, 7.0, n_components=16, direction=0.4, seed=3),
    "jonswap64_h12": lambda: waves.jonswap(1.5, 9.0, n_components=64, direction=-1.0, seed=5, depth=12.0),
    "mixed_h3": lambda: waves.WaveField(np.concatenate([
        waves.regular(0.3, 5.0, direction=2.0, phase=0.7, depth=3.0).components,
        waves.regular(0.05, 1.3, direction=-2.5, depth=3.0).components,
        waves.regular(0.2, 20.0, phase=-1.0, depth=3.0).components]), 3.0),
}


def _ak(field):
    c = field.components
    return float((c[:, 0] * np.hypot(c[:, 1], c[:, 2])).sum())


def _cond(rng, n_envs):
    return waves.env_conditions(n_envs, current=rng.uniform(-0.5, 0.5, (n_envs, 3)),
                                surface_dz=rng.uniform(-0.3, 0.3, n_envs), wave_scale=rng.uniform(0.0, 2.0, n_envs),
                                time_offset=rng.uniform(0.0, 100.0, n_envs), origin=rng.uniform(-80, 80, (n_envs, 2)))


# --------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", sorted(FIELDS))
def test_slope_is_the_gradient_of_eta(name):
    """waves.slope against central differences of waves.evaluate's eta; slope_env against those of evaluate_env."""
    field = FIELDS[name]()
    rng = np.random.default_rng(1)
    m, h, t = 2000, 1e-4, 321.25
    p = np.stack([rng.uniform(-300, 300, m), rng.uniform(-300, 300, m), rng.uniform(-2, 1, m)], axis=1)
    ex, ey = np.array([h, 0.0, 0.0]), np.array([0.0, h, 0.0])
    fd = np.stack([(waves.evaluate(field, p + ex, t)[:, 0] - waves.evaluate(field, p - ex, t)[:, 0]) / (2 * h),
                   (waves.evaluate(field, p + ey, t)[:, 0] - waves.evaluate(field, p - ey, t)[:, 0]) / (2 * h)], axis=1)
    got = waves.slope(field, p, t)
    assert got.shape == (m, 2)
    assert np.abs(got - fd).max() <= 1e-6 * _ak(field)
    cond = _cond(rng, 7)
    env = rng.integers(0, 7, m)
    fd_env = np.stack([(waves.evaluate_env(field, p + e, t, cond, env)[:, 0] -
                        waves.evaluate_env(field, p - e, t, cond, env)[:, 0]) / (2 * h) for e in (ex, ey)], axis=1)
    got_env = waves.slope_env(field, p, t, cond, env)
    assert np.abs(got_env - fd_env).max() <= 2e-6 * _ak(field)
    # the env variant is the scaled slope at the env-local position and env time
    r = cond[env]
    q = p.copy()
    q[:, 0] -= r[:, waves.COND_X0]
    q[:, 1] -= r[:, waves.COND_Y0]
    assert np.array_equal(got_env, r[:, waves.COND_SCALE:waves.COND_SCALE + 1] *
                          waves.slope(field, q, t + r[:, waves.COND_TAU]))


@pytest.mark.parametrize("f32", [False, True], ids=["fp64", "fp32"])
@pytest.mark.parametrize("name", sorted(FIELDS))
def test_host_slope_evaluator_matches_reference(slope_emul, name, f32):
    """The evaluator the kernels inline (water_at with the slope) against waves.slope / waves.slope_env: fp64 within
    a few ulps of sum a_j k_j, fp32 within 2e-6 of it; a NaN row for an env index outside [0, E)."""
    field = FIELDS[name]()
    rng = np.random.default_rng(2)
    m = 20000
    p = np.stack([rng.uniform(-500, 500, m), rng.uniform(-500, 500, m), rng.uniform(-5, 2, m)], axis=1)
    if f32:
        p = p.astype(np.float32).astype(np.float64)
    tol = (2e-6 if f32 else 16 * EPS) * _ak(field)
    for t in (0.0, 1234.5, 99999.37):
        got = _emul_slope(slope_emul, field, p, t, f32)
        assert np.abs(got - waves.slope(field, p, t)).max() <= tol, t
        cond = _cond(rng, 5)
        env = rng.integers(-1, 6, m)
        got = _emul_slope(slope_emul, field, p, t, f32, env, cond)
        bad = (env < 0) | (env >= 5)
        assert np.isnan(got[bad]).all() and np.isfinite(got[~bad]).all()
        want = waves.slope_env(field, p[~bad], t, cond, env[~bad])
        assert np.abs(got[~bad] - want).max() <= 2.0 * tol, t


def _centred(pos):
    """Body positions for the float64 reference with x = y = 0: its world-form plane test subtracts p from the world
    keypoints, which at |p_xy| = 150 m costs 1e-14 m of cancellation by itself; the model does not depend on p_xy."""
    p = np.array(pos, dtype=np.float64)
    p[:, 0:2] = 0.0
    return p


def _random_bodies(rng, n, f32=False):
    """Random boxes with random state: dims, coefficient records, velocities, accelerations."""
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
        coeff, v, w = (x.astype(np.float32).astype(np.float64) for x in (coeff, v, w))
    return coeff, v, w, a, b


def _quat_between_ez(nhat):
    """xyzw quaternion of the smallest rotation taking e_z to the unit vectors nhat (n, 3)."""
    axis = np.stack([-nhat[:, 1], nhat[:, 0], np.zeros(len(nhat))], axis=1)   # e_z x nhat
    s = np.linalg.norm(axis, axis=1)
    ang = np.arctan2(s, nhat[:, 2])
    u = axis / np.where(s > 0, s, 1.0)[:, None]
    return np.concatenate([u * np.sin(ang / 2)[:, None], np.cos(ang / 2)[:, None]], axis=1)


def test_tilt_invariance_on_host_model(slope_emul):
    """A box rotated by the rotation that takes e_z to the plane normal n, its height scaled by |n|, is the level box on
    a flat surface: same wet mask (bodies with a keypoint on the surface excepted), same ratio and same body-frame
    centre of buoyancy to a few ulps."""
    rng = np.random.default_rng(3)
    n = 20000
    coeff, v, w, a, b = _random_bodies(rng, n)
    dims = coeff[:, 0:3]
    h0 = rng.uniform(-0.7, 0.7, n) * dims[:, 2]
    sl = rng.uniform(-0.6, 0.6, (n, 2))
    nvec = np.stack([-sl[:, 0], -sl[:, 1], np.ones(n)], axis=1)
    nn = np.linalg.norm(nvec, axis=1)
    q_tilt = _quat_between_ez(nvec / nn[:, None])
    q_level = np.tile([0.0, 0.0, 0.0, 1.0], (n, 1))
    pos_level = np.stack([np.zeros(n), np.zeros(n), h0], axis=1)
    pos_tilt = np.stack([np.zeros(n), np.zeros(n), h0 * nn], axis=1)
    _, _, lev = _emul_step(slope_emul, 0, True, pos_level, q_level, v, w, a, b, coeff, 1025.0, 9.81, np.zeros((n, 2)))
    _, _, til = _emul_step(slope_emul, 0, True, pos_tilt, q_tilt, v, w, a, b, coeff, 1025.0, 9.81, sl)
    # keypoint heights of the level box: h0 + {-1, 0, 1} dz / 2; a tie is a keypoint within rounding of the surface
    tie = (np.abs(h0[:, None] + np.array([-0.5, 0.0, 0.5])[None, :] * dims[:, 2:3]) < 1e-12 * dims.max(axis=1)[:, None]).any(axis=1)
    ok = ~tie
    assert ok.mean() > 0.99
    assert np.array_equal(lev[ok, 11], til[ok, 11])
    wet = lev[:, 0] > 0
    assert 0.2 < (wet & (lev[:, 0] < 1)).mean()                          # partially wet bodies are exercised
    assert np.abs(lev[ok, 0] - til[ok, 0]).max() <= 8 * EPS
    # body-frame centre of buoyancy: R^T (cob - p) of the tilted box against the level box's
    x, y, z, s = q_tilt.T
    R = np.stack([np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - s * z), 2 * (x * z + s * y)], -1),
                  np.stack([2 * (x * y + s * z), 1 - 2 * (x * x + z * z), 2 * (y * z - s * x)], -1),
                  np.stack([2 * (x * z - s * y), 2 * (y * z + s * x), 1 - 2 * (x * x + y * y)], -1)], axis=1)
    cob_b = np.einsum("nji,nj->ni", R, til[:, 1:4])
    assert np.abs(cob_b[ok] - lev[ok, 1:4]).max(axis=1).max() <= 16 * EPS * dims.max()


@pytest.mark.parametrize("mode,warp", [(0, False), (0, True), (1, False)], ids=["fp64", "fp64_warp", "fp32_fast"])
def test_zero_slope_is_bit_identical_to_slope_off(slope_emul, mode, warp):
    """The slope instantiation with a zero slope reproduces the one without, bit for bit."""
    wl = W.heterogeneous_boxes(50000, seed=21)
    coeff, v, w, a, b = _random_bodies(np.random.default_rng(4), wl.n, f32=mode == 1)
    pos = wl.pos.astype(np.float64)
    zero = np.zeros((wl.n, 2))
    on = _emul_step(slope_emul, mode, True, pos, wl.quat_xyzw, v, w, a, b, coeff, 1025.0, 9.81, zero, warp)
    off = _emul_step(slope_emul, mode, False, pos, wl.quat_xyzw, v, w, a, b, coeff, 1025.0, 9.81, zero, warp)
    for x, y in zip(on, off):
        assert np.array_equal(x.view(np.int64), y.view(np.int64))


@pytest.mark.parametrize("variant", ["numba", "warp_compat", "dense_added_mass"])
def test_reference_without_slope_is_the_oracle(oracle, variant):
    """tests/slope_reference.py without a slope against the C oracle: the same arithmetic in the same order, so every
    vector agrees to a few float64 ulps of its magnitude (asin / sin / sqrt come from different libraries), and the
    submersion ratio bit for bit."""
    wl = W.heterogeneous_boxes(100000, seed=23, xy_range=150.0)
    rng = np.random.default_rng(6)
    q = wl.quat_xyzw.astype(np.float64) * rng.uniform(0.999, 1.001, (wl.n, 1))   # not unit: R(q) and C7 matter
    M = slots = None
    if variant == "dense_added_mass":
        M = rng.uniform(-20.0, 20.0, (3, 6, 6)) + np.eye(6)[None] * 200.0
        slots = np.array([0, 2, 1, 1], dtype=np.int32)
        oracle.set_added_mass_dense(M, slots)
    oracle.set_warp_compat(variant == "warp_compat")
    try:
        args = (wl.ctor_rows(), wl.masses(), wl.pos, q, wl.lin_vel, wl.ang_vel, wl.prev_lin, wl.prev_ang, wl.dt)
        want = oracle.step(*args)
    finally:
        oracle.set_warp_compat(False)
        oracle.set_added_mass_dense(None)
    got = SR.step(*args, warp_compat=variant == "warp_compat", dense=M, dense_slot=slots)
    assert 0.2 < ((want.components["sub_ratio"] > 0) & (want.components["sub_ratio"] < 1)).mean()
    assert np.array_equal(got.sub_ratio, want.components["sub_ratio"])
    scale = scoring.force_scale(wl.coeff_per_body(), wl.rho, wl.g)
    pn = np.abs(wl.pos.astype(np.float64)).max(axis=1) * np.abs(want.force).max(axis=1)
    assert scoring.fp64_ok(got.force, want.force, scale, rel=1e-14).all()
    assert scoring.fp64_ok(got.torque, want.torque, scale, extra=pn, rel=1e-14).all()


@pytest.mark.parametrize("mode", [0, 1], ids=["fp64", "fp32_fast"])
def test_host_model_with_slope_matches_reference(slope_emul, mode):
    """The host model with the tangent-plane waterline against the float64 reference fed the same slope, under the
    parity bounds of the step tests (fp32: the fast path plus the float64 re-evaluation of flagged bodies)."""
    wl = W.heterogeneous_boxes(100000, seed=22, xy_range=150.0)
    rng = np.random.default_rng(5)
    pos = wl.pos.astype(np.float64)
    sl = rng.uniform(-0.4, 0.4, (wl.n, 2))
    vel, ang = wl.lin_vel.astype(np.float64), wl.ang_vel.astype(np.float64)
    pl, pa = wl.prev_lin.astype(np.float64), wl.prev_ang.astype(np.float64)
    acc, aacc = (vel - pl) / wl.dt, (ang - pa) / wl.dt
    F, T, comp = _emul_step(slope_emul, mode, True, pos, wl.quat_xyzw, vel, ang, acc, aacc, wl.coeff_per_body(), wl.rho,
                            wl.g, sl)
    pos = _centred(pos)
    ref = SR.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vel, ang, pl, pa, wl.dt, slope=sl)
    flat = SR.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vel, ang, pl, pa, wl.dt)
    changed = (ref.sub_ratio != flat.sub_ratio).mean()
    assert changed > 0.1                                                  # the slope does move the waterline
    if mode == 1:
        assert comp[:, 12].sum() > 0                                      # flagged bodies were re-evaluated
        scoring.assert_fp32(F, ref.force, "slope fp32 force")
        scoring.assert_fp32(T, ref.torque, "slope fp32 torque")
    else:
        scale = scoring.force_scale(wl.coeff_per_body(), wl.rho, wl.g)
        assert scoring.fp64_ok(F, ref.force, scale).all()
        pn = np.abs(pos).max(axis=1) * np.abs(ref.force).max(axis=1)
        assert scoring.fp64_ok(T, ref.torque, scale, extra=pn).all()
        assert np.abs(comp[:, 0] - ref.sub_ratio).max() <= 1e-12


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
@pytest.mark.parametrize("name", sorted(FIELDS))
def test_sampler_matches_reference(dev, dtype, name):
    from silver2_isaacsim_b200 import HydroEngine

    field = FIELDS[name]()
    f32 = dtype == torch.float32
    rng = np.random.default_rng(7)
    m = 100_000
    e = HydroEngine(40, dtype=dtype, device=dev)
    p = np.stack([rng.uniform(-500, 500, m), rng.uniform(-500, 500, m), rng.uniform(-5, 2, m)], axis=1)
    p = p.astype(np.float32 if f32 else np.float64).astype(np.float64)
    e.set_wave_slope(True)
    assert e.wave_slope
    assert not e.sample_surface_slope(_t(p, dtype, dev)).any()           # no field: no slope
    e.set_wave_field(field)
    e.set_wave_slope(False)
    assert not e.sample_surface_slope(_t(p, dtype, dev)).any()           # mode off: no slope
    e.set_wave_slope(True)
    tol = (2e-6 if f32 else 16 * EPS) * _ak(field)
    cond = _cond(rng, 10)
    ct = torch.as_tensor(cond, device=dev)
    for t in (0.0, 1234.5, 99999.37):
        e.set_wave_time(t)
        got = e.sample_surface_slope(_t(p, dtype, dev))
        assert got.dtype == torch.float64 and tuple(got.shape) == (m, 2)
        assert np.abs(got.cpu().numpy() - waves.slope(field, p, t)).max() <= tol, t
        with pytest.raises(Exception):
            e.sample_surface_slope(_t(p, dtype, dev), env=0)             # env rows without conditions
        e.set_env_conditions(ct, 4)
        env = rng.integers(-2, 12, m)
        got = e.sample_surface_slope(_t(p, dtype, dev), env=env).cpu().numpy()
        bad = (env < 0) | (env >= 10)
        assert np.isnan(got[bad]).all() and np.isfinite(got[~bad]).all()
        want = waves.slope_env(field, p[~bad], t, cond, env[~bad])
        assert np.abs(got[~bad] - want).max() <= 2.0 * tol, t
        e.set_env_conditions(None)
    with pytest.raises(ValueError):
        e.sample_surface_slope(np.zeros((4, 2)))


def _wave_workload(n=200_000, seed=2026):
    """Heterogeneous boxes over several wavelengths with p_z in [-3, 2] m, as robots of 4 bodies."""
    wl = W.heterogeneous_boxes(n, seed=seed, xy_range=150.0)
    rng = np.random.default_rng(seed + 1)
    wl.pos[:, 2] = rng.uniform(-3.0, 2.0, n).astype(np.float32)
    wl.bodies_per_robot = 4
    return wl


def _oracle_inputs(wl, dtype, water):
    """What the kernel feeds the model: p_z - waterline in float64 (x, y centred, _centred), v - S(flow) formed in S."""
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


def _sea_engine(wl, dtype, dev, **kw):
    field = waves.jonswap(2.0, 6.0, n_components=16, direction=0.5, seed=9, depth=40.0)
    cur = np.array([0.3, -0.2, 0.05]).astype(np.float32).astype(np.float64)
    e = _engine(wl, dtype, dev, "auto", stats=True, **kw)
    e.set_environment(current=cur, surface_z=0.15)
    e.set_wave_field(field)
    e.set_wave_time(1234.5)
    e.set_wave_slope(True)
    pts = _t(wl.pos, dtype, dev)
    return e, e.sample_water(pts).cpu().numpy(), e.sample_surface_slope(pts).cpu().numpy()


@gpu
@DTYPES
@pytest.mark.parametrize("layout", ["split", "view"])
def test_step_with_slope_matches_reference(oracle, dev, dtype, layout):
    """Strict parity: 2e5 boxes cut by a finite-depth JONSWAP sea with a current, the float64 reference (the C oracle's
    arithmetic with a sloped waterline plane, tests/slope_reference.py) fed the waterline, flow and
    slope the kernel forms (sample_water, sample_surface_slope at the same clock); fp32 flagged bodies re-evaluated
    with the slope too; per-robot wrench."""
    wl = _wave_workload()
    e, water, sl = _sea_engine(wl, dtype, dev)
    assert np.abs(sl).max() > 0.2
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
    ref = SR.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vrel, wl.ang_vel, prel, wl.prev_ang, wl.dt, slope=sl)
    _check(wl, pos, dtype, ref, F, T, f"slope {layout}")
    flat = oracle.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vrel, wl.ang_vel, prel, wl.prev_ang, wl.dt)
    assert (ref.sub_ratio != flat.components["sub_ratio"]).mean() > 0.05
    want = oracle.robot_wrench(wl.pos.astype(np.float64), ref.force, ref.torque, 4)
    F4 = np.abs(ref.force).reshape(-1, 4, 3).sum(axis=(1, 2)) + np.abs(ref.torque).reshape(-1, 4, 3).sum(axis=(1, 2))
    lever = np.abs(wl.pos.astype(np.float64)).reshape(-1, 12).max(axis=1) * np.abs(ref.force).reshape(-1, 12).max(axis=1)
    rel = 2e-4 if dtype == torch.float32 else 1e-10
    assert (np.abs(Wr - want).max(axis=1) <= rel * (F4 + lever) + 1e-6).all()


@gpu
@DTYPES
@pytest.mark.parametrize("variant", ["warp_compat", "dense_added_mass"])
def test_step_with_slope_variants_match_reference(dev, dtype, variant):
    """The fused Warp-compat step and dense added mass with the slope, against the float64 reference with the same
    switches."""
    wl = _wave_workload(40_000, seed=31)
    wl.bodies_per_robot = 0
    e, water, sl = _sea_engine(wl, dtype, dev)
    rng = np.random.default_rng(8)
    M = slots = None
    if variant == "warp_compat":
        e.set_warp_compat(True)
    else:
        M = rng.uniform(-20.0, 20.0, (3, 6, 6)) + np.eye(6)[None] * 200.0
        slots = np.array([0, 2, 1, 1], dtype=np.int32)
        e.set_added_mass_dense(M, slots)
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    F, T = e.step(_t(wl.pos, dtype, dev), _t(wl.quat_xyzw, dtype, dev), _t(wl.lin_vel, dtype, dev),
                  _t(wl.ang_vel, dtype, dev), wl.dt)
    F, T = F.double().cpu().numpy(), T.double().cpu().numpy()
    pos, vrel, prel = _oracle_inputs(wl, dtype, water)
    ref = SR.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vrel, wl.ang_vel, prel, wl.prev_ang, wl.dt, slope=sl,
                  warp_compat=variant == "warp_compat", dense=M, dense_slot=slots)
    _check(wl, pos, dtype, ref, F, T, f"slope {variant}")


def _run_paths(dev, dtype, setup, paths=("eager", "bound", "graph", "host", "persistent")):
    """Run one start state through each step path on a fresh handle prepared by setup(e); returns path -> tensors."""
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
    """Without the call, or with the mode on and no wave field, every step path is bit-identical to a handle that never
    heard of the slope; with a field of zero amplitudes, mode on equals mode off bit for bit (the persistent rollout
    runs its own slope instantiation: to rounding there, include/h2o.h)."""
    field = waves.jonswap(1.5, 7.0, n_components=16, direction=0.4, seed=3)
    zero = waves.WaveField(np.concatenate([np.zeros((16, 1)), field.components[:, 1:]], axis=1))

    def with_field(f, slope):
        def setup(e):
            e.set_environment(current=(0.2, -0.1, 0.0))
            if f is not None:
                e.set_wave_field(f)
            if slope is not None:
                e.set_wave_slope(slope)
        return setup

    cases = [(with_field(None, None), with_field(None, True)),          # no field: the mode changes nothing
             (with_field(field, None), with_field(field, False)),       # mode off: as never called
             (with_field(zero, False), with_field(zero, True))]         # zero amplitudes: zero slope
    for k, (a, b) in enumerate(cases):
        ra, rb = _run_paths(dev, dtype, a), _run_paths(dev, dtype, b)
        for path in ra:
            for x, y in zip(ra[path], rb[path]):
                if k == 2 and path == "persistent":
                    assert torch.allclose(x.double(), y.double(), rtol=1e-5 if dtype == torch.float32 else 1e-12,
                                          atol=1e-6 if dtype == torch.float32 else 1e-12), (k, path)
                else:
                    assert torch.equal(_bits(x), _bits(y)), (k, path)


def _rollout_state(dev, dtype, n=3000, seed=51):
    wl = W.heterogeneous_boxes(n, seed=seed, xy_range=60.0)
    wl.pos[:, 2] = np.random.default_rng(seed + 1).uniform(-2.0, 1.0, wl.n).astype(np.float32)
    return wl


def _slope_rollout_engine(wl, dtype, dev, envs):
    e = _engine(wl, dtype, dev)
    e.set_wave_field(waves.jonswap(1.5, 7.0, n_components=16, direction=0.4, seed=3))
    e.set_wave_slope(True)
    keep = None
    if envs:
        keep = torch.as_tensor(_cond(np.random.default_rng(14), wl.n // 4), device=dev)
        e.set_env_conditions(keep, 4)
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    F, T = e.bind(*ten)
    return e, ten, F, T, keep


@gpu
@DTYPES
@pytest.mark.parametrize("envs", [False, True], ids=["global", "envs"])
def test_persistent_rollout_with_slope_k_steps_equal_single_steps(dev, dtype, envs):
    """K steps in one launch == K one-step launches, bit for bit, trace rows included."""
    wl = _rollout_state(dev, dtype)
    K, res = 20, []
    for plan in ([(K, 1)], [(1, 1)] * K):
        e, ten, F, T, keep = _slope_rollout_engine(wl, dtype, dev, envs)
        traces = [e.rollout_persistent(s, wl.dt, gravity=wl.g, trace_every=te) for s, te in plan]
        torch.cuda.synchronize()
        res.append(([t.cpu() for t in ten + [F, T, e.prev_velocities()]], torch.cat([t.cpu() for t in traces]),
                    e.wave_time))
    (a, ta, ca), (b, tb, cb) = res
    for name, x, y in zip(("pos", "quat", "lin_vel", "ang_vel", "force", "torque", "prev"), a, b):
        assert torch.equal(_bits(x), _bits(y)), name
    assert torch.equal(_bits(ta), _bits(tb)) and ca == cb


@gpu
@DTYPES
def test_graph_rollout_with_slope_equals_eager(dev, dtype):
    """Graph rollout in free-body mode with the slope == eager step_bound + integrate_free_bodies, bit for bit."""
    wl = _rollout_state(dev, dtype, seed=61)
    K, res = 5, []
    for mode in ("eager", "graph"):
        e, ten, F, T, keep = _slope_rollout_engine(wl, dtype, dev, True)
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
def test_persistent_rollout_with_slope_tracks_float64_reference(dev):
    """The README buoy released into a regular wave, 200 persistent steps with the slope (fp64), against a float64
    rollout of the reference step with the slope (waves.evaluate / waves.slope at each step) and free_body.integrate: the C1
    bounds (1e-11 after 100 steps, 1e-9 after 200)."""
    from oracle import free_body
    from silver2_isaacsim_b200 import HydroEngine
    from silver2_isaacsim_b200 import params as P

    wl = W.readme_buoy()
    ctor = P.HydroParams().ctor_row()
    mass = float(wl.table[0, 10])
    field = waves.regular(0.25, 4.0, direction=0.3, phase=0.4)
    dt, steps, t0 = wl.dt, 200, 3.0
    p, q, v, w = (np.array(a[0], dtype=np.float64) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel))
    p[2] = 0.1
    pv, pw = np.zeros(3), np.zeros(3)
    t = t0
    ref_pos, tilt = [], 0.0
    for k in range(steps):
        smp = waves.evaluate(field, p[None], t)[0]
        sl = waves.slope(field, p[None], t)
        rel = p.copy()
        rel[2] = p[2] - smp[0]
        flow = smp[1:]
        r = SR.step(ctor, [mass], rel[None], q[None], (v - flow)[None], w[None], (pv - flow)[None], pw[None], dt,
                    slope=sl)
        pv, pw = v.copy(), w.copy()
        p, q, v, w = free_body.integrate(p, q, v, w, r.force[0], r.torque[0], mass, ctor[0:3], dt, wl.g)
        t = t + dt
        ref_pos.append(p.copy())
        tilt = max(tilt, float(np.abs(w).max()))
    assert tilt > 1e-2                                                    # the slope does roll and pitch the buoy
    e = HydroEngine(1, dtype=torch.float64, device=dev)
    e.set_params_uniform(ctor, mass)
    e.set_wave_field(field)
    e.set_wave_time(t0)
    e.set_wave_slope(True)
    d = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64), device=dev).contiguous()
    start = wl.pos.astype(np.float64).copy()
    start[0, 2] = 0.1
    pos = d(start)
    e.bind(pos, d(wl.quat_xyzw), d(wl.lin_vel), d(wl.ang_vel))
    trace = e.rollout_persistent(steps, dt, gravity=wl.g, trace_every=100).cpu().numpy()[:, 0]
    drift = {n: float(np.abs(trace[n // 100 - 1, :3] - ref_pos[n - 1]).max()) for n in (100, 200)}
    assert drift[100] < 1e-11 and drift[200] < 1e-9, drift


@gpu
@DTYPES
def test_mirror_symmetry_of_the_pitch_torque(dev, dtype):
    """A level box where the slope is largest, with buoyancy as the only load: mode off gives the reference's zero
    pitch torque exactly (its wet keypoints are symmetric); mode on a nonzero one; mirroring the scene in x mirrors the
    wrench bit for bit."""
    from silver2_isaacsim_b200 import HydroEngine

    a, period = 0.5, 3.0
    k = waves.wavenumber(2 * math.pi / period)
    # theta = pi/2 at x = 0, t = 0: eta = 0 and sx = -a k (e_x hx = 0.11 m) there; each box has a keypoint layer
    # within 0.11 m of the waterline, so that the tangent plane cuts it differently from the horizontal one
    z = np.array([-0.08, -0.03, 0.02, 0.07, 0.25, 0.32, -0.26, -0.34])
    n = len(z)
    pos = np.stack([np.zeros(n), np.linspace(-3.0, 3.0, n), z], axis=1)
    q = np.tile([0.0, 0.0, 0.0, 1.0], (n, 1))
    zero = np.zeros((n, 3))
    # README box, buoyancy only: no drag, damping, lift or added mass
    ctor = [1.0, 0.8, 0.6, 0.0, 0.0, 0.0, 0.0, 1025.0, 9.81, 0.0, 0.0, 0.0]
    res = {}
    for mirror in (False, True):
        field = waves.WaveField(np.array([[a, -k if mirror else k, 0.0, 2 * math.pi / period, math.pi / 2]]))
        for slope in (False, True):
            e = HydroEngine(n, dtype=dtype, device=dev)
            e.set_params_uniform(ctor, 300.0)
            e.set_wave_field(field)
            e.set_wave_slope(slope)
            F, T = e.step(_t(pos, dtype, dev), _t(q, dtype, dev), _t(zero, dtype, dev), _t(zero, dtype, dev), 1 / 60)
            res[mirror, slope] = (F.double().cpu().numpy(), T.double().cpu().numpy())
    F0, T0 = res[False, False]
    assert (T0[:, 1] == 0).all() and (T0 == 0).all()                      # level box, flat waterline: no torque
    F1, T1 = res[False, True]
    assert (np.abs(T1[:, 1]) > 1e-3 * np.abs(F1[:, 2]).max()).all()      # the tangent plane pitches the box
    Fm, Tm = res[True, True]
    flip = np.array([-1.0, 1.0, 1.0])
    assert np.array_equal(Fm, F1 * flip) and np.array_equal(Tm, T1 * -flip)


@gpu
def test_setter_drops_a_captured_rollout(dev):
    """set_wave_slope drops a captured rollout; a refused call leaves it intact."""
    from silver2_isaacsim_b200 import _lib as L

    wl = W.uniform_small_batch(2048)
    e = _engine(wl, torch.float64, dev)
    e.set_wave_field(waves.regular(0.2, 5.0))
    e.bind(*[_t(a, torch.float64, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)])
    e.capture_rollout(2, wl.dt)
    e.launch_rollout()
    e.set_wave_slope(True)
    with pytest.raises(L.H2OError):
        e.launch_rollout()
    e.capture_rollout(2, wl.dt)
    pts = _t(wl.pos, torch.float64, dev)
    out = torch.empty(wl.n, 2, dtype=torch.float64, device=dev)
    idx = torch.zeros(wl.n, dtype=torch.int32, device=dev)
    rc = e._lib.h2o_water_slope_sample(e._h, ctypes.c_void_p(pts.data_ptr()), ctypes.c_void_p(idx.data_ptr()), wl.n,
                                       ctypes.c_void_p(out.data_ptr()), None)
    assert rc == 8                                                        # H2O_ERR_NOT_CONFIGURED: no env conditions
    assert e._lib.h2o_set_wave_slope(None, 1) == 1                        # H2O_ERR_BAD_HANDLE
    e.launch_rollout()                                                    # still captured
    torch.cuda.synchronize()
