"""Gridded water currents (include/h2o.h, h2o_set_current_grid / h2o_water_sample): the NumPy module, the evaluator
and the composition of csrc/h2o_waves.cuh (grid_eval, water_at) on the host, and on the GPU the sampler, the step,
the rollouts, the clock, env behaviour, a seabed boundary layer and input validation."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from silver2_isaacsim_b200 import currents, waves
from silver2_isaacsim_b200 import workloads as W
from tests import scoring
from tests.test_env_conditions import _cond_t, _identity_workload, _random_cond, _run_path, _same_bits
from tests.test_waves import FIELDS, _check, _engine, _t, _wave_workload

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def current_emul(tmp_path_factory):
    """tests/host_emul/current_emul.cpp (grid_eval and water_at instantiated for the host), built into a temporary
    directory with the flags of the other emulators."""
    so = str(tmp_path_factory.mktemp("current_emul") / "libh2o_current_emul.so")
    subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-shared", "-mfma", "-ffp-contract=fast", "-fvisibility=hidden",
                    "-o", so, os.path.join(ROOT, "tests", "host_emul", "current_emul.cpp")], check=True)
    lib = ctypes.CDLL(so)
    lib.emul_current_eval.restype = ctypes.c_int
    lib.emul_water.restype = ctypes.c_int
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _dims(grid):
    return np.ascontiguousarray(grid.dims, dtype=np.int64)


def _emul_eval(lib, grid, x, y, z, t):
    q = [np.ascontiguousarray(np.broadcast_to(np.asarray(a, dtype=np.float64), np.shape(x))) for a in (x, y, z, t)]
    out = np.zeros((len(q[0]), 3))
    dims, geom = _dims(grid), grid.geometry
    assert lib.emul_current_eval(_ptr(dims), _ptr(grid.values), _ptr(geom), ctypes.c_int64(len(out)),
                                 *[_ptr(a) for a in q], _ptr(out)) == 0
    return out


def _emul_water(lib, points, t, f32, grid=None, field=None, cond=None, env=None, surface_z=0.0, current=(0, 0, 0)):
    p = np.ascontiguousarray(points, dtype=np.float64)
    comps = np.ascontiguousarray(field.components if field else np.zeros((0, 5)), dtype=np.float64)
    idx = None if env is None else np.ascontiguousarray(env, dtype=np.int32)
    cnd = None if cond is None else np.ascontiguousarray(cond, dtype=np.float64)
    cur = np.ascontiguousarray(current, dtype=np.float64)
    fld, water = np.zeros((len(p), 4)), np.zeros((len(p), 4))
    dims, vals, geom = (None, None, None) if grid is None else (_dims(grid), grid.values, grid.geometry)
    rc = lib.emul_water(int(f32), len(comps), _ptr(comps), ctypes.c_double(field.depth if field else math.inf),
                        _ptr(dims), _ptr(vals), _ptr(geom), ctypes.c_int64(len(p)), _ptr(p), _ptr(idx),
                        ctypes.c_int64(0 if cnd is None else len(cnd)), _ptr(cnd), ctypes.c_double(t),
                        ctypes.c_double(surface_z), _ptr(cur), _ptr(fld), _ptr(water))
    assert rc == 0
    return fld, water


def compose(grid, points, t, surface_z, current, cond=None, env=None, field=None):
    """The NumPy composition of include/h2o.h: rows [waterline, flow] from the env rows, the grid (currents.evaluate)
    and the sea's contribution ``field`` ((m,4) [s eta, s u] of the same points, or None without a sea)."""
    p = np.asarray(points, dtype=np.float64)
    cur = np.broadcast_to(np.asarray(current, dtype=np.float64), (len(p), 3))
    level, flow = np.full(len(p), float(surface_z)), cur.copy()
    x, y, tt = p[:, 0], p[:, 1], np.full(len(p), float(t))
    if env is not None:
        r = np.asarray(cond)[np.asarray(env)]
        level = level + r[:, waves.COND_DZ]
        flow = cur + r[:, waves.COND_CX:waves.COND_CZ + 1]
        x, y, tt = x - r[:, waves.COND_X0], y - r[:, waves.COND_Y0], tt + r[:, waves.COND_TAU]
    if grid is not None:
        flow = flow + currents.evaluate(grid, x, y, p[:, 2] - level, tt)
    out = np.empty((len(p), 4))
    out[:, 0], out[:, 1:] = level, flow
    if field is not None:
        out[:, 0], out[:, 1:] = level + field[:, 0], flow + field[:, 1:]
    return out


def _random_grid(rng, dims, origin=(-100.0, -80.0, -4.0), spacing=(25.0, 30.0, 0.8), t0=1230.0, frame_dt=10.0, c=0.6):
    return currents.CurrentGrid(rng.uniform(-c, c, (*dims, 3)), origin=origin, spacing=spacing, t0=t0,
                                frame_dt=frame_dt if dims[0] > 1 else 0.0)


def _grid_points(rng, m, f32=False):
    """Inside and outside the lattice of _random_grid on every side (x in [-100, 75], y in [-80, 100], z in [-4, 0])."""
    p = np.stack([rng.uniform(-160, 140, m), rng.uniform(-130, 150, m), rng.uniform(-6.0, 2.0, m)], axis=1)
    return p.astype(np.float32).astype(np.float64) if f32 else p


SHAPES = {"3d_2frames": (2, 6, 7, 8), "profile": (1, 32, 1, 1), "one_node": (1, 1, 1, 1),
          "xt_only": (3, 1, 1, 5), "yz_4frames": (4, 5, 6, 1)}


# --------------------------------------------------------------------------- CPU: currents.py
def test_builders_and_validation():
    g = currents.CurrentGrid(np.zeros((2, 3, 4, 3)), origin=(1, 2, 3), spacing=(0.5, 1, 2))
    assert g.dims == (1, 2, 3, 4) and g.values.shape == (1, 2, 3, 4, 3) and not g.values.flags.writeable
    assert (g.geometry == [1, 2, 3, 0.5, 1, 2, 0, 0]).all()
    g = currents.CurrentGrid(np.zeros((2, 1, 1, 1, 3)), t0=5.0, frame_dt=2.0)
    assert g.dims == (2, 1, 1, 1) and g.geometry[6:].tolist() == [5.0, 2.0]
    for bad in (dict(values=np.zeros((2, 3, 4))), dict(values=np.zeros((1, 2, 3, 4, 2))),
                dict(values=np.zeros((0, 1, 1, 1, 3))), dict(values=np.full((1, 1, 1, 3), np.nan)),
                dict(values=np.zeros((1, 1, 1, 3)), spacing=(1, 0, 1)), dict(values=np.zeros((1, 1, 1, 3)), origin=(0, 0)),
                dict(values=np.zeros((1, 1, 1, 3)), origin=(0, math.inf, 0)),
                dict(values=np.zeros((2, 1, 1, 1, 3)), frame_dt=0.0), dict(values=np.zeros((1, 1, 1, 3)), t0=math.nan)):
        with pytest.raises(ValueError):
            currents.CurrentGrid(**bad)
    p = currents.profile([-3.0, -2.0, -1.0], [[1, 0, 0], [2, 0, 0], [3, 0, 0]])
    assert p.dims == (1, 3, 1, 1) and p.origin == (0.0, 0.0, -3.0) and p.spacing == (1.0, 1.0, 1.0)
    with pytest.raises(ValueError):
        currents.profile([-3.0, -2.0, -0.5], np.zeros((3, 3)))       # uneven
    with pytest.raises(ValueError):
        currents.profile([-1.0, -2.0], np.zeros((2, 3)))             # decreasing
    with pytest.raises(ValueError):
        currents.profile([-1.0, 0.0], np.zeros((3, 3)))
    b = currents.power_law_profile(0.8, 0.3, seabed_z=-18.4, nz=32)
    assert currents.CurrentGrid(np.broadcast_to(np.arange(3.0), (2, 3, 4, 3))).values.flags.c_contiguous
    assert b.dims == (1, 32, 1, 1) and b.origin[2] == -18.4 and b.spacing[2] == pytest.approx(18.4 / 31)
    speed = np.hypot(b.values[0, :, 0, 0, 0], b.values[0, :, 0, 0, 1])
    assert speed[0] == 0.0 and speed[-1] == pytest.approx(0.8) and (np.diff(speed) > 0).all()
    assert np.allclose(np.arctan2(b.values[0, 1:, 0, 0, 1], b.values[0, 1:, 0, 0, 0]), 0.3)
    assert (b.values[..., 2] == 0).all()
    z = np.array([-18.4, -10.0, -1.0, 0.0, 5.0, -30.0])
    got = currents.evaluate(b, 0.0, 0.0, z, 0.0)
    want = 0.8 * np.clip((z + 18.4) / 18.4, 0, 1) ** (1 / 7)
    assert np.allclose(np.hypot(got[:, 0], got[:, 1]), want, rtol=0.02, atol=1e-12)
    for bad in (dict(top_z=-20.0), dict(alpha=0.0), dict(nz=1), dict(speed=math.nan)):
        with pytest.raises(ValueError):
            currents.power_law_profile(**{**dict(speed=1.0, direction=0.0, seabed_z=-18.4), **bad})


@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_host_evaluator_matches_reference(current_emul, shape):
    """grid_eval on the host == currents.evaluate bit for bit: random grids, points outside on every side, times
    before, between and after the frames, and NaN coordinates."""
    rng = np.random.default_rng(sorted(SHAPES).index(shape))
    g = _random_grid(rng, SHAPES[shape])
    m = 40_000
    p = _grid_points(rng, m)
    t = rng.uniform(1200.0, 1290.0, m)                                # frames at 1230, 1240, 1250 (, 1260)
    t[:6] = [1230.0, 1240.0, 1250.0, -1e9, 1e9, 1235.0]
    for k, col in enumerate((p[:, 0], p[:, 1], p[:, 2], t)):
        col[10 + k] = np.nan
        col[20 + k] = np.inf
        col[30 + k] = -np.inf
    got = _emul_eval(current_emul, g, p[:, 0], p[:, 1], p[:, 2], t)
    want = currents.evaluate(g, p[:, 0], p[:, 1], p[:, 2], t)
    assert np.array_equal(got, want, equal_nan=True)
    assert np.isnan(want[10:14]).all() and np.isfinite(want[14:]).all()
    assert (np.abs(want[14:]) <= 0.6 + 1e-12).all()                    # a convex combination of the nodes


def test_nodes_and_multilinear_fields(current_emul):
    """Node values at nodes: exactly where the node is the lower corner of its cell (weight 0; the last node of an
    axis is reached with weight 1, a + (b - a), so to rounding); a multilinear field to rounding."""
    rng = np.random.default_rng(4)
    g = _random_grid(rng, (3, 4, 5, 6), spacing=(25.0, 30.0, 0.75))
    nt, nz, ny, nx = g.dims
    f, k, j, i = (a.reshape(-1) for a in np.meshgrid(*(np.arange(n) for n in g.dims), indexing="ij"))
    x, y, z = (g.origin[a] + b * g.spacing[a] for a, b in ((0, i), (1, j), (2, k)))
    t = g.t0 + f * g.frame_dt
    want = g.values[f, k, j, i]
    lower = (f < nt - 1) & (k < nz - 1) & (j < ny - 1) & (i < nx - 1)
    for got in (currents.evaluate(g, x, y, z, t), _emul_eval(current_emul, g, x, y, z, t)):
        assert np.array_equal(got[lower], want[lower])
        assert np.allclose(got, want, rtol=0, atol=1e-15)
    # a multilinear field is reproduced to rounding anywhere inside, and held outside
    coef = rng.uniform(-1, 1, (5, 3))
    lin = lambda x, y, z, t: coef[0] + np.outer(x, coef[1]) + np.outer(y, coef[2]) + np.outer(z, coef[3]) + \
        np.outer(t - g.t0, coef[4]) / 10
    vals = lin(x, y, z, t).reshape(nt, nz, ny, nx, 3)
    h = currents.CurrentGrid(vals, origin=g.origin, spacing=g.spacing, t0=g.t0, frame_dt=g.frame_dt)
    m = 20_000
    q = [rng.uniform(g.origin[a], g.origin[a] + (n - 1) * g.spacing[a], m) for a, n in ((0, nx), (1, ny), (2, nz))]
    tq = rng.uniform(g.t0, g.t0 + (nt - 1) * g.frame_dt, m)
    got = _emul_eval(current_emul, h, *q, tq)
    assert np.abs(got - lin(*q, tq)).max() <= 1e-12 * np.abs(vals).max() * 10
    far = _emul_eval(current_emul, h, q[0] + 1e6, q[1], q[2], tq)
    assert np.allclose(far, lin(np.full(m, h.origin[0] + (nx - 1) * h.spacing[0]), q[1], q[2], tq), rtol=0, atol=1e-10)


@pytest.mark.parametrize("sea", [None, "jonswap16_deep", "mixed_h3"])
@pytest.mark.parametrize("f32", [False, True], ids=["fp64", "fp32"])
def test_host_water_at_with_grid_matches_composition(current_emul, sea, f32):
    """water_at on the host with a grid == the NumPy composition bit for bit (with the host's own sea samples),
    with and without env rows; the grid leaves the sea's samples unchanged."""
    field = FIELDS[sea]() if sea else None
    rng = np.random.default_rng(12)
    g = _random_grid(rng, (2, 6, 7, 8))
    cond = _random_cond(rng, 50, origin=30.0, tau=20.0)
    cur = np.array([0.3, -0.2, 0.05])
    for t in (1220.0, 1234.5, 1300.0):
        p = _grid_points(rng, 20_000, f32)
        env = rng.integers(0, 50, len(p))
        for rows in (False, True):
            kw = dict(cond=cond, env=env) if rows else {}
            fld, water = _emul_water(current_emul, p, t, f32, grid=g, field=field, surface_z=0.25, current=cur, **kw)
            fld0, _ = _emul_water(current_emul, p, t, f32, field=field, surface_z=0.25, current=cur, **kw)
            assert np.array_equal(fld, fld0)
            want = compose(g, p, t, 0.25, cur, field=fld if field else None, **kw)
            assert np.array_equal(water, want), (t, rows)
    bad_f, bad_w = _emul_water(current_emul, p[:2], 0.0, f32, grid=g, cond=cond, env=[-1, 50])
    assert np.isnan(bad_w).all() and np.isnan(bad_f).all()


@pytest.mark.parametrize("f32", [False, True], ids=["fp64", "fp32"])
def test_host_zero_and_uniform_grids(current_emul, f32):
    """A zero grid == no grid; a uniform grid g with a zero global current == no grid with current g: bit for bit."""
    rng = np.random.default_rng(21)
    field = FIELDS["jonswap16_deep"]()
    cond = _random_cond(rng, 20)
    p = _grid_points(rng, 10_000, f32)
    env = rng.integers(0, 20, len(p))
    gval = np.array([0.35, -0.6, 0.02])
    zero = currents.CurrentGrid(np.zeros((2, 3, 4, 5, 3)), frame_dt=1.0)
    uni = currents.CurrentGrid(np.broadcast_to(gval, (2, 3, 4, 5, 3)), frame_dt=1.0)
    for kw in (dict(), dict(cond=cond, env=env)):
        cur = (0.2, -0.1, 0.0)
        a = _emul_water(current_emul, p, 500.25, f32, grid=zero, field=field, current=cur, **kw)
        b = _emul_water(current_emul, p, 500.25, f32, field=field, current=cur, **kw)
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
        a = _emul_water(current_emul, p, 500.25, f32, grid=uni, field=field, **kw)
        b = _emul_water(current_emul, p, 500.25, f32, field=field, current=gval, **kw)
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


# --------------------------------------------------------------------------- GPU
torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu
DTYPES = pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda:0")


def _grid_t(grid, dev):
    return torch.as_tensor(np.ascontiguousarray(grid.values), dtype=torch.float64, device=dev).contiguous()


def _set_grid(e, grid, dev, values=None):
    v = _grid_t(grid, dev) if values is None else values
    e.set_current_grid(v, grid.origin, grid.spacing, grid.t0, grid.frame_dt)
    return v


@gpu
@DTYPES
@pytest.mark.parametrize("sea", [True, False], ids=["waves", "still"])
def test_sample_water_matches_composition(dev, dtype, sea):
    from silver2_isaacsim_b200 import HydroEngine
    from silver2_isaacsim_b200 import _lib as L

    f32 = dtype == torch.float32
    rng = np.random.default_rng(31)
    e = HydroEngine(1000, dtype=dtype, device=dev)
    cur = np.array([0.3, -0.2, 0.05])
    e.set_environment(current=cur, surface_z=-0.4)
    with pytest.raises(L.H2OError, match="NOT_CONFIGURED"):
        e.sample_water(np.zeros((2, 3)), env=0)
    assert np.array_equal(e.sample_water(np.zeros((2, 3))).cpu().numpy(), [[-0.4, *cur]] * 2)
    g = _random_grid(rng, (2, 6, 7, 8))
    vt = _set_grid(e, g, dev)
    assert e.current_grid is vt
    cond = _random_cond(rng, 1000, origin=30.0, tau=20.0)
    e.set_env_conditions(_cond_t(cond, dev), 1)
    if sea:
        e.set_wave_field(FIELDS["mixed_h3"]())
    for t in (1200.0, 1234.5, 1245.0, 1300.0):
        e.set_wave_time(t)
        p = _grid_points(rng, 100_000, f32)
        pt = _t(p, dtype, dev)
        env = rng.integers(0, 1000, len(p))
        envt = torch.as_tensor(env, device=dev)
        got = e.sample_water(pt).cpu().numpy()
        fld = e.sample_waves(pt).cpu().numpy() if sea else None
        assert np.array_equal(got, compose(g, p, t, -0.4, cur, field=fld)), t
        got = e.sample_water(pt, env=envt).cpu().numpy()
        fld = e.sample_waves(pt, env=envt).cpu().numpy() if sea else None
        assert np.array_equal(got, compose(g, p, t, -0.4, cur, cond=cond, env=env, field=fld)), t
    bad = e.sample_water(pt[:4], env=[-1, 1000, 2 ** 40, 3]).cpu().numpy()
    assert np.isnan(bad[:3]).all() and np.isfinite(bad[3]).all()


@gpu
@DTYPES
def test_step_with_grid_matches_oracle(oracle, dev, dtype):
    """Strict parity: 2e5 boxes as 4-body envs and robots with random env rows, a 3-D two-frame grid and a
    16-component finite-depth sea, against the oracle fed with the waterline and flow sample_water returns; fp32
    flagged bodies included, per-robot wrench too."""
    wl = _wave_workload()
    n_envs = wl.n // 4
    rng = np.random.default_rng(99)
    cond = _random_cond(rng, n_envs, dz=0.6, origin=30.0, tau=20.0)
    env = np.arange(wl.n) // 4
    g = currents.CurrentGrid(rng.uniform(-0.8, 0.8, (2, 8, 16, 16, 3)), origin=(-200.0, -200.0, -4.0),
                             spacing=(25.0, 25.0, 0.75), t0=1230.0, frame_dt=15.0)
    cur = np.array([0.3, -0.2, 0.05])
    e = _engine(wl, dtype, dev, "auto", stats=True)
    e.set_environment(current=cur, surface_z=0.15)
    e.set_env_conditions(_cond_t(cond, dev), 4)
    _set_grid(e, g, dev)
    e.set_wave_field(waves.jonswap(2.0, 6.0, n_components=16, direction=0.5, seed=9, depth=40.0))
    e.set_wave_time(1234.5)
    smp = e.sample_water(_t(wl.pos, dtype, dev), env=torch.as_tensor(env, device=dev)).cpu().numpy()
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    F, T, Wr = e.step(_t(wl.pos, dtype, dev), _t(wl.quat_xyzw, dtype, dev), _t(wl.lin_vel, dtype, dev),
                      _t(wl.ang_vel, dtype, dev), wl.dt, robot_wrench=True)
    F, T, Wr = (x.double().cpu().numpy() for x in (F, T, Wr))
    assert e.last_kernel == "direct" and e.wave_time == 1234.5 + wl.dt
    if dtype == torch.float32:
        assert e.stats()["reevaluated_bodies"] > 0
    pos = wl.pos.astype(np.float64).copy()
    pos[:, 2] = pos[:, 2] - smp[:, 0]
    flow = smp[:, 1:]
    if dtype == torch.float32:
        vrel = (wl.lin_vel - flow.astype(np.float32)).astype(np.float64)
        prel = (wl.prev_lin.astype(np.float64) - wl.lin_vel.astype(np.float64)) + vrel
    else:
        vrel = wl.lin_vel.astype(np.float64) - flow
        prel = wl.prev_lin.astype(np.float64) - flow
    ref = oracle.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vrel, wl.ang_vel, prel, wl.prev_ang, wl.dt)
    _check(wl, pos, dtype, ref, F, T, "current grid")
    want = oracle.robot_wrench(wl.pos.astype(np.float64), ref.force, ref.torque, 4)
    F4 = np.abs(ref.force).reshape(-1, 4, 3).sum(axis=(1, 2)) + np.abs(ref.torque).reshape(-1, 4, 3).sum(axis=(1, 2))
    lever = np.abs(wl.pos.astype(np.float64)).reshape(-1, 12).max(axis=1) * np.abs(ref.force).reshape(-1, 12).max(axis=1)
    rel = 2e-4 if dtype == torch.float32 else 1e-10
    assert (np.abs(Wr - want).max(axis=1) <= rel * (F4 + lever) + 1e-6).all()
    # the grid does move the flow by its own magnitude
    no_grid = compose(None, wl.pos.astype(np.float64), 1234.5, 0.15, cur, cond=cond, env=env)
    assert np.abs(smp[:, 1:] - no_grid[:, 1:]).max() > 0.3


@gpu
@DTYPES
@pytest.mark.parametrize("kind", ["zero", "uniform"])
@pytest.mark.parametrize("path", ["eager", "bound", "graph", "persistent", "host"])
def test_zero_and_uniform_grids_are_bit_identical(dev, dtype, kind, path):
    """With random env rows and a sea: a zero grid == no grid, and a uniform grid g with a zero global current ==
    no grid with current g, bit for bit through every step path (the clock too).  The persistent rollout with a grid
    is its own kernel instantiation, which may contract the model's multiply-adds differently from the one without:
    there both sides carry a grid (a uniform g with current 0 == a zero grid with current g, bit for bit), and the
    grid-less rollout agrees to the rounding of test_persistent_rollout_with_conditions_equals_stepwise."""
    wl = _identity_workload()
    field = waves.jonswap(1.5, 6.0, n_components=8, seed=12, depth=30.0)
    cond = _random_cond(np.random.default_rng(3), wl.n // 4, origin=50.0)
    gval = (0.35, -0.6, 0.02)
    persistent = path == "persistent"
    res = []
    for with_grid in (False, True, None):
        if with_grid is None and not persistent:
            break
        e = _engine(wl, dtype, dev, "direct")
        cur = (0.2, -0.1, 0.0) if kind == "zero" else ((0.0, 0.0, 0.0) if with_grid else gval)
        e.set_environment(current=cur, surface_z=0.1)
        e.set_wave_field(field)
        e.set_wave_time(500.25)
        e.set_env_conditions(_cond_t(cond, dev), 4)
        if with_grid or (persistent and with_grid is False):
            vals = torch.zeros(2, 3, 4, 5, 3, dtype=torch.float64, device=dev)
            if kind == "uniform" and with_grid:
                vals[:] = torch.tensor(gval, dtype=torch.float64)
            e.set_current_grid(vals, (-50.0, -50.0, -3.0), (20.0, 25.0, 1.0), t0=500.0, frame_dt=0.01)
            if not with_grid and kind == "zero":                        # a zero grid of other dims and geometry
                e.set_current_grid(vals[:1, :2, :1].contiguous(), (7.0, -3.0, 1.0), (1.0, 2.0, 0.5))
        res.append(_run_path(e, wl, dtype, dev, path))
        assert e.last_kernel == "direct"
    for k, (a, b) in enumerate(zip(res[0], res[1])):
        assert (_same_bits(a, b) if isinstance(a, torch.Tensor) else a == b), (path, k)
    if persistent:
        tol = 2e-4 if dtype == torch.float32 else 1e-9
        for k, (a, b) in enumerate(zip(res[1], res[2])):
            if not isinstance(a, torch.Tensor):
                assert a == b                                           # the clock
                continue
            a, b = a.double().numpy().reshape(len(a), -1), b.double().numpy().reshape(len(b), -1)
            ok = (a == b) | (np.isnan(a) & np.isnan(b))
            with np.errstate(invalid="ignore"):
                ok |= np.abs(a - b) <= tol * (np.abs(a).max(axis=1, keepdims=True) + 1e-3)
            assert float(ok.all(axis=1).mean()) >= 0.995, k


def _frames_grid(rng):
    """Three frames 0.05 s apart: a 1/60 s step crosses frames."""
    return currents.CurrentGrid(rng.uniform(-0.8, 0.8, (3, 4, 5, 6, 3)), origin=(-150.0, -150.0, -3.0),
                                spacing=(60.0, 75.0, 1.5), t0=0.02, frame_dt=0.05)


@gpu
@DTYPES
def test_time_frames_clock_graph_and_persistent(dev, dtype):
    """A time-varying grid without waves advances the clock; graph replays == eager steps bit for bit; the
    persistent rollout == stepwise steps; a single-frame grid leaves the clock alone."""
    wl = W.uniform_small_batch(1024)
    rng = np.random.default_rng(8)
    g = _frames_grid(rng)
    K, res = 10, {}
    for mode in ("eager", "graph", "persistent", "stepwise"):
        e = _engine(wl, dtype, dev, stats=True)
        _set_grid(e, g, dev)
        ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
        e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
        F, T = e.bind(*ten)
        if mode in ("eager", "stepwise"):
            for _ in range(2 * K):
                e.step_bound(wl.dt)
                e.integrate_free_bodies(*ten, F, T, wl.dt, wl.g)
        elif mode == "graph":
            e.set_rollout_mode(free_bodies=True, gravity=wl.g)
            e.capture_rollout(K, wl.dt)
            e.launch_rollout()
            e.launch_rollout()
        else:
            e.rollout_persistent(2 * K, wl.dt, gravity=wl.g)
            assert e.launch_count == 2                                  # the rollout + one clock advance
        torch.cuda.synchronize()
        assert e.stats(reset=True)["nonfinite_bodies"] == 0
        res[mode] = ([x.cpu() for x in ten + [F, T, e.prev_velocities()]], e.wave_time)
    want = 0.0
    for _ in range(2 * K):
        want += wl.dt
    assert all(r[1] == want for r in res.values())
    assert all(torch.equal(a, b) for a, b in zip(res["eager"][0], res["graph"][0]))
    tol = 2e-4 if dtype == torch.float32 else 1e-9
    for name, a, b in zip(("pos", "quat", "lin_vel", "ang_vel", "force", "torque", "prev"), res["stepwise"][0],
                          res["persistent"][0]):
        a, b = a.double().numpy(), b.double().numpy()
        scale = np.abs(a).max(axis=1, keepdims=True) + 1e-3
        frac = float((np.abs(a - b) <= tol * scale).all(axis=1).mean())
        assert frac >= 0.995, (name, frac)
    # the frames matter: the first frame alone gives other forces; a single frame leaves the clock alone
    e = _engine(wl, dtype, dev)
    first = currents.CurrentGrid(g.values[:1], origin=g.origin, spacing=g.spacing)
    _set_grid(e, first, dev)
    ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    F, T = e.bind(*ten)
    for _ in range(2 * K):
        e.step_bound(wl.dt)
        e.integrate_free_bodies(*ten, F, T, wl.dt, wl.g)
    assert e.wave_time == 0.0 and not torch.equal(F.cpu(), res["eager"][0][4])


@gpu
@DTYPES
def test_graph_replay_follows_in_place_edits(dev, dtype):
    """An in-place edit of the borrowed grid between two replays reaches the second replay (== eager steps with the
    same edit, bit for bit); set_current_grid drops the graph, a refused call keeps it."""
    from silver2_isaacsim_b200 import _lib as L

    wl = _identity_workload(8000, seed=4)
    rng = np.random.default_rng(6)
    g0, g1 = _frames_grid(rng), _frames_grid(rng)
    res = []
    for mode in ("eager", "graph"):
        e = _engine(wl, dtype, dev, "auto")
        vt = _set_grid(e, g0, dev)
        ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
        e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
        F, T = e.bind(*ten)
        if mode == "graph":
            e.capture_rollout(3, wl.dt)
            e.launch_rollout()
            vt.copy_(torch.as_tensor(g1.values, device=dev))
            e.launch_rollout()
        else:
            for k in range(6):
                if k == 3:
                    vt.copy_(torch.as_tensor(g1.values, device=dev))
                e.step_bound(wl.dt)
        torch.cuda.synchronize()
        res.append([F.cpu(), T.cpu(), e.prev_velocities().cpu(), e.wave_time])
    for a, b in zip(*res):
        assert (torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b)
    lib = L.load()
    dims = (ctypes.c_int64 * 4)(*g1.dims)
    geom = (ctypes.c_double * 8)(*g1.geometry)
    assert lib.h2o_set_current_grid(e._h, ctypes.c_void_p(vt.data_ptr() + 4), dims, geom) == 7   # refused
    e.launch_rollout()
    _set_grid(e, g1, dev, vt)
    with pytest.raises(L.H2OError, match="NOT_CONFIGURED"):
        e.launch_rollout()


@gpu
@DTYPES
def test_origins_give_the_same_current(dev, dtype):
    """Env 1 = env 0 shifted by D with origin D, in a 3-D grid and a sea: the same force and torque (bit for bit on
    the fast path; flagged fp32 bodies, re-evaluated from world p_x, p_y, within the strict fp32 bound)."""
    from silver2_isaacsim_b200 import HydroEngine

    B = 20_000
    base = W.heterogeneous_boxes(B, seed=77, xy_range=150.0)
    rng = np.random.default_rng(78)
    p = np.round(np.stack([rng.uniform(-150, 150, B), rng.uniform(-150, 150, B), rng.uniform(-3, 2, B)], 1) * 64) / 64
    D = np.array([1024.0, -512.0, 0.0])
    pos = np.concatenate([p, p + D])
    tile = lambda a: np.concatenate([a, a])
    cond = waves.env_conditions(2, current=(0.1, 0.05, 0.0), surface_dz=0.2, time_offset=3.0, origin=[[0.0, 0.0], D[:2]])
    g = currents.CurrentGrid(rng.uniform(-0.8, 0.8, (2, 8, 16, 16, 3)), origin=(-160.0, -160.0, -4.0),
                             spacing=(21.0, 21.0, 0.75), t0=400.0, frame_dt=8.0)
    out = []
    for with_grid in (True, False):
        e = HydroEngine(2 * B, dtype=dtype, device=dev)
        e.set_globals(base.rho, base.g)
        e.set_params_per_body(tile(base.coeff_per_body()))
        e.enable_stats(True)
        e.set_environment(current=(0.2, -0.1, 0.0), surface_z=0.1)
        e.set_env_conditions(_cond_t(cond, dev), B)
        if with_grid:
            _set_grid(e, g, dev)
        e.set_wave_field(waves.jonswap(2.0, 6.0, n_components=16, direction=0.5, seed=9, depth=40.0))
        e.set_wave_time(401.0)
        e.set_prev(_t(tile(base.prev_lin), dtype, dev), _t(tile(base.prev_ang), dtype, dev))
        F, T = e.step(_t(pos, dtype, dev), _t(tile(base.quat_xyzw), dtype, dev), _t(tile(base.lin_vel), dtype, dev),
                      _t(tile(base.ang_vel), dtype, dev), base.dt)
        out.append((F.double().cpu().numpy(), T.double().cpu().numpy(), e.stats()["reevaluated_bodies"]))
    (F, T, redo), (F0, _, _) = out
    same = (F[:B] == F[B:]).all(axis=1) & (T[:B] == T[B:]).all(axis=1)
    if dtype == torch.float32:
        assert (~same).sum() <= redo, ((~same).sum(), redo)
        scoring.assert_fp32(F[B:], F[:B], "shifted env force")
        scoring.assert_fp32(T[B:], T[:B], "shifted env torque")
    else:
        assert same.all()
    assert not np.array_equal(F, F0)                                    # the grid does act


@gpu
@DTYPES
def test_masked_reset_restarts_the_frames(dev, dtype):
    wl = _identity_workload(4096, seed=21)
    n_envs = wl.n // 4
    rng = np.random.default_rng(23)
    cond = _random_cond(rng, n_envs, origin=30.0)
    g = currents.CurrentGrid(rng.uniform(-0.8, 0.8, (3, 4, 5, 6, 3)), origin=(-150.0, -150.0, -3.0),
                             spacing=(60.0, 75.0, 1.5), t0=0.0, frame_dt=20.0)
    e = _engine(wl, dtype, dev)
    ct = _cond_t(cond, dev)
    e.set_env_conditions(ct, 4)
    _set_grid(e, g, dev)
    e.set_wave_time(-25.0)
    ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    e.bind(*ten)
    for _ in range(3):
        e.step_bound(wl.dt)
    ids = np.array([0, 7, 100, n_envs - 2])
    clock = e.wave_time
    assert clock == ((-25.0 + wl.dt) + wl.dt) + wl.dt                   # the grid alone runs the clock
    e.reset_envs(ids, restart_waves=True)
    after = ct.cpu().numpy()
    assert (after[ids, waves.COND_TAU] == -clock).all()
    p = wl.pos.astype(np.float64)[ids * 4]
    if dtype == torch.float32:
        p = p.astype(np.float32).astype(np.float64)
    got = e.sample_water(_t(p, dtype, dev), env=ids).cpu().numpy()
    at_zero = after[ids].copy()
    at_zero[:, waves.COND_TAU] = 0.0
    want = compose(g, p, 0.0, 0.0, (0, 0, 0), cond=at_zero, env=np.arange(len(ids)))
    assert np.array_equal(got, want)                                    # env time clock + (-clock) == 0: frame 0
    other = e.sample_water(_t(p, dtype, dev), env=ids + 1).cpu().numpy()
    assert np.array_equal(other, compose(g, p, clock, 0.0, (0, 0, 0), cond=after, env=ids + 1))


@gpu
def test_boxes_drift_with_a_seabed_boundary_layer(dev):
    """Physics: neutrally buoyant, fully submerged 1 m cubes released at rest in a power-law seabed boundary layer
    (seabed 18.4 m below the mean level, as SILVER2 at the Obsea site) drift, in a persistent rollout, at the
    profile's speed at their own depth."""
    from silver2_isaacsim_b200 import HydroEngine
    from silver2_isaacsim_b200 import params as P

    prm = P.HydroParams()
    n = 64
    speed, direction = 0.6, 0.4
    bl = currents.power_law_profile(speed, direction, seabed_z=-18.4, top_z=-2.0)
    e = HydroEngine(n, dtype=torch.float64, device=dev)
    e.set_globals(prm.waterDensity, prm.gravity)
    e.set_part_table(np.asarray([prm.coeff_record(prm.waterDensity * 1.0)]), np.zeros(1, np.int32))
    _set_grid(e, bl, dev)
    z0 = np.linspace(-17.5, -3.0, n)
    pos = torch.as_tensor(np.stack([np.zeros(n), np.arange(n) * 3.0, z0], 1), device=dev)
    quat = torch.tensor([[0.0, 0.0, 0.0, 1.0]] * n, dtype=torch.float64, device=dev)
    v, w = torch.zeros(n, 3, dtype=torch.float64, device=dev), torch.zeros(n, 3, dtype=torch.float64, device=dev)
    e.bind(pos, quat, v, w)
    dt = 1.0 / 60.0
    e.rollout_persistent(3600, dt, gravity=prm.gravity)                # 60 s
    torch.cuda.synchronize()
    p, vel = pos.cpu().numpy(), v.cpu().numpy()
    want = currents.evaluate(bl, p[:, 0], p[:, 1], p[:, 2], 0.0)
    print("depth, drift speed, profile speed:", [(round(a, 2), round(b, 4), round(c, 4)) for a, b, c in
                                                  zip(p[::16, 2], np.hypot(vel[::16, 0], vel[::16, 1]),
                                                      np.hypot(want[::16, 0], want[::16, 1]))])
    assert np.abs(p[:, 2] - z0).max() < 0.5                            # neutrally buoyant: the depth is kept
    assert np.abs(vel - want).max() <= 0.02 * speed
    assert (np.diff(np.hypot(vel[:, 0], vel[:, 1])) > 0).all()          # faster further from the seabed


@gpu
def test_current_grid_inputs_are_validated(dev):
    from silver2_isaacsim_b200 import _lib as L

    wl = _identity_workload(4000, seed=3)
    e = _engine(wl, torch.float64, dev)
    ten = [_t(a, torch.float64, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    e.bind(*ten)
    e.capture_rollout(2, wl.dt)
    good = torch.zeros(2, 3, 4, 5, 3, dtype=torch.float64, device=dev)
    for bad in (good.float(), good.cpu(), good[..., :2].contiguous(), good.transpose(1, 2), good[0, 0],
                good[:0], good.cpu().numpy()):
        with pytest.raises(ValueError):
            e.set_current_grid(bad, (0, 0, 0), (1, 1, 1), 0.0, 1.0)
    with pytest.raises(ValueError):
        e.set_current_grid(good, (0, 0), (1, 1, 1), 0.0, 1.0)
    for geo in (dict(spacing=(1, 0, 1)), dict(spacing=(1, 1, -1)), dict(origin=(0, math.nan, 0)),
                dict(t0=math.inf), dict(frame_dt=0.0), dict(frame_dt=-1.0)):
        kw = {**dict(origin=(0, 0, 0), spacing=(1, 1, 1), t0=0.0, frame_dt=1.0), **geo}
        with pytest.raises(L.H2OError, match="BAD_ARGUMENT"):
            e.set_current_grid(good, **kw)
    lib = L.load()
    geom = (ctypes.c_double * 8)(0, 0, 0, 1, 1, 1, 0, 1)
    ptr = ctypes.c_void_p(good.data_ptr())
    for dims in ((0, 3, 4, 5), (2, 3, -1, 5), (1 << 40, 1 << 20, 1, 1), (1 << 62, 2, 1, 1)):
        assert lib.h2o_set_current_grid(e._h, ptr, (ctypes.c_int64 * 4)(*dims), geom) == 2      # BAD_ARGUMENT
    dims = (ctypes.c_int64 * 4)(2, 3, 4, 5)
    assert lib.h2o_set_current_grid(e._h, ctypes.c_void_p(good.data_ptr() + 4), dims, geom) == 7  # ALIGNMENT
    host = np.zeros((2, 3, 4, 5, 3))
    assert lib.h2o_set_current_grid(e._h, host.ctypes.data_as(ctypes.c_void_p), dims, geom) == 5  # BAD_DEVICE
    e.launch_rollout()                                                  # every refused call kept the graph
    e.set_current_grid(good[0], (0, 0, 0), (1, 1, 1))                    # one frame: 4-D, frame_dt unused
    assert e.current_grid is not None
    with pytest.raises(L.H2OError, match="NOT_CONFIGURED"):
        e.launch_rollout()
    e.step_bound(wl.dt)
    assert e.last_kernel == "direct" and e.wave_time == 0.0
    e.set_current_grid(None)
    assert e.current_grid is None
