"""Per-env water conditions (include/h2o.h, h2o_set_env_conditions / h2o_reset_envs / h2o_wave_sample_env): the
NumPy module, the composition of csrc/h2o_waves.cuh (water_at) on the host, and on the GPU the sampler, the step,
the rollouts, the masked reset and the bit-identity of identity rows."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from silver2_isaacsim_b200 import waves
from silver2_isaacsim_b200 import workloads as W
from tests import scoring
from tests.test_waves import FIELDS, _check, _engine, _points, _scales, _t, _wave_workload, wave_emul  # noqa: F401

IDENTITY = np.array([0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0])
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def env_emul(tmp_path_factory):
    """tests/host_emul/env_emul.cpp (water_at instantiated for the host), built into a temporary directory with
    the flags of the wave emulator."""
    so = str(tmp_path_factory.mktemp("env_emul") / "libh2o_env_emul.so")
    subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-shared", "-mfma", "-ffp-contract=fast", "-fvisibility=hidden",
                    "-o", so, os.path.join(ROOT, "tests", "host_emul", "env_emul.cpp")], check=True)
    lib = ctypes.CDLL(so)
    lib.emul_wave_sample_env.restype = ctypes.c_int
    return lib


def _random_cond(rng, n_envs, c=0.5, dz=0.5, tau=1e4, origin=200.0, smax=2.0):
    return waves.env_conditions(n_envs, current=rng.uniform(-c, c, (n_envs, 3)), surface_dz=rng.uniform(-dz, dz, n_envs),
                                wave_scale=rng.uniform(0.0, smax, n_envs), time_offset=rng.uniform(0.0, tau, n_envs),
                                origin=rng.uniform(-origin, origin, (n_envs, 2)))


def _emul_env(lib, field, points, env_index, cond, t, f32, surface_z=0.0, current=(0.0, 0.0, 0.0)):
    p = np.ascontiguousarray(points, dtype=np.float64)
    idx = np.ascontiguousarray(env_index, dtype=np.int32)
    cond = np.ascontiguousarray(cond, dtype=np.float64)
    comps = np.ascontiguousarray(field.components, dtype=np.float64)
    cur = np.ascontiguousarray(current, dtype=np.float64)
    fld, water = np.zeros((len(p), 4)), np.zeros((len(p), 4))
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = lib.emul_wave_sample_env(int(f32), len(comps), ptr(comps), ctypes.c_double(field.depth), ctypes.c_int64(len(p)),
                                  ptr(p), ptr(idx), ctypes.c_int64(len(cond)), ptr(cond), ctypes.c_double(t),
                                  ctypes.c_double(surface_z), ptr(cur), ptr(fld), ptr(water))
    assert rc == 0
    return fld, water


def _assert_env_field_close(got, want, field, s, rel, what):
    """The bounds of test_waves.py, scaled row by row by |s|."""
    s_eta, s_u = _scales(field)
    s = np.abs(s)
    assert (np.abs(got[:, 0] - want[:, 0]) <= rel * s * s_eta).all(), what
    assert (np.abs(got[:, 1:] - want[:, 1:]).max(axis=1) <= rel * s * s_u).all(), what


# --------------------------------------------------------------------------- CPU
def test_env_conditions_defaults_and_validation():
    c = waves.env_conditions(5)
    assert c.shape == (5, 8) and c.dtype == np.float64 and (c == IDENTITY).all()
    c = waves.env_conditions(3, current=(0.1, 0.2, 0.3), surface_dz=[0.0, 1.0, 2.0], wave_scale=0.5, time_offset=7.0,
                             origin=np.array([[1, 2], [3, 4], [5, 6]]))
    assert (c[:, waves.COND_CX:waves.COND_CZ + 1] == [0.1, 0.2, 0.3]).all()
    assert (c[:, waves.COND_DZ] == [0, 1, 2]).all() and (c[:, waves.COND_SCALE] == 0.5).all()
    assert (c[:, waves.COND_TAU] == 7.0).all() and (c[:, waves.COND_X0] == [1, 3, 5]).all()
    assert (c[:, waves.COND_Y0] == [2, 4, 6]).all()
    assert waves.COND_COLS == 8 and waves.COND_Y0 == 7
    for bad in (dict(current=(1.0, 2.0)), dict(surface_dz=[0.0, 1.0]), dict(origin=(1.0, 2.0, 3.0)),
                dict(wave_scale=math.nan), dict(time_offset=[0.0, math.inf, 0.0]), dict(current=np.zeros((2, 3)))):
        with pytest.raises(ValueError):
            waves.env_conditions(3, **bad)
    for n in (0, -1):
        with pytest.raises(ValueError):
            waves.env_conditions(n)


def test_evaluate_takes_per_point_time_and_level():
    field = FIELDS["jonswap64_h12"]()
    rng = np.random.default_rng(3)
    p = _points(rng, 2000, field.depth, False)
    want = waves.evaluate(field, p, 1234.5, surface_z=0.3)
    assert np.array_equal(waves.evaluate(field, p, np.full(len(p), 1234.5), surface_z=np.full(len(p), 0.3)), want)
    with pytest.raises(ValueError):
        waves.evaluate(field, p, np.zeros(3))


@pytest.mark.parametrize("name", sorted(FIELDS))
def test_evaluate_env_equals_per_env_evaluate(name):
    field = FIELDS[name]()
    rng = np.random.default_rng(11)
    cond = _random_cond(rng, 40)
    p = _points(rng, 4000, field.depth, False)
    env = rng.integers(0, 40, len(p))
    t, sz = 321.25, -0.2
    got = waves.evaluate_env(field, p, t, cond, env, surface_z=sz)
    for e in range(40):
        r = cond[e]
        q = p[env == e].copy()
        q[:, 0] -= r[waves.COND_X0]
        q[:, 1] -= r[waves.COND_Y0]
        want = r[waves.COND_SCALE] * waves.evaluate(field, q, t + r[waves.COND_TAU], sz + r[waves.COND_DZ])
        assert np.array_equal(got[env == e], want), e


@pytest.mark.parametrize("name", sorted(FIELDS))
@pytest.mark.parametrize("f32", [False, True], ids=["fp64", "fp32"])
def test_host_env_evaluator_matches_reference(env_emul, name, f32):
    """water_at on the host against waves.evaluate_env (1000 random env rows), and the waterline and flow it
    composes, bit for bit: (surface_z + dz) + s eta and (current + c) + s u."""
    field = FIELDS[name]()
    rng = np.random.default_rng(5)
    cond = _random_cond(rng, 1000)
    cur = np.array([0.3, -0.2, 0.05])
    for t in (0.0, 1234.5, 99999.37):
        p = _points(rng, 50_000, field.depth, f32)
        env = rng.integers(0, 1000, len(p))
        got, water = _emul_env(env_emul, field, p, env, cond, t, f32, surface_z=0.25, current=cur)
        want = waves.evaluate_env(field, p, t, cond, env, surface_z=0.25)
        _assert_env_field_close(got, want, field, cond[env, waves.COND_SCALE], 2e-6 if f32 else 1e-12, (name, t))
        r = cond[env]
        assert np.array_equal(water[:, 0], (0.25 + r[:, waves.COND_DZ]) + got[:, 0])
        assert np.array_equal(water[:, 1:], (cur[None, :] + r[:, waves.COND_CX:waves.COND_CZ + 1]) + got[:, 1:])
    bad, _ = _emul_env(env_emul, field, p[:3], [-1, 1000, 2 ** 31 - 1], cond, 0.0, f32)
    assert np.isnan(bad).all()


@pytest.mark.parametrize("name", sorted(FIELDS))
@pytest.mark.parametrize("f32", [False, True], ids=["fp64", "fp32"])
def test_identity_row_reproduces_the_env_free_evaluator(env_emul, wave_emul, name, f32):
    from tests.test_waves import _emul_sample

    field = FIELDS[name]()
    rng = np.random.default_rng(8)
    cond = waves.env_conditions(4)
    for t in (0.0, 1234.5, 99999.37):
        p = _points(rng, 20_000, field.depth, f32)
        got, water = _emul_env(env_emul, field, p, rng.integers(0, 4, len(p)), cond, t, f32, surface_z=0.25)
        want = _emul_sample(wave_emul, field, p, t, f32, surface_z=0.25)
        assert np.array_equal(got, want)
        assert np.array_equal(water[:, 0], 0.25 + want[:, 0]) and np.array_equal(water[:, 1:], want[:, 1:])


# --------------------------------------------------------------------------- GPU
torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu
DTYPES = pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda:0")


def _cond_t(cond, dev):
    return torch.as_tensor(np.ascontiguousarray(cond), dtype=torch.float64, device=dev).contiguous()


@gpu
@DTYPES
@pytest.mark.parametrize("name", sorted(FIELDS))
def test_sample_env_matches_reference(dev, dtype, name):
    from silver2_isaacsim_b200 import HydroEngine
    from silver2_isaacsim_b200 import _lib as L

    field = FIELDS[name]()
    f32 = dtype == torch.float32
    rng = np.random.default_rng(17)
    e = HydroEngine(1000, dtype=dtype, device=dev)
    with pytest.raises(L.H2OError, match="NOT_CONFIGURED"):
        e.sample_waves(np.zeros((2, 3)), env=0)
    cond = _random_cond(rng, 1000)
    ct = _cond_t(cond, dev)
    e.set_env_conditions(ct, 1)
    assert e.env_conditions is ct
    assert np.array_equal(e.sample_waves(np.ones((3, 3)), env=[0, 5, 999]).cpu().numpy(), np.zeros((3, 4)))  # no field
    e.set_environment(surface_z=-0.4)
    e.set_wave_field(field)
    for t in (0.0, 1234.5, 99999.37):
        e.set_wave_time(t)
        p = _points(rng, 100_000, field.depth, f32)
        env = rng.integers(0, 1000, len(p))
        got = e.sample_waves(_t(p, dtype, dev), env=torch.as_tensor(env, device=dev)).cpu().numpy()
        want = waves.evaluate_env(field, p, t, cond, env, surface_z=-0.4)
        _assert_env_field_close(got, want, field, cond[env, waves.COND_SCALE], 2e-6 if f32 else 1e-12, (name, t))
    bad = e.sample_waves(_t(p[:4], dtype, dev), env=[-1, 1000, 2 ** 40, 3]).cpu().numpy()
    assert np.isnan(bad[:3]).all() and np.isfinite(bad[3]).all()


def _env_oracle_inputs(wl, dtype, cur, surface_z, cond, env, smp):
    """What the kernel feeds the model: p_z - ((surface_z + dz) + s eta) in float64, v - S((current + c) + s u)."""
    r = cond[env]
    pos = wl.pos.astype(np.float64).copy()
    pos[:, 2] = pos[:, 2] - ((surface_z + r[:, waves.COND_DZ]) + smp[:, 0])
    flow = (cur[None, :] + r[:, waves.COND_CX:waves.COND_CZ + 1]) + smp[:, 1:]
    if dtype == torch.float32:
        vrel = (wl.lin_vel - flow.astype(np.float32)).astype(np.float64)
        prel = (wl.prev_lin.astype(np.float64) - wl.lin_vel.astype(np.float64)) + vrel
    else:
        vrel = wl.lin_vel.astype(np.float64) - flow
        prel = wl.prev_lin.astype(np.float64) - flow
    return pos, vrel, prel


@gpu
@DTYPES
@pytest.mark.parametrize("layout", ["split", "view"])
@pytest.mark.parametrize("sea", [True, False], ids=["waves", "still"])
def test_step_with_env_conditions_matches_oracle(oracle, dev, dtype, layout, sea):
    """Strict parity: 2e5 boxes as 4-body envs and robots with random c_e, dz, s, tau and origins, in a 16-component
    finite-depth JONSWAP sea (or none) with a global current and surface_z, against the oracle fed with the
    waterline and flow the kernel forms; fp32 flagged bodies included, per-robot wrench too."""
    wl = _wave_workload()
    n_envs = wl.n // 4
    rng = np.random.default_rng(99)
    cond = _random_cond(rng, n_envs, dz=0.6)
    env = np.arange(wl.n) // 4
    cur = np.array([0.3, -0.2, 0.05])
    surface_z = 0.15
    e = _engine(wl, dtype, dev, "auto", stats=True)
    e.set_environment(current=cur, surface_z=surface_z)
    e.set_env_conditions(_cond_t(cond, dev), 4)
    if sea:
        e.set_wave_field(waves.jonswap(2.0, 6.0, n_components=16, direction=0.5, seed=9, depth=40.0))
        e.set_wave_time(1234.5)
    smp = e.sample_waves(_t(wl.pos, dtype, dev), env=torch.as_tensor(env, device=dev)).cpu().numpy()
    assert (np.abs(smp[:, 0]).max() > 0.5) == sea                       # the sea does cut the boxes
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
        assert e.stats()["reevaluated_bodies"] > 0                     # the float64 re-evaluation sees the env too
    pos, vrel, prel = _env_oracle_inputs(wl, dtype, cur, surface_z, cond, env, smp)
    ref = oracle.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vrel, wl.ang_vel, prel, wl.prev_ang, wl.dt)
    _check(wl, pos, dtype, ref, F, T, f"env conditions {layout} sea={sea}")
    want = oracle.robot_wrench(wl.pos.astype(np.float64), ref.force, ref.torque, 4)
    F4 = np.abs(ref.force).reshape(-1, 4, 3).sum(axis=(1, 2)) + np.abs(ref.torque).reshape(-1, 4, 3).sum(axis=(1, 2))
    lever = np.abs(wl.pos.astype(np.float64)).reshape(-1, 12).max(axis=1) * np.abs(ref.force).reshape(-1, 12).max(axis=1)
    rel = 2e-4 if dtype == torch.float32 else 1e-10
    assert (np.abs(Wr - want).max(axis=1) <= rel * (F4 + lever) + 1e-6).all()


def _identity_workload(n=20_000, seed=31):
    wl = W.heterogeneous_boxes(n, seed=seed, xy_range=150.0)
    wl.pos[:, 2] = np.random.default_rng(seed).uniform(-3.0, 2.0, n).astype(np.float32)
    wl.bodies_per_robot = 4
    return wl


def _run_path(e, wl, dtype, dev, path):
    """One path through the engine; returns the tensors it produces, the carried state and the clock."""
    ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    if path == "eager":
        out = list(e.step(*ten, wl.dt, robot_wrench=True))
        out += list(e.step(*ten, wl.dt, robot_wrench=True))
    elif path == "bound":
        out = list(e.bind(*ten, robot_wrench=True))
        e.step_bound(wl.dt)
        e.step_bound(wl.dt)
    elif path == "graph":
        F, T = e.bind(*ten)
        e.set_rollout_mode(free_bodies=True, gravity=wl.g)
        e.capture_rollout(5, wl.dt)
        e.launch_rollout()
        e.launch_rollout()
        out = ten + [F, T]
    elif path == "persistent":
        F, T = e.bind(*ten)
        e.rollout_persistent(10, wl.dt, gravity=wl.g)
        out = ten + [F, T]
    else:  # host, pinned buffers
        ins = [torch.as_tensor(np.ascontiguousarray(a)).to(dtype).pin_memory()
               for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
        outs = [torch.empty(wl.n, 3, dtype=dtype).pin_memory() for _ in range(2)]
        outs.append(torch.empty(wl.n // 4, 6, dtype=dtype).pin_memory())
        e.step_host(*ins, wl.dt, out_force=outs[0], out_torque=outs[1], out_robot_wrench=outs[2])
        e.step_host(*ins, wl.dt, out_force=outs[0], out_torque=outs[1], out_robot_wrench=outs[2])
        out = outs
    torch.cuda.synchronize()
    return [x.cpu() for x in out] + [e.prev_velocities().cpu(), e.wave_time]


def _same_bits(a, b):
    """Bit for bit (a free-body rollout of boxes may leave non-finite states, which torch.equal calls unequal)."""
    ints = {torch.float32: torch.int32, torch.float64: torch.int64}
    return a.dtype == b.dtype and torch.equal(a.view(ints[a.dtype]), b.view(ints[b.dtype]))


@gpu
@DTYPES
@pytest.mark.parametrize("sea", [True, False], ids=["waves", "still"])
@pytest.mark.parametrize("path", ["eager", "bound", "graph", "persistent", "host"])
def test_identity_rows_are_bit_identical(dev, dtype, sea, path):
    wl = _identity_workload()
    field = waves.jonswap(1.5, 6.0, n_components=8, seed=12, depth=30.0)
    res = []
    for with_cond in (False, True):
        e = _engine(wl, dtype, dev, "direct")
        e.set_environment(current=(0.2, -0.1, 0.0), surface_z=0.1)
        if sea:
            e.set_wave_field(field)
            e.set_wave_time(500.25)
        if with_cond:
            cond = _cond_t(waves.env_conditions(wl.n // 4), dev)
            e.set_env_conditions(cond, 4)
        res.append(_run_path(e, wl, dtype, dev, path))
        assert e.last_kernel == "direct"
    for k, (a, b) in enumerate(zip(*res)):
        assert (_same_bits(a, b) if isinstance(a, torch.Tensor) else a == b), (path, k)


@gpu
@DTYPES
def test_removing_conditions_returns_to_the_tile_kernel(dev, dtype):
    wl = W.heterogeneous_boxes(60_000, seed=5)

    def run(e):
        e.set_environment(current=(0.2, 0.1, 0.0), surface_z=0.1)
        e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
        F, T = e.step(*[_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)], wl.dt)
        return F.cpu(), T.cpu()

    e0 = _engine(wl, dtype, dev, "auto")
    F0, T0 = run(e0)
    assert e0.last_kernel == "tile"
    e1 = _engine(wl, dtype, dev, "auto")
    e1.set_env_conditions(_cond_t(waves.env_conditions(wl.n // 4), dev), 4)
    F1, T1 = run(e1)
    assert e1.last_kernel == "direct"
    e1.set_env_conditions(None)
    assert e1.env_conditions is None
    F2, T2 = run(e1)
    assert e1.last_kernel == "tile" and torch.equal(F0, F2) and torch.equal(T0, T2)


@gpu
@DTYPES
def test_graph_replay_follows_in_place_edits(dev, dtype):
    """An in-place edit of the borrowed tensor between two replays reaches the second replay (== eager steps with
    the same edit, bit for bit); a new tensor drops the graph."""
    from silver2_isaacsim_b200 import _lib as L

    wl = _identity_workload(8000, seed=4)
    field = waves.jonswap(1.0, 5.0, n_components=8, seed=2)
    rng = np.random.default_rng(6)
    cond0 = _random_cond(rng, wl.n // 4, tau=100.0, origin=50.0)
    cond1 = _random_cond(rng, wl.n // 4, tau=100.0, origin=50.0)
    res = []
    for mode in ("eager", "graph"):
        e = _engine(wl, dtype, dev, "auto")
        e.set_wave_field(field)
        ct = _cond_t(cond0, dev)
        e.set_env_conditions(ct, 4)
        ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
        e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
        F, T = e.bind(*ten)
        if mode == "graph":
            e.capture_rollout(3, wl.dt)
            e.launch_rollout()
            ct.copy_(torch.as_tensor(cond1, device=dev))
            e.launch_rollout()
        else:
            for k in range(6):
                if k == 3:
                    ct.copy_(torch.as_tensor(cond1, device=dev))
                e.step_bound(wl.dt)
        torch.cuda.synchronize()
        res.append([F.cpu(), T.cpu(), e.prev_velocities().cpu(), e.wave_time])
    for a, b in zip(*res):
        assert (torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b)
    e.set_env_conditions(_cond_t(cond1, dev), 4)
    with pytest.raises(L.H2OError, match="NOT_CONFIGURED"):
        e.launch_rollout()


@gpu
@DTYPES
def test_persistent_rollout_with_conditions_equals_stepwise(dev, dtype):
    wl = W.uniform_small_batch(1024)
    field = waves.jonswap(1.0, 5.0, n_components=8, seed=4, depth=15.0)
    cond = _random_cond(np.random.default_rng(13), wl.n // 4, dz=0.3, origin=100.0)
    K, res = 25, []
    for mode in ("stepwise", "persistent"):
        e = _engine(wl, dtype, dev, stats=True)
        e.set_wave_field(field)
        e.set_wave_time(77.7)
        e.set_env_conditions(_cond_t(cond, dev), 4)
        ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
        e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
        F, T = e.bind(*ten)
        if mode == "stepwise":
            for _ in range(K):
                e.step_bound(wl.dt)
                e.integrate_free_bodies(*ten, F, T, wl.dt, wl.g)
        else:
            e.rollout_persistent(K, wl.dt, gravity=wl.g)
        torch.cuda.synchronize()
        st = e.stats(reset=True)
        assert st["bodies"] == K * wl.n and st["nonfinite_bodies"] == 0
        res.append(([x.double().cpu().numpy() for x in ten] +
                    [F.double().cpu().numpy(), T.double().cpu().numpy(), e.prev_velocities().double().cpu().numpy()],
                    e.wave_time))
    assert res[0][1] == res[1][1]
    tol = 2e-4 if dtype == torch.float32 else 1e-9   # as test_persistent_rollout_in_waves_equals_stepwise
    for name, a, b in zip(("pos", "quat", "lin_vel", "ang_vel", "force", "torque", "prev"), res[0][0], res[1][0]):
        scale = np.abs(a).max(axis=1, keepdims=True) + 1e-3
        frac = float((np.abs(a - b) <= tol * scale).all(axis=1).mean())
        assert frac >= 0.995, (name, frac)


@gpu
@DTYPES
def test_masked_reset(dev, dtype):
    from silver2_isaacsim_b200 import _lib as L

    wl = _identity_workload(4096, seed=21)
    n_envs = wl.n // 4
    field = FIELDS["jonswap16_deep"]()
    rng = np.random.default_rng(23)
    cond = _random_cond(rng, n_envs)
    e = _engine(wl, dtype, dev)
    with pytest.raises(L.H2OError, match="NOT_CONFIGURED"):
        e.reset_envs([0])
    e.set_wave_field(field)
    e.set_wave_time(55.5)
    ct = _cond_t(cond, dev)
    e.set_env_conditions(ct, 4)
    ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    e.bind(*ten)
    e.capture_rollout(2, wl.dt)
    e.launch_rollout()
    prev0 = e.prev_velocities().clone()
    assert (prev0 != 0).any(dim=1).all()
    mask = torch.as_tensor(rng.random(n_envs) < 0.3, device=dev)
    e.reset_envs(mask)
    body_mask = mask.repeat_interleave(4)
    prev1 = e.prev_velocities()
    assert (prev1[body_mask] == 0).all() and torch.equal(prev1[~body_mask], prev0[~body_mask])
    assert torch.equal(ct.cpu(), torch.as_tensor(cond))                  # no restart: the rows are untouched
    # restart the waves of a few envs given by id
    ids = np.array([0, 7, 100, n_envs - 1])
    clock = e.wave_time
    e.reset_envs(ids, restart_waves=True)
    after = ct.cpu().numpy()
    other = np.ones(n_envs, bool)
    other[ids] = False
    assert (after[ids, waves.COND_TAU] == -clock).all()
    assert np.array_equal(after[other], cond[other]) and np.array_equal(np.delete(after[ids], waves.COND_TAU, axis=1),
                                                                        np.delete(cond[ids], waves.COND_TAU, axis=1))
    p = wl.pos.astype(np.float64)[ids * 4]
    if dtype == torch.float32:
        p = p.astype(np.float32).astype(np.float64)
    got = e.sample_waves(_t(p, dtype, dev), env=ids).cpu().numpy()
    at_zero = after.copy()
    at_zero[:, waves.COND_TAU] = 0.0
    want = waves.evaluate_env(field, p, 0.0, at_zero, ids)
    assert np.array_equal(want, waves.evaluate_env(field, p, clock, after, ids))   # clock + (-clock) == 0 exactly
    _assert_env_field_close(got, want, field, after[ids, waves.COND_SCALE], 2e-6 if dtype == torch.float32 else 1e-12,
                            "restart")
    e.launch_rollout()                                                   # the captured rollout is kept
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        e.reset_envs([n_envs])
    with pytest.raises(ValueError):
        e.reset_envs(torch.ones(n_envs + 1, dtype=torch.bool))


@gpu
@DTYPES
def test_origins_give_the_same_sea(dev, dtype):
    """Env 1 = env 0 shifted by D with origin D: the same force and torque (bit for bit on the fast path; flagged
    fp32 bodies, re-evaluated from world p_x, p_y, within the strict fp32 bound).  Env 2 (s = 0) = still water."""
    from silver2_isaacsim_b200 import HydroEngine

    B = 20_000
    base = W.heterogeneous_boxes(B, seed=77, xy_range=150.0)
    rng = np.random.default_rng(78)
    p = np.round(np.stack([rng.uniform(-150, 150, B), rng.uniform(-150, 150, B), rng.uniform(-3, 2, B)], 1) * 64) / 64
    D = np.array([1024.0, -512.0, 0.0])
    pos = np.concatenate([p, p + D, p])
    tile = lambda a: np.concatenate([a, a, a])
    cond = waves.env_conditions(3, current=(0.1, 0.05, 0.0), surface_dz=0.2, wave_scale=[1.0, 1.0, 0.0],
                                time_offset=[30.0, 30.0, 30.0], origin=[[0.0, 0.0], D[:2], [5.0, 5.0]])
    field = waves.jonswap(2.0, 6.0, n_components=16, direction=0.5, seed=9, depth=40.0)
    out = []
    for sea in (True, False):
        e = HydroEngine(3 * B, dtype=dtype, device=dev)
        e.set_globals(base.rho, base.g)
        e.set_params_per_body(tile(base.coeff_per_body()))
        e.enable_stats(True)
        e.set_environment(current=(0.2, -0.1, 0.0), surface_z=0.1)
        e.set_env_conditions(_cond_t(cond, dev), B)
        if sea:
            e.set_wave_field(field)
            e.set_wave_time(400.0)
        e.set_prev(_t(tile(base.prev_lin), dtype, dev), _t(tile(base.prev_ang), dtype, dev))
        F, T = e.step(_t(pos, dtype, dev), _t(tile(base.quat_xyzw), dtype, dev), _t(tile(base.lin_vel), dtype, dev),
                      _t(tile(base.ang_vel), dtype, dev), base.dt)
        out.append((F.double().cpu().numpy(), T.double().cpu().numpy(), e.stats()["reevaluated_bodies"]))
    (F, T, redo), (Fs, Ts, _) = out
    same = (F[:B] == F[B:2 * B]).all(axis=1) & (T[:B] == T[B:2 * B]).all(axis=1)
    if dtype == torch.float32:
        assert (~same).sum() <= redo, ((~same).sum(), redo)
        scoring.assert_fp32(F[B:2 * B], F[:B], "shifted env force")
        scoring.assert_fp32(T[B:2 * B], T[:B], "shifted env torque")
    else:
        assert same.all()
    assert np.array_equal(F[2 * B:], Fs[2 * B:]) and np.array_equal(T[2 * B:], Ts[2 * B:])
    assert not np.array_equal(F[:B], Fs[:B])                              # the sea does act on env 0


@gpu
def test_env_condition_inputs_are_validated(dev):
    from silver2_isaacsim_b200 import _lib as L

    wl = _identity_workload(4000, seed=3)
    e = _engine(wl, torch.float64, dev)
    ten = [_t(a, torch.float64, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    e.bind(*ten)
    e.capture_rollout(2, wl.dt)
    good = _cond_t(waves.env_conditions(1000), dev)
    with pytest.raises(L.H2OError, match="BAD_SHAPE"):
        e.set_env_conditions(_cond_t(waves.env_conditions(571), dev), 7)   # 7 does not divide 4000
    for bad in (good[:999], good.float(), good.cpu(), good.t().contiguous(), good[:, :4].contiguous(),
                _cond_t(waves.env_conditions(2000), dev)[::2], waves.env_conditions(1000)):
        with pytest.raises(ValueError):
            e.set_env_conditions(bad, 4)
    with pytest.raises(ValueError):
        e.set_env_conditions(good, 0)
    lib = L.load()
    assert lib.h2o_set_env_conditions(e._h, 4, ctypes.c_void_p(good.data_ptr() + 4)) == 7     # H2O_ERR_ALIGNMENT
    host = waves.env_conditions(1000)
    assert lib.h2o_set_env_conditions(e._h, 4, host.ctypes.data_as(ctypes.c_void_p)) == 5     # H2O_ERR_BAD_DEVICE
    e.launch_rollout()                                                   # every refused call kept the graph
    e.set_env_conditions(good, 4)
    with pytest.raises(L.H2OError, match="NOT_CONFIGURED"):
        e.launch_rollout()
    e.set_env_conditions(None)
    assert e.env_conditions is None
