"""Built-in linear wave field (include/h2o.h, h2o_set_wave_field): the NumPy module, the evaluator of
csrc/h2o_waves.cuh on the host, and on the GPU the sampler, the step, the clock and the rollouts."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from silver2_isaacsim_b200 import waves
from silver2_isaacsim_b200 import workloads as W
from tests import scoring

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def wave_emul(tmp_path_factory):
    """tests/host_emul/waves_emul.cpp (the evaluator header instantiated for the host), built into a temporary
    directory with the flags of the model emulator."""
    so = str(tmp_path_factory.mktemp("wave_emul") / "libh2o_wave_emul.so")
    subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-shared", "-mfma", "-ffp-contract=fast", "-fvisibility=hidden",
                    "-o", so, os.path.join(ROOT, "tests", "host_emul", "waves_emul.cpp")], check=True)
    lib = ctypes.CDLL(so)
    lib.emul_wave_sample.restype = ctypes.c_int
    return lib


def _emul_sample(lib, field, points, t, f32, surface_z=0.0):
    p = np.ascontiguousarray(points, dtype=np.float64)
    c = np.ascontiguousarray(field.components, dtype=np.float64)
    out = np.zeros((len(p), 4))
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = lib.emul_wave_sample(int(f32), len(c), ptr(c), ctypes.c_double(field.depth), ctypes.c_int64(len(p)), ptr(p),
                              ctypes.c_double(t), ctypes.c_double(surface_z), ptr(out))
    assert rc == 0
    return out


def _points(rng, m, depth, f32):
    zlo = -(depth + 2.0) if math.isfinite(depth) else -60.0   # below the bottom: the velocity depth is clamped
    p = np.stack([rng.uniform(-500, 500, m), rng.uniform(-500, 500, m), rng.uniform(zlo, 2.0, m)], axis=1)
    return p.astype(np.float32).astype(np.float64) if f32 else p


FIELDS = {
    "jonswap16_deep": lambda: waves.jonswap(2.0, 7.0, n_components=16, direction=0.4, seed=3),
    "jonswap64_h12": lambda: waves.jonswap(1.5, 9.0, n_components=64, direction=-1.0, seed=5, depth=12.0),
    "mixed_h3": lambda: waves.WaveField(np.concatenate([
        waves.regular(0.3, 5.0, direction=2.0, phase=0.7, depth=3.0).components,
        waves.regular(0.05, 1.3, direction=-2.5, depth=3.0).components,
        waves.regular(0.2, 20.0, phase=-1.0, depth=3.0).components]), 3.0),
}


def _scales(field):
    c = field.components
    return c[:, 0].sum(), (c[:, 0] * c[:, 3]).sum()


def _assert_field_close(got, want, field, rel, what):
    s_eta, s_u = _scales(field)
    e_eta = np.abs(got[:, 0] - want[:, 0]).max() / s_eta
    e_u = np.abs(got[:, 1:] - want[:, 1:]).max() / s_u
    assert e_eta <= rel and e_u <= rel, (what, e_eta, e_u)


# --------------------------------------------------------------------------- CPU: waves.py
def test_wavenumber_dispersion_residual_and_limits():
    g = 9.81
    omega = np.geomspace(0.02, 20.0, 200)
    for depth in (0.05, 0.5, 3.0, 20.0, 200.0, 5000.0, math.inf):
        k = waves.wavenumber(omega, depth, g)
        th = 1.0 if math.isinf(depth) else np.tanh(k * depth)
        assert (np.abs(g * k * th - omega ** 2) <= 1e-12 * omega ** 2).all(), depth
    w = np.array([0.5, 1.0, 3.0])
    assert np.allclose(waves.wavenumber(w, 1e4), w ** 2 / g, rtol=1e-6, atol=0)        # deep limit
    assert np.allclose(waves.wavenumber(1e-3 * w, 0.01), 1e-3 * w / math.sqrt(g * 0.01), rtol=1e-6, atol=0)  # shallow
    assert waves.wavenumber(1.0) == 1.0 / g and isinstance(waves.wavenumber(1.0, 5.0), float)


def test_regular_field():
    f = waves.regular(0.4, 6.0, direction=math.pi / 2, phase=0.3, depth=10.0)
    a, kx, ky, w, ph = f.components[0]
    assert (a, ph, f.depth) == (0.4, 0.3, 10.0) and w == 2 * math.pi / 6.0
    assert abs(kx) < 1e-15 and ky == pytest.approx(waves.wavenumber(w, 10.0), rel=1e-15)


def test_jonswap_variance_seed_and_peak():
    hs, tp = 2.5, 8.0
    f = waves.jonswap(hs, tp, n_components=32, seed=11)
    a, w = f.components[:, 0], f.components[:, 3]
    assert abs((a ** 2 / 2).sum() / (hs / 4) ** 2 - 1) <= 0.02
    assert np.array_equal(f.components, waves.jonswap(hs, tp, n_components=32, seed=11).components)
    assert not np.array_equal(f.components[:, 4], waves.jonswap(hs, tp, n_components=32, seed=12).components[:, 4])
    fr = w / (2 * math.pi)
    df = fr[1] - fr[0]
    assert np.allclose(np.diff(fr), df) and abs(fr[np.argmax(a)] - 1 / tp) <= df   # peak bin at 1 / tp
    assert ((f.components[:, 4] >= 0) & (f.components[:, 4] < 2 * math.pi)).all()


def test_evaluate_matches_hyperbolic_form_and_linear_theory():
    f = waves.regular(0.5, 4.0, direction=0.3, phase=0.2, depth=6.0)
    a, kx, ky, w, ph = f.components[0]
    k = math.hypot(kx, ky)
    rng = np.random.default_rng(1)
    p = np.stack([rng.uniform(-50, 50, 500), rng.uniform(-50, 50, 500), rng.uniform(-8, 1, 500)], axis=1)
    t = 17.3
    got = waves.evaluate(f, p, t, surface_z=0.5)
    z = np.clip(p[:, 2] - 0.5, -6.0, 0.0)
    th = kx * p[:, 0] + ky * p[:, 1] - w * t + ph
    C, S = np.cosh(k * (z + 6.0)) / np.sinh(k * 6.0), np.sinh(k * (z + 6.0)) / np.sinh(k * 6.0)
    want = np.stack([a * np.cos(th), a * w * C * np.cos(th) * kx / k, a * w * C * np.cos(th) * ky / k,
                     a * w * S * np.sin(th)], axis=1)
    assert np.abs(got - want).max() <= 1e-13
    # the vertical orbital velocity at the mean level is the rate of change of the elevation
    top = np.array([[3.0, -2.0, 0.0]])
    h = 1e-5
    deta = (waves.evaluate(f, top, t + h)[0, 0] - waves.evaluate(f, top, t - h)[0, 0]) / (2 * h)
    assert waves.evaluate(f, top, t)[0, 3] == pytest.approx(deta, rel=1e-8)


@pytest.mark.parametrize("name", sorted(FIELDS))
@pytest.mark.parametrize("f32", [False, True], ids=["fp64", "fp32"])
def test_host_evaluator_matches_reference(wave_emul, name, f32):
    """csrc/h2o_waves.cuh on the host against waves.evaluate: 10^5 points, clocks up to 10^5 s."""
    field = FIELDS[name]()
    rng = np.random.default_rng(42)
    for t in (0.0, 1234.5, 99999.37):
        p = _points(rng, 100_000, field.depth, f32)
        got = _emul_sample(wave_emul, field, p, t, f32, surface_z=0.25)
        want = waves.evaluate(field, p, t, surface_z=0.25)
        _assert_field_close(got, want, field, 2e-6 if f32 else 1e-12, (name, t))


def test_wave_inputs_are_validated():
    from silver2_isaacsim_b200.engine import HydroEngine

    good = waves.regular(0.2, 5.0).components
    bad = {
        "shape": np.zeros((2, 4)),
        "too many": np.repeat(good, 65, axis=0),
        "nan": np.array([[0.1, np.nan, 0.0, 1.0, 0.0]]),
        "inf": np.array([[0.1, 0.1, 0.0, np.inf, 0.0]]),
        "negative amplitude": np.array([[-0.1, 0.1, 0.0, 1.0, 0.0]]),
        "zero k": np.array([[0.1, 0.0, 0.0, 1.0, 0.0]]),
        "zero omega": np.array([[0.1, 0.1, 0.0, 0.0, 0.0]]),
    }
    for what, comps in bad.items():
        with pytest.raises(ValueError):
            waves.WaveField(comps)
    for depth in (0.0, -1.0, -math.inf, math.nan):
        with pytest.raises(ValueError):
            waves.WaveField(good, depth)
        with pytest.raises(ValueError):
            waves.wavenumber(1.0, depth)
    for omega in (0.0, -1.0, math.nan, math.inf):
        with pytest.raises(ValueError):
            waves.wavenumber(omega)
    with pytest.raises(ValueError):
        waves.jonswap(1.0, 8.0, n_components=65)
    with pytest.raises(ValueError):
        waves.jonswap(0.0, 8.0)
    with pytest.raises(ValueError):
        waves.regular(0.1, 0.0)
    f = waves.WaveField(good)
    assert not f.components.flags.writeable and f.n_components == 1 and f.depth == math.inf
    # HydroEngine.set_wave_field takes a WaveField (or None); the check comes before any device call
    eng = object.__new__(HydroEngine)
    for x in (good, [[0.2, 0.1, 0.0, 1.0, 0.0]], "regular"):
        with pytest.raises(TypeError):
            eng.set_wave_field(x)


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
def test_sample_matches_reference(dev, dtype, name):
    from silver2_isaacsim_b200 import HydroEngine

    field = FIELDS[name]()
    f32 = dtype == torch.float32
    rng = np.random.default_rng(7)
    e = HydroEngine(1, dtype=dtype, device=dev)
    assert np.array_equal(e.sample_waves(np.zeros((3, 3))).cpu().numpy(), np.zeros((3, 4)))   # no field: still water
    e.set_environment(surface_z=-0.4)
    e.set_wave_field(field)
    for t in (0.0, 1234.5, 99999.37):
        e.set_wave_time(t)
        assert e.wave_time == t
        p = _points(rng, 100_000, field.depth, f32)
        got = e.sample_waves(_t(p, dtype, dev))
        assert got.dtype == torch.float64 and tuple(got.shape) == (len(p), 4)
        _assert_field_close(got.cpu().numpy(), waves.evaluate(field, p, t, surface_z=-0.4), field,
                            2e-6 if f32 else 1e-12, (name, t))
    with pytest.raises(ValueError):
        e.sample_waves(np.zeros((4, 2)))


def _wave_workload(n=200_000, seed=2026):
    """Heterogeneous boxes over several wavelengths with p_z in [-3, 2] m, as robots of 4 bodies."""
    wl = W.heterogeneous_boxes(n, seed=seed, xy_range=150.0)
    rng = np.random.default_rng(seed + 1)
    wl.pos[:, 2] = rng.uniform(-3.0, 2.0, n).astype(np.float32)
    wl.bodies_per_robot = 4
    return wl


def _oracle_inputs(wl, dtype, cur, surface_z, smp):
    """What the kernel feeds the model: p_z - (surface_z + eta) in float64, v - S(current + u) formed in S."""
    pos = wl.pos.astype(np.float64).copy()
    pos[:, 2] = pos[:, 2] - (surface_z + smp[:, 0])
    flow = cur[None, :] + smp[:, 1:]
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


@gpu
@DTYPES
@pytest.mark.parametrize("layout", ["split", "view"])
def test_step_in_waves_matches_oracle(oracle, dev, dtype, layout):
    """Strict parity: 2e5 boxes cut by a 16-component JONSWAP sea (finite depth) with a uniform current, clock at
    1234.5 s, against the oracle fed with the surface-relative heights and flow-relative velocities the kernel
    forms from sample_waves at the same clock; fp32 flagged bodies included, per-robot wrench too."""
    wl = _wave_workload()
    field = waves.jonswap(2.0, 6.0, n_components=16, direction=0.5, seed=9, depth=40.0)
    cur = np.array([0.3, -0.2, 0.05]).astype(np.float32).astype(np.float64)
    surface_z = 0.15
    e = _engine(wl, dtype, dev, "auto", stats=True)
    e.set_environment(current=cur, surface_z=surface_z)
    e.set_wave_field(field)
    e.set_wave_time(1234.5)
    smp = e.sample_waves(_t(wl.pos, dtype, dev)).cpu().numpy()
    assert np.abs(smp[:, 0]).max() > 0.5                              # the sea does cut the boxes
    e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
    if layout == "split":
        F, T, Wr = e.step(_t(wl.pos, dtype, dev), _t(wl.quat_xyzw, dtype, dev), _t(wl.lin_vel, dtype, dev),
                          _t(wl.ang_vel, dtype, dev), wl.dt, robot_wrench=True)
    else:
        F, T, Wr = e.step_view(_t(wl.pos, dtype, dev), _t(wl.quat_xyzw, dtype, dev), _t(wl.velocities(), dtype, dev),
                               wl.dt, robot_wrench=True)
    F, T, Wr = (x.double().cpu().numpy() for x in (F, T, Wr))
    assert e.last_kernel == "direct" and e.wave_time == 1234.5 + wl.dt
    st = e.stats()
    if dtype == torch.float32:
        assert st["reevaluated_bodies"] > 0                            # the float64 re-evaluation sees the waves too
    pos, vrel, prel = _oracle_inputs(wl, dtype, cur, surface_z, smp)
    ref = oracle.step(wl.ctor_rows(), wl.masses(), pos, wl.quat_xyzw, vrel, wl.ang_vel, prel, wl.prev_ang, wl.dt)
    _check(wl, pos, dtype, ref, F, T, f"waves {layout}")
    want = oracle.robot_wrench(wl.pos.astype(np.float64), ref.force, ref.torque, 4)
    F4 = np.abs(ref.force).reshape(-1, 4, 3).sum(axis=(1, 2)) + np.abs(ref.torque).reshape(-1, 4, 3).sum(axis=(1, 2))
    lever = np.abs(wl.pos.astype(np.float64)).reshape(-1, 12).max(axis=1) * np.abs(ref.force).reshape(-1, 12).max(axis=1)
    rel = 2e-4 if dtype == torch.float32 else 1e-10
    assert (np.abs(Wr - want).max(axis=1) <= rel * (F4 + lever) + 1e-6).all()
    prev = e.prev_velocities().double().cpu().numpy()
    assert (prev[:, :3] == wl.lin_vel.astype(np.float64)).all()        # the carried state stays the body velocity


@gpu
def test_clock_steps_and_graph_invalidation(dev):
    from silver2_isaacsim_b200 import _lib as L

    wl = W.uniform_small_batch(2048)
    e = _engine(wl, torch.float64, dev)
    ten = [_t(a, torch.float64, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
    assert e.wave_time == 0.0
    e.set_wave_field(waves.regular(0.3, 6.0))
    t0, dt = 12.34, 1.0 / 120.0
    e.set_wave_time(t0)
    want = t0
    for _ in range(37):
        e.step(*ten, dt)
        want += dt
    assert e.wave_time == want                                         # the same additions, bit for bit
    n0 = e.launch_count
    e.step(*ten, 0.0)                                                  # dt <= 1e-6: a no-op, clock included
    assert e.wave_time == want and e.launch_count == n0
    e.bind(*ten)
    e.capture_rollout(3, dt)
    e.set_wave_time(5.0)                                               # the clock is graph input: graph kept
    e.launch_rollout()
    assert e.wave_time == ((5.0 + dt) + dt) + dt
    e.set_wave_field(waves.regular(0.2, 6.0))                          # a setter: graph dropped
    with pytest.raises(L.H2OError, match="NOT_CONFIGURED"):
        e.launch_rollout()
    e.capture_rollout(2, dt)
    e.set_wave_field(None)
    with pytest.raises(L.H2OError, match="NOT_CONFIGURED"):
        e.launch_rollout()
    with pytest.raises(ValueError):
        e.set_wave_time(math.nan)


@gpu
@DTYPES
def test_graph_rollout_in_waves_equals_eager(dev, dtype):
    """Free bodies: a captured K-step rollout replayed twice == 2K eager (step + integrate_free_bodies), bit for bit,
    the clock included (every captured step advances it on the device)."""
    wl = W.uniform_small_batch(3000)
    field = waves.jonswap(1.0, 5.0, n_components=8, seed=2)
    K, res = 20, []
    for mode in ("eager", "graph"):
        e = _engine(wl, dtype, dev)
        e.set_environment(current=(0.1, 0.0, 0.0))
        e.set_wave_field(field)
        e.set_wave_time(300.0)
        ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
        e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
        F, T = e.bind(*ten)
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
        res.append([x.cpu() for x in ten + [F, T, e.prev_velocities()]] + [e.wave_time])
    for a, b in zip(*res[:2]):
        assert (torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b)


@gpu
@DTYPES
def test_persistent_rollout_in_waves_equals_stepwise(dev, dtype):
    """K steps in one persistent launch in waves == K x (fused step + free-body stepper); the clock bit for bit."""
    wl = W.uniform_small_batch(1024)
    field = waves.jonswap(1.0, 5.0, n_components=8, seed=4, depth=15.0)
    K, res = 25, []
    for mode in ("stepwise", "persistent"):
        e = _engine(wl, dtype, dev, stats=True)
        e.set_wave_field(field)
        e.set_wave_time(77.7)
        ten = [_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)]
        e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
        F, T = e.bind(*ten)
        if mode == "stepwise":
            for _ in range(K):
                e.step_bound(wl.dt)
                e.integrate_free_bodies(*ten, F, T, wl.dt, wl.g)
        else:
            e.rollout_persistent(K, wl.dt, gravity=wl.g)
            assert e.launch_count == 2                                  # the rollout + one clock advance
        torch.cuda.synchronize()
        st = e.stats(reset=True)
        assert st["bodies"] == K * wl.n and st["nonfinite_bodies"] == 0
        res.append(([x.double().cpu().numpy() for x in ten] +
                    [F.double().cpu().numpy(), T.double().cpu().numpy(), e.prev_velocities().double().cpu().numpy()],
                    e.wave_time))
    assert res[0][1] == res[1][1]
    tol = 2e-4 if dtype == torch.float32 else 1e-9   # as test_persistent_rollout_equals_stepwise
    for name, a, b in zip(("pos", "quat", "lin_vel", "ang_vel", "force", "torque", "prev"), res[0][0], res[1][0]):
        scale = np.abs(a).max(axis=1, keepdims=True) + 1e-3
        frac = float((np.abs(a - b) <= tol * scale).all(axis=1).mean())
        assert frac >= 0.995, (name, frac)


@gpu
@DTYPES
def test_no_behaviour_change_without_waves(dev, dtype):
    wl = W.heterogeneous_boxes(60_000, seed=5)
    cur = (0.2, 0.1, 0.0)

    def run(e):
        e.set_environment(current=cur, surface_z=0.1)
        e.set_prev(_t(wl.prev_lin, dtype, dev), _t(wl.prev_ang, dtype, dev))
        F, T = e.step(*[_t(a, dtype, dev) for a in (wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel)], wl.dt)
        return F.cpu(), T.cpu()

    flat = waves.regular(0.3, 6.0).components.copy()
    flat[:, 0] = 0.0                                                    # zero amplitude
    e0 = _engine(wl, dtype, dev, "direct")
    F0, T0 = run(e0)
    e1 = _engine(wl, dtype, dev, "direct")
    e1.set_wave_field(waves.WaveField(np.repeat(flat, 8, axis=0)))
    e1.set_wave_time(1e4)
    F1, T1 = run(e1)
    assert torch.equal(F0, F1) and torch.equal(T0, T1)
    # removing the field sends auto steps back to the tile kernel, bit-identical to an engine that never had one
    e2 = _engine(wl, dtype, dev, "auto")
    F2, T2 = run(e2)
    assert e2.last_kernel == "tile"
    e3 = _engine(wl, dtype, dev, "auto")
    e3.set_wave_field(waves.regular(0.3, 6.0))
    run(e3)
    assert e3.last_kernel == "direct"
    e3.set_wave_field(None)
    F3, T3 = run(e3)
    assert e3.last_kernel == "tile" and torch.equal(F2, F3) and torch.equal(T2, T3)


@gpu
def test_floating_cube_follows_a_long_wave(dev):
    """Physics: the C1 buoy (1 m cube, m = rho V / 2) in a regular deep-water wave whose period is >= 5x its natural
    heave period heaves with the surface: amplitude within 15 % of a, correlation with eta at the buoy > 0.95."""
    from silver2_isaacsim_b200 import HydroEngine

    wl = W.readme_buoy()
    m, area = float(wl.table[0, 10]), float(wl.table[0, 0] * wl.table[0, 1])
    t_heave = 2 * math.pi * math.sqrt(m / (wl.rho * wl.g * area))
    period, amp = 8.0, 0.15
    assert period >= 5 * t_heave
    field = waves.regular(amp, period)
    e = HydroEngine(1, dtype=torch.float64, device=dev)
    e.set_globals(wl.rho, wl.g)
    e.set_part_table(wl.table, wl.slot_type)
    e.set_wave_field(field)
    pos = torch.zeros(1, 3, dtype=torch.float64, device=dev)           # floating level at its waterline
    quat = torch.tensor([[0.0, 0.0, 0.0, 1.0]], dtype=torch.float64, device=dev)
    v, w = torch.zeros(1, 3, dtype=torch.float64, device=dev), torch.zeros(1, 3, dtype=torch.float64, device=dev)
    e.bind(pos, quat, v, w)
    n_steps = int(round(5 * period / wl.dt))
    trace = e.rollout_persistent(n_steps, wl.dt, gravity=wl.g, trace_every=1).cpu().numpy()[:, 0]
    assert e.wave_time == pytest.approx(n_steps * wl.dt, rel=1e-12)
    t = (np.arange(n_steps) + 1) * wl.dt
    eta = np.array([waves.evaluate(field, trace[k:k + 1, :3], t[k])[0, 0] for k in range(n_steps)])
    win = t > 3 * period
    z = trace[win, 2]
    heave = 0.5 * (z.max() - z.min())
    corr = float(np.corrcoef(z, eta[win])[0, 1])
    print(f"natural heave period {t_heave:.3f} s; heave amplitude {heave:.4f} m for a = {amp} m; correlation {corr:.4f}")
    assert abs(heave / amp - 1) <= 0.15 and corr > 0.95
