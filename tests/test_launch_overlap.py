"""Launch overlap of consecutive captured tile kernels.

A tile launch captured right after another tile launch of the library in the same stream may load, compute and store
its first tile before the earlier grid has finished -- but only when the two launches' memory accesses do not
conflict.  The CPU tests check the access records and the decision without a device; the GPU tests check that
captured graphs compute exactly what the same steps compute when every boundary is serialised, and that every
aliasing pattern is refused (a launch that started early over aliased memory would race, so the refusal is asserted
directly, not left to a race to show up).
"""
import ctypes

import numpy as np
import pytest

MB = 1 << 20


# ---------------------------------------------------------------------------------------------------------------
# CPU: access records and the overlap decision
# ---------------------------------------------------------------------------------------------------------------
EAGER, SOLE_DEP, OTHER_DEPS, OTHER_CAPTURE = 0, 1, 2, 3
NAMES = ("pos", "quat", "lin", "ang", "prev", "coeff", "force", "torque", "wrench", "stats", "bitmap")


def _fake_launch(base, n):
    """Device addresses of an fp32 split-layout launch over n bodies, every array in its own 16 MB-aligned slot."""
    return {name: base + i * 16 * MB for i, name in enumerate(NAMES)}


def _decide(lib, earlier, n_e, later, n_l, relation=SOLE_DEP, bodies_per_robot=0):
    fn = lib.h2o_diag_overlap_decision
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int]
    arr = lambda d: (ctypes.c_void_p * 11)(*[d[k] for k in NAMES])
    e, l = arr(earlier), arr(later)
    return fn(ctypes.cast(e, ctypes.c_void_p), n_e, ctypes.cast(l, ctypes.c_void_p), n_l, bodies_per_robot, relation)


@pytest.fixture()
def two(built_lib):
    n = 1 << 14
    return built_lib, _fake_launch(1 << 40, n), _fake_launch(2 << 40, n), n


def test_independent_launches_overlap_only_when_captured_back_to_back(two):
    lib, a, b, n = two
    assert _decide(lib, a, n, b, n) == 1
    assert _decide(lib, a, n, b, n, relation=EAGER) == 0
    assert _decide(lib, a, n, b, n, relation=OTHER_DEPS) == 0
    assert _decide(lib, a, n, b, n, relation=OTHER_CAPTURE) == 0


def test_shared_read_only_inputs_do_not_conflict(two):
    lib, a, b, n = two
    for k in ("pos", "quat", "lin", "ang", "coeff"):
        assert _decide(lib, a, n, dict(b, **{k: a[k]}), n) == 1, k


@pytest.mark.parametrize("src", ["force", "torque", "prev"])
@pytest.mark.parametrize("dst", ["pos", "quat", "lin", "ang", "prev", "coeff"])
def test_read_after_write_is_refused(two, src, dst):
    lib, a, b, n = two
    assert _decide(lib, a, n, dict(b, **{dst: a[src]}), n) == 0


@pytest.mark.parametrize("dst", ["force", "torque", "prev"])
@pytest.mark.parametrize("src", ["pos", "quat", "lin", "ang", "prev", "coeff"])
def test_write_after_read_is_refused(two, src, dst):
    lib, a, b, n = two
    assert _decide(lib, a, n, dict(b, **{dst: a[src]}), n) == 0


@pytest.mark.parametrize("k", ["force", "torque", "stats", "bitmap"])
def test_write_after_write_is_refused(two, k):
    lib, a, b, n = two
    assert _decide(lib, a, n, dict(b, **{k: a[k]}), n) == 0


def test_same_engine_twice_is_refused(two):
    lib, a, _, n = two
    assert _decide(lib, a, n, a, n) == 0


def test_intervals_are_half_open_and_cover_the_tiled_bodies(two):
    lib, a, b, n = two
    force_bytes = n * 3 * 4
    # the later launch reads from the byte right after the earlier force array, then from its last byte
    assert _decide(lib, a, n, dict(b, pos=a["force"] + force_bytes), n) == 1
    assert _decide(lib, a, n, dict(b, pos=a["force"] + force_bytes - 16), n) == 0
    # bodies past the last full tile belong to the per-body kernel: not in the tile launch's record
    n_odd = n + 100
    tiled = (n_odd // 128) * 128
    assert _decide(lib, a, n_odd, dict(b, pos=a["force"] + tiled * 3 * 4), n) == 1
    assert _decide(lib, a, n_odd, dict(b, pos=a["force"] + (tiled - 4) * 3 * 4), n) == 0


def test_redo_bitmap_words_of_a_shared_bitmap(two):
    lib, a, b, n = two
    # the same bitmap allocation: both launches cover bodies from 0, so their words meet
    assert _decide(lib, a, n, dict(b, bitmap=a["bitmap"]), n) == 0
    assert _decide(lib, a, n, dict(b, bitmap=a["bitmap"] + n // 8), n) == 1


def test_robot_wrench_is_a_write(two):
    lib, a, b, n = two
    bpr = 19
    n_r = (n // 76) * 76
    assert _decide(lib, a, n_r, b, n_r, bodies_per_robot=bpr) == 1
    assert _decide(lib, a, n_r, dict(b, pos=a["wrench"]), n_r, bodies_per_robot=bpr) == 0
    assert _decide(lib, a, n_r, dict(b, wrench=a["pos"]), n_r, bodies_per_robot=bpr) == 0
    assert _decide(lib, a, n_r, dict(b, wrench=a["wrench"]), n_r, bodies_per_robot=bpr) == 0


# ---------------------------------------------------------------------------------------------------------------
# GPU: captured graphs against serialised execution, bit for bit
# ---------------------------------------------------------------------------------------------------------------
def _last_overlap(eng):
    fn = eng._lib.h2o_diag_last_overlap
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p]
    return fn(eng._h)


class Scene:
    """Engines over resident tensors; every run starts from the same state (carried velocities and the tensors the
    steps or the foreign kernels write)."""

    def __init__(self, torch):
        self.torch = torch
        self.dev = torch.device("cuda", 0)
        self.engines = []
        self.state = []   # (tensor, saved copy)
        self.prev0 = []   # (engine, prev_lin, prev_ang)

    def tensor(self, a):
        t = self.torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32), device=self.dev)
        self.state.append((t, t.clone()))
        return t

    def engine(self, wl, inputs=None, outputs=None, stats=False, robot=False):
        from silver2_isaacsim_b200 import HydroEngine

        e = HydroEngine(wl.n, device=self.dev)
        e.set_workload_params(wl)
        if stats:
            e.enable_stats(True)
        pos, quat, lin, ang = inputs or (self.tensor(wl.pos), self.tensor(wl.quat_xyzw), self.tensor(wl.lin_vel),
                                         self.tensor(wl.ang_vel))
        F, T = outputs or (None, None)
        out = e.bind(pos, quat, lin, ang, out_force=F, out_torque=T, robot_wrench=robot)
        e.out = out
        for t in out:
            self.state.append((t, t.clone()))
        self.prev0.append((e, self.tensor(wl.prev_lin), self.tensor(wl.prev_ang)))
        e.dt = wl.dt
        self.engines.append(e)
        return e

    def restore(self):
        torch = self.torch
        torch.cuda.synchronize()
        for t, saved in self.state:
            t.copy_(saved)
        for e, pl, pa in self.prev0:
            e.set_prev(pl, pa)
        for e in self.engines:
            e.stats(reset=True)
        torch.cuda.synchronize()

    def results(self):
        self.torch.cuda.synchronize()
        out = [t.cpu().numpy().copy() for e in self.engines for t in e.out]
        out += [e.prev_velocities().cpu().numpy().copy() for e in self.engines]
        return out

    def warm(self, seq):
        for fn in seq:
            fn()
        self.torch.cuda.synchronize()

    def graph(self, seq):
        torch = self.torch
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            self.warm(seq)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for fn in seq:
                fn()
        return g

    def run_graph(self, g):
        self.restore()
        g.replay()
        return self.results()

    def run_eager(self, seq):
        self.restore()
        for fn in seq:
            fn()
        return self.results()


def _equal(xs, ys):
    assert len(xs) == len(ys)
    for i, (x, y) in enumerate(zip(xs, ys)):
        assert x.shape == y.shape
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), f"array {i} differs"


@pytest.fixture()
def torch_gpu():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch


def _noop(torch):
    scratch = torch.zeros(4, device="cuda")
    return lambda: scratch.mul_(1.0)


def _boxes(n, seed):
    from silver2_isaacsim_b200 import workloads as W
    return W.heterogeneous_boxes(n, seed=W.SEED_BASE + seed)


def _hexapods(n_envs, seed):
    from silver2_isaacsim_b200 import workloads as W
    return W.hexapod_envs(n_envs, seed=W.SEED_BASE + seed)


@pytest.mark.gpu
@pytest.mark.parametrize("n_engines", [6, 2])
@pytest.mark.parametrize("kind", ["boxes", "boxes_stats", "boxes_tail", "hexapods_wrench", "hexapods_wrench_tail"])
def test_rotation_graph_matches_serialised_steps(torch_gpu, n_engines, kind):
    torch = torch_gpu
    sc = Scene(torch)
    for k in range(n_engines):
        if kind.startswith("boxes"):
            n = (1 << 18) + (52 if kind == "boxes_tail" else 0)
            e = sc.engine(_boxes(n, 10 + k), stats=kind == "boxes_stats")
        else:
            envs = 2048 + (2 if kind.endswith("tail") else 0)
            e = sc.engine(_hexapods(envs, 20 + k), robot=True)
        e.set_kernel("tile")
    rounds = 3
    seq = [(lambda e=e: e.step_bound(e.dt)) for _ in range(rounds) for e in sc.engines]
    noop = _noop(torch)
    serial = [f for fn in seq for f in (fn, noop)]
    g = sc.graph(seq)
    overlapped = [_last_overlap(e) for e in sc.engines]
    g_ref = sc.graph(serial)
    assert [_last_overlap(e) for e in sc.engines] == [0] * n_engines
    if kind.endswith("tail"):
        assert overlapped == [0] * n_engines  # the per-body tail kernel sits between the tile launches
    else:
        assert overlapped == [1] * n_engines
    stats_ref = None
    ref = sc.run_graph(g_ref)
    if kind == "boxes_stats":
        stats_ref = [e.stats() for e in sc.engines]
    got = sc.run_graph(g)
    _equal(got, ref)
    _equal(got, sc.run_eager(seq))
    if stats_ref is not None:
        for e, s in zip(sc.engines, stats_ref):
            s2 = e.stats()
            for key in s:
                assert s2[key] == pytest.approx(s[key], rel=1e-12), key


def _pair_check(torch, sc, seq, later):
    """Graph of `seq` against the same steps run eagerly (every boundary serialised): bit for bit; `later` (the
    engine whose launch follows the aliasing one) must have been captured to wait first."""
    g = sc.graph(seq)
    assert _last_overlap(later) == 0
    got = sc.run_graph(g)
    _equal(got, sc.run_eager(seq))
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("src", ["force", "torque"])
def test_read_after_write_across_engines_waits(torch_gpu, src):
    torch = torch_gpu
    sc = Scene(torch)
    a = sc.engine(_boxes(1 << 18, 30))
    wl_b = _boxes(1 << 16, 31)
    # B reads the rows A writes in its last round (the tail of A's output): a launch that started early would
    # read them before A stored them
    tail = a.out[0 if src == "force" else 1][-wl_b.n:]
    b = sc.engine(wl_b, inputs=(tail, sc.tensor(wl_b.quat_xyzw), tail, sc.tensor(wl_b.ang_vel)))
    seq = [lambda: a.step_bound(a.dt), lambda: b.step_bound(b.dt)] * 2
    _pair_check(torch, sc, seq, b)


@pytest.mark.gpu
def test_write_after_read_across_engines_waits(torch_gpu):
    torch = torch_gpu
    sc = Scene(torch)
    a = sc.engine(_boxes(1 << 18, 40))
    wl_b = _boxes(1 << 16, 41)
    pos_a = a._bound[0]
    lin_a = a._bound[2]
    # B writes its force / torque over the rows of A's inputs that A reads in its last round
    b = sc.engine(wl_b, outputs=(pos_a[-wl_b.n:], lin_a[-wl_b.n:]))
    seq = [lambda: a.step_bound(a.dt), lambda: b.step_bound(b.dt), lambda: a.step_bound(a.dt)]
    _pair_check(torch, sc, seq, b)


@pytest.mark.gpu
def test_same_engine_twice_waits(torch_gpu):
    torch = torch_gpu
    sc = Scene(torch)
    a = sc.engine(_boxes(1 << 18, 50))
    seq = [lambda: a.step_bound(a.dt)] * 3  # each step reads the velocities the one before wrote
    _pair_check(torch, sc, seq, a)


@pytest.mark.gpu
def test_foreign_writer_between_launches_waits(torch_gpu):
    torch = torch_gpu
    sc = Scene(torch)
    a = sc.engine(_boxes(1 << 18, 60))
    b = sc.engine(_boxes(1 << 18, 61))
    pos_b = b._bound[0]
    seq = [lambda: a.step_bound(a.dt), lambda: pos_b.add_(0.25), lambda: b.step_bound(b.dt)]
    _pair_check(torch, sc, seq, b)


@pytest.mark.gpu
@pytest.mark.parametrize("who", ["foreign_kernel", "library_step"])
def test_cross_stream_join_waits(torch_gpu, who):
    """A second stream joins the capture through an event; the work it adds must order B after it."""
    torch = torch_gpu
    sc = Scene(torch)
    a = sc.engine(_boxes(1 << 18, 70))
    b = sc.engine(_boxes(1 << 18, 71))
    c = sc.engine(_boxes(1 << 16, 72))
    pos_b = b._bound[0]
    other = torch.cuda.Stream(device=sc.dev)

    def joined():
        cur = torch.cuda.current_stream(sc.dev)
        other.wait_stream(cur)
        with torch.cuda.stream(other):
            if who == "foreign_kernel":
                pos_b.add_(0.25)
            else:
                c.step_bound(c.dt)
        cur.wait_stream(other)

    seq = [lambda: a.step_bound(a.dt), joined, lambda: b.step_bound(b.dt)]
    _pair_check(torch, sc, seq, b)
