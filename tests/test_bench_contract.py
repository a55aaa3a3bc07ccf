"""bench.py contract (CPU side): the reference arm prints exactly one JSON line with the agreed keys."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


import pytest


@pytest.mark.parametrize("kind", ["port", "auto"])
def test_reference_arm_line(oracle, kind):
    """--impl reference: the unmodified Numba reference (live tree or the bytecode staged in oracle/_ref)
    when it is available, else the C port; either way one JSON line on the B200 arm's config."""
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3",
                          "--warmup", "1", "--bodies-per-gpu", "65536", "--ref-kind", kind],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-1500:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "body-force updates/sec" and d["unit"] == "bodies/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and "workload" in d["config"]
    from oracle import ref_numba
    want = "reference" if (kind == "auto" and ref_numba.available()) else "port"
    assert d["cpu_baseline"]["kind"] == want and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["config"]["bodies_per_gpu"] == 65536 and d["steps"] == 3  # the B200 arm's config, not a capped one
    assert d["e2e"] == {"value": d["value"], "unit": "bodies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 1e5 and d["gpu_launches"] == 0


def test_reference_arm_other_ranks_stay_silent(oracle):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=120, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_b200_arm_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode != 0 and "no CPU path" in (res.stderr + res.stdout)
    assert res.stdout.strip() == ""  # no fabricated line


def test_tools_and_harnesses_compile(tmp_path):
    """Every stand-alone script (tools/, tests/harness/, examples/) at least byte-compiles."""
    import glob
    import py_compile

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    scripts = [p for d in ("tools", os.path.join("tests", "harness"), "examples")
               for p in glob.glob(os.path.join(root, d, "*.py"))]
    assert len(scripts) >= 15
    for p in scripts:
        py_compile.compile(p, doraise=True, cfile=str(tmp_path / (os.path.basename(p) + "c")))


def test_step_regions_launch_exactly_the_steps():
    """The timed steps are exactly --steps, cycling through the batches in order across the regions."""
    import bench

    ran = []
    fns = [lambda b=b: ran.append(b) for b in range(6)]
    for steps, regions in ((200, 20), (23, 5), (7, 7), (1, 1)):
        ran.clear()
        regs, counts, _ = bench.build_step_regions(None, fns, steps, regions, None, use_graph=False)
        assert len(regs) == regions and counts.sum() == steps and counts.min() >= 1
        for r in regs:
            r()
        assert ran == [i % 6 for i in range(steps)]


def test_dump_outputs_writes_a_seeded_sample_above_the_limit(tmp_path):
    import bench
    import torch

    g = torch.Generator().manual_seed(1)
    arrays = {"force": torch.randn(1000, 3, generator=g), "torque": torch.randn(1000, 3, generator=g).double()}
    info = bench.dump_outputs(str(tmp_path / "all"), arrays)
    assert info["rows"] == "all" and info["files"] == ["force.npy", "torque.npy"]
    F = np.load(tmp_path / "all" / "force.npy")
    assert F.dtype == np.float32 and np.array_equal(F, arrays["force"].numpy())
    limit = 100 * (3 * 4 + 3 * 8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, limit_bytes=limit)
    F, T = np.load(tmp_path / "a" / "force.npy"), np.load(tmp_path / "a" / "torque.npy")
    assert F.shape == (100, 3) and T.shape == (100, 3) and T.dtype == np.float64
    assert F.nbytes + T.nbytes <= limit
    rows = [int(np.nonzero((arrays["force"].numpy() == f).all(axis=1))[0][0]) for f in F]
    assert np.array_equal(T, arrays["torque"].numpy()[rows])  # the same rows from every array
    assert np.array_equal(F, np.load(tmp_path / "b" / "force.npy"))  # the same sample every run


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(oracle, tmp_path):
    """--dump-outputs holds what step --steps returned (batch (K - 1) % batches), the same from run to run."""
    import torch
    from silver2_isaacsim_b200 import workloads as W
    from tests import scoring

    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    n = 1 << 16
    out = {}
    for tag, steps in (("k7", 7), ("k8", 8), ("k7_again", 7)):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                              "--bodies-per-gpu", str(n), "--no-extra", "--no-e2e", "--no-cpu-baseline",
                              "--dump-outputs", str(tmp_path / tag)], capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-1500:]
        d = json.loads(res.stdout)
        assert d["steps"] == steps and d["gpu_launches"] == steps
        assert sum(d["extra"]["timing"]["steps_per_region"]) == steps
        assert d["extra"]["dump_outputs"]["rows"] == "all"
        out[tag] = [np.load(tmp_path / tag / f) for f in ("force.npy", "torque.npy")]
    for a, b in zip(out["k7"], out["k7_again"]):
        assert a.dtype == np.float32 and a.shape == (n, 3) and a.tobytes() == b.tobytes()
    # batch b is heterogeneous_boxes(seed=SEED_BASE + 3 + b); every batch has been stepped before the timed
    # steps, so its previous velocities are its velocities
    for tag, batch in (("k7", 0), ("k8", 1)):
        wl = W.heterogeneous_boxes(n, seed=W.SEED_BASE + 3 + batch)
        ref = oracle.step(wl.ctor_rows(), wl.masses(), wl.pos, wl.quat_xyzw, wl.lin_vel, wl.ang_vel, wl.lin_vel,
                          wl.ang_vel, wl.dt)
        scoring.assert_fp32(out[tag][0], ref.force, tag + " force")
        scoring.assert_fp32(out[tag][1], ref.torque, tag + " torque")
