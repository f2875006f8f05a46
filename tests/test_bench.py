"""bench.py's --dump-outputs and --steps: the dumped rays are the traced rays of the seeded source at the sampled
indices (recomputed here on the CPU oracle), identical from run to run, and --steps is the number of steps timed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import chains, pyref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("x", "y", "z", "l", "m", "n", "ux", "uy", "uz", "hpd")
N = 300_000                 # more than bench.DUMP_RAYS: the dump is a sample


def bench_module():
    """bench.py for its constants and ``dump_sample`` (importing it turns bytecode writing off: restore that)."""
    old = sys.dont_write_bytecode
    import bench
    sys.dont_write_bytecode = old
    return bench


def run_bench(*args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                       timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


def load_dump(path):
    assert sorted(os.listdir(path)) == sorted(n + ".npy" for n in NAMES)
    out = {n: np.load(os.path.join(path, n + ".npy")) for n in NAMES}
    for n, a in out.items():
        assert a.dtype == np.float64 and a.shape == ((1,) if n == "hpd" else (1 << 18,)), n
    return out


def assert_dump_is_the_trace(dump, source_rows):
    """The oracle traces the same source with the bench's chain: the sampled rows must be its rows bit for bit."""
    b = bench_module()
    rays = [np.array(r, dtype=np.float64) for r in source_rows]
    chains.run_steps_cpu(rays, chains.wolter1_steps(b.R0, b.Z0, b.PSI))
    idx = b.dump_sample(N)
    for k, name in enumerate(b.DUMP_ROWS, 1):
        assert np.array_equal(dump[name], rays[k][idx], equal_nan=True), name
    return pyref.hpd(rays)


def test_reference_arm_dump_is_the_trace_and_repeatable(tmp_path):
    lines = [run_bench("--impl", "reference", "--warmup", "1", "--steps", "3", "--ref-rays", str(N),
                       "--dump-outputs", str(tmp_path / run)) for run in ("a", "b")]
    a, b = load_dump(tmp_path / "a"), load_dump(tmp_path / "b")
    for name in NAMES:
        assert np.array_equal(a[name], b[name], equal_nan=True), name
    bm = bench_module()
    np.random.seed(0)
    hpd = assert_dump_is_the_trace(a, pyref.subannulus(bm.RIN, bm.ROUT, 2 * np.pi, N, zhat=-1.))
    assert a["hpd"][0] == hpd == lines[0]["config"]["hpd"]
    assert lines[0]["steps"] == 3


@pytest.mark.gpu
def test_engine_dump_is_the_trace_and_steps_are_timed(tmp_path):
    """The engine arm at two step counts: twice the steps launch twice the kernels in the timed region, and the dump
    of the last timed step equals the oracle's trace of the same Philox source."""
    import torch
    import pyxfocus_b200 as pxf
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    common = ["--gpus", "1", "--warmup", "3", "--rays", str(N), "--no-e2e", "--no-configs", "--no-cpu-baseline"]
    two = run_bench(*common, "--steps", "2")
    four = run_bench(*common, "--steps", "4", "--dump-outputs", str(tmp_path))
    assert four["steps"] == 4 and four["gpu_launches"] == 2 * two["gpu_launches"] > 0
    b = bench_module()
    src = pxf.sources.subannulus(b.RIN, b.ROUT, 2 * np.pi, N, zhat=-1., rng="philox", seed=0, first=0, device="cuda:0")
    dump = load_dump(tmp_path)
    hpd = assert_dump_is_the_trace(dump, pxf.sources.to_numpy(src))
    assert dump["hpd"][0] == four["config"]["hpd"]
    assert dump["hpd"][0] == pytest.approx(hpd, rel=1e-9)


def test_steps_must_be_positive():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 2 and "--steps" in p.stderr
