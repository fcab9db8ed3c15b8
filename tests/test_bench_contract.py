"""bench.py's contract pieces that do not need a GPU: the reference arm (--impl reference) runs the reference's own CPU generator on
a bounded sample and prints one JSON line with the keys the driver reads; the B200 arm refuses to run without a device."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line(oracle):
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg5-small", "--steps", "2",
                        "--warmup", "1", "--gpus", "1"], capture_output=True, text=True, timeout=600, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "pixel-diffs/sec" and line["unit"] == "pixel-diffs/s"
    assert line["higher_is_better"] is True and line["steps"] == 2 and line["warmup"] == 1 and line["value"] > 1e6
    assert line["e2e"] == {"value": line["value"], "unit": "pixel-diffs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] == 1 and cb["value"] == line["value"] and "library images" in cb["sample"]
    assert 0.0 < cb["visited_fraction"] <= 1.0
    # the same `config` object as the B200 arm prints for this workload (bench.describe), so that the driver can pair the lines
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.describe(bench.WORKLOADS["cfg5-small"], "cfg5-small", 1)
    assert line["config"]["cell_shape"] == "Puzzle"


def test_other_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True, text=True,
                       timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_reference_arm_refuses_to_dump_outputs(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
    assert p.returncode != 0 and "--dump-outputs" in p.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_b200_arm_dumps_the_same_outputs_on_every_run(tmp_path):
    """--dump-outputs: the best-fit grid of the last timed step, float64, identical for two runs with the same arguments."""
    import numpy as np
    grids = []
    for run in range(2):
        out = tmp_path / ("run%d" % run)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                            "--workload", "cfg4-small", "--configs", "none", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads(p.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2
        assert sorted(os.listdir(out)) == ["cfg4-small_best_fits0.npy"]
        g = np.load(out / "cfg4-small_best_fits0.npy")
        assert g.dtype == np.float64 and g.shape == (11, 17)  # 1080 x 1920 in 128 px cells (GridGenerator's grid, edge ring included)
        assert int((g >= 0).sum()) == line["valid_cells"] and g.max() < 1000 and np.array_equal(g, np.round(g))
        grids.append(g)
    assert np.array_equal(grids[0], grids[1])


def test_b200_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg4-small", "--configs", "none"], capture_output=True,
                       text=True, timeout=300, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)
