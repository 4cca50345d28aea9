"""bench.py's command line: the reference arm (`--impl reference`, CPU) prints ONE JSON line with the expected
keys; the CUDA arm's --dump-outputs and --steps (-m gpu)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert d["metric"] == "raft_corr_build_plus_12iter_lookup_frame_pairs_per_s_1080p"
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] and "sample" in d["cpu_baseline"]
    # the arm runs the STOCK class on the FULL configuration every step: no slicing, no extrapolation
    assert "1 full frame pair 1920x1088" in d["cpu_baseline"]["sample"] and "stock torchvision CorrBlock" in d["cpu_baseline"]["sample"]
    assert "scaled" not in d["cpu_baseline"]["sample"] and "1/" not in d["cpu_baseline"]["sample"]
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"]["workload"] == bench.WORKLOAD and d["config"]["fmap"] == [1, 256, 136, 240]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_and_steps(tmp_path):
    """--dump-outputs writes the last timed step's results as float32 .npy (64 MB at most), identical over two runs
    with the same arguments; --steps sets the number of timed steps (the timed launches scale with it)."""
    runs = {}
    for name, steps in (("a", 2), ("b", 2), ("c", 3)):
        d = tmp_path / name
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3",
                              "--no-alt", "--no-gop", "--no-gpu-baseline", "--no-cpu-baseline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
        assert len(lines) == 1
        runs[name] = (json.loads(lines[0]), {f.stem: np.load(f) for f in d.glob("*.npy")})
    line, arrays = runs["a"]
    assert line["steps"] == 2 and runs["c"][0]["steps"] == 3
    assert runs["c"][0]["gpu_launches"] * 2 == line["gpu_launches"] * 3
    assert sorted(arrays) == ["lookup"] + [f"pyramid_level{l}" for l in range(4)]
    assert arrays["lookup"].shape == (1, 324, 136, 240)
    for l in range(4):
        assert arrays[f"pyramid_level{l}"].shape == (64, 1, 136 >> l, 240 >> l)
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for k, a in arrays.items():
        assert a.dtype == np.float32 and np.isfinite(a).all() and np.abs(a).max() > 0, k
        assert np.array_equal(a, runs["b"][1][k]), k
