"""CPU: the parts of bench.py's contract that need no GPU - the reference arm's JSON line (the reference's own kernels on the host
cores, keys the driver reads) and the per-block structure of the synthetic capture (equal work per GPU at every N)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-log2n", "18"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("MSamples/s") and d["unit"] == "MSamples/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"].startswith("2-FSK complex64")


def test_dump_outputs_are_reproducible(tmp_path):
    """--dump-outputs: the last step's center, pulse table and qad as float .npy files, the same from run to run"""
    import numpy as np

    runs = []
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                              "--cpu-log2n", "16", "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        runs.append({f[:-4]: np.load(str(tmp_path / d / f)) for f in os.listdir(str(tmp_path / d))})
    a, b = runs
    assert sorted(a) == ["center", "pulses", "pulses_index", "qad", "qad_index"] == sorted(b)
    for f in a:
        assert a[f].dtype in (np.float32, np.float64) and np.array_equal(a[f], b[f]), f
    assert len(a["qad"]) == 1 << 16 and np.array_equal(a["qad_index"], np.arange(1 << 16))
    assert a["pulses"][:, 1].sum() == (1 << 16) - 5                      # every sample but the tolerance lies in some pulse


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_capture_blocks_are_alike():
    sys.path.insert(0, ROOT)
    import bench

    n = 1 << 20
    base = bench.capture_gaps(n, 0)
    assert base == (int(0.40 * n), int(0.43 * n), int(0.97 * n))       # N = 1: the single-GPU capture of BASELINE configs[1]
    for rank in range(1, 8):
        g = bench.capture_gaps(n, rank)
        assert tuple(x - rank * n for x in g) == base                    # every block is built like the first
        assert rank * n <= g[0] < g[1] < g[2] < (rank + 1) * n
