"""bench.py contract pieces that run without a GPU: the reference arm (the reference's CPU objects / the oracle port on the
host cores) prints ONE JSON line with the keys the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(built):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--width", "192", "--height", "288",
                        "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "fields/s" and d["value"] > 0
    for key in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config"):
        assert key in d
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["gpu_launches"] == 0
    # whole fields, and the workload string of our own arm (the driver compares the two arms' configs)
    assert "whole fields" in d["config"]["workload"] and "192x288" in d["config"]["workload"]
    assert "288 = 1.000 field" in d["cpu_baseline"]["sample"]
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"]["workload"] == bench.WORKLOAD % (192, 288)


def test_reference_arm_other_ranks_exit_silently(built):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                       text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_our_arm_fails_loudly_without_a_gpu(built):
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--pairs", "1"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_driver_secondary_never_takes_the_bench_line_down(built):
    """secondary.config5_mt_driver: without a GPU the sharded driver refuses (no CPU fallback) and the secondary reports
    that instead of raising; with a GPU it carries the jets/s of the window loop."""
    sys.path.insert(0, ROOT)
    import bench
    from slowflow_b200.api import load_library
    res = bench.run_driver_secondary(96, 64, 1, 3)
    assert "workload" in res and "error" not in res
    for tpg in (1, 2):
        leg = res["threads_per_gpu_%d" % tpg]
        if load_library().sfgpu_device_count() > 0:
            assert leg["jets_per_sec"] > 0 and abs(leg["windows_per_sec"] - 2 * leg["jets_per_sec"]) < 1e-9
        else:
            assert "no CUDA device" in leg["error"]


def test_dump_outputs_crops_the_stride_and_samples_large_outputs(tmp_path, monkeypatch):
    """--dump-outputs: the flows as the caller holds them, (pairs, H, W) float32; above the size limit a seeded sample of both
    components at the same positions, with those positions in sample_index.npy."""
    torch = pytest.importorskip("torch")
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    W, H, S, B = 61, 45, 64, 3
    wx = [torch.arange(S * H, dtype=torch.float32) + 1e4 * j for j in range(B)]
    wy = [-x for x in wx]
    ref = np.stack([x.numpy().reshape(H, S)[:, :W] for x in wx])
    bench.dump_outputs(str(tmp_path / "whole"), wx, wy, W, H, S)
    fx, fy = np.load(tmp_path / "whole" / "flow_x.npy"), np.load(tmp_path / "whole" / "flow_y.npy")
    assert fx.dtype == np.float32 and np.array_equal(fx, ref) and np.array_equal(fy, -ref)
    assert sorted(os.listdir(tmp_path / "whole")) == ["flow_x.npy", "flow_y.npy"]
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1024)
    monkeypatch.setattr(bench, "DUMP_SAMPLES", 100)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), wx, wy, W, H, S)
    ix = np.load(tmp_path / "s1" / "sample_index.npy")
    assert ix.dtype == np.float64 and 0 < len(ix) <= 100 and np.array_equal(ix, np.load(tmp_path / "s2" / "sample_index.npy"))
    k = ix.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "s1" / "flow_x.npy"), ref.reshape(-1)[k])
    assert np.array_equal(np.load(tmp_path / "s1" / "flow_y.npy"), -ref.reshape(-1)[k])


def test_reference_arm_rejects_dump_outputs(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not (tmp_path / "d").exists()
