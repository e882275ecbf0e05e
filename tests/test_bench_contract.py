"""bench.py's JSON contract on the parts that run without a GPU: the reference arm (oracle port on the host
cores), the refusal of our arm to run without a device, the argument checks and --dump-outputs' file layout;
on the GPU, that --dump-outputs writes the images of the timed renders."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def run(*args, env=None):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, cwd=ROOT,
                          timeout=600, env=env)


def test_reference_arm_prints_one_contract_line():
    p = run("--impl", "reference", "--workload", "c1", "--steps", "2", "--warmup", "1", "--ref-seconds", "3")
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Mrays/s (all bounces)" and d["unit"] == "Mrays/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None and d["dtype"] == "f64"
    assert d["config"]["workload"].startswith("diffuse_single_sphere") or "512" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "spp" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_runs_on_rank_zero_only():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = run("--impl", "reference", "--workload", "c1", "--gpus", "2", "--steps", "1", "--warmup", "0", env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_our_arm_refuses_to_run_without_a_device():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    p = run("--steps", "1", "--warmup", "0")
    assert p.returncode != 0
    assert "no CPU fallback" in (p.stderr + p.stdout)


def test_argument_checks():
    p = run("--steps", "0")
    assert p.returncode == 2 and "--steps" in p.stderr
    p = run("--impl", "reference", "--dump-outputs", "unused")
    assert p.returncode == 2 and "--dump-outputs" in p.stderr


def test_dump_outputs_writes_small_images_whole_and_samples_large_ones(tmp_path, monkeypatch):
    # bench.py sets these on import unless they are set already: set here, they are restored after the test
    monkeypatch.setenv("NCCL_DEBUG", "WARN")
    monkeypatch.setenv("NCCL_DEBUG_FILE", "/dev/stderr")
    monkeypatch.syspath_prepend(str(ROOT))
    import bench
    rng = np.random.default_rng(1)
    small = rng.random((24, 40, 3), dtype=np.float32)
    big = rng.random((2160, 3840, 3), dtype=np.float32)   # the 4K image of the default workload: 99.5 MB
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, [("small", small), ("big", big)])
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["big.npy", "big_pixels.npy", "small.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 64 << 20
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)
    rows, idx = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "a" / "big_pixels.npy")
    assert rows.dtype == np.float32 and idx.dtype == np.float64 and rows.shape == (idx.size, 3)
    pix = idx.astype(np.int64)
    assert np.array_equal(pix, idx) and (np.diff(pix) > 0).all() and pix[0] >= 0 and pix[-1] < 2160 * 3840
    assert idx.size > 2160 * 3840 // 8
    assert np.array_equal(rows, big.reshape(-1, 3)[pix])
    for f in files:   # the same sample every time
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


@pytest.mark.gpu
def test_dumped_outputs_are_the_timed_renders(tmp_path, native_built):
    p = run("--workload", "c1", "--steps", "3", "--warmup", "1", "--no-per-config", "--no-cpu-baseline",
            "--dump-outputs", str(tmp_path))
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3
    assert sorted(f.name for f in tmp_path.iterdir()) == ["diffuse_single_sphere.npy"]
    img = np.load(tmp_path / "diffuse_single_sphere.npy")
    assert img.dtype == np.float32 and img.shape == (512, 512, 3)
    # the same samples through the one-GPU render call
    from rayrs_b200 import api, scenes
    cfg = scenes.CONFIGS["c1"]
    spec = cfg.specs()[0]
    sc = spec.scene(scenes.synthetic_hdri(2048, 1024), device=0, with_f64=False)
    ref = api.render_gpu(spec.camera(), sc, cfg.spp, cfg.max_bounces)
    sc.close()
    assert np.max(np.abs(img - ref) / (np.abs(ref) + 1e-3)) <= 1e-4
