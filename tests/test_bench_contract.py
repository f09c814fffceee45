"""CPU: the bench contract that can be exercised without a GPU -- `bench.py --impl reference` (the reference arm the
driver launches next to ours) prints ONE JSON line with the agreed keys, times the unmodified reference when
baseline/_ref or /root/reference exists (else the oracle port, and says which), and non-zero ranks of a torchrun
launch exit 0 without work.  Run on a tiny architecture so that it takes seconds."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--impl", "reference", "--config", "tiny_swin", "--tris", "64", "--resolution", "64", "--total-views", "2",
        "--steps", "2", "--warmup", "1"]


def _run(extra_env=None, gpus=1):
    env = dict(os.environ, **(extra_env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", str(gpus)] + ARGS,
                          capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)


def test_reference_arm_prints_one_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    j = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in j, k
    assert j["impl"] == "reference" and j["unit"] == "frames/s" and j["higher_is_better"] is True
    assert j["vs_baseline"] is None and j["data"] == "synthetic" and j["dtype"] == "f32" and j["scaling"] == "strong"
    assert j["value"] > 0 and j["ms_per_step"] > 0 and j["gpu_launches"] == 0
    assert "workload" in j["config"] and "model" not in j["config"]
    cb = j["cpu_baseline"]
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(cb) and cb["value"] == j["value"]
    have_ref = any(os.path.isdir(os.path.join(p, "renderformer", "models"))
                   for p in (os.path.join(ROOT, "baseline", "_ref"), "/root/reference"))
    assert cb["kind"] == ("reference" if have_ref else "port") and cb["cores"] == (os.cpu_count() or 1)
    e = j["e2e"]
    assert e["value"] == j["value"] and e["unit"] == j["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, gpus=2)
    assert r.returncode == 0 and r.stdout.strip() == "", (r.stdout, r.stderr[-500:])


def test_dump_outputs_is_whole_or_a_fixed_sample_within_64_mb(tmp_path, monkeypatch):
    """--dump-outputs: a job's images go out whole while they fit in 64 MB, else as the same seeded pixel sample on
    every run (here pixel value = flat pixel index, so the sample shows which pixels it holds)."""
    import numpy as np
    import torch
    for k in ("NCCL_DEBUG", "NCCL_DEBUG_FILE"):  # importing bench sets these; monkeypatch restores them after the test
        had = os.environ.get(k)
        monkeypatch.setenv(k, "")
        if had is None:
            monkeypatch.delenv(k)
        else:
            monkeypatch.setenv(k, had)
    import bench
    small = torch.rand(1, 2, 8, 8, 3)
    p = bench.dump_images(small, str(tmp_path / "small"))
    assert os.path.basename(p) == "image.npy" and np.array_equal(np.load(p), small.numpy())
    npix = 32 * 512 * 512  # the metric's job: 32 views at 512^2, 100 MB of float32
    big = torch.arange(npix, dtype=torch.float32)[:, None].expand(npix, 3).reshape(1, 32, 512, 512, 3)
    p1, p2 = bench.dump_images(big, str(tmp_path / "a")), bench.dump_images(big, str(tmp_path / "b"))
    a = np.load(p1)
    assert os.path.basename(p1) == "image_sample.npy" and os.path.getsize(p1) <= 64_000_000
    assert a.dtype == np.float32 and a.shape[1] == 3 and a.shape[0] > npix // 2
    assert np.array_equal(a, np.load(p2))
    idx = a[:, 0].astype(np.int64)
    assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < npix and (a == a[:, :1]).all()


def test_steps_below_one_are_rejected():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert r.returncode != 0 and "--steps" in r.stderr
