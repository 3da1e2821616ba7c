"""bench.py contract on CPU: the reference arm prints ONE JSON line with the agreed keys (the
GPU arm is exercised by the driver and by tools/gpu_round.sh)."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def test_reference_arm_json_line():
    env = dict(os.environ, AGCM_BENCH_REF_BUDGET_S="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "aes_gcm_enc_tag_throughput" and d["unit"] == "GB/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, env=env, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_below_one_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_dump_outputs_files(tmp_path):
    """--dump-outputs: the tag and seeded 4 KiB ciphertext windows, as float32, within 64 MB."""
    import numpy as np
    import torch
    import bench
    g = torch.Generator()
    g.manual_seed(0)
    ct = torch.randint(0, 256, (1 << 24,), dtype=torch.uint8, generator=g)
    tag = torch.arange(16, dtype=torch.uint8)
    bench.dump_outputs(str(tmp_path), 0, 1, ct, tag)
    assert sorted(os.listdir(tmp_path)) == ["ciphertext_sample.npy", "tag.npy"]
    assert np.load(tmp_path / "tag.npy").tolist() == list(range(16))
    got = np.load(tmp_path / "ciphertext_sample.npy")
    assert got.dtype == np.float32 and got.shape == (bench.DUMP_WINDOWS, bench.DUMP_WINDOW)
    pick = np.sort(np.random.default_rng(3).choice(ct.numel() // bench.DUMP_WINDOW, bench.DUMP_WINDOWS, replace=False))
    want = ct.numpy().reshape(-1, bench.DUMP_WINDOW)[pick]
    assert np.array_equal(got, want)
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    # one file per rank when the stream is split, the tag once
    bench.dump_outputs(str(tmp_path / "n2"), 1, 2, ct, tag)
    assert os.listdir(tmp_path / "n2") == ["ciphertext_sample_rank1.npy"]
    assert np.load(tmp_path / "n2" / "ciphertext_sample_rank1.npy").shape == (bench.DUMP_WINDOWS // 2, bench.DUMP_WINDOW)
