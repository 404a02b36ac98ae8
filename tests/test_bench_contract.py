"""bench.py: the reference arm (`--impl reference`) runs without a GPU and prints the contract's JSON line; what
`--dump-outputs` writes (on CPU tensors, and through the CUDA arm on the GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "cirim_320x320x15coil_slices_per_sec" and d["unit"] == "slices/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and abs(d["value"] - 1e3 / d["ms_per_step"]) < 1e-6 * d["value"] + 1e-9  # 1 slice per step
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_dump_outputs_files(tmp_path):
    """bench.dump_outputs on CPU tensors: the final estimate in full, the same seeded positions of every estimate, and
    a seeded sample of the reconstruction once it exceeds DUMP_RECON_MAX values."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    g = torch.Generator().manual_seed(0)
    casc = [[torch.randn(2, 320, 320, dtype=torch.complex64, generator=g) for _ in range(8)] for _ in range(5)]
    bench.dump_outputs(str(tmp_path / "a"), casc)
    bench.dump_outputs(str(tmp_path / "b"), casc)
    rec, est = np.load(tmp_path / "a" / "reconstruction.npy"), np.load(tmp_path / "a" / "estimates_sample.npy")
    assert rec.dtype == est.dtype == np.float32
    assert np.array_equal(rec, torch.view_as_real(casc[-1][-1]).numpy())
    assert est.shape == (5, 8, bench.DUMP_ESTIMATE_SAMPLES, 2)
    idx = bench._seeded_sample(2 * 320 * 320, bench.DUMP_ESTIMATE_SAMPLES)
    assert np.array_equal(est[3, 6], torch.view_as_real(casc[3][6].reshape(-1))[idx].numpy())
    assert np.array_equal(est, np.load(tmp_path / "b" / "estimates_sample.npy"))
    big = torch.randn(bench.DUMP_RECON_MAX // (320 * 320) + 1, 320, 320, dtype=torch.complex64, generator=g)
    bench.dump_outputs(str(tmp_path / "c"), casc, big)
    assert np.load(tmp_path / "c" / "reconstruction.npy").shape == (bench.DUMP_RECON_MAX, 2)
    assert sum(f.stat().st_size for f in (tmp_path / "c").iterdir()) <= 64 * 2 ** 20


@pytest.mark.gpu
def test_dump_outputs_cli_repeats(tmp_path):
    """--dump-outputs on the CUDA arm: shapes of the last step's outputs, and the same arrays for a different --steps."""
    import numpy as np

    for steps, d in ((1, "a"), (2, "b")):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0",
                              "--batch", "2", "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
    for name, shape in (("reconstruction", (2, 320, 320, 2)), ("estimates_sample", (5, 8, 1 << 16, 2))):
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.shape == shape and a.dtype == np.float32 and np.isfinite(a).all()
        assert np.array_equal(a, b), name


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
