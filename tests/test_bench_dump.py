"""bench.py --dump-outputs: the arrays it writes (float64, within 64 MB, seeded samples of large outputs) and, on the GPU,
that two runs with the same arguments write identical outputs and time exactly --steps steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_seeded_sample_is_fixed_and_sorted():
    a, b = bench.seeded_sample(1 << 20, 256), bench.seeded_sample(1 << 20, 256)
    assert np.array_equal(a, b) and a.size == 256 and np.all(np.diff(a) > 0)
    assert np.array_equal(bench.seeded_sample(100, 256), np.arange(100))


def test_large_rows_are_sampled_within_the_limit(tmp_path):
    big = np.arange((1 << 21) * 5, dtype=np.float64).reshape(-1, 5)          # 80 MiB
    out = {}
    bench.sample_rows("particles", big, out)
    assert np.array_equal(out["particles"], big[out["particles_index"]])
    bench.write_outputs(str(tmp_path), out)
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= bench.DUMP_LIMIT_BYTES + 4096
    assert np.load(tmp_path / "particles.npy").dtype == np.float64
    with pytest.raises(RuntimeError):
        bench.write_outputs(str(tmp_path / "over"), {"particles": big})


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
           "--no-cpu-baseline", "--no-second", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.splitlines()[-1])


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    a, b = _bench(tmp_path / "a", 4), _bench(tmp_path / "b", 4)
    assert a["steps"] == b["steps"] == 4
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "particles.npy" in names and "landmarks.npy" in names
    for n in names:
        x, y = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert x.dtype == np.float64 and np.array_equal(x, y), n
    p = np.load(tmp_path / "a" / "particles.npy")
    assert p.shape == (bench.N_PARTICLES, 4) and np.isfinite(p).all()
    assert abs(p[:, 0].sum() - 1.0) < 1e-9                                     # weights are normalised after a step
