"""bench.py's reference arm runs on the CPU (the unmodified reference through oracle/_ref): its JSON line must carry the keys the
driver reads, on the same metric / unit / config as the B200 arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "oracle_dump")), reason="oracle/_ref not built (make -C oracle ref)")
def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--step-bytes", "256"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-800:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "input_MB_per_s" and d["unit"] == "MB/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_samples_past_the_limit(tmp_path):
    """bench.dump_outputs (--dump-outputs): arrays within the limit are written whole; past it every array becomes the same
    seeded sample of its elements on every run, and the files stay within the limit."""
    code = ("import sys, numpy as np; sys.path.insert(0, %r); import bench\n"
            "a = np.arange(1000, dtype=np.float32).reshape(10, 100)\n"
            "bench.dump_outputs(sys.argv[1], {'p': a})\n"
            "for d in sys.argv[2:]: bench.dump_outputs(d, {'p': a, 'q': a.astype(np.float64)}, limit=3000)\n" % ROOT)
    dirs = [str(tmp_path / d) for d in ("whole", "s1", "s2")]
    subprocess.run([sys.executable, "-c", code] + dirs, check=True, cwd=ROOT)
    np.testing.assert_array_equal(np.load(os.path.join(dirs[0], "p.npy")), np.arange(1000, dtype=np.float32).reshape(10, 100))
    p1, q1 = np.load(os.path.join(dirs[1], "p.npy")), np.load(os.path.join(dirs[1], "q.npy"))
    assert p1.dtype == np.float32 and q1.dtype == np.float64 and p1.nbytes + q1.nbytes <= 3000 and p1.size == 250
    assert np.all(np.diff(p1) > 0)
    np.testing.assert_array_equal(p1, np.load(os.path.join(dirs[2], "p.npy")))
    np.testing.assert_array_equal(q1, np.load(os.path.join(dirs[2], "q.npy")))
