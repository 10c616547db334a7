"""bench.py's output contract (CPU): exactly ONE JSON line on stdout even when a library (NCCL prints its version banner)
writes to file descriptor 1 during the run."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_single_json_line_on_stdout():
    code = (
        "import os, sys\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import bench\n"
        "sys.stdout.flush()\n"
        "bench._REAL_STDOUT = os.dup(1)\n"
        "os.dup2(2, 1)\n"
        "os.write(1, b'NCCL version 0.0.0 (library chatter on fd 1)\\n')\n"
        "print('python-level chatter')\n"
        "bench._emit({'metric': 'flows/sec DDIM-50 @436x1024', 'value': 1.5})\n"
    )
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    assert len(lines) == 1, r.stdout
    assert json.loads(lines[0]) == {"metric": "flows/sec DDIM-50 @436x1024", "value": 1.5}
    assert "NCCL version" in r.stderr and "python-level chatter" in r.stderr


def test_reduction_rate_profile_is_parsed():
    """bench.py's `frac_of_l2_reduction_rate` divides by the rate measured by scripts/micro/red_rate.cu for the white-noise
    scatter pattern (profiles/r2_red_rate.txt): the committed profile must parse to a plausible number of reductions / s."""
    sys.path.insert(0, ROOT)
    import bench
    rate = bench.load_red_rate()
    assert rate is not None and 1e11 < rate < 1e12, rate


def test_dump_outputs_whole_or_a_fixed_sample(tmp_path):
    """--dump-outputs: a small output is written whole, a large one as the same seeded sample on every run, both float32."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    small = torch.arange(6, dtype=torch.float64).reshape(2, 3)
    big = torch.arange(bench.DUMP_FULL_MAX + 1, dtype=torch.float32)          # value == flat index
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"small": small, "big": big})
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and np.array_equal(s, small.numpy())
    b = np.load(tmp_path / "a" / "big.npy")
    assert b.dtype == np.float32 and b.shape == (bench.DUMP_SAMPLE,)
    assert np.array_equal(b, np.load(tmp_path / "b" / "big.npy"))
    assert np.all(np.diff(b) >= 0) and 0 <= b.min() and b.max() <= bench.DUMP_FULL_MAX


def test_dump_outputs_are_finite_with_a_mask_of_the_holes(tmp_path):
    """The forward splat leaves NaN holes in the samples: the dump writes 0 there and marks them in <name>_nonfinite.npy."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    holes = torch.tensor([[1.0, float("nan")], [float("inf"), -2.0]])
    bench.dump_outputs(str(tmp_path), {"samples": holes, "flow": torch.ones(3)})
    assert np.array_equal(np.load(tmp_path / "samples.npy"), np.array([[1, 0], [0, -2]], dtype=np.float32))
    assert np.array_equal(np.load(tmp_path / "samples_nonfinite.npy"), np.array([[0, 1], [1, 0]], dtype=np.float32))
    assert np.load(tmp_path / "samples_nonfinite.npy").dtype == np.float32
    assert not (tmp_path / "flow_nonfinite.npy").exists()
