"""bench.py --dump-outputs: what the last timed step computed, as float .npy files, comparable from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def _bench(out_dir, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-cpu-baseline",
                        "--dump-outputs", str(out_dir)] + list(args), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    files = sorted(os.listdir(out_dir))
    assert sum(os.path.getsize(out_dir / f) for f in files) <= 64 << 20
    arrays = {f[:-4]: np.load(out_dir / f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in arrays.values())
    return line, arrays


def test_training_dump_is_the_last_timed_step_and_repeats(tmp_path):
    a_line, a = _bench(tmp_path / "a", "--steps", "2", "--warmup", "1")
    _, b = _bench(tmp_path / "b", "--steps", "2", "--warmup", "1")
    _, c = _bench(tmp_path / "c", "--steps", "3", "--warmup", "1")
    assert sorted(a) == ["loss", "params_sample"] and a["loss"].dtype == np.float64 and a["params_sample"].dtype == np.float32
    assert float(a["loss"][0]) == a_line["config"]["loss_last_step"]
    # same arguments: same inputs, so the outputs agree up to the order of floating-point sums
    assert abs(float(a["loss"][0] - b["loss"][0])) < 1e-4 and float(np.abs(a["params_sample"] - b["params_sample"]).max()) < 1e-3
    # one more timed step ends on the next of the rotating batches: a different loss than the run-to-run noise
    assert abs(float(a["loss"][0] - c["loss"][0])) > 1e-3


def test_decode_dump(tmp_path):
    line, d = _bench(tmp_path, "--workload", "decode", "--steps", "1", "--warmup", "1")
    assert line["steps"] == 1 and line["config"]["tokens_per_step"] == 200
    assert sorted(d) == ["fp16_log_probs", "fp16_token_ids", "fp32_log_probs", "fp32_token_ids"]
    for p in ("fp32", "fp16"):
        ids = d[p + "_token_ids"]
        assert ids.dtype == np.float64 and ids.shape[0] == 1 and np.array_equal(ids, np.round(ids)) and ids.max() < 8192
