"""bench.py --dump-outputs: the last timed step's outputs are written as float .npy files, and two runs with the same
arguments write the same values (fixed seeds for weights, conditioning and the sampler's Philox key), so that two
builds can be compared output for output."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = {"1b_lyrics": ["logits", "tokens"], "vqvae_decode": ["audio_level0", "audio_level1", "audio_level2"]}


def _run(workload, out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--small", "--steps", "3",
           "--warmup", "2", "--no-cpu-baseline", "--no-secondary", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    files = sorted(f[:-4] for f in os.listdir(out_dir))
    assert files == NAMES[workload]
    return {k: np.load(os.path.join(out_dir, k + ".npy")) for k in files}


@pytest.mark.parametrize("workload", sorted(NAMES))
def test_dumped_outputs_repeat_exactly(workload, tmp_path):
    a = _run(workload, tmp_path / "a")
    b = _run(workload, tmp_path / "b")
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and a[k].size > 0 and np.isfinite(a[k]).all(), k
        assert np.array_equal(a[k], b[k]), f"{k}: two runs with the same arguments differ"
    if workload == "1b_lyrics":
        assert a["tokens"].shape[0] == a["logits"].shape[0] == 16
        assert (a["tokens"] == np.round(a["tokens"])).all() and (a["tokens"] >= 0).all()
