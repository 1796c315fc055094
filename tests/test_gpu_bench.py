"""GPU: bench.py --dump-outputs writes what the last timed step computed, the same arrays for the same arguments, and
--steps is the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(tmp_path, name, *args):
    out = tmp_path / name
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-bind", *args,
                           "--dump-outputs", str(out)], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert proc.returncode == 0, proc.stderr[-4000:]
    line = json.loads([ln for ln in proc.stdout.splitlines() if ln.startswith("{")][-1])
    arrays = {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    return line, arrays


def test_streaming_dump_is_reproducible_and_follows_steps(tmp_path):
    S = 1024
    common = ["--streams", str(S), "--warmup", "1", "--no-e2e", "--no-ops", "--no-cpu", "--no-parity"]
    line_a, a = _bench(tmp_path, "a", "--steps", "3", *common)
    line_b, b = _bench(tmp_path, "b", "--steps", "3", *common)
    line_c, c = _bench(tmp_path, "c", "--steps", "4", *common)
    assert (line_a["steps"], line_b["steps"], line_c["steps"]) == (3, 3, 4)
    assert sorted(a) == ["sample_streams", "state", "triggers", "window_label_counts", "window_labels"]
    assert a["triggers"].shape == (S,) and a["state"].shape == (2, S, 128) and a["window_labels"].shape == (S, 64)
    np.testing.assert_array_equal(a["sample_streams"], np.arange(S))
    assert np.isfinite(a["state"]).all() and np.abs(a["state"]).max() > 0
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert not np.array_equal(a["state"], c["state"])      # one more timed step: the carried state moved on


def test_attention_dump(tmp_path):
    line, a = _bench(tmp_path, "att", "--workload", "attention", "--utterances", "4", "--steps", "2", "--warmup", "1")
    assert line["steps"] == 2
    assert sorted(a) == ["sample_utterances", "softmax"]
    assert a["softmax"].shape == (4, 400, 6)
    np.testing.assert_allclose(a["softmax"].sum(-1), 1.0, atol=1e-5)
