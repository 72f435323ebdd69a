"""bench.py --dump-outputs on a small model: the outputs of the last timed step are written as float32 / float64 .npy files,
and two runs with the same arguments write the same arrays (seeded inputs, deterministic kernels)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from blama_b200 import gguf_synth as gs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--shape", "small-llama-q4km", "--prompt", "64", "--new", "32", "--verify", "48",
           "--verify-reps", "2", "--steps", "2", "--warmup", "1", "--no-cpu", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, check=True, timeout=600, capture_output=True, text=True).stdout.strip().splitlines()[-1]
    return json.loads(out), {p.stem: np.load(p) for p in out_dir.iterdir()}


def test_dump_outputs_are_reproducible(tmp_path):
    line, a = run_bench(tmp_path / "a")
    _, b = run_bench(tmp_path / "b")
    assert line["steps"] == 2 and line["value"] > 0
    assert sorted(a) == ["complete_tokens", "complete_top10_logits", "complete_top10_tokens", "decode_loop_logits",
                         "decode_loop_top10_logits", "decode_loop_top10_tokens", "verify_score"]
    assert sum(x.nbytes for x in a.values()) <= 64 * 10**6
    n = len(a["complete_tokens"])
    assert n > 0 and a["complete_top10_tokens"].shape == a["complete_top10_logits"].shape == (n, 10)
    assert a["decode_loop_logits"].shape == (gs.SHAPES["small-llama-q4km"].vocab,) and a["decode_loop_logits"].dtype == np.float32
    # the device top-10 after the loop is the top of the logits row it returned
    assert np.array_equal(np.sort(a["decode_loop_logits"])[::-1][:10], a["decode_loop_top10_logits"])
    assert a["complete_tokens"].dtype == np.float64 and np.array_equal(a["complete_tokens"], a["complete_tokens"].round())
    assert 0.0 < a["verify_score"][0] <= 1.0
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
