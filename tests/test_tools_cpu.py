"""CPU checks of the measurement helpers: the parity bookkeeping of bench.py / the GPU tests, bench.py's output dump, and the ncu
launch-list summariser."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from blama_b200 import parity_stats as ps  # noqa: E402


def test_parity_stats_top10_figures():
    rng = np.random.default_rng(3)
    want = (rng.standard_normal(4000) * 2).astype(np.float32)
    want[[7, 99, 1234]] += 20.0                                  # three ranks far above the rest: pinned whatever the noise
    st = ps.StepStats()
    st.add_floor(want + 1e-6, want)                              # a second implementation of the reference: same order
    got = want + (rng.standard_normal(4000) * 0.05).astype(np.float32)
    err, bad = st.add(got, want, ps.top_sorted(got, 10)[0])
    s = st.summary()
    assert not bad and s["pinned_ranks"] >= 2 and s["pinned_ranks_ok"] == s["pinned_ranks"]
    assert s["top1_match_frac"] == 1.0 and 0.5 <= s["top10_overlap_mean"] <= 1.0
    assert s["floor_top10_id_match_frac"] == 1.0 and s["floor_top1_match_frac"] == 1.0 and s["floor_top10_overlap_mean"] == 1.0
    assert s["within_floor"] is False                            # 0.05 of noise against a floor of 1e-6
    assert abs(s["max_abs"] - err) < 1e-9


def test_bench_write_outputs_dtypes_and_limit(tmp_path):
    import bench

    toks = np.array([5, 128255, 2**31 - 1], dtype=np.int32)
    logits = np.linspace(-3, 3, 7, dtype=np.float32)
    bench.write_outputs(str(tmp_path / "d"), {"tokens": toks, "logits": logits, "score": np.array([0.25])})
    got = {p.stem: np.load(p) for p in (tmp_path / "d").iterdir()}
    assert sorted(got) == ["logits", "score", "tokens"]
    assert got["tokens"].dtype == np.float64 and np.array_equal(got["tokens"], toks)
    assert got["logits"].dtype == np.float32 and np.array_equal(got["logits"], logits)
    assert got["score"].dtype == np.float64 and got["score"][0] == 0.25
    with pytest.raises(ValueError):
        bench.write_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT_BYTES // 8 + 1)})
    assert not (tmp_path / "big").exists()
    # the reference arm has no device outputs to write: refused before any work
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "ref")],
                       capture_output=True, text=True)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "ref").exists()


def test_ncu_summary_selects_the_last_pass(tmp_path):
    csv_text = "\n".join([
        "==PROF== noise line",
        '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"',
        '"0","1","python","h","embed_kernel(int)","1","7","(256, 1, 1)","(32, 1, 1)","0","10.0","Command line profiler metrics","gpu__time_duration.sum","ns","1,000"',
        '"1","1","python","h","void gemm<1>(int)","1","7","(320, 1, 1)","(148, 1, 1)","0","10.0","Command line profiler metrics","gpu__time_duration.sum","ns","5,000"',
        '"2","1","python","h","embed_kernel(int)","1","7","(256, 1, 1)","(2048, 1, 1)","0","10.0","Command line profiler metrics","gpu__time_duration.sum","ns","2,000"',
        '"3","1","python","h","void gemm<1>(int)","1","7","(320, 1, 1)","(148, 1, 1)","0","10.0","Command line profiler metrics","gpu__time_duration.sum","ns","7,000"',
        '"3","1","python","h","void gemm<1>(int)","1","7","(320, 1, 1)","(148, 1, 1)","0","10.0","Command line profiler metrics","dram__bytes_read.sum","byte","4,000,000"',
    ])
    p = tmp_path / "launches.csv"
    p.write_text(csv_text)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ncu_summary.py"), str(p), "--from-last", "embed_kernel", "--grid", "2048",
                          "--meta", "shape=x", "tokens=2048"], capture_output=True, text=True, check=True).stdout
    d = json.loads(out)
    assert d["shape"] == "x" and d["tokens"] == 2048 and d["kernels"] == 2
    assert abs(d["gpu_time_ms_serialised"] - 0.009) < 1e-12 and d["dram__bytes_read"] == 4e6
    assert d["per_kernel"]["void gemm<1>"]["launches"] == 1 and abs(d["per_kernel"]["void gemm<1>"]["ms"] - 0.007) < 1e-9
