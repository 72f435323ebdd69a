"""Wall time of a 2048-token verify request (fillCtx + LogitComparer through the host API, L2 flushed before each, median of 5) for the
form selected by the environment: default two-pass (bf16 panels), BLK_PANEL_MIN=0 (de-quantisation fused into the GEMM)."""
import os, statistics, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import ensure_model
from blama_b200 import gguf_synth, host_api
shape = sys.argv[1] if len(sys.argv) > 1 else "llama-3.1-8b-q4km"
T = int(sys.argv[2]) if len(sys.argv) > 2 else 2048
path = ensure_model(shape, 0, lambda: None)
hm = host_api.Model(path)
inst = host_api.Instance(hm, T + 128)
ctx = inst.raw_ctx()
prompt = gguf_synth.synth_prompt(shape, 32, 1)
inst.start_session(seed=1).set_initial_prompt(prompt); toks, top = inst.complete(T); inst.stop_session()
ts = []
for r in range(6):
    ctx.flush_l2()
    inst.start_session(seed=1).set_initial_prompt(prompt)
    t0 = time.perf_counter(); score = inst.verify(toks, top); dt = time.perf_counter() - t0
    inst.stop_session()
    if r: ts.append(dt * 1e3)
print(f"{shape} T={T} PANEL_MIN={os.environ.get('BLK_PANEL_MIN','default')}: median {statistics.median(ts):.2f} ms (min {min(ts):.2f}, max {max(ts):.2f}), score {score:.5f}")
