"""Prompt prefill time vs token count: the two-pass GEMM form and the fused form (BLK_PANEL_MIN)."""
import os, sys, time
sys.path.insert(0, '.')
from bench import ensure_model
from blama_b200 import capi, gguf_synth
shape = sys.argv[1] if len(sys.argv) > 1 else "llama-3.1-8b-q4km"
path = ensure_model(shape, 0, lambda: None)
m = capi.Model(path)
for name, pm in (("fused form", 1 << 30), ("two-pass  ", 32)):
    os.environ["BLK_PANEL_MIN"] = str(pm)
    c = capi.Ctx(m, 2304)
    row = []
    for T in (32, 64, 128, 256, 384, 512, 768, 1024, 2048):
        toks = gguf_synth.synth_prompt(shape, T, 3)
        c.clear(); c.decode(toks); c.topk(1)                    # warm (allocations, attributes)
        best = 1e9
        for _ in range(3):
            c.clear()
            t0 = time.perf_counter(); c.decode(toks); c.topk(1); best = min(best, time.perf_counter() - t0)
        row.append(f"T={T}: {best*1e3:6.2f}")
    print(name, " | ".join(row), "ms")
    c.close()
