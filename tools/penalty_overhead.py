"""Cost of the logit-bias / repetition-penalty edit pass: tok/s with and without the stages, alternated in one process.

    python tools/penalty_overhead.py [--rounds 3] [--new 256] [--server-new 128] [--out FILE]

Workload: the synthetic Llama-3.1-8B-arch Q4_K_M model, a 512-token prompt and --new tokens through Session::complete (batch-1
decode), in three configurations: no stages; window 64, repeat 1.1, freq 0.1, present 0.1; the same plus a 1000-entry bias map.
Then a batching server (max_batch 32) with 32 requests in flight, without and with the penalties + bias.  Every timing ends in
a device synchronise (complete() and the server's answers read results back).  The card's name and power limit are printed
with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import ensure_model  # noqa: E402
from blama_b200 import gguf_synth as gs, host_api as H  # noqa: E402

SHAPE = "llama-3.1-8b-q4km"


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:      # the numbers still print; the card line says why it is missing
        return f"unknown ({e})"


def configs(n_vocab: int):
    rng = np.random.default_rng(0)
    bias = {int(t): float(b) for t, b in zip(rng.choice(n_vocab, 1000, replace=False), rng.uniform(-5.0, 2.0, 1000))}
    pen = dict(penalty_last_n=64, repeat_penalty=1.1, freq_penalty=0.1, present_penalty=0.1)
    return {"off": {}, "penalties": pen, "penalties+bias1000": dict(pen, logit_bias=bias)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--new", type=int, default=256)
    ap.add_argument("--server-new", type=int, default=128)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    H.lib()
    path = ensure_model(SHAPE, 0, lambda: None)
    m = H.Model(path)
    prompt = [int(t) for t in gs.synth_prompt(SHAPE, 512, 1)]
    inst = H.Instance(m, 1024)
    n_vocab = inst.raw_ctx().m.n_vocab
    cfgs = configs(n_vocab)
    lines = [f"card: {card()}", f"model: {SHAPE} (synthetic weights), prompt 512 tokens, {a.new} new tokens per Session::complete"]
    res = {k: [] for k in cfgs}
    for name, st in cfgs.items():            # warm-up of every configuration (allocations, first launches)
        inst.start_session(seed=1, **st).set_initial_prompt(prompt)
        inst.complete(8)
        inst.stop_session()
    for r in range(a.rounds):
        for name, st in cfgs.items():
            inst.start_session(seed=1, **st).set_initial_prompt(prompt)
            t0 = time.perf_counter()
            toks, _ = inst.complete(a.new)
            dt = time.perf_counter() - t0
            inst.stop_session()
            res[name].append(len(toks) / dt)
            lines.append(f"round {r} session {name:20s} {len(toks):4d} tokens {len(toks) / dt:8.1f} tok/s")
    for name, v in res.items():
        lines.append(f"session {name:20s} median {np.median(v):8.1f} tok/s  (rounds: {', '.join(f'{x:.1f}' for x in v)})")
    inst.close()

    srv = H.Server([m], ctx_size=1024, max_batch=32)
    prompts = [[int(t) for t in gs.synth_prompt(SHAPE, 512, 10 + k)] for k in range(32)]
    scfg = {"off": cfgs["off"], "penalties+bias1000": cfgs["penalties+bias1000"]}
    sres = {k: [] for k in scfg}
    for rr in range(a.rounds + 1):           # round 0 warms up
        for name, st in scfg.items():
            t0 = time.perf_counter()
            tickets = [srv.submit_complete(p, a.server_new, seed=k, **st) for k, p in enumerate(prompts)]
            n = sum(len(srv.wait_complete(t)[0]) for t in tickets)
            dt = time.perf_counter() - t0
            if rr:
                sres[name].append(n / dt)
                lines.append(f"round {rr - 1} server {name:20s} {n:5d} tokens {n / dt:8.1f} tok/s (32 requests in flight, prompts included)")
    for name, v in sres.items():
        lines.append(f"server {name:20s} median {np.median(v):8.1f} tok/s  (rounds: {', '.join(f'{x:.1f}' for x in v)})")
    err = srv.last_worker_error()
    if err:
        lines.append(f"server worker error: {err}")
    srv.close(); m.close()
    text = "\n".join(lines)
    print(text, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
            f.write(json.dumps({"session": {k: float(np.median(v)) for k, v in res.items()},
                                "server": {k: float(np.median(v)) for k, v in sres.items()}}) + "\n")


if __name__ == "__main__":
    main()
