#!/usr/bin/env python
"""bench.py -- decode tok/s (+ verified tok/s) of the blama hot path on B200, one model replica per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--shape llama-3.1-8b-q4km] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...        (one rank per GPU)

A "step" is one /complete request of BASELINE.json configs[1]: a 512-token synthetic prompt, then 256 new tokens on
random-init Llama-3.1-8B-arch Q4_K_M weights.  Printed JSON line (rank 0):
  value    decode tok/s with everything resident in HBM: the 256 decode steps run back to back with the arg-max token
           fed back on the device (blk_decode_loop), timed with CUDA events on the engine's stream
  e2e      the same 256 tokens through the reference-shaped public API (bl::llama::Session::complete over the C ABI):
           host sampler chain in the loop, token id host->device and top-64 device->host every step, wall clock
  roofline the dominant kernel (gate/up mat-vec + SwiGLU) timed alone with CUDA events, algorithmic bytes / duration
           against the measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  the oracle (CPU restatement of the reference's ggml-cpu arithmetic, kind "port") on the box's host cores
--impl reference times that CPU port on the same metric (the real blama CPU build cannot be produced offline, DESIGN.md).
--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy, float32 or float64: the /complete
tokens and top-10 lists, the logits row and top-10 after the device-resident loop, and (--verify > 0) the score of the last
verify request.
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "decode tok/s (Llama-3.1-8B-arch Q4_K_M, 512-tok prompt + 256 new tokens, batch 1)"


def env_int(k, d):
    try:
        return int(os.environ.get(k, d))
    except ValueError:
        return d


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                d = json.load(f)
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst)"
        except Exception:
            pass
    return 2250.0, "fallback (B200_PROFILING.md nominal dense bf16)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu: int):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for i, n in enumerate(names):
                if len(r) > 3 + i and r[3 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def model_path(shape: str) -> str:
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
    return os.path.join(base, f"blama_b200_{shape}.gguf")


def ensure_model(shape: str, rank: int, barrier) -> str:
    from blama_b200 import gguf_synth

    path = model_path(shape)
    want = gguf_synth.model_bytes(gguf_synth.SHAPES[shape])
    if rank == 0 and not (os.path.exists(path) and os.path.getsize(path) >= want):
        t0 = time.time()
        tmp = path + ".tmp"
        gguf_synth.write_gguf(tmp, shape)
        os.replace(tmp, path)
        print(f"[bench] wrote {path} ({want / 1e9:.2f} GB) in {time.time() - t0:.1f}s", file=sys.stderr)
    barrier()
    return path


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's CPU path, bounded sample
# ---------------------------------------------------------------------------------------------------------------------
def cpu_decode_sample(path: str, shape: str, budget_s: float, steps: int = 1, warmup: int = 0, keep: int = 0, cross: int = 0):
    """decode tok/s of the CPU port on a bounded sample: a 16-token prompt, then n_new single-token decodes per step.
    keep > 0: also returns the reference rows of the run (last prompt token + the first `keep` greedy steps) for the parity block;
    cross > 0: additionally a /complete of `cross` tokens by the CPU port (prover for the cross-backend verdict) and a callable that
    runs the CPU port as the verifier of a response."""
    from blama_b200 import gguf_synth
    from oracle import pyoracle as po

    cores = os.cpu_count() or 1
    m = po.Model(path)
    c = po.Ctx(m, 512, po.MODE_GGML, cores)
    prompt = gguf_synth.synth_prompt(shape, 16, 1)
    t0 = time.time()
    c.decode(prompt)
    t_prompt = time.time() - t0
    t0 = time.time()
    c.decode([int(prompt[0])])
    t_tok = max(1e-4, time.time() - t0)
    total_steps = max(1, steps + warmup)
    n_new = int(max(2, min(64, (budget_s / total_steps - t_prompt) / t_tok)))
    times = []
    trace = {"prompt": [int(t) for t in prompt], "rows": []}
    for s in range(total_steps):
        c.clear()
        lg = c.decode(prompt)[0]
        if s == 0 and keep:
            trace["rows"].append((None, lg.copy()))          # the row after the whole prompt
        tok = int(np.argmax(lg))
        t0 = time.time()
        for i in range(n_new):
            lg = c.decode([tok])[0]
            if s == 0 and i < keep:
                trace["rows"].append((tok, lg.copy()))
            tok = int(np.argmax(lg))
        dt = time.time() - t0
        if s >= warmup:
            times.append(dt)
    if keep:
        # the noise floor of the reference arithmetic on the same tokens: the port against itself with the fp32 partial sums added
        # in the opposite order (blama_b200/parity_stats.py)
        alt = po.Ctx(m, 512, po.MODE_GGML_ALT, cores)
        trace["floor_rows"] = [alt.decode(prompt)[0].copy()]
        for tok, _ in trace["rows"][1:]:
            trace["floor_rows"].append(alt.decode([tok])[0].copy())
        alt.close()
    if cross:
        c.clear()
        trace["cpu_prover"] = c.complete(prompt, cross, seed=5)
        trace["cpu_verifier"] = lambda toks, claimed_ids: c.fill_ctx(prompt, toks, claimed_ids)
        trace["close"] = lambda: (c.close(), m.close())
    else:
        c.close(); m.close()
    tok_s = n_new * len(times) / sum(times)
    return {"value": tok_s, "unit": "tok/s", "cores": cores, "kind": "port",
            "sample": f"{len(times)} x ({len(prompt)}-token prompt, then {n_new} batch-1 decode steps) of the same GGUF; "
                      f"oracle/liboracle.so (ggml-cpu arithmetic restated, {cores} threads)"}, n_new, sum(times) / len(times), trace


def gpu_parity(hm, n_ctx: int, trace: dict) -> dict:
    """The GPU path against the rows the CPU port just produced (same GGUF, same tokens): logits of the batch-1 decode kernel per step,
    and the reference's cross-backend verdict test in both directions (inference/test/t-LogitComparer.cpp:41-79)."""
    from blama_b200 import host_api, parity_stats as ps

    inst = host_api.Instance(hm, n_ctx)
    ctx = inst.raw_ctx()
    st = ps.StepStats()
    prompt = trace["prompt"]
    ctx.clear()
    for t in prompt[:-1]:
        ctx.decode([t])
    feed = prompt[-1]
    for k, (tok, want) in enumerate(trace["rows"]):
        top = ctx.decode_topk(feed if tok is None else tok, 10)
        st.add(ctx.logits(), want, top["token"])
        if "floor_rows" in trace:
            st.add_floor(trace["floor_rows"][k], want)
    out = st.summary()
    out["mode"] = "batch-1 decode kernel vs CPU port (ggml-cpu arithmetic), teacher-forced with the port's arg-max"
    if "cpu_prover" in trace:
        c_toks, c_top = trace["cpu_prover"]
        n = len(c_toks)
        # CPU prover -> GPU verifier (sequential fill = the decode kernel)
        inst.start_session(seed=5, sequential_verify=True).set_initial_prompt(prompt)
        g_out, g_n = inst.fill_ctx(c_toks, c_top)
        inst.stop_session()
        s_cg = host_api.lc_score([host_api.lc_compare(c_top[i], g_out[i][: g_n[i]]) for i in range(n)])
        # GPU prover -> CPU verifier
        inst.start_session(seed=5).set_initial_prompt(prompt)
        g_toks, g_top = inst.complete(n)
        inst.stop_session()
        o_out, o_n = trace["cpu_verifier"](g_toks, g_top["token"])
        s_gc = host_api.lc_score([host_api.lc_compare(g_top[i], o_out[i][: o_n[i]]) for i in range(len(g_toks))])
        trace["close"]()
        out.update({"score_cpu_prover_gpu_verifier": s_cg, "score_gpu_prover_cpu_verifier": s_gc, "verdict_tokens": n,
                    "verdict_equal": bool((s_cg >= 0.95) == (s_gc >= 0.95) and s_cg >= 0.95),
                    "same_tokens_sampled": bool(len(g_toks) == n and np.array_equal(g_toks, c_toks))})
    inst.close()
    return out


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    path = ensure_model(args.shape, 0, lambda: None)
    cb, n_new, step_s, _ = cpu_decode_sample(path, args.shape, budget_s=150.0, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "tok/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int8", "data": "synthetic",
        "config": {"workload": f"{args.shape}: {args.prompt}-token prompt + {args.new} new tokens per request (BASELINE configs[1]), "
                               "one replica per GPU, independent requests", "shape": args.shape, "prompt_tokens": args.prompt,
                   "new_tokens": args.new, "sample": f"bounded: 16-token prompt + {n_new} decode steps per step on the host cores (the full "
                                                     "512 + 256 request takes minutes on the CPU); shorter context favours the CPU arm"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "CPU restatement of the reference's llama.cpp CPU path (the upstream binary cannot be built offline)",
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------------------------
# multi-GPU plumbing: requests are partitioned, never sharded -- the only collectives are the barrier and the max / sum of
# the per-rank timings and token counts (NCCL on GPUs; gloo in the CPU tests)
# ---------------------------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self, rank: int, world: int, local_rank: int, backend=None):
        self.rank, self.world, self.local_rank, self.pg, self.device = rank, world, local_rank, None, "cpu"
        if world > 1 and backend:
            import torch
            import torch.distributed as td

            if backend == "nccl":
                torch.cuda.set_device(local_rank)
                self.device = f"cuda:{local_rank}"
                td.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            else:
                td.init_process_group(backend)
            self.pg = td

    def barrier(self):
        if self.pg is not None:
            self.pg.barrier()

    def _reduce(self, x: float, op_name: str) -> float:
        if self.pg is None:
            return x
        import torch

        t = torch.tensor([x], dtype=torch.float64, device=self.device)
        self.pg.all_reduce(t, op=getattr(self.pg.ReduceOp, op_name))
        return float(t.item())

    def max(self, x: float) -> float:
        return self._reduce(x, "MAX")

    def sum(self, x: float) -> float:
        return self._reduce(x, "SUM")

    def close(self):
        if self.pg is not None:
            self.pg.destroy_process_group()
            self.pg = None


def aggregate_throughput(dist: "Dist", units_this_rank: float, seconds_this_rank: float) -> float:
    """whole-job throughput: units all ranks processed / the slowest rank's time (bench contract)"""
    return dist.sum(units_this_rank) / dist.max(seconds_this_rank)


def request_seed(rank: int, step: int) -> int:
    """independent requests per rank and step (one replica per GPU, no request is split across GPUs)"""
    return 1 + rank * 100003 + step


# ---------------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------------
def run_ours(args, rank: int, world: int, local_rank: int):
    dist = Dist(rank, world, local_rank, backend="nccl" if world > 1 else None)
    barrier, max_over_ranks, sum_over_ranks = dist.barrier, dist.max, dist.sum

    from blama_b200 import capi, gguf_synth, host_api

    path = ensure_model(args.shape, rank, barrier)
    t0 = time.time()
    hm = host_api.Model(path, device=local_rank)
    load_s = time.time() - t0
    n_ctx = args.prompt + max(args.new, args.verify) + 64
    inst = host_api.Instance(hm, n_ctx)
    inst.warmup()
    ctx = inst.raw_ctx()
    prompt = gguf_synth.synth_prompt(args.shape, args.prompt, request_seed(rank, 0))

    sampler = ClockSampler(local_rank)
    dev_ms, e2e_s, prompt_ms, e2e_tokens = [], [], [], 0
    launches0 = None
    total = args.warmup + args.steps
    barrier()
    for s in range(total):
        timed = s >= args.warmup
        if s == args.warmup:
            barrier()
            sampler.start()
            launches0 = ctx.kernel_launches
        # --- e2e: the public API, host buffers in / out -----------------------------------------------------------------
        ctx.flush_l2()
        inst.start_session(seed=s)
        t0 = time.perf_counter()
        inst.set_initial_prompt(prompt)
        t1 = time.perf_counter()
        toks, top = inst.complete(args.new)
        t2 = time.perf_counter()
        inst.stop_session()
        # --- value: device-resident loop ---------------------------------------------------------------------------------
        ctx.flush_l2()
        ctx.clear()
        ctx.decode(prompt)
        first = int(ctx.topk(1)["token"][0])
        ctx.timer_start()
        ctx.decode_loop(first, args.new, wait=False)
        ms = ctx.timer_stop()
        if timed:
            dev_ms.append(ms); e2e_s.append(t2 - t1); prompt_ms.append((t1 - t0) * 1e3)
            e2e_tokens += len(toks)                # complete() stops early at an end-of-generation token
        assert len(toks) > 0
        if args.dump_outputs and s == total - 1:      # read back after the timer stopped: the timed region is unchanged
            loop_top = ctx.topk(10)
            outputs = {"complete_tokens": toks, "complete_top10_tokens": top["token"], "complete_top10_logits": top["logit"],
                       "decode_loop_logits": ctx.logits(), "decode_loop_top10_tokens": loop_top["token"],
                       "decode_loop_top10_logits": loop_top["logit"]}
    barrier()
    sampler.stop_flag.set()
    launches = ctx.kernel_launches - (launches0 or 0)

    # aggregate: value = tokens all ranks produced / max-over-ranks device time
    value = aggregate_throughput(dist, float(args.new * args.steps), sum(dev_ms) / 1e3)
    e2e = aggregate_throughput(dist, float(e2e_tokens), sum(e2e_s))
    t_dev = max_over_ranks(sum(dev_ms) / 1e3)

    # --- verified tok/s (BASELINE configs[2] shape: re-fill `verify` response tokens, top-10 gather + LogitComparer) -------
    verify = None
    if args.verify > 0:
        # the prover's side of the round trip (not timed): a real /complete of `verify` tokens with its top-10 per token
        inst.start_session(seed=1)
        inst.set_initial_prompt(prompt[:32])
        vt_l, vtop_l = inst.complete(args.verify)
        inst.stop_session()
        vt_l = np.ascontiguousarray(vt_l, dtype=np.int32); vtop_l = np.ascontiguousarray(vtop_l)      # the request, unmarshalled
        reps, vt = (1, []) if args.sequential_verify else (args.verify_reps, [])
        for r in range(reps + (0 if args.sequential_verify else 1)):              # one untimed warm-up, then `reps` timed requests
            ctx.flush_l2()
            inst.start_session(seed=1, sequential_verify=args.sequential_verify)
            inst.set_initial_prompt(prompt[:32])
            t0 = time.perf_counter()
            score = inst.verify(vt_l, vtop_l)          # fillCtx + LogitComparer over every position, in C++ (Server::verify)
            dt = time.perf_counter() - t0
            inst.stop_session()
            if r > 0 or args.sequential_verify:
                vt.append(dt)
        if args.dump_outputs:
            outputs["verify_score"] = np.array([score])
        t_v = max_over_ranks(statistics.median(vt))
        verify = {"tokens": int(len(vt_l)), "tok_s": sum_over_ranks(float(len(vt_l))) / t_v, "ms": t_v * 1e3, "reps": len(vt),
                  "ms_min": min(vt) * 1e3, "ms_max": max(vt) * 1e3, "timing": "median wall time of the timed requests (host buffers in, score out), L2 flushed before each",
                  "score": score, "score_note": "prover = int8 decode arithmetic, verifier = bf16 tensor-core prefill: same verdict at the reference's 0.95 bar, "
                                                "not the bit-identical 1.0 of the sequential mode",
                  "mode": "batched prefill" if not args.sequential_verify else "sequential decode"}
        # tensor roofline of the verify prefill: the work the default path EXECUTES -- layer GEMMs + attention + the claimed-id rows of the
        # vocabulary projection (10 per position) + one full row for the last position -- against the measured dense bf16 peak.  SURVEY 8d's
        # count with the full-vocabulary head (not computed by this path) is reported beside it.  The wall time includes fillCtx's host
        # side and the LogitComparer pass.
        sh_v = gguf_synth.SHAPES[args.shape]
        T, p0 = int(len(vt_l)), 32
        dq, dkv = sh_v.n_head * sh_v.d_head, sh_v.n_head_kv * sh_v.d_head
        p_layers = sh_v.n_layer * (sh_v.d_model * (dq + 2 * dkv) + dq * sh_v.d_model + 3 * sh_v.d_model * sh_v.d_ffn)
        attn = 4.0 * dq * sh_v.n_layer * (T * p0 + T * (T + 1) / 2)
        flops = 2.0 * T * p_layers + attn + 2.0 * T * 10 * sh_v.d_model + 2.0 * sh_v.vocab * sh_v.d_model
        flops_full_head = 2.0 * T * (p_layers + sh_v.vocab * sh_v.d_model) + attn
        tf_peak, tf_src = measured_tensor_peak()
        traffic_v = None
        try:
            with open(os.path.join(ROOT, "profiles", "r2_ncu_verify_summary.json")) as fh:
                nv = json.load(fh)
            if nv.get("shape") == args.shape and nv.get("tokens") == T:
                traffic_v = nv["dram__bytes_read"] + nv["dram__bytes_write"]
        except (OSError, ValueError, KeyError):
            pass
        try:      # resident bf16 panels of the multi-token GEMMs (built by the first prefill; blama_b200.h blk_model_panel_bytes)
            nr, nm = C.c_int32(0), C.c_int32(0)
            pb = int(capi.lib().blk_model_panel_bytes(capi.lib().blk_ctx_model(ctx.h), C.byref(nr), C.byref(nm)))
            verify["weights_bf16_resident"] = {"bytes": pb, "matrices": int(nr.value), "of": int(nm.value),
                                               "note": "de-quantised once at the first multi-token pass and kept in HBM; BLK_PANEL_CACHE_GB=0 streams them per request instead"}
        except Exception as e:      # noqa: BLE001
            verify["weights_bf16_resident"] = {"error": str(e)}
        verify["roofline"] = {"bound": "tensor", "achieved": flops / t_v / 1e12, "peak": tf_peak, "unit": "TFLOP/s", "frac": flops / t_v / 1e12 / tf_peak,
                              "flops": flops, "flops_if_full_vocab_head": flops_full_head, "peak_source": tf_src, "traffic": traffic_v,
                              "traffic_source": "profiles/r2_ncu_verify_summary.json (sum of dram__bytes over the kernels of one verify prefill)" if traffic_v else None,
                              "note": "flops = executed work (claimed-id rows of the head only); flops_if_full_vocab_head = SURVEY 8d's count"}

    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, outputs)
    if rank != 0:
        dist.close()
        return

    # --- roofline of the dominant kernel, timed alone ------------------------------------------------------------------------
    peak, peak_src = measured_peaks()
    kernels = {}
    if ctx.persistent_decode:
        # the whole token is ONE kernel: time it alone (no top-k, position held at the end of the last request)
        ctx.clear(); ctx.decode(prompt)
        runs = [ctx.bench_kernel(5, 64) for _ in range(3)]          # three batches of 64 launches (CUDA events): the median batch
        ms, nbytes = sorted(runs)[1]
        kernels["mega_decode_kernel"] = {"ms": ms, "bytes": nbytes, "gbs": nbytes / ms / 1e6, "ms_batches": [round(r[0], 5) for r in runs]}
        dom, dom_name = kernels["mega_decode_kernel"], ("mega_decode_kernel (persistent cooperative kernel: the whole forward of one token, "
                                                        f"weights + KV of a {args.prompt}-token context), timed alone")
    else:
        names = ["ffn_gate_up_swiglu_gemv", "ffn_down_gemv", "attn_qkv_rope_gemv", "attn_out_gemv", "lm_head_gemv"]
        for which, nm in enumerate(names):
            ms, nbytes = ctx.bench_kernel(which, 64 if which < 4 else 16)
            kernels[nm] = {"ms": ms, "bytes": nbytes, "gbs": nbytes / ms / 1e6}
        dom, dom_name = kernels[names[0]], "gemv_pairs_kernel<EPI_SWIGLU> (ffn gate/up mat-vec + SiLU*mul), timed alone over all layers"
    # bytes one decoded token must stream (weights once + KV read at the mean context of the run)
    # (the host Model does not expose its blk handle to Python; recompute from the GGUF plan)
    wbytes = 0
    for name, ne, t, _, _ in gguf_synth.plan_tensors(gguf_synth.SHAPES[args.shape]):
        if name in ("token_embd.weight", "rope_freqs.weight") and not (name == "token_embd.weight" and gguf_synth.SHAPES[args.shape].tied):
            continue
        bs, nb = gguf_synth.BLOCK[t]
        wbytes += int(np.prod(ne)) // bs * nb
    sh = gguf_synth.SHAPES[args.shape]
    kv_per_tok = sh.n_layer * sh.n_head_kv * sh.d_head * 2 * 2
    mean_ctx = args.prompt + args.new / 2
    bytes_per_token = wbytes + kv_per_tok * mean_ctx
    # DRAM traffic of the dominant kernel per launch, from the committed `ncu --set full` capture of the same kernel and shape
    traffic, traffic_file = None, None
    for cand in ("r2_ncu_mega_decode_summary.json", "r1_ncu_mega_decode_summary.json"):
        try:
            with open(os.path.join(ROOT, "profiles", cand)) as fh:
                ns = json.load(fh)
            if ctx.persistent_decode and ns.get("shape") == args.shape:
                traffic, traffic_file = ns["dram__bytes_read"] + ns["dram__bytes_write"], cand
                break
        except (OSError, ValueError, KeyError):
            pass
    roofline = {
        "bound": "hbm", "kernel": dom_name,
        "achieved": dom["gbs"], "peak": peak, "unit": "GB/s", "frac": dom["gbs"] / peak, "traffic": traffic,
        "traffic_source": f"profiles/{traffic_file} (ncu --set full, one launch at a 512-token context)" if traffic else None,
        "peak_source": peak_src, "bytes_per_launch": dom["bytes"], "ms_per_launch": dom["ms"],
        "kernels": {k: {"gbs": round(v["gbs"], 1), "ms": round(v["ms"], 5), "bytes": v["bytes"], **({"ms_batches": v["ms_batches"]} if "ms_batches" in v else {})}
                    for k, v in kernels.items()},
        "step": {"bytes_per_token": int(bytes_per_token), "achieved_gbs": bytes_per_token * (value / world) / 1e9,
                 "frac": bytes_per_token * (value / world) / 1e9 / peak},
    }

    cpu, parity = None, None
    if world == 1 and not args.no_cpu:
        try:
            cpu, _, _, trace = cpu_decode_sample(path, args.shape, budget_s=20.0, keep=8, cross=16)
            parity = gpu_parity(hm, 256, trace)      # the CPU port's rows are the checker here, never the thing measured
        except Exception as e:  # the CPU port is a reported baseline, never on the product path
            cpu = cpu or {"value": None, "unit": "tok/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
            parity = parity or {"error": str(e)}

    clocks = sampler.summary()
    line = {
        "metric": METRIC, "value": value, "unit": "tok/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": (t_dev / args.steps) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int8", "data": "synthetic",
        "config": {"workload": f"{args.shape}: {args.prompt}-token prompt + {args.new} new tokens per request (BASELINE configs[1]), "
                               "one replica per GPU, independent requests", "shape": args.shape, "prompt_tokens": args.prompt,
                   "new_tokens": args.new, "l2": f"flushed (256 MiB memset) before every timed region; per-token weight stream {wbytes / 1e9:.1f} GB >> 126 MB L2",
                   "parallelism": f"replicas x{world} (no collective on the data path)"},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "tok/s", "h2d_bytes_per_step": 4 * (args.prompt + args.new), "d2h_bytes_per_step": 512 * (args.new + 1),
                "prompt_ms": statistics.mean(prompt_ms)},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity": parity,
        "verify": verify,
        "model_load_s": load_s,
    }
    emit(line)
    inst.close(); hm.close()
    dist.close()


# ---------------------------------------------------------------------------------------------------------------------
# dispatcher arm: ONE process, ONE bl::llama::server::Server, one replica + worker thread per GPU, whole requests from a shared queue
# (reference server/code/server/Server.cpp:45-161; north_star: "independent complete/verify requests are partitioned across the GPUs")
# ---------------------------------------------------------------------------------------------------------------------
def verify_flops(sh, T: int, p0: int) -> float:
    """executed work of one batched verify of T response tokens behind a p0-token prompt (see the verify roofline of run_ours)"""
    dq, dkv = sh.n_head * sh.d_head, sh.n_head_kv * sh.d_head
    p_layers = sh.n_layer * (sh.d_model * (dq + 2 * dkv) + dq * sh.d_model + 3 * sh.d_model * sh.d_ffn)
    return 2.0 * T * p_layers + 4.0 * dq * sh.n_layer * (T * p0 + T * (T + 1) / 2) + 2.0 * T * 10 * sh.d_model + 2.0 * sh.vocab * sh.d_model


def run_dispatcher(args):
    from concurrent.futures import ThreadPoolExecutor

    from blama_b200 import gguf_synth, host_api

    n_gpus, R = args.gpus, args.requests
    path = ensure_model(args.shape, 0, lambda: None)
    t0 = time.time()
    with ThreadPoolExecutor(n_gpus) as ex:
        models = list(ex.map(lambda g: host_api.Model(path, device=g), range(n_gpus)))
    load_s = time.time() - t0
    sh = gguf_synth.SHAPES[args.shape]
    p0 = 32
    v_max = args.verify if args.mode == "stream" else 64 if args.mode == "batch" else min(args.verify, 1024)
    workers = [m for m in models for _ in range(max(1, args.workers_per_gpu))]      # several Instances may share one Model (t-integration.cpp:220-224)
    srv = host_api.Server(workers, ctx_size=p0 + max(v_max, args.new) + 64, batch_size=4096, max_batch=args.max_batch if args.mode == "batch" else 1)
    prompt = gguf_synth.synth_prompt(args.shape, p0, 1)
    # the prover's side (not timed): ONE /complete of v_max tokens through the same Server; the queued verify requests re-fill
    # prefixes of that response (lengths spread over [v_max / 2, v_max]) -- the cost of a verify depends on its length only
    toks, top, nl = srv.wait_complete(srv.submit_complete(prompt, v_max, seed=1), cap=v_max)
    assert len(toks) == v_max, f"the prover stopped at an end-of-generation token after {len(toks)} tokens"
    lens = [int(x) for x in np.linspace(v_max // 2, v_max, R).round()]
    rng = np.random.default_rng(7)
    rng.shuffle(lens)
    kinds = ["verify"] * R if args.mode == "stream" else ["complete"] * R if args.mode == "batch" else ["complete" if i % 2 == 0 else "verify" for i in range(R)]

    def submit(i):
        if kinds[i] == "verify":
            return srv.submit_verify(prompt, toks[: lens[i]], top[: lens[i]], nl[: lens[i]], seed=1)
        return srv.submit_complete(gguf_synth.synth_prompt(args.shape, p0, 100 + i), args.new, seed=i)

    def wait(i, t):
        return srv.wait_verify(t) if kinds[i] == "verify" else len(srv.wait_complete(t, cap=args.new)[0])

    for t in [srv.submit_verify(prompt, toks[: lens[0]], top[: lens[0]], nl[: lens[0]], seed=1) for _ in range(2 * len(workers))]:      # warm-up: every worker
        srv.wait_verify(t)
    if args.mode == "batch":      # ... and every slot of the batching worker (first-use allocations of its context, the batched-step scratch)
        for t in [srv.submit_complete(gguf_synth.synth_prompt(args.shape, p0, 900 + i), 4, seed=i) for i in range(args.max_batch)]:
            srv.wait_complete(t, cap=4)
    srv.drain()
    sampler = ClockSampler(0)
    sampler.start()
    st0 = srv.stats()
    w0 = time.perf_counter()
    tickets = [submit(i) for i in range(R)]
    results = [wait(i, t) for i, t in enumerate(tickets)]
    wall = time.perf_counter() - w0
    srv.drain()                                  # the workers book a request after answering it
    st1 = srv.stats()
    sampler.stop_flag.set()
    per_worker = [{"device": b["device"], "requests": b["requests"] - a["requests"], "gpu_ms": b["gpu_ms"] - a["gpu_ms"]} for a, b in zip(st0, st1)]
    dev_s = max(w["gpu_ms"] for w in per_worker) / 1e3            # device clock (CUDA events around every request), max over the workers
    v_tokens = sum(lens[i] for i in range(R) if kinds[i] == "verify")
    d_tokens = sum(int(results[i]) for i in range(R) if kinds[i] == "complete")
    scores = [float(results[i]) for i in range(R) if kinds[i] == "verify"]
    flops = sum(verify_flops(sh, lens[i], p0) for i in range(R) if kinds[i] == "verify")
    tf_peak, tf_src = measured_tensor_peak()
    busy = sum(w["gpu_ms"] for w in per_worker) / 1e3
    if args.mode == "batch":
        metric = f"aggregate decode tok/s ({sh.name}, {R} concurrent /complete requests of {args.new} tokens, up to {args.max_batch} in flight per replica)"
        value = d_tokens / wall          # admission (prompt prefills) and the batched steps interleave on the host: wall clock is the honest figure
    else:
        metric = ("verified tok/s" if args.mode == "stream" else "verified tok/s within a complete+verify mix") + \
                 f" ({sh.name}, queued /verify_completion requests through one Server, one replica per GPU)"
        value = v_tokens / dev_s
    line = {
        "metric": metric,
        "value": value, "unit": "tok/s", "n_gpus": n_gpus, "steps": R, "warmup": 2 * n_gpus, "ms_per_step": dev_s / R * 1e3, "max_batch": args.max_batch if args.mode == "batch" else 1,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "mode": args.mode,
        "config": {"workload": f"{args.shape}: {R} queued requests ({'all /verify_completion' if args.mode == 'stream' else 'alternating /complete of ' + str(args.new) + ' tokens and /verify_completion'}"
                               f", responses of {min(lens)}..{max(lens)} tokens behind a {p0}-token prompt) through ONE bl::llama::server::Server in one process, "
                               f"{n_gpus} worker threads = {n_gpus} GPU replicas, shared queue, no collective (BASELINE configs[{4 if args.mode == 'stream' else 3}])",
                   "shape": args.shape, "requests": R, "response_tokens": [min(lens), max(lens)],
                   "responses": "prefixes of one prover run (a /complete of the longest length through the same Server)",
                   "l2": "per-request weight stream >> 126 MB L2"},
        "timing": "CUDA events on every replica's stream around each request, summed per replica; value = tokens / max over replicas",
        "wall_s": wall, "value_wall": v_tokens / wall, "dispatch_efficiency": busy / (len(workers) * wall), "workers_per_gpu": max(1, args.workers_per_gpu),
        "decode_tokens": d_tokens, "decode_tok_s_wall": d_tokens / wall if d_tokens else None,
        "per_worker": per_worker, "score_min": min(scores) if scores else None, "score_max": max(scores) if scores else None,
        "roofline": {"bound": "tensor", "achieved": flops / dev_s / 1e12 / n_gpus, "peak": tf_peak, "unit": "TFLOP/s per GPU",
                     "frac": flops / dev_s / 1e12 / n_gpus / tf_peak, "flops": flops, "peak_source": tf_src},
        "clocks": sampler.summary(), "gpu_launches": None, "model_load_s": load_s, "worker_error": srv.last_worker_error() or None,
    }
    emit(line)
    srv.close()
    for m in models:
        m.close()


_JSON_FD = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner on the first communicator,
    with NCCL_DEBUG=VERSION set by some launchers), so everything else is sent to stderr and the line goes to the saved fd."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


DUMP_LIMIT_BYTES = 64 * 10**6


def write_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: DIR/<name>.npy per array; float32 stays float32, everything else (token ids, scores) becomes float64,
    which holds every int32 exactly.  Refuses to write more than DUMP_LIMIT_BYTES in all."""
    conv = {name: np.ascontiguousarray(a, dtype=np.float32 if np.asarray(a).dtype == np.float32 else np.float64)
            for name, a in arrays.items()}
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in conv.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="llama-3.1-8b-q4km")
    ap.add_argument("--prompt", type=int, default=512)
    ap.add_argument("--new", type=int, default=256)
    ap.add_argument("--verify", type=int, default=2048, help="response tokens of the verify measurement (0 = skip)")
    ap.add_argument("--verify-reps", type=int, default=9, help="timed repeats of the verify request (median reported)")
    ap.add_argument("--sequential-verify", action="store_true")
    ap.add_argument("--max-batch", type=int, default=1, help="--mode batch: /complete requests in flight per replica (continuous batching)")
    ap.add_argument("--mode", default="step", choices=["step", "stream", "mix", "batch"],
                    help="step: the contract's per-GPU replica benchmark; stream: queued /verify_completion requests through ONE Server with "
                         "--gpus replicas in one process (BASELINE configs[4]); mix: alternating /complete and /verify_completion requests (configs[3])")
    ap.add_argument("--requests", type=int, default=64, help="queued requests of --mode stream / mix")
    ap.add_argument("--workers-per-gpu", type=int, default=1, help="--mode stream / mix: Server workers (Instances) sharing each replica: with 2, "
                    "one request's host work (claimed-id preparation, LogitComparer) overlaps the other's prefill")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="--mode step: write the outputs of the last timed step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "step"):
        ap.error("--dump-outputs applies to --impl ours --mode step")
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if not (args.gpus > 1 and world == 1 and args.mode == "step"):
        quiet_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.mode != "step":
        if rank == 0:
            run_dispatcher(args)          # one process drives all --gpus replicas
        return
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
