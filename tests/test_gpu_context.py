"""Context management on the paged KV cache (reference Session.cpp:284-347; SURVEY.md section 8f item 3):
  * blk_kv_shift = llama_kv_self_seq_rm + llama_kv_self_seq_add + llama.cpp's K-shift, against the oracle's restatement;
  * Session's infinite-context shifting inside complete() against the oracle replaying the same schedule;
  * getState / setState: the reference's "states" test shape (inference/test/t-integration.cpp:304-421)."""
import numpy as np
import pytest

from blama_b200 import gguf_synth as gs
from blama_b200 import parity_stats as ps

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["small-llama-q4km", "small-qwen2-q8", "tiny-llama-q8"])      # NORM rotary + rope_freqs, NEOX rotary, d_head 64
def test_kv_shift_matches_oracle(name, gguf_path, oracle):
    from blama_b200 import capi

    path = gguf_path(name)
    om = oracle.Model(path); oc = oracle.Ctx(om, 128, oracle.MODE_GGML, 4)
    m = capi.Model(path); c = capi.Ctx(m, 128)
    toks = [int(t) for t in gs.synth_prompt(name, 90, 77)]
    for t in toks[:70]:                       # crosses a 64-token KV page
        oc.decode([t]); c.decode([t])
    oc.kv_shift(6, 37); c.kv_shift(6, 37)     # drop 31 cells behind a 6-token prefix; the 33 cells behind them move (two chunks of <= 31)
    assert c.n_past == oc.n_past == 39
    worst = 0.0
    for t in toks[70:82]:
        want = oc.decode([t])[0]
        c.decode([t])
        worst = max(worst, float(np.abs(c.logits() - want).max()))
    print(f"\n[kv shift {name}] max |dlogit| after the shift = {worst:.3g}")
    assert worst <= ps.FLIP_TOL, worst
    # a second shift on the shifted cache, then errors
    oc.kv_shift(2, 3); c.kv_shift(2, 3)
    want = oc.decode([toks[82]])[0]; c.decode([toks[82]])
    assert float(np.abs(c.logits() - want).max()) <= ps.FLIP_TOL
    with pytest.raises(capi.BlkError):
        c.kv_shift(10, 10)
    with pytest.raises(capi.BlkError):
        c.kv_shift(5, 1000)
    c.close(); m.close(); oc.close(); om.close()


def test_infinite_context_generation_follows_the_reference_schedule(gguf_path, oracle):
    """complete() past the end of a 64-token context: Session::doDecode drops numLeft / 2 cells behind the prompt whenever
    numPast + 1 >= n_ctx (reference Session.cpp:324-347).  The oracle replays the produced tokens with the same schedule; the
    top-10 logits reported for every token must agree with the oracle's rows."""
    from blama_b200 import host_api as H

    name = "small-llama-q4km"
    path = gguf_path(name)
    prompt = [int(t) for t in gs.synth_prompt(name, 10, 5)]
    hm = H.Model(path)
    inst = H.Instance(hm, 64)
    inst.start_session(seed=4).set_initial_prompt(prompt)
    toks, top = inst.complete(150)
    assert len(toks) == 150                                   # 160 tokens through a 64-token context
    inst.stop_session()
    inst.start_session(seed=4, infinite_context=False).set_initial_prompt(prompt)
    with pytest.raises(H.HostError, match="^context limit of 64 reached$"):
        inst.complete(150)
    inst.close()
    om = oracle.Model(path); oc = oracle.Ctx(om, 64, oracle.MODE_GGML, 4)
    oc.decode(prompt)
    n_keep, n_past, worst, shifts = len(prompt), len(prompt), 0.0, 0
    for i, t in enumerate(toks):
        if n_past + 1 >= 64:
            n_discard = (n_past - n_keep) // 2
            oc.kv_shift(n_keep, n_keep + n_discard)
            n_past -= n_discard; shifts += 1
        row = oc.decode([int(t)])[0]
        n_past += 1
        worst = max(worst, float(np.abs(row[top[i]["token"]] - top[i]["logit"]).max()))
    print(f"\n[context shift] {shifts} shifts over 150 generated tokens, max |dlogit| on the reported top-10 = {worst:.3g}")
    assert shifts >= 4 and worst <= ps.FLIP_TOL, (shifts, worst)
    oc.close(); om.close(); hm.close()


def test_fill_ctx_past_the_context_end_shifts_like_the_reference_loop(gguf_path):
    from blama_b200 import host_api as H

    name = "small-llama-q4km"
    hm = H.Model(gguf_path(name))
    prompt = gs.synth_prompt(name, 8, 2)
    a, b = H.Instance(hm, 64), H.Instance(hm, 64)
    a.start_session(seed=2).set_initial_prompt(prompt)
    toks, top = a.complete(100)
    b.start_session(seed=2).set_initial_prompt(prompt)
    out, out_n = b.fill_ctx(toks, top)                        # does not fit: per-token loop with the same shifts -> bit-equal
    assert np.array_equal(out["token"], top["token"]) and np.array_equal(out["logit"], top["logit"])
    a.close(); b.close(); hm.close()


def test_states(gguf_path):
    """t-integration.cpp:304-421: same state + fresh sampler -> same text; a mid-session state restores the cache but not the RNG"""
    from blama_b200 import host_api as H

    name = "small-llama-q4km"
    hm = H.Model(gguf_path(name))
    inst = H.Instance(hm, 256)
    prompt = hm.tokenize("France has a long history of", add_special=True)
    n = 15
    inst.start_session().set_initial_prompt(prompt)
    initial = inst.get_state()
    p1, top1 = inst.complete(n)
    middle = inst.get_state()
    p2, _ = inst.complete(n)
    inst.stop_session()
    assert len(initial) < len(middle)                         # the blob grows with the cache
    # the initial state + a sampler in its initial state -> the same tokens (and the same reported logits)
    inst.start_session().set_state(initial)
    r1, rtop1 = inst.complete(n)
    assert np.array_equal(r1, p1) and np.array_equal(rtop1["logit"], top1["logit"])
    inst.stop_session()
    # the middle state: the RNG is not part of the state, so the continuation differs from the original one ...
    inst.start_session().set_state(middle)
    m1, _ = inst.complete(n)
    inst.stop_session()
    assert not np.array_equal(m1, p2)
    # ... but is the same for every session started from that state
    other = H.Instance(hm, 256)
    other.start_session().set_state(middle)
    m2, _ = other.complete(n)
    assert np.array_equal(m1, m2)
    other.stop_session()
    # errors: the reference's texts
    other.start_session()
    with pytest.raises(H.HostError, match="^Failed to set state$"):
        other.set_state(np.frombuffer(b"not a state blob, definitely not", dtype=np.uint8))
    with pytest.raises(H.HostError, match="^Failed to set state$"):
        other.set_state(middle[: len(middle) // 2])           # truncated
    other.set_state(initial)
    with pytest.raises(H.HostError, match="^Session already started$"):
        other.set_state(initial)
    small = H.Instance(hm, 16)                                # a context the state does not fit into
    small.start_session()
    with pytest.raises(H.HostError, match="^Failed to set state$"):
        small.set_state(middle)
    for i in (inst, other, small):
        i.close()
    hm.close()


def _regroup(ctxs, n_pos, ga_i, F, W):
    """Session::ensureRoom's Self-Extend loop (reference Session.cpp:348-368) applied to every context in `ctxs`"""
    while n_pos >= ga_i + W:
        ib = (F * ga_i) // W
        bd = (W // F) * (F - 1)
        dd = (W // F) - ib * bd - W
        for c in ctxs:
            c.kv_seq_add(ga_i, n_pos, ib * bd)
            c.kv_seq_div(ga_i + ib * bd, ga_i + ib * bd + W, F)
            c.kv_seq_add(ga_i + ib * bd + W, n_pos + ib * bd, dd)
        n_pos -= bd
        ga_i += W // F
    return n_pos, ga_i


@pytest.mark.parametrize("name,F,W", [("small-llama-q4km", 2, 32), ("small-qwen2-q8", 4, 32), ("tiny-llama-q8", 2, 16)])
def test_self_extend_positions_match_oracle(name, F, W, gguf_path, oracle):
    """llama_kv_self_seq_add / seq_div on cell positions + the K-shift, against the oracle's restatement, driven by the reference's
    schedule; the next token's rotary position is one past the largest cell position"""
    from blama_b200 import capi

    path = gguf_path(name)
    om = oracle.Model(path); oc = oracle.Ctx(om, 256, oracle.MODE_GGML, 4)
    m = capi.Model(path); c = capi.Ctx(m, 256)
    toks = [int(t) for t in gs.synth_prompt(name, 140, 61)]
    n_pos, ga_i, worst, regroups = 0, 0, 0.0, 0
    # a 40-token prompt in one call (the tcgen05 prefill on the GPU), then token by token
    oc.decode(toks[:40]); c.decode(toks[:40])
    n_pos = 40
    for i, t in enumerate(toks[40:]):
        before = ga_i
        n_pos, ga_i = _regroup([c, oc], n_pos, ga_i, F, W)
        regroups += ga_i != before
        assert c.next_pos == oc.next_pos == n_pos and c.n_past == 40 + i
        want = oc.decode([t])[0]
        c.decode([t])
        n_pos += 1
        err = float(np.abs(c.logits() - want).max())
        worst = max(worst, err)
        # the prompt went through the bf16 prefill on the GPU and the int8 path in the oracle: quantisation-noise bound
        assert err <= 0.5, (i, err)
    print(f"\n[self-extend {name} F={F} W={W}] {regroups} regroupings over 100 tokens, max |dlogit| = {worst:.3g}")
    assert regroups >= 3
    # the state blob carries the positions: a second context continues identically
    c2 = capi.Ctx(m, 256)
    c2.state_set(c.state_get())
    assert c2.next_pos == c.next_pos and c2.n_past == c.n_past
    c.decode([toks[0]]); c2.decode([toks[0]])
    assert np.array_equal(c.logits(), c2.logits())
    with pytest.raises(capi.BlkError):
        c.kv_shift(2, 5)                                   # compaction is not defined once positions have been regrouped
    c.close(); c2.close(); m.close(); oc.close(); om.close()


def test_self_extend_session_follows_the_reference_schedule(gguf_path, oracle):
    from blama_b200 import host_api as H

    name, F, W = "small-llama-q4km", 2, 32
    path = gguf_path(name)
    prompt = [int(t) for t in gs.synth_prompt(name, 10, 8)]
    hm = H.Model(path)
    inst = H.Instance(hm, 256)
    inst.start_session_self_extend(F, W, seed=6).set_initial_prompt(prompt)
    toks, top = inst.complete(120)
    assert len(toks) == 120
    inst.stop_session()
    with pytest.raises(H.HostError, match="^Group-attention width 33 must be a multiple of group-attention factor 2$"):
        inst.start_session_self_extend(2, 33).set_initial_prompt(prompt)
    inst.close()
    om = oracle.Model(path); oc = oracle.Ctx(om, 256, oracle.MODE_GGML, 4)
    oc.decode(prompt)
    n_pos, ga_i, worst = len(prompt), 0, 0.0
    for i, t in enumerate(toks):
        n_pos, ga_i = _regroup([oc], n_pos, ga_i, F, W)
        row = oc.decode([int(t)])[0]
        n_pos += 1
        worst = max(worst, float(np.abs(row[top[i]["token"]] - top[i]["logit"]).max()))
    print(f"\n[self-extend session] ga index {ga_i} after 120 tokens, max |dlogit| on the reported top-10 = {worst:.3g}")
    assert ga_i >= 3 * (W // F) and worst <= ps.FLIP_TOL, (ga_i, worst)
    oc.close(); om.close(); hm.close()


@pytest.mark.parametrize("persistent", [True, False], ids=["persistent", "per-op"])
def test_profile_step_adds_its_cell_like_decode(persistent, gguf_path, monkeypatch):
    """blk_profile_step between Self-Extend regroupings: the pending K re-rotation is applied before the step and the new cell's
    position is recorded for the next regrouping, exactly as blk_decode does it (BLK_MEGA=0: the eagerly enqueued per-op step)"""
    from blama_b200 import capi

    name, F, W = "small-llama-q4km", 2, 32
    if not persistent:
        monkeypatch.setenv("BLK_MEGA", "0")                  # read when the model is loaded
    m = capi.Model(gguf_path(name))
    monkeypatch.delenv("BLK_MEGA", raising=False)
    a, b = capi.Ctx(m, 256), capi.Ctx(m, 256)
    assert a.persistent_decode == persistent
    toks = [int(t) for t in gs.synth_prompt(name, 69, 61)]
    a.decode(toks[:40]); b.decode(toks[:40])
    n_pos, ga_i, regroups = 40, 0, 0
    for t in toks[40:68]:
        before = ga_i
        n_pos, ga_i = _regroup([a, b], n_pos, ga_i, F, W)
        regroups += ga_i != before
        a.profile_step(t); b.decode([t])
        n_pos += 1
        assert np.array_equal(a.logits(), b.logits())
        assert a.n_past == b.n_past and a.next_pos == b.next_pos == n_pos
    assert regroups >= 2
    a.decode([toks[68]]); b.decode([toks[68]])
    assert np.array_equal(a.logits(), b.logits())
    a.close(); b.close(); m.close()


def test_profile_step_rejects_a_bad_token(gguf_path):
    from blama_b200 import capi

    name = "small-llama-q4km"
    m = capi.Model(gguf_path(name)); c = capi.Ctx(m, 64)
    c.decode([int(t) for t in gs.synth_prompt(name, 5, 3)])
    for bad in (m.n_vocab, -1):
        with pytest.raises(capi.BlkError):
            c.profile_step(bad)
        assert c.n_past == 5
    c.close(); m.close()


def test_bench_kernel_resets_the_context(gguf_path, monkeypatch):
    """the per-op kernel benchmark leaves an empty context behind, Self-Extend positions included"""
    from blama_b200 import capi

    name = "small-llama-q4km"
    monkeypatch.setenv("BLK_MEGA", "0")                      # the kernels of the per-op step, as bench.py times them
    m = capi.Model(gguf_path(name))
    monkeypatch.delenv("BLK_MEGA", raising=False)
    c, fresh = capi.Ctx(m, 256), capi.Ctx(m, 256)
    toks = [int(t) for t in gs.synth_prompt(name, 52, 9)]
    c.decode(toks[:40])
    _regroup([c], 40, 0, 2, 32)
    assert c.next_pos != c.n_past
    c.bench_kernel(0, 4)
    assert c.n_past == 0 and c.next_pos == 0
    c.decode(toks[40:]); fresh.decode(toks[40:])
    assert np.array_equal(c.logits(), fresh.logits())
    c.close(); fresh.close(); m.close()
