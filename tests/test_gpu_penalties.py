"""Logit bias and repetition penalties on the device: the edit pass (logit_edit_kernel + the threshold selector on the edited
copy) against the numpy restatement (tests/penalty_ref.py), bit for bit; a Session with the stages on both batch-1 paths and
after every operation that leaves a logits row; the batched step; the batching server."""
import math

import numpy as np
import pytest

import penalty_ref as pr
from blama_b200 import gguf_synth as gs

pytestmark = pytest.mark.gpu

STAGES = dict(penalty_last_n=16, repeat_penalty=1.3, freq_penalty=0.2, present_penalty=0.3)


def _chunk(V: int) -> int:
    shift = 6
    while (V + (1 << shift) - 1) >> shift > 256:
        shift += 1
    return 1 << shift


def _same(got, want):
    assert np.array_equal(got["token"], want["token"]), (got["token"][:12], want["token"][:12])
    assert np.array_equal(got["logit"].view(np.uint32), want["logit"].astype(np.float32).view(np.uint32))


@pytest.mark.parametrize("V", [32000, 128256, 152064])
def test_edit_pass_matches_numpy(V):
    from blama_b200 import capi

    rng = np.random.default_rng(V)
    c = _chunk(V)
    base = (rng.standard_normal((6, V)) * 2.0).astype(np.float32)
    rows = []
    # 0: edits on chunk boundaries and at the last id, ids that the raw top-64 holds, penalised
    ids = sorted({0, c - 1, c, 2 * c - 1, 2 * c, 5 * c, V - 2, V - 1})
    base[0, ids] = 8.0 + np.arange(len(ids), dtype=np.float32) * 0.25
    base[0, ids[::2]] *= -1.0                                     # negative logits: the repeat penalty multiplies
    rows.append(([(t, 1 + k % 3, 0.0 if k % 2 else 0.5) for k, t in enumerate(ids)], 1.3, 0.2, 0.4))
    # 1: an id from below raw rank 1000 lifted into the top 40 by its bias, another to the very top
    order = np.argsort(-base[1], kind="stable")
    lift, top = int(order[1500]), int(order[4000])
    rows.append((sorted([(lift, 0, float(base[1, order[20]] - base[1, lift]) + 0.01), (top, 0, float(base[1].max() - base[1, top]) + 1.0)]),
                 1.0, 0.0, 0.0))
    # 2: the arg-max and the next nine banned
    rows.append((sorted((int(t), 0, -math.inf) for t in np.argsort(-base[2], kind="stable")[:10]), 1.0, 0.0, 0.0))
    # 3: a degenerate row of equal logits (the selector's exact fallback), a few ids edited
    base[3] = 1.0
    rows.append(([(3, 2, 0.0), (70, 0, -1.0), (c + 1, 1, 0.0), (V - 1, 0, 0.5)], 1.1, 0.1, 0.0))
    # 4: no edits
    rows.append(([], 1.0, 0.0, 0.0))
    # 5: thousands of bans plus penalties on the raw top-64
    bans = set(int(t) for t in rng.choice(V, 3000, replace=False))
    pen = set(int(t) for t in np.argsort(-base[5], kind="stable")[:64])
    rows.append((sorted((t, 2 if t in pen else 0, -math.inf if t in bans else 0.0) for t in bans | pen), 1.5, 0.3, 0.2))
    got = capi.test_logit_edits(base, rows, 64)
    for r, (edits, rep, fr, pres) in enumerate(rows):
        e = np.array(edits, dtype=pr.EDIT_DTYPE)
        want = pr.topk(pr.apply_edits(base[r], e, rep, fr, pres), 64)
        _same(got[r], want)
    assert lift in got[1]["token"][:40].tolist() and int(got[1]["token"][0]) == top
    assert int(np.argmax(base[2])) not in got[2]["token"].tolist()


@pytest.mark.parametrize("edits,repeat", [
    ([(5, 0, 1.0), (5, 0, 1.0)], 1.0),          # duplicate id
    ([(7, 0, 1.0), (3, 0, 1.0)], 1.0),          # descending
    ([(32000, 0, 1.0)], 1.0),                   # out of range
    ([(-1, 0, 1.0)], 1.0),
    ([(3, -1, 0.0)], 1.1),                      # negative count
    ([(3, 0, math.nan)], 1.0),
    ([(3, 0, math.inf)], 1.0),
    ([(3, 1, 0.0)], 0.0),                       # repeat must be > 0
])
def test_malformed_edit_lists_are_refused(edits, repeat):
    from blama_b200 import capi

    row = np.zeros((1, 32000), dtype=np.float32)
    with pytest.raises(capi.BlkError) as e:
        capi.test_logit_edits(row, [(edits, repeat, 0.0, 0.0)], 10)
    assert e.value.code == 4


def _model(gguf_path, monkeypatch, persistent: bool, name="small-llama-q4km"):
    from blama_b200 import host_api as H

    if not persistent:
        monkeypatch.setenv("BLK_MEGA", "0")
    H.lib()
    return H.Model(gguf_path(name))


def _check_session(inst, hist, bias, stages=STAGES):
    ctx = inst.raw_ctx()
    row = ctx.logits()
    want = pr.topk(pr.edited_row(row, hist, stages["penalty_last_n"], stages["repeat_penalty"], stages["freq_penalty"],
                                 stages["present_penalty"], bias), 64)
    _same(inst.sampling_candidates(), want)
    return row


@pytest.mark.parametrize("persistent", [True, False])
def test_session_steps_match_numpy(gguf_path, monkeypatch, persistent):
    from blama_b200 import host_api as H

    name = "small-llama-q4km"
    m = _model(gguf_path, monkeypatch, persistent, name)
    inst = H.Instance(m, 256)
    V = inst.raw_ctx().m.n_vocab
    prompt = [int(t) for t in gs.synth_prompt(name, 40, 3)]             # >= 32 tokens: the prompt prefill path
    bias = {11: 6.0, 250: -math.inf, V - 1: 4.5, 1000: 2.0}
    inst.start_session(seed=1, logit_bias=bias, **STAGES).set_initial_prompt(prompt)
    assert inst.raw_ctx().persistent_decode == persistent
    hist = list(prompt)
    _check_session(inst, hist, bias)
    launches = inst.raw_ctx().kernel_launches
    for _ in range(10):
        toks, top = inst.complete(1)
        if len(toks) == 0:
            break
        assert int(toks[0]) != 250
        hist.append(int(toks[0]))
        row = _check_session(inst, hist, bias)
        _same(top[0], pr.topk(row, 10))                                  # the reported top-10 stays the raw row's
    assert inst.raw_ctx().kernel_launches > launches
    # state restore: a new session's sampler has an empty window; the restored row is edited by the bias alone
    blob = inst.get_state()
    inst2 = H.Instance(m, 256)
    inst2.start_session(seed=1, logit_bias=bias, **STAGES)
    inst2.set_state(blob)
    _check_session(inst2, [], bias)
    # a sampler replaced after a decode: the kept row, re-selected with the new stages
    other = dict(penalty_last_n=4, repeat_penalty=1.7, freq_penalty=0.0, present_penalty=0.5)
    inst.reset_sampler(seed=2, logit_bias={5: 3.0}, **other)
    _check_session(inst, [], {5: 3.0}, other)
    toks, _ = inst.complete(1)
    _check_session(inst, [int(toks[0])], {5: 3.0}, other)
    inst.close(); inst2.close(); m.close()


def test_batched_fill_leaves_the_last_response_token_in_the_window(gguf_path, monkeypatch):
    from blama_b200 import host_api as H

    name = "small-llama-q4km"
    m = _model(gguf_path, monkeypatch, True, name)
    prompt = [int(t) for t in gs.synth_prompt(name, 12, 4)]
    resp = [int(t) for t in gs.synth_prompt(name, 40, 5)]           # >= 32: the batched fill runs the prefill path
    bias = {17: 3.0}
    for sequential in (False, True):
        inst = H.Instance(m, 256)
        inst.start_session(seed=1, sequential_verify=sequential, logit_bias=bias, **STAGES).set_initial_prompt(prompt)
        claimed = np.zeros((len(resp), 10), dtype=H.TD_DTYPE)
        inst.fill_ctx(resp, claimed, np.zeros(len(resp), dtype=np.int32))
        edits, _ = inst.logit_edits()
        # the reference's fillCtx pushes each response token as a prompt of its own: reset, accept -- only the last remains
        assert edits.tolist() == pr.edit_list(inst.raw_ctx().m.n_vocab, [resp[-1]], bias=bias, **_kw(STAGES)).tolist()
        _check_session(inst, [resp[-1]], bias)
        inst.close()
    m.close()


def _kw(stages):
    return dict(last_n=stages["penalty_last_n"], repeat=stages["repeat_penalty"], freq=stages["freq_penalty"], present=stages["present_penalty"])


def test_default_parameters_launch_what_the_plain_path_launches(gguf_path):
    from blama_b200 import capi, host_api as H

    name = "small-llama-q4km"
    path = gguf_path(name)
    H.lib()
    m = H.Model(path)
    inst = H.Instance(m, 256)
    prompt = [int(t) for t in gs.synth_prompt(name, 10, 6)]
    inst.start_session(seed=2).set_initial_prompt(prompt)
    ctx = inst.raw_ctx()
    l0 = ctx.kernel_launches
    toks, top = inst.complete(12)
    used = ctx.kernel_launches - l0
    # the parent's path through the C ABI: the prompt, then one blk_decode_topk per emitted token
    cm = capi.Model(path)
    c = capi.Ctx(cm, 256)
    c.decode(prompt)
    c0 = c.kernel_launches
    for i, t in enumerate(toks):
        _same(c.decode_topk(int(t), 10), top[i])
    assert c.kernel_launches - c0 == used
    c.close(); cm.close(); inst.close(); m.close()


def test_edited_decode_refuses_a_bad_list_before_launching(gguf_path):
    from blama_b200 import capi

    name = "small-llama-q4km"
    cm = capi.Model(gguf_path(name))
    c = capi.Ctx(cm, 256)
    c.decode([int(t) for t in gs.synth_prompt(name, 8, 1)])
    n_past, launches = c.n_past, c.kernel_launches
    with pytest.raises(capi.BlkError) as e:
        c.decode_topk_edited(5, [(9, 0, 1.0), (4, 0, 1.0)])
    assert e.value.code == 4 and c.n_past == n_past and c.kernel_launches == launches
    raw, ed = c.decode_topk_edited(5, [(9, 0, 1.0)], k=64)
    row = c.logits()
    _same(raw, pr.topk(row, 64))
    _same(ed, pr.topk(pr.apply_edits(row, np.array([(9, 0, 1.0)], dtype=pr.EDIT_DTYPE)), 64))
    c.close(); cm.close()


def test_complete_matches_oracle_session_with_penalties(gguf_path, oracle):
    """the CUDA Session and the oracle's Session restated with the two stages (numpy edits + the oracle's chain) emit the same
    tokens while the arithmetic stays on the clean branch, as test_complete_matches_oracle_session"""
    from blama_b200 import host_api as H

    name = "tiny-llama-q8"
    path = gguf_path(name)
    prompt = [int(t) for t in gs.synth_prompt(name, 10, 6)]
    om = oracle.Model(path)
    oc = oracle.Ctx(om, 128, oracle.MODE_GGML, 2)
    bias = {7: 2.0, 100: -math.inf}
    row = oc.decode(prompt)[0]
    s = oracle.Sampler(seed=5)
    hist = list(prompt)
    want_t, want_top = [], []
    for _ in range(16):
        tok = s.sample(pr.edited_row(row, hist, bias=bias, **_kw(STAGES)))
        if om.is_eog(tok):
            break
        row = oc.decode([tok])[0]
        hist.append(tok)
        want_t.append(tok); want_top.append(pr.topk(row, 10))
    hm = H.Model(path)
    inst = H.Instance(hm, 128)
    inst.start_session(seed=5, logit_bias=bias, **STAGES).set_initial_prompt(prompt)
    got_t, got_top = inst.complete(16)
    n_same = 0
    for i in range(min(len(want_t), len(got_t))):
        if want_t[i] != got_t[i]:
            break
        n_same += 1
        assert np.abs(got_top[i]["logit"] - want_top[i]["logit"]).max() <= 0.25
    assert n_same >= 4, (want_t, got_t)
    s.close(); inst.close(); hm.close(); oc.close(); om.close()


def test_decode_batch_edited_matches_oracle_bf16(gguf_path, oracle):
    from blama_b200 import capi

    name = "small-llama-q4km"
    path = gguf_path(name)
    m = capi.Model(path)
    om = oracle.Model(path)
    lens = [40, 33, 70]
    ctxs = [capi.Ctx(m, 256) for _ in lens]
    ocs = [oracle.Ctx(om, 256, oracle.MODE_BF16, 4) for _ in lens]
    ws = capi.Ctx(m, 256)
    for i, n in enumerate(lens):
        p = gs.synth_prompt(name, n, 50 + i)
        ctxs[i].decode(p); ocs[i].decode(p)
    worst = 0.0
    for step in range(4):
        toks = [int(t) for t in gs.synth_prompt(name, len(lens), 90 + step)]
        per_row = [
            ([], 1.0, 0.0, 0.0),                                                          # no edits: edited == raw
            ([(t, 0, b) for t, b in sorted({3: 5.0, int(toks[1]): -math.inf}.items())], 1.0, 0.0, 0.0),     # bias only
            (sorted((int(t), 1 + k % 2, 0.0) for k, t in enumerate(set(toks + [1, 2, 9, 40]))), 1.4, 0.2, 0.1),
        ]
        raw, ed = capi.decode_batch_edited(ws, ctxs, toks, per_row, 64)
        _same(ed[0], raw[0])
        for i in range(len(lens)):
            want = ocs[i].decode([toks[i]])[0]
            e = np.array(per_row[i][0], dtype=pr.EDIT_DTYPE)
            want_ed = pr.apply_edits(want, e, *per_row[i][1:])
            fin = np.isfinite(ed[i]["logit"])
            assert np.all(np.diff(ed[i]["logit"][fin]) <= 0)
            worst = max(worst, float(np.abs(ed[i]["logit"][fin] - want_ed[ed[i]["token"][fin]]).max()))
            worst = max(worst, float(np.abs(raw[i]["logit"] - want[raw[i]["token"]]).max()))
        assert int(toks[1]) not in ed[1]["token"].tolist()
    assert worst <= 0.15, worst
    for c in ctxs + [ws]:
        c.close()
    for o in ocs:
        o.close()
    m.close(); om.close()


def test_batching_server_with_penalties(gguf_path):
    from blama_b200 import host_api as H

    name = "small-llama-q4km"
    H.lib()
    m = H.Model(gguf_path(name))
    plain = H.Server([m], ctx_size=512)
    batched = H.Server([m], ctx_size=512, max_batch=4)
    prompts = [gs.synth_prompt(name, 6 + 3 * k, 70 + k) for k in range(7)]
    free = plain.wait_complete(plain.submit_complete(prompts[0], 20, seed=3))
    banned = int(free[0][0])
    stages = dict(STAGES, logit_bias={banned: -math.inf, 12: 1.5})
    # a lone request on the batching server takes the batch-1 path: bit-identical to the plain server
    a = plain.wait_complete(plain.submit_complete(prompts[0], 20, seed=3, **stages))
    b = batched.wait_complete(batched.submit_complete(prompts[0], 20, seed=3, **stages))
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1]["logit"], b[1]["logit"])
    assert banned not in a[0].tolist()
    want_len = [24, 40, 8, 33, 16, 40, 5]
    tickets = [batched.submit_complete(p, n, seed=k, **(stages if k % 2 == 0 else dict(penalty_last_n=8, repeat_penalty=1.2)))
               for k, (p, n) in enumerate(zip(prompts, want_len))]
    got = [batched.wait_complete(t) for t in tickets]
    assert batched.last_worker_error() == ""
    for k, g in enumerate(got):
        assert len(g[0]) == want_len[k]
        if k % 2 == 0:
            assert banned not in g[0].tolist()
        s = plain.wait_verify(plain.submit_verify(prompts[k], g[0], g[1], g[2], seed=k))
        assert s >= 0.95, (k, s)
    batched.close(); plain.close(); m.close()
