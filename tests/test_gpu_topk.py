"""The device threshold top-64 (topk_select_kernel) on every path that leaves a selection behind, against numpy's sort of the row
the context itself reports (logit descending, ties to the lower id), bit for bit: the decode step on both batch-1 forms, the
prompt prefill, the decode loop, both verify forms, a restored state, the edit pass with no edits and the batched step."""
import numpy as np
import pytest

import penalty_ref as pr
from blama_b200 import gguf_synth as gs

pytestmark = pytest.mark.gpu

NAME = "small-llama-q4km"
BATCH_MAX = 64


def _same(got, want):
    assert np.array_equal(got["token"], want["token"]), (got["token"][:12], want["token"][:12])
    assert np.array_equal(got["logit"].view(np.uint32), want["logit"].astype(np.float32).view(np.uint32))


def _model(gguf_path, monkeypatch, persistent: bool):
    from blama_b200 import capi

    if not persistent:
        monkeypatch.setenv("BLK_MEGA", "0")                  # read when the model is loaded
    m = capi.Model(gguf_path(NAME))
    monkeypatch.delenv("BLK_MEGA", raising=False)
    return m


def _check(c):
    """the context's raw top-64 is the sorted head of its logits row; the edit pass with no edits selects the same list"""
    want = pr.topk(c.logits(), 64)
    _same(c.topk(64), want)
    _same(c.topk_edited(), want)
    return want


@pytest.mark.parametrize("persistent", [True, False], ids=["persistent", "per-op"])
def test_topk_matches_the_logits_row_on_every_path(persistent, gguf_path, monkeypatch):
    from blama_b200 import capi

    m = _model(gguf_path, monkeypatch, persistent)
    c = capi.Ctx(m, 256)
    assert c.persistent_decode == persistent
    toks = [int(t) for t in gs.synth_prompt(NAME, 120, 17)]
    c.decode(toks[:40])                                      # >= 32 tokens: the prefill path (topk_of_logits)
    _check(c)
    c.decode([toks[40]])                                     # one decode step
    _check(c)
    for t in toks[41:44]:
        got = c.decode_topk(t, 64)
        want = _check(c)
        _same(got, want)
    raw, ed = c.decode_topk_edited(toks[44])
    want = _check(c)
    _same(raw, want); _same(ed, want)
    c.decode_loop(toks[45], 6)
    _check(c)
    if persistent:                                           # the kernel alone leaves chunk maxima behind; the next step must not see them
        c.bench_kernel(5, 8)
        c.decode([toks[46]])
        _check(c)
    # a restored state carries the selection and its logits row
    c2 = capi.Ctx(m, 256)
    c2.state_set(c.state_get())
    _check(c2)
    c2.decode([toks[47]])
    _check(c2)
    # verify mode 0: the batched prefill of >= 32 tokens; mode 1: one decode step per token
    claimed = np.tile(np.arange(10, dtype=np.int32), (40, 1))
    c.set_verify_mode(0)
    c.verify_prefill(toks[48:88], claimed)
    _check(c)
    c.set_verify_mode(1)
    _, top = c.verify_prefill(toks[88:96], claimed[:8])
    want = _check(c)
    _same(top[-1], want[:10])
    c.close(); c2.close(); m.close()


def test_batched_raw_and_unedited_lists_agree_on_every_row(gguf_path):
    from blama_b200 import capi

    m = capi.Model(gguf_path(NAME))
    ctxs = [capi.Ctx(m, 128) for _ in range(BATCH_MAX)]
    ws = capi.Ctx(m, 128)
    for i, c in enumerate(ctxs):
        c.decode([int(t) for t in gs.synth_prompt(NAME, 3 + i % 5, 200 + i)])
    for step, n in enumerate([1, 7, BATCH_MAX, 7]):          # the edit rows grow (1 -> 7 -> 64) and are reused
        toks = [int(t) for t in gs.synth_prompt(NAME, n, 300 + step)]
        raw, ed = capi.decode_batch_edited(ws, ctxs[:n], toks, [([], 1.0, 0.0, 0.0)] * n, 64)
        for i in range(n):
            _same(ed[i], raw[i])
            assert np.all(np.isfinite(raw[i]["logit"])) and np.all(np.diff(raw[i]["logit"]) <= 0), (n, i)
    for c in ctxs + [ws]:
        c.close()
    m.close()
