"""Logit bias and repetition penalties in the host Sampler (no device): its full-row path draws what the oracle's sampler chain
draws from the row edited by the numpy restatement (tests/penalty_ref.py), draw for draw, and its edit list (what the device
edit pass receives) equals the restatement's."""
import math

import numpy as np
import pytest

import penalty_ref as pr

V = 3000


@pytest.fixture(scope="module")
def host():
    from blama_b200 import host_api

    host_api.lib_nodevice()
    return host_api


def _row(seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    row = (rng.standard_normal(V) * 3.0 - 1.0).astype(np.float32)      # mostly negative: the repeat penalty multiplies there
    return row


def _oracle_draws(oracle, row, n, history, seed, temp, top_p, top_k, min_p, last_n, repeat, freq, present, bias):
    s = oracle.Sampler(seed=seed, temp=temp, top_p=top_p, top_k=top_k, min_p=min_p)
    hist = list(history)
    out = []
    for _ in range(n):
        tok = s.sample(pr.edited_row(row, hist, last_n, repeat, freq, present, bias))
        out.append(tok)
        hist.append(tok)
    s.close()
    return np.array(out, dtype=np.int32)


CASES = [
    # (last_n, repeat, freq, present, bias builder, temp, top_p, top_k)
    (64, 1.1, 0.1, 0.1, lambda top: {}, 0.8, 0.95, 40),
    (64, 1.3, 0.0, 0.0, lambda top: {int(top[0]): -math.inf}, 0.8, 0.95, 40),                 # the arg-max banned
    (8, 1.1, 0.5, 0.3, lambda top: {int(top[2000]): 12.0, int(top[5]): -2.5}, 1.0, 0.9, 40),  # window shorter than the history
    (0, 1.5, 0.4, 0.4, lambda top: {int(top[900]): 9.0}, 0.7, 0.95, 40),                      # numTokens 0: bias only
    (32, 0.9, -0.2, 0.0, lambda top: {}, 0.0, 0.95, 40),                                        # greedy, repeat < 1
    (64, 1.2, 0.05, 0.2, lambda top: {int(t): -math.inf for t in top[:30]}, 0.8, 1.0, 0),    # top-k off, many bans
]


@pytest.mark.parametrize("case", range(len(CASES)))
@pytest.mark.parametrize("seed", [0, 7, 1234])
def test_full_row_draws_match_oracle(host, oracle, case, seed):
    last_n, repeat, freq, present, mk_bias, temp, top_p, top_k = CASES[case]
    row = _row(seed + 100 * case)
    top = np.argsort(-row, kind="stable")
    bias = mk_bias(top)
    # a history that repeats the best ids, so the penalties reorder the head of the row
    history = [int(t) for t in np.concatenate([top[:12], top[:6], top[3:9], top[40:60]])]
    got = host.sampler_draw_penalized(row, 24, history, seed=seed, temp=temp, top_p=top_p, top_k=top_k, min_p=0.05, penalty_last_n=last_n,
                                      repeat_penalty=repeat, freq_penalty=freq, present_penalty=present, logit_bias=bias)
    want = _oracle_draws(oracle, row, 24, history, seed, temp, top_p, top_k, 0.05, last_n, repeat, freq, present, bias)
    assert np.array_equal(got, want), (got, want)
    if bias and any(v == -math.inf for v in bias.values()):
        assert not set(got.tolist()) & {k for k, v in bias.items() if v == -math.inf}


def test_defaults_draw_what_the_plain_chain_draws(host, oracle):
    row = _row(5)
    got = host.sampler_draw_penalized(row, 16, [1, 2, 3], seed=3)
    s = oracle.Sampler(seed=3)
    want = [s.sample(row) for _ in range(16)]
    assert got.tolist() == want


@pytest.mark.parametrize("last_n", [0, 1, 5, 64])
def test_edit_list_matches_numpy(host, last_n):
    rng = np.random.default_rng(last_n)
    history = rng.integers(0, 50, size=40).tolist()
    bias = {3: 1.25, 7: -math.inf, 11: 0.0, 49: -0.5, V + 5: 2.0, -1: 1.0}      # out-of-vocabulary ids and zero biases edit nothing
    got, params = host.sampler_logit_edits(V, history, last_n, 1.1, 0.25, 0.5, bias)
    want = pr.edit_list(V, history, last_n, 1.1, 0.25, 0.5, bias)
    assert got.tolist() == want.tolist()
    if pr.penalties_active(last_n, 1.1, 0.25, 0.5):
        assert params == (np.float32(1.1), 0.25, 0.5)
    # inactive penalties: the window counts are not listed
    got, _ = host.sampler_logit_edits(V, history, last_n, 1.0, 0.0, 0.0, bias)
    assert got.tolist() == pr.edit_list(V, history, last_n, 1.0, 0.0, 0.0, bias).tolist()
    assert (got["count"] == 0).all()


def test_reset_empties_the_window(host):
    got, _ = host.sampler_logit_edits(V, [4, 4, 9], 64, 1.3, 0.0, 0.0, {2: 1.0}, reset_after=True)
    assert got.tolist() == [(2, 0, 1.0)]
    got, _ = host.sampler_logit_edits(V, [4, 4, 9], 64, 1.3, 0.0, 0.0, None, reset_after=False)
    assert got.tolist() == [(4, 2, 0.0), (9, 1, 0.0)]


def test_edited_values_are_bit_exact(host, oracle):
    """the host's edit arithmetic against the restatement on awkward values (greedy draw = arg-max of the edited row)"""
    row = np.array([-0.0, 0.0, -1e-30, 3.5, -7.25, 1e30, -1e30, 0.1, -0.1, 2.0], dtype=np.float32)
    for tgt in range(len(row)):
        history = [tgt, tgt, tgt, (tgt + 1) % len(row)]
        bias = {tgt: 50.0}
        got = host.sampler_draw_penalized(row, 1, history, temp=0.0, top_k=40, min_p=0.0, penalty_last_n=64, repeat_penalty=1.7,
                                          freq_penalty=0.3, present_penalty=0.9, logit_bias=bias)
        want = int(np.argmax(pr.edited_row(row, history, 64, 1.7, 0.3, 0.9, bias)))
        assert got[0] == want


@pytest.mark.parametrize("bad", [math.nan, math.inf])
def test_nan_and_plus_inf_biases_are_rejected(host, bad):
    with pytest.raises(host.HostError, match="NaN or \\+inf"):
        host.sampler_draw_penalized(_row(0), 1, logit_bias={5: bad})


def test_bad_penalties_are_rejected(host):
    with pytest.raises(host.HostError, match="must not be negative"):
        host.sampler_draw_penalized(_row(0), 1, penalty_last_n=-1, repeat_penalty=1.1)
    with pytest.raises(host.HostError, match="repeat penalty > 0"):
        host.sampler_draw_penalized(_row(0), 1, repeat_penalty=0.0)
    # a negative window with the stage off changes nothing and stays accepted
    host.sampler_draw_penalized(_row(0), 1, penalty_last_n=-1)


def test_mirostat_and_grammar_still_raise(host):
    with pytest.raises(host.HostError, match="mirostat"):
        host.sampler_check(mirostat=2)
    with pytest.raises(host.HostError, match="grammar"):
        host.sampler_check(grammar="root ::= \"a\"")
    host.sampler_check()
