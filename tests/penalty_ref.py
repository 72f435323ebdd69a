"""numpy restatement of the logit-bias and repetition-penalty stages (llama.cpp b5187 llama_sampler_logit_bias_apply and
llama_sampler_penalties_apply, as blama configures its chain), shared by the CPU and GPU tests.

Every operation is a float32 numpy scalar operation (correctly rounded, never fused), so the edited logits are bit-equal to
those of the host Sampler and of the device edit kernel."""
from __future__ import annotations

from collections import Counter

import numpy as np

F32 = np.float32
EDIT_DTYPE = np.dtype([("token", np.int32), ("count", np.int32), ("bias", np.float32)])


def penalties_active(last_n: int, repeat: float, freq: float, present: float) -> bool:
    return last_n > 0 and (F32(repeat), F32(freq), F32(present)) != (F32(1), F32(0), F32(0))


def window_counts(history, last_n: int) -> Counter:
    """ids of the last last_n accepted tokens with their counts (the penalty sampler's ring buffer)"""
    return Counter(int(t) for t in list(history)[-last_n:]) if last_n > 0 else Counter()


def edit_list(n_vocab: int, history=(), last_n: int = 64, repeat: float = 1.0, freq: float = 0.0, present: float = 0.0, bias=None):
    """one (token, count, bias) per edited id in [0, n_vocab), ascending; zero biases and inactive penalties edit nothing"""
    bias = {int(k): F32(v) for k, v in (bias or {}).items() if 0 <= int(k) < n_vocab}
    counts = window_counts(history, last_n) if penalties_active(last_n, repeat, freq, present) else Counter()
    ids = sorted(set(k for k, v in bias.items() if v != 0) | set(k for k in counts if 0 <= k < n_vocab))
    return np.array([(t, counts.get(t, 0), bias.get(t, F32(0))) for t in ids], dtype=EDIT_DTYPE)


def edit_value(logit, count: int, bias, repeat, freq, present):
    l = F32(logit)
    if F32(bias) != 0:
        l = F32(l + F32(bias))
    if count > 0:
        l = F32(l * F32(repeat)) if l <= 0 else F32(l / F32(repeat))
        l = F32(l - F32(F32(F32(count) * F32(freq)) + F32(present)))
    return l


def apply_edits(row: np.ndarray, edits: np.ndarray, repeat: float = 1.0, freq: float = 0.0, present: float = 0.0) -> np.ndarray:
    out = np.array(row, dtype=np.float32, copy=True)
    for t, c, b in edits:
        out[t] = edit_value(out[t], int(c), b, repeat, freq, present)
    return out


def edited_row(row: np.ndarray, history=(), last_n: int = 64, repeat: float = 1.0, freq: float = 0.0, present: float = 0.0, bias=None):
    return apply_edits(row, edit_list(len(row), history, last_n, repeat, freq, present, bias), repeat, freq, present)


def topk(row: np.ndarray, k: int) -> np.ndarray:
    """logit descending, ties to the lower id (the device selector's order)"""
    order = np.lexsort((np.arange(len(row)), -row.astype(np.float64)))[:k]
    out = np.zeros(k, dtype=[("token", np.int32), ("logit", np.float32)])
    out["token"] = order
    out["logit"] = row[order]
    return out
