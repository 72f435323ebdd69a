"""ctypes view of the C ABI in include/blama_b200.h (the library a blama maintainer would bind; see INTEGRATION.md).

This module is the thin Python harness the tests and bench.py drive the product through.  It loads
blama_b200/lib/libblama_b200.so and fails loudly if the library is missing or no CUDA device is present:
there is no CPU fallback and nothing under oracle/ is ever imported from here."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence, Tuple

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# BLAMA_B200_LIB: an alternative build of the same library (build-against-build A/B runs: tools/decode_lib_ab.py)
LIB_PATH = os.environ.get("BLAMA_B200_LIB") or os.path.join(HERE, "lib", "libblama_b200.so")

TD_DTYPE = np.dtype([("token", np.int32), ("logit", np.float32)])

# every symbol include/blama_b200.h declares: name -> (restype, argtypes)
_vp, _i32, _i64, _f32p = C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_float)
LOG_CB = C.CFUNCTYPE(None, C.c_int, C.c_char_p, C.c_void_p)
PROGRESS_CB = C.CFUNCTYPE(C.c_int32, C.c_float, C.c_void_p)
SYMBOLS = {
    "blk_init": (_i32, []),
    "blk_set_log_callback": (None, [LOG_CB, _vp]),
    "blk_last_error": (C.c_char_p, []),
    "blk_device_count": (_i32, []),
    "blk_version": (C.c_char_p, []),
    "blk_model_load": (_vp, [C.c_char_p, _i32, PROGRESS_CB, _vp]),
    "blk_model_load_vocab": (_vp, [C.c_char_p]),
    "blk_model_free": (None, [_vp]),
    "blk_model_add_eos": (_i32, [_vp]),
    "blk_model_vocab_only": (_i32, [_vp]),
    "blk_model_token_type": (_i32, [_vp, _i32]),
    "blk_model_n_merges": (_i32, [_vp]),
    "blk_model_merge_text": (_i32, [_vp, _i32, C.c_char_p, _i32]),
    "blk_model_n_vocab": (_i32, [_vp]),
    "blk_model_n_ctx_train": (_i32, [_vp]),
    "blk_model_n_embd": (_i32, [_vp]),
    "blk_model_n_layer": (_i32, [_vp]),
    "blk_model_token_bos": (_i32, [_vp]),
    "blk_model_token_eos": (_i32, [_vp]),
    "blk_model_is_eog": (_i32, [_vp, _i32]),
    "blk_model_add_bos": (_i32, [_vp]),
    "blk_model_device": (_i32, [_vp]),
    "blk_model_weight_bytes_per_token": (_i64, [_vp]),
    "blk_model_kv_bytes_per_token": (_i64, [_vp]),
    "blk_model_panel_bytes": (_i64, [_vp, _vp, _vp]),
    "blk_model_token_text": (_i32, [_vp, _i32, C.c_char_p, _i32]),
    "blk_model_meta_str": (_i32, [_vp, C.c_char_p, C.c_char_p, _i32]),
    "blk_ctx_create": (_vp, [_vp, _i32, _i32]),
    "blk_ctx_free": (None, [_vp]),
    "blk_ctx_n_ctx": (_i32, [_vp]),
    "blk_ctx_n_batch": (_i32, [_vp]),
    "blk_ctx_n_past": (_i32, [_vp]),
    "blk_ctx_model": (_vp, [_vp]),
    "blk_kv_clear": (_i32, [_vp]),
    "blk_sync": (_i32, [_vp]),
    "blk_kv_shift": (_i32, [_vp, _i32, _i32]),
    "blk_kv_seq_add": (_i32, [_vp, _i32, _i32, _i32]),
    "blk_kv_seq_div": (_i32, [_vp, _i32, _i32, _i32]),
    "blk_ctx_next_pos": (_i32, [_vp]),
    "blk_state_size": (_i64, [_vp]),
    "blk_state_get": (_i32, [_vp, _vp, _i64, C.POINTER(_i64)]),
    "blk_state_set": (_i32, [_vp, _vp, _i64]),
    "blk_decode": (_i32, [_vp, _vp, _i32]),
    "blk_topk_last": (_i32, [_vp, _i32, _vp]),
    "blk_gather_last": (_i32, [_vp, _vp, _i32, _vp]),
    "blk_get_logits_last": (_i32, [_vp, _vp]),
    "blk_decode_topk": (_i32, [_vp, _i32, _i32, _vp]),
    "blk_decode_loop": (_i32, [_vp, _i32, _i32, C.POINTER(_i32)]),
    "blk_decode_batch": (_i32, [_vp, _vp, _vp, _i32, _i32, _vp]),
    "blk_decode_topk_edited": (_i32, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "blk_topk_last_edited": (_i32, [_vp, _i32, _vp, _vp]),
    "blk_decode_batch_edited": (_i32, [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "blk_verify_prefill": (_i32, [_vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "blk_ctx_set_verify_mode": (_i32, [_vp, _i32]),
    "blk_timer_start": (_i32, [_vp]),
    "blk_timer_stop": (_i32, [_vp, _f32p]),
    "blk_ctx_kernel_launches": (_i64, [_vp]),
    "blk_ctx_persistent_decode": (_i32, [_vp]),
    "blk_debug_trace": (_i32, [_vp, _vp, _i32, _vp, _vp]),
    "blk_flush_l2": (_i32, [_vp]),
    "blk_profile_step": (_i32, [_vp, _i32, C.c_char_p, _i32]),
    "blk_profile_verify": (_i32, [_vp, _vp, _i32, C.c_char_p, _i32]),
    "blk_bench_kernel": (_i32, [_vp, _i32, _i32, _f32p, C.POINTER(C.c_int64)]),
    "blk_test_gemv": (_i32, [_i32, _i32, _vp, _i64, _i64, _vp, _vp]),
    "blk_test_gemm": (_i32, [_i32, _i32, _vp, _i32, _i64, _vp, _i64, _i32, _i32, _vp, C.c_float, _vp, _vp, _vp]),
    "blk_bench_gemm": (_i32, [_i32, _i32, _vp, _i64, _i64, _i64, _i32, _f32p]),
    "blk_test_dequant": (_i32, [_i32, _i32, _vp, _i64, _i64, _vp]),
    "blk_test_rmsnorm": (_i32, [_i32, _vp, _vp, _i32, _i32, C.c_float, _vp]),
    "blk_test_qkv_post": (_i32, [_i32, _vp, _i32, _i32, _i32, _i32, _i32, _i32, C.c_float, _vp, _vp, _vp, _vp]),
    "blk_test_prefill_attn": (_i32, [_i32, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, C.POINTER(_i32)]),
    "blk_test_decode_attn": (_i32, [_i32, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i64, _vp, C.POINTER(_i32)]),
    "blk_test_decode_attn_batch": (_i32, [_i32, _i32, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i64, _vp]),
    "blk_test_logit_edits": (_i32, [_i32, _vp, _i32, _i32, _vp, _i32, _vp]),
    "blk_test_row_topk": (_i32, [_i32, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "blk_test_claimed_logits": (_i32, [_i32, _i32, _vp, _i64, _i64, _vp, _i32, _vp, _vp, _vp]),
}

_lib: Optional[C.CDLL] = None


class BlkError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[blk status {code}] {msg}")
        self.code = code
        self.msg = msg


def lib() -> C.CDLL:
    """Load the CUDA engine.  Raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(blama_b200 has no CPU fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def _check(rc: int) -> None:
    if rc != 0:
        raise BlkError(rc, (lib().blk_last_error() or b"").decode(errors="replace"))


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def init() -> None:
    _check(lib().blk_init())


def test_rmsnorm(x: np.ndarray, w: np.ndarray, eps: float, device: int = 0) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.float32); w = np.ascontiguousarray(w, dtype=np.float32)
    out = np.zeros_like(x)
    _check(lib().blk_test_rmsnorm(device, _p(x), _p(w), x.shape[0], x.shape[1], eps, _p(out)))
    return out


def test_qkv_post(qkv: np.ndarray, n_head: int, n_head_kv: int, d_head: int, neox: bool, pos0: int, theta: float, freq_factors=None, device: int = 0):
    qkv = np.ascontiguousarray(qkv, dtype=np.float32)
    T = qkv.shape[0]
    q = np.zeros((T, n_head * d_head), dtype=np.float32); k = np.zeros((T, n_head_kv * d_head), dtype=np.float32); v = np.zeros_like(k)
    ff = None if freq_factors is None else np.ascontiguousarray(freq_factors, dtype=np.float32)
    _check(lib().blk_test_qkv_post(device, _p(qkv), T, n_head, n_head_kv, d_head, int(neox), pos0, theta, _p(ff) if ff is not None else None, _p(q), _p(k), _p(v)))
    return q, k, v


def test_prefill_attn(q: np.ndarray, k: np.ndarray, v: np.ndarray, pos0: int, n_head: int, n_head_kv: int, d_head: int, device: int = 0):
    q = np.ascontiguousarray(q, dtype=np.float32); k = np.ascontiguousarray(k, dtype=np.float32); v = np.ascontiguousarray(v, dtype=np.float32)
    T = q.shape[0]
    out = np.zeros_like(q)
    tc = _i32(0)
    _check(lib().blk_test_prefill_attn(device, _p(q), _p(k), _p(v), T, pos0, n_head, n_head_kv, d_head, _p(out), C.byref(tc)))
    return out, bool(tc.value)


def test_decode_attn(q: np.ndarray, k: np.ndarray, v: np.ndarray, n_ctx: int, n_head: int, n_head_kv: int, d_head: int, form: int = -1,
                     seed: int = 0, device: int = 0):
    """Decode attention of q [n_head*d_head] over the n_kv = len(k) cells of a context of n_ctx cells.  form: -1 the engine's plan,
    0 the split form, 1 the cluster form.  Returns (out [n_head*d_head] f32, True when the cluster form ran)."""
    q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1)
    k = np.ascontiguousarray(k, dtype=np.float32); v = np.ascontiguousarray(v, dtype=np.float32)
    out = np.zeros_like(q)
    used = _i32(-1)
    _check(lib().blk_test_decode_attn(device, _p(q), _p(k), _p(v), k.shape[0], n_ctx, n_head, n_head_kv, d_head, form, seed, _p(out), C.byref(used)))
    return out, bool(used.value)


def test_decode_attn_batch(q: np.ndarray, k: np.ndarray, v: np.ndarray, n_kv: Sequence[int], n_head: int, n_head_kv: int, d_head: int,
                           seed: int = 0, device: int = 0) -> np.ndarray:
    """Batched decode attention: row b of q [n][n_head*d_head] over its own n_kv[b] cells, whose keys / values are rows
    sum(n_kv[:b]) .. of k / v.  Returns the bf16 output [n][n_head*d_head] as f32."""
    q = np.ascontiguousarray(q, dtype=np.float32)
    k = np.ascontiguousarray(k, dtype=np.float32); v = np.ascontiguousarray(v, dtype=np.float32)
    nk = np.ascontiguousarray(n_kv, dtype=np.int32)
    assert q.shape[0] == nk.shape[0] and k.shape[0] == v.shape[0] == int(nk.sum())
    out = np.zeros_like(q)
    _check(lib().blk_test_decode_attn_batch(device, q.shape[0], _p(q), _p(k), _p(v), _p(nk), n_head, n_head_kv, d_head, seed, _p(out)))
    return out


EDIT_DTYPE = np.dtype([("token", np.int32), ("count", np.int32), ("bias", np.float32)])     # blk_logit_edit


class LogitEdits(C.Structure):
    """blk_logit_edits: one row's (repeat, freq, present) and its edit list, ids ascending"""
    _fields_ = [("repeat", C.c_float), ("freq", C.c_float), ("present", C.c_float), ("edits", C.c_void_p), ("n_edits", C.c_int32)]


def logit_edits(edits=None, repeat: float = 1.0, freq: float = 0.0, present: float = 0.0):
    """(LogitEdits, the array it points into) from [(token, count, bias), ...] or an EDIT_DTYPE array; keep both alive while in use"""
    arr = np.zeros(0, dtype=EDIT_DTYPE) if edits is None else (np.ascontiguousarray(edits) if isinstance(edits, np.ndarray)
                                                               else np.array([tuple(e) for e in edits], dtype=EDIT_DTYPE))
    assert arr.dtype == EDIT_DTYPE
    return LogitEdits(repeat, freq, present, arr.ctypes.data if len(arr) else None, len(arr)), arr


def _edit_rows(per_row):
    """[(edits, repeat, freq, present), ...] -> (LogitEdits array, arrays to keep alive)"""
    made = [logit_edits(*r) for r in per_row]
    return (LogitEdits * len(made))(*[m[0] for m in made]), [m[1] for m in made]


def test_logit_edits(logits: np.ndarray, per_row, k: int = 64, device: int = 0) -> np.ndarray:
    """edited top-k of every row of logits [n][V]; per_row[i] = (edits, repeat, freq, present) as logit_edits takes them"""
    lg = np.ascontiguousarray(logits, dtype=np.float32).reshape(len(per_row), -1)
    rows, keep = _edit_rows(per_row)
    out = np.zeros((lg.shape[0], k), dtype=TD_DTYPE)
    _check(lib().blk_test_logit_edits(device, _p(lg), lg.shape[0], lg.shape[1], C.cast(rows, C.c_void_p), k, _p(out)))
    return out


test_rmsnorm.__test__ = test_qkv_post.__test__ = test_prefill_attn.__test__ = False      # (not pytest tests)
test_logit_edits.__test__ = False
test_decode_attn.__test__ = test_decode_attn_batch.__test__ = False


def decode_batch(ws: "Ctx", ctxs: Sequence["Ctx"], tokens: Sequence[int], k: int = 40) -> np.ndarray:
    """one forward pass for len(ctxs) sequences, one new token each (blk_decode_batch); returns [n][k] top-k lists"""
    n = len(ctxs)
    arr = (_vp * n)(*[c.h for c in ctxs])
    t = np.ascontiguousarray(tokens, dtype=np.int32)
    out = np.zeros((n, k), dtype=TD_DTYPE)
    _check(lib().blk_decode_batch(ws.h, arr, _p(t), n, k, _p(out)))
    return out


def decode_batch_edited(ws: "Ctx", ctxs: Sequence["Ctx"], tokens: Sequence[int], per_row, k: int = 64):
    """blk_decode_batch_edited: (raw [n][k], edited [n][k]); per_row[i] = (edits, repeat, freq, present)"""
    n = len(ctxs)
    arr = (_vp * n)(*[c.h for c in ctxs])
    t = np.ascontiguousarray(tokens, dtype=np.int32)
    rows, keep = _edit_rows(per_row)
    raw = np.zeros((n, k), dtype=TD_DTYPE); ed = np.zeros((n, k), dtype=TD_DTYPE)
    _check(lib().blk_decode_batch_edited(ws.h, arr, _p(t), n, k, C.cast(rows, C.c_void_p), _p(raw), _p(ed)))
    return raw, ed


def device_count() -> int:
    return int(lib().blk_device_count())


class Model:
    """blk_model handle (reference: bl::llama::Model, Model.hpp:26-58)."""

    def __init__(self, path: str, device: int = 0, progress=None):
        init()
        cb = PROGRESS_CB(lambda p, u: 1 if progress is None else int(bool(progress(p) is not False)))
        self._cb = cb
        self.h = lib().blk_model_load(path.encode(), device, cb, None)
        if not self.h:
            raise BlkError(-1, (lib().blk_last_error() or b"").decode(errors="replace"))
        L = lib()
        self.n_vocab = L.blk_model_n_vocab(self.h)
        self.n_ctx_train = L.blk_model_n_ctx_train(self.h)
        self.n_embd = L.blk_model_n_embd(self.h)
        self.n_layer = L.blk_model_n_layer(self.h)
        self.bos = L.blk_model_token_bos(self.h)
        self.eos = L.blk_model_token_eos(self.h)
        self.weight_bytes_per_token = int(L.blk_model_weight_bytes_per_token(self.h))
        self.kv_bytes_per_token = int(L.blk_model_kv_bytes_per_token(self.h))

    def is_eog(self, tok: int) -> bool:
        return bool(lib().blk_model_is_eog(self.h, int(tok)))

    def panel_cache(self):
        """(bytes, resident matrices, matrices) of the resident bf16 panels (0 before the first multi-token pass)"""
        nr, nm = C.c_int32(0), C.c_int32(0)
        b = lib().blk_model_panel_bytes(self.h, C.byref(nr), C.byref(nm))
        return int(b), int(nr.value), int(nm.value)

    def token_text(self, tok: int) -> str:
        buf = C.create_string_buffer(256)
        n = lib().blk_model_token_text(self.h, int(tok), buf, 256)
        return buf.raw[: min(n, 256)].decode(errors="replace")

    def close(self):
        if self.h:
            lib().blk_model_free(self.h)
            self.h = None


class Ctx:
    """blk_ctx handle (reference: bl::llama::Instance + llama_context, Instance.hpp:21-50)."""

    def __init__(self, model: Model, n_ctx: int = 4096, n_batch: int = 2048):
        self.m = model
        self.h = lib().blk_ctx_create(model.h, n_ctx, n_batch)
        if not self.h:
            raise BlkError(-1, (lib().blk_last_error() or b"").decode(errors="replace"))

    @property
    def n_past(self) -> int:
        return int(lib().blk_ctx_n_past(self.h))

    def clear(self):
        _check(lib().blk_kv_clear(self.h))

    def sync(self):
        _check(lib().blk_sync(self.h))

    def kv_shift(self, p0: int, p1: int):
        """drop the cells of positions [p0, p1), move the rest down (K re-rotated): reference Session.cpp:341-342"""
        _check(lib().blk_kv_shift(self.h, p0, p1))

    def kv_seq_add(self, p0: int, p1: int, delta: int):
        _check(lib().blk_kv_seq_add(self.h, p0, p1, delta))

    def kv_seq_div(self, p0: int, p1: int, d: int):
        _check(lib().blk_kv_seq_div(self.h, p0, p1, d))

    @property
    def next_pos(self) -> int:
        return int(lib().blk_ctx_next_pos(self.h))

    def state_get(self) -> np.ndarray:
        n = int(lib().blk_state_size(self.h))
        buf = np.zeros(n, dtype=np.uint8)
        w = _i64(0)
        _check(lib().blk_state_get(self.h, _p(buf), n, C.byref(w)))
        return buf[: w.value]

    def state_set(self, blob: np.ndarray):
        b = np.ascontiguousarray(blob, dtype=np.uint8)
        _check(lib().blk_state_set(self.h, _p(b), len(b)))

    def decode(self, tokens: Sequence[int]):
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        _check(lib().blk_decode(self.h, _p(t), len(t)))

    def topk(self, k: int = 10) -> np.ndarray:
        out = np.zeros(k, dtype=TD_DTYPE)
        _check(lib().blk_topk_last(self.h, k, _p(out)))
        return out

    def decode_topk(self, token: int, k: int = 40) -> np.ndarray:
        out = np.zeros(k, dtype=TD_DTYPE)
        _check(lib().blk_decode_topk(self.h, int(token), k, _p(out)))
        return out

    def decode_topk_edited(self, token: int, edits=None, repeat: float = 1.0, freq: float = 0.0, present: float = 0.0, k: int = 64):
        """blk_decode_topk_edited: (raw top-k, edited top-k)"""
        e, keep = logit_edits(edits, repeat, freq, present)
        raw = np.zeros(k, dtype=TD_DTYPE); ed = np.zeros(k, dtype=TD_DTYPE)
        _check(lib().blk_decode_topk_edited(self.h, int(token), k, C.byref(e), _p(raw), _p(ed)))
        return raw, ed

    def topk_edited(self, edits=None, repeat: float = 1.0, freq: float = 0.0, present: float = 0.0, k: int = 64) -> np.ndarray:
        e, keep = logit_edits(edits, repeat, freq, present)
        out = np.zeros(k, dtype=TD_DTYPE)
        _check(lib().blk_topk_last_edited(self.h, k, C.byref(e), _p(out)))
        return out

    def decode_loop(self, first_token: int, n_steps: int, wait: bool = True) -> int:
        last = _i32(-1)
        _check(lib().blk_decode_loop(self.h, int(first_token), n_steps, C.byref(last) if wait else None))
        return int(last.value)

    def gather(self, ids: Sequence[int]) -> np.ndarray:
        i = np.ascontiguousarray(ids, dtype=np.int32)
        out = np.zeros(len(i), dtype=np.float32)
        _check(lib().blk_gather_last(self.h, _p(i), len(i), _p(out)))
        return out

    def logits(self) -> np.ndarray:
        out = np.zeros(self.m.n_vocab, dtype=np.float32)
        _check(lib().blk_get_logits_last(self.h, _p(out)))
        return out

    def set_verify_mode(self, mode: int):
        _check(lib().blk_ctx_set_verify_mode(self.h, mode))

    def verify_prefill(self, tokens: Sequence[int], claimed: np.ndarray, n_claimed: Optional[np.ndarray] = None, want_top: bool = True):
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        n = len(t)
        cl = np.ascontiguousarray(claimed, dtype=np.int32).reshape(n, 10)
        nc = np.full(n, 10, dtype=np.int32) if n_claimed is None else np.ascontiguousarray(n_claimed, dtype=np.int32)
        g = np.zeros((n, 10), dtype=np.float32)
        top = np.zeros((n, 10), dtype=TD_DTYPE) if want_top else None
        _check(lib().blk_verify_prefill(self.h, _p(t), n, _p(cl), _p(nc), _p(g), _p(top) if want_top else None))
        return g, top

    def timer_start(self):
        _check(lib().blk_timer_start(self.h))

    def timer_stop(self) -> float:
        ms = C.c_float(0)
        _check(lib().blk_timer_stop(self.h, C.byref(ms)))
        return float(ms.value)

    def bench_kernel(self, which: int, iters: int = 64) -> Tuple[float, int]:
        """(average ms per launch, algorithmic bytes per launch) of one decode kernel timed alone"""
        ms = C.c_float(0)
        b = C.c_int64(0)
        _check(lib().blk_bench_kernel(self.h, which, iters, C.byref(ms), C.byref(b)))
        return float(ms.value), int(b.value)

    def profile_step(self, token: int) -> str:
        buf = C.create_string_buffer(8192)
        _check(lib().blk_profile_step(self.h, int(token), buf, 8192))
        return buf.value.decode()

    def profile_verify(self, tokens: Sequence[int]) -> str:
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        buf = C.create_string_buffer(8192)
        _check(lib().blk_profile_verify(self.h, _p(t), len(t), buf, 8192))
        return buf.value.decode()

    def flush_l2(self):
        _check(lib().blk_flush_l2(self.h))

    @property
    def persistent_decode(self) -> bool:
        return bool(lib().blk_ctx_persistent_decode(self.h))

    def debug_trace(self) -> np.ndarray:
        buf = np.zeros(512 * 1024, dtype=np.int64)
        n_cta, per = C.c_int32(0), C.c_int32(0)
        _check(lib().blk_debug_trace(self.h, buf.ctypes.data_as(C.c_void_p), buf.size, C.byref(n_cta), C.byref(per)))
        return buf[: n_cta.value * per.value].reshape(n_cta.value, per.value)

    @property
    def kernel_launches(self) -> int:
        return int(lib().blk_ctx_kernel_launches(self.h))

    def close(self):
        if self.h:
            lib().blk_ctx_free(self.h)
            self.h = None


def test_gemv(gtype: int, blocks: np.ndarray, rows: int, k: int, x: np.ndarray, device: int = 0) -> np.ndarray:
    b = np.ascontiguousarray(blocks, dtype=np.uint8)
    xx = np.ascontiguousarray(x, dtype=np.float32)
    y = np.zeros(rows, dtype=np.float32)
    _check(lib().blk_test_gemv(device, gtype, _p(b), rows, k, _p(xx), _p(y)))
    return y


class TestMatrix(C.Structure):
    """blk_test_matrix: one weight matrix of blk_test_gemm"""
    _fields_ = [("type", C.c_int32), ("blocks", C.c_void_p), ("rows", C.c_int64), ("bias", C.c_void_p)]
    __test__ = False


class GemmPlan(C.Structure):
    """blk_test_gemm_plan: what a blk_test_gemm call ran"""
    _fields_ = [("n_sm", C.c_int32), ("launches", C.c_int32), ("k_splits", C.c_int32), ("n_whole", C.c_int32), ("deferred", C.c_int32),
                ("panel", C.c_int32)]

    def as_dict(self) -> dict:
        return {f: int(getattr(self, f)) for f, _ in self._fields_}


GEMM_STORE, GEMM_ACCUM, GEMM_SWIGLU = 0, 1, 2


def test_gemm_layer(op: int, mats, k: int, x: np.ndarray, form: int = 0, split: int = 0, c: Optional[np.ndarray] = None,
                    norm_w: Optional[np.ndarray] = None, eps: float = 1e-5, device: int = 0):
    """The prefill GEMM as a multi-token pass calls it (blk_test_gemm).  mats: [(ggml type, blocks, rows, bias or None), ...].
    op GEMM_STORE: C = X W_i^T (+bias_i) side by side; GEMM_ACCUM: C += X W^T (c = the residual) then, with norm_w, the RMSNorm;
    GEMM_SWIGLU: H = silu(X Wg^T) * (X Wu^T).  form 0 fused / 1 panel; split 0 none / 1 workspace / 2 workspace + deferred reduce.
    Returns (C or None, H / xn or None, plan dict).  c: the initial C (op GEMM_STORE: NaN when omitted, so a column left unwritten shows)."""
    xx = np.ascontiguousarray(x, dtype=np.float32)
    T = xx.shape[0]
    keep = []
    arr = (TestMatrix * len(mats))()
    for i, (gtype, blocks, rows, bias) in enumerate(mats):
        b = np.ascontiguousarray(blocks, dtype=np.uint8)
        bb = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32)
        keep += [b, bb]
        arr[i] = TestMatrix(gtype, b.ctypes.data, rows, bb.ctypes.data if bb is not None else None)
    n_out = mats[0][2] if op == GEMM_SWIGLU else sum(m[2] for m in mats)
    cc = None
    if op != GEMM_SWIGLU:
        cc = np.full((T, n_out), np.nan, dtype=np.float32) if c is None else np.array(c, dtype=np.float32, order="C", copy=True)
        assert cc.shape == (T, n_out)
    w = None if norm_w is None else np.ascontiguousarray(norm_w, dtype=np.float32)
    h = np.zeros((T, n_out), dtype=np.float32) if (op == GEMM_SWIGLU or w is not None) else None
    plan = GemmPlan()
    _check(lib().blk_test_gemm(device, op, C.cast(arr, C.c_void_p), len(mats), k, _p(xx), T, form, split, _p(w) if w is not None else None, eps,
                               _p(cc) if cc is not None else None, _p(h) if h is not None else None, C.byref(plan)))
    return cc, h, plan.as_dict()


def test_gemm(gtype: int, blocks: np.ndarray, rows: int, k: int, x: np.ndarray, device: int = 0, form: int = 0, split: int = 0) -> np.ndarray:
    """Y[t][r] = W[r,:] . X[t,:] through the prefill GEMM: one matrix, store (test_gemm_layer with GEMM_STORE); returns Y [n_tok][rows]"""
    y, _, _ = test_gemm_layer(GEMM_STORE, [(gtype, blocks, rows, None)], k, x, form=form, split=split, device=device)
    return y


def test_row_topk(logits: np.ndarray, claimed: np.ndarray, n_claimed: np.ndarray, rows_per_launch: int = 256, top: bool = True, device: int = 0):
    """row_topk_gather_kernel (blk_test_row_topk): (gathered [n][10], top ids [n][10], top logits [n][10]) (the last two None without top)"""
    lg = np.ascontiguousarray(logits, dtype=np.float32)
    n, V = lg.shape
    cl = np.ascontiguousarray(claimed, dtype=np.int32).reshape(n, 10)
    nc = np.ascontiguousarray(n_claimed, dtype=np.int32).reshape(n)
    g = np.zeros((n, 10), dtype=np.float32)
    ti = np.zeros((n, 10), dtype=np.int32) if top else None
    tl = np.zeros((n, 10), dtype=np.float32) if top else None
    _check(lib().blk_test_row_topk(device, _p(lg), n, V, rows_per_launch, _p(cl), _p(nc), _p(g), _p(ti) if top else None, _p(tl) if top else None))
    return g, ti, tl


def test_claimed_logits(gtype: int, blocks: np.ndarray, rows: int, k: int, xn: np.ndarray, claimed: np.ndarray, n_claimed: np.ndarray,
                        device: int = 0) -> np.ndarray:
    """claimed_logits_kernel (blk_test_claimed_logits): gathered [n][10]"""
    b = np.ascontiguousarray(blocks, dtype=np.uint8)
    xx = np.ascontiguousarray(xn, dtype=np.float32)
    n = xx.shape[0]
    cl = np.ascontiguousarray(claimed, dtype=np.int32).reshape(n, 10)
    nc = np.ascontiguousarray(n_claimed, dtype=np.int32).reshape(n)
    g = np.zeros((n, 10), dtype=np.float32)
    _check(lib().blk_test_claimed_logits(device, gtype, _p(b), rows, k, _p(xx), n, _p(cl), _p(nc), _p(g)))
    return g


def test_dequant(gtype: int, blocks: np.ndarray, rows: int, k: int, device: int = 0) -> np.ndarray:
    b = np.ascontiguousarray(blocks, dtype=np.uint8)
    out = np.zeros((rows, k), dtype=np.float32)
    _check(lib().blk_test_dequant(device, gtype, _p(b), rows, k, _p(out)))
    return out


def bench_gemm(gtype: int, blocks: np.ndarray, rows: int, k: int, n_tok: int, iters: int = 10, device: int = 0) -> float:
    """average ms of one prefill GEMM [n_tok x k] . [rows x k]^T"""
    b = np.ascontiguousarray(blocks, dtype=np.uint8)
    ms = C.c_float(0)
    _check(lib().blk_bench_gemm(device, gtype, _p(b), rows, k, n_tok, iters, C.byref(ms)))
    return float(ms.value)


test_gemm.__test__ = test_gemm_layer.__test__ = test_row_topk.__test__ = test_claimed_logits.__test__ = False      # (not pytest tests)
