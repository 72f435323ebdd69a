"""ctypes view of the reference-shaped host API (blama_b200/host/host_capi.cpp): bl::llama::Model / Instance / Session /
LogitComparer / MetricsAggregator / Sampler.  Errors surface as HostError carrying the C++ exception text, which are the
strings the reference's own tests pin (inference/test/t-integration.cpp:137-217)."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import capi

TD_DTYPE = capi.TD_DTYPE
_vp, _i32, _u32, _f32 = C.c_void_p, C.c_int32, C.c_uint32, C.c_float

HOST_SYMBOLS = {
    "blh_last_error": (C.c_char_p, []),
    "blh_init": (None, []),
    "blh_model_create": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "blh_model_free": (None, [_vp]),
    "blh_model_train_ctx": (C.c_int, [_vp]),
    "blh_model_create_vocab_only": (C.c_int, [C.c_char_p, C.POINTER(_vp)]),
    "blh_model_tokenize": (C.c_int, [_vp, C.c_char_p, C.c_int, C.c_int, C.c_int, _vp, C.c_int]),
    "blh_model_token_to_string": (C.c_int, [_vp, _i32, C.c_int, C.c_char_p, C.c_int]),
    "blh_model_is_eog": (C.c_int, [_vp, _i32]),
    "blh_instance_create": (C.c_int, [_vp, _u32, _u32, C.POINTER(_vp)]),
    "blh_instance_free": (None, [_vp]),
    "blh_instance_warmup": (C.c_int, [_vp]),
    "blh_instance_ctx": (_vp, [_vp]),
    "blh_session_start": (C.c_int, [_vp, _u32, _f32, _f32, C.c_int]),
    "blh_session_stop": (None, [_vp]),
    "blh_session_set_initial_prompt": (C.c_int, [_vp, _vp, C.c_int]),
    "blh_session_complete": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp, _vp]),
    "blh_session_stream": (C.c_int, [_vp, C.c_int, _vp, _vp]),
    "blh_session_fill_ctx": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    "blh_session_verify": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.POINTER(_f32)]),
    "blh_session_get_state": (C.c_int, [_vp, _vp, C.c_int64, C.POINTER(C.c_int64)]),
    "blh_session_set_state": (C.c_int, [_vp, _vp, C.c_int64]),
    "blh_session_start_ex": (C.c_int, [_vp, _u32, _f32, _f32, C.c_int, C.c_int]),
    "blh_session_start_ga": (C.c_int, [_vp, _u32, _f32, _f32, _u32, _u32]),
    "blh_lc_compare": (None, [_vp, _i32, _vp, _i32, _vp]),
    "blh_lc_similarity": (_f32, [_vp, _i32, _vp, _i32]),
    "blh_lc_score": (_f32, [_vp, _i32]),
    "blh_sampler_draw": (C.c_int, [_u32, _f32, _f32, _i32, _f32, _i32, _vp, _i32, _i32, _i32, _vp]),
    "blh_sampler_draw_penalized": (C.c_int, [_u32, _f32, _f32, _i32, _f32, _i32, _i32, _f32, _f32, _f32, _vp, _vp, C.c_int,
                                             _vp, _i32, _vp, _i32, _i32, _vp]),
    "blh_sampler_logit_edits": (C.c_int, [_i32, _f32, _f32, _f32, _vp, _vp, C.c_int, _vp, _i32, _i32, _i32, _vp, C.c_int, _vp, _vp]),
    "blh_sampler_check": (C.c_int, [_i32, C.c_char_p]),
    "blh_session_reset_sampler": (C.c_int, [_vp, _u32, _f32, _f32, _i32, _f32, _f32, _f32, _vp, _vp, C.c_int]),
    "blh_session_logit_edits": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp]),
    "blh_session_candidates": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "blh_server_submit_complete_ex": (C.c_int, [_vp, _vp, C.c_int, _u32, _u32, _f32, _f32, _i32, _f32, _f32, _f32, _vp, _vp, C.c_int,
                                                C.POINTER(C.c_int64)]),
    "blh_server_create": (C.c_int, [_vp, C.c_int, _u32, _u32, C.POINTER(_vp)]),
    "blh_server_create_ex": (C.c_int, [_vp, C.c_int, _u32, _u32, _u32, C.POINTER(_vp)]),
    "blh_server_free": (None, [_vp]),
    "blh_server_workers": (C.c_int, [_vp]),
    "blh_server_drain": (None, [_vp]),
    "blh_server_last_worker_error": (C.c_int, [_vp, C.c_char_p, C.c_int]),
    "blh_server_submit_complete": (C.c_int, [_vp, _vp, C.c_int, _u32, _u32, _f32, _f32, C.POINTER(C.c_int64)]),
    "blh_server_submit_verify": (C.c_int, [_vp, _vp, C.c_int, _u32, _f32, _f32, _vp, C.c_int, _vp, _vp, C.POINTER(C.c_int64)]),
    "blh_server_submit_complete_json": (C.c_int, [_vp, C.c_char_p, C.POINTER(C.c_int64)]),
    "blh_server_submit_verify_json": (C.c_int, [_vp, C.c_char_p, C.POINTER(C.c_int64)]),
    "blh_server_wait_complete": (C.c_int, [_vp, C.c_int64, C.c_int, _vp, _vp, _vp, _vp]),
    "blh_server_wait_verify": (C.c_int, [_vp, C.c_int64, C.POINTER(_f32)]),
    "blh_server_wait_complete_json": (C.c_int, [_vp, C.c_int64, C.c_char_p, C.c_int, C.POINTER(C.c_int)]),
    "blh_server_wait_verify_json": (C.c_int, [_vp, C.c_int64, C.c_char_p, C.c_int, C.POINTER(C.c_int)]),
    "blh_server_stats": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int]),
    "blh_server_http_start": (C.c_int, [_vp, C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "blh_server_http_stop": (None, [_vp]),
    "blh_wire_verify_json": (C.c_int, [_f32, C.c_char_p, C.c_int]),
    "blh_wire_json_roundtrip": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(C.c_int)]),
    "blh_wire_parse_request": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(_u32), C.POINTER(_u32), C.POINTER(_f32), C.POINTER(_f32)]),
    "blh_wire_parse_verify": (C.c_int, [C.c_char_p, C.c_int, _vp, _vp, _vp, _vp]),
    "blh_wire_complete_json": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_char_p, C.c_int, C.POINTER(C.c_int)]),
}

_bound = False


def lib() -> C.CDLL:
    global _bound
    l = capi.lib()
    if not _bound:
        for name, (res, args) in HOST_SYMBOLS.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        l.blh_init()
        _bound = True
    return l


def lib_nodevice() -> C.CDLL:
    """the host-only entry points (verdict, sampler, wire format, tokenizer) need no CUDA device: same library, same binding"""
    return lib()


class HostError(RuntimeError):
    pass


def _check(rc: int):
    if rc:
        raise HostError((lib().blh_last_error() or b"").decode(errors="replace"))


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def as_td(pairs) -> np.ndarray:
    if isinstance(pairs, np.ndarray) and pairs.dtype == TD_DTYPE:
        return np.ascontiguousarray(pairs)
    out = np.zeros(len(pairs), dtype=TD_DTYPE)
    for i, (t, l) in enumerate(pairs):
        out[i] = (t, l)
    return out


EDIT_DTYPE = capi.EDIT_DTYPE


def _bias_arrays(logit_bias):
    """{token: bias} -> (ids int32, values float32)"""
    items = sorted((logit_bias or {}).items())
    return np.array([k for k, _ in items], dtype=np.int32), np.array([v for _, v in items], dtype=np.float32)


def _stages_active(penalty_last_n, repeat_penalty, freq_penalty, present_penalty, logit_bias) -> bool:
    return bool(logit_bias) or (repeat_penalty, freq_penalty, present_penalty) != (1.0, 0.0, 0.0)


def _edits_out(call, cap: int = 1 << 16):
    """call(out, cap, byref(n), out3) -> rc: (EDIT_DTYPE array, (repeat, freq, present))"""
    out = np.zeros(cap, dtype=EDIT_DTYPE); n = _i32(0); p3 = np.zeros(3, dtype=np.float32)
    _check(call(_p(out), cap, C.byref(n), _p(p3)))
    assert n.value <= cap
    return out[: n.value].copy(), tuple(float(x) for x in p3)


class Model:
    def __init__(self, path: str, device: int = 0, gpu: bool = True, prefix_bos: bool = False, vocab_only: bool = False):
        h = _vp()
        if vocab_only:
            _check(lib().blh_model_create_vocab_only(path.encode(), C.byref(h)))
        else:
            _check(lib().blh_model_create(path.encode(), device, int(gpu), int(prefix_bos), C.byref(h)))
        self.h = h
        self.path = path

    def train_ctx(self) -> int:
        return lib().blh_model_train_ctx(self.h)

    def tokenize(self, text, add_special: bool = True, parse_special: bool = True) -> np.ndarray:
        raw = text if isinstance(text, (bytes, bytearray)) else text.encode("utf-8")
        out = np.zeros(len(raw) + 4, dtype=np.int32)
        n = lib().blh_model_tokenize(self.h, bytes(raw), len(raw), int(add_special), int(parse_special), _p(out), len(out))
        if n < 0:
            raise HostError((lib().blh_last_error() or b"").decode(errors="replace"))
        return out[:n].copy()

    def token_to_bytes(self, tok: int, special: bool = True) -> bytes:
        buf = C.create_string_buffer(512)
        n = lib().blh_model_token_to_string(self.h, int(tok), int(special), buf, 512)
        if n < 0:
            raise HostError((lib().blh_last_error() or b"").decode(errors="replace"))
        return buf.raw[:min(n, 512)]

    def token_to_string(self, tok: int, special: bool = True) -> str:
        return self.token_to_bytes(tok, special).decode(errors="replace")

    def is_eog(self, tok: int) -> bool:
        return bool(lib().blh_model_is_eog(self.h, int(tok)))

    def close(self):
        if self.h:
            lib().blh_model_free(self.h)
            self.h = None


class Instance:
    """Instance + its (single) Session, addressed together like the reference's Instance::startSession."""

    def __init__(self, model: Model, ctx_size: int = 0, batch_size: int = 0):
        h = _vp()
        _check(lib().blh_instance_create(model.h, ctx_size, batch_size, C.byref(h)))
        self.h = h
        self.model = model

    def warmup(self):
        _check(lib().blh_instance_warmup(self.h))

    def raw_ctx(self) -> "capi.Ctx":
        """non-owning capi.Ctx view of this instance's C-ABI context (timers, launch counters)"""
        import types

        c = capi.Ctx.__new__(capi.Ctx)
        c.h = lib().blh_instance_ctx(self.h)
        c.m = types.SimpleNamespace(n_vocab=int(capi.lib().blk_model_n_vocab(capi.lib().blk_ctx_model(c.h))))
        c.close = lambda: None
        return c

    def start_session(self, seed: int = 0, temperature: float = 0.8, top_p: float = 0.95, sequential_verify: bool = False,
                      infinite_context: bool = True, penalty_last_n: int = 64, repeat_penalty: float = 1.0, freq_penalty: float = 0.0,
                      present_penalty: float = 0.0, logit_bias: Optional[dict] = None):
        """logit_bias {token: bias} and the repetition penalties are the first two stages of the reference's sampler chain (off by
        default); when given, the session's sampler is replaced by one that has them (Session::resetSampler) before any decode"""
        _check(lib().blh_session_start_ex(self.h, seed, temperature, top_p, int(sequential_verify), int(infinite_context)))
        if _stages_active(penalty_last_n, repeat_penalty, freq_penalty, present_penalty, logit_bias):
            self.reset_sampler(seed, temperature, top_p, penalty_last_n, repeat_penalty, freq_penalty, present_penalty, logit_bias)
        return self

    def reset_sampler(self, seed: int = 0, temperature: float = 0.8, top_p: float = 0.95, penalty_last_n: int = 64, repeat_penalty: float = 1.0,
                      freq_penalty: float = 0.0, present_penalty: float = 0.0, logit_bias: Optional[dict] = None):
        """Session::resetSampler: a new sampler chain (empty penalty window) for the rest of the session"""
        ids, vals = _bias_arrays(logit_bias)
        _check(lib().blh_session_reset_sampler(self.h, seed, temperature, top_p, penalty_last_n, repeat_penalty, freq_penalty, present_penalty,
                                               _p(ids), _p(vals), len(ids)))

    def sampling_candidates(self) -> np.ndarray:
        """the list the next draw samples from (the edited top-64 with logit bias / penalties active, else the raw top-64)"""
        out = np.zeros(64, dtype=TD_DTYPE); n = _i32(0)
        _check(lib().blh_session_candidates(self.h, _p(out), 64, C.byref(n)))
        return out[: min(n.value, 64)].copy()

    def logit_edits(self):
        """the session sampler's edit list now: (EDIT_DTYPE array, (repeat, freq, present))"""
        return _edits_out(lambda out, cap, n, p3: lib().blh_session_logit_edits(self.h, out, cap, n, p3))

    def start_session_self_extend(self, ga_factor: int, ga_width: int, seed: int = 0, temperature: float = 0.8, top_p: float = 0.95):
        """Session with group attention (Self-Extend, reference Session.cpp:348-368)"""
        _check(lib().blh_session_start_ga(self.h, seed, temperature, top_p, ga_factor, ga_width))
        return self

    def stop_session(self):
        lib().blh_session_stop(self.h)

    def set_initial_prompt(self, tokens: Sequence[int]):
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        _check(lib().blh_session_set_initial_prompt(self.h, _p(t), len(t)))

    def complete(self, max_tokens: int, prompt: Sequence[int] = ()):
        p = np.ascontiguousarray(prompt, dtype=np.int32)
        toks = np.zeros(max(1, max_tokens), dtype=np.int32)
        top = np.zeros((max(1, max_tokens), 10), dtype=TD_DTYPE)
        nl = np.zeros(max(1, max_tokens), dtype=np.int32)
        n = _i32(0)
        _check(lib().blh_session_complete(self.h, _p(p), len(p), max_tokens, _p(toks), _p(top), _p(nl), C.byref(n)))
        return toks[: n.value].copy(), top[: n.value].copy()

    def stream(self, max_tokens: int) -> np.ndarray:
        toks = np.zeros(max(1, max_tokens), dtype=np.int32)
        n = _i32(0)
        _check(lib().blh_session_stream(self.h, max_tokens, _p(toks), C.byref(n)))
        return toks[: n.value].copy()

    def fill_ctx(self, tokens: Sequence[int], claimed: np.ndarray, n_claimed: Optional[np.ndarray] = None):
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        n = len(t)
        cl = np.ascontiguousarray(claimed).reshape(n, 10)
        assert cl.dtype == TD_DTYPE
        nc = np.full(n, 10, dtype=np.int32) if n_claimed is None else np.ascontiguousarray(n_claimed, dtype=np.int32)
        out = np.zeros((n, 10), dtype=TD_DTYPE)
        out_n = np.zeros(n, dtype=np.int32)
        _check(lib().blh_session_fill_ctx(self.h, _p(t), n, _p(cl), _p(nc), _p(out), _p(out_n)))
        return out, out_n

    def verify(self, tokens: Sequence[int], claimed: np.ndarray, n_claimed: Optional[np.ndarray] = None) -> float:
        """fillCtx + LogitComparer + MetricsAggregator in C++ (what Server::verify runs); returns the score"""
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        n = len(t)
        cl = np.ascontiguousarray(claimed).reshape(n, 10)
        assert cl.dtype == TD_DTYPE
        nc = np.full(n, 10, dtype=np.int32) if n_claimed is None else np.ascontiguousarray(n_claimed, dtype=np.int32)
        score = _f32(0)
        _check(lib().blh_session_verify(self.h, _p(t), n, _p(cl), _p(nc), C.byref(score)))
        return float(score.value)

    def get_state(self) -> np.ndarray:
        cap = int(capi.lib().blk_state_size(lib().blh_instance_ctx(self.h))) + (1 << 16)
        buf = np.zeros(cap, dtype=np.uint8)
        n = C.c_int64(0)
        _check(lib().blh_session_get_state(self.h, _p(buf), cap, C.byref(n)))
        return buf[: n.value].copy()

    def set_state(self, blob=None):
        b = np.zeros(0, dtype=np.uint8) if blob is None else np.ascontiguousarray(blob, dtype=np.uint8)
        _check(lib().blh_session_set_state(self.h, _p(b) if len(b) else None, len(b)))

    def close(self):
        if self.h:
            lib().blh_instance_free(self.h)
            self.h = None


def lc_compare(a, b) -> Tuple[float, float, float]:
    a, b = as_td(a), as_td(b)
    out = np.zeros(3, dtype=np.float32)
    lib().blh_lc_compare(_p(a), len(a), _p(b), len(b), _p(out))
    return (float(out[0]), float(out[1]), float(out[2]))


def lc_similarity(a, b) -> float:
    a, b = as_td(a), as_td(b)
    return float(lib().blh_lc_similarity(_p(a), len(a), _p(b), len(b)))


def lc_score(metrics) -> float:
    m = np.ascontiguousarray(np.asarray(metrics, dtype=np.float32).reshape(-1, 3))
    return float(lib().blh_lc_score(_p(m), len(m)))


def sampler_draw(cand, n_draws: int, seed: int = 0, temp: float = 0.8, top_p: float = 0.95, top_k: int = 40, min_p: float = 0.05,
                 min_keep: int = 0, is_sorted: bool = True) -> np.ndarray:
    c = as_td(cand)
    out = np.zeros(n_draws, dtype=np.int32)
    _check(lib().blh_sampler_draw(seed, temp, top_p, top_k, min_p, min_keep, _p(c), len(c), int(is_sorted), n_draws, _p(out)))
    return out


def sampler_draw_penalized(logits: np.ndarray, n_draws: int, history: Sequence[int] = (), seed: int = 0, temp: float = 0.8, top_p: float = 0.95,
                           top_k: int = 40, min_p: float = 0.05, min_keep: int = 0, penalty_last_n: int = 64, repeat_penalty: float = 1.0,
                           freq_penalty: float = 0.0, present_penalty: float = 0.0, logit_bias: Optional[dict] = None) -> np.ndarray:
    """the host Sampler's full-row path: accept `history`, then per draw edit a copy of `logits` with bias + penalties, draw, accept"""
    lg = np.ascontiguousarray(logits, dtype=np.float32)
    h = np.ascontiguousarray(history, dtype=np.int32)
    ids, vals = _bias_arrays(logit_bias)
    out = np.zeros(max(1, n_draws), dtype=np.int32)
    _check(lib().blh_sampler_draw_penalized(seed, temp, top_p, top_k, min_p, min_keep, penalty_last_n, repeat_penalty, freq_penalty, present_penalty,
                                            _p(ids), _p(vals), len(ids), _p(h), len(h), _p(lg), len(lg), n_draws, _p(out)))
    return out[:n_draws]


def sampler_check(mirostat: int = 0, grammar: str = ""):
    """raises HostError when the Sampler refuses these parameters"""
    _check(lib().blh_sampler_check(mirostat, grammar.encode()))


def sampler_logit_edits(n_vocab: int, history: Sequence[int] = (), penalty_last_n: int = 64, repeat_penalty: float = 1.0, freq_penalty: float = 0.0,
                        present_penalty: float = 0.0, logit_bias: Optional[dict] = None, reset_after: bool = False):
    """Sampler::logitEdits after accepting `history` (then reset() when reset_after): (EDIT_DTYPE array, (repeat, freq, present))"""
    h = np.ascontiguousarray(history, dtype=np.int32)
    ids, vals = _bias_arrays(logit_bias)
    return _edits_out(lambda out, cap, n, p3: lib().blh_sampler_logit_edits(penalty_last_n, repeat_penalty, freq_penalty, present_penalty, _p(ids),
                                                                            _p(vals), len(ids), _p(h), len(h), int(reset_after), n_vocab, out, cap, n, p3))


# ---- wire format (host only) ----------------------------------------------------------------------------------------------
def _text_out(call, cap: int = 1 << 16) -> str:
    """call(buf, cap, byref(len)) -> rc; grows the buffer once when the text is longer than cap"""
    for _ in range(2):
        buf = C.create_string_buffer(cap)
        n = C.c_int(0)
        rc = call(buf, cap, C.byref(n))
        if rc:
            raise HostError((lib_nodevice().blh_last_error() or b"").decode(errors="replace"))
        if n.value <= cap:
            return buf.raw[: n.value].decode("utf-8")
        cap = n.value + 16
    raise HostError("text did not fit")


def wire_verify_json(score: float) -> str:
    buf = C.create_string_buffer(256)
    n = lib_nodevice().blh_wire_verify_json(score, buf, 256)
    return buf.raw[:n].decode()


def wire_json_roundtrip(text: str) -> str:
    b = text.encode("utf-8")
    return _text_out(lambda buf, cap, n: lib_nodevice().blh_wire_json_roundtrip(b, buf, cap, n), max(1 << 12, 2 * len(b)))


def wire_parse_request(body: str):
    pb = C.create_string_buffer(1 << 16)
    mt, seed, temp, top_p = _u32(0), _u32(0), _f32(0), _f32(0)
    rc = lib_nodevice().blh_wire_parse_request(body.encode(), pb, len(pb), C.byref(mt), C.byref(seed), C.byref(temp), C.byref(top_p))
    if rc:
        raise HostError((lib_nodevice().blh_last_error() or b"").decode(errors="replace"))
    return {"prompt": pb.value.decode(), "max_tokens": mt.value, "seed": seed.value, "temp": temp.value, "top_p": top_p.value}


def wire_parse_verify(body: str, cap: int = 4096):
    toks = np.zeros(cap, dtype=np.int32); cl = np.zeros((cap, 10), dtype=TD_DTYPE); nc = np.zeros(cap, dtype=np.int32); n = _i32(0)
    rc = lib_nodevice().blh_wire_parse_verify(body.encode(), cap, _p(toks), _p(cl), _p(nc), C.byref(n))
    if rc:
        raise HostError((lib_nodevice().blh_last_error() or b"").decode(errors="replace"))
    return toks[: n.value].copy(), cl[: n.value].copy(), nc[: n.value].copy()


def wire_complete_json(tokens, top10: np.ndarray, n_logits=None, model: Optional[Model] = None) -> str:
    t = np.ascontiguousarray(tokens, dtype=np.int32)
    n = len(t)
    cl = np.ascontiguousarray(top10).reshape(n, 10)
    nl = np.full(n, 10, dtype=np.int32) if n_logits is None else np.ascontiguousarray(n_logits, dtype=np.int32)
    l = lib_nodevice()
    return _text_out(lambda buf, cap, ln: l.blh_wire_complete_json(model.h if model else None, _p(t), n, _p(cl), _p(nl), buf, cap, ln), 1 << 20)


# ---- Server: N replicas behind one request queue (reference server/code/server/Server.hpp) -----------------------------------
class Server:
    def __init__(self, models: Sequence[Model], ctx_size: int = 0, batch_size: int = 0, max_batch: int = 1):
        """max_batch > 1: continuous batching -- up to max_batch /complete requests in flight per replica, one batched step per token"""
        arr = (_vp * len(models))(*[m.h for m in models])
        h = _vp()
        _check(lib().blh_server_create_ex(arr, len(models), ctx_size, batch_size, max_batch, C.byref(h)))
        self.h = h
        self.models = list(models)

    def workers(self) -> int:
        return lib().blh_server_workers(self.h)

    def submit_complete(self, prompt: Sequence[int], max_tokens: int, seed: int = 0, temp: float = 0.8, top_p: float = 0.95,
                        penalty_last_n: int = 64, repeat_penalty: float = 1.0, freq_penalty: float = 0.0, present_penalty: float = 0.0,
                        logit_bias: Optional[dict] = None) -> int:
        p = np.ascontiguousarray(prompt, dtype=np.int32)
        t = C.c_int64(0)
        if not _stages_active(penalty_last_n, repeat_penalty, freq_penalty, present_penalty, logit_bias):
            _check(lib().blh_server_submit_complete(self.h, _p(p), len(p), max_tokens, seed, temp, top_p, C.byref(t)))
        else:
            ids, vals = _bias_arrays(logit_bias)
            _check(lib().blh_server_submit_complete_ex(self.h, _p(p), len(p), max_tokens, seed, temp, top_p, penalty_last_n, repeat_penalty,
                                                       freq_penalty, present_penalty, _p(ids), _p(vals), len(ids), C.byref(t)))
        return t.value

    def submit_verify(self, prompt: Sequence[int], tokens: Sequence[int], claimed: np.ndarray, n_claimed=None, seed: int = 0,
                      temp: float = 0.8, top_p: float = 0.95) -> int:
        p = np.ascontiguousarray(prompt, dtype=np.int32)
        tk = np.ascontiguousarray(tokens, dtype=np.int32)
        n = len(tk)
        cl = np.ascontiguousarray(claimed).reshape(n, 10)
        assert cl.dtype == TD_DTYPE
        nc = np.full(n, 10, dtype=np.int32) if n_claimed is None else np.ascontiguousarray(n_claimed, dtype=np.int32)
        t = C.c_int64(0)
        _check(lib().blh_server_submit_verify(self.h, _p(p), len(p), seed, temp, top_p, _p(tk), n, _p(cl), _p(nc), C.byref(t)))
        return t.value

    def submit_complete_json(self, body: str) -> int:
        t = C.c_int64(0)
        _check(lib().blh_server_submit_complete_json(self.h, body.encode("utf-8"), C.byref(t)))
        return t.value

    def submit_verify_json(self, body: str) -> int:
        t = C.c_int64(0)
        _check(lib().blh_server_submit_verify_json(self.h, body.encode("utf-8"), C.byref(t)))
        return t.value

    def wait_complete(self, ticket: int, cap: int = 4096):
        toks = np.zeros(cap, dtype=np.int32); top = np.zeros((cap, 10), dtype=TD_DTYPE); nl = np.zeros(cap, dtype=np.int32); n = _i32(0)
        _check(lib().blh_server_wait_complete(self.h, ticket, cap, _p(toks), _p(top), _p(nl), C.byref(n)))
        k = min(n.value, cap)
        return toks[:k].copy(), top[:k].copy(), nl[:k].copy()

    def wait_verify(self, ticket: int) -> float:
        s = _f32(0)
        _check(lib().blh_server_wait_verify(self.h, ticket, C.byref(s)))
        return float(s.value)

    def wait_complete_json(self, ticket: int) -> str:
        # a ticket can be waited for once: size the buffer generously (a 2048-token answer is ~1.5 MB)
        cap = 1 << 23
        buf = C.create_string_buffer(cap); n = C.c_int(0)
        _check(lib().blh_server_wait_complete_json(self.h, ticket, buf, cap, C.byref(n)))
        return buf.raw[: min(n.value, cap)].decode("utf-8")

    def wait_verify_json(self, ticket: int) -> str:
        buf = C.create_string_buffer(256); n = C.c_int(0)
        _check(lib().blh_server_wait_verify_json(self.h, ticket, buf, 256, C.byref(n)))
        return buf.raw[: n.value].decode()

    def drain(self):
        lib().blh_server_drain(self.h)

    def last_worker_error(self) -> str:
        buf = C.create_string_buffer(4096)
        n = lib().blh_server_last_worker_error(self.h, buf, 4096)
        return buf.raw[: min(n, 4096)].decode(errors="replace")

    def stats(self):
        k = self.workers()
        dev = np.zeros(k, dtype=np.int32); req = np.zeros(k, dtype=np.uint64); ms = np.zeros(k, dtype=np.float64)
        lib().blh_server_stats(self.h, _p(dev), _p(req), _p(ms), k)
        return [{"device": int(dev[i]), "requests": int(req[i]), "gpu_ms": float(ms[i])} for i in range(k)]

    def http_start(self, host: str = "127.0.0.1", port: int = 0, io_threads: int = 4) -> int:
        out = C.c_int(0)
        _check(lib().blh_server_http_start(self.h, host.encode(), port, io_threads, C.byref(out)))
        return out.value

    def http_stop(self):
        lib().blh_server_http_stop(self.h)

    def close(self):
        if self.h:
            lib().blh_server_free(self.h)
            self.h = None
