"""The non-GEMM kernels of the verify / prefill path one at a time, against float64 numpy on the ROUNDED operands (the GEMV, the
de-quantisation and the GEMM are pinned the same way in test_gpu_kernels.py / test_gpu_prefill_gemm.py):
  rmsnorm_bf16_kernel    bf16(x / sqrt(mean(x^2) + eps) * w)                      within one bf16 rounding of the exact value
  qkv_post_kernel        RoPE (NORM / NEOX, rope_freqs) on q and k -> f16, v -> f16, rows through the page table   within one f16 ulp
  prefill_attn_tc_kernel causal soft-max(q k^T / sqrt(d)) v on f16 operands -> bf16 (tcgen05; the mma.sync kernels for d_head 64)"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BF16_ULP = 2.0 ** -7          # relative spacing of bf16 at the bottom of a binade (8 significand bits): half an ulp = 2^-8 = 3.9e-3
F16_ULP = 2.0 ** -10          # ... of f16 (11 significand bits): half an ulp = 4.9e-4


@pytest.mark.parametrize("T,K", [(5, 256), (64, 2048), (33, 4096), (7, 8192)])
def test_rmsnorm_bf16(T, K):
    from blama_b200 import capi

    capi.init()
    rng = np.random.default_rng(K + T)
    x = (rng.standard_normal((T, K)) * rng.uniform(0.1, 30.0, (T, 1))).astype(np.float32)
    w = (1.0 + 0.1 * rng.standard_normal(K)).astype(np.float32)
    eps = 1e-5
    got = capi.test_rmsnorm(x, w, eps).astype(np.float64)
    x64, w64 = x.astype(np.float64), w.astype(np.float64)
    ref = x64 / np.sqrt((x64 * x64).mean(axis=1, keepdims=True) + eps) * w64
    rel = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-30)
    print(f"\n[rmsnorm {T}x{K}] max rel err {rel.max():.3g} (bf16 half ulp = {BF16_ULP / 2:.3g})")
    assert rel.max() <= BF16_ULP * 0.51 + 1e-6          # the correctly rounded bf16 of the f32 result: within half a bf16 ulp (+ f32 noise)


@pytest.mark.parametrize("n_head,n_head_kv,d_head,neox,pos0,ff", [(4, 2, 128, False, 0, True), (4, 2, 128, True, 57, False), (8, 2, 64, False, 1000, True),
                                                                    (14, 2, 128, True, 130, False)])
def test_qkv_post_rope_and_cache_rows(n_head, n_head_kv, d_head, neox, pos0, ff):
    from blama_b200 import capi

    capi.init()
    rng = np.random.default_rng(n_head * 131 + pos0)
    T, dq, dkv, half = 70, n_head * d_head, n_head_kv * d_head, d_head // 2
    theta = 5e5 if not neox else 1e6
    qkv = (rng.standard_normal((T, dq + 2 * dkv)) * 2.0).astype(np.float32)
    factors = rng.uniform(1.0, 8.0, half).astype(np.float32) if ff else None
    q, k, v = capi.test_qkv_post(qkv, n_head, n_head_kv, d_head, neox, pos0, theta, factors)
    # v: exactly the f16 rounding of the input, at the row the page table names
    assert np.array_equal(v, qkv[:, dq + dkv:].astype(np.float16).astype(np.float32))
    # the angle as the kernel (and ggml) builds it: theta_i = pos * scale^i in f32, iterated, / freq_factor_i
    scale = np.float32(np.float32(theta) ** np.float32(-2.0 / d_head))
    worst = 0.0
    for t in range(T):
        th = np.zeros(half, dtype=np.float32)
        cur = np.float32(pos0 + t)
        for i in range(half):
            th[i] = cur / (factors[i] if ff else np.float32(1.0))
            cur = np.float32(cur * scale)
        c, s = np.cos(th.astype(np.float64)), np.sin(th.astype(np.float64))
        for src, got, heads in ((qkv[t, :dq], q[t], n_head), (qkv[t, dq:dq + dkv], k[t], n_head_kv)):
            x = src.astype(np.float64).reshape(heads, d_head)
            if neox:
                x0, x1 = x[:, :half], x[:, half:]
                ref = np.concatenate([x0 * c - x1 * s, x0 * s + x1 * c], axis=1)
            else:
                x0, x1 = x[:, 0::2], x[:, 1::2]
                ref = np.empty_like(x); ref[:, 0::2] = x0 * c - x1 * s; ref[:, 1::2] = x0 * s + x1 * c
            err = np.abs(got.reshape(heads, d_head) - ref)
            tol = F16_ULP * np.maximum(np.abs(ref), 1e-3) + 2e-6 * max(1, pos0 + t)      # one f16 ulp + the f32 angle error at this position
            assert np.all(err <= tol), (t, float((err / tol).max()))
            worst = max(worst, float((err / np.maximum(np.abs(ref), 1e-3)).max()))
    print(f"\n[qkv_post heads {n_head}/{n_head_kv} d {d_head} neox {neox} pos0 {pos0}] max rel err {worst:.3g} (f16 ulp {F16_ULP:.3g})")


@pytest.mark.parametrize("n_head,n_head_kv,d_head,T,pos0,scores", [
    (4, 1, 128, 200, 0, "random"), (8, 2, 128, 64, 100, "random"), (7, 1, 128, 130, 31, "random"), (8, 1, 128, 96, 64, "random"),
    (1, 1, 128, 40, 5, "random"), (4, 2, 64, 100, 20, "random"),
    # many key tiles (the K ring runs ahead of the V ring, both wrap several times)
    (8, 2, 128, 700, 333, "random"), (2, 1, 128, 1100, 0, "random"),
    # scores that grow by ~13 per 128-key tile: the one-pass kernel raises its reference maximum and rescales O in TMEM at EVERY tile;
    # falling scores: it never does after the first tile and the late probabilities underflow
    (4, 1, 128, 600, 100, "rising"), (8, 1, 128, 300, 77, "rising"), (4, 2, 128, 500, 0, "falling")])
def test_prefill_attention(n_head, n_head_kv, d_head, T, pos0, scores):
    from blama_b200 import capi

    capi.init()
    rng = np.random.default_rng(n_head * 17 + T)
    n_keys, gq = pos0 + T, n_head // n_head_kv
    q = rng.standard_normal((T, n_head * d_head)).astype(np.float32) * 1.5
    k = rng.standard_normal((n_keys, n_head_kv * d_head)).astype(np.float32)
    v = rng.standard_normal((n_keys, n_head_kv * d_head)).astype(np.float32)
    if scores != "random":
        # every query = sqrt(d) e + noise, key j = (+-0.1 j) e + noise: score_j ~ +-0.1 j (+ O(1) noise)
        e = np.zeros(d_head, dtype=np.float32); e[::2] = 1.0; e /= np.linalg.norm(e)
        q = (0.3 * q.reshape(T, n_head, d_head) + np.sqrt(d_head) * e).reshape(T, -1).astype(np.float32)
        ramp = (0.1 if scores == "rising" else -0.1) * np.arange(n_keys, dtype=np.float32)
        k = (k.reshape(n_keys, n_head_kv, d_head) + ramp[:, None, None] * e).reshape(n_keys, -1).astype(np.float32)
    got, used_tc = capi.test_prefill_attn(q, k, v, pos0, n_head, n_head_kv, d_head)
    assert used_tc == (d_head == 128)
    qh = q.astype(np.float16).astype(np.float64).reshape(T, n_head, d_head)
    kh = k.astype(np.float16).astype(np.float64).reshape(n_keys, n_head_kv, d_head)
    vh = v.astype(np.float16).astype(np.float64).reshape(n_keys, n_head_kv, d_head)
    ref = np.zeros((T, n_head, d_head))
    for h in range(n_head):
        s = qh[:, h] @ kh[:, h // gq].T / np.sqrt(d_head)                       # [T][n_keys]
        mask = np.arange(n_keys)[None, :] > (pos0 + np.arange(T))[:, None]
        s[mask] = -np.inf
        p = np.exp(s - s.max(axis=1, keepdims=True))
        ref[:, h] = (p / p.sum(axis=1, keepdims=True)) @ vh[:, h // gq]
    ref = ref.reshape(T, n_head * d_head)
    scale = np.abs(ref).max(axis=1, keepdims=True)
    err = np.abs(got - ref)
    rel = float((err / scale).max())
    print(f"\n[prefill attention heads {n_head}/{n_head_kv} d {d_head} T {T} pos0 {pos0} {scores} tc {used_tc}] max err / row max = {rel:.3g}")
    # bf16 output (half ulp 2^-9 of the value) + f16 probabilities (2^-11 each, averaged over the row): bounded by 1e-3 of the row's
    # largest value beside the output rounding
    assert np.all(err <= BF16_ULP * 0.51 * np.abs(ref) + 1e-3 * scale), rel


def test_prefill_attention_rejects_a_shape_without_a_kernel():
    """d_head 128 runs only on the tcgen05 kernel, which covers GQA ratios up to 8: a ratio of 16 is an argument error, not a launch."""
    from blama_b200 import capi

    capi.init()
    T = 16
    q = np.zeros((T, 16 * 128), dtype=np.float32)
    kv = np.zeros((T, 128), dtype=np.float32)
    with pytest.raises(capi.BlkError) as e:
        capi.test_prefill_attn(q, kv, kv, 0, 16, 1, 128)
    assert e.value.code == 4      # BLK_ERR_ARG
