"""Decode attention kernels against float64 numpy on the operands they see (q, K, V rounded to f16, scale = 1/sqrt(d_head) in f32).

Per-op decode step (attn_cluster_kernel, or attn_scores / attn_pv / attn_combine): ggml's order of operations -- f32 scores, row
maximum, expf, the sum in double, p = e * (1/S) rounded to f16, V.p accumulated in f32.  Batched decode step
(decode_attn_batch_kernel): an f32 flash soft-max over 512-key tiles with p not rounded, bf16 output.

Every case goes through a seeded random page table over a pool larger than the context needs, and every cell a kernel should not
read (unmapped pages, cells past n_kv, the batch's other layer) holds NaN.  The error bounds are elementwise:
  delta_j  relative f32 error of probability j before any rounding: the score's dot product, s_j - M, expf (and the batch kernel's
           running-maximum corrections), plus the normalisation, which inherits the errors of every e_i
  eps      f32 error of the output: (delta * p) . |V| + 8 * 2^-24 * sqrt(n_kv) * (p . |V|) + 1e-7 (the middle term: f32 accumulation)
  A        |o - p.V| <= u16(p) . |V| + eps, u16(p) = max(2^-11 p, 2^-25) is half an f16 ulp including the subnormals below 2^-14
  B        |o - f16(p).V| <= sum_j ulp16(p_j) |v_j| [p_j within delta_j p_j of an f16 rounding midpoint] + eps
B fails a kernel that skips the rounding of p or rounds before normalising; A alone allows both.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U22, U24 = 2.0 ** -22, 2.0 ** -24
BF16_HALF_ULP = 2.0 ** -8         # relative half ulp of bf16 (8 significant bits)
# (n_head, n_head_kv): every GQA ratio from 1 to 8
HEADS = [(2, 2), (4, 2), (6, 2), (4, 1), (5, 1), (12, 2), (14, 2), (8, 1)]
PER_OP_NKV = [1, 2, 7, 64, 65, 129, 1000, 4097]
BATCH_NKV = [1, 2, 511, 512, 513, 1024, 1025, 1536, 3000]
BD_TK = 512                       # decode_attn_batch_kernel's key tile


def _operands(rng, n_q, n_kv, n_head, n_head_kv, d_head, pattern):
    """q [n_q][n_head*dh], k / v [n_kv][n_head_kv*dh] (f32) for one score pattern over the same n_kv keys"""
    gq = n_head // n_head_kv
    q = rng.standard_normal((n_q, n_head, d_head)).astype(np.float32) * 1.5
    k = rng.standard_normal((n_kv, n_head_kv, d_head)).astype(np.float32)
    v = rng.standard_normal((n_kv, n_head_kv, d_head)).astype(np.float32)
    if pattern == "uniform":
        # every score 0, p = 1/n_kv; V's mean of 1 turns the f16 rounding of p into a shift of the whole output
        q[:] = 0.0
        v = (1.0 + 0.1 * v).astype(np.float32)
    elif pattern == "peaked":
        # q = 20 k_j0 (its own j0 per query head): s_j0 ~ 20 scale |k|^2 dominates, every other p underflows in f16
        for r in range(n_q):
            for h in range(n_head):
                q[r, h] = 20.0 * k[rng.integers(n_kv), h // gq]
    elif pattern in ("rising", "falling"):
        # every query = sqrt(d) e + noise, key j = (+-0.1 j) e + noise: score_j ~ +-0.1 j (+ O(1) noise).  Rising raises the batch
        # kernel's running maximum in every tile; falling never does after the first tile.
        e = np.zeros(d_head, dtype=np.float32); e[::2] = 1.0; e /= np.linalg.norm(e)
        q = (0.3 * q + np.sqrt(d_head) * e).astype(np.float32)
        ramp = (0.1 if pattern == "rising" else -0.1) * np.arange(n_kv, dtype=np.float32)
        k = (k + ramp[:, None, None] * e).astype(np.float32)
    else:
        assert pattern == "random"
    return q.reshape(n_q, -1), k.reshape(n_kv, -1), v.reshape(n_kv, -1)


def _reference(q, k, v, n_head, n_head_kv, d_head, n_corr):
    """float64 reference of one query row over all rows of k / v.  n_corr: expf evaluations that multiply into one probability
    beside its own (the batch kernel's per-tile corrections).  Returns per head: p, |V|, V, o_exact, delta, eps (lists)."""
    gq = n_head // n_head_kv
    scale = float(np.float32(1.0) / np.sqrt(np.float32(d_head)))     # the kernels' 1.0f / sqrtf((float)d_head)
    n_kv = k.shape[0]
    qh = q.astype(np.float16).astype(np.float64).reshape(n_head, d_head)
    kh = k.astype(np.float16).astype(np.float64).reshape(n_kv, n_head_kv, d_head)
    vh = v.astype(np.float16).astype(np.float64).reshape(n_kv, n_head_kv, d_head)
    out = []
    for h in range(n_head):
        K, V = kh[:, h // gq], vh[:, h // gq]
        s = scale * (K @ qh[h])
        a = scale * (np.abs(K) @ np.abs(qh[h]))
        M = s.max()
        e = np.exp(s - M)
        p = e / e.sum()
        # the score (dot product a, then s_j - M), expf and the corrections; then the normalisation: S carries every e_i's error
        delta = U22 * (a + np.abs(s) + abs(M) + 1.0 + n_corr)
        delta = delta + p @ delta
        aV = np.abs(V)
        eps = (delta * p) @ aV + 8.0 * U24 * np.sqrt(n_kv) * (p @ aV) + 1e-7
        out.append((p, aV, V, p @ V, delta, eps))
    return out


def _check_per_op(got, ref, d_head, tag):
    """checks A and B of every head; returns the largest error / bound ratio of each"""
    worst_a = worst_b = 0.0
    for h, (p, aV, V, o_exact, delta, eps) in enumerate(ref):
        o = got[h * d_head:(h + 1) * d_head].astype(np.float64)
        assert np.all(np.isfinite(o)), f"{tag} head {h}: non-finite output (a read through the wrong page or past n_kv)"
        bound_a = np.maximum(2.0 ** -11 * p, 2.0 ** -25) @ aV + eps
        err_a = np.abs(o - o_exact)
        # f16 neighbours of every p: the rounding midpoint between them, and the ulp
        r = p.astype(np.float16)
        lo = np.where(r.astype(np.float64) <= p, r, np.nextafter(r, np.float16(-np.inf))).astype(np.float64)
        hi = np.where(r.astype(np.float64) > p, r, np.nextafter(r, np.float16(np.inf))).astype(np.float64)
        near_mid = np.abs(p - 0.5 * (lo + hi)) <= delta * p
        bound_b = ((hi - lo) * near_mid) @ aV + eps
        err_b = np.abs(o - r.astype(np.float64) @ V)
        worst_a = max(worst_a, float((err_a / bound_a).max()))
        worst_b = max(worst_b, float((err_b / bound_b).max()))
        assert np.all(err_a <= bound_a), f"{tag} head {h}: check A, worst err / bound {(err_a / bound_a).max():.3g}"
        assert np.all(err_b <= bound_b), f"{tag} head {h}: check B (p rounded to f16 after normalising), worst err / bound {(err_b / bound_b).max():.3g}"
    return worst_a, worst_b


def _run_per_op(n_head, n_head_kv, d_head, n_kv, pattern, forms, seed, n_ctx=None):
    from blama_b200 import capi

    rng = np.random.default_rng(seed)
    q, k, v = _operands(rng, 1, n_kv, n_head, n_head_kv, d_head, pattern)
    ref = _reference(q[0], k, v, n_head, n_head_kv, d_head, 0)
    for form in forms:
        got, cluster = capi.test_decode_attn(q[0], k, v, n_ctx or n_kv, n_head, n_head_kv, d_head, form=form, seed=seed)
        if form >= 0:
            assert cluster == bool(form)
        tag = f"[decode attn heads {n_head}/{n_head_kv} d {d_head} n_kv {n_kv} {pattern} {'cluster' if cluster else 'split'}]"
        wa, wb = _check_per_op(got, ref, d_head, tag)
        print(f"\n{tag} max err / bound: A {wa:.3g}, B {wb:.3g}")


@pytest.mark.parametrize("d_head", [64, 128])
@pytest.mark.parametrize("n_head,n_head_kv", HEADS)
def test_decode_attn_per_op_shapes(n_head, n_head_kv, d_head):
    """every GQA ratio (both template instances of the cluster kernel), n_kv from fewer keys than CTAs / splits to several pages,
    both forms forced"""
    from blama_b200 import capi

    capi.init()
    for n_kv in PER_OP_NKV:
        _run_per_op(n_head, n_head_kv, d_head, n_kv, "random", (0, 1), seed=n_head * 1000 + d_head + n_kv)


@pytest.mark.parametrize("pattern", ["uniform", "peaked", "rising", "falling"])
@pytest.mark.parametrize("n_head,n_head_kv,d_head", [(8, 1, 128), (6, 2, 64), (2, 2, 128), (5, 1, 64)])
def test_decode_attn_per_op_patterns(n_head, n_head_kv, d_head, pattern):
    from blama_b200 import capi

    capi.init()
    for n_kv in (65, 1000, 4097):
        _run_per_op(n_head, n_head_kv, d_head, n_kv, pattern, (0, 1), seed=7 * n_kv + n_head)


@pytest.mark.parametrize("n_head,n_head_kv,last_cluster,first_split", [
    (8, 1, 24576, 24640),     # GQA 8: one CTA's scores (cap = n_ctx / 8) + 16 warps' partial outputs reach 160 KB
    (4, 1, 65536, 65600),     # GQA 4
    (1, 1, 261632, 261696),   # MHA: shared memory would allow more, but cap > 511 * 64 + 1 would overflow the 512-entry page buffer
])
def test_decode_attn_plan_boundary(n_head, n_head_kv, last_cluster, first_split):
    """the plan picks the cluster form up to last_cluster cells and the split form from first_split on; both compute the same
    attention over a short n_kv, and a forced cluster launch beyond the boundary is an argument error"""
    from blama_b200 import capi

    capi.init()
    d_head, n_kv = 128, 100
    for n_ctx, want in ((last_cluster, True), (first_split, False)):
        rng = np.random.default_rng(n_ctx)
        q, k, v = _operands(rng, 1, n_kv, n_head, n_head_kv, d_head, "random")
        got, cluster = capi.test_decode_attn(q[0], k, v, n_ctx, n_head, n_head_kv, d_head, form=-1, seed=n_ctx)
        assert cluster == want, (n_ctx, cluster)
        tag = f"[decode attn plan heads {n_head}/{n_head_kv} n_ctx {n_ctx} {'cluster' if cluster else 'split'}]"
        wa, wb = _check_per_op(got, _reference(q[0], k, v, n_head, n_head_kv, d_head, 0), d_head, tag)
        print(f"\n{tag} max err / bound: A {wa:.3g}, B {wb:.3g}")
    with pytest.raises(capi.BlkError) as e:
        capi.test_decode_attn(q[0], k, v, first_split, n_head, n_head_kv, d_head, form=1)
    assert e.value.code == 4


def test_decode_attn_mha_long_context_takes_the_split_form():
    """MHA at 300,000 cells: one cluster CTA's slice would span 586 pages, more than its 512-entry page buffer holds.  The plan
    picks the split form, which meets A and B with uniform scores (p = 1/300000 is subnormal in f16), and a forced cluster launch is
    refused before it starts."""
    from blama_b200 import capi

    capi.init()
    n_kv = 300_000
    rng = np.random.default_rng(5)
    q, k, v = _operands(rng, 1, n_kv, 1, 1, 128, "uniform")
    got, cluster = capi.test_decode_attn(q[0], k, v, n_kv, 1, 1, 128, form=-1, seed=3)
    assert not cluster
    tag = f"[decode attn heads 1/1 d 128 n_kv {n_kv} uniform split]"
    wa, wb = _check_per_op(got, _reference(q[0], k, v, 1, 1, 128, 0), 128, tag)
    print(f"\n{tag} max err / bound: A {wa:.3g}, B {wb:.3g}")
    with pytest.raises(capi.BlkError) as e:
        capi.test_decode_attn(q[0], k, v, n_kv, 1, 1, 128, form=1)
    assert e.value.code == 4


def _run_batch(n_head, n_head_kv, d_head, lengths, patterns, seed):
    """one launch over rows of the given lengths; row b uses patterns[b % len(patterns)].  Returns the largest error / bound."""
    from blama_b200 import capi

    rng = np.random.default_rng(seed)
    rows = [_operands(rng, 1, n, n_head, n_head_kv, d_head, patterns[b % len(patterns)]) for b, n in enumerate(lengths)]
    q = np.concatenate([r[0] for r in rows]); k = np.concatenate([r[1] for r in rows]); v = np.concatenate([r[2] for r in rows])
    got = capi.test_decode_attn_batch(q, k, v, lengths, n_head, n_head_kv, d_head, seed=seed)
    worst = 0.0
    for b, (n, (qb, kb, vb)) in enumerate(zip(lengths, rows)):
        # the running maximum is corrected once per tile: up to n_tiles expf factors in one probability
        ref = _reference(qb[0], kb, vb, n_head, n_head_kv, d_head, (n + BD_TK - 1) // BD_TK)
        for h, (p, aV, V, o_exact, delta, eps) in enumerate(ref):
            o = got[b, h * d_head:(h + 1) * d_head].astype(np.float64)
            tag = f"[decode attn batch heads {n_head}/{n_head_kv} d {d_head} row {b} n_kv {n} {patterns[b % len(patterns)]} head {h}]"
            assert np.all(np.isfinite(o)), f"{tag}: non-finite output (a read through the wrong page, past n_kv or of the wrong layer)"
            bound = BF16_HALF_ULP * (np.abs(o_exact) + eps) + eps
            err = np.abs(o - o_exact)
            worst = max(worst, float((err / bound).max()))
            assert np.all(err <= bound), f"{tag}: worst err / bound {(err / bound).max():.3g}"
    return got, worst


@pytest.mark.parametrize("d_head", [64, 128])
@pytest.mark.parametrize("n_head,n_head_kv", HEADS)
def test_decode_attn_batch_lengths(n_head, n_head_kv, d_head):
    """rows on both sides of every 512-key tile boundary in one launch, every GQA ratio"""
    from blama_b200 import capi

    capi.init()
    _, worst = _run_batch(n_head, n_head_kv, d_head, BATCH_NKV, ["random"], seed=n_head * 100 + d_head)
    print(f"\n[decode attn batch heads {n_head}/{n_head_kv} d {d_head} n_kv {BATCH_NKV}] max err / bound {worst:.3g}")


@pytest.mark.parametrize("n_head,n_head_kv,d_head", [(8, 1, 128), (6, 2, 64), (2, 2, 128)])
def test_decode_attn_batch_patterns(n_head, n_head_kv, d_head):
    """uniform, peaked and ramp scores side by side in one launch (each length takes every pattern)"""
    from blama_b200 import capi

    capi.init()
    pats = ["uniform", "peaked", "rising", "falling"]
    lengths = [n for n in (2, 513, 1025, 3000) for _ in pats]
    patterns = [pats[i % 4] for i in range(len(lengths))]
    _, worst = _run_batch(n_head, n_head_kv, d_head, lengths, patterns, seed=d_head + n_head)
    print(f"\n[decode attn batch heads {n_head}/{n_head_kv} d {d_head} patterns] max err / bound {worst:.3g}")


@pytest.mark.parametrize("d_head", [64, 128])
def test_decode_attn_batch_64_rows(d_head):
    """a full batch of 64 rows with random lengths from 1 to 2000"""
    from blama_b200 import capi

    capi.init()
    lengths = [int(n) for n in np.random.default_rng(d_head).integers(1, 2001, 64)]
    _, worst = _run_batch(8, 1, d_head, lengths, ["random"], seed=11)
    print(f"\n[decode attn batch 64 rows d {d_head}] max err / bound {worst:.3g}")


def test_decode_attn_is_deterministic():
    """the same call twice gives the same bits, in both per-op forms and the batch kernel"""
    from blama_b200 import capi

    capi.init()
    rng = np.random.default_rng(1)
    q, k, v = _operands(rng, 1, 3000, 8, 1, 128, "random")
    for form in (0, 1):
        a, _ = capi.test_decode_attn(q[0], k, v, 3000, 8, 1, 128, form=form, seed=2)
        b, _ = capi.test_decode_attn(q[0], k, v, 3000, 8, 1, 128, form=form, seed=2)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), form
    lengths = [1, 700, 3000]
    rows = [_operands(rng, 1, n, 8, 1, 128, "random") for n in lengths]
    qb = np.concatenate([r[0] for r in rows]); kb = np.concatenate([r[1] for r in rows]); vb = np.concatenate([r[2] for r in rows])
    a = capi.test_decode_attn_batch(qb, kb, vb, lengths, 8, 1, 128, seed=4)
    b = capi.test_decode_attn_batch(qb, kb, vb, lengths, 8, 1, 128, seed=4)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
