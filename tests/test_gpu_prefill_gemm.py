"""The tcgen05 prefill GEMM (bf16 operands, f32 TMEM accumulation) called the way the layer loop calls it, against float64 on the operands
the kernel sees: bf16(x) and bf16(dequantised W) (de-quantisation itself is pinned bit-exact in test_gpu_kernels.py).

  op STORE   QKV (1 - 3 matrices side by side, mixed weight types, biases) and the lm_head chunk   C = X W^T (+ bias)
  op ACCUM   Wo / down onto the f32 residual, then the RMSNorm of the pass                        C += X W^T, xn = bf16(rmsnorm(C) w)
  op SWIGLU  gate + up                                                                              H = bf16(silu(X Wg^T) (X Wu^T))

each in the fused form (de-quantised in the GEMM) and the panel form (bf16 tile images filled first), with and without the deterministic
split-K: every tile split, only the partial last wave split, or an accumulate whose reduce the RMSNorm does (the deferred reduce).  Every
case checks that the plan which ran is the one launch_gemm's rule gives (restated below) and the one its id names.

Bounds (each printed beside the measured value):
  f32 outputs   |got - ref| <= 2e-4 max|ref| (per matrix): f32 accumulation over K <= 28672 products of bf16 operands stays two
                orders below this, while one 64-wide K block dropped or counted twice moves an output by ~1/8 of its std (~3e-2 max|ref|)
  accumulate    the same on the update, plus half an f32 ulp of the new residual (the residual is ~10x the update: that rounding is real)
  SwiGLU        half a bf16 ulp of the value, plus the propagated GEMM error 1.1 |u| dg + |silu(g)| du (|silu'| <= 1.1), plus 2^-18 of
                the value for __expf / __fdividef (relative error of ex2.approx after the f32 scaling of |g| < 30)
  deferred xn   within 0.51 bf16 ulp of bf16(rmsnorm(C_device) w) on the device's own C, as test_rmsnorm_bf16 states it
Exact: the deferred reduce equals the reduce kernel + the plain RMSNorm (C and xn), fused equals panel at the same plan, and a split-K
call gives the same bits twice."""
import math

import numpy as np
import pytest

from blama_b200 import gguf_synth as gs

STORE, ACCUM, SWIGLU = 0, 1, 2
PG_BM, PG_BN, PG_BK = 256, 256, 64
WS_TILES = 1                   # split-K workspace: n_SM x 65536 floats = one 256 x 256 f32 tile per SM
BF16_ULP = 2.0 ** -7           # relative spacing of bf16 at the bottom of a binade: half an ulp = 2^-8
REL = 2e-4
EXPF_REL = 2.0 ** -18
CHAIN_PDL_MAX_TOKENS = 1024
TYPE_NAME = {gs.Q4_K: "Q4_K", gs.Q5_K: "Q5_K", gs.Q6_K: "Q6_K", gs.Q8_0: "Q8_0", gs.F32: "F32"}
FUSED_PAIRS = {(t, t) for t in (gs.Q4_K, gs.Q5_K, gs.Q6_K, gs.Q8_0, gs.F32, gs.F16)} | {(gs.Q4_K, gs.Q6_K), (gs.Q4_K, gs.Q5_K)}
PANEL_TYPES = (gs.Q4_K, gs.Q5_K, gs.Q6_K, gs.Q8_0)


def bf16_round(x: np.ndarray) -> np.ndarray:
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


# ---- launch_gemm's plan, restated ----------------------------------------------------------------------------------------------------
def expected_plan(op, types, Ns, K, T, n_sm, form, split):
    """What prefill_gemm / prefill_gemm_multi / prefill_gemm_swiglu launch on n_sm SMs (prefill.cu): a partial last wave of at most half
    the SMs, after at most two whole waves, is split S = min(8, n_sm // rem, k_blocks // 8) ways, fewer if S * rem tiles do not fit the
    workspace; the reduce is deferred only for a full-width accumulate (N % 256 == 0) with every tile split."""
    n = len(Ns)
    panel = form == 1 and all(t in PANEL_TYPES for t in types)
    launches = 1
    sk = split > 0
    if op == STORE and n > 1:
        fuse = types[0] == types[1] and (n == 2 or (types[0], types[2]) in FUSED_PAIRS)
        if not panel and not fuse:
            launches, sk = n, False          # one launch per matrix, no split-K (column-offset C)
    m_tiles = -(-T // PG_BM)
    n_tiles = -(-Ns[0] // 128) if op == SWIGLU else sum(-(-N // PG_BN) for N in Ns)
    if launches > 1:
        n_tiles = -(-Ns[-1] // PG_BN)        # the plan reported is the last launch's
    tiles = m_tiles * n_tiles
    S, n_whole = 1, tiles
    kb = K // PG_BK
    if sk:
        nw = (tiles // n_sm) * n_sm
        rem = tiles - nw
        if rem > 0 and 2 * rem <= n_sm and nw <= 2 * n_sm:
            s = min(8, n_sm // rem, kb // 8)
            while s > 1 and s * rem > n_sm * WS_TILES:
                s -= 1
            if s > 1 and all(N % 4 == 0 for N in Ns):
                S, n_whole = s, nw
    deferred = split == 2 and op == ACCUM and S > 1 and n_whole == 0 and Ns[0] % PG_BN == 0
    return dict(n_sm=n_sm, launches=launches, k_splits=S, n_whole=n_whole, deferred=int(deferred), panel=int(panel))


def path_of(plan):
    if plan["deferred"]:
        return "deferred"
    if plan["k_splits"] == 1:
        return "nosplit"
    return "wave" if plan["n_whole"] > 0 else "split"


def ragged(plan, K):
    """the last K split is shorter than the others"""
    S, kb = plan["k_splits"], K // PG_BK
    k_per = math.ceil(kb / S)
    return S > 1 and kb - (S - 1) * k_per < k_per


# ---- operands and the float64 reference --------------------------------------------------------------------------------------------
def make_weights(rng, oracle, gtype, rows, K, max_elems=1 << 25):
    """(raw blocks of a rows x K matrix, its distinct rows bf16(dequant) as float32).  Matrices above max_elems repeat a block of U
    distinct rows (row r = row r % U, U odd so no multiple of the 256-row tile maps a row onto an equal one): the kernel reads the full
    production shape, the reference computes U rows."""
    U = rows if rows * K <= max_elems else (max_elems // K) | 1
    blk = gs.random_blocks(rng, gtype, U * K, 1.0 / np.sqrt(K))
    w = bf16_round(oracle.dequantize(gtype, blk, U * K).reshape(U, K))
    if U != rows:
        blk = np.tile(blk.reshape(U, -1), (-(-rows // U), 1))[:rows].reshape(-1)
    return blk, w


def ref_gemm(xb64: np.ndarray, w: np.ndarray, rows: int) -> np.ndarray:
    """float64 X W^T over the distinct rows of w (blocks of rows: float64 temporaries stay under ~1 GB), repeated out to `rows` columns"""
    T, K = xb64.shape
    U = w.shape[0]
    out = np.empty((T, U))
    step = max(1, (1 << 25) // K)
    for r0 in range(0, U, step):
        out[:, r0:r0 + step] = xb64 @ w[r0:r0 + step].astype(np.float64).T
    return out if U == rows else np.tile(out, (1, -(-rows // U)))[:, :rows]


# ---- the cases -----------------------------------------------------------------------------------------------------------------------
Q4, Q5, Q6, Q8 = gs.Q4_K, gs.Q5_K, gs.Q6_K, gs.Q8_0
# id: (op, [(type, N, bias)], K, T, split, path on 148 SMs).  Production K always; the ids name the model whose layer has the shape.
PROD = {
    "8b-qkv-T1": (STORE, [(Q4, 4096, False), (Q4, 1024, False), (Q6, 1024, False)], 4096, 1, 1, "split"),
    "8b-qkv-T200": (STORE, [(Q4, 4096, False), (Q4, 1024, False), (Q6, 1024, False)], 4096, 200, 1, "split"),
    "8b-qkv-T2048": (STORE, [(Q4, 4096, False), (Q4, 1024, False), (Q6, 1024, False)], 4096, 2048, 1, "wave"),
    "qwen7b-qkv-bias-T64": (STORE, [(Q8, 3584, True), (Q8, 512, True), (Q8, 512, True)], 3584, 64, 1, "split"),
    "qwen7b-qkv-bias-T300": (STORE, [(Q8, 3584, True), (Q8, 512, True), (Q8, 512, True)], 3584, 300, 1, "split"),
    "70b-qkv-T48": (STORE, [(Q4, 8192, False), (Q4, 1024, False), (Q5, 1024, False)], 8192, 48, 1, "split"),
    # a type mix without a fused kernel: one launch per matrix in the fused form, one launch in the panel form
    "q6q6q4-qkv-bias-T64": (STORE, [(Q6, 2048, True), (Q6, 512, True), (Q4, 512, True)], 2048, 64, 1, "nosplit"),
    "8b-wo-T1": (ACCUM, [(Q4, 4096, False)], 4096, 1, 2, "deferred"),
    "8b-wo-T130": (ACCUM, [(Q4, 4096, False)], 4096, 130, 2, "deferred"),
    "8b-wo-T700": (ACCUM, [(Q4, 4096, False)], 4096, 700, 2, "deferred"),
    "8b-wo-T1100": (ACCUM, [(Q4, 4096, False)], 4096, 1100, 2, "nosplit"),
    "8b-down-T64": (ACCUM, [(Q6, 4096, False)], 14336, 64, 2, "deferred"),
    "8b-down-T700": (ACCUM, [(Q6, 4096, False)], 14336, 700, 2, "deferred"),
    "qwen7b-down-T40": (ACCUM, [(Q8, 3584, False)], 18944, 40, 2, "deferred"),
    "70b-down-T16": (ACCUM, [(Q4, 8192, False)], 28672, 16, 2, "deferred"),
    "70b-wo-T300": (ACCUM, [(Q4, 8192, False)], 8192, 300, 2, "deferred"),
    "1b-swiglu-T100": (SWIGLU, [(Q8, 8192, False)] * 2, 2048, 100, 1, "split"),
    "small-qwen2-gq7-swiglu-T75": (SWIGLU, [(Q8, 2304, False)] * 2, 1792, 75, 1, "split"),
    "8b-swiglu-T32": (SWIGLU, [(Q4, 14336, False)] * 2, 4096, 32, 1, "nosplit"),
    "qwen7b-swiglu-T32": (SWIGLU, [(Q8, 18944, False)] * 2, 3584, 32, 1, "nosplit"),
    "8b-lm-head-T512": (STORE, [(Q6, 128256, False)], 4096, 512, 0, "nosplit"),
}
# the kernel-level shapes the file started from, as single-matrix STORE inputs (both forms, with and without the split-K workspace)
CASES = [(256, 256, 256), (300, 384, 1024), (1, 256, 512), (77, 1000, 256), (512, 1024, 4096), (640, 512, 14336)]
GTYPES = [(gs.Q4_K, "Q4_K"), (gs.Q6_K, "Q6_K"), (gs.Q8_0, "Q8_0"), (gs.Q5_K, "Q5_K"), (gs.F32, "F32")]


def _plan_148(case):
    op, mats, K, T, split, _ = case
    return expected_plan(op, [m[0] for m in mats], [m[1] for m in mats], K, T, 148, 0, split)


def test_cases_cover_every_plan_on_148_sms():
    """Across the cases: both forms, every op (one matrix, three mixed-type matrices with biases), every split path, the three token
    classes (one accumulator, both halves of one M tile, several M tiles) and a last K split shorter than the others -- and every
    production case's id names the path the rule gives on a 148-SM B200."""
    paths, ops, t_classes, short_last = set(), set(), set(), False
    for name, case in PROD.items():
        op, mats, K, T, split, path = case
        plan = _plan_148(case)
        assert path_of(plan) == path, (name, plan)
        paths.add(path)
        kinds = {m[0] for m in mats}
        ops.add((op, len(mats), len(kinds) > 1 and any(m[2] for m in mats)) if op == STORE else (op,))
        t_classes.add(0 if T <= 128 else 1 if T <= 256 else 2)
        short_last |= ragged(plan, K)
    for T, N, K in CASES:
        plan = expected_plan(STORE, [gs.Q4_K], [N], K, T, 148, 0, 1)
        paths.add(path_of(plan))
        ops.add((STORE, 1, False))
        short_last |= ragged(plan, K)
    assert paths == {"nosplit", "split", "wave", "deferred"}, paths
    assert {(STORE, 1, False), (STORE, 3, True), (ACCUM,), (SWIGLU,)} <= ops, ops
    assert t_classes == {0, 1, 2}
    assert short_last
    # the named plans of the case table, worked out by hand from the rule
    assert _plan_148(PROD["8b-qkv-T1"])["k_splits"] == 6 and ragged(_plan_148(PROD["8b-qkv-T1"]), 4096)
    assert _plan_148(PROD["8b-qkv-T2048"]) == dict(n_sm=148, launches=1, k_splits=3, n_whole=148, deferred=0, panel=0)
    assert _plan_148(PROD["70b-down-T16"])["k_splits"] == 4
    assert _plan_148(PROD["small-qwen2-gq7-swiglu-T75"])["k_splits"] == 3
    assert _plan_148(PROD["q6q6q4-qkv-bias-T64"])["launches"] == 3
    assert _plan_148(PROD["8b-lm-head-T512"])["n_whole"] == 1002


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------
def _run(capi, op, mats, K, x, form, split, c=None, norm_w=None, eps=1e-5):
    return capi.test_gemm_layer(op, mats, K, x, form=form, split=split, c=c, norm_w=norm_w, eps=eps)


def _check_plan(name, got, op, types, Ns, K, T, form, split, path=None):
    want = expected_plan(op, types, Ns, K, T, got["n_sm"], form, split)
    print(f"[{name} form {form} split {split}] plan {got}")
    assert got == want, (got, want)
    if path is not None:
        assert path_of(got) == path, f"{name}: ran the {path_of(got)} path on {got['n_sm']} SMs, the case names {path}"


def _check_store(name, got, ref, Ns):
    col = 0
    for N in Ns:
        g, r = got[:, col:col + N], ref[:, col:col + N]
        err, bound = float(np.abs(g - r).max()), REL * float(np.abs(r).max())
        print(f"  [{name}] cols {col}..{col + N}: max err {err:.3g} <= {bound:.3g}")
        assert np.isfinite(g).all() and err <= bound, (col, err, bound)
        col += N


def _check_accum(name, got, c0, upd):
    ref = c0.astype(np.float64) + upd
    err = np.abs(got - ref)
    bound = REL * np.abs(upd).max() + 2.0 ** -24 * np.abs(ref)
    print(f"  [{name}] accumulate: max err {err.max():.3g}, max err / bound {(err / bound).max():.3g}")
    assert np.isfinite(got).all() and np.all(err <= bound), float((err / bound).max())


def _check_xn(name, xn, c_dev, w, eps):
    c64 = c_dev.astype(np.float64)
    ref = c64 / np.sqrt((c64 * c64).mean(axis=1, keepdims=True) + eps) * w.astype(np.float64)
    rel = np.abs(xn - ref) / np.maximum(np.abs(ref), 1e-30)
    print(f"  [{name}] rmsnorm on the device's C: max rel err {rel.max():.3g} <= {BF16_ULP * 0.51 + 1e-6:.3g}")
    assert rel.max() <= BF16_ULP * 0.51 + 1e-6


def _check_swiglu(name, h, g, u):
    dg, du = REL * np.abs(g).max(), REL * np.abs(u).max()
    silu = g / (1.0 + np.exp(-g))
    ref = silu * u
    e = 1.1 * np.abs(u) * dg + np.abs(silu) * du + EXPF_REL * np.abs(ref)
    bound = BF16_ULP / 2 * (np.abs(ref) + e) + e
    err = np.abs(h - ref)
    print(f"  [{name}] swiglu: max err {err.max():.3g}, max err / bound {(err / bound).max():.3g}")
    assert np.isfinite(h).all() and np.all(err <= bound), float((err / bound).max())


@pytest.mark.gpu
@pytest.mark.parametrize("gtype,name", GTYPES)
@pytest.mark.parametrize("T,N,K", CASES)
@pytest.mark.parametrize("form", ["fused", "panel"])
def test_prefill_gemm(gtype, name, T, N, K, form, oracle):
    """One matrix, STORE: form = fused (weights de-quantised inside the GEMM) or panel (de-quantised once to bf16 tile images), each
    without and with the split-K workspace."""
    from blama_b200 import capi

    if form == "panel" and gtype == gs.F32:
        pytest.skip("the panel form covers the quantised types")
    if gtype == gs.F32 and K > 4096:
        pytest.skip("F32 weights are a test-only format")
    f = 1 if form == "panel" else 0
    rng = np.random.default_rng(T * 3 + N + K)
    blk = gs.random_blocks(rng, gtype, N * K, 1.0 / np.sqrt(K))
    x = rng.standard_normal((T, K)).astype(np.float32)
    w = bf16_round(oracle.dequantize(gtype, blk, N * K).reshape(N, K))
    want = ref_gemm(bf16_round(x).astype(np.float64), w, N)
    for split in (0, 1):
        got, _, plan = _run(capi, STORE, [(gtype, blk, N, None)], K, x, f, split)
        _check_plan(f"{name} {T}x{N}x{K}", plan, STORE, [gtype], [N], K, T, f, split)
        _check_store(f"{name} {T}x{N}x{K}", got, want, [N])


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PROD))
def test_prefill_gemm_as_the_layer_loop_calls_it(case, oracle):
    from blama_b200 import capi

    op, spec, K, T, split, path = PROD[case]
    rng = np.random.default_rng(sum(map(ord, case)))
    types, Ns = [s[0] for s in spec], [s[1] for s in spec]
    mats, ws = [], []
    for gtype, N, has_bias in spec:
        blk, w = make_weights(rng, oracle, gtype, N, K)
        bias = (rng.standard_normal(N) * 0.5).astype(np.float32) if has_bias else None
        mats.append((gtype, blk, N, bias)); ws.append(w)
    x = rng.standard_normal((T, K)).astype(np.float32)
    xb = bf16_round(x).astype(np.float64)
    forms = (0, 1) if all(t in PANEL_TYPES for t in types) else (0,)
    outs, plans = {}, {}
    if op == STORE:
        ref = np.concatenate([ref_gemm(xb, w, N) + (0.0 if b is None else b.astype(np.float64)) for (_, _, N, b), w in zip(mats, ws)], axis=1)
        for f in forms:
            got, _, plan = _run(capi, STORE, mats, K, x, f, split)
            _check_plan(case, plan, op, types, Ns, K, T, f, split, path if f == 0 else None)
            _check_store(case, got, ref, Ns)
            outs[f] = (got,)
            plans[f] = plan
    elif op == SWIGLU:
        g, u = ref_gemm(xb, ws[0], Ns[0]), ref_gemm(xb, ws[1], Ns[1])
        for f in forms:
            _, h, plan = _run(capi, SWIGLU, mats, K, x, f, split)
            _check_plan(case, plan, op, types, Ns, K, T, f, split, path)
            _check_swiglu(case, h, g, u)
            outs[f] = (h,)
            plans[f] = plan
    else:
        N = Ns[0]
        upd = ref_gemm(xb, ws[0], N)
        c0 = (rng.standard_normal((T, N)) * 10.0 * upd.std()).astype(np.float32)        # the residual, ~10x the update
        norm_w = (1.0 + 0.1 * rng.standard_normal(N)).astype(np.float32)
        eps = 1e-5
        for f in forms:
            res = {}
            for sp in (1, 2) if split == 2 else (split,):
                got, xn, plan = _run(capi, ACCUM, mats, K, x, f, sp, c=c0, norm_w=norm_w, eps=eps)
                _check_plan(case, plan, op, types, Ns, K, T, f, sp, path if sp == split else None)
                _check_accum(case, got, c0, upd)
                _check_xn(case, xn, got, norm_w, eps)
                res[sp] = (got, xn)
                plans[f] = plan
            if split == 2:
                # DESIGN §5: the RMSNorm adds the partial sums in the reduce kernel's order (splits, then the residual): bit-identical
                assert np.array_equal(res[1][0], res[2][0]), "deferred reduce: C differs from the reduce kernel's"
                assert np.array_equal(res[1][1], res[2][1]), "deferred reduce: xn differs from reduce kernel + RMSNorm"
            outs[f] = res[split]
        if T > CHAIN_PDL_MAX_TOKENS:
            print(f"  [{case}] {T} tokens: launched without programmatic dependent launch, as a pass of that size is")
    if len(forms) == 2 and {**plans[0], "panel": 1} == plans[1]:
        # at the same plan both forms write the same bf16 B tile (RawK64<T>::expand) and issue the same MMAs: the same bits
        for a, b in zip(outs[0], outs[1]):
            assert np.array_equal(a, b), f"fused and panel differ: max {np.nanmax(np.abs(a - b)):.3g}"
    if path != "nosplit":
        # run to run: the split-K partial sums are added in split order by one thread per output
        c2, h2, _ = _run(capi, op, mats, K, x, 0, split, c=c0 if op == ACCUM else None, norm_w=norm_w if op == ACCUM else None)
        again = (c2,) if op == STORE else (h2,) if op == SWIGLU else (c2, h2)
        for a, b in zip(outs[0], again):
            assert np.array_equal(a, b), "split-K GEMM is not deterministic"
