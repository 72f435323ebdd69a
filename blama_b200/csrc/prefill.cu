// prefill.cu -- launchers of the multi-token prefill path (tcgen05 GEMM + helpers).
#include "prefill.hpp"
#include "prefill_gemm.cuh"
#include "prefill_attn_tc.cuh"

#include <mutex>

namespace blk {
namespace {

using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else (void)cudaGetLastError();
    });
    return fn;
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, size_t n) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < n) {
        const float4 v = *reinterpret_cast<const float4*>(x + i);
        __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
        uint2 o; o.x = *reinterpret_cast<uint32_t*>(&a); o.y = *reinterpret_cast<uint32_t*>(&b);
        *reinterpret_cast<uint2*>(y + i) = o;
    } else {
        for (size_t j = i; j < n; j++) y[j] = __float2bfloat16_rn(x[j]);
    }
}

} // namespace

cudaError_t convert_f32_to_bf16(const float* x, __nv_bfloat16* y, size_t n, cudaStream_t st) {
    const size_t threads = (n + 3) / 4;
    f32_to_bf16_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(x, y, n);
    return cudaGetLastError();
}

namespace {
using GemmKernel = void (*)(const CUtensorMap, const PrefillGemmArgs);

GemmKernel pick_kernel(int ta, int tb) {
#define BLK_K(A, B) if (ta == A && tb == B) return prefill_gemm_kernel<A, B>;
    BLK_K(QT_Q4_K, QT_Q4_K) BLK_K(QT_Q6_K, QT_Q6_K) BLK_K(QT_Q8_0, QT_Q8_0) BLK_K(QT_Q5_K, QT_Q5_K) BLK_K(QT_F32, QT_F32) BLK_K(QT_F16, QT_F16)
    BLK_K(QT_Q4_K, QT_Q6_K) BLK_K(QT_Q4_K, QT_Q5_K) BLK_K(QT_PANEL, QT_PANEL)
#undef BLK_K
    return nullptr;
}

// panel: nullptr for the fused (in-kernel dequantisation) form, else the bf16 panel (panel_layout) the B tiles are read from
cudaError_t launch_gemm(PrefillGemmArgs& a, int ta, int tb, const __nv_bfloat16* X, cudaStream_t st, const __nv_bfloat16* panel = nullptr,
                        const SplitKWs* sk = nullptr, GemmPlan* plan = nullptr) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return cudaErrorNotSupported;
    if (a.K % PG_BK || a.T <= 0 || a.n_tiles <= 0) return cudaErrorInvalidValue;
    GemmKernel kernel = panel ? pick_kernel(QT_PANEL, QT_PANEL) : pick_kernel(ta, tb);
    if (!kernel) return cudaErrorInvalidValue;
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {(cuuint64_t)a.K, (cuuint64_t)a.T};
    const cuuint64_t gstride[1] = {(cuuint64_t)a.K * sizeof(__nv_bfloat16)};
    const cuuint32_t box[2] = {(cuuint32_t)PG_BK, 128u};
    const cuuint32_t estr[2] = {1u, 1u};
    CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(X), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    a.panel = reinterpret_cast<const unsigned char*>(panel);      // tile images, fetched with plain bulk copies (no tensor map)
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PG_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int tiles = ((a.T + PG_BM - 1) / PG_BM) * a.n_tiles;
    // The last, partial wave of tiles (all of them when there are fewer tiles than SMs) is split along K so that its work items fill
    // the SMs; partial sums go to the workspace and are added in split order by a second kernel (deterministic).  Every split gets
    // at least 8 K blocks (hence never an empty one); a wave that is at least half full is left alone.
    a.k_splits = 1; a.n_whole = tiles; a.ws = nullptr;
    if (sk && sk->ws && sms > 0) {
        const int n_whole = (tiles / sms) * sms, rem = tiles - n_whole;
        if (rem > 0 && 2 * rem <= sms && n_whole <= 2 * sms) {      // (after many whole waves the partial one is a small share: not worth a second kernel)
            int S = std::min(8, std::min(sms / rem, (a.K / PG_BK) / 8));
            while (S > 1 && (size_t)S * (size_t)rem * (size_t)(PG_BM * PG_BN) > sk->elems) S--;
            bool ok = S > 1;
            for (int i = 0; i < a.nseg && ok; i++) ok = a.seg[i].W.N % 4 == 0 && a.seg[i].col0 % 4 == 0;
            if (a.mode == PG_SWIGLU) ok = ok && a.ldh % 4 == 0; else ok = ok && a.ldc % 4 == 0;
            if (ok) { a.k_splits = S; a.n_whole = n_whole; a.ws = sk->ws; }
        }
    }
    const int items = a.n_whole + (tiles - a.n_whole) * a.k_splits;
    const int grid = items < sms ? items : sms;
    e = launch_chain(kernel, dim3((unsigned)grid), dim3(PG_THREADS), PG_SMEM_BYTES, st, tmap, a);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (plan) { plan->n_sm = sms; plan->launches++; plan->k_splits = a.k_splits; plan->n_whole = a.n_whole; plan->deferred = false; plan->panel = panel != nullptr; }
    if (e != cudaSuccess || a.k_splits == 1) return e;
    if (sk && sk->defer && a.mode == PG_ACCUM && a.n_whole == 0 && a.nseg == 1 && a.seg[0].col0 == 0 && !a.seg[0].bias &&
        a.seg[0].W.N % PG_BN == 0 && a.ldc == a.seg[0].W.N) {
        // every tile is split and full width: the caller's next RMSNorm over C adds the partial sums (same order: splits, then the residual)
        if (sk->defer->ws) return cudaErrorInvalidValue;      // an earlier deferred reduce was never consumed: fail loudly, never drop partial sums
        *sk->defer = PendingReduce{a.ws, a.k_splits, (a.T + PG_BM - 1) / PG_BM};
        if (plan) plan->deferred = true;
        return cudaSuccess;
    }
    e = launch_chain(splitk_reduce_kernel, dim3((unsigned)(tiles - a.n_whole), 32), dim3(256), 0, st, a);
    return e == cudaSuccess ? cudaGetLastError() : e;
}

// first pass of the two-pass form: W -> panel rows [row0, row0 + W.N)
cudaError_t panel_dequant(const QMat& W, __nv_bfloat16* panel, long long row0, cudaStream_t st) {
    if (row0 % 128) return cudaErrorInvalidValue;
    const long long total = (long long)((W.N + 127) / 128) * 128 * (W.K >> 6);
    const unsigned grid = (unsigned)((total + 255) / 256);
    unsigned char* dst = reinterpret_cast<unsigned char*>(panel);
    switch (W.type) {
        case QT_Q4_K: panel_dequant_kernel<QT_Q4_K><<<grid, 256, 0, st>>>(W, dst, row0); break;
        case QT_Q5_K: panel_dequant_kernel<QT_Q5_K><<<grid, 256, 0, st>>>(W, dst, row0); break;
        case QT_Q6_K: panel_dequant_kernel<QT_Q6_K><<<grid, 256, 0, st>>>(W, dst, row0); break;
        case QT_Q8_0: panel_dequant_kernel<QT_Q8_0><<<grid, 256, 0, st>>>(W, dst, row0); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}
bool panel_type_ok(int t) { return t == QT_Q4_K || t == QT_Q5_K || t == QT_Q6_K || t == QT_Q8_0; }

// The bf16 panel layout of the two-pass form: part i's rows start at panel row row0[i] (if row0 is given); returns the rows the
// panel holds.  The parts of one GEMM take whole 256-row tiles one after another.  A SwiGLU tile pairs 128 gate rows with the
// matching 128 up rows, so there up starts at the first 128-aligned row after gate.
long long panel_layout(const GemmPart* parts, int n_parts, bool swiglu, long long* row0 = nullptr) {
    const int align = swiglu ? 128 : PG_BN;
    long long rows = 0;
    for (int i = 0; i < n_parts; i++) {
        if (row0) row0[i] = rows;
        rows += (long long)((parts[i].W->N + align - 1) / align) * align;
    }
    return rows;
}
} // namespace

cudaError_t prefill_gemm(const QMat& W, const __nv_bfloat16* X, int T, float* C, long long ldc, const float* bias, int mode, cudaStream_t st,
                         const __nv_bfloat16* panel, const SplitKWs* sk, GemmPlan* plan) {
    PrefillGemmArgs a{};
    a.nseg = 1; a.seg[0] = {W, bias, 0, 0};
    a.C = C; a.ldc = ldc; a.T = T; a.K = W.K; a.mode = mode;
    a.n_tiles = (W.N + PG_BN - 1) / PG_BN;
    const bool use_panel = panel && panel_type_ok(W.type) && W.K % 64 == 0;
    return launch_gemm(a, W.type, W.type, X, st, use_panel ? panel : nullptr, (W.N % 4 == 0 && ldc % 4 == 0) ? sk : nullptr, plan);
}
// the dequantisation passes alone, so that a caller can run them on a second stream one GEMM ahead; false = this combination takes
// the fused form (the GEMM call must then get panel = nullptr)
bool prefill_panel_fill(const GemmPart* parts, int n_parts, bool swiglu, __nv_bfloat16* panel, cudaStream_t st, cudaError_t* err) {
    *err = cudaSuccess;
    if (!panel || n_parts < 1 || n_parts > 3 || (swiglu && (n_parts != 2 || parts[1].W->type != parts[0].W->type))) return false;
    for (int i = 0; i < n_parts; i++) if (!panel_type_ok(parts[i].W->type) || parts[i].W->K != parts[0].W->K || parts[i].col0 % 4 || parts[i].W->K % 64) return false;
    long long row0[3];
    panel_layout(parts, n_parts, swiglu, row0);
    for (int i = 0; i < n_parts; i++) {
        *err = panel_dequant(*parts[i].W, panel, row0[i], st);
        if (*err != cudaSuccess) return true;
    }
    return true;
}
size_t prefill_panel_elems(const GemmPart* parts, int n_parts, bool swiglu) {
    return (size_t)panel_layout(parts, n_parts, swiglu) * (size_t)parts[0].W->K;
}

cudaError_t prefill_gemm_multi(const GemmPart* parts, int n_parts, const __nv_bfloat16* X, int T, float* C, long long ldc, cudaStream_t st,
                               const __nv_bfloat16* panel, const SplitKWs* sk, GemmPlan* plan) {
    bool all_panel = panel != nullptr && n_parts >= 1 && n_parts <= 3;
    for (int i = 0; i < n_parts && all_panel; i++) all_panel = panel_type_ok(parts[i].W->type) && parts[i].W->K == parts[0].W->K && parts[i].col0 % 4 == 0;
    bool fuse = n_parts >= 2 && n_parts <= 3 && parts[0].W->type == parts[1].W->type;
    for (int i = 0; i < n_parts && fuse; i++) fuse = (parts[i].col0 % 4 == 0) && parts[i].W->K == parts[0].W->K;
    if (fuse && n_parts == 3 && !pick_kernel(parts[0].W->type, parts[2].W->type)) fuse = false;
    if (!all_panel && !fuse) {
        for (int i = 0; i < n_parts; i++) {
            cudaError_t e = prefill_gemm(*parts[i].W, X, T, C + parts[i].col0, ldc, parts[i].bias, 0, st, nullptr, nullptr, plan);     // (column-offset C: no split-K)
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    }
    // one launch over every segment; the panel form takes any mix of weight types (each segment is dequantised to its own rows)
    PrefillGemmArgs a{};
    a.nseg = n_parts; a.C = C; a.ldc = ldc; a.T = T; a.K = parts[0].W->K; a.mode = PG_STORE;
    long long row0[3];
    a.n_tiles = (int)(panel_layout(parts, n_parts, false, row0) / PG_BN);
    for (int i = 0; i < n_parts; i++) a.seg[i] = {*parts[i].W, parts[i].bias, parts[i].col0, (int)(row0[i] / PG_BN)};
    bool sk_ok = ldc % 4 == 0;
    for (int i = 0; i < n_parts; i++) sk_ok = sk_ok && parts[i].W->N % 4 == 0;
    return launch_gemm(a, parts[0].W->type, n_parts == 3 ? parts[2].W->type : parts[0].W->type, X, st, all_panel ? panel : nullptr, sk_ok ? sk : nullptr, plan);
}

cudaError_t prefill_gemm_swiglu(const QMat& gate, const QMat& up, const __nv_bfloat16* X, int T, __nv_bfloat16* H, long long ldh, cudaStream_t st,
                                const __nv_bfloat16* panel, const SplitKWs* sk, GemmPlan* plan) {
    if (gate.type != up.type || gate.N != up.N || gate.K != up.K || ldh % 8) return cudaErrorInvalidValue;
    PrefillGemmArgs a{};
    a.nseg = 2; a.seg[0] = {gate, nullptr, 0, 0}; a.seg[1] = {up, nullptr, 0, 0};
    a.H = H; a.ldh = ldh; a.T = T; a.K = gate.K; a.mode = PG_SWIGLU;
    a.n_tiles = (gate.N + 127) / 128;
    if (!(panel && panel_type_ok(gate.type) && gate.K % 64 == 0)) return launch_gemm(a, gate.type, gate.type, X, st, nullptr, sk, plan);
    const GemmPart parts[2] = {{&gate, nullptr, 0}, {&up, nullptr, 0}};
    long long row0[2];
    panel_layout(parts, 2, true, row0);
    a.panel_up_row0 = (int)row0[1];
    return launch_gemm(a, gate.type, gate.type, X, st, panel, sk, plan);
}

namespace {
bool encode_2d_f16(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t row_stride_elems, uint32_t box_inner, uint32_t box_outer) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
    const cuuint64_t gstride[1] = {(cuuint64_t)row_stride_elems * sizeof(__half)};
    const cuuint32_t box[2] = {box_inner, box_outer};
    const cuuint32_t estr[2] = {1u, 1u};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
template <int GQ, int GQS = GQ>
cudaError_t launch_attn_tc(const CUtensorMap& mq, const CUtensorMap& mk, const CUtensorMap& mv, const AttnTcArgs& a, int n_head_kv, cudaStream_t st) {
    {   // the opt-in is per (function, device): one replica per GPU in one process launches this on every device
        cudaError_t e = cudaFuncSetAttribute(prefill_attn_tc_kernel<GQ, GQS>, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM_BYTES);
        if (e != cudaSuccess) return e;
    }
    constexpr int BQ = 128 / GQS;
    (void)launch_chain(prefill_attn_tc_kernel<GQ, GQS>, dim3((a.T + BQ - 1) / BQ, n_head_kv), dim3(AT_THREADS), AT_SMEM_BYTES, st, mq, mk, mv, a);
    return cudaGetLastError();
}
int attn_tc_slots(int gq) { return gq <= 1 ? 1 : gq <= 2 ? 2 : gq <= 4 ? 4 : 8; }
} // namespace

// ---- verifier logits at the claimed ids only (Session.cpp:263-282 reads nothing else of the row) -------------------------
// One warp per (position, claimed id): dot(bf16(dequant(W[id])), xn[t]) in f32 -- the arithmetic of the GEMM form (bf16
// operands, f32 accumulation) without the 2 T V d flops of the full vocabulary projection.
__global__ void __launch_bounds__(256) claimed_logits_kernel(const QMat W, const __nv_bfloat16* __restrict__ xn, const int32_t* __restrict__ claimed,
                                                             const int32_t* __restrict__ n_claimed, int n, float* __restrict__ gathered) {
    const int gw = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int t = gw / 10, j = gw - t * 10;
    if (t >= n) return;
    float out = 0.0f;
    if (j < n_claimed[t]) {
        const int id = claimed[(size_t)t * 10 + j];
        if (id < 0 || id >= W.N) out = -INFINITY;
        else {
            float acc = 0.0f;
            const __nv_bfloat16* x = xn + (size_t)t * W.K;
            for (int kb = lane; kb < (W.K >> 6); kb += 32) {
                float w[64];
                dequant_k64(W, id, kb, w);
                const uint4* xv = reinterpret_cast<const uint4*>(x + (size_t)kb * 64);
#pragma unroll
                for (int c = 0; c < 8; c++) {
                    const uint4 xx = xv[c];
                    const __nv_bfloat162* xb = reinterpret_cast<const __nv_bfloat162*>(&xx);
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const float2 xf = __bfloat1622float2(xb[i]);
                        acc += __bfloat162float(__float2bfloat16_rn(w[c * 8 + 2 * i])) * xf.x;
                        acc += __bfloat162float(__float2bfloat16_rn(w[c * 8 + 2 * i + 1])) * xf.y;
                    }
                }
            }
            out = warp_sum(acc);
        }
    }
    if (lane == 0) gathered[(size_t)t * 10 + j] = out;
}

cudaError_t prefill_claimed_logits(const QMat& W, const __nv_bfloat16* xn, const int32_t* claimed, const int32_t* n_claimed, int n, float* gathered, cudaStream_t st) {
    if (W.K % 64 || n <= 0) return cudaErrorInvalidValue;
    const long long warps = (long long)n * 10;
    claimed_logits_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, st>>>(W, xn, claimed, n_claimed, n, gathered);
    return cudaGetLastError();
}

bool prefill_attn_tc_supported(int d_head, int n_head, int n_head_kv) {
    const int gq = n_head_kv > 0 ? n_head / n_head_kv : 0;
    return d_head == 128 && gq >= 1 && gq <= 8 && encode_tiled() != nullptr;
}

cudaError_t prefill_attn_tc(const __half* q, const __half* k_pool, const __half* v_pool, const int32_t* page_table, int n_pages, const int32_t* pos0_dev,
                            int pos0, __nv_bfloat16* out, __half* vt, int ctx_pad, int T, int n_head, int n_head_kv, int kv_dim, float scale, cudaStream_t st) {
    const int gq = n_head / n_head_kv, dq = n_head * 128, n_keys = pos0 + T;
    if (n_keys > ctx_pad || ctx_pad % 128) return cudaErrorInvalidValue;
    // V^T of every key this chunk can see (zero padded to the key tile)
    (void)launch_chain(vt_transpose_kernel, dim3((n_keys + 127) / 128 * 2, n_head_kv), dim3(256), 0, st, v_pool, page_table, kv_dim, n_keys, ctx_pad, vt);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    CUtensorMap mq, mk, mv;
    if (!encode_2d_f16(&mq, q, (uint64_t)dq, (uint64_t)T, (uint64_t)dq, 64, (uint32_t)(128 / attn_tc_slots(gq)))) return cudaErrorInvalidValue;
    if (!encode_2d_f16(&mk, k_pool, (uint64_t)kv_dim, (uint64_t)n_pages * KV_PAGE, (uint64_t)kv_dim, 64, 64)) return cudaErrorInvalidValue;
    if (!encode_2d_f16(&mv, vt, (uint64_t)ctx_pad, (uint64_t)n_head_kv * 128, (uint64_t)ctx_pad, 64, 128)) return cudaErrorInvalidValue;
    AttnTcArgs a{};
    a.page_table = page_table; a.pos0 = pos0_dev; a.out = out; a.T = T; a.n_head = n_head; a.n_pages = n_pages; a.scale = scale;
    switch (gq) {
        case 1: return launch_attn_tc<1>(mq, mk, mv, a, n_head_kv, st);
        case 2: return launch_attn_tc<2>(mq, mk, mv, a, n_head_kv, st);
        case 3: return launch_attn_tc<3, 4>(mq, mk, mv, a, n_head_kv, st);
        case 4: return launch_attn_tc<4>(mq, mk, mv, a, n_head_kv, st);
        case 5: return launch_attn_tc<5, 8>(mq, mk, mv, a, n_head_kv, st);
        case 6: return launch_attn_tc<6, 8>(mq, mk, mv, a, n_head_kv, st);
        case 7: return launch_attn_tc<7, 8>(mq, mk, mv, a, n_head_kv, st);
        case 8: return launch_attn_tc<8>(mq, mk, mv, a, n_head_kv, st);
        default: return cudaErrorInvalidValue;
    }
}

} // namespace blk
