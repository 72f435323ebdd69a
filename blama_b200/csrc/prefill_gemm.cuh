// prefill_gemm.cuh -- dequant-fused tcgen05 / TMEM GEMM for multi-token prefill (the /verify_completion context fill,
// reference Session::fillCtx, Session.cpp:231-244, done as ONE causal prefill instead of N single-token decodes).
//
//   C[T][N] (f32) (+)= X[T][K] (bf16) . W[N][K]^T      W = device-resident quant blocks (Q4_K / Q5_K / Q6_K / Q8_0 / F32)
//
// Per CTA tile: 256 tokens x 256 weight rows, K walked in steps of 64.
//   warp 8  (1 thread)  : TMA producer -- two 128x64 bf16 boxes of X per stage (cp.async.bulk.tensor, SWIZZLE_128B)
//   warps 0-7 (256 thr) : dequant producers -- thread r turns 64 K-elements of weight row n0+r into bf16 and writes them
//                         as one 128-byte row of the canonical K-major SWIZZLE_128B tile the UMMA descriptor describes
//                         (weights are dequantised once per 256 tokens and never touch HBM in bf16)
//   warp 9  (1 thread)  : MMA issuer -- tcgen05.mma.cta_group::1.kind::f16, M=128, N=256, K=16; two accumulators
//                         (token rows 0-127 / 128-255) x 256 f32 columns = all 512 TMEM columns
//   warps 4-7 double as the epilogue after the main loop of a tile: tcgen05.ld 32x32b -> registers -> global
// Operands are bf16 (weights: bf16(dequantised f32), activations: bf16), accumulation is f32 in TMEM: this is the
// ORC_MODE_BF16 arithmetic of the oracle; tolerance against the reference's int8 path is stated in the tests.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "gemv_kernels.cuh"   // QMat
#include "tma_ptx.cuh"        // mbarrier / bulk-copy wrappers

namespace blk {

constexpr int PG_BM = 256, PG_BN = 256, PG_BK = 64;
constexpr int PG_STAGES = 3;                              // full tiles: three 64 KB stages (A 32 KB + B 32 KB)
constexpr int PG_STAGES_FEW = 4;                          // batches of at most 128 tokens (one M half): four 48 KB stages (A 16 KB + B 32 KB) in the
                                                          // same 192 KB -- a third more weight bytes in flight per SM, which is what bounds a few-token GEMM
constexpr int PG_PRODUCER_THREADS = 256;
constexpr int PG_THREADS = PG_PRODUCER_THREADS + 64;      // + TMA warp + MMA warp
constexpr int PG_A_BYTES = PG_BM * PG_BK * 2;             // 32 KB (two 128-row boxes)
constexpr int PG_B_BYTES = PG_BN * PG_BK * 2;             // 32 KB
constexpr int PG_STAGE_BYTES = PG_A_BYTES + PG_B_BYTES;
constexpr int PG_SMEM_BYTES = PG_STAGES * PG_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;

enum : int { PG_STORE = 0, PG_ACCUM = 1, PG_SWIGLU = 2 };
// pseudo weight type of the two-pass form: the weights were dequantised once into a bf16 "panel" [rows][K] in global memory
// (panel_dequant_kernel) and the B tile is fetched by TMA like the activations; no dequantisation inside the GEMM
constexpr int QT_PANEL = 100;

// Up to three weight matrices share one launch (q | k | v, or gate | up): more tiles per launch = less wave-quantisation
// loss on 148 SMs.  Segment s covers output columns [col0, col0 + W.N); its tiles are 256 rows of W (the last may be
// partial).  PG_SWIGLU: seg[0] = gate, seg[1] = up; a tile holds 128 gate rows + the 128 matching up rows and the epilogue
// writes h = silu(g) * u as bf16.
struct PgSeg { QMat W; const float* bias; int col0; int tile0; };
struct PrefillGemmArgs {
    PgSeg seg[3];
    int nseg;
    float* C; long long ldc;    // f32 output (PG_STORE / PG_ACCUM), row stride in elements
    __nv_bfloat16* H; long long ldh;   // bf16 output (PG_SWIGLU)
    int T, K;
    int n_tiles;                // total column tiles over all segments
    int mode;
    int panel_up_row0;          // QT_PANEL + PG_SWIGLU: panel row of ffn_up row 0 (ffn_gate starts at panel row 0)
    // QT_PANEL: the bf16 weights as TILE IMAGES -- block (rb, kb) = rows 128 rb .. +127, columns 64 kb .. +63 is 16 KB at
    // panel + (rb * K / 64 + kb) * 16384 bytes, laid out exactly as the K-major SWIZZLE_128B shared-memory tile (row r at
    // (r >> 3) * 1024 + (r & 7) * 128, 16-byte chunk c at position c ^ (r & 7)): one contiguous cp.async.bulk per half tile instead of a
    // 2-D tensor-map box of 128 pieces of 128 bytes at an 8-16 KB stride (which touched 128 DRAM pages for 16 KB)
    const unsigned char* panel;
    // deterministic split-K of the LAST, partial wave of tiles (and of every tile when the batch has fewer tiles than SMs): tiles
    // [0, n_whole) are computed whole; each tile t >= n_whole becomes k_splits work items, item (t, s) stores its partial sums as a
    // 256 x 256 f32 tile at ws + ((t - n_whole) * k_splits + s) * 65536 and splitk_reduce_kernel adds the partials in split order and
    // applies the epilogue (bias / accumulate / SwiGLU).  k_splits == 1: off.
    int n_whole, k_splits;
    float* ws;
};

// ---- PTX wrappers ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem desc] . B[smem desc]^T, bf16 x bf16 -> f32
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// kind::f16 covers f16 and bf16 inputs; the instruction descriptor says which
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    tc_mma_bf16(tmem_d, desc_a, desc_b, idesc, accumulate);
}
__device__ __forceinline__ void tc_ld_32x32b_x32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major SWIZZLE_128B shared-memory descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO(=1)<<16 | SBO(1024 B >>4)<<32 |
// version(1)<<46 | layout SWIZZLE_128B(2)<<61
__device__ __forceinline__ uint64_t umma_desc_sw128(const void* smem) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_u32(smem) >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (1) @4, a/b format BF16 (1) @7/@10, K-major both,
// n_dim = N>>3 @17, m_dim = M>>4 @24
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- 64 consecutive K-elements of one weight row, dequantised (f32) -----------------------------------------------------
// kb = index of the 64-element block inside the row.  Same float expressions as ggml's dequantize_row_* (no FMA).
__device__ __forceinline__ void dequant_k64(const QMat& W, int64_t row, int kb, float* out) {
    if (W.type == QT_Q4_K) { dequant_unit_q4k(W, row, kb, out); return; }
    if (W.type == QT_Q5_K) { dequant_unit_q5k(W, row, kb, out); return; }
    if (W.type == QT_Q8_0) { dequant_unit_q80(W, row, 2 * kb, out); dequant_unit_q80(W, row, 2 * kb + 1, out + 32); return; }
    if (W.type == QT_Q6_K) {
        const int s = kb >> 2, hh = (kb >> 1) & 1, hi = kb & 1;           // quarters (2*hi, 2*hi+1) of half hh
        const uint8_t* ql = W.p0 + (size_t)row * (W.K >> 1) + (size_t)s * 128 + hh * 64;
        const uint8_t* qh = W.p1 + (size_t)row * (W.K >> 2) + (size_t)s * 64 + hh * 32;
        const int8_t* sc = reinterpret_cast<const int8_t*>(W.p2) + (size_t)row * (W.K >> 4) + s * 16 + hh * 8 + hi * 4;
        const float d = __half2float(reinterpret_cast<const __half*>(W.p3)[(size_t)row * (W.K >> 8) + s]);
#pragma unroll
        for (int l = 0; l < 32; l++) {
            const uint8_t a = ql[l], b = ql[l + 32], h = qh[l];
            const int qa = (int)(((hi ? (a >> 4) : (a & 0xF))) | (((h >> (4 * hi)) & 3) << 4)) - 32;
            const int qb = (int)(((hi ? (b >> 4) : (b & 0xF))) | (((h >> (4 * hi + 2)) & 3) << 4)) - 32;
            out[l] = d * (float)sc[l >> 4] * (float)qa;
            out[32 + l] = d * (float)sc[2 + (l >> 4)] * (float)qb;
        }
        return;
    }
    if (W.type == QT_F32) {
        const float* src = reinterpret_cast<const float*>(W.p0) + (size_t)row * W.K + (size_t)kb * 64;
#pragma unroll
        for (int i = 0; i < 64; i++) out[i] = src[i];
        return;
    }
    const __half* src = reinterpret_cast<const __half*>(W.p0) + (size_t)row * W.K + (size_t)kb * 64;
#pragma unroll
    for (int i = 0; i < 64; i++) out[i] = __half2float(src[i]);
}

// ---- optimised producers: raw 64-element slices held in registers (loaded one stage ahead), expanded to bf16 ----------
// byte -> float without I2F: PRMT drops the byte into the mantissa of 2^23 (0x4B000000), one FADD removes the bias
__device__ __forceinline__ float byte_to_float(uint32_t word, int i) {      // (float) byte i of word
    const uint32_t m = __byte_perm(word, 0x4B000000u, 0x7650 + i);          // {byte i, 0x00, 0x00, 0x4B}
    return __uint_as_float(m) - 8388608.0f;
}
__device__ __forceinline__ float byte_to_float_off(uint32_t word, int i, float off) {      // (float) byte i of word + 2^23 - off
    const uint32_t m = __byte_perm(word, 0x4B000000u, 0x7650 + i);
    return __uint_as_float(m) - off;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&p);
}
// store 8 consecutive K-elements (one 16 B chunk c of the 128 B row) into the SWIZZLE_128B tile
__device__ __forceinline__ void store_chunk(unsigned char* srow, int r, int c, const float* v) {
    uint4 o;
    o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]); o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(srow + ((c ^ (r & 7)) << 4)) = o;
}

template <int TYPE> struct RawK64;
template <> struct RawK64<QT_Q4_K> {
    uint4 q0, q1, hdr;
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int kb) {
        const uint8_t* q = W.p0 + (size_t)row * (W.K >> 1) + (size_t)kb * 32;
        q0 = ldg_stream(q); q1 = ldg_stream(q + 16);
        hdr = __ldg(reinterpret_cast<const uint4*>(W.p1 + ((size_t)row * (W.K >> 8) + (kb >> 2)) * 16));
    }
    __device__ __forceinline__ void expand(unsigned char* srow, int r, int kb) const {
        uint32_t sc2, mn2; k4_scale_min_pair(hdr, kb & 3, sc2, mn2);
        const float2 dm = hdr_d_dmin(hdr);
        const float d1 = dm.x * (float)(sc2 & 0xFF), m1 = dm.y * (float)(mn2 & 0xFF);
        const float d2 = dm.x * (float)(sc2 >> 8), m2 = dm.y * (float)(mn2 >> 8);
        const uint32_t w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
        for (int c = 0; c < 4; c++) {           // chunk c: low nibbles of bytes 8c..8c+7; chunk c+4: their high nibbles
            float lo[8], hi[8];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint32_t wl = w[2 * c + h] & 0x0F0F0F0Fu, wh = (w[2 * c + h] >> 4) & 0x0F0F0F0Fu;
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    lo[4 * h + i] = __fmaf_rn(d1, byte_to_float(wl, i), -m1);
                    hi[4 * h + i] = __fmaf_rn(d2, byte_to_float(wh, i), -m2);
                }
            }
            store_chunk(srow, r, c, lo);
            store_chunk(srow, r, c + 4, hi);
        }
    }
};
template <> struct RawK64<QT_Q5_K> {
    uint4 q0, q1, hdr, h0, h1;
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int kb) {
        const uint8_t* q = W.p0 + (size_t)row * (W.K >> 1) + (size_t)kb * 32;
        q0 = ldg_stream(q); q1 = ldg_stream(q + 16);
        const size_t sb = (size_t)row * (W.K >> 8) + (kb >> 2);
        hdr = __ldg(reinterpret_cast<const uint4*>(W.p1 + sb * 16));
        h0 = __ldg(reinterpret_cast<const uint4*>(W.p2 + sb * 32));
        h1 = __ldg(reinterpret_cast<const uint4*>(W.p2 + sb * 32 + 16));
    }
    __device__ __forceinline__ void expand(unsigned char* srow, int r, int kb) const {
        const int j = kb & 3;
        uint32_t sc2, mn2; k4_scale_min_pair(hdr, j, sc2, mn2);
        const float2 dm = hdr_d_dmin(hdr);
        const float d1 = dm.x * (float)(sc2 & 0xFF), m1 = dm.y * (float)(mn2 & 0xFF);
        const float d2 = dm.x * (float)(sc2 >> 8), m2 = dm.y * (float)(mn2 >> 8);
        const uint32_t w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
        const uint32_t hb[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
        for (int c = 0; c < 4; c++) {
            float lo[8], hi[8];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint32_t hw = hb[2 * c + h];
                const uint32_t wl = (w[2 * c + h] & 0x0F0F0F0Fu) | (((hw >> (2 * j)) & 0x01010101u) << 4);
                const uint32_t wh = ((w[2 * c + h] >> 4) & 0x0F0F0F0Fu) | (((hw >> (2 * j + 1)) & 0x01010101u) << 4);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    lo[4 * h + i] = __fmaf_rn(d1, byte_to_float(wl, i), -m1);
                    hi[4 * h + i] = __fmaf_rn(d2, byte_to_float(wh, i), -m2);
                }
            }
            store_chunk(srow, r, c, lo);
            store_chunk(srow, r, c + 4, hi);
        }
    }
};
template <> struct RawK64<QT_Q6_K> {
    uint4 l0, l1, l2, l3, h0, h1; uint32_t sc4; uint16_t dh;      // 64 B of ql, 32 B of qh, 4 scales, d
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int kb) {
        const int s = kb >> 2, hh = (kb >> 1) & 1, hi = kb & 1;
        const uint8_t* ql = W.p0 + (size_t)row * (W.K >> 1) + (size_t)s * 128 + hh * 64;
        l0 = ldg_stream(ql); l1 = ldg_stream(ql + 16); l2 = ldg_stream(ql + 32); l3 = ldg_stream(ql + 48);
        const uint8_t* qh = W.p1 + (size_t)row * (W.K >> 2) + (size_t)s * 64 + hh * 32;
        h0 = ldg_stream(qh); h1 = ldg_stream(qh + 16);
        sc4 = __ldg(reinterpret_cast<const uint32_t*>(W.p2 + (size_t)row * (W.K >> 4) + s * 16 + hh * 8 + hi * 4));
        dh = __ldg(reinterpret_cast<const uint16_t*>(W.p3) + (size_t)row * (W.K >> 8) + s);
    }
    __device__ __forceinline__ void expand(unsigned char* srow, int r, int kb) const {
        if (kb & 1) expand_half<1>(srow, r); else expand_half<0>(srow, r);      // compile-time nibble / bit selection
    }
    template <int HI>
    __device__ __forceinline__ void expand_half(unsigned char* srow, int r) const {
        const float d = __half2float(__ushort_as_half(dh));
        float dsc[4];
#pragma unroll
        for (int i = 0; i < 4; i++) dsc[i] = d * (float)(int)(int8_t)((sc4 >> (8 * i)) & 0xFF);
        const uint32_t la[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};      // ql[0..31]
        const uint32_t lb[8] = {l2.x, l2.y, l2.z, l2.w, l3.x, l3.y, l3.z, l3.w};      // ql[32..63]
        const uint32_t hq[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};      // qh[0..31]
        // elements 0..31: quarter 2*HI (ql[l], qh bits 4*HI..), elements 32..63: quarter 2*HI+1 (ql[32+l], qh bits 4*HI+2..)
#pragma unroll
        for (int c = 0; c < 4; c++) {
            float qa[8], qb[8];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int wi = 2 * c + h;
                const uint32_t na = HI ? ((la[wi] >> 4) & 0x0F0F0F0Fu) : (la[wi] & 0x0F0F0F0Fu);
                const uint32_t nb = HI ? ((lb[wi] >> 4) & 0x0F0F0F0Fu) : (lb[wi] & 0x0F0F0F0Fu);
                const uint32_t ha = HI ? (hq[wi] & 0x30303030u) : ((hq[wi] << 4) & 0x30303030u);
                const uint32_t hbq = HI ? ((hq[wi] >> 2) & 0x30303030u) : ((hq[wi] << 2) & 0x30303030u);
                const uint32_t wa = na | ha, wb = nb | hbq;
                const float sa = dsc[wi >> 2], sb = dsc[2 + (wi >> 2)];      // 16 elements per scale
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    qa[4 * h + i] = sa * byte_to_float_off(wa, i, 8388640.0f);      // (2^23 + q) - (2^23 + 32) = q - 32, exact
                    qb[4 * h + i] = sb * byte_to_float_off(wb, i, 8388640.0f);
                }
            }
            store_chunk(srow, r, c, qa);
            store_chunk(srow, r, c + 4, qb);
        }
    }
};
template <> struct RawK64<QT_Q8_0> {
    uint4 q0, q1, q2, q3; uint32_t d2;
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int kb) {
        const uint8_t* q = W.p0 + (size_t)row * W.K + (size_t)kb * 64;
        q0 = ldg_stream(q); q1 = ldg_stream(q + 16); q2 = ldg_stream(q + 32); q3 = ldg_stream(q + 48);
        d2 = __ldg(reinterpret_cast<const uint32_t*>(W.p1 + ((size_t)row * (W.K >> 5) + 2 * kb) * 2));
    }
    __device__ __forceinline__ void expand(unsigned char* srow, int r, int) const {
        const float2 d = __half22float2(*reinterpret_cast<const __half2*>(&d2));
        const uint32_t w[16] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w, q3.x, q3.y, q3.z, q3.w};
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const float dd = c < 4 ? d.x : d.y;
            float v[8];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint32_t u = w[2 * c + h] ^ 0x80808080u;          // int8 -> biased uint8
#pragma unroll
                for (int i = 0; i < 4; i++) v[4 * h + i] = byte_to_float_off(u, i, 8388736.0f) * dd;      // biased byte - 128
            }
            store_chunk(srow, r, c, v);
        }
    }
};
// generic (test-only formats F32 / F16): plain loads at expand time
template <int TYPE> struct RawK64 {
    const QMat* W; int64_t row;
    __device__ __forceinline__ void load(const QMat& w, int64_t r, int) { W = &w; row = r; }
    __device__ __forceinline__ void expand(unsigned char* srow, int r, int kb) const {
        float v[64];
        dequant_k64(*W, row, kb, v);
#pragma unroll
        for (int c = 0; c < 8; c++) store_chunk(srow, r, c, v + 8 * c);
    }
};

// work item -> (tile, K split, K-block range); `part`: the item stores partial sums to the workspace
struct PgItem { int tile, split, kb0, kb1; bool part; };
__device__ __forceinline__ PgItem pg_item(int item, int n_whole, int n_split, int k_per, int k_blocks_all) {
    PgItem w;
    if (item < n_whole || n_split <= 1) { w.tile = item; w.split = 0; w.kb0 = 0; w.kb1 = k_blocks_all; w.part = false; }
    else {
        const int r = item - n_whole;
        w.tile = n_whole + r / n_split; w.split = r - (w.tile - n_whole) * n_split;
        w.kb0 = w.split * k_per; w.kb1 = min(k_blocks_all, w.kb0 + k_per); w.part = true;
    }
    return w;
}

template <int TA, int TB>
__global__ void __launch_bounds__(PG_THREADS, 1) prefill_gemm_kernel(const __grid_constant__ CUtensorMap tmap_x, const PrefillGemmArgs a) {
    constexpr bool PANEL = (TA == QT_PANEL);
    // The tiles need 1024-byte alignment (SWIZZLE_128B atoms).  The dynamic shared memory of a kernel without static shared memory
    // starts 1024-aligned on this part; it is checked, not assumed, and NOT re-aligned through an integer cast -- that hides the
    // address space from the compiler, and every shared-memory access of the producers became a generic ST.E / LD.E.
    extern __shared__ __align__(1024) unsigned char pg_smem_raw[];
    unsigned char* smem = pg_smem_raw;
    if (threadIdx.x == 0 && (smem_u32(pg_smem_raw) & 1023u)) __trap();
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PG_STAGES * PG_STAGE_BYTES);
    uint64_t* full = bars;                          // [n_st]  TMA bytes + 8 producer-warp arrivals
    uint64_t* empty = bars + PG_STAGES_FEW;         // [n_st]  tcgen05.commit
    uint64_t* tmem_full = bars + 2 * PG_STAGES_FEW;     // accumulators complete
    uint64_t* tmem_empty = bars + 2 * PG_STAGES_FEW + 1;    // epilogue drained them (8 warps)
    uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2 * PG_STAGES_FEW + 2);
    // stage geometry: kernel-uniform (few = every tile has one M half only)
    const bool few = a.T <= 128;
    const int n_st = few ? PG_STAGES_FEW : PG_STAGES;
    const int a_bytes = few ? PG_A_BYTES / 2 : PG_A_BYTES;
    const int st_bytes = a_bytes + PG_B_BYTES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < PG_STAGES_FEW; s++) { mbar_init(full + s, PANEL ? 1 : 1 + PG_PRODUCER_THREADS / 32); mbar_init(empty + s, 1); }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 8);
        mbar_fence_init();
    }
    if (warp == 9) {    // one warp allocates all 512 TMEM columns (two 128 x 256 f32 accumulators)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_base_slot;
    // the prologue above touched no global memory: from here on the kernel reads what the previous kernel of the stream wrote
    pdl_launch_dependents(); pdl_wait();

    const int m_tiles = (a.T + PG_BM - 1) / PG_BM, n_tiles = a.n_tiles;
    const int k_blocks_all = a.K / PG_BK;
    const int n_split = a.k_splits, n_whole = a.k_splits > 1 ? a.n_whole : m_tiles * n_tiles;
    const int k_per = (k_blocks_all + n_split - 1) / n_split;      // K blocks per split (the last split may be shorter)
    const int total_tiles = n_whole + (m_tiles * n_tiles - n_whole) * n_split;     // work items (pg_item)

    if (warp == 8) {
        // ===================== TMA producer (activations) =====================
        if (lane == 0) {
            int s = 0; uint32_t ph = 0;                        // stage and its phase
            for (int wi = 0;; wi++) {
                const int item = (int)blockIdx.x + wi * (int)gridDim.x;
                if (item >= total_tiles) break;
                const PgItem w = pg_item(item, n_whole, n_split, k_per, k_blocks_all);
                const int tile = w.tile, kb0 = w.kb0, kb1 = w.kb1;
                const int m0 = (tile % m_tiles) * PG_BM, nt = tile / m_tiles;
                // panel rows of the two 128-row halves of the B tile
                const int w0 = a.mode == PG_SWIGLU ? nt * 128 : nt * PG_BN;
                const int w1 = a.mode == PG_SWIGLU ? a.panel_up_row0 + nt * 128 : nt * PG_BN + 128;
                const bool two = m0 + 128 < a.T;                   // token rows 128-255 of the tile exist (few-token batches: one M half only)
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(empty + s, ph ^ 1);
                    unsigned char* sa = smem + s * st_bytes;
                    mbar_expect_tx(full + s, (PANEL ? PG_A_BYTES + PG_B_BYTES : PG_A_BYTES) - (two ? 0 : PG_A_BYTES / 2));
                    tma_load_2d(sa, &tmap_x, kb * PG_BK, m0, full + s);
                    if (two) tma_load_2d(sa + PG_A_BYTES / 2, &tmap_x, kb * PG_BK, m0 + 128, full + s);
                    if (PANEL) {
                        bulk_g2s(sa + a_bytes, a.panel + (((size_t)(w0 >> 7) * k_blocks_all + kb) << 14), PG_B_BYTES / 2, full + s);
                        bulk_g2s(sa + a_bytes + PG_B_BYTES / 2, a.panel + (((size_t)(w1 >> 7) * k_blocks_all + kb) << 14), PG_B_BYTES / 2, full + s);
                    }
                    if (++s == n_st) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 9) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(128, PG_BN);
            int s = 0; uint32_t ph = 0;
            for (int tile_i = 0;; tile_i++) {
                const int item = (int)blockIdx.x + tile_i * (int)gridDim.x;
                if (item >= total_tiles) break;
                const PgItem w = pg_item(item, n_whole, n_split, k_per, k_blocks_all);
                const int kb0 = w.kb0, kb1 = w.kb1;
                const bool two = (w.tile % m_tiles) * PG_BM + 128 < a.T;      // the second accumulator's token rows exist
                mbar_wait(tmem_empty, (tile_i & 1) ^ 1);          // epilogue of the previous tile has drained TMEM
                tc_fence_after();
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(full + s, ph);
                    tc_fence_after();
                    unsigned char* sa = smem + s * st_bytes;
                    unsigned char* sb = sa + a_bytes;
                    const uint64_t da0 = umma_desc_sw128(sa), da1 = umma_desc_sw128(sa + PG_A_BYTES / 2), db = umma_desc_sw128(sb);
#pragma unroll
                    for (int k = 0; k < PG_BK / 16; k++) {
                        const uint64_t koff = (uint64_t)((k * 32) >> 4);       // 16 bf16 = 32 B along K inside the swizzle atom
                        const uint32_t acc = (kb > kb0 || k > 0) ? 1u : 0u;
                        tc_mma_bf16(tmem_base, da0 + koff, db + koff, idesc, acc);
                        if (two) tc_mma_bf16(tmem_base + PG_BN, da1 + koff, db + koff, idesc, acc);
                    }
                    tc_commit(empty + s);                         // frees the stage when these MMAs have read it
                    if (++s == n_st) { s = 0; ph ^= 1; }
                }
                tc_commit(tmem_full);                             // accumulators of this tile are final
            }
        }
    } else {
        // ===================== dequant producers (warps 0-7); warps 4-7 also run the epilogue =====================
        const int r = threadIdx.x;                                // B-tile row handled by this thread
        int s = 0; uint32_t ph = 0;
        for (int tile_i = 0;; tile_i++) {
            const int item = (int)blockIdx.x + tile_i * (int)gridDim.x;
            if (item >= total_tiles) break;
            const PgItem w = pg_item(item, n_whole, n_split, k_per, k_blocks_all);
            const int tile = w.tile, kb0 = w.kb0, kb1 = w.kb1;
            const int m0 = (tile % m_tiles) * PG_BM, nt = tile / m_tiles;
            // which matrix / row this thread dequantises, and where the tile's columns land in the output
            int si = 0;
            if (a.mode != PG_SWIGLU) {
                if (a.nseg > 1 && nt >= a.seg[1].tile0) si = 1;
                if (a.nseg > 2 && nt >= a.seg[2].tile0) si = 2;
            } else {
                si = r >> 7;                                      // rows 0-127: gate, 128-255: up
            }
            const PgSeg& Sg = a.seg[si];
            const int n_local0 = (a.mode == PG_SWIGLU) ? nt * 128 : (nt - Sg.tile0) * PG_BN;
            const int64_t row = (a.mode == PG_SWIGLU) ? (int64_t)n_local0 + (r & 127) : (int64_t)n_local0 + r;
            const bool row_ok = row < Sg.W.N;
            auto produce = [&](auto raw_tag) {
                using Raw = decltype(raw_tag);
                constexpr bool DEEP = sizeof(Raw) <= 64;           // small raw slices (Q4_K): three in flight; large ones: two
                Raw cur, nxt, nx2;
                if (row_ok) { cur.load(Sg.W, row, kb0); if (DEEP && kb0 + 1 < kb1) nxt.load(Sg.W, row, kb0 + 1); }
                for (int kb = kb0; kb < kb1; kb++) {
                    if (DEEP) { if (row_ok && kb + 2 < kb1) nx2.load(Sg.W, row, kb + 2); }      // loads fly while the current slice is expanded
                    else { if (row_ok && kb + 1 < kb1) nxt.load(Sg.W, row, kb + 1); }
                    mbar_wait(empty + s, ph ^ 1);
                    unsigned char* srow = smem + s * st_bytes + a_bytes + (r >> 3) * 1024 + (r & 7) * 128;
                    if (row_ok) cur.expand(srow, r, kb);
                    else {
#pragma unroll
                        for (int c = 0; c < 8; c++) *reinterpret_cast<uint4*>(srow + (c << 4)) = make_uint4(0, 0, 0, 0);
                    }
                    fence_proxy_async();                           // generic-proxy stores -> visible to the tensor core (async proxy)
                    __syncwarp();
                    if (lane == 0) mbar_arrive(full + s);
                    cur = nxt;
                    if (DEEP) nxt = nx2;
                    if (++s == n_st) { s = 0; ph ^= 1; }
                }
            };
            if constexpr (!PANEL) { if (TA != TB && si == 2) produce(RawK64<TB>{}); else produce(RawK64<TA>{}); }
            else { (void)produce; (void)row_ok; }
            {
                // ---- epilogue: warp q = warp % 4 owns TMEM lanes 32q .. 32q+31; warps 0-3 drain the first accumulator
                //      (token rows 0-127), warps 4-7 the second (rows 128-255) ----
                const int q = warp & 3;
                mbar_wait(tmem_full, tile_i & 1);
                tc_fence_after();
                // tile-level segment (the producer's `si` is per thread in SwiGLU mode)
                int ts = 0;
                if (a.mode != PG_SWIGLU) {
                    if (a.nseg > 1 && nt >= a.seg[1].tile0) ts = 1;
                    if (a.nseg > 2 && nt >= a.seg[2].tile0) ts = 2;
                }
                const PgSeg& Ts = a.seg[ts];
                const int tn0 = (a.mode == PG_SWIGLU) ? nt * 128 : (nt - Ts.tile0) * PG_BN;     // first row of W in this tile
                const int n_valid = Ts.W.N - tn0;                                                 // columns of the tile that exist
                {
                    const int h = warp >> 2;
                    const int trow = m0 + h * 128 + q * 32 + lane;
                    const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(h * PG_BN);
                    if (m0 + h * 128 >= a.T) {
                        // this accumulator's token rows do not exist (few-token batch): nothing was accumulated, nothing to drain
                    } else if (w.part) {
                        // a K split: the raw partial sums of the tile go to the workspace (row-major 256 x 256), nothing else
                        float* wt = a.ws + ((size_t)(tile - n_whole) * n_split + w.split) * (size_t)(PG_BM * PG_BN) + (size_t)(h * 128 + q * 32 + lane) * PG_BN;
#pragma unroll 1
                        for (int cc = 0; cc < PG_BN / 32; cc++) {
                            uint32_t v[32];
                            tc_ld_32x32b_x32(tbase + cc * 32, v);
                            tc_wait_ld();
                            if (trow < a.T) {
#pragma unroll
                                for (int j = 0; j < 32; j += 4)
                                    *reinterpret_cast<float4*>(wt + cc * 32 + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                            }
                        }
                    } else if (a.mode == PG_SWIGLU) {
#pragma unroll 1
                        for (int cc = 0; cc < 4; cc++) {
                            uint32_t g[32], u[32];
                            tc_ld_32x32b_x32(tbase + cc * 32, g);
                            tc_ld_32x32b_x32(tbase + 128 + cc * 32, u);
                            tc_wait_ld();
                            if (trow < a.T) {
                                __nv_bfloat16* dst = a.H + (size_t)trow * a.ldh + tn0 + cc * 32;
#pragma unroll
                                for (int j = 0; j < 32; j += 8) {
                                    if (cc * 32 + j + 7 < n_valid) {
                                        uint4 o;
                                        uint32_t* op = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
                                        for (int e = 0; e < 4; e++) {
                                            const float g0 = __uint_as_float(g[j + 2 * e]), g1 = __uint_as_float(g[j + 2 * e + 1]);
                                            op[e] = pack_bf16x2(__fdividef(g0, 1.0f + __expf(-g0)) * __uint_as_float(u[j + 2 * e]),
                                                                __fdividef(g1, 1.0f + __expf(-g1)) * __uint_as_float(u[j + 2 * e + 1]));
                                        }
                                        *reinterpret_cast<uint4*>(dst + j) = o;
                                    } else {
                                        for (int e = 0; e < 8; e++) if (cc * 32 + j + e < n_valid) {
                                            const float gg = __uint_as_float(g[j + e]);
                                            dst[j + e] = __float2bfloat16_rn((gg / (1.0f + expf(-gg))) * __uint_as_float(u[j + e]));
                                        }
                                    }
                                }
                            }
                        }
                    } else {
                    // PG_ACCUM: the residual values of column chunk cc + 1 are requested before chunk cc is drained (one exposed L2
                    // round trip per tile instead of eight)
                    float4 cres[8];
                    auto fetch_res = [&](int cc) {
                        if (a.mode == PG_ACCUM && trow < a.T) {
                            const float* src = a.C + (size_t)trow * a.ldc + Ts.col0 + tn0 + cc * 32;
#pragma unroll
                            for (int j = 0; j < 32; j += 4) if (cc * 32 + j + 3 < n_valid) cres[j >> 2] = *reinterpret_cast<const float4*>(src + j);
                        }
                    };
                    fetch_res(0);
#pragma unroll 1
                    for (int cc = 0; cc < PG_BN / 32; cc++) {
                        uint32_t v[32];
                        tc_ld_32x32b_x32(tbase + cc * 32, v);
                        float4 ccur[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) ccur[j] = cres[j];
                        if (cc + 1 < PG_BN / 32) fetch_res(cc + 1);
                        tc_wait_ld();
                        if (trow < a.T && cc * 32 < n_valid) {
                            float* dst = a.C + (size_t)trow * a.ldc + Ts.col0 + tn0 + cc * 32;
                            const float* bias = Ts.bias ? Ts.bias + tn0 + cc * 32 : nullptr;
                            const int mode = a.mode;
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                if (cc * 32 + j + 3 < n_valid) {
                                    float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                                    if (mode == PG_ACCUM) { const float4 c0 = ccur[j >> 2]; o.x += c0.x; o.y += c0.y; o.z += c0.z; o.w += c0.w; }
                                    else if (bias) { o.x += bias[j]; o.y += bias[j + 1]; o.z += bias[j + 2]; o.w += bias[j + 3]; }
                                    *reinterpret_cast<float4*>(dst + j) = o;
                                } else {
                                    for (int jj = 0; jj < 4; jj++) if (cc * 32 + j + jj < n_valid) {
                                        float o = __uint_as_float(v[j + jj]);
                                        if (mode == PG_ACCUM) o += dst[j + jj]; else if (bias) o += bias[j + jj];
                                        dst[j + jj] = o;
                                    }
                                }
                            }
                        }
                    }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tmem_empty);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 9) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// ---- second step of a split-K GEMM: the split tiles' partial sums are added in split order, then the tile's epilogue runs --------
// grid = (split tiles, 32): block (i, y) finishes rows 8 y .. 8 y + 7 of tile n_whole + i
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const PrefillGemmArgs a) {
    pdl_launch_dependents(); pdl_wait();
    const int m_tiles = (a.T + PG_BM - 1) / PG_BM;
    const int tile = a.n_whole + blockIdx.x, S = a.k_splits;
    const int m0 = (tile % m_tiles) * PG_BM, nt = tile / m_tiles;
    const float* wt = a.ws + (size_t)blockIdx.x * S * (size_t)(PG_BM * PG_BN);
    int ts = 0;
    if (a.mode != PG_SWIGLU) {
        if (a.nseg > 1 && nt >= a.seg[1].tile0) ts = 1;
        if (a.nseg > 2 && nt >= a.seg[2].tile0) ts = 2;
    }
    const PgSeg& Ts = a.seg[ts];
    const int tn0 = (a.mode == PG_SWIGLU) ? nt * 128 : (nt - Ts.tile0) * PG_BN;
    const int n_valid = Ts.W.N - tn0;
    const int ncol4 = a.mode == PG_SWIGLU ? 32 : 64;          // float4 columns of the output per row
    for (int idx = threadIdx.x; idx < 8 * ncol4; idx += 256) {
        const int r = blockIdx.y * 8 + idx / ncol4, c = (idx % ncol4) * 4;
        const int trow = m0 + r;
        if (trow >= a.T || c >= n_valid) continue;
        auto sum4 = [&](int col) {
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int s = 0; s < S; s++) {
                const float4 p = __ldcg(reinterpret_cast<const float4*>(wt + (size_t)s * (PG_BM * PG_BN) + (size_t)r * PG_BN + col));
                o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w;
            }
            return o;
        };
        if (a.mode == PG_SWIGLU) {
            const float4 g = sum4(c), u = sum4(128 + c);
            uint2 o;
            o.x = pack_bf16x2(__fdividef(g.x, 1.0f + __expf(-g.x)) * u.x, __fdividef(g.y, 1.0f + __expf(-g.y)) * u.y);
            o.y = pack_bf16x2(__fdividef(g.z, 1.0f + __expf(-g.z)) * u.z, __fdividef(g.w, 1.0f + __expf(-g.w)) * u.w);
            *reinterpret_cast<uint2*>(a.H + (size_t)trow * a.ldh + tn0 + c) = o;
        } else {
            float4 o = sum4(c);
            float* dst = a.C + (size_t)trow * a.ldc + Ts.col0 + tn0 + c;
            if (a.mode == PG_ACCUM) { const float4 c0 = *reinterpret_cast<const float4*>(dst); o.x += c0.x; o.y += c0.y; o.z += c0.z; o.w += c0.w; }
            else if (Ts.bias) { const float* b = Ts.bias + tn0 + c; o.x += b[0]; o.y += b[1]; o.z += b[2]; o.w += b[3]; }
            *reinterpret_cast<float4*>(dst) = o;
        }
    }
}

// ---- one weight matrix -> bf16 tile images of the panel (PrefillGemmArgs::panel): the same values the fused producers write into
// shared memory (bf16 of ggml's dequantised f32), in the same swizzled tile layout.  One thread expands one 64-element slice of a
// row (128 bytes); consecutive threads take consecutive rows of the same (row block, K block), so a warp writes 4 KB contiguous.
// row0 = panel row of W's row 0 (a multiple of 128) -------------------------------------------------------------------------------
template <int TYPE>
__global__ void __launch_bounds__(256) panel_dequant_kernel(const QMat W, unsigned char* __restrict__ panel, long long row0) {
    const int kbs = W.K >> 6;
    const int64_t n_rb = (W.N + 127) >> 7;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_rb * kbs * 128) return;
    const int r = (int)(idx & 127);
    const int64_t bk = idx >> 7;
    const int64_t rb = bk / kbs; const int kb = (int)(bk - rb * kbs);
    const int64_t row = rb * 128 + r;
    if (row >= W.N) return;
    RawK64<TYPE> raw;
    raw.load(W, row, kb);
    unsigned char* dst = panel + ((((size_t)(row0 >> 7) + (size_t)rb) * kbs + kb) << 14) + (r >> 3) * 1024 + (r & 7) * 128;
    raw.expand(dst, r, kb);
}

} // namespace blk
