// prefill_kernels.cuh -- the non-GEMM kernels of the multi-token prefill path (verification context fill / prompt
// prefill): RMSNorm -> bf16, RoPE + KV-page write, causal flash attention over the paged f16 KV cache (mma.sync f16),
// SwiGLU, and per-row top-10 + claimed-id gather over vocabulary logits.
// Arithmetic class: bf16 GEMM operands, f16 attention operands, f32 accumulation everywhere (oracle mode ORC_MODE_BF16 for
// the GEMMs); tolerances against the reference's int8 path are stated in tests/test_gpu_prefill.py.
#pragma once
#include <cuda_bf16.h>
#include "tma_ptx.cuh"

#include "decode_kernels.cuh"
#include "prefill.hpp"          // PendingReduce

namespace blk {

// ---- RMSNorm * weight -> bf16 (one CTA per token row) -------------------------------------------------------------------
// The row is read ONCE with 16-byte loads and stays in registers between the two passes (K <= 8192; longer rows re-read it).
__device__ __forceinline__ double rms_sq4(float4 v) {
    return ((double)__fmul_rn(v.x, v.x) + (double)__fmul_rn(v.y, v.y)) + ((double)__fmul_rn(v.z, v.z) + (double)__fmul_rn(v.w, v.w));
}
__device__ __forceinline__ uint2 rms_out4(float4 v, float scale, float4 w) {
    const __nv_bfloat162 p0 = __floats2bfloat162_rn(__fmul_rn(__fmul_rn(v.x, scale), w.x), __fmul_rn(__fmul_rn(v.y, scale), w.y));
    const __nv_bfloat162 p1 = __floats2bfloat162_rn(__fmul_rn(__fmul_rn(v.z, scale), w.z), __fmul_rn(__fmul_rn(v.w, scale), w.w));
    uint2 o; o.x = *reinterpret_cast<const uint32_t*>(&p0); o.y = *reinterpret_cast<const uint32_t*>(&p1);
    return o;
}
template <int NV, bool REDUCE>     // NV: 16-byte words of the row a thread keeps in registers: rows up to NV * 1024 elements are read once
__global__ void __launch_bounds__(256) rmsnorm_bf16_kernel(float* __restrict__ x, const float* __restrict__ w, int K, float eps,
                                                          __nv_bfloat16* __restrict__ y, const float* __restrict__ ws, int S, int m_tiles) {
    // ws != nullptr: the row's pending split-K partial sums (256 x 256 f32 tiles at ws + ((nt * m_tiles + mt) * S + s) * 65536, the layout
    // prefill_gemm_kernel writes) are added first -- splits in order, then the residual, as splitk_reduce_kernel does -- and the new
    // residual row is written back
    pdl_launch_dependents(); pdl_wait();
    const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    float4* x4 = reinterpret_cast<float4*>(x + (size_t)row * K);
    const float4* w4 = reinterpret_cast<const float4*>(w);
    uint2* y2 = reinterpret_cast<uint2*>(y + (size_t)row * K);
    const int n4 = K >> 2;                               // K % 4 == 0 (checked at load: every row length is a multiple of 32)
    const bool in_regs = n4 <= NV * 256;
    __shared__ double red[8];
    __shared__ float s_scale;
    auto fetch = [&](int i) -> float4 {
        float4 v = REDUCE ? x4[i] : __ldg(reinterpret_cast<const float4*>(x4) + i);
        if (REDUCE) {
            const int col = i << 2;
            const float* p = ws + ((size_t)((col >> 8) * m_tiles + (row >> 8)) * S) * 65536 + (size_t)(row & 255) * 256 + (col & 255);
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int s = 0; s < S; s++) { const float4 q = __ldcg(reinterpret_cast<const float4*>(p + (size_t)s * 65536)); o.x += q.x; o.y += q.y; o.z += q.z; o.w += q.w; }
            v = make_float4(o.x + v.x, o.y + v.y, o.z + v.z, o.w + v.w);
            x4[i] = v;
        }
        return v;
    };
    float4 v[NV];
    double sum = 0.0;
    if (in_regs) {
#pragma unroll
        for (int j = 0; j < NV; j++) { const int i = tid + j * 256; if (i < n4) { v[j] = fetch(i); sum += rms_sq4(v[j]); } }
    } else {
        for (int i = tid; i < n4; i += 256) sum += rms_sq4(fetch(i));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) red[wid] = sum;
    __syncthreads();
    if (tid == 0) {
        double tot = 0.0;
        for (int i = 0; i < 8; i++) tot += red[i];
        s_scale = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn((float)(tot / (double)K), eps)));
    }
    __syncthreads();
    const float scale = s_scale;
    if (in_regs) {
#pragma unroll
        for (int j = 0; j < NV; j++) { const int i = tid + j * 256; if (i < n4) y2[i] = rms_out4(v[j], scale, __ldg(w4 + i)); }
    } else {
        for (int i = tid; i < n4; i += 256) y2[i] = rms_out4(x4[i], scale, __ldg(w4 + i));      // (REDUCE: the row was written back above)
    }
}

// pend: a deferred split-K accumulate over x (launch_gemm, SplitKWs::defer); consumed here
__host__ inline void rmsnorm_bf16_launch(float* x, const float* w, int K, float eps, __nv_bfloat16* y, int rows, cudaStream_t st, PendingReduce* pend = nullptr) {
    const float* ws = pend ? pend->ws : nullptr;
    const int S = pend ? pend->S : 0, mt = pend ? pend->m_tiles : 0;
    if (pend) *pend = PendingReduce{};
    if (ws) {
        if (K <= 4096) (void)launch_chain(rmsnorm_bf16_kernel<4, true>, dim3(rows), dim3(256), 0, st, x, w, K, eps, y, ws, S, mt);
        else (void)launch_chain(rmsnorm_bf16_kernel<8, true>, dim3(rows), dim3(256), 0, st, x, w, K, eps, y, ws, S, mt);
    } else {
        if (K <= 4096) (void)launch_chain(rmsnorm_bf16_kernel<4, false>, dim3(rows), dim3(256), 0, st, x, w, K, eps, y, (const float*)nullptr, 0, 0);
        else (void)launch_chain(rmsnorm_bf16_kernel<8, false>, dim3(rows), dim3(256), 0, st, x, w, K, eps, y, (const float*)nullptr, 0, 0);
    }
}

// ---- RoPE on q,k; q -> f16 [T][dq]; k,v -> f16 KV pages (one CTA per token, four elements per thread and step) --------------------
struct QkvPostArgs {
    const float* qkv; long long ld;            // [T][dq + 2*dkv] f32 (bias already added by the GEMM)
    const float2* rope_cs;                     // [T][d_head/2]
    const int32_t* pos0;                       // device scalar: position of token 0
    __half* q_out;                             // [T][dq]
    __half* k_pool; __half* v_pool; const int32_t* page_table;
    int dq, dkv, d_head, neox;
};
__device__ __forceinline__ uint2 pack_h4(float a, float b, float c, float d) {
    const __half2 p0 = __floats2half2_rn(a, b), p1 = __floats2half2_rn(c, d);
    uint2 o; o.x = *reinterpret_cast<const uint32_t*>(&p0); o.y = *reinterpret_cast<const uint32_t*>(&p1);
    return o;
}
// row t of the batch at cache position `pos` of the sequence whose pools / page table are given
__device__ __forceinline__ void qkv_post_row(const QkvPostArgs& a, int t, int pos, __half* k_pool, __half* v_pool, const int32_t* page_table) {
    const int tid = threadIdx.x;
    const float* row = a.qkv + (size_t)t * a.ld;
    const float2* cs = a.rope_cs + (size_t)t * (a.d_head / 2);
    const size_t base = ((size_t)page_table[pos / KV_PAGE] * KV_PAGE + (pos % KV_PAGE)) * a.dkv;
    const int dh = a.d_head, hd = dh >> 1;               // d_head is 64 or 128 (checked at load)
    const int nqk = a.dq + a.dkv;                        // q then k: contiguous in the row, both whole heads
    __half* qdst = a.q_out + (size_t)t * a.dq;
    __half* kdst = k_pool + base;
    if (!a.neox) {
        // NORM pairs (2i, 2i+1): four consecutive elements are two pairs
        for (int e = tid * 4; e < nqk; e += 1024) {
            const float4 x = *reinterpret_cast<const float4*>(row + e);
            const float4 c = *reinterpret_cast<const float4*>(cs + ((e & (dh - 1)) >> 1));      // {cos, sin} of the two pairs
            const float y0 = x.x * c.x - x.y * c.y, y1 = x.x * c.y + x.y * c.x;
            const float y2 = x.z * c.z - x.w * c.w, y3 = x.z * c.w + x.w * c.z;
            *reinterpret_cast<uint2*>(e < a.dq ? qdst + e : kdst + (e - a.dq)) = pack_h4(y0, y1, y2, y3);
        }
    } else {
        // NEOX pairs (i, i + d_head/2) inside a head: four consecutive i
        const int hsh = dh == 128 ? 6 : 5;
        for (int idx = tid * 4; idx < (nqk >> 1); idx += 1024) {
            const int h = idx >> hsh, i = idx & (hd - 1);
            const int r0 = h * dh + i;
            const float4 x0 = *reinterpret_cast<const float4*>(row + r0), x1 = *reinterpret_cast<const float4*>(row + r0 + hd);
            const float4 c01 = *reinterpret_cast<const float4*>(cs + i), c23 = *reinterpret_cast<const float4*>(cs + i + 2);
            const uint2 lo = pack_h4(x0.x * c01.x - x1.x * c01.y, x0.y * c01.z - x1.y * c01.w, x0.z * c23.x - x1.z * c23.y, x0.w * c23.z - x1.w * c23.w);
            const uint2 hi = pack_h4(x0.x * c01.y + x1.x * c01.x, x0.y * c01.w + x1.y * c01.z, x0.z * c23.y + x1.z * c23.x, x0.w * c23.w + x1.w * c23.z);
            __half* dst = r0 < a.dq ? qdst + r0 : kdst + (r0 - a.dq);
            *reinterpret_cast<uint2*>(dst) = lo;
            *reinterpret_cast<uint2*>(dst + hd) = hi;
        }
    }
    for (int e = tid * 4; e < a.dkv; e += 1024) {
        const float4 x = *reinterpret_cast<const float4*>(row + nqk + e);
        *reinterpret_cast<uint2*>(v_pool + base + e) = pack_h4(x.x, x.y, x.z, x.w);
    }
}
__global__ void __launch_bounds__(256) qkv_post_kernel(const QkvPostArgs a) {
    pdl_launch_dependents(); pdl_wait();
    qkv_post_row(a, blockIdx.x, a.pos0[0] + (int)blockIdx.x, a.k_pool, a.v_pool, a.page_table);
}

// ---- causal flash attention over the paged KV cache (mma.sync m16n8k16 f16, f32 accumulate) -------------------------------------
// grid = (ceil(T/64), n_head); block = 128 (4 warps x 16 query rows).  Keys 0 .. pos0+T-1 (the chunk's own K/V are already
// in the cache).  Output bf16 [T][n_head*DH].
struct PrefillAttnArgs {
    const __half* q; const __half* k_pool; const __half* v_pool; const int32_t* page_table; const int32_t* pos0;
    __nv_bfloat16* out;
    int T, n_head, n_head_kv, kv_dim;
    float scale;
};
__device__ __forceinline__ void ldsm_x4(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void mma_f16(float* c, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_f16x2(float a, float b) { __half2 h = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }

template <int DH>
__global__ void __launch_bounds__(128) prefill_attn_kernel(const PrefillAttnArgs a) {
    constexpr int BQ = 64, BKV = 64, LD = DH + 8;        // padded rows: conflict-free ldmatrix
    extern __shared__ __align__(16) unsigned char pa_smem[];
    __half* sQ = reinterpret_cast<__half*>(pa_smem);
    __half* sK = sQ + BQ * LD;
    __half* sV = sK + BKV * LD;
    const int qt = blockIdx.x, h = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int hk = h / (a.n_head / a.n_head_kv);
    const int pos0 = a.pos0[0];
    const int q0 = qt * BQ;
    const int dq = a.n_head * DH;
    // Q tile -> smem
    for (int i = tid; i < BQ * (DH / 8); i += 128) {
        const int r = i / (DH / 8), c = i % (DH / 8);
        uint4 v = make_uint4(0, 0, 0, 0);
        if (q0 + r < a.T) v = *reinterpret_cast<const uint4*>(a.q + (size_t)(q0 + r) * dq + (size_t)h * DH + c * 8);
        *reinterpret_cast<uint4*>(sQ + r * LD + c * 8) = v;
    }
    float o[DH / 8][4];
#pragma unroll
    for (int i = 0; i < DH / 8; i++) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.0f; }
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.0f, 0.0f};
    const int g = lane >> 2, t4 = lane & 3;
    const int qrow0 = q0 + warp * 16 + g;                 // this thread's two query rows: qrow0, qrow0 + 8
    const int kv_end = min(pos0 + a.T, pos0 + q0 + BQ);  // causal: keys up to the last query of the tile
    const float sl2 = a.scale * 1.4426950408889634f;
    for (int k0 = 0; k0 < kv_end; k0 += BKV) {
        __syncthreads();
        for (int i = tid; i < BKV * (DH / 8); i += 128) {
            const int r = i / (DH / 8), c = i % (DH / 8);
            const int key = k0 + r;
            uint4 kv = make_uint4(0, 0, 0, 0), vv = make_uint4(0, 0, 0, 0);
            if (key < kv_end) {
                const size_t off = ((size_t)a.page_table[key / KV_PAGE] * KV_PAGE + (key % KV_PAGE)) * a.kv_dim + (size_t)hk * DH + c * 8;
                kv = *reinterpret_cast<const uint4*>(a.k_pool + off);
                vv = *reinterpret_cast<const uint4*>(a.v_pool + off);
            }
            *reinterpret_cast<uint4*>(sK + r * LD + c * 8) = kv;
            *reinterpret_cast<uint4*>(sV + r * LD + c * 8) = vv;
        }
        __syncthreads();
        // S = Q K^T for this warp's 16 rows x 64 keys
        float s[BKV / 8][4];
#pragma unroll
        for (int i = 0; i < BKV / 8; i++) { s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.0f; }
#pragma unroll
        for (int kk = 0; kk < DH / 16; kk++) {
            uint32_t a0, a1, a2, a3;
            ldsm_x4(a0, a1, a2, a3, sQ + (warp * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * LD + kk * 16 + 8 * (lane >> 4));
#pragma unroll
            for (int nb = 0; nb < BKV / 16; nb++) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4(b0, b1, b2, b3, sK + (nb * 16 + (lane & 7) + 8 * (lane >> 4)) * LD + kk * 16 + 8 * ((lane >> 3) & 1));
                mma_f16(s[2 * nb], a0, a1, a2, a3, b0, b1);
                mma_f16(s[2 * nb + 1], a0, a1, a2, a3, b2, b3);
            }
        }
        // scale, causal mask, online softmax
        float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int i = 0; i < BKV / 8; i++) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int key = k0 + i * 8 + 2 * t4 + (j & 1);
                const int qr = qrow0 + 8 * (j >> 1);
                const bool ok = (key <= pos0 + qr) && (qr < a.T);
                s[i][j] = ok ? s[i][j] * sl2 : -INFINITY;
                mx[j >> 1] = fmaxf(mx[j >> 1], s[i][j]);
            }
        }
        float corr[2];
#pragma unroll
        for (int r = 0; r < 2; r++) {
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
            const float mn = fmaxf(m_run[r], mx[r]);
            corr[r] = (m_run[r] == -INFINITY) ? 0.0f : exp2f(m_run[r] - mn);
            m_run[r] = mn;
        }
        float ls[2] = {0.0f, 0.0f};
        uint32_t pfrag[BKV / 8][2];
#pragma unroll
        for (int i = 0; i < BKV / 8; i++) {
            float p[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                p[j] = (m_run[j >> 1] == -INFINITY) ? 0.0f : exp2f(s[i][j] - m_run[j >> 1]);
                ls[j >> 1] += p[j];
            }
            pfrag[i][0] = pack_f16x2(p[0], p[1]);
            pfrag[i][1] = pack_f16x2(p[2], p[3]);
        }
#pragma unroll
        for (int r = 0; r < 2; r++) {
            ls[r] += __shfl_xor_sync(0xffffffffu, ls[r], 1);
            ls[r] += __shfl_xor_sync(0xffffffffu, ls[r], 2);
            l_run[r] = l_run[r] * corr[r] + ls[r];
        }
#pragma unroll
        for (int i = 0; i < DH / 8; i++) { o[i][0] *= corr[0]; o[i][1] *= corr[0]; o[i][2] *= corr[1]; o[i][3] *= corr[1]; }
        // O += P V
#pragma unroll
        for (int kk = 0; kk < BKV / 16; kk++) {
            const uint32_t a0 = pfrag[2 * kk][0], a1 = pfrag[2 * kk][1], a2 = pfrag[2 * kk + 1][0], a3 = pfrag[2 * kk + 1][1];
#pragma unroll
            for (int nb = 0; nb < DH / 16; nb++) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4_t(b0, b1, b2, b3, sV + (kk * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * LD + nb * 16 + 8 * (lane >> 4));
                mma_f16(o[2 * nb], a0, a1, a2, a3, b0, b1);
                mma_f16(o[2 * nb + 1], a0, a1, a2, a3, b2, b3);
            }
        }
    }
    // normalise and store bf16
#pragma unroll
    for (int r = 0; r < 2; r++) {
        const int qr = qrow0 + 8 * r;
        if (qr >= a.T) continue;
        const float inv = l_run[r] > 0.0f ? 1.0f / l_run[r] : 0.0f;
        __nv_bfloat16* dst = a.out + (size_t)qr * dq + (size_t)h * DH;
#pragma unroll
        for (int i = 0; i < DH / 8; i++) {
            __nv_bfloat162 p = __floats2bfloat162_rn(o[i][2 * r] * inv, o[i][2 * r + 1] * inv);
            *reinterpret_cast<__nv_bfloat162*>(dst + i * 8 + 2 * t4) = p;
        }
    }
}

// ---- the same attention with the query heads of one KV head sharing a CTA -----------------------------------------------------
// grid = (ceil(T / BQ), n_head_kv), block = 256 (8 warps).  BQ = 128 / GQ tokens x GQ query heads = 128 rows per CTA: a K / V tile
// is fetched ONCE for all GQ heads (the per-head kernel above fetches it GQ times), by cp.async into a double buffer so the next
// tile streams in while this one is multiplied.  Heavy (late, causal) query tiles are scheduled first.
__device__ __forceinline__ void pa_cp16(void* smem_dst, const void* g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(g) : "memory");
}
template <int DH, int GQ>
__global__ void __launch_bounds__(256, 2) prefill_attn_gqa_kernel(const PrefillAttnArgs a) {
    constexpr int BQ = 128 / GQ, BKV = 64, LD = DH + 8, MT = BQ / 16;      // MT m16 tiles per head
    extern __shared__ __align__(16) unsigned char pa_smem[];
    __half* sQ = reinterpret_cast<__half*>(pa_smem);                        // [GQ][BQ][LD]
    __half* sKV = sQ + GQ * BQ * LD;                                        // [2 buffers][K | V][BKV][LD]
    const int qt = (int)gridDim.x - 1 - (int)blockIdx.x, hk = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g_h = warp / MT, mt = warp % MT, h = hk * GQ + g_h;
    const int pos0 = a.pos0[0];
    const int q0 = qt * BQ;
    const int dq = a.n_head * DH;
    const int kv_end = min(pos0 + a.T, pos0 + q0 + BQ);                     // causal: keys up to the last query of the tile
    const int n_tiles = (kv_end + BKV - 1) / BKV;
    auto load_tile = [&](int ti, int buf) {
        __half* dK = sKV + (size_t)buf * 2 * BKV * LD; __half* dV = dK + BKV * LD;
        for (int i = tid; i < BKV * (DH / 8); i += 256) {
            const int r = i / (DH / 8), c = i % (DH / 8);
            const int key = min(ti * BKV + r, kv_end - 1);                  // rows past the end repeat the last key (masked below)
            const size_t off = ((size_t)a.page_table[key / KV_PAGE] * KV_PAGE + (key % KV_PAGE)) * a.kv_dim + (size_t)hk * DH + c * 8;
            pa_cp16(dK + r * LD + c * 8, a.k_pool + off);
            pa_cp16(dV + r * LD + c * 8, a.v_pool + off);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    load_tile(0, 0);
    // Q tiles of the GQ heads -> smem
    for (int i = tid; i < GQ * BQ * (DH / 8); i += 256) {
        const int c = i % (DH / 8), r = (i / (DH / 8)) % BQ, gg = i / (BQ * (DH / 8));
        uint4 v = make_uint4(0, 0, 0, 0);
        if (q0 + r < a.T) v = *reinterpret_cast<const uint4*>(a.q + (size_t)(q0 + r) * dq + (size_t)(hk * GQ + gg) * DH + c * 8);
        *reinterpret_cast<uint4*>(sQ + (gg * BQ + r) * LD + c * 8) = v;
    }
    float o[DH / 8][4];
#pragma unroll
    for (int i = 0; i < DH / 8; i++) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.0f; }
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.0f, 0.0f};
    const int g = lane >> 2, t4 = lane & 3;
    const int qrow0 = q0 + mt * 16 + g;                   // this thread's two query tokens: qrow0, qrow0 + 8
    const __half* myQ = sQ + (g_h * BQ + mt * 16) * LD;
    const float sl2 = a.scale * 1.4426950408889634f;
    for (int ti = 0; ti < n_tiles; ti++) {
        const int k0 = ti * BKV, buf = ti & 1;
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                   // tile ti landed for everyone; everyone is done with buffer buf ^ 1
        if (ti + 1 < n_tiles) load_tile(ti + 1, buf ^ 1);
        const __half* sK = sKV + (size_t)buf * 2 * BKV * LD; const __half* sV = sK + BKV * LD;
        if (k0 > pos0 + q0 + mt * 16 + 15) continue;      // every key of this tile is in the future of this warp's rows
        float s[BKV / 8][4];
#pragma unroll
        for (int i = 0; i < BKV / 8; i++) { s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.0f; }
#pragma unroll
        for (int kk = 0; kk < DH / 16; kk++) {
            uint32_t a0, a1, a2, a3;
            ldsm_x4(a0, a1, a2, a3, myQ + ((lane & 7) + 8 * ((lane >> 3) & 1)) * LD + kk * 16 + 8 * (lane >> 4));
#pragma unroll
            for (int nb = 0; nb < BKV / 16; nb++) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4(b0, b1, b2, b3, sK + (nb * 16 + (lane & 7) + 8 * (lane >> 4)) * LD + kk * 16 + 8 * ((lane >> 3) & 1));
                mma_f16(s[2 * nb], a0, a1, a2, a3, b0, b1);
                mma_f16(s[2 * nb + 1], a0, a1, a2, a3, b2, b3);
            }
        }
        float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int i = 0; i < BKV / 8; i++) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int key = k0 + i * 8 + 2 * t4 + (j & 1);
                const int qr = qrow0 + 8 * (j >> 1);
                const bool ok = (key <= pos0 + qr) && (qr < a.T);
                s[i][j] = ok ? s[i][j] * sl2 : -INFINITY;
                mx[j >> 1] = fmaxf(mx[j >> 1], s[i][j]);
            }
        }
        float corr[2];
#pragma unroll
        for (int r = 0; r < 2; r++) {
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
            const float mn = fmaxf(m_run[r], mx[r]);
            corr[r] = (m_run[r] == -INFINITY) ? 0.0f : exp2f(m_run[r] - mn);
            m_run[r] = mn;
        }
        float ls[2] = {0.0f, 0.0f};
        uint32_t pfrag[BKV / 8][2];
#pragma unroll
        for (int i = 0; i < BKV / 8; i++) {
            float pp[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                pp[j] = (m_run[j >> 1] == -INFINITY) ? 0.0f : exp2f(s[i][j] - m_run[j >> 1]);
                ls[j >> 1] += pp[j];
            }
            pfrag[i][0] = pack_f16x2(pp[0], pp[1]);
            pfrag[i][1] = pack_f16x2(pp[2], pp[3]);
        }
#pragma unroll
        for (int r = 0; r < 2; r++) {
            ls[r] += __shfl_xor_sync(0xffffffffu, ls[r], 1);
            ls[r] += __shfl_xor_sync(0xffffffffu, ls[r], 2);
            l_run[r] = l_run[r] * corr[r] + ls[r];
        }
#pragma unroll
        for (int i = 0; i < DH / 8; i++) { o[i][0] *= corr[0]; o[i][1] *= corr[0]; o[i][2] *= corr[1]; o[i][3] *= corr[1]; }
#pragma unroll
        for (int kk = 0; kk < BKV / 16; kk++) {
            const uint32_t a0 = pfrag[2 * kk][0], a1 = pfrag[2 * kk][1], a2 = pfrag[2 * kk + 1][0], a3 = pfrag[2 * kk + 1][1];
#pragma unroll
            for (int nb = 0; nb < DH / 16; nb++) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4_t(b0, b1, b2, b3, sV + (kk * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * LD + nb * 16 + 8 * (lane >> 4));
                mma_f16(o[2 * nb], a0, a1, a2, a3, b0, b1);
                mma_f16(o[2 * nb + 1], a0, a1, a2, a3, b2, b3);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 2; r++) {
        const int qr = qrow0 + 8 * r;
        if (qr >= a.T) continue;
        const float inv = l_run[r] > 0.0f ? 1.0f / l_run[r] : 0.0f;
        __nv_bfloat16* dst = a.out + (size_t)qr * dq + (size_t)h * DH;
#pragma unroll
        for (int i = 0; i < DH / 8; i++) {
            __nv_bfloat162 pr = __floats2bfloat162_rn(o[i][2 * r] * inv, o[i][2 * r + 1] * inv);
            *reinterpret_cast<__nv_bfloat162*>(dst + i * 8 + 2 * t4) = pr;
        }
    }
}
template <int DH, int GQ> constexpr int prefill_attn_gqa_smem() { return (128 * (DH + 8) + 2 * 2 * 64 * (DH + 8)) * 2; }

// ---- per-row top-10 + gather at claimed ids over a chunk of vocabulary logits (one CTA per row) --------------------------------
// Session::getLogitsFromCtx(10) / getLogitsFromCtx(TokenDataVector) for every position of the verification fill.
struct RowTopkArgs {
    const float* logits; long long ld; int n_vocab; int row0;      // logits of rows row0 .. row0+gridDim.x-1
    const int32_t* claimed; const int32_t* n_claimed;              // [n][10], [n]  (indexed by absolute row)
    float* gathered;                                               // [n][10]
    int32_t* top_ids; float* top_logits;                           // [n][10]
};
// Threshold selection, two streaming passes over the row (the full-row bitonic sort this replaces cost 470 us per 256 rows):
//   pass 1: every thread keeps the maximum of its share; tau = the 10th largest of the 256 thread maxima is a lower bound of the
//           10th largest logit (ten distinct elements are >= tau);
//   pass 2: the few elements >= tau are appended to a shared list, which is sorted (logit descending, ties by lower id, so the
//           result does not depend on the append order).  A degenerate row (> 1024 survivors, e.g. constant logits) falls back
//           to per-thread insertion + a block-wide sort.
__global__ void __launch_bounds__(256) row_topk_gather_kernel(const RowTopkArgs a) {
    const int rl = blockIdx.x, row = a.row0 + rl, tid = threadIdx.x;
    const float* lg = a.logits + (size_t)rl * a.ld;
    if (a.claimed && tid < 10) {
        float v = 0.0f;
        if (tid < a.n_claimed[row]) { const int id = a.claimed[(size_t)row * 10 + tid]; v = (id >= 0 && id < a.n_vocab) ? lg[id] : -INFINITY; }
        a.gathered[(size_t)row * 10 + tid] = v;
    }
    if (!a.top_ids) return;
    __shared__ float key[4096];
    __shared__ int idx[4096];
    __shared__ unsigned int s_cnt;
    const bool vec = (a.ld % 4 == 0) && (a.n_vocab % 4 == 0);
    const int n4 = vec ? a.n_vocab >> 2 : 0;
    // pass 1
    float m = -INFINITY;
    if (vec) {
        const float4* lg4 = reinterpret_cast<const float4*>(lg);
        for (int i = tid; i < n4; i += 256) { const float4 v = lg4[i]; m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w))); }
    } else {
        for (int i = tid; i < a.n_vocab; i += 256) m = fmaxf(m, lg[i]);
    }
    key[tid] = m; idx[tid] = tid;
    if (tid == 0) s_cnt = 0u;
    __syncthreads();
    bitonic_sort_desc_n<256>(key, idx, 256);
    const float tau = key[9];
    __syncthreads();
    // pass 2
    constexpr unsigned int CAP = 1024;
    auto push = [&](float v, int i) {
        if (v >= tau) { const unsigned int s = atomicAdd(&s_cnt, 1u); if (s < CAP) { key[s] = v; idx[s] = i; } }
    };
    if (vec) {
        const float4* lg4 = reinterpret_cast<const float4*>(lg);
        for (int i = tid; i < n4; i += 256) { const float4 v = lg4[i]; push(v.x, 4 * i); push(v.y, 4 * i + 1); push(v.z, 4 * i + 2); push(v.w, 4 * i + 3); }
    } else {
        for (int i = tid; i < a.n_vocab; i += 256) push(lg[i], i);
    }
    __syncthreads();
    const unsigned int total = s_cnt;
    if (total <= CAP) {
        int n2 = 16;
        while (n2 < (int)total) n2 <<= 1;
        for (int i = (int)total + tid; i < n2; i += 256) { key[i] = -INFINITY; idx[i] = 0x7fffffff; }
        __syncthreads();
        bitonic_sort_desc_n<256>(key, idx, n2);
    } else {
        // thread-local top-10 by insertion, then a block-wide merge through shared memory
        __syncthreads();
        float bl[10]; int bi[10];
#pragma unroll
        for (int i = 0; i < 10; i++) { bl[i] = -INFINITY; bi[i] = 0x7fffffff; }
        for (int i = tid; i < a.n_vocab; i += 256) {
            const float v = lg[i];
            if (td_before(v, i, bl[9], bi[9])) {
                bl[9] = v; bi[9] = i;
#pragma unroll
                for (int j = 9; j > 0; j--) {
                    if (td_before(bl[j], bi[j], bl[j - 1], bi[j - 1])) { const float tv = bl[j]; bl[j] = bl[j - 1]; bl[j - 1] = tv; const int ti = bi[j]; bi[j] = bi[j - 1]; bi[j - 1] = ti; }
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 10; i++) { key[tid * 10 + i] = bl[i]; idx[tid * 10 + i] = bi[i]; }
        for (int i = 2560 + tid; i < 4096; i += 256) { key[i] = -INFINITY; idx[i] = 0x7fffffff; }
        __syncthreads();
        bitonic_sort_desc_n<256>(key, idx, 4096);
    }
    if (tid < 10) { a.top_ids[(size_t)row * 10 + tid] = idx[tid]; a.top_logits[(size_t)row * 10 + tid] = key[tid]; }
}

// per-chunk maxima of a logits row (feeds topk_select_kernel when the row was not produced by the decode lm_head mat-vec)
// blockIdx.y = row of a batch (rows ld floats apart, 256 chunk maxima per row)
__global__ void __launch_bounds__(256) chunk_max_kernel(const float* __restrict__ logits, int n, int chunk_shift, int* chunk_max, long long ld = 0) {
    logits += (size_t)blockIdx.y * (size_t)ld; chunk_max += blockIdx.y * 256;
    const int c = blockIdx.x, begin = c << chunk_shift, end = min(n, begin + (1 << chunk_shift));
    float m = -INFINITY;
    for (int i = begin + threadIdx.x; i < end; i += 256) m = fmaxf(m, logits[i]);
    m = warp_max(m);
    __shared__ float red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) { for (int i = 1; i < 8; i++) m = fmaxf(m, red[i]); chunk_max[c] = float_order_key(m); }
}

} // namespace blk
