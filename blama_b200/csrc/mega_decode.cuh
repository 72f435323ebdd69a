// mega_decode.cuh -- the whole batch-1 decode step (Session::getToken -> llama_decode(1 token), reference
// inference/code/llama/Session.cpp:169-190, 395-401) as ONE persistent cooperative kernel.
//
// Why: a decode step of an 8B model is ~290 dependent operations of 2-20 us each.  As separate kernels (even with
// PDL + CUDA graph) every boundary drains the memory system; measured 34 % of the HBM roofline.  Here one CTA per SM
// stays resident for the whole token and HBM never stops streaming:
//
//   * weights live in a second, "stream" copy laid out at load time as [pair][K-slice][row a | row b] chunks: the bytes one
//     warp needs for one row slice are contiguous (2-4 KB).  Q4_K / Q5_K chunks are ggml's own blocks (144 / 176 B are
//     16 B multiples); Q6_K / Q8_0 are re-tiled to 208 B / 272 B super-blocks.
//   * every warp owns a private 3-slot shared-memory ring that its lane 0 keeps full with cp.async.bulk (TMA 1-D) copies,
//     completion on an mbarrier.  The chunk sequence of a warp is a pure function of (cta, warp): it never depends on
//     activations, so the ring runs AHEAD across phase boundaries and across the grid barriers: while the CTAs
//     synchronise and re-quantise activations, the next phase's weights are already landing.
//   * one lane owns one HALF super-block (128 weights) of a row slice; the 128 int8 activations it needs are the same for
//     every row of the phase, so they sit in 32 registers (loaded once per phase) -- the inner loop reads only weights
//     from shared memory: ~0.5 instructions per weight for Q4_K.
//   * phases of a layer: QKV (+bias, RoPE, KV-page write) | attention scores | softmax + V.p (+ split combine by the
//     last CTA of each KV head) | Wo (+residual) | gate/up (SwiGLU) | down (+residual); then final norm + lm_head.
//     Phases are separated by a grid barrier (one atomic + spin per CTA); activations are exchanged through L2
//     (ld.global.cg) and re-quantised redundantly by every CTA in the prologue of the phase that consumes them.
//
// Arithmetic contract: identical to the per-kernel path (decode_kernels.cuh): activations quantised exactly as ggml's
// quantize_row_q8_K / q8_0, integer dot products bit-identical to ggml_vec_dot_*, attention in ggml's order
// (max -> expf -> sum in double -> p * (1/sum) -> f16 -> V.p).  Only the order of fp32 additions differs.
#pragma once
#include "gemv_kernels.cuh"
#include "tma_ptx.cuh"       // mbarrier / bulk-copy PTX wrappers
#include "mega_decode.hpp"

namespace blk {

// ---- small PTX helpers ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int dp4a_us(uint32_t a_u8, int b_s8, int c) {
    int d; asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_u8), "r"(b_s8), "r"(c)); return d;
}
__device__ __forceinline__ uint4 lds128(const void* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
    unsigned int v; asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ int sext8(uint32_t w, int k) { return (int)(w << (24 - 8 * k)) >> 24; }

__device__ __forceinline__ unsigned int ld_relaxed_u32(const unsigned int* p) {
    unsigned int v; asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void red_release_add(unsigned int* p, unsigned int v) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- LL exchange: every value that crosses CTAs travels with an epoch tag in ONE 8-byte store; readers poll the data itself.
// Measured on B200 (tools/micro/lat.cu): store -> visible -> read = ~900 cycles, against ~3500 for grid barrier + read.
// No fences: an 8-byte store is single-copy atomic, so a reader sees {value, tag} of the same store or an older one.
__device__ __forceinline__ uint32_t mg_tag(uint32_t seq, int phi, int sub) { return seq * 4096u + (uint32_t)(phi + 1) * 4u + (uint32_t)sub; }
__device__ __forceinline__ uint2 ll_ld(const uint2* p) {
    uint2 v; asm volatile("ld.relaxed.gpu.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ uint4 ll_ld2(const uint2* p) {      // two consecutive {value, tag} words
    uint4 v; asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void ll_st(uint2* p, float v, uint32_t tag) {
    asm volatile("st.relaxed.gpu.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(__float_as_uint(v)), "r"(tag) : "memory");
}
__device__ __forceinline__ void ll_st2(uint2* p, float v0, float v1, uint32_t tag) {
    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(__float_as_uint(v0)), "r"(tag), "r"(__float_as_uint(v1)), "r"(tag) : "memory");
}
constexpr int MG_SPIN_LIMIT = 1 << 20;       // a few 100 ms of polling: a phase that never arrives sets *P.err instead of hanging the GPU
struct MgV8F { uint4 a, b, c, d; };          // 8 x {value, tag}
__device__ __forceinline__ MgV8F ll_ld8(const uint2* p) { MgV8F r; r.a = ll_ld2(p); r.b = ll_ld2(p + 2); r.c = ll_ld2(p + 4); r.d = ll_ld2(p + 6); return r; }
__device__ __forceinline__ bool ll_ok8(const MgV8F& r, uint32_t tag) {
    return r.a.y == tag && r.a.w == tag && r.b.y == tag && r.b.w == tag && r.c.y == tag && r.c.w == tag && r.d.y == tag && r.d.w == tag;
}

// activations of one lane: the 128 int8 values of its half super-block plus their scales / partial sums
struct LaneAct {
    int q[32];
    float d0;            // Q8_K: the block scale
    uint32_t aux[6];     // Q8_K: [0..3] 8 x int16 sums of 16 consecutive activations, [4..5] 4 x int16 sums of 32
                         // Q8_0: [0..3] the four 32-element block scales (float bits)
};

// ---- per-type dot product of one half super-block (weights in wb, loaded from the ring) ---------------------------------
__device__ __forceinline__ float mg_dot_q4k(const uint4* wb, int hf, const LaneAct& A) {
    const uint4 hdr = wb[0];
    uint32_t sc4, mn4;
    if (hf == 0) { sc4 = hdr.y & 0x3F3F3F3Fu; mn4 = hdr.z & 0x3F3F3F3Fu; }
    else { sc4 = (hdr.w & 0x0F0F0F0Fu) | ((hdr.y >> 2) & 0x30303030u); mn4 = ((hdr.w >> 4) & 0x0F0F0F0Fu) | ((hdr.z >> 2) & 0x30303030u); }
    const uint32_t* qw = reinterpret_cast<const uint32_t*>(wb + 1);
    int i0 = 0, i1 = 0, i2 = 0, i3 = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        i0 = __dp4a((int)(qw[i] & 0x0F0F0F0Fu), A.q[i], i0);
        i1 = dp4a_us(qw[i] & 0xF0F0F0F0u, A.q[8 + i], i1);            // 16 x the high-nibble sum (exact)
        i2 = __dp4a((int)(qw[8 + i] & 0x0F0F0F0Fu), A.q[16 + i], i2);
        i3 = dp4a_us(qw[8 + i] & 0xF0F0F0F0u, A.q[24 + i], i3);
    }
    i1 >>= 4; i3 >>= 4;
    const int p = (int)(sc4 & 0xff) * i0 + (int)((sc4 >> 8) & 0xff) * i1 + (int)((sc4 >> 16) & 0xff) * i2 + (int)(sc4 >> 24) * i3;
    int pm = __dp2a_lo((int)A.aux[4], (int)mn4, 0);
    pm = __dp2a_hi((int)A.aux[5], (int)mn4, pm);
    const float2 dm = __half22float2(*reinterpret_cast<const __half2*>(&hdr.x));
    return (dm.x * A.d0) * (float)p - (dm.y * A.d0) * (float)pm;
}

__device__ __forceinline__ float mg_dot_q5k(const uint4* wb, int hf, const LaneAct& A) {
    const uint4 hdr = wb[0];
    uint32_t sc4, mn4;
    if (hf == 0) { sc4 = hdr.y & 0x3F3F3F3Fu; mn4 = hdr.z & 0x3F3F3F3Fu; }
    else { sc4 = (hdr.w & 0x0F0F0F0Fu) | ((hdr.y >> 2) & 0x30303030u); mn4 = ((hdr.w >> 4) & 0x0F0F0F0Fu) | ((hdr.z >> 2) & 0x30303030u); }
    const uint32_t* hw = reinterpret_cast<const uint32_t*>(wb + 1);      // 8 words: high bits of elements l = 4i..4i+3
    const uint32_t* qw = reinterpret_cast<const uint32_t*>(wb + 3);
    const uint32_t M = 0x0F0F0F0Fu, B = 0x01010101u;
    const int j0 = 4 * hf;                                              // bit of the first 32-element sub-block of this half
    int i0 = 0, i1 = 0, i2 = 0, i3 = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint32_t h = hw[i] >> j0;
        i0 = __dp4a((int)((qw[i] & M) | ((h & B) << 4)), A.q[i], i0);
        i1 = __dp4a((int)(((qw[i] >> 4) & M) | (((h >> 1) & B) << 4)), A.q[8 + i], i1);
        i2 = __dp4a((int)((qw[8 + i] & M) | (((h >> 2) & B) << 4)), A.q[16 + i], i2);
        i3 = __dp4a((int)(((qw[8 + i] >> 4) & M) | (((h >> 3) & B) << 4)), A.q[24 + i], i3);
    }
    const int p = (int)(sc4 & 0xff) * i0 + (int)((sc4 >> 8) & 0xff) * i1 + (int)((sc4 >> 16) & 0xff) * i2 + (int)(sc4 >> 24) * i3;
    int pm = __dp2a_lo((int)A.aux[4], (int)mn4, 0);
    pm = __dp2a_hi((int)A.aux[5], (int)mn4, pm);
    const float2 dm = __half22float2(*reinterpret_cast<const __half2*>(&hdr.x));
    return (dm.x * A.d0) * (float)p - (dm.y * A.d0) * (float)pm;
}

// Q6_K half: ql words l0[i] = wb[0..1], l1[i] = wb[2..3] (elements l and l + 32), qh words wb[4..5], scales wb[6].xy, d wb[6].z
__device__ __forceinline__ float mg_dot_q6k(const uint4* wb, const LaneAct& A) {
    const uint32_t* l0 = reinterpret_cast<const uint32_t*>(wb);
    const uint32_t* l1 = reinterpret_cast<const uint32_t*>(wb + 2);
    const uint32_t* hw = reinterpret_cast<const uint32_t*>(wb + 4);
    const uint32_t M = 0x0F0F0F0Fu, H = 0x30303030u;
    int is[8];
#pragma unroll
    for (int k = 0; k < 8; k++) is[k] = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int t = i >> 2;
        const uint32_t h = hw[i];
        is[0 + t] = __dp4a((int)((l0[i] & M) | ((h << 4) & H)), A.q[i], is[0 + t]);
        is[2 + t] = __dp4a((int)((l1[i] & M) | ((h << 2) & H)), A.q[8 + i], is[2 + t]);
        is[4 + t] = __dp4a((int)(((l0[i] >> 4) & M) | (h & H)), A.q[16 + i], is[4 + t]);
        is[6 + t] = __dp4a((int)(((l1[i] >> 4) & M) | ((h >> 2) & H)), A.q[24 + i], is[6 + t]);
    }
    const uint32_t sx = wb[6].x, sy = wb[6].y;
    int p = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) { p += sext8(sx, k) * is[k]; p += sext8(sy, k) * is[4 + k]; }
    // sum (q - 32) a = sum q a - 32 sum a, with the 16-element activation sums
    int t = __dp2a_lo((int)A.aux[0], (int)sx, 0);
    t = __dp2a_hi((int)A.aux[1], (int)sx, t);
    t = __dp2a_lo((int)A.aux[2], (int)sy, t);
    t = __dp2a_hi((int)A.aux[3], (int)sy, t);
    p -= 32 * t;
    const float d = __half2float(__ushort_as_half((unsigned short)(wb[6].z & 0xffff)));
    return (d * A.d0) * (float)p;
}

// Q8_0 half super-block = four 32-element blocks: int8 weights wb[0..7], f16 scales wb[8].xy
__device__ __forceinline__ float mg_dot_q80(const uint4* wb, const LaneAct& A) {
    const int* qw = reinterpret_cast<const int*>(wb);
    const __half2 d01 = *reinterpret_cast<const __half2*>(&wb[8].x), d23 = *reinterpret_cast<const __half2*>(&wb[8].y);
    const float dw[4] = {__low2float(d01), __high2float(d01), __low2float(d23), __high2float(d23)};
    float v = 0.0f;
#pragma unroll
    for (int b = 0; b < 4; b++) {
        int s = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) s = __dp4a(qw[8 * b + j], A.q[8 * b + j], s);
        v += (float)s * (dw[b] * __uint_as_float(A.aux[b]));
    }
    return v;
}

// ---- activation quantisation of one 256-element block by one warp (8 values per lane, in registers), into the swizzled
// shared-memory layout.  Same arithmetic as quantize_256_warp (gemv_kernels.cuh).  The int8 values of half super-block hs
// live at sq + hs*128, 16-byte chunk c stored at chunk position c ^ (hs & 7): the per-lane register loads (stride 128 B
// between lanes) are then bank-conflict free.
__device__ __noinline__ void mg_quantize_regs(float4 va, float4 vb, int fmt, int b, int8_t* sq, float* sd, int16_t* sbs) {
    const int lane = threadIdx.x & 31;
    const float v[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
    int qi[8];
    if (fmt == ACT_Q8_K) {
        // max |x| of the block, then the FIRST element attaining it decides the sign of the scale (quantize_row_q8_K_ref)
        float amax = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; i++) amax = fmaxf(amax, fabsf(v[i]));
        amax = warp_max(amax);
        float mine = 0.0f; bool has = false;
#pragma unroll
        for (int i = 7; i >= 0; i--) if (fabsf(v[i]) == amax) { mine = v[i]; has = true; }      // lowest i wins
        const unsigned int who = __ballot_sync(0xffffffffu, has);
        const float mx = __shfl_sync(0xffffffffu, mine, who ? __ffs(who) - 1 : 0);
        if (amax == 0.0f) {
#pragma unroll
            for (int i = 0; i < 8; i++) qi[i] = 0;
            if (lane == 0) sd[b] = 0.0f;
        } else {
            const float iscale = __fdiv_rn(-127.0f, mx);
#pragma unroll
            for (int i = 0; i < 8; i++) qi[i] = min(127, __float2int_rn(__fmul_rn(iscale, v[i])));
            if (lane == 0) sd[b] = __fdiv_rn(1.0f, iscale);
        }
        int s = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) s += qi[i];
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        if ((lane & 1) == 0) sbs[b * 16 + (lane >> 1)] = (int16_t)s;
    } else {   // ACT_Q8_0
        float amax = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; i++) amax = fmaxf(amax, fabsf(v[i]));
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
        const float d = __fdiv_rn(amax, 127.0f);
        const float id = d != 0.0f ? __fdiv_rn(1.0f, d) : 0.0f;
#pragma unroll
        for (int i = 0; i < 8; i++) qi[i] = (int)roundf(__fmul_rn(v[i], id));
        if ((lane & 3) == 0) sd[b * 8 + (lane >> 2)] = __half2float(__float2half_rn(d));
    }
    uint2 pk;
    pk.x = (uint32_t)(qi[0] & 0xff) | ((uint32_t)(qi[1] & 0xff) << 8) | ((uint32_t)(qi[2] & 0xff) << 16) | ((uint32_t)(qi[3] & 0xff) << 24);
    pk.y = (uint32_t)(qi[4] & 0xff) | ((uint32_t)(qi[5] & 0xff) << 8) | ((uint32_t)(qi[6] & 0xff) << 16) | ((uint32_t)(qi[7] & 0xff) << 24);
    const int hs = 2 * b + (lane >> 4), c = (lane >> 1) & 7;
    *reinterpret_cast<uint2*>(sq + hs * 128 + ((c ^ (hs & 7)) << 4) + (lane & 1) * 8) = pk;
}
struct MgV8 { float4 a, b; };
__device__ __forceinline__ MgV8 mg_load8(const float* p) {
    MgV8 r; r.a = __ldcg(reinterpret_cast<const float4*>(p)); r.b = __ldcg(reinterpret_cast<const float4*>(p) + 1); return r;
}

// ---- stream cursor: the chunk sequence of one warp over the whole token ---------------------------------------------
// Used once per (model, device) by mg_chunk_list_kernel to write every warp's chunk descriptors {address, bytes} to global
// memory; the decode kernel's producer then just walks its list (one 16 B load per 2-4 KB chunk).
struct MgCursor {
    int ph, s, k, c;          // phase, segment, item (row pair), chunk of the item
    int n;                    // items of this warp's group in the current segment
    int cpp;                  // chunks per item (1 if the chunk holds both rows, else 2)
    uint32_t bytes;           // bytes per chunk
    const uint8_t* addr0;     // chunk (item 0, 0)
    size_t item_stride;
};

// group bookkeeping of a warp in a phase
struct MgGroup { int W, L, rpc, NG, NGtot, gg, ws; bool active; };
__device__ __forceinline__ MgGroup mg_group(const MegaPhase* ph, int n_cta, int cta, int warp) {
    MgGroup g;
    g.W = ph->W; g.L = ph->L; g.rpc = ph->rpc;
    g.NG = MG_WARPS / g.W; g.NGtot = n_cta * g.NG;
    g.active = warp < g.NG * g.W;
    g.gg = cta * g.NG + warp / g.W;
    g.ws = warp % g.W;
    return g;
}
__device__ __forceinline__ void mg_seg_items(const MgGroup& g, const MegaSeg* sg, int& vg, int& n) {
    vg = (g.gg + sg->rot) % g.NGtot;
    n = (g.active && vg < sg->n_pairs) ? (sg->n_pairs - 1 - vg) / g.NGtot + 1 : 0;
}
__device__ inline void mg_cursor_load(MgCursor& cu, const MegaPhase* phases, int n_cta, int cta, int warp) {
    const MegaPhase* ph = phases + cu.ph;
    const MgGroup g = mg_group(ph, n_cta, cta, warp);
    const MegaSeg* sg = ph->seg + cu.s;
    int vg; mg_seg_items(g, sg, vg, cu.n);
    cu.cpp = 2 / g.rpc;
    cu.bytes = (uint32_t)(sg->slice_bytes * g.rpc);
    cu.addr0 = sg->base + ((size_t)vg * g.W + g.ws) * 2 * (size_t)sg->slice_bytes;
    cu.item_stride = (size_t)g.NGtot * g.W * 2 * (size_t)sg->slice_bytes;
    cu.k = 0; cu.c = 0;
}
// move to the first chunk at or after (ph, s) that exists; returns false at the end of the token
__device__ inline bool mg_cursor_seek(MgCursor& cu, const MegaPhase* phases, int n_phases, int n_cta, int cta, int warp) {
    while (cu.ph < n_phases) {
        if (cu.s < phases[cu.ph].nseg) {
            mg_cursor_load(cu, phases, n_cta, cta, warp);
            if (cu.n > 0) return true;
            cu.s++;
        } else { cu.ph++; cu.s = 0; }
    }
    return false;
}
__device__ inline bool mg_cursor_next(MgCursor& cu, const MegaPhase* phases, int n_phases, int n_cta, int cta, int warp) {
    if (++cu.c < cu.cpp) return true;
    cu.c = 0;
    if (++cu.k < cu.n) return true;
    cu.s++;
    return mg_cursor_seek(cu, phases, n_phases, n_cta, cta, warp);
}

// one thread per (cta, warp): list == nullptr -> only count; else write descriptors {addr.lo, addr.hi, bytes, 0}
__global__ void mg_chunk_list_kernel(const MegaPhase* phases, int n_phases, int n_cta, uint4* list, int list_stride, int* counts) {
    const int id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= n_cta * MG_WARPS) return;
    const int cta = id / MG_WARPS, warp = id % MG_WARPS;
    MgCursor cu; cu.ph = 0; cu.s = 0; cu.k = 0; cu.c = 0; cu.n = 0; cu.cpp = 1; cu.bytes = 0; cu.addr0 = nullptr; cu.item_stride = 0;
    bool more = mg_cursor_seek(cu, phases, n_phases, n_cta, cta, warp);
    int n = 0;
    while (more) {
        if (list) {
            const unsigned long long a = (unsigned long long)(cu.addr0 + (size_t)cu.k * cu.item_stride + (size_t)cu.c * cu.bytes);
            list[(size_t)id * list_stride + n] = make_uint4((uint32_t)a, (uint32_t)(a >> 32), cu.bytes, 0u);
        }
        n++;
        more = mg_cursor_next(cu, phases, n_phases, n_cta, cta, warp);
    }
    counts[id] = n;
}

// ---- shared memory carve-up ------------------------------------------------------------------------------------------
struct MgSmem {
    uint64_t* bars; MegaPhase* ph; __half** kp; __half** vp; float2* part; float2* rope; double* redd; float* stat; int* misc;
    unsigned char* act;        // quantised activations of the running phase
    unsigned char* attn;       // attention tiles (behind the activations of an n_embd-long row, so they can be filled early)
};
__device__ __forceinline__ MgSmem mg_carve(const MegaParams& P, unsigned char* smem) {
    MgSmem s;
    unsigned char* sp = smem + (size_t)MG_WARPS * MG_SLOTS * P.slot_bytes;
    s.bars = reinterpret_cast<uint64_t*>(sp); sp += MG_WARPS * MG_SLOTS * 8;
    s.ph = reinterpret_cast<MegaPhase*>(sp); sp += 2 * sizeof(MegaPhase);
    s.kp = reinterpret_cast<__half**>(sp); sp += (size_t)P.n_layer * sizeof(__half*);
    s.vp = reinterpret_cast<__half**>(sp); sp += (size_t)P.n_layer * sizeof(__half*);
    s.part = reinterpret_cast<float2*>(sp); sp += (size_t)P.max_items * MG_WARPS * sizeof(float2);
    s.rope = reinterpret_cast<float2*>(sp); sp += (size_t)(P.d_head / 2) * sizeof(float2);
    s.redd = reinterpret_cast<double*>(sp); sp += 8 * MG_WARPS * sizeof(double);
    s.stat = reinterpret_cast<float*>(sp); sp += 32 * sizeof(float);
    s.misc = reinterpret_cast<int*>(sp); sp += 32 * sizeof(int);
    s.act = sp;
    s.attn = sp + P.attn_off;
    return s;
}

// ---- optional event trace: thread 0 of every CTA appends (SM clock << 8 | tag); see tools/mega_trace.py --------------------
template <bool TR>
__device__ __forceinline__ void mg_tr(const MegaParams& P, const MgSmem& S, int tag) {
    if (TR && threadIdx.x == 0) {
        const int i = S.misc[16]++;
        long long t;
        if (P.trace_global) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); else t = clock64();     // ns, common to all SMs | SM clock
        if (i < P.trace_cap) P.trace[(size_t)blockIdx.x * P.trace_cap + i] = (t << 8) | (long long)tag;
    }
}

// ---- step 0: embedding row -> x (rows spread over the CTAs) -------------------------------------------------------------
__device__ __noinline__ void mg_embed(const MegaParams& P) {
    const int tid = threadIdx.x;
    const int tok = P.tok[0];
    const uint32_t tag = P.seq * 4096u;               // epoch of the embedding row
    const int per = (P.n_embd / 64 + P.n_cta - 1) / P.n_cta;      // 64-element units per CTA
    const int u0 = (int)blockIdx.x * per, u1 = min(P.n_embd / 64, u0 + per);
    const QMat& E = P.tok_embd;
    if (E.type == QT_Q4_K || E.type == QT_Q5_K || E.type == QT_Q6_K) {
        for (int u = u0 + tid; u < u1; u += MG_THREADS) {
            float v[64];
            if (E.type == QT_Q4_K) dequant_unit_q4k(E, tok, u, v); else if (E.type == QT_Q5_K) dequant_unit_q5k(E, tok, u, v); else dequant_unit_q6k(E, tok, u, v);
            if (E.type == QT_Q6_K) { for (int l = 0; l < 64; l++) ll_st(P.x2 + q6k_unit_elem(u, l), v[l], tag); }
            else { for (int l = 0; l < 64; l++) ll_st(P.x2 + u * 64 + l, v[l], tag); }
        }
    } else if (E.type == QT_Q8_0) {
        for (int u = 2 * u0 + tid; u < 2 * u1; u += MG_THREADS) { float v[32]; dequant_unit_q80(E, tok, u, v); for (int l = 0; l < 32; l++) ll_st(P.x2 + u * 32 + l, v[l], tag); }
    } else if (E.type == QT_F32) {
        const float* src = reinterpret_cast<const float*>(E.p0) + (size_t)tok * E.K;
        for (int i = u0 * 64 + tid; i < u1 * 64; i += MG_THREADS) ll_st(P.x2 + i, src[i], tag);
    } else {
        const __half* src = reinterpret_cast<const __half*>(E.p0) + (size_t)tok * E.K;
        for (int i = u0 * 64 + tid; i < u1 * 64; i += MG_THREADS) ll_st(P.x2 + i, __half2float(src[i]), tag);
    }
}

// a poll that never completes: record it (mapped host word) and carry on with whatever is there -- never hang the GPU
__device__ __noinline__ void mg_poll_timeout(const MegaParams& P, const MgSmem& S, int where) {
    if (P.err && !S.misc[20]) *reinterpret_cast<volatile int*>(P.err) = where;
    S.misc[20] = 1;                                   // every later poll of this CTA gives up at once: the launch drains quickly
}
__device__ __forceinline__ bool mg_spin_out(const MgSmem& S, int& spins) { return ++spins > (S.misc[20] ? 0 : MG_SPIN_LIMIT); }

// ---- attention of one layer, two stages chained through LL words ------------------------------------------------------------
// CTA c serves KV head c % n_head_kv, context split c / n_head_kv.  The K and V rows of the CTA's token slice are copied
// into shared memory with cp.async at the START of the layer's QKV phase (only the row of the token being decoded has to wait
// for that phase: it arrives as f32 LL words), so both stages work out of shared memory.
struct MgAttn { int hk, split, n_split, t0, nt; bool on; };
__device__ __forceinline__ MgAttn mg_attn_get(const MgSmem& S) {   // computed once per token (mg_attn_setup), kept in shared memory
    MgAttn a; a.hk = S.misc[1]; a.split = S.misc[2]; a.n_split = S.misc[3]; a.t0 = S.misc[4]; a.nt = S.misc[5]; a.on = S.misc[6] != 0; return a;
}
__device__ __forceinline__ void mg_attn_setup(const MegaParams& P, int n_kv, const MgSmem& S) {
    const int n_split = max(1, min(P.max_split, (n_kv + P.ts_cap - 1) / P.ts_cap));
    const int hk = (int)blockIdx.x % P.n_head_kv, split = (int)blockIdx.x / P.n_head_kv;
    const int per = (n_kv + n_split - 1) / n_split;
    const int t0 = split * per;
    S.misc[1] = hk; S.misc[2] = split; S.misc[3] = n_split; S.misc[4] = t0; S.misc[5] = max(0, min(n_kv, t0 + per) - t0); S.misc[6] = split < n_split ? 1 : 0;
}
__device__ __forceinline__ size_t mg_kv_row(const MegaParams& P, int hk, int t) {
    return ((size_t)P.page_table[t / KV_PAGE] * KV_PAGE + (t % KV_PAGE)) * P.kv_dim + (size_t)hk * P.d_head;
}
struct MgAttnSmem { __half* q; float* sc; __half* k; __half* v; float* red; };
__device__ __forceinline__ MgAttnSmem mg_attn_carve(const MegaParams& P, unsigned char* base) {
    const int gq = P.n_head / P.n_head_kv;
    MgAttnSmem s;
    s.q = reinterpret_cast<__half*>(base);
    s.sc = reinterpret_cast<float*>(base + (size_t)gq * P.d_head * 2);
    s.k = reinterpret_cast<__half*>(reinterpret_cast<unsigned char*>(s.sc) + (size_t)gq * P.ts_cap * 4);
    s.v = s.k + (size_t)P.ts_cap * P.d_head;
    s.red = reinterpret_cast<float*>(s.k);          // [token group][gq][dh] partial outputs, once the tiles are dead
    return s;
}
// rows [tile0, tile0 + cn) of the slice, restricted to tokens < t_limit -> shared memory (cp.async)
__device__ __forceinline__ void mg_attn_load_rows(const MegaParams& P, const MgAttn& a, const __half* pool, __half* dst, int tile0, int cn, int t_limit) {
    const int dh = P.d_head, csh = dh == 128 ? 4 : 3;               // 16-byte chunks per row: dh / 8
    for (int idx = threadIdx.x; idx < (cn << csh); idx += MG_THREADS) {
        const int tl = idx >> csh, c = idx & ((1 << csh) - 1);
        const int t = a.t0 + tile0 + tl;
        if (t >= t_limit) continue;
        const __half* src = pool + mg_kv_row(P, a.hk, t) + c * 8;
        cp_async16(dst + (size_t)tl * dh + c * 8, src);
    }
}

// first tile of K and V of this CTA's slice, except the token being decoded
__device__ __noinline__ void mg_attn_prefetch(const MegaParams& P, int layer, int n_kv, const MgSmem& S) {
    const MgAttn a = mg_attn_get(S);
    if (!a.on || a.nt == 0) return;
    const MgAttnSmem s = mg_attn_carve(P, S.attn);
    const int cn = min(a.nt, P.ts_cap);
    mg_attn_load_rows(P, a, S.kp[layer], s.k, 0, cn, n_kv - 1);
    mg_attn_load_rows(P, a, S.vp[layer], s.v, 0, cn, n_kv - 1);
    cp_async_commit();
}

// scaled scores of ONE tile (rows [0, cn) of s.k) against the gq query heads in s.q -> s.sc: 8 lanes per token, dh / 8 dims each
template <int GQ>
__device__ __forceinline__ void mg_scores_tile(const MegaParams& P, const MgAttnSmem& s, int cn, int gq, int dh) {
    const int tid = threadIdx.x;
    const int ld = tid & 7, tl = tid >> 3;
    const int DL = dh >> 3;
    float sc[GQ];
#pragma unroll
    for (int gI = 0; gI < GQ; gI++) sc[gI] = 0.0f;
    if (tl < cn) {
        for (int c = 0; c < DL; c += 8) {
            const uint4 kv = *reinterpret_cast<const uint4*>(s.k + (size_t)tl * dh + ld * DL + c);
            const __half2* kh = reinterpret_cast<const __half2*>(&kv);
            float kf[8];
#pragma unroll
            for (int i = 0; i < 4; i++) { const float2 f = __half22float2(kh[i]); kf[2 * i] = f.x; kf[2 * i + 1] = f.y; }
#pragma unroll
            for (int gI = 0; gI < GQ; gI++) if (gI < gq) {
                const uint4 qq = *reinterpret_cast<const uint4*>(s.q + gI * dh + ld * DL + c);
                const __half2* qh = reinterpret_cast<const __half2*>(&qq);
#pragma unroll
                for (int i = 0; i < 4; i++) { const float2 f = __half22float2(qh[i]); sc[gI] += kf[2 * i] * f.x; sc[gI] += kf[2 * i + 1] * f.y; }
            }
        }
    }
#pragma unroll
    for (int gI = 0; gI < GQ; gI++) if (gI < gq) {
        float v = sc[gI];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        v = __fmul_rn(v, P.attn_scale);
        if (tl < cn && ld == 0) s.sc[gI * P.ts_cap + tl] = v;
    }
}

// stage 1: scaled scores of the first tile of this CTA's token slice for the gq query heads of its KV head -> shared memory
// (stage 2 scores the later tiles)
template <int GQ>
__device__ __noinline__ void mg_attn_scores(const MegaParams& P, int phi, int n_kv, const MgSmem& S) {
    const MgAttn a = mg_attn_get(S);
    if (!a.on || a.nt == 0) return;
    const MgAttnSmem s = mg_attn_carve(P, S.attn);
    const int tid = threadIdx.x, dh = P.d_head, gq = P.n_head / P.n_head_kv;
    const uint32_t tag_in = mg_tag(P.seq, phi, 0);
    // poll: the query heads, and (slice holding the new token only) the K / V rows this layer's QKV phase produced
    const int cn0 = min(P.ts_cap, a.nt);
    const int tl_new = n_kv - 1 - a.t0;                             // local index of the token being decoded
    const bool has_new = tl_new >= 0 && tl_new < cn0;
    const int nq = gq * dh, nnew = has_new ? 2 * dh : 0;            // words this CTA needs: thread i takes i, i + 512, ...
    {
        uint2 w[3];
        int spins = 0;
        bool ok;
        do {
            ok = true;
#pragma unroll
            for (int r = 0; r < 3; r++) {
                const int i = tid + r * MG_THREADS;
                if (i < nq) w[r] = ll_ld(P.q2 + (size_t)(a.hk * gq) * dh + i);
                else if (i < nq + nnew) { const int j = i - nq; w[r] = ll_ld(P.kvn2 + (size_t)(j < dh ? 0 : P.kv_dim) + a.hk * dh + (j < dh ? j : j - dh)); }
                else w[r] = make_uint2(0u, tag_in);
                ok = ok && w[r].y == tag_in;
            }
            if (mg_spin_out(S, spins)) { mg_poll_timeout(P, S, 1); break; }
        } while (!__syncthreads_and(ok));
#pragma unroll
        for (int r = 0; r < 3; r++) {
            const int i = tid + r * MG_THREADS;
            if (i < nq) s.q[i] = __float2half_rn(__uint_as_float(w[r].x));
            else if (i < nq + nnew) { const int j = i - nq; (j < dh ? s.k : s.v)[(size_t)tl_new * dh + (j < dh ? j : j - dh)] = __float2half_rn(__uint_as_float(w[r].x)); }
        }
    }
    cp_async_wait_all();
    __syncthreads();
    mg_scores_tile<GQ>(P, s, cn0, gq, dh);
}

// stage 2: soft-max over the CTA's OWN scores (local maximum and sum, merged by the CTAs of the head): the scores never leave the CTA.
//   one slice (n_split == 1): that is the whole row -- ggml's order exactly (max -> expf -> sum in double -> p * (1/sum) -> f16 -> V.p),
//     the result goes straight to the attention output;
//   several slices: flash-style -- p = f16(expf(s - m_local)), o = sum p v, and (m_local, l_local) travel with the partial; the CTAs
//     of the head merge: M = max m_s, w_s = expf(m_s - M), out = (sum_s w_s o_s) / (sum_s w_s l_s).  Against ggml this moves the f16
//     rounding of the probabilities in front of the normalisation (a 2^-11 relative change per probability, the size of every other
//     rounding difference between two implementations of this arithmetic); it removes the all-to-all exchange of the scores and the
//     statistics pass over the whole row.
//   a slice longer than one shared-memory tile (contexts beyond max_split x ts_cap = 1152 tokens on the 8B model) is walked tile by
//     tile with a running maximum: the later tiles' K / V rows are fetched synchronously, their scores computed here, and the
//     accumulator rescaled by expf(m_old - m_new) -- the same flash order, now inside the CTA too.
template <int GQ, bool TR>
__device__ __noinline__ void mg_attn_pv(const MegaParams& P, int layer, int phi, int n_kv, const MgSmem& S) {
    const MgAttn a = mg_attn_get(S);
    if (!a.on) return;
    const MgAttnSmem s = mg_attn_carve(P, S.attn);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, dh = P.d_head, gq = P.n_head / P.n_head_kv;
    const uint32_t tag_in = mg_tag(P.seq, phi, 0), tag_po = mg_tag(P.seq, phi, 2), tag_ao = mg_tag(P.seq, phi, 3);
    const int TG = MG_THREADS / dh;
    const int d = tid & (dh - 1), tg = dh == 128 ? tid >> 7 : tid >> 6;
    const bool single = a.n_split == 1;
    const bool multi = a.nt > P.ts_cap;                    // more than one tile in this slice (never with a single slice)
    float m_run = -INFINITY, l_run = 0.0f;                 // warps < gq: running statistics of their query head
    float acc[GQ];
#pragma unroll
    for (int gI = 0; gI < GQ; gI++) acc[gI] = 0.0f;
    __syncthreads();                                       // the scores of stage 1 (written by the token's lane group) are in shared memory
    if (a.nt > 0) {
        // later tiles travel behind the computation: K of tile c + 1 is requested when the scores of tile c are done (the K rows are
        // dead), V of tile c + 1 when P.V of tile c is (cp.async groups in that order)
        if (multi) { mg_attn_load_rows(P, a, S.kp[layer], s.k, P.ts_cap, min(P.ts_cap, a.nt - P.ts_cap), n_kv - 1); cp_async_commit(); }
        for (int c0 = 0; c0 < a.nt; c0 += P.ts_cap) {
            const int cn = min(P.ts_cap, a.nt - c0);
            const bool more = c0 + P.ts_cap < a.nt;
            const int tl_new = n_kv - 1 - a.t0 - c0;       // the token being decoded: its rows are this layer's LL words (polled: other CTAs than q's)
            const bool new_here = c0 > 0 && tl_new >= 0 && tl_new < cn;
            if (c0 > 0) {
                __syncthreads();                           // P.V of the previous tile has read its V rows and probabilities
                mg_attn_load_rows(P, a, S.vp[layer], s.v, c0, cn, n_kv - 1);
                cp_async_commit();
                cp_async_wait_group<1>();                  // this tile's K rows have landed (its V rows may still fly)
                if (new_here && tid < dh) {
                    const uint2* src = P.kvn2 + a.hk * dh + tid;
                    uint2 w = ll_ld(src);
                    int spins = 0;
                    while (w.y != tag_in) { if (mg_spin_out(S, spins)) { mg_poll_timeout(P, S, 1); break; } w = ll_ld(src); }
                    s.k[(size_t)tl_new * dh + tid] = __float2half_rn(__uint_as_float(w.x));
                }
                __syncthreads();
                mg_scores_tile<GQ>(P, s, cn, gq, dh);
                __syncthreads();
                if (more) { mg_attn_load_rows(P, a, S.kp[layer], s.k, c0 + P.ts_cap, min(P.ts_cap, a.nt - c0 - P.ts_cap), n_kv - 1); cp_async_commit(); }
            }
            if (warp < gq) {                               // warp g: statistics and probabilities of query head g
                float* row = s.sc + warp * P.ts_cap;
                float m = -INFINITY;
                for (int tl = lane; tl < cn; tl += 32) m = fmaxf(m, row[tl]);
                m = warp_max(m);
                if (multi) m = fmaxf(m, m_run);
                double sum = 0.0;
                for (int tl = lane; tl < cn; tl += 32) { const float e = expf(row[tl] - m); row[tl] = e; sum += (double)e; }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
                __syncwarp();
                if (single) {
                    const float inv = (float)(1.0 / sum);
                    for (int tl = lane; tl < cn; tl += 32) row[tl] = __half2float(__float2half_rn(__fmul_rn(row[tl], inv)));
                } else {
                    for (int tl = lane; tl < cn; tl += 32) row[tl] = __half2float(__float2half_rn(row[tl]));
                    if (!multi) { if (lane == 0) ll_st2(P.st2 + ((size_t)(a.hk * gq + warp) * P.max_split + a.split) * 2, m, (float)sum, tag_po); }
                    else {
                        const float corr = expf(m_run - m);                 // 0 on the first tile
                        l_run = l_run * corr + (float)sum; m_run = m;
                        if (lane == 0) S.stat[16 + warp] = corr;
                    }
                }
            }
            if (c0 > 0) {
                if (more) cp_async_wait_group<1>(); else cp_async_wait_all();      // this tile's V rows have landed
                if (new_here && tid >= dh && tid < 2 * dh) {
                    const int j = tid - dh;
                    const uint2* src = P.kvn2 + P.kv_dim + a.hk * dh + j;
                    uint2 w = ll_ld(src);
                    int spins = 0;
                    while (w.y != tag_in) { if (mg_spin_out(S, spins)) { mg_poll_timeout(P, S, 1); break; } w = ll_ld(src); }
                    s.v[(size_t)tl_new * dh + j] = __float2half_rn(__uint_as_float(w.x));
                }
            }
            __syncthreads();
            if (c0 == 0) mg_tr<TR>(P, S, 13);
            if (multi && c0 > 0) {
#pragma unroll
                for (int gI = 0; gI < GQ; gI++) if (gI < gq) acc[gI] *= S.stat[16 + gI];
            }
#pragma unroll 4
            for (int tl = tg; tl < cn; tl += TG) {
                const float v = __half2float(s.v[(size_t)tl * dh + d]);
#pragma unroll
                for (int gI = 0; gI < GQ; gI++) if (gI < gq) acc[gI] += s.sc[gI * P.ts_cap + tl] * v;
            }
        }
        if (multi && warp < gq && lane == 0) ll_st2(P.st2 + ((size_t)(a.hk * gq + warp) * P.max_split + a.split) * 2, m_run, l_run, tag_po);
    } else if (!single && warp < gq && lane == 0) {
        ll_st2(P.st2 + ((size_t)(a.hk * gq + warp) * P.max_split + a.split) * 2, -INFINITY, 0.0f, tag_po);
    }
    __syncthreads();
    mg_tr<TR>(P, S, 14);
#pragma unroll
    for (int gI = 0; gI < GQ; gI++) if (gI < gq) s.red[(tg * gq + gI) * dh + d] = acc[gI];
    __syncthreads();
    const int E = gq * dh, NO = P.n_head * dh;
    for (int e = tid; e < E; e += MG_THREADS) {
        float o = 0.0f;
        for (int k = 0; k < TG; k++) o += s.red[k * E + e];
        if (single) ll_st(P.ao2 + (size_t)a.hk * E + e, o, tag_ao);
        else ll_st(P.po2 + (size_t)a.split * NO + a.hk * E + e, o, tag_po);
    }
    mg_tr<TR>(P, S, 15);
    if (single) return;
    // ---- merge, spread over the CTAs of the KV head: split s owns elements [s per, s per + per) of the head group's output.  One
    //      thread per (element, slice) pair, statistics and partials polled TOGETHER (one L2 round trip behind the slowest slice
    //      instead of the split-0 CTA's three dependent ones); the sum runs in split order as before (bit-identical). ----
    const int ns = a.n_split;
    const int per = (E + ns - 1) / ns;
    const int e0 = a.split * per, ne = max(0, min(E, e0 + per) - e0);
    const int n_items = ne * ns;
    float* wgt = reinterpret_cast<float*>(S.redd);          // [gq <= 8][32] merge weights (the double reduction scratch: 256 floats)
    float* wp = s.red;                                      // [ne][ns] partials of this CTA's elements (the reduction scratch is dead after the sync below)
    {
        const uint2* sp = P.st2 + (size_t)(a.hk * gq + min(warp, gq - 1)) * P.max_split * 2;
        const bool st_on = warp < gq && lane < ns;
        int el[3], sl[3];                                 // n_items <= E + ns - 1 <= 8 * 128 + 31 < 3 * MG_THREADS
#pragma unroll
        for (int r = 0; r < 3; r++) { const int it = tid + r * MG_THREADS; el[r] = it / ns; sl[r] = it - el[r] * ns; }
        float m = -INFINITY, l = 0.0f, pv[3] = {0.0f, 0.0f, 0.0f};
        int spins = 0;
        bool ok;
        do {
            ok = true;
            if (st_on) { const uint4 w = ll_ld2(sp + lane * 2); m = __uint_as_float(w.x); l = __uint_as_float(w.z); ok = w.y == tag_po && w.w == tag_po; }
#pragma unroll
            for (int r = 0; r < 3; r++) if (tid + r * MG_THREADS < n_items) {
                const uint2 w = ll_ld(P.po2 + (size_t)sl[r] * NO + a.hk * E + e0 + el[r]);
                pv[r] = __uint_as_float(w.x); ok = ok && w.y == tag_po;
            }
            if (mg_spin_out(S, spins)) { mg_poll_timeout(P, S, 2); break; }
        } while (!__syncthreads_and(ok));
        if (warp < gq) {
            const float M = warp_max(lane < ns ? m : -INFINITY);
            const float w = lane < ns ? expf(m - M) : 0.0f;
            float L = w * l;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) L += __shfl_xor_sync(0xffffffffu, L, o);
            if (lane < ns) wgt[warp * 32 + lane] = w;
            if (lane == 0) S.stat[warp] = __fdiv_rn(1.0f, L);
        }
#pragma unroll
        for (int r = 0; r < 3; r++) if (tid + r * MG_THREADS < n_items) wp[tid + r * MG_THREADS] = pv[r];
    }
    __syncthreads();
    if (tid < ne) {
        const int e = e0 + tid;
        const int g = dh == 128 ? e >> 7 : e >> 6;
        float o = 0.0f;
        for (int s0 = 0; s0 < ns; s0++) o += wgt[g * 32 + s0] * wp[tid * ns + s0];
        ll_st(P.ao2 + (size_t)a.hk * E + e, o * S.stat[g], tag_ao);
    }
}

// ---- warp group bookkeeping without integer divisions ---------------------------------------------------------------------------
__device__ __forceinline__ void mg_warp_group(const MegaPhase* ph, int warp, int& g_local, int& ws, bool& active) {
    if (ph->wsh >= 0) { g_local = warp >> ph->wsh; ws = warp & (ph->W - 1); }
    else { g_local = warp / ph->W; ws = warp - g_local * ph->W; }
    active = g_local < ph->NG;
}
// first pair of group gg in a segment (pairs gg', gg' + NGtot, ... with gg' = (gg + rot) mod NGtot)
__device__ __forceinline__ int mg_first_pair(const MegaSeg& sg, int gg, int NGtot) { const int v = gg + sg.rot; return v >= NGtot ? v - NGtot : v; }

// row pair e of this CTA in a phase: e -> (warp group, partial-sum slot) -> (segment, pair index)
__device__ __forceinline__ bool mg_item_of(const MegaPhase* ph, int n_cta, int e, int& gl, int& ks, int& seg, int& p) {
    const int NG = ph->NG, NGtot = n_cta * NG;
    if (ph->ngsh >= 0) { gl = e & (NG - 1); ks = e >> ph->ngsh; } else { ks = e / NG; gl = e - ks * NG; }
    const int gg = (int)blockIdx.x * NG + gl;
    seg = 0;
    if (ph->nseg > 1 && ks >= ph->seg[1].slot0) seg = 1;
    if (ph->nseg > 2 && ks >= ph->seg[2].slot0) seg = 2;
    const MegaSeg& sg = ph->seg[seg];
    p = mg_first_pair(sg, gg, NGtot) + (ks - sg.slot0) * NGtot;
    return p < sg.n_pairs;
}

// ---- epilogue of a stream phase: combine the K-slice partials of every row pair of this CTA and publish the rows ---------
// res: x[r0], x[r1] of the pair of thread tid (residual phases: fetched before the mat-vec, see the kernel)
__device__ __noinline__ void mg_epilogue(const MegaParams& P, const MegaPhase* ph, int phi, int pos, const MgSmem& S, float2 res, bool have_res) {
    const int tid = threadIdx.x, dh = P.d_head;
    const int NG = ph->NG, W = ph->W;
    const uint32_t tag = mg_tag(P.seq, phi, 0);
    for (int e = tid; e < NG * ph->items; e += MG_THREADS) {
        int gl, ks, s, p;
        if (!mg_item_of(ph, P.n_cta, e, gl, ks, s, p)) continue;
        const MegaSeg& sg = ph->seg[s];
        float v0 = 0.0f, v1 = 0.0f;
        for (int w = 0; w < W; w++) { const float2 t = S.part[ks * MG_WARPS + gl * W + w]; v0 += t.x; v1 += t.y; }
        const int kind = sg.kind;
        if (kind == MK_SWIGLU) { ll_st(P.h2 + p, (v0 / (1.0f + expf(-v0))) * v1, tag); continue; }     // ggml_silu_f32 then ggml_mul
        int r0 = 2 * p, r1 = 2 * p + 1;
        if ((kind == MK_Q || kind == MK_K) && P.neox) { const int hd = dh >> 1; const int hh = dh == 128 ? p >> 6 : p >> 5; r0 = hh * dh + (p & (hd - 1)); r1 = r0 + hd; }
        if (sg.bias) { v0 += sg.bias[r0]; v1 += sg.bias[r1]; }
        if (kind == MK_RESID) {
            if (!(have_res && e == tid)) { res.x = __uint_as_float(ll_ld(P.x2 + r0).x); res.y = __uint_as_float(ll_ld(P.x2 + r1).x); }
            ll_st2(P.x2 + r0, res.x + v0, res.y + v1, tag);
        } else if (kind == MK_LOGITS) {
            *reinterpret_cast<float2*>(P.logits + r0) = make_float2(v0, v1);
            atomicMax(P.chunk_max + (r0 >> P.chunk_shift), float_order_key(fmaxf(v0, v1)));
        } else {
            if (kind != MK_V) {                                   // rotary embedding on the pair: ggml rope NORM / NEOX
                const int i = P.neox ? (r0 & (dh - 1)) : ((r0 & (dh - 1)) >> 1);
                const float2 cs = S.rope[i];
                const float x0 = v0, x1 = v1;
                v0 = x0 * cs.x - x1 * cs.y;
                v1 = x0 * cs.y + x1 * cs.x;
            }
            if (kind == MK_Q) { ll_st(P.q2 + r0, v0, tag); ll_st(P.q2 + r1, v1, tag); }
            else {
                const size_t base = ((size_t)S.misc[0] * KV_PAGE + (pos % KV_PAGE)) * P.kv_dim;
                __half* dst = (kind == MK_K ? S.kp : S.vp)[ph->layer];
                dst[base + r0] = __float2half_rn(v0);           // ggml_cpy f32 -> f16 into the cache (read by later tokens)
                dst[base + r1] = __float2half_rn(v1);
                uint2* kn = P.kvn2 + (kind == MK_K ? 0 : P.kv_dim);     // ... and as LL words for this token's attention
                ll_st(kn + r0, v0, tag); ll_st(kn + r1, v1, tag);
            }
        }
    }
}

// ---- prologue of a stream phase: wait for the source vector (LL words), (RMSNorm *) quantise it into shared memory ---------
// One warp per 256-element block, redundantly per CTA.  With a norm the row has at most 2 blocks per warp (K <= 8192), held in
// registers for both the sum of squares and the quantisation; nw: this lane's norm weights, fetched before the wait.
// Code size matters here (the whole decode loop has to stay resident in the instruction cache): ONE quantiser instance.
__device__ __forceinline__ float4 mg_norm4(float4 v, float scale, float4 w) {
    return make_float4(__fmul_rn(__fmul_rn(v.x, scale), w.x), __fmul_rn(__fmul_rn(v.y, scale), w.y), __fmul_rn(__fmul_rn(v.z, scale), w.z), __fmul_rn(__fmul_rn(v.w, scale), w.w));
}
__device__ __forceinline__ double mg_sq4(float4 v) {
    return ((double)__fmul_rn(v.x, v.x) + (double)__fmul_rn(v.y, v.y)) + ((double)__fmul_rn(v.z, v.z) + (double)__fmul_rn(v.w, v.w));
}
__device__ __forceinline__ MgV8 mg_ll_vals(const MgV8F& r) {
    MgV8 v;
    v.a = make_float4(__uint_as_float(r.a.x), __uint_as_float(r.a.z), __uint_as_float(r.b.x), __uint_as_float(r.b.z));
    v.b = make_float4(__uint_as_float(r.c.x), __uint_as_float(r.c.z), __uint_as_float(r.d.x), __uint_as_float(r.d.z));
    return v;
}
// 8 consecutive values of a block (this lane's share), polled until every word carries the tag (warp-uniform exit)
__device__ __forceinline__ MgV8 mg_ll_wait8(const MegaParams& P, const MgSmem& S, const uint2* p, uint32_t tag, bool active) {
    MgV8F r = ll_ld8(p);
    int spins = 0;
    while (!__all_sync(0xffffffffu, !active || ll_ok8(r, tag))) {
        if (mg_spin_out(S, spins)) { mg_poll_timeout(P, S, 4); break; }
        r = ll_ld8(p);
    }
    return mg_ll_vals(r);
}
template <bool TR>
__device__ __noinline__ void mg_prologue(const MegaParams& P, const MegaPhase* ph, int phi, const MgSmem& S, float4 nw0, float4 nw1, float4 nw2, float4 nw3) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int K = ph->K, fmt = ph->act_fmt, nblk = K >> 8;
    int8_t* sq = reinterpret_cast<int8_t*>(S.act);
    float* sd = reinterpret_cast<float*>(S.act + K);
    int16_t* sbs = reinterpret_cast<int16_t*>(S.act + K + (K >> 5) * 4);
    const uint2* src = (ph->src == MSRC_X ? P.x2 : (ph->src == MSRC_ATTN ? P.ao2 : P.h2)) + lane * 8;
    const uint32_t tag = phi == 0 ? P.seq * 4096u : mg_tag(P.seq, phi - 1, ph->src == MSRC_ATTN ? 3 : 0);
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ph->norm_w) {
        const int b0 = warp, b1 = warp + MG_WARPS;
        MgV8 v0, v1; v0.a = v0.b = v1.a = v1.b = z4;
        if (b0 < nblk) v0 = mg_ll_wait8(P, S, src + b0 * 256, tag, true);
        if (b1 < nblk) v1 = mg_ll_wait8(P, S, src + b1 * 256, tag, true);
        double sum = (mg_sq4(v0.a) + mg_sq4(v0.b)) + (mg_sq4(v1.a) + mg_sq4(v1.b));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) S.redd[warp] = sum;
        mg_tr<TR>(P, S, 30);
        __syncthreads();
        double t4[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int i = 0; i < MG_WARPS; i++) t4[i & 3] += S.redd[i];
        const double tot = (t4[0] + t4[1]) + (t4[2] + t4[3]);
        const float mean = (float)(tot / (double)K);
        const float scale = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(mean, P.eps)));
        mg_tr<TR>(P, S, 31);
#pragma unroll 1
        for (int r = 0; r < 2; r++) {
            const int b = r ? b1 : b0;
            if (b < nblk) mg_quantize_regs(mg_norm4(r ? v1.a : v0.a, scale, r ? nw2 : nw0), mg_norm4(r ? v1.b : v0.b, scale, r ? nw3 : nw1), fmt, b, sq, sd, sbs);
        }
    } else {
#pragma unroll 1
        for (int b = warp; b < nblk; b += MG_WARPS) {
            const MgV8 cur = mg_ll_wait8(P, S, src + b * 256, tag, true);
            if (b == warp) mg_tr<TR>(P, S, 32);
            mg_quantize_regs(cur.a, cur.b, fmt, b, sq, sd, sbs);
        }
    }
    mg_tr<TR>(P, S, 34);
    __syncthreads();
}

// =================================================================================================================
// the kernel
// =================================================================================================================
template <int GQ, bool TR>
__global__ void __launch_bounds__(MG_THREADS, 1) mega_decode_kernel(const __grid_constant__ MegaParams P) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const MgSmem S = mg_carve(P, smem);
    unsigned char* ring = smem + (size_t)warp * MG_SLOTS * P.slot_bytes;
    uint64_t* my_bar = S.bars + warp * MG_SLOTS;

    if (lane == 0) { for (int s = 0; s < MG_SLOTS; s++) mbar_init(my_bar + s, 1); mbar_fence_init(); }
    __syncwarp();

    // ---- producer: this warp's chunk list; prime the ring (weights do not depend on anything) ----
    const uint4* plist = P.chunk_list + ((size_t)blockIdx.x * MG_WARPS + warp) * P.list_stride;
    const int p_total = P.chunk_counts[blockIdx.x * MG_WARPS + warp];
    int p_issued = 0, c_done = 0;
    uint4 p_desc = p_total > 0 ? __ldg(plist) : make_uint4(0, 0, 0, 0);
    auto issue_next = [&]() {
        if (p_issued < p_total) {
            if (lane == 0) {
                const int slot = p_issued % MG_SLOTS;
                mbar_expect_tx(my_bar + slot, p_desc.z);
                bulk_g2s(ring + (size_t)slot * P.slot_bytes, reinterpret_cast<const void*>(((unsigned long long)p_desc.y << 32) | p_desc.x), p_desc.z, my_bar + slot);
            }
            p_issued++;
            if (p_issued < p_total) p_desc = __ldg(plist + p_issued);
        }
    };
#pragma unroll 1
    for (int s = 0; s < MG_SLOTS; s++) issue_next();

    // ---- per-token constants into shared memory: phase descriptors 0 / 1, KV pool pointers, the page of this position,
    //      this CTA's attention assignment ----
    const int pos = P.pos[0];
    const int n_kv = pos + 1;
    auto fetch_phase = [&](int phi) {     // one warp copies descriptor phi into its shared-memory slot (visible after a CTA sync)
        if (phi < P.n_phases && lane < (int)(sizeof(MegaPhase) / 16))
            reinterpret_cast<uint4*>(S.ph + (phi & 1))[lane] = __ldg(reinterpret_cast<const uint4*>(P.phases + phi) + lane);
    };
    if (warp == 0) fetch_phase(0);
    if (warp == 1) fetch_phase(1);
    for (int l = tid; l < P.n_layer; l += MG_THREADS) { S.kp[l] = P.k_pools[l]; S.vp[l] = P.v_pools[l]; }
    if (tid == 0) {
        S.misc[0] = P.page_table[pos / KV_PAGE]; S.misc[16] = 0; S.misc[20] = 0;
        mg_attn_setup(P, n_kv, S);
    }
    __syncthreads();

    mg_tr<TR>(P, S, 1);
    mg_embed(P);
    rope_table_fill(S.rope, P.d_head / 2, pos + P.pos[1], P.theta_scale, P.rope_freqs);      // P.pos = {cell index, rotary offset (Self-Extend)}
    __syncthreads();

    // ================================= the token: one stream phase per iteration =================================
    // pre-wait part | prologue (waits for the source vector's LL words) | mat-vec | epilogue (publishes LL words)
    //   (| the two attention stages after a QKV phase).  There is no grid barrier: the data carries its own epoch.
    // ONE instance of this body (the kernel must stay small enough for the instruction cache): the phase table drives it.
    const int n_run = P.with_head ? P.n_phases : P.n_phases - 1;
#pragma unroll 1
    for (int phi = 0; phi < n_run; phi++) {
        const MegaPhase* ph = S.ph + (phi & 1);
        const bool is_qkv = ph->seg[0].kind == MK_Q;
        const int layer = ph->layer;
        const int trk = (is_qkv ? 0 : ph->seg[0].kind == MK_SWIGLU ? 2 : ph->seg[0].kind == MK_LOGITS ? 4 : (ph->src == MSRC_ATTN ? 1 : 3)) << 5;
        mg_tr<TR>(P, S, trk | 2);
        // -- before the wait: everything that does not depend on the other CTAs --
        float4 nw[4];
        nw[0] = nw[1] = nw[2] = nw[3] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ph->norm_w) {
#pragma unroll
            for (int r = 0; r < 2; r++) {
                const int b = warp + r * MG_WARPS;
                if (b < (ph->K >> 8)) { const float4* wp = reinterpret_cast<const float4*>(ph->norm_w + b * 256 + lane * 8); nw[2 * r] = __ldg(wp); nw[2 * r + 1] = __ldg(wp + 1); }
            }
        }
        if (is_qkv) mg_attn_prefetch(P, layer, n_kv, S);      // this layer's K / V tiles start streaming into shared memory
        int g_local, ws; bool g_active;
        mg_warp_group(ph, warp, g_local, ws, g_active);
        const int L = ph->L, rpc = ph->rpc, NGtot = P.n_cta * ph->NG, gg = (int)blockIdx.x * ph->NG + g_local;
        const int K = ph->K, fmt = ph->act_fmt;
        const int sub = lane >= L ? (lane >= 2 * L ? 2 : 1) : 0;     // row of the chunk this lane works on
        const int hsl = lane - sub * L;                   // half super-block inside the slice
        const int hs = ws * L + hsl;                      // ... inside the row
        const bool lane_on = g_active && sub < rpc && hs < (K >> 7);
        // residual rows of the pair this thread will finish in the epilogue (x is stable: its last writer phase was waited for
        // by this CTA's previous normed prologue, the next writer is this phase)
        float2 res = make_float2(0.f, 0.f);
        const bool have_res = ph->seg[0].kind == MK_RESID && ph->NG * ph->items <= MG_THREADS;
        if (have_res && tid < ph->NG * ph->items) {
            int gl, ks, s, p;
            if (mg_item_of(ph, P.n_cta, tid, gl, ks, s, p)) { const uint4 t = ll_ld2(P.x2 + 2 * p); res = make_float2(__uint_as_float(t.x), __uint_as_float(t.z)); }
        }
        if (warp == 2) fetch_phase(phi + 1);              // next phase's descriptor (its slot's last reader was phase phi - 1)
        mg_prologue<TR>(P, ph, phi, S, nw[0], nw[1], nw[2], nw[3]);
        mg_tr<TR>(P, S, trk | 3);
        // -- this lane's activations --
        LaneAct A;
        if (lane_on) {
            const int8_t* sq = reinterpret_cast<const int8_t*>(S.act);
            const float* sd = reinterpret_cast<const float*>(S.act + K);
            const int16_t* sbs = reinterpret_cast<const int16_t*>(S.act + K + (K >> 5) * 4);
#pragma unroll
            for (int c = 0; c < 8; c++) {
                const uint4 t = lds128(sq + hs * 128 + ((c ^ (hs & 7)) << 4));
                A.q[4 * c] = (int)t.x; A.q[4 * c + 1] = (int)t.y; A.q[4 * c + 2] = (int)t.z; A.q[4 * c + 3] = (int)t.w;
            }
            if (fmt == ACT_Q8_K) {
                A.d0 = sd[hs >> 1];
                const uint4 t = lds128(sbs + hs * 8);
                A.aux[0] = t.x; A.aux[1] = t.y; A.aux[2] = t.z; A.aux[3] = t.w;
                auto pair_sum = [](uint32_t w) -> int { return (int)(int16_t)(w & 0xffff) + (int)(int16_t)(w >> 16); };
                A.aux[4] = (uint32_t)(pair_sum(t.x) & 0xffff) | ((uint32_t)pair_sum(t.y) << 16);
                A.aux[5] = (uint32_t)(pair_sum(t.z) & 0xffff) | ((uint32_t)pair_sum(t.w) << 16);
            } else {
                A.d0 = 0.0f;
#pragma unroll
                for (int b = 0; b < 4; b++) A.aux[b] = __float_as_uint(sd[hs * 4 + b]);
                A.aux[4] = A.aux[5] = 0u;
            }
        } else {
#pragma unroll
            for (int i = 0; i < 32; i++) A.q[i] = 0;
            A.d0 = 0.0f;
#pragma unroll
            for (int i = 0; i < 6; i++) A.aux[i] = 0u;
        }
        mg_tr<TR>(P, S, trk | 4);
        // -- main loop: every chunk of this warp in this phase --
        const int sb = hsl >> 1, hf = hsl & 1;
        for (int s = 0; s < ph->nseg; s++) {
            const MegaSeg* sg = ph->seg + s;
            const int type = sg->type, n_pairs = g_active ? sg->n_pairs : 0;
            const int sub_off = sub * sg->slice_bytes;
            const int tail_off = (L >> 1) * 208 + sb * 2;     // Q6_K: this super-block's d in the slice tail
            int slot_i = sg->slot0;
            for (int p = mg_first_pair(*sg, gg, NGtot); p < n_pairs; p += NGtot, slot_i++) {
                float va = 0.0f, vb = 0.0f;
#pragma unroll 1
                for (int c = 0; c < 2 / rpc; c++) {           // one code instance for both rows of the pair
                    const int slot = c_done % MG_SLOTS;
                    mbar_wait(my_bar + slot, (uint32_t)((c_done / MG_SLOTS) & 1));
                    const unsigned char* sl = ring + (size_t)slot * P.slot_bytes + sub_off;
                    float v = 0.0f;
                    if (lane_on) {
                        uint4 wb[9];
                        if (type == QT_Q4_K) {
                            const unsigned char* b = sl + sb * 144;
                            wb[0] = lds128(b);
#pragma unroll
                            for (int i = 0; i < 4; i++) wb[1 + i] = lds128(b + 16 + hf * 64 + 16 * i);
                            v = mg_dot_q4k(wb, hf, A);
                        } else if (type == QT_Q6_K) {
                            const unsigned char* b = sl + sb * 208;
#pragma unroll
                            for (int i = 0; i < 2; i++) { wb[i] = lds128(b + hf * 64 + 16 * i); wb[2 + i] = lds128(b + hf * 64 + 32 + 16 * i); }
#pragma unroll
                            for (int i = 0; i < 2; i++) wb[4 + i] = lds128(b + 128 + hf * 32 + 16 * i);
                            const uint2 sc = *reinterpret_cast<const uint2*>(b + 192 + hf * 8);
                            wb[6].x = sc.x; wb[6].y = sc.y;
                            wb[6].z = *reinterpret_cast<const unsigned short*>(sl + tail_off);
                            v = mg_dot_q6k(wb, A);
                        } else if (type == QT_Q8_0) {
                            const unsigned char* b = sl + sb * 272;
#pragma unroll
                            for (int i = 0; i < 8; i++) wb[i] = lds128(b + hf * 128 + 16 * i);
                            const uint2 dd = *reinterpret_cast<const uint2*>(b + 256 + hf * 8);
                            wb[8].x = dd.x; wb[8].y = dd.y;
                            v = mg_dot_q80(wb, A);
                        } else {   // QT_Q5_K
                            const unsigned char* b = sl + sb * 176;
                            wb[0] = lds128(b); wb[1] = lds128(b + 16); wb[2] = lds128(b + 32);
#pragma unroll
                            for (int i = 0; i < 4; i++) wb[3 + i] = lds128(b + 48 + hf * 64 + 16 * i);
                            v = mg_dot_q5k(wb, hf, A);
                        }
                    }
                    __syncwarp();                             // every lane has read the slot: refill it
                    c_done++;
                    issue_next();
                    if (c == 0) va = v; else vb = v;
                }
                float v0, v1;
                if (rpc == 2) {     // both rows in one chunk: lanes [0, L) row a, [L, 2L) row b
                    v0 = warp_sum(sub == 0 ? va : 0.0f); v1 = warp_sum(sub == 1 ? va : 0.0f);
                } else {            // ONE butterfly for both rows: lanes 0-15 carry row a, lanes 16-31 row b
                    const float oa = __shfl_xor_sync(0xffffffffu, va, 16), ob = __shfl_xor_sync(0xffffffffu, vb, 16);
                    float y = lane < 16 ? va + oa : vb + ob;
#pragma unroll
                    for (int o = 8; o > 0; o >>= 1) y += __shfl_xor_sync(0xffffffffu, y, o);
                    v0 = y; v1 = __shfl_sync(0xffffffffu, y, 16);
                }
                if (lane == 0) S.part[slot_i * MG_WARPS + warp] = make_float2(v0, v1);
            }
        }
        __syncthreads();
        mg_tr<TR>(P, S, trk | 5);
        mg_epilogue(P, ph, phi, pos, S, res, have_res);
        mg_tr<TR>(P, S, trk | 6);
        if (is_qkv) {
            mg_attn_scores<GQ>(P, phi, n_kv, S);
            mg_tr<TR>(P, S, 11);
            mg_attn_pv<GQ, TR>(P, layer, phi, n_kv, S);
            mg_tr<TR>(P, S, 16);
        }
        __syncthreads();                                  // S.part, S.act and the phase descriptor slot are reused by the next phase
    }
    mg_tr<TR>(P, S, 20);
    if (tid == 0 && blockIdx.x == 0 && P.advance_pos) P.pos[0] = pos + 1;
}

} // namespace blk
