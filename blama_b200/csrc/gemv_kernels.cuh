// gemv_kernels.cuh -- the dequant-fused decode mat-vec (templates only; instantiated in gemv_*.cu).
// See decode_kernels.cuh for the rest of the decode path and for the arithmetic contract.
#pragma once
#include <cstdlib>
#include "qweights.cuh"

namespace blk {


constexpr int KV_PAGE = 64;          // tokens per KV page
constexpr int GEMV_THREADS = 256;    // 8 warps per CTA
constexpr int MAX_GQ = 8;            // query heads per KV head (70B: 8, Qwen2.5-7B: 7)
constexpr int TOPK_MAX = 64;

// activations prepared for a quantised mat-vec
struct ActBuf {
    float* f32 = nullptr;     // [K]   (always written: residual / debug / F32 weights)
    int8_t* q = nullptr;      // [K]
    float* d = nullptr;       // [K/256] (Q8_K) or [K/32] (Q8_0; value already rounded through fp16)
    int16_t* bs = nullptr;    // [K/16]  (Q8_K only)
};

__device__ __forceinline__ uint4 ldg_stream(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// rope table: cs[i] = {cos(theta_i), sin(theta_i)}, theta_i = pos * theta_scale^i / freq_factor_i, theta built by
// repeated multiplication exactly as ggml_rope_cache_init does
__device__ inline void rope_table_fill(float2* cs, int half_rot, int pos, float theta_scale, const float* freq_factors) {
    for (int i = threadIdx.x; i < half_rot; i += blockDim.x) {
        float theta = (float)pos;
        for (int k = 0; k < i; k++) theta *= theta_scale;
        const float ff = freq_factors ? freq_factors[i] : 1.0f;
        const float th = theta / ff;
        float s, c; sincosf(th, &s, &c);
        cs[i] = make_float2(c, s);
    }
}

// Programmatic dependent launch (PDL): every kernel of the decode step lets its successor start early
// (launch_dependents) and only blocks (wait) right before it touches data its predecessor produced.  The mat-vecs
// issue all their weight loads BEFORE waiting, so HBM keeps streaming across kernel boundaries.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// =================================================================================================================
// activation quantisation (one warp per 256-element block)
//   Q8_K : upstream ggml-quants.c quantize_row_q8_K_ref   (iscale = -127/max, first max wins, nearest_int)
//   Q8_0 : upstream ggml-quants.c quantize_row_q8_0_ref   (d = amax/127 stored as f16, roundf)
// =================================================================================================================
// One warp quantises one 256-element block.  The values are y[i] (NORM = false) or (y[i] * scale) * w[i] (NORM = true,
// the RMSNorm output); `coherent` reads bypass L1 (data written by other CTAs of the same kernel).
template <bool NORM = false, bool COHERENT = false>
__device__ __forceinline__ void quantize_256_warp(const float* y /*smem or global, 256-aligned block*/, int valid, int fmt,
                                                   int8_t* q, float* dq, int16_t* bs, int blk_index,
                                                   float scale = 1.0f, const float* w = nullptr, float* f32_out = nullptr) {
    const int lane = threadIdx.x & 31;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        float t = 0.0f;
        if (lane * 8 + i < valid) {
            t = COHERENT ? __ldcg(y + lane * 8 + i) : y[lane * 8 + i];
            if (NORM) t = __fmul_rn(__fmul_rn(t, scale), w[lane * 8 + i]);
            if (f32_out) f32_out[lane * 8 + i] = t;
        }
        v[i] = t;
    }
    if (fmt == ACT_F32) return;
    int qi[8];
    if (fmt == ACT_Q8_K) {
        // first element attaining the max |x| decides the sign of the scale
        float amax = 0.0f; int idx = 0x7fffffff;
#pragma unroll
        for (int i = 0; i < 8; i++) { const float ax = fabsf(v[i]); if (ax > amax) { amax = ax; idx = lane * 8 + i; } }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float oa = __shfl_xor_sync(0xffffffffu, amax, o);
            const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
            if (oa > amax || (oa == amax && oi < idx)) { amax = oa; idx = oi; }
        }
        float mx = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; i++) if (lane * 8 + i == idx) mx = v[i];
        mx = __shfl_sync(0xffffffffu, mx, (idx == 0x7fffffff ? 0 : idx) >> 3);
        if (amax == 0.0f) {
#pragma unroll
            for (int i = 0; i < 8; i++) qi[i] = 0;
            if (lane == 0) dq[blk_index] = 0.0f;
        } else {
            const float iscale = __fdiv_rn(-127.0f, mx);
#pragma unroll
            for (int i = 0; i < 8; i++) qi[i] = min(127, __float2int_rn(__fmul_rn(iscale, v[i])));
            if (lane == 0) dq[blk_index] = __fdiv_rn(1.0f, iscale);
        }
        int s = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) s += qi[i];
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        if ((lane & 1) == 0) bs[blk_index * 16 + (lane >> 1)] = (int16_t)s;
    } else {   // ACT_Q8_0: 32-element blocks = 4 lanes
        float amax = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; i++) amax = fmaxf(amax, fabsf(v[i]));
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
        const float d = __fdiv_rn(amax, 127.0f);
        const float id = d != 0.0f ? __fdiv_rn(1.0f, d) : 0.0f;
#pragma unroll
        for (int i = 0; i < 8; i++) qi[i] = (int)roundf(__fmul_rn(v[i], id));
        if ((lane & 3) == 0 && lane * 8 < valid) dq[blk_index * 8 + (lane >> 2)] = __half2float(__float2half_rn(d));
    }
    if (lane * 8 < valid) {
        uint2 pk;
        pk.x = (uint32_t)(qi[0] & 0xff) | ((uint32_t)(qi[1] & 0xff) << 8) | ((uint32_t)(qi[2] & 0xff) << 16) | ((uint32_t)(qi[3] & 0xff) << 24);
        pk.y = (uint32_t)(qi[4] & 0xff) | ((uint32_t)(qi[5] & 0xff) << 8) | ((uint32_t)(qi[6] & 0xff) << 16) | ((uint32_t)(qi[7] & 0xff) << 24);
        *reinterpret_cast<uint2*>(q + lane * 8) = pk;
    }
}


// =================================================================================================================
// dequant-fused mat-vec: one warp owns a PAIR of rows at a time; each lane streams 2 x 128 bit of quantised weights
// per row per step and multiplies them with the int8 activations held in shared memory.
// =================================================================================================================
struct ActView { const int8_t* q; const float* d; const int16_t* bs; const float* f32; };

template <int TYPE> struct RowUnit;
template <> struct RowUnit<QT_Q4_K> {
    uint4 q0, q1, hdr;
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int u) {
        const uint8_t* q = W.p0 + (size_t)row * (W.K >> 1) + (size_t)u * 32;
        q0 = ldg_stream(q); q1 = ldg_stream(q + 16);
        hdr = __ldg(reinterpret_cast<const uint4*>(W.p1 + ((size_t)row * (W.K >> 8) + (u >> 2)) * 16));
    }
    __device__ __forceinline__ float dot(const ActView& A, int u) const {
        const int4* a = reinterpret_cast<const int4*>(A.q + (size_t)u * 64);
        const int4 l0 = a[0], l1 = a[1], h0 = a[2], h1 = a[3];
        int ilo = 0, ihi = 0;
        const uint32_t M = 0x0F0F0F0Fu;
        ilo = __dp4a((int)(q0.x & M), l0.x, ilo); ihi = __dp4a((int)((q0.x >> 4) & M), h0.x, ihi);
        ilo = __dp4a((int)(q0.y & M), l0.y, ilo); ihi = __dp4a((int)((q0.y >> 4) & M), h0.y, ihi);
        ilo = __dp4a((int)(q0.z & M), l0.z, ilo); ihi = __dp4a((int)((q0.z >> 4) & M), h0.z, ihi);
        ilo = __dp4a((int)(q0.w & M), l0.w, ilo); ihi = __dp4a((int)((q0.w >> 4) & M), h0.w, ihi);
        ilo = __dp4a((int)(q1.x & M), l1.x, ilo); ihi = __dp4a((int)((q1.x >> 4) & M), h1.x, ihi);
        ilo = __dp4a((int)(q1.y & M), l1.y, ilo); ihi = __dp4a((int)((q1.y >> 4) & M), h1.y, ihi);
        ilo = __dp4a((int)(q1.z & M), l1.z, ilo); ihi = __dp4a((int)((q1.z >> 4) & M), h1.z, ihi);
        ilo = __dp4a((int)(q1.w & M), l1.w, ilo); ihi = __dp4a((int)((q1.w >> 4) & M), h1.w, ihi);
        uint32_t sc2, mn2; k4_scale_min_pair(hdr, u & 3, sc2, mn2);
        const uint2 bsw = *reinterpret_cast<const uint2*>(A.bs + (size_t)u * 4);   // 4 x int16 sums of 16
        const int blo = (int)(int16_t)(bsw.x & 0xffff) + (int)(int16_t)(bsw.x >> 16);
        const int bhi = (int)(int16_t)(bsw.y & 0xffff) + (int)(int16_t)(bsw.y >> 16);
        const int p = (int)(sc2 & 0xff) * ilo + (int)(sc2 >> 8) * ihi;
        const int pm = (int)(mn2 & 0xff) * blo + (int)(mn2 >> 8) * bhi;
        const float2 dm = hdr_d_dmin(hdr);
        const float ad = A.d[u >> 2];
        return (dm.x * ad) * (float)p - (dm.y * ad) * (float)pm;
    }
};
template <> struct RowUnit<QT_Q5_K> {
    uint4 q0, q1, hdr, h0, h1;
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int u) {
        const uint8_t* q = W.p0 + (size_t)row * (W.K >> 1) + (size_t)u * 32;
        q0 = ldg_stream(q); q1 = ldg_stream(q + 16);
        const size_t sb = (size_t)row * (W.K >> 8) + (u >> 2);
        hdr = __ldg(reinterpret_cast<const uint4*>(W.p1 + sb * 16));
        h0 = __ldg(reinterpret_cast<const uint4*>(W.p2 + sb * 32));
        h1 = __ldg(reinterpret_cast<const uint4*>(W.p2 + sb * 32 + 16));
    }
    __device__ __forceinline__ float dot(const ActView& A, int u) const {
        const int4* a = reinterpret_cast<const int4*>(A.q + (size_t)u * 64);
        const int4 l0 = a[0], l1 = a[1], g0 = a[2], g1 = a[3];
        const int j = u & 3;
        const uint32_t M = 0x0F0F0F0Fu, B = 0x01010101u;
        int ilo = 0, ihi = 0;
#define BLK_Q5_STEP(QW, HW, AL, AH)                                                                  \
        ilo = __dp4a((int)(((QW) & M) | ((((HW) >> (2 * j)) & B) << 4)), (AL), ilo);                 \
        ihi = __dp4a((int)((((QW) >> 4) & M) | ((((HW) >> (2 * j + 1)) & B) << 4)), (AH), ihi);
        BLK_Q5_STEP(q0.x, h0.x, l0.x, g0.x) BLK_Q5_STEP(q0.y, h0.y, l0.y, g0.y)
        BLK_Q5_STEP(q0.z, h0.z, l0.z, g0.z) BLK_Q5_STEP(q0.w, h0.w, l0.w, g0.w)
        BLK_Q5_STEP(q1.x, h1.x, l1.x, g1.x) BLK_Q5_STEP(q1.y, h1.y, l1.y, g1.y)
        BLK_Q5_STEP(q1.z, h1.z, l1.z, g1.z) BLK_Q5_STEP(q1.w, h1.w, l1.w, g1.w)
#undef BLK_Q5_STEP
        uint32_t sc2, mn2; k4_scale_min_pair(hdr, j, sc2, mn2);
        const uint2 bsw = *reinterpret_cast<const uint2*>(A.bs + (size_t)u * 4);
        const int blo = (int)(int16_t)(bsw.x & 0xffff) + (int)(int16_t)(bsw.x >> 16);
        const int bhi = (int)(int16_t)(bsw.y & 0xffff) + (int)(int16_t)(bsw.y >> 16);
        const int p = (int)(sc2 & 0xff) * ilo + (int)(sc2 >> 8) * ihi;
        const int pm = (int)(mn2 & 0xff) * blo + (int)(mn2 >> 8) * bhi;
        const float2 dm = hdr_d_dmin(hdr);
        const float ad = A.d[u >> 2];
        return (dm.x * ad) * (float)p - (dm.y * ad) * (float)pm;
    }
};
template <> struct RowUnit<QT_Q6_K> {
    uint4 l0, l1, h; uint2 sc; uint16_t dh;
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int u) {
        const int s = u >> 2, hh = (u >> 1) & 1, t = u & 1;
        const uint8_t* ql = W.p0 + (size_t)row * (W.K >> 1) + (size_t)s * 128 + hh * 64 + t * 16;
        l0 = ldg_stream(ql); l1 = ldg_stream(ql + 32);
        h = ldg_stream(W.p1 + (size_t)row * (W.K >> 2) + (size_t)s * 64 + hh * 32 + t * 16);
        sc = __ldg(reinterpret_cast<const uint2*>(W.p2 + (size_t)row * (W.K >> 4) + s * 16 + hh * 8));
        dh = __ldg(reinterpret_cast<const uint16_t*>(W.p3) + (size_t)row * (W.K >> 8) + s);
    }
    __device__ __forceinline__ float dot(const ActView& A, int u) const {
        const int s = u >> 2, hh = (u >> 1) & 1, t = u & 1;
        const int e0 = 256 * s + 128 * hh + 16 * t;
        const int4 a0 = *reinterpret_cast<const int4*>(A.q + e0);
        const int4 a1 = *reinterpret_cast<const int4*>(A.q + e0 + 32);
        const int4 a2 = *reinterpret_cast<const int4*>(A.q + e0 + 64);
        const int4 a3 = *reinterpret_cast<const int4*>(A.q + e0 + 96);
        const uint32_t M = 0x0F0F0F0Fu, H = 0x30303030u;
        int i0 = 0, i1 = 0, i2 = 0, i3 = 0;
#define BLK_Q6_STEP(LA, LB, HW, A0, A1, A2, A3)                                     \
        i0 = __dp4a((int)(((LA) & M) | (((HW) << 4) & H)), (A0), i0);               \
        i1 = __dp4a((int)(((LB) & M) | (((HW) << 2) & H)), (A1), i1);               \
        i2 = __dp4a((int)((((LA) >> 4) & M) | ((HW) & H)), (A2), i2);               \
        i3 = __dp4a((int)((((LB) >> 4) & M) | (((HW) >> 2) & H)), (A3), i3);
        BLK_Q6_STEP(l0.x, l1.x, h.x, a0.x, a1.x, a2.x, a3.x)
        BLK_Q6_STEP(l0.y, l1.y, h.y, a0.y, a1.y, a2.y, a3.y)
        BLK_Q6_STEP(l0.z, l1.z, h.z, a0.z, a1.z, a2.z, a3.z)
        BLK_Q6_STEP(l0.w, l1.w, h.w, a0.w, a1.w, a2.w, a3.w)
#undef BLK_Q6_STEP
        // 16-element sums of the activations give the "-32" offset: sum (q-32) a = sum q a - 32 sum a
        const int bi = 16 * s + 8 * hh + t;
        const int b0 = A.bs[bi], b1 = A.bs[bi + 2], b2 = A.bs[bi + 4], b3 = A.bs[bi + 6];
        const uint32_t sl = t ? (sc.x >> 8) : sc.x, sh = t ? (sc.y >> 8) : sc.y;   // bytes t, t+2 | t+4, t+6
        const int s0 = (int)(int8_t)(sl & 0xff), s1 = (int)(int8_t)((sl >> 16) & 0xff);
        const int s2 = (int)(int8_t)(sh & 0xff), s3 = (int)(int8_t)((sh >> 16) & 0xff);
        const int p = s0 * (i0 - 32 * b0) + s1 * (i1 - 32 * b1) + s2 * (i2 - 32 * b2) + s3 * (i3 - 32 * b3);
        const float d = __half2float(__ushort_as_half(dh));
        return (d * A.d[s]) * (float)p;
    }
};
template <> struct RowUnit<QT_Q8_0> {
    uint4 q0, q1; uint16_t dh;
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int u) {
        const uint8_t* q = W.p0 + (size_t)row * W.K + (size_t)u * 32;
        q0 = ldg_stream(q); q1 = ldg_stream(q + 16);
        dh = __ldg(reinterpret_cast<const uint16_t*>(W.p1) + (size_t)row * (W.K >> 5) + u);
    }
    __device__ __forceinline__ float dot(const ActView& A, int u) const {
        const int4* a = reinterpret_cast<const int4*>(A.q + (size_t)u * 32);
        const int4 a0 = a[0], a1 = a[1];
        int i = 0;
        i = __dp4a((int)q0.x, a0.x, i); i = __dp4a((int)q0.y, a0.y, i); i = __dp4a((int)q0.z, a0.z, i); i = __dp4a((int)q0.w, a0.w, i);
        i = __dp4a((int)q1.x, a1.x, i); i = __dp4a((int)q1.y, a1.y, i); i = __dp4a((int)q1.z, a1.z, i); i = __dp4a((int)q1.w, a1.w, i);
        return (float)i * (__half2float(__ushort_as_half(dh)) * A.d[u]);
    }
};
template <> struct RowUnit<QT_F32> {
    float4 w0, w1;
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int u) {
        const float4* p = reinterpret_cast<const float4*>(W.p0) + ((size_t)row * W.K + (size_t)u * 8) / 4;
        w0 = __ldg(p); w1 = __ldg(p + 1);
    }
    __device__ __forceinline__ float dot(const ActView& A, int u) const {
        const float4* x = reinterpret_cast<const float4*>(A.f32 + (size_t)u * 8);
        const float4 x0 = x[0], x1 = x[1];
        return w0.x * x0.x + w0.y * x0.y + w0.z * x0.z + w0.w * x0.w + w1.x * x1.x + w1.y * x1.y + w1.z * x1.z + w1.w * x1.w;
    }
};
template <> struct RowUnit<QT_F16> {
    uint4 w;
    __device__ __forceinline__ void load(const QMat& W, int64_t row, int u) {
        w = __ldg(reinterpret_cast<const uint4*>(W.p0 + ((size_t)row * W.K + (size_t)u * 8) * 2));
    }
    __device__ __forceinline__ float dot(const ActView& A, int u) const {
        // ggml converts the activations to f16 for F16 weights (vec_dot_type F16) and accumulates in f32
        const float* x = A.f32 + (size_t)u * 8;
        const __half2* h = reinterpret_cast<const __half2*>(&w);
        float acc = 0.0f;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float2 wf = __half22float2(h[i]);
            acc += wf.x * __half2float(__float2half_rn(x[2 * i])) + wf.y * __half2float(__float2half_rn(x[2 * i + 1]));
        }
        return acc;
    }
};

// one K-slice (U units per lane) of two rows (possibly of two different matrices of the same type) against the same
// activations.  load() issues all 2*U weight loads of the lane; dot() consumes them once the activations exist.
template <int TYPE, int U>
struct PairSlice {
    RowUnit<TYPE> ua[U], ub[U];
    __device__ __forceinline__ void load(const QMat& Wa, int64_t ra, const QMat& Wb, int64_t rb, int u0, int units) {
        const int lane = threadIdx.x & 31;
#pragma unroll
        for (int i = 0; i < U; i++) {
            const int u = u0 + i * 32 + lane;
            if (u < units) { ua[i].load(Wa, ra, u); ub[i].load(Wb, rb, u); }
        }
    }
    __device__ __forceinline__ void dot(const ActView& A, int u0, int units, float& oa, float& ob) const {
        const int lane = threadIdx.x & 31;
        float sa = 0.0f, sb = 0.0f;
#pragma unroll
        for (int i = 0; i < U; i++) {
            const int u = u0 + i * 32 + lane;
            if (u < units) { sa += ua[i].dot(A, u); sb += ub[i].dot(A, u); }
        }
        oa = warp_sum(sa); ob = warp_sum(sb);
    }
};

enum : int { EPI_STORE = 0, EPI_RESID = 1, EPI_QKV = 2, EPI_SWIGLU = 3 };

struct GemvSeg {
    QMat W;                 // rows of this segment
    const float* bias;      // optional [N]
    int pair0;              // first pair index of this segment
    int kind;               // EPI_QKV only: 0 = q, 1 = k, 2 = v
};

// Work fused behind the lm_head mat-vec: per-chunk maxima of the logits for the threshold top-k (decode_kernels.cuh)
enum : int { TAIL_NONE = 0, TAIL_CHUNKMAX = 3 };
struct GemvTail {
    int kind = TAIL_NONE;
    int* chunk_max = nullptr;   // order-preserving int encoding of the per-chunk max logit (atomicMax)
    int chunk_shift = 10;       // log2(chunk size)
};

__device__ __forceinline__ int float_order_key(float f) { const int i = __float_as_int(f); return i >= 0 ? i : (i ^ 0x7fffffff); }
__device__ __forceinline__ float float_from_order_key(int k) { return __int_as_float(k >= 0 ? k : (k ^ 0x7fffffff)); }

struct GemvArgs {
    GemvTail tail;
    GemvSeg seg[3];
    int nseg;
    int total_pairs;
    ActBuf act;             // global-memory activations (prepared by act_prepare_kernel)
    int act_fmt;
    float* out;             // EPI_STORE / EPI_RESID / EPI_SWIGLU destination; EPI_QKV: q vector [n_head*d_head] f32
    // EPI_QKV
    int d_head, neox;
    const float2* rope_cs;  // [d_head/2] {cos, sin} of this step's position
    const int32_t* pos;     // device scalar: position of the token being decoded
    __half* k_pool; __half* v_pool;   // this layer's KV pages [n_pages][KV_PAGE][n_kv*d_head]
    const int32_t* page_table;
    int kv_dim;             // n_head_kv * d_head
};

// Mat-vec kernel.  A CTA of 8 warps handles G = 8/S row pairs, each pair split along K into S slices of 32*U units
// (one warp per slice); slice partials meet in shared memory and are added in slice order (deterministic).  There is
// no loop: every lane issues all of its weight loads up front, so the whole matrix is in flight at once and the grid
// (pairs/G CTAs) load-balances itself.  Activations (int8 + scales, a few KB) are read through L1 straight from global.
//   TA = weight type of segments 0 and 1 (q,k | gate,up | the single matrix), TB = type of segment 2 (v).
template <int EPI, int TA, int TB, int U>
__global__ void __launch_bounds__(GEMV_THREADS) gemv_pairs_kernel(const GemvArgs a, const int S) {
    __shared__ float part[GEMV_THREADS / 32][2];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int G = (GEMV_THREADS / 32) / S;
    const int g = w / S, ks = w % S;
    const int pair = blockIdx.x * G + g;
    const bool valid = pair < a.total_pairs;
    const ActView A{a.act.q, a.act.d, a.act.bs, a.act.f32};
    float v0 = 0.0f, v1 = 0.0f;
    int r0 = 0, r1 = 0, si = 0;
    float res0 = 0.0f, res1 = 0.0f;
    pdl_launch_dependents();
    if (EPI == EPI_SWIGLU) {
        r0 = r1 = pair;
        const int units = a.seg[0].W.K / qmat_unit_elems(TA);
        PairSlice<TA, U> ps;
        if (valid) ps.load(a.seg[0].W, pair, a.seg[1].W, pair, ks * 32 * U, units);
        pdl_wait();
        if (valid) ps.dot(A, ks * 32 * U, units, v0, v1);
    } else {
        if (a.nseg > 1 && pair >= a.seg[1].pair0) si = 1;
        if (a.nseg > 2 && pair >= a.seg[2].pair0) si = 2;
        const GemvSeg& Sg = a.seg[si];
        const int p = pair - Sg.pair0;
        r0 = 2 * p; r1 = 2 * p + 1;
        if (EPI == EPI_QKV && a.neox && Sg.kind != 2) {
            const int hd = a.d_head >> 1;
            r0 = (p / hd) * a.d_head + (p % hd); r1 = r0 + hd;
        }
        if (TA != TB && si == 2) {
            const int units = Sg.W.K / qmat_unit_elems(TB);
            PairSlice<TB, U> ps;
            if (valid) ps.load(Sg.W, r0, Sg.W, r1, ks * 32 * U, units);
            pdl_wait();
            if (valid) ps.dot(A, ks * 32 * U, units, v0, v1);
        } else {
            const int units = Sg.W.K / qmat_unit_elems(TA);
            PairSlice<TA, U> ps;
            if (valid) ps.load(Sg.W, r0, Sg.W, r1, ks * 32 * U, units);
            pdl_wait();
            if (EPI == EPI_RESID && valid && ks == 0 && lane == 0) { res0 = a.out[r0]; res1 = a.out[r1]; }
            if (valid) ps.dot(A, ks * 32 * U, units, v0, v1);
        }
    }
    if (S > 1) {
        if (lane == 0) { part[w][0] = v0; part[w][1] = v1; }
        __syncthreads();
        if (ks == 0) {
            v0 = part[w][0]; v1 = part[w][1];
            for (int k = 1; k < S; k++) { v0 += part[w + k][0]; v1 += part[w + k][1]; }
        }
    }
    const bool writer = (S == 1 || ks == 0);
    if (valid && lane == 0 && writer) {
        if (EPI == EPI_SWIGLU) { a.out[pair] = (v0 / (1.0f + expf(-v0))) * v1; }     // ggml_silu_f32 then ggml_mul
        else {
            const GemvSeg& Sg = a.seg[si];
            if (Sg.bias) { v0 += Sg.bias[r0]; v1 += Sg.bias[r1]; }
            if (EPI == EPI_STORE) {
                a.out[r0] = v0; a.out[r1] = v1;
                if (a.tail.kind == TAIL_CHUNKMAX) atomicMax(a.tail.chunk_max + (r0 >> a.tail.chunk_shift), float_order_key(fmaxf(v0, v1)));
            }
            else if (EPI == EPI_RESID) { a.out[r0] = res0 + v0; a.out[r1] = res1 + v1; }
            else if (EPI == EPI_QKV) {
                if (Sg.kind != 2) {     // rotary embedding on the (r0, r1) pair: ggml rope NORM / NEOX
                    const int i = a.neox ? (r0 % a.d_head) : ((r0 % a.d_head) >> 1);
                    const float2 cs = a.rope_cs[i];
                    const float x0 = v0, x1 = v1;
                    v0 = x0 * cs.x - x1 * cs.y;
                    v1 = x0 * cs.y + x1 * cs.x;
                }
                if (Sg.kind == 0) { a.out[r0] = v0; a.out[r1] = v1; }
                else {
                    const int pos = a.pos[0];
                    const size_t base = ((size_t)a.page_table[pos / KV_PAGE] * KV_PAGE + (pos % KV_PAGE)) * a.kv_dim;
                    __half* dst = (Sg.kind == 1) ? a.k_pool : a.v_pool;
                    dst[base + r0] = __float2half_rn(v0);      // ggml_cpy f32 -> f16 into the cache
                    dst[base + r1] = __float2half_rn(v1);
                }
            }
        }
    }
}

// launch with the programmatic-stream-serialization attribute (PDL edge to the previous kernel in the stream / graph)
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// the kernels of the multi-token chain (RMSNorm, GEMM, split-K reduce, RoPE / KV write, V transpose, attention): every one executes
// griddepcontrol.wait before its first global access and releases its dependents at its start, so the next kernel's launch latency and
// prologue (barrier initialisation, TMEM allocation) hide under the tail of the current one.  Measured on the 8B model: a 32-token
// prompt 4.71 -> 4.01 ms, 512 tokens 8.84 -> 8.36, a 32-row batched decode step 5.14 -> 4.67 ms; at 2048 tokens nothing (28.3-29.5 ms
// either way, if anything slower), so a pass switches it on only up to CHAIN_PDL_MAX_TOKENS (ChainPdl scope, per host thread).
constexpr int CHAIN_PDL_MAX_TOKENS = 1024;
inline bool& chain_pdl_flag() { static thread_local bool on = false; return on; }
struct ChainPdl {      // RAII: the launches of this host thread inside the scope are programmatic dependents of their predecessors
    bool prev;
    explicit ChainPdl(int n_tokens) : prev(chain_pdl_flag()) { chain_pdl_flag() = n_tokens <= CHAIN_PDL_MAX_TOKENS; }
    ~ChainPdl() { chain_pdl_flag() = prev; }
};
template <class... KArgs, class... Args>
inline cudaError_t launch_chain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    if (chain_pdl_flag()) return launch_pdl(kernel, grid, block, smem, st, args...);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// same, as a thread-block cluster of `cluster` CTAs
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, int cluster, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = (unsigned)cluster; attr[1].val.clusterDim.y = 1; attr[1].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 2;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// host-side launch helpers (one translation unit per epilogue so the instantiations compile in parallel)
struct GemvPlan { int U; int S; int ctas; };
inline GemvPlan gemv_plan(int K, int type, int total_pairs) {
    const int units = K / qmat_unit_elems(type);
    GemvPlan p{1, 1, 0};
    const int per_lane = (units + 31) / 32;
    if (per_lane <= 1) { p.U = 1; p.S = 1; }
    else if (per_lane <= 2) { p.U = 2; p.S = 1; }
    else if (per_lane <= 4) { p.U = 2; p.S = 2; }
    else if (per_lane <= 8) { p.U = 2; p.S = 4; }
    else if (per_lane <= 16) { p.U = 2; p.S = 8; }
    else if (per_lane <= 24) { p.U = 3; p.S = 8; }
    else if (per_lane <= 32) { p.U = 4; p.S = 8; }
    else { p.U = 0; }
    const int G = (GEMV_THREADS / 32) / p.S;
    p.ctas = (total_pairs + G - 1) / G;
    return p;
}
// implemented in gemv_*.cu; return cudaError of the launch, or cudaErrorInvalidValue when no instantiation exists
cudaError_t launch_gemv_store(const GemvArgs& a, cudaStream_t st);
cudaError_t launch_gemv_resid(const GemvArgs& a, cudaStream_t st);
cudaError_t launch_gemv_qkv(const GemvArgs& a, cudaStream_t st);
cudaError_t launch_gemv_swiglu(const GemvArgs& a, cudaStream_t st);


} // namespace blk
