// decode_kernels.cuh -- batch-1 decode path (Session::getToken -> llama_decode(1 token), reference
// inference/code/llama/Session.cpp:169-190, 395-401) as hand-written sm_100a kernels.
//
// Arithmetic follows the reference's CPU backend (upstream ggml-cpu): the activation vector of every W.x is
// quantised row-wise to Q8_K (K-quant weights) or Q8_0 (Q8_0 weights) and multiplied with the still-quantised weights
// through integer dot products (dp4a) whose partial sums are scaled in fp32.  All integer partial sums are therefore
// bit-identical to ggml_vec_dot_q4_K_q8_K & co; only the order of the fp32 additions differs.
//
// All kernels here are HBM-bound byte/integer work: coalesced 128-bit loads (two per lane per step), warp-shuffle
// reductions, grids sized in multiples of the SM count.  No tensor cores (SURVEY.md section 8d: decode -> HBM roofline).
#pragma once
#include <cooperative_groups.h>
#include "gemv_kernels.cuh"

namespace blk {

// =================================================================================================================
// weight re-tiling (load time): ggml blocks -> split planes (qweights.cuh)
// =================================================================================================================
__global__ void retile_q4k_kernel(const uint8_t* __restrict__ src, uint8_t* qs, uint8_t* hdr, int64_t nblk) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk) return;
    const uint8_t* s = src + b * 144;
    for (int i = 0; i < 16; i++) hdr[b * 16 + i] = s[i];
    for (int i = 0; i < 128; i++) qs[b * 128 + i] = s[16 + i];
}
__global__ void retile_q5k_kernel(const uint8_t* __restrict__ src, uint8_t* qs, uint8_t* hdr, uint8_t* qh, int64_t nblk) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk) return;
    const uint8_t* s = src + b * 176;
    for (int i = 0; i < 16; i++) hdr[b * 16 + i] = s[i];
    for (int i = 0; i < 32; i++) qh[b * 32 + i] = s[16 + i];
    for (int i = 0; i < 128; i++) qs[b * 128 + i] = s[48 + i];
}
__global__ void retile_q6k_kernel(const uint8_t* __restrict__ src, uint8_t* ql, uint8_t* qh, uint8_t* sc, uint8_t* d, int64_t nblk) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk) return;
    const uint8_t* s = src + b * 210;
    for (int i = 0; i < 128; i++) ql[b * 128 + i] = s[i];
    for (int i = 0; i < 64; i++) qh[b * 64 + i] = s[128 + i];
    for (int i = 0; i < 16; i++) sc[b * 16 + i] = s[192 + i];
    d[b * 2] = s[208]; d[b * 2 + 1] = s[209];
}
__global__ void retile_q80_kernel(const uint8_t* __restrict__ src, uint8_t* qs, uint8_t* d, int64_t nblk) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk) return;
    const uint8_t* s = src + b * 34;
    d[b * 2] = s[0]; d[b * 2 + 1] = s[1];
    for (int i = 0; i < 32; i++) qs[b * 32 + i] = s[2 + i];
}

// =================================================================================================================
// embedding gather (get_rows with dequant) + per-step RoPE table
// =================================================================================================================
// grid = n_tok CTAs.  x[t] = dequant(token_embd[tok[t]]); CTA 0.. also fill the rope table rows for their token
__global__ void embed_kernel(QMat E, const int32_t* __restrict__ tokens, const int32_t* __restrict__ pos0, float* x,
                             float2* rope_cs, int half_rot, float theta_scale, const float* freq_factors) {
    pdl_launch_dependents(); pdl_wait();
    const int t = blockIdx.x;
    dequant_row_cta(E, tokens[t], x + (size_t)t * E.K);
    rope_table_fill(rope_cs + (size_t)t * half_rot, half_rot, pos0[0] + pos0[1] + t, theta_scale, freq_factors);      // pos0 = {cell index, rotary offset}
}

// =================================================================================================================
// activation preparation: (optional RMSNorm * weight) -> f32 copy + Q8_K / Q8_0 quantisation
//   rms_norm: upstream ggml-cpu ops.cpp ggml_compute_forward_rms_norm_f32 (row sum of squares in double)
//   Q8_K    : upstream ggml-quants.c quantize_row_q8_K_ref   (iscale = -127/max, first max wins, nearest_int)
//   Q8_0    : upstream ggml-quants.c quantize_row_q8_0_ref   (d = amax/127 stored as f16, roundf)
// grid = n_rows (tokens), block = 512.  K % 32 == 0.
// =================================================================================================================
template <bool NORM>
__global__ void __launch_bounds__(512) act_prepare_kernel(const float* __restrict__ x, const float* __restrict__ w, int K, float eps,
                                                          int fmt, ActBuf out, int64_t row_stride_q, int64_t row_stride_d, int64_t row_stride_bs) {
    pdl_launch_dependents(); pdl_wait();
    // row-strided outputs so the same kernel serves the batch (prefill) case: row = blockIdx.x
    const int row = blockIdx.x;
    x += (size_t)row * K;
    float* of = out.f32 ? out.f32 + (size_t)row * K : nullptr;
    int8_t* oq = out.q ? out.q + (size_t)row * row_stride_q : nullptr;
    float* od = out.d ? out.d + (size_t)row * row_stride_d : nullptr;
    int16_t* ob = out.bs ? out.bs + (size_t)row * row_stride_bs : nullptr;
    __shared__ double red[16];
    __shared__ float s_scale;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    float scale = 1.0f;
    if (NORM) {
        double sum = 0.0;
        for (int i = tid; i < K; i += 512) { const float v = x[i]; sum += (double)__fmul_rn(v, v); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) red[wid] = sum;
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0;
            for (int i = 0; i < 16; i++) tot += red[i];
            const float mean = (float)(tot / (double)K);
            s_scale = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(mean, eps)));
        }
        __syncthreads();
        scale = s_scale;
    }
    extern __shared__ float ybuf[];   // [K] normalised row
    for (int i = tid; i < K; i += 512) {
        float v = x[i];
        if (NORM) v = __fmul_rn(__fmul_rn(v, scale), w[i]);
        ybuf[i] = v;
        if (of) of[i] = v;
    }
    __syncthreads();
    if (fmt == ACT_F32) return;
    const int nblk = (K + 255) >> 8;
    for (int b = wid; b < nblk; b += 16)
        quantize_256_warp(ybuf + b * 256, min(256, K - b * 256), fmt, oq + b * 256, od, ob, b);
}

// =================================================================================================================
// decode attention over the paged f16 KV cache, split along the context.
//   follows llama-graph.cpp build_attn_mha with flash_attn = false, in ggml's own order of operations:
//     kq = K.q (q rounded to f16, f32 accumulate) * scale ; soft_max_ext: max, expf, sum in double, p = e * (1/sum) ;
//     p rounded to f16 ; out = V.p (f32 accumulate).
//   The probabilities must be normalised BEFORE the f16 rounding: the Q8_K quantisation that follows amplifies a
//   2^-11 relative change of the attention output into ~0.1 logit differences.
//   kernel 1 (scores): grid (n_head_kv, n_split), block d_head: thread = token; writes scaled scores.
//   kernel 2 (pv)    : grid (n_head_kv, n_split), block d_head: every CTA reduces max / sum over the whole row
//                      (scores are L2 resident), then its own token slice: thread = output dim.
//   kernel 3 (combine): sums the split partials in fixed order and quantises for the Wo mat-vec.
// =================================================================================================================
struct AttnArgs {
    const float* q;            // [n_head][d_head] f32 (post-RoPE)
    const __half* k_pool; const __half* v_pool; const int32_t* page_table;
    const int32_t* pos;        // device scalar: n_kv = pos + 1
    int n_head, n_head_kv, d_head, kv_dim, n_split;
    float scale;
    float* scores;             // [n_head][score_stride]
    int score_stride;
    float* part_o;             // [n_head][n_split][d_head]
};

template <int DH>
__global__ void __launch_bounds__(DH) attn_scores_kernel(const AttnArgs a) {
    pdl_launch_dependents(); pdl_wait();
    const int hk = blockIdx.x, split = blockIdx.y, tid = threadIdx.x;
    const int gq = a.n_head / a.n_head_kv;
    const int n_kv = a.pos[0] + 1;
    const int per = (n_kv + a.n_split - 1) / a.n_split;
    const int t_begin = split * per, t_end = min(n_kv, t_begin + per);
    if (t_begin >= t_end) return;
    __shared__ __half sq[MAX_GQ * DH];
    for (int i = tid; i < gq * DH; i += DH) sq[i] = __float2half_rn(a.q[(size_t)(hk * gq) * DH + i]);
    __syncthreads();
    for (int t = t_begin + tid; t < t_end; t += DH) {
        const __half* kr = a.k_pool + ((size_t)a.page_table[t / KV_PAGE] * KV_PAGE + (t % KV_PAGE)) * a.kv_dim + (size_t)hk * DH;
        float s[MAX_GQ];
#pragma unroll
        for (int g = 0; g < MAX_GQ; g++) s[g] = 0.0f;
#pragma unroll 4
        for (int c = 0; c < DH / 8; c++) {
            const uint4 kv = *reinterpret_cast<const uint4*>(kr + c * 8);
            const __half2* kh = reinterpret_cast<const __half2*>(&kv);
            float kf[8];
#pragma unroll
            for (int i = 0; i < 4; i++) { const float2 f = __half22float2(kh[i]); kf[2 * i] = f.x; kf[2 * i + 1] = f.y; }
#pragma unroll
            for (int g = 0; g < MAX_GQ; g++) if (g < gq) {
                const __half2* qh = reinterpret_cast<const __half2*>(sq + g * DH + c * 8);
#pragma unroll
                for (int i = 0; i < 4; i++) { const float2 f = __half22float2(qh[i]); s[g] += kf[2 * i] * f.x; s[g] += kf[2 * i + 1] * f.y; }
            }
        }
#pragma unroll
        for (int g = 0; g < MAX_GQ; g++) if (g < gq) a.scores[(size_t)(hk * gq + g) * a.score_stride + t] = __fmul_rn(s[g], a.scale);
    }
}

template <int DH>
__global__ void __launch_bounds__(DH) attn_pv_kernel(const AttnArgs a) {
    pdl_launch_dependents(); pdl_wait();
    const int hk = blockIdx.x, split = blockIdx.y, tid = threadIdx.x;
    const int gq = a.n_head / a.n_head_kv;
    const int n_kv = a.pos[0] + 1;
    const int per = (n_kv + a.n_split - 1) / a.n_split;
    const int t_begin = split * per, t_end = min(n_kv, t_begin + per);
    const int lane = tid & 31, wid = tid >> 5;
    constexpr int NW = DH / 32;
    float* po = a.part_o + ((size_t)(hk * gq) * a.n_split + split) * DH;
    if (t_begin >= t_end) {
        for (int g = 0; g < gq; g++) po[(size_t)g * a.n_split * DH + tid] = 0.0f;
        return;
    }
    __shared__ float sred[MAX_GQ][NW];
    __shared__ double dred[MAX_GQ][NW];
    __shared__ float sp[MAX_GQ][DH];
    float M[MAX_GQ], inv[MAX_GQ];
    // row max
#pragma unroll
    for (int g = 0; g < MAX_GQ; g++) if (g < gq) {
        const float* sr = a.scores + (size_t)(hk * gq + g) * a.score_stride;
        float mx = -INFINITY;
        for (int t = tid; t < n_kv; t += DH) mx = fmaxf(mx, sr[t]);
        mx = warp_max(mx);
        if (lane == 0) sred[g][wid] = mx;
    }
    __syncthreads();
#pragma unroll
    for (int g = 0; g < MAX_GQ; g++) if (g < gq) {
        float mx = sred[g][0];
#pragma unroll
        for (int w = 1; w < NW; w++) mx = fmaxf(mx, sred[g][w]);
        M[g] = mx;
    }
    // row sum of expf(s - max) in double (ggml_float)
#pragma unroll
    for (int g = 0; g < MAX_GQ; g++) if (g < gq) {
        const float* sr = a.scores + (size_t)(hk * gq + g) * a.score_stride;
        double sum = 0.0;
        for (int t = tid; t < n_kv; t += DH) sum += (double)expf(sr[t] - M[g]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) dred[g][wid] = sum;
    }
    __syncthreads();
#pragma unroll
    for (int g = 0; g < MAX_GQ; g++) if (g < gq) {
        double sum = 0.0;
#pragma unroll
        for (int w = 0; w < NW; w++) sum += dred[g][w];
        inv[g] = (float)(1.0 / sum);
    }
    float acc[MAX_GQ];
#pragma unroll
    for (int g = 0; g < MAX_GQ; g++) acc[g] = 0.0f;
    for (int t0 = t_begin; t0 < t_end; t0 += DH) {
        const int t = t0 + tid;
#pragma unroll
        for (int g = 0; g < MAX_GQ; g++) if (g < gq) {
            float p = 0.0f;
            if (t < t_end) p = __fmul_rn(expf(a.scores[(size_t)(hk * gq + g) * a.score_stride + t] - M[g]), inv[g]);
            sp[g][tid] = __half2float(__float2half_rn(p));
        }
        __syncthreads();
        const int nt = min(DH, t_end - t0);
        for (int j = 0; j < nt; j++) {
            const int tj = t0 + j;
            const float v = __half2float(a.v_pool[((size_t)a.page_table[tj / KV_PAGE] * KV_PAGE + (tj % KV_PAGE)) * a.kv_dim + (size_t)hk * DH + tid]);
#pragma unroll
            for (int g = 0; g < MAX_GQ; g++) if (g < gq) acc[g] += sp[g][j] * v;
        }
        __syncthreads();
    }
#pragma unroll
    for (int g = 0; g < MAX_GQ; g++) if (g < gq) po[(size_t)g * a.n_split * DH + tid] = acc[g];
}

// -----------------------------------------------------------------------------------------------------------------
// Single-kernel decode attention: one thread-block CLUSTER per KV head, the context split across the cluster's CTAs,
// the cross-CTA reductions (row max, row sum, output) done through distributed shared memory.  Same arithmetic order as
// the three-kernel path above (max -> expf -> sum in double -> p = e * (1/sum) -> f16 -> V.p), but the scores never leave
// shared memory and there is one launch instead of three.
//   grid = n_head_kv * CS CTAs (cluster dims (CS,1,1)), block = 128 threads, dynamic smem = gq * cap * 4 bytes (scores)
// -----------------------------------------------------------------------------------------------------------------
struct AttnClusterArgs {
    const float* q; const __half* k_pool; const __half* v_pool; const int32_t* page_table; const int32_t* pos;
    int n_head, n_head_kv, kv_dim, cap;      // cap = tokens of the context one CTA can hold scores for
    float scale;
    float* out;                              // [n_head * d_head] f32 attention output
};

constexpr int ATTN_THREADS = 512;
constexpr int ATTN_CLUSTER_PAGES = 512;      // KV pages one CTA's token slice may span (s_page below)

template <int DH, int GQ>      // GQ = compile-time bound on query heads per KV head (4 or 8)
__global__ void __launch_bounds__(ATTN_THREADS) attn_cluster_kernel(const AttnClusterArgs a) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    pdl_launch_dependents(); pdl_wait();
    constexpr int NW = ATTN_THREADS / 32;
    extern __shared__ float s_sc[];                  // [gq][cap] scores, then [NW][gq][DH] per-warp partial outputs
    __shared__ __half sq[GQ * DH];
    __shared__ float c_max[GQ];                      // read by the other CTAs of the cluster
    __shared__ double c_sum[GQ];                     //   "
    __shared__ float c_out[GQ * DH];                 //   "   this CTA's partial V.p
    __shared__ float s_M[GQ], s_inv[GQ];
    __shared__ float red_f[GQ][NW];
    __shared__ double red_d[GQ][NW];
    // The slice's physical page numbers.  Nothing here checks the slice length: the host plan (plan_decode_attn in engine.cu) picks
    // this kernel only when cap tokens starting anywhere inside a page span at most ATTN_CLUSTER_PAGES pages, i.e.
    // cap <= (ATTN_CLUSTER_PAGES - 1) * KV_PAGE + 1.  Longer slices (MHA models at contexts above ~262k cells) take the split form.
    __shared__ int s_page[ATTN_CLUSTER_PAGES];

    const int CS = (int)cluster.num_blocks(), r = (int)cluster.block_rank();
    const int hk = blockIdx.x / CS, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int gq = a.n_head / a.n_head_kv;
    float* red_o = s_sc + (size_t)gq * a.cap;        // [NW][gq][DH]
    const int n_kv = a.pos[0] + 1;
    const int per = (n_kv + CS - 1) / CS;
    const int t0 = r * per, t1 = min(n_kv, t0 + per);
    const int nt = max(0, t1 - t0);
    for (int i = tid; i < gq * DH; i += ATTN_THREADS) sq[i] = __float2half_rn(a.q[(size_t)(hk * gq) * DH + i]);
    // physical pages of this CTA's token slice (removes a dependent global load from every K / V row address)
    const int pg0 = t0 / KV_PAGE;
    const int npg = nt > 0 ? (t1 - 1) / KV_PAGE - pg0 + 1 : 0;
    for (int i = tid; i < npg && i < ATTN_CLUSTER_PAGES; i += ATTN_THREADS) s_page[i] = a.page_table[pg0 + i];
    __syncthreads();
    auto row_off = [&](int t) -> size_t { return ((size_t)s_page[t / KV_PAGE - pg0] * KV_PAGE + (t % KV_PAGE)) * a.kv_dim + (size_t)hk * DH; };

    // ---- 1. scores: 4 lanes per token, each a quarter of the head dim; local row max ----
    constexpr int QD = DH / 4;                       // dims per lane
    float lmax[GQ];
#pragma unroll
    for (int g = 0; g < GQ; g++) lmax[g] = -INFINITY;
    const int qd = tid & 3;
    for (int tl0 = 0; tl0 < nt; tl0 += ATTN_THREADS / 4) {
        const int tl = tl0 + (tid >> 2);
        float s[GQ];
#pragma unroll
        for (int g = 0; g < GQ; g++) s[g] = 0.0f;
        if (tl < nt) {
            const uint4* kr = reinterpret_cast<const uint4*>(a.k_pool + row_off(t0 + tl) + qd * QD);
            uint4 kreg[QD / 8];
#pragma unroll
            for (int c = 0; c < QD / 8; c++) kreg[c] = kr[c];
#pragma unroll
            for (int c = 0; c < QD / 8; c++) {
                const __half2* kh = reinterpret_cast<const __half2*>(&kreg[c]);
                float kf[8];
#pragma unroll
                for (int i = 0; i < 4; i++) { const float2 f = __half22float2(kh[i]); kf[2 * i] = f.x; kf[2 * i + 1] = f.y; }
#pragma unroll
                for (int g = 0; g < GQ; g++) if (g < gq) {
                    const __half2* qh = reinterpret_cast<const __half2*>(sq + g * DH + qd * QD + c * 8);
#pragma unroll
                    for (int i = 0; i < 4; i++) { const float2 f = __half22float2(qh[i]); s[g] += kf[2 * i] * f.x; s[g] += kf[2 * i + 1] * f.y; }
                }
            }
        }
#pragma unroll
        for (int g = 0; g < GQ; g++) if (g < gq) {
            float v = s[g];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            v = __fmul_rn(v, a.scale);
            if (tl < nt) { if (qd == 0) s_sc[g * a.cap + tl] = v; lmax[g] = fmaxf(lmax[g], v); }
        }
    }
#pragma unroll
    for (int g = 0; g < GQ; g++) if (g < gq) { const float m = warp_max(lmax[g]); if (lane == 0) red_f[g][wid] = m; }
    __syncthreads();
    if (tid < gq) { float m = red_f[tid][0]; for (int k = 1; k < NW; k++) m = fmaxf(m, red_f[tid][k]); c_max[tid] = m; }
    cluster.sync();                                                                   // [1] every CTA's c_max is final
    if (tid < gq) {
        float M = -INFINITY;
        for (int rr = 0; rr < CS; rr++) M = fmaxf(M, *cluster.map_shared_rank(&c_max[tid], rr));
        s_M[tid] = M;
    }
    __syncthreads();

    // ---- 2. e = expf(s - max), row sum in double ----
    double lsum[GQ];
#pragma unroll
    for (int g = 0; g < GQ; g++) lsum[g] = 0.0;
    for (int i = tid; i < nt * gq; i += ATTN_THREADS) {
        const int g = i / nt, tl = i - g * nt;
        const float e = expf(s_sc[g * a.cap + tl] - s_M[g]);
        s_sc[g * a.cap + tl] = e;
#pragma unroll
        for (int gg = 0; gg < GQ; gg++) if (gg == g) lsum[gg] += (double)e;
    }
#pragma unroll
    for (int g = 0; g < GQ; g++) if (g < gq) {
        double v = lsum[g];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red_d[g][wid] = v;
    }
    __syncthreads();
    if (tid < gq) { double v = 0.0; for (int k = 0; k < NW; k++) v += red_d[tid][k]; c_sum[tid] = v; }
    cluster.sync();                                                                   // [2] every CTA's c_sum is final
    if (tid < gq) {
        double S = 0.0;
        for (int rr = 0; rr < CS; rr++) S += *cluster.map_shared_rank(&c_sum[tid], rr);
        s_inv[tid] = (float)(1.0 / S);
    }
    __syncthreads();
    // p = e * (1/sum), rounded to f16 (ggml converts the probabilities to f16 for the V product)
    for (int i = tid; i < nt * gq; i += ATTN_THREADS) {
        const int g = i / nt, tl = i - g * nt;
        s_sc[g * a.cap + tl] = __half2float(__float2half_rn(__fmul_rn(s_sc[g * a.cap + tl], s_inv[g])));
    }
    __syncthreads();

    // ---- 3. partial V.p over this CTA's tokens: thread = (8 head dims) x (token group) ----
    constexpr int DG = DH / 8;                       // threads across the head dim (one 128-bit load each)
    constexpr int TG = ATTN_THREADS / DG;            // token groups
    constexpr int TGW = 32 / DG;                     // token groups inside one warp
    const int dg = tid % DG, tg = tid / DG;
    float acc[GQ][8];
#pragma unroll
    for (int g = 0; g < GQ; g++)
#pragma unroll
        for (int i = 0; i < 8; i++) acc[g][i] = 0.0f;
    for (int tl = tg; tl < nt; tl += 2 * TG) {          // two V rows in flight per thread
        uint4 vv[2];
#pragma unroll
        for (int j = 0; j < 2; j++) {
            const int tj = tl + j * TG;
            vv[j] = (tj < nt) ? *reinterpret_cast<const uint4*>(a.v_pool + row_off(t0 + tj) + dg * 8) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int j = 0; j < 2; j++) {
            const int tj = tl + j * TG;
            if (tj >= nt) break;
            const __half2* vh = reinterpret_cast<const __half2*>(&vv[j]);
            float vf[8];
#pragma unroll
            for (int i = 0; i < 4; i++) { const float2 f = __half22float2(vh[i]); vf[2 * i] = f.x; vf[2 * i + 1] = f.y; }
#pragma unroll
            for (int g = 0; g < GQ; g++) if (g < gq) {
                const float p = s_sc[g * a.cap + tj];
#pragma unroll
                for (int i = 0; i < 8; i++) acc[g][i] += p * vf[i];
            }
        }
    }
    // token groups of one warp meet by shuffle, warps meet in shared memory; both in fixed order
#pragma unroll
    for (int g = 0; g < GQ; g++) if (g < gq) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            float v = acc[g][i];
#pragma unroll
            for (int o = DG; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane < DG) red_o[((size_t)wid * gq + g) * DH + dg * 8 + i] = v;
        }
    }
    (void)TGW;
    __syncthreads();
    for (int e = tid; e < gq * DH; e += ATTN_THREADS) {
        const int g = e / DH, dd = e - g * DH;
        float o = 0.0f;
#pragma unroll
        for (int k = 0; k < NW; k++) o += red_o[((size_t)k * gq + g) * DH + dd];
        c_out[e] = o;
    }
    cluster.sync();                                                                   // [3] every CTA's c_out is final
    // ---- 4. sum the CTAs' partials in rank order; CTA r finishes its share of the gq*DH outputs ----
    const int E = gq * DH;
    const int share = (E + CS - 1) / CS;
    for (int e = r * share + tid; e < min(E, (r + 1) * share); e += ATTN_THREADS) {
        float o = 0.0f;
        for (int rr = 0; rr < CS; rr++) o += *cluster.map_shared_rank(&c_out[e], rr);
        a.out[(size_t)hk * E + e] = o;
    }
    cluster.sync();                                                                   // [4] remote reads done before any CTA exits
}

// sum the split partials (fixed order) and quantise the attention output for the Wo mat-vec.
// grid = n_head*d_head/256 CTAs, block = 256 (one Q8_K super-block of the output each)
__global__ void __launch_bounds__(256) attn_combine_kernel(const float* __restrict__ part_o, int d_head, int n_split, int fmt, ActBuf out) {
    pdl_launch_dependents(); pdl_wait();
    const int e = blockIdx.x * 256 + threadIdx.x;
    const int h = e / d_head, dd = e % d_head;
    float o = 0.0f;
    for (int s = 0; s < n_split; s++) o += part_o[((size_t)h * n_split + s) * d_head + dd];
    __shared__ float y[256];
    y[threadIdx.x] = o;
    if (out.f32) out.f32[e] = o;
    __syncthreads();
    if (fmt == ACT_F32) return;
    if (threadIdx.x < 32) quantize_256_warp(y, 256, fmt, out.q + blockIdx.x * 256, out.d, out.bs, blockIdx.x);
}

// quantise an f32 vector (no norm): grid = ceil(K/256/8), block = 256 (8 warps, one super-block each)
__global__ void __launch_bounds__(256) act_quant_kernel(const float* __restrict__ x, int K, int fmt, ActBuf out) {
    pdl_launch_dependents(); pdl_wait();
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b * 256 >= K) return;
    quantize_256_warp(x + (size_t)b * 256, min(256, K - b * 256), fmt, out.q + (size_t)b * 256, out.d, out.bs, b);
}

// =================================================================================================================
// top-k of the vocabulary logits (Session.cpp:246-261 does a full std::sort of n_vocab pairs per token on the host).
// Order: logit descending, ties by lower id.
// =================================================================================================================
__device__ __forceinline__ bool td_before(float la, int ia, float lb, int ib) { return la > lb || (la == lb && ia < ib); }

// runtime-size variant (n a power of two <= 2048)
template <int THREADS>
__device__ inline void bitonic_sort_desc_n(float* key, int* idx, int n) {
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += THREADS) {
                const int p = i ^ j;
                if (p > i) {
                    const bool up = ((i & k) == 0);
                    const float a = key[i], b = key[p]; const int ia = idx[i], ib = idx[p];
                    const bool a_first = td_before(a, ia, b, ib);
                    if (up ? !a_first : a_first) { key[i] = b; key[p] = a; idx[i] = ib; idx[p] = ia; }
                }
            }
            __syncthreads();
        }
    }
}

// Threshold top-k.  The lm_head mat-vec leaves the maximum logit of
// every vocabulary chunk in chunk_max (atomicMax in its epilogue).  With C >= 64 chunks, the 64th largest chunk maximum
// tau is a lower bound of the 64th largest logit, so only logits >= tau can be in the top 64: a few hundred survivors
// out of 128k.  Every CTA derives tau, scans its share of the row and appends survivors; the last CTA to finish sorts
// them (logit descending, ties by lower id -> deterministic whatever the append order) and resets the scratch state.
struct TopkArgs {
    const float* logits; int n;
    int* chunk_max; int n_chunks;
    float* cand_l; int* cand_i; int cap;
    unsigned int* count; unsigned int* done;
    int32_t* out_ids; float* out_logits;
    int32_t* feed_tok;          // optional: receives the arg-max (greedy on-device feedback of the decode loop)
    long long ld;               // rows of a batch (blockIdx.y): logits ld floats apart; every per-row array below is laid out row-major:
                                // chunk_max [row][256], cand_l / cand_i [row][cap], count / done [row][2], out_* [row][TOPK_MAX]
};

__global__ void __launch_bounds__(1024) topk_select_kernel(TopkArgs a) {
    pdl_launch_dependents(); pdl_wait();
    if (blockIdx.y) {       // batched rows
        const size_t r = blockIdx.y;
        a.logits += r * (size_t)a.ld; a.chunk_max += r * 256; a.cand_l += r * (size_t)a.cap; a.cand_i += r * (size_t)a.cap;
        a.count += 2 * r; a.done += 2 * r; a.out_ids += r * TOPK_MAX; a.out_logits += r * TOPK_MAX;
    }
    __shared__ float key[2048];
    __shared__ int idx[2048];
    __shared__ unsigned int s_last, s_n;
    const int tid = threadIdx.x, lane = tid & 31;
    // 1. tau from the chunk maxima
    for (int i = tid; i < 256; i += 1024) { key[i] = i < a.n_chunks ? float_from_order_key(a.chunk_max[i]) : -INFINITY; idx[i] = i; }
    __syncthreads();
    bitonic_sort_desc_n<1024>(key, idx, 256);
    const float tau = (a.n_chunks >= TOPK_MAX) ? key[TOPK_MAX - 1] : -INFINITY;
    __syncthreads();
    // 2. scan this CTA's share, append survivors
    const int per = (a.n + gridDim.x - 1) / gridDim.x;
    const int begin = blockIdx.x * per, end = min(a.n, begin + per);
    for (int i0 = begin; i0 < end; i0 += 1024) {
        const int i = i0 + tid;
        const float v = i < end ? a.logits[i] : -INFINITY;
        const bool keep = (i < end) && (v >= tau);
        const unsigned int m = __ballot_sync(0xffffffffu, keep);
        if (m) {
            unsigned int base = 0;
            if (lane == 0) base = atomicAdd(a.count, (unsigned int)__popc(m));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (keep) {
                const unsigned int slot = base + __popc(m & ((1u << lane) - 1u));
                if (slot < (unsigned int)a.cap) { a.cand_l[slot] = v; a.cand_i[slot] = i; }
            }
        }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned int old = atomicAdd(a.done, 1u);
        s_last = (old == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (tid == 0) s_n = *reinterpret_cast<volatile unsigned int*>(a.count);
    __syncthreads();
    const unsigned int total = s_n;
    if (total <= (unsigned int)a.cap) {
        int n2 = 64;
        while (n2 < (int)total) n2 <<= 1;
        for (int i = tid; i < n2; i += 1024) {
            const bool ok = i < (int)total;
            key[i] = ok ? __ldcg(a.cand_l + i) : -INFINITY;
            idx[i] = ok ? __ldcg(a.cand_i + i) : 0x7fffffff;
        }
        __syncthreads();
        bitonic_sort_desc_n<1024>(key, idx, n2);
    } else {
        // degenerate row (e.g. thousands of equal logits): exact fallback over the whole row, 1984 at a time
        for (int i = tid; i < TOPK_MAX; i += 1024) { key[i] = -INFINITY; idx[i] = 0x7fffffff; }
        for (int base = 0; base < a.n; base += 2048 - TOPK_MAX) {
            for (int i = tid; i < 2048 - TOPK_MAX; i += 1024) {
                const int g = base + i;
                key[TOPK_MAX + i] = g < a.n ? a.logits[g] : -INFINITY;
                idx[TOPK_MAX + i] = g < a.n ? g : 0x7fffffff;
            }
            __syncthreads();
            bitonic_sort_desc_n<1024>(key, idx, 2048);
        }
    }
    for (int i = tid; i < TOPK_MAX; i += 1024) { a.out_ids[i] = idx[i]; a.out_logits[i] = key[i]; }
    if (tid == 0 && a.feed_tok) a.feed_tok[0] = idx[0];
    for (int i = tid; i < a.n_chunks; i += 1024) a.chunk_max[i] = (int)0x80000000;
    if (tid == 0) { *a.count = 0u; *a.done = 0u; }
}

__global__ void gather_logits_kernel(const float* __restrict__ logits, int n_vocab, const int32_t* __restrict__ ids, int n, float* out) {
    pdl_launch_dependents(); pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { const int id = ids[i]; out[i] = (id >= 0 && id < n_vocab) ? logits[id] : -INFINITY; }
}

// greedy on-device feedback for the device-resident decode loop (bench): next token = arg-max of the step just computed
__global__ void feed_top1_kernel(const int32_t* top_ids, int32_t* tok) {
    pdl_launch_dependents(); pdl_wait(); if (threadIdx.x == 0 && blockIdx.x == 0) tok[0] = top_ids[0]; }

__global__ void advance_pos_kernel(int32_t* pos, int n) {
    pdl_launch_dependents(); pdl_wait(); if (threadIdx.x == 0 && blockIdx.x == 0) pos[0] += n; }

} // namespace blk
