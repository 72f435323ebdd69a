// mega_decode.hpp -- descriptors and host entry points of the persistent decode kernel (mega_decode.cuh / mega_decode.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "qweights.cuh"

namespace blk {

constexpr int MG_WARPS = 16;
constexpr int MG_THREADS = MG_WARPS * 32;
#ifndef MG_SLOTS_N
#define MG_SLOTS_N 3
#endif
constexpr int MG_SLOTS = MG_SLOTS_N;
constexpr int MG_PCAP = 512;          // tokens of one softmax / V.p sub-slice held in shared memory

enum : int { MK_Q = 0, MK_K = 1, MK_V = 2, MK_RESID = 3, MK_SWIGLU = 4, MK_LOGITS = 5 };
enum : int { MSRC_X = 0, MSRC_ATTN = 1, MSRC_H = 2 };

// super-block (256 weights) bytes in the stream copy
__host__ __device__ inline int mg_sb_bytes(int type) {
    switch (type) {
        case QT_Q4_K: return 144;
        case QT_Q5_K: return 176;
        case QT_Q6_K: return 208;      // + 2 B of d per super-block in the slice tail
        case QT_Q8_0: return 272;
        default: return 0;
    }
}
// bytes of one row slice of `sbs` super-blocks (multiple of 16)
__host__ __device__ inline int mg_slice_bytes(int type, int sbs) {
    int b = sbs * mg_sb_bytes(type);
    if (type == QT_Q6_K) b += (sbs * 2 + 15) / 16 * 16;
    return b;
}

struct MegaSeg {
    const uint8_t* base;     // chunks [pair][slice][a|b], slice_bytes each
    const float* bias;       // optional, indexed by output row
    int type;                // QT_*
    int n_pairs;
    int slice_bytes;
    int rot;                 // rotation of the pair -> warp-group assignment (balances the remainder across phases)
    int kind;                // MK_*
    int slot0;               // first partial-sum slot of this segment: items of the earlier segments (ceil(n_pairs / groups))
};
struct MegaPhase {
    MegaSeg seg[3];
    const float* norm_w;     // RMSNorm weight applied to the source vector (nullptr: none)
    int nseg;
    int K;                   // row length
    int W;                   // warps per row pair (K-slices)
    int L;                   // lanes (half super-blocks) per slice, even
    int rpc;                 // row slices per chunk: 2 when both rows of a pair fit in one warp (2L <= 32), else 1
    int act_fmt;             // ACT_Q8_K / ACT_Q8_0
    int src;                 // MSRC_*
    int layer;
    int items;               // upper bound of row pairs per warp group in this phase (all segments)
    int NG;                  // warp groups per CTA = MG_WARPS / W
    int wsh;                 // log2(W) when W is a power of two, else -1
    int ngsh;                // log2(NG) when NG is a power of two, else -1
};
static_assert(sizeof(MegaPhase) % 16 == 0, "MegaPhase must be a whole number of 16-byte words");

struct MegaParams {
    const MegaPhase* phases; int n_phases; int n_layer;
    const uint4* chunk_list; const int* chunk_counts; int list_stride;     // per (cta, warp): chunk descriptors {addr.lo, addr.hi, bytes, 0}
    int n_cta; int slot_bytes; int max_items; int act_bytes;
    int attn_off;            // offset of the attention tiles inside the activation scratch (behind an n_embd-long row's activations)
    int ts_cap;              // tokens of one attention tile (K and V rows of a CTA's context slice held in shared memory) = tokens per context split
    // model
    QMat tok_embd;
    int n_embd, n_head, n_head_kv, d_head, n_ff, n_vocab, neox;
    float eps, theta_scale, attn_scale;
    const float* rope_freqs;
    // context
    const int32_t* tok; int32_t* pos;
    // cross-CTA vectors as LL words {value bits, epoch tag} (mega_decode.cuh): residual stream, q, SwiGLU output, attention output,
    // split partials [max_split][n_head * d_head], the new token's K | V rows [2][kv_dim]
    uint2* x2; uint2* q2; uint2* h2; uint2* ao2; uint2* po2; uint2* kvn2;
    uint2* st2;              // soft-max statistics of the split partials [n_head][max_split] x {local max, local sum}
    int max_split;
    uint32_t seq;            // launch counter of the context (epoch base of every tag)
    int* err;                // mapped host word: set when a poll timed out
    __half* const* k_pools; __half* const* v_pools; const int32_t* page_table; int kv_dim;
    float* logits; int* chunk_max; int chunk_shift;
    int with_head; int advance_pos;
    long long* trace; int trace_cap; int trace_global;      // optional event trace [n_cta][trace_cap] (debug / profiling)
};

// ---- host entry points (mega_decode.cu) ----
// dynamic shared memory the kernel needs for these parameters
size_t mega_smem_bytes(const MegaParams& P);
// opt the kernel in to `smem` bytes of dynamic shared memory; returns the device's per-block opt-in limit in *limit
cudaError_t mega_setup(size_t smem, int* limit);
// cooperative launch of one decode step: P.n_cta CTAs (must all be co-resident: one per SM)
cudaError_t mega_launch(const MegaParams& P, size_t smem, cudaStream_t st);
// scatter one raw ggml tensor (device copy) into the stream layout of a segment.
//   rowmap: 0 = pairs (2p, 2p+1); 1 = NEOX rotary pairs (r, r + d_head/2) inside each head; 2 = every row is half `ab` of pair r
// per (cta, warp) chunk lists of the whole token; list == nullptr: only counts[n_cta * MG_WARPS]
cudaError_t mega_chunk_lists(const MegaPhase* d_phases, int n_phases, int n_cta, uint4* list, int list_stride, int* counts, cudaStream_t st);
cudaError_t mega_build_stream(const uint8_t* raw, uint8_t* base, int type, int N, int K, int W, int sbs, int slice_bytes,
                              int rowmap, int d_head, int ab, cudaStream_t st);

} // namespace blk
