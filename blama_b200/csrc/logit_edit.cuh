// logit_edit.cuh -- the logit-bias and repetition-penalty stages of the sampler chain on the device (llama.cpp b5187
// llama_sampler_logit_bias_apply + llama_sampler_penalties_apply), applied to a copy of a logits row.
//
// The host sampler only sees a top-k list, which is exact only while nothing ahead of top-k changes the logits.  With a
// bias or a penalty active, any id can enter the top 40, so the edited row gets a top-k of its own: this kernel writes the
// edited copy plus its per-chunk maxima, and topk_select_kernel (unchanged) selects from it.  The raw row is never written.
#pragma once
#include "gemv_kernels.cuh"

namespace blk {

struct LogitEdit { int32_t token; int32_t count; float bias; };     // layout of blk_logit_edit (include/blama_b200.h)

// One edited logit, bit-identical to the host Sampler's restatement: rounded operations only, so nvcc cannot contract
// the multiply and the subtraction into an FMA.  A zero bias is no edit (the id may only be listed for its count).
__device__ __forceinline__ float edit_logit(float l, int count, float bias, float repeat, float freq, float present) {
    if (bias != 0.0f) l = __fadd_rn(l, bias);
    if (count > 0) {
        l = l <= 0.0f ? __fmul_rn(l, repeat) : __fdiv_rn(l, repeat);
        l = __fsub_rn(l, __fadd_rn(__fmul_rn((float)count, freq), present));
    }
    return l;
}

struct LogitEditArgs {
    const float* logits; long long ld; int n;    // raw rows (blockIdx.y), ld floats apart, n = vocabulary size
    const float* params;                         // [row][3]: repeat, freq, present
    const int32_t* row_off;                      // [rows + 1]: CSR offsets into edits
    const LogitEdit* edits;                      // per row ascending by token, ids in [0, n)
    float* out;                                  // edited rows, same layout as logits
    int* chunk_max; int chunk_shift;             // [row][256] float_order_key of every chunk's maximum (exact)
};

// One CTA per vocabulary chunk of 1 << chunk_shift ids (dynamic shared memory holds the chunk).  The CTA finds its slice
// of the row's edit list by binary search, edits the staged chunk, then writes it out with its exact maximum:
// topk_select_kernel's "at least 64 survivors" rests on the chunk maxima never over-estimating.
__global__ void __launch_bounds__(256) logit_edit_kernel(LogitEditArgs a) {
    extern __shared__ float s_row[];
    __shared__ int s_lo, s_hi;
    __shared__ float red[8];
    const int r = blockIdx.y, tid = threadIdx.x;
    const int begin = (int)blockIdx.x << a.chunk_shift, end = min(a.n, begin + (1 << a.chunk_shift));
    const float* in = a.logits + (size_t)r * (size_t)a.ld;
    float* out = a.out + (size_t)r * (size_t)a.ld;
    if (tid < 2) {      // lower bound of begin (thread 0) and of end (thread 1) in the row's edits
        const int key = tid == 0 ? begin : end;
        int lo = a.row_off[r], hi = a.row_off[r + 1];
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (a.edits[mid].token < key) lo = mid + 1; else hi = mid; }
        if (tid == 0) s_lo = lo; else s_hi = lo;
    }
    for (int i = begin + tid; i < end; i += 256) s_row[i - begin] = in[i];
    __syncthreads();
    const float repeat = a.params[3 * r], freq = a.params[3 * r + 1], present = a.params[3 * r + 2];
    for (int e = s_lo + tid; e < s_hi; e += 256) {       // ids are distinct: one writer per element
        const LogitEdit ed = a.edits[e];
        float& v = s_row[ed.token - begin];
        v = edit_logit(v, ed.count, ed.bias, repeat, freq, present);
    }
    __syncthreads();
    float m = -INFINITY;
    for (int i = begin + tid; i < end; i += 256) { const float v = s_row[i - begin]; out[i] = v; m = fmaxf(m, v); }
    m = warp_max(m);
    if ((tid & 31) == 0) red[tid >> 5] = m;
    __syncthreads();
    if (tid == 0) {
        for (int i = 1; i < 8; i++) m = fmaxf(m, red[i]);
        a.chunk_max[r * 256 + (int)blockIdx.x] = float_order_key(m);
    }
}

} // namespace blk
