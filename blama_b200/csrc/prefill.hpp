// prefill.hpp -- host-side entry points of the multi-token prefill path (implemented in prefill.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "qweights.cuh"

namespace blk {

// C[T][N] (f32, row stride ldc) = or += X[T][K] (bf16, row-major, device) . W^T  through the tcgen05 GEMM
// mode: 0 store (+bias), 1 accumulate into C.  Returns a CUDA error (cudaErrorNotSupported if the driver lacks TMA).
// panel != nullptr selects the two-pass form: W was dequantised once into the bf16 panel (prefill_panel_fill) and the GEMM reads
// its B tiles from there -- for many-token batches, where the fused form would dequantise every weight tile T / 256 times.
// sk != nullptr: workspace for the deterministic split-K of the last, partial wave of tiles (all tiles when the batch has fewer
// tiles than SMs); n_sm * 65536 floats always suffice (split tiles * splits never exceeds the SM count)
// a split-K ACCUMULATE (C += X W^T over the residual stream, every tile split) whose partial sums are still in the workspace: the RMSNorm
// that follows adds them while it reads the row anyway (rmsnorm_bf16_launch), instead of a reduce kernel of its own
struct PendingReduce { const float* ws = nullptr; int S = 0, m_tiles = 0; };
struct SplitKWs { float* ws; size_t elems; PendingReduce* defer = nullptr; };
// plan != nullptr: what the call launched (unit tests check that a case runs the path it names).  launches counts GEMM kernel
// launches and accumulates; the other fields describe the last one (k_splits 1 and n_whole = every tile when nothing was split)
struct GemmPlan { int n_sm = 0, launches = 0, k_splits = 0, n_whole = 0; bool deferred = false, panel = false; };
cudaError_t prefill_gemm(const QMat& W, const __nv_bfloat16* X, int T, float* C, long long ldc, const float* bias, int mode, cudaStream_t st,
                         const __nv_bfloat16* panel = nullptr, const SplitKWs* sk = nullptr, GemmPlan* plan = nullptr);

// several matrices with the same K in one launch: C[:, col0_s : col0_s + N_s] = X . W_s^T (+bias_s).  Matrices 0 and 1 must share
// a weight type.  Falls back to one launch per matrix when a column offset is not 4-element aligned.
struct GemmPart { const QMat* W; const float* bias; int col0; };
cudaError_t prefill_gemm_multi(const GemmPart* parts, int n_parts, const __nv_bfloat16* X, int T, float* C, long long ldc, cudaStream_t st,
                               const __nv_bfloat16* panel = nullptr, const SplitKWs* sk = nullptr, GemmPlan* plan = nullptr);

// H[T][ff] (bf16) = silu(X . Wgate^T) * (X . Wup^T), one launch, SwiGLU in the GEMM epilogue
cudaError_t prefill_gemm_swiglu(const QMat& gate, const QMat& up, const __nv_bfloat16* X, int T, __nv_bfloat16* H, long long ldh, cudaStream_t st,
                                const __nv_bfloat16* panel = nullptr, const SplitKWs* sk = nullptr, GemmPlan* plan = nullptr);
// The dequantisation passes of the two-pass form: the panel of one GEMM over parts (prefill_gemm, prefill_gemm_multi), or with
// swiglu = true over {gate, up} (prefill_gemm_swiglu).  A caller can run them on a second stream one GEMM ahead.
// Return false when the combination takes the fused form (the GEMM call must then get panel = nullptr).
bool prefill_panel_fill(const GemmPart* parts, int n_parts, bool swiglu, __nv_bfloat16* panel, cudaStream_t st, cudaError_t* err);
// bf16 elements of that panel
size_t prefill_panel_elems(const GemmPart* parts, int n_parts, bool swiglu);

// Causal attention of a prefill chunk on tcgen05 (prefill_attn_tc.cuh): d_head = 128, GQA ratio 1 .. 8.
//   q [T][n_head*128] f16 (post-RoPE), paged f16 K / V pools of the layer, out [T][n_head*128] bf16;
//   vt: scratch [n_head_kv*128][ctx_pad] f16 for the transposed V of this layer (ctx_pad: multiple of 128 >= pos0 + T).
bool prefill_attn_tc_supported(int d_head, int n_head, int n_head_kv);
cudaError_t prefill_attn_tc(const __half* q, const __half* k_pool, const __half* v_pool, const int32_t* page_table, int n_pages, const int32_t* pos0_dev,
                            int pos0, __nv_bfloat16* out, __half* vt, int ctx_pad, int T, int n_head, int n_head_kv, int kv_dim, float scale, cudaStream_t st);

// gathered[t][j] = logit of vocabulary row claimed[t][j] at position t (j < n_claimed[t]; 0 past that, -inf for an id outside the
// vocabulary): sparse rows of the vocabulary projection, bf16 operands / f32 accumulation like the GEMM form
cudaError_t prefill_claimed_logits(const QMat& W, const __nv_bfloat16* xn, const int32_t* claimed, const int32_t* n_claimed, int n, float* gathered, cudaStream_t st);

// y[i] = bf16(x[i])
cudaError_t convert_f32_to_bf16(const float* x, __nv_bfloat16* y, size_t n, cudaStream_t st);

} // namespace blk
