/*
 * blama_b200.h -- C ABI of the B200-native engine behind blama's inference hot path.
 *
 * blama has no plugin registry: the seam its hot path sits behind is the llama.cpp C API called from
 * bl::llama::{Model,Instance,Session,Sampler} (SURVEY.md section 8b).  This header is the narrower ABI that
 * replaces those call sites; each entry point cites the reference interface it stands in for
 * (paths relative to the reference tree, inference/code/llama/ unless noted).  The C++ classes in
 * blama_b200/host/llama/ re-implement bl::llama::* over exactly these functions, and INTEGRATION.md shows the
 * binding a blama maintainer would add.
 *
 * Conventions: plain pointers and sizes only; every function returns a blk_status (0 = ok) unless it returns a
 * handle (NULL on failure) or a value; no exceptions cross the boundary; blk_last_error() gives the message of the
 * last failure on the calling thread.  One thread drives one blk_ctx at a time (Server.cpp:36); several contexts may
 * share one blk_model (t-integration.cpp:220-224).  There is NO CPU fallback: without a CUDA device every call
 * that needs one fails with BLK_ERR_NO_DEVICE.
 */
#ifndef BLAMA_B200_H
#define BLAMA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BLK_API __attribute__((visibility("default")))

typedef int32_t blk_status;
enum {
    BLK_OK = 0,
    BLK_ERR_NO_DEVICE = 1,   /* no CUDA device / driver (the product never falls back to the CPU) */
    BLK_ERR_IO = 2,          /* file missing / unreadable */
    BLK_ERR_FORMAT = 3,      /* not a GGUF v2/v3 file, unsupported arch or tensor type */
    BLK_ERR_ARG = 4,         /* bad argument (token id out of range, n <= 0, ...) */
    BLK_ERR_CTX_FULL = 5,    /* n_past + n > n_ctx            (llama_decode != 0, Session.cpp:388-390) */
    BLK_ERR_CUDA = 6,        /* CUDA runtime error */
    BLK_ERR_OOM = 7
};

typedef struct blk_model blk_model;
typedef struct blk_ctx blk_ctx;

/* TokenData of the reference (Token.hpp:12-15): 8 bytes, {int32 token; float logit} */
typedef struct { int32_t token; float logit; } blk_token_data;

/* ---- library -------------------------------------------------------------------------------------------- */
/* llama_backend_init + llama_log_set (Init.cpp:34-38).  Idempotent. */
BLK_API blk_status blk_init(void);
typedef void (*blk_log_cb)(int level, const char* text, void* user);      /* level: 0 debug 1 info 2 warn 3 error */
BLK_API void blk_set_log_callback(blk_log_cb cb, void* user);              /* Init.cpp:11-30 llamaLogCb */
BLK_API const char* blk_last_error(void);
BLK_API int32_t blk_device_count(void);                                   /* ggml_backend_dev_by_type(GPU), Model.cpp:14-19 */
BLK_API const char* blk_version(void);

/* ---- model (Model.cpp:50-53 llama_model_load_from_file, llama_model_free) -------------------------------- */
typedef int32_t (*blk_progress_cb)(float progress, void* user);           /* Model.cpp:37-43; return 0 to abort */
/* Parses the GGUF, uploads every tensor to `device` as device-resident quant blocks (Q4_K/Q5_K/Q6_K/Q8_0/F16/F32),
 * re-tiled on the device into the split layout the kernels stream (DESIGN.md "Data layout"). */
BLK_API blk_model* blk_model_load(const char* gguf_path, int32_t device, blk_progress_cb cb, void* user);
/* Model::Params::vocabOnly (Model.hpp:30; llama_model_params.vocab_only, Model.cpp:33): metadata + vocabulary only.  Needs no
 * CUDA device; such a model cannot back a context (n_ctx_train reads 0, as the reference's "vocab only" test expects). */
BLK_API blk_model* blk_model_load_vocab(const char* gguf_path);
BLK_API void       blk_model_free(blk_model*);
BLK_API int32_t blk_model_n_vocab(const blk_model*);        /* llama_vocab_n_tokens    Session.cpp:27 */
BLK_API int32_t blk_model_n_ctx_train(const blk_model*);    /* llama_model_n_ctx_train Model.cpp:59 */
BLK_API int32_t blk_model_n_embd(const blk_model*);         /* llama_model_n_embd */
BLK_API int32_t blk_model_n_layer(const blk_model*);        /* llama_model_n_layer */
BLK_API int32_t blk_model_token_bos(const blk_model*);      /* llama_vocab_bos         Session.cpp:73 */
BLK_API int32_t blk_model_token_eos(const blk_model*);      /* llama_vocab_eos         Instance.cpp:94 */
BLK_API int32_t blk_model_is_eog(const blk_model*, int32_t token);   /* llama_vocab_is_eog Vocab.cpp:30 */
BLK_API int32_t blk_model_add_bos(const blk_model*);        /* llama_vocab_get_add_bos Model.cpp:63 */
BLK_API int32_t blk_model_add_eos(const blk_model*);        /* llama_vocab_get_add_eos (llama_tokenize appends EOS when set) */
BLK_API int32_t blk_model_vocab_only(const blk_model*);
BLK_API int32_t blk_model_device(const blk_model*);
/* bytes of weights one decoded token streams from HBM (all matmul tensors once + lm_head; SURVEY.md 8d) */
BLK_API int64_t blk_model_weight_bytes_per_token(const blk_model*);
/* KV bytes per context token (K+V, all layers, f16) */
BLK_API int64_t blk_model_kv_bytes_per_token(const blk_model*);
/* Bytes of the resident bf16 weight panels (the multi-token GEMMs' B operands, built by the first prefill of >= 32 tokens into
   free device memory beyond a reserve; BLK_PANEL_CACHE_GB caps it, 0 disables) and how many of the 4 n_layer + 1 matrices they
   cover (n_resident may be NULL).  0 before the first multi-token pass.  No llama.cpp counterpart: ggml keeps quantised weights only. */
BLK_API int64_t blk_model_panel_bytes(blk_model*, int32_t* n_resident, int32_t* n_matrices);
/* token text (tokenizer.ggml.tokens[token]); returns length, copies at most cap bytes (llama_token_to_piece, Vocab.cpp:57) */
BLK_API int32_t blk_model_token_text(const blk_model*, int32_t token, char* buf, int32_t cap);
/* The vocabulary behind llama_tokenize / llama_token_to_piece (Vocab.cpp:40,57): token attribute (tokenizer.ggml.token_type:
 * 1 normal, 2 unknown, 3 control, 4 user defined, 5 unused, 6 byte) and the BPE merge list in rank order ("left right").  The
 * tokenizer itself is host code above this boundary (blama_b200/host/llama/Tokenizer.cpp). */
BLK_API int32_t blk_model_token_type(const blk_model*, int32_t token);
BLK_API int32_t blk_model_n_merges(const blk_model*);
BLK_API int32_t blk_model_merge_text(const blk_model*, int32_t rank, char* buf, int32_t cap);
/* metadata string lookup (llama_model_meta_val_str, Model.cpp:77); returns length or -1 */
BLK_API int32_t blk_model_meta_str(const blk_model*, const char* key, char* buf, int32_t cap);

/* ---- context (Instance.cpp:34-48 llama_init_from_model, llama_free) -------------------------------------- */
/* n_ctx = 0 -> training context (Instance.hpp:22).  n_batch = logical prefill batch (Instance.hpp:23). */
BLK_API blk_ctx*   blk_ctx_create(blk_model*, int32_t n_ctx, int32_t n_batch);
BLK_API void       blk_ctx_free(blk_ctx*);
BLK_API int32_t    blk_ctx_n_ctx(const blk_ctx*);           /* llama_n_ctx   Session.cpp:57 */
BLK_API int32_t    blk_ctx_n_batch(const blk_ctx*);         /* llama_n_batch Session.cpp:381 */
BLK_API int32_t    blk_ctx_n_past(const blk_ctx*);
BLK_API const blk_model* blk_ctx_model(const blk_ctx*);     /* llama_get_model Session.cpp:26 */
BLK_API blk_status blk_kv_clear(blk_ctx*);                  /* llama_kv_self_clear Session.cpp:53 */
BLK_API blk_status blk_sync(blk_ctx*);                      /* llama_synchronize   Session.cpp:54 */
/* Context shift (Session.cpp:341-342): llama_kv_self_seq_rm(ctx, 0, p0, p1) followed by llama_kv_self_seq_add(ctx, 0, p1, n_past,
 * -(p1 - p0)).  The cells of positions [p0, p1) are dropped, the cells behind them move down by p1 - p0 and their K rows are
 * re-rotated by that position change exactly as llama.cpp's K-shift does (RoPE applied to the f16 cache row); n_past shrinks by
 * p1 - p0. */
BLK_API blk_status blk_kv_shift(blk_ctx*, int32_t p0, int32_t p1);
/* Self-Extend group attention (Session.cpp:348-368): llama_kv_self_seq_add(ctx, 0, p0, p1, delta) and llama_kv_self_seq_div(ctx, 0, p0,
 * p1, d).  Cells whose POSITION lies in [p0, p1) get position + delta / position / d; the cells stay where they are, their K rows
 * are re-rotated by the accumulated position change before the next decode (llama.cpp's K-shift), and the next token takes the
 * position one past the largest one (blk_ctx_next_pos), which from then on differs from the number of cells (blk_ctx_n_past). */
BLK_API blk_status blk_kv_seq_add(blk_ctx*, int32_t p0, int32_t p1, int32_t delta);
BLK_API blk_status blk_kv_seq_div(blk_ctx*, int32_t p0, int32_t p1, int32_t d);
BLK_API int32_t    blk_ctx_next_pos(const blk_ctx*);
/* llama_state_get_size / llama_state_get_data / llama_state_set_data (Session.cpp:291-304): the KV rows of every layer, the
 * last logits row and its top-k list, as one blob (engine-specific layout, not llama.cpp's).  The sampler's RNG is not part of
 * it, as in the reference (t-integration.cpp:371-376). */
BLK_API int64_t    blk_state_size(const blk_ctx*);
BLK_API blk_status blk_state_get(blk_ctx*, void* dst, int64_t cap, int64_t* written);
BLK_API blk_status blk_state_set(blk_ctx*, const void* src, int64_t size);

/* ---- decode (Session.cpp:388 llama_decode on a llama_batch_get_one batch) -------------------------------- */
/* Appends n tokens at positions n_past.. ; afterwards the logits of the LAST token are resident on the device
 * (the reference's llama_get_logits_ith(-1) row).  n == 1 is the batch-1 decode step (dequant-fused GEMV path,
 * CUDA graph); n > 1 is prompt prefill (tcgen05 GEMM path). */
BLK_API blk_status blk_decode(blk_ctx*, const int32_t* tokens, int32_t n);

/* Session::getLogitsFromCtx(topK) (Session.cpp:246-261) without the host sort: top-k (k <= 64) of the last
 * token's logits, descending (ties: lower id first). */
BLK_API blk_status blk_topk_last(blk_ctx*, int32_t k, blk_token_data* out);
/* Session::getLogitsFromCtx(TokenDataVector) (Session.cpp:263-282) without the V-long host loop: logits of the last
 * token at `ids` (raw, in the order given; the caller applies the reference's de-dup + sort). */
BLK_API blk_status blk_gather_last(blk_ctx*, const int32_t* ids, int32_t n, float* out);
/* llama_get_logits_ith(-1) (Session.cpp:24, Sampler.cpp:111): copies all n_vocab logits to the host.  Test / debug
 * path: the product never needs the full row. */
BLK_API blk_status blk_get_logits_last(blk_ctx*, float* out);

/* One fused decode step for Session::getToken (Session.cpp:169-190): decode `token`, then return the top-k of the new
 * distribution in one device->host copy. */
BLK_API blk_status blk_decode_topk(blk_ctx*, int32_t token, int32_t k, blk_token_data* out);

/* Continuous batching (not in the reference, whose Server serialises requests: server/code/server/Server.cpp:36; SURVEY.md 8f
 * item 4): ONE forward pass for n <= 64 sequences, one new token each.  ctxs[i] are distinct contexts of the workspace context's
 * model; tokens[i] is appended to ctxs[i] at that context's own position, into its own KV pages.  The weights are streamed once for
 * all rows through the tcgen05 GEMM path (bf16 operand arithmetic: that of the verify prefill, not the int8 arithmetic of the
 * batch-1 kernel).  out[i * k .. i * k + k - 1] = top-k of sequence i's new distribution, descending.  `ws` lends its stream and
 * prefill workspaces and may or may not be one of ctxs.  The contexts' "last logits" are not kept (blk_topk_last / blk_gather_last
 * need a blk_decode first). */
BLK_API blk_status blk_decode_batch(blk_ctx* ws, blk_ctx* const* ctxs, const int32_t* tokens, int32_t n, int32_t k, blk_token_data* out);

/* ---- logit bias and repetition penalties (llama.cpp b5187 llama_sampler_logit_bias_apply + llama_sampler_penalties_apply) ----
 * The two stages at the head of the reference's sampler chain change logits before its top-k, so the top-k of the raw row no
 * longer decides the draw.  These entry points apply them on the device to a COPY of the last logits row and select the top-k
 * of that copy; the raw row, its top-k (the reported top-10), blk_gather_last, blk_get_logits_last and the state blob stay raw.
 * Per edited id, in this order (float arithmetic, no contraction):
 *     if (bias != 0)  logit += bias;
 *     if (count > 0)  { logit = logit <= 0 ? logit * repeat : logit / repeat;  logit -= (float)count * freq + present; }
 * Edit lists come from outside the library and are checked before anything is launched (BLK_ERR_ARG): ids in [0, n_vocab) and
 * strictly ascending, counts >= 0, biases not NaN or +inf (-inf bans an id), repeat finite and > 0, freq / present finite.
 * Lists of any length are staged (a bias map may ban thousands of ids). */
typedef struct { int32_t token; int32_t count; float bias; } blk_logit_edit;      /* count 0 = bias only */
typedef struct { float repeat, freq, present; const blk_logit_edit* edits; int32_t n_edits; } blk_logit_edits;
/* blk_decode_topk plus the edit pass: raw = top-k of the new raw row (what blk_decode_topk returns), edited = top-k of the edited
 * row.  One synchronise. */
BLK_API blk_status blk_decode_topk_edited(blk_ctx*, int32_t token, int32_t k, const blk_logit_edits* edits, blk_token_data* raw,
                                          blk_token_data* edited);
/* top-k of the edited copy of the kept last row (after a prompt prefill, a verify fill, blk_state_set, or for a sampler replaced
 * after a decode).  Needs a last row, as blk_topk_last does. */
BLK_API blk_status blk_topk_last_edited(blk_ctx*, int32_t k, const blk_logit_edits* edits, blk_token_data* edited);
/* blk_decode_batch plus the edit pass of every row (per_row[n]): raw as blk_decode_batch's out, edited[i * k ..] = top-k of row i
 * after its own edits.  One edit launch and one selection launch for all rows. */
BLK_API blk_status blk_decode_batch_edited(blk_ctx* ws, blk_ctx* const* ctxs, const int32_t* tokens, int32_t n, int32_t k,
                                           const blk_logit_edits* per_row, blk_token_data* raw, blk_token_data* edited);

/* Device-resident greedy decode loop (measurement aid for bench.py's `value`): n_steps decode steps back to back with the
 * arg-max token fed back ON THE DEVICE, no host round trip inside the loop.  Asynchronous unless last_token != NULL. */
BLK_API blk_status blk_decode_loop(blk_ctx*, int32_t first_token, int32_t n_steps, int32_t* last_token);

/* ---- verification context fill (Session::fillCtx, Session.cpp:231-244) ----------------------------------- */
/* Appends the n response tokens as ONE causal prefill (chunked by n_batch) instead of n single-token decodes, and for
 * every position i returns
 *   gathered[i*10 + j] = verifier logit at claimed[i*10 + j]  (j < n_claimed[i]; raw, unsorted), and
 *   top[i*10 .. i*10+9] = the verifier's own top-10 (descending),
 * without ever materialising the n x n_vocab logits.  `top` may be NULL. */
BLK_API blk_status blk_verify_prefill(blk_ctx*, const int32_t* tokens, int32_t n,
                                      const int32_t* claimed /* [n][10] */, const int32_t* n_claimed /* [n] */,
                                      float* gathered /* [n][10] */, blk_token_data* top /* [n][10] or NULL */);

/* 0 (default) = batched prefill (tcgen05 GEMM path; results within the stated fp tolerance of the decode path);
 * 1 = sequential: n batch-1 decodes, exactly the reference's algorithm, logits bit-identical to blk_decode_topk. */
BLK_API blk_status blk_ctx_set_verify_mode(blk_ctx*, int32_t mode);

/* ---- measurement ------------------------------------------------------------------------------------------ */
/* CUDA-event timing on the context's own stream (torch.cuda.Event cannot see it). */
BLK_API blk_status blk_timer_start(blk_ctx*);
BLK_API blk_status blk_timer_stop(blk_ctx*, float* ms);     /* synchronises the stream */
/* number of kernels this context has launched since creation (graph replays count their kernel nodes) */
BLK_API int64_t    blk_ctx_kernel_launches(const blk_ctx*);
/* 1 when batch-1 decode steps of this context run as the single persistent cooperative kernel (mega_decode.cuh), 0 when
 * they run as the per-operation CUDA graph (weight types or shapes the persistent kernel does not take, or BLK_MEGA=0) */
BLK_API int32_t    blk_ctx_persistent_decode(const blk_ctx*);
/* Debug: per-CTA stage-boundary clocks of the last persistent decode step (context created with BLK_MEGA_TRACE=1);
 * out receives n_cta x per_cta SM-clock samples. */
BLK_API blk_status blk_debug_trace(blk_ctx*, int64_t* out, int32_t cap, int32_t* n_cta, int32_t* per_cta);
/* Times ONE kernel of the decode path in isolation, for the roofline line of bench.py: launches it `iters` times back to
 * back, cycling through the layers so consecutive launches stream different weights (working set >> L2), bracketed by
 * CUDA events on the context's stream.  which: 0 = gate/up + SwiGLU mat-vec, 1 = down-proj mat-vec, 2 = QKV mat-vec,
 * 3 = attention-output mat-vec, 4 = lm_head mat-vec, 5 = the persistent decode kernel (one launch = the whole forward of
 * one token at the context's current position, top-k not included; needs blk_ctx_persistent_decode() == 1).  Returns the
 * average launch duration and the algorithmic bytes one launch must move (quantised weights + KV rows read / activations). */
BLK_API blk_status blk_bench_kernel(blk_ctx*, int32_t which, int32_t iters, float* avg_ms, int64_t* bytes_per_launch);
/* Decodes `token` with the step's kernels launched eagerly and a CUDA event between every pair of launches (so without
 * the cross-kernel overlap of the graph), and writes a CSV breakdown (kernel, launches, total_us, avg_us, share). */
BLK_API blk_status blk_profile_step(blk_ctx*, int32_t token, char* report, int32_t cap);
/* same for one verification prefill of n tokens (event between every kernel of the tcgen05 path) */
BLK_API blk_status blk_profile_verify(blk_ctx*, const int32_t* tokens, int32_t n, char* report, int32_t cap);
/* writes >= bytes of device memory to evict L2 between timed iterations */
BLK_API blk_status blk_flush_l2(blk_ctx*);

/* ---- unit-level entry points (kernel parity tests) --------------------------------------------------------- */
/* y[r] = W[r,:] . x through the decode GEMV kernel of ggml type `type` (raw ggml blocks in, host buffers) */
BLK_API blk_status blk_test_gemv(int32_t device, int32_t type, const void* w_blocks, int64_t rows, int64_t k,
                                 const float* x, float* y);
/* The prefill tcgen05 GEMM (bf16 operands, f32 accumulate) called the way a multi-token pass calls it, inside the pass's programmatic
 * dependent launch scope.  mats: weights of ggml type `type`, rows x k (raw ggml blocks), optional bias [rows]; x [n_tok][k] f32 (rounded
 * to bf16 on the device).
 *   op 0: C[:, col0_i .. col0_i + rows_i) = X W_i^T (+ bias_i) for 1 - 3 matrices side by side (col0_i = rows of the matrices before i;
 *         QKV / lm_head); c_inout [n_tok][sum rows] in / out (columns the GEMM must write can be preset to NaN)
 *   op 1: C += X W^T, one matrix (Wo / down onto the residual); c_inout [n_tok][rows] in / out.  norm_w [rows] != NULL: then the RMSNorm
 *         of the pass, h_or_xn [n_tok][rows] = bf16(rmsnorm(C) * norm_w) as f32
 *   op 2: h_or_xn [n_tok][rows] = bf16(silu(X Wgate^T) * (X Wup^T)) as f32, mats = {gate, up}
 * form: 0 fused (de-quantised inside the GEMM), 1 panel (the bf16 panel filled first; BLK_ERR_ARG for weights that take the fused form only).
 * split: 0 no split-K workspace, 1 a workspace of n_SM x 65536 floats, 2 the same with the reduce deferred to the RMSNorm (op 1 with norm_w).
 * plan (may be NULL) receives what ran: the SM count, GEMM launches, K splits, whole tiles (all tiles when not split), whether the reduce was
 * deferred and whether the panel kernel ran. */
typedef struct { int32_t type; const void* blocks; int64_t rows; const float* bias; } blk_test_matrix;
typedef struct { int32_t n_sm, launches, k_splits, n_whole, deferred, panel; } blk_test_gemm_plan;
BLK_API blk_status blk_test_gemm(int32_t device, int32_t op, const blk_test_matrix* mats, int32_t n_mats, int64_t k, const float* x, int64_t n_tok,
                                 int32_t form, int32_t split, const float* norm_w, float eps, float* c_inout, float* h_or_xn, blk_test_gemm_plan* plan);
/* average duration of the prefill GEMM on the given weights with n_tok resident bf16 activations (CUDA events) */
BLK_API blk_status blk_bench_gemm(int32_t device, int32_t type, const void* w_blocks, int64_t rows, int64_t k, int64_t n_tok, int32_t iters, float* avg_ms);
/* The non-GEMM kernels of the prefill path, one at a time (host buffers in / out; f16 / bf16 results come back as the exact values in
 * f32): rmsnorm_bf16_kernel; qkv_post_kernel (RoPE on q and k, q -> f16, k / v -> the f16 cache rows, read back through a reversed
 * page table); the causal prefill attention (tcgen05 kernel for d_head 128, *used_tc tells) over a cache of pos0 + T keys. */
BLK_API blk_status blk_test_rmsnorm(int32_t device, const float* x, const float* w, int32_t T, int32_t K, float eps, float* out);
BLK_API blk_status blk_test_qkv_post(int32_t device, const float* qkv, int32_t T, int32_t n_head, int32_t n_head_kv, int32_t d_head, int32_t neox,
                                     int32_t pos0, float rope_theta, const float* freq_factors, float* q_out, float* k_out, float* v_out);
BLK_API blk_status blk_test_prefill_attn(int32_t device, const float* q, const float* k, const float* v, int32_t T, int32_t pos0, int32_t n_head,
                                         int32_t n_head_kv, int32_t d_head, float* out, int32_t* used_tc);
/* The decode attention kernels over a paged f16 cache behind a seeded random page table (pages and cells nothing should read hold NaN).
 * blk_test_decode_attn: one query row q [n_head*d_head] over cells 0 .. n_kv - 1 of a context of n_ctx cells (k / v [n_kv][n_head_kv*d_head]),
 * through the per-op decode step's form plan and launch; form -1 = the plan's choice, 0 = the three-kernel split form, 1 = the cluster form
 * (BLK_ERR_ARG without a launch when the plan does not allow it); *used_form = 1 when the cluster form ran.
 * blk_test_decode_attn_batch: the batched decode step's attention over n rows of their own lengths n_kv[n] in one launch (k / v: the
 * rows' keys / values one after another); out [n][n_head*d_head] = the bf16 output as f32. */
BLK_API blk_status blk_test_decode_attn(int32_t device, const float* q, const float* k, const float* v, int32_t n_kv, int32_t n_ctx, int32_t n_head,
                                        int32_t n_head_kv, int32_t d_head, int32_t form, int64_t seed, float* out, int32_t* used_form);
BLK_API blk_status blk_test_decode_attn_batch(int32_t device, int32_t n, const float* q, const float* k, const float* v, const int32_t* n_kv,
                                              int32_t n_head, int32_t n_head_kv, int32_t d_head, int64_t seed, float* out);
/* The edit pass of blk_decode_batch_edited on host rows: logits [n_rows][n_vocab] and per_row[n_rows] in, out [n_rows][k] = the
 * edited rows' top-k (descending, ties to the lower id), through the same two launches. */
BLK_API blk_status blk_test_logit_edits(int32_t device, const float* logits, int32_t n_rows, int32_t n_vocab, const blk_logit_edits* per_row,
                                        int32_t k, blk_token_data* out);
/* The output kernels of a verify pass.  blk_test_row_topk: row_topk_gather_kernel over logits [n_rows][n_vocab], rows_per_launch rows per
 * launch as the pass chunks them: gathered[r][j] = logit of claimed[r][j] (j < n_claimed[r]; 0 past it, -inf outside the vocabulary) and,
 * when top_ids != NULL, the top 10 of each row (descending, ties to the lower id).  blk_test_claimed_logits: claimed_logits_kernel, the same
 * gathered[n][10] computed as dot(bf16(dequant(W[id])), bf16(xn[t])) with W of ggml type `type`, rows x k. */
BLK_API blk_status blk_test_row_topk(int32_t device, const float* logits, int32_t n_rows, int32_t n_vocab, int32_t rows_per_launch,
                                     const int32_t* claimed, const int32_t* n_claimed, float* gathered, int32_t* top_ids, float* top_logits);
BLK_API blk_status blk_test_claimed_logits(int32_t device, int32_t type, const void* w_blocks, int64_t rows, int64_t k, const float* xn, int32_t n,
                                           const int32_t* claimed, const int32_t* n_claimed, float* gathered);
/* dequantise through the device re-tile + dequant kernels */
BLK_API blk_status blk_test_dequant(int32_t device, int32_t type, const void* w_blocks, int64_t rows, int64_t k, float* out);

#ifdef __cplusplus
}
#endif
#endif /* BLAMA_B200_H */
