// engine.hpp -- model / context objects behind the C ABI (include/blama_b200.h).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>
#include <mutex>

#include "../../include/blama_b200.h"
#include <cuda_bf16.h>
#include "decode_kernels.cuh"
#include "mega_decode.hpp"

namespace blk {

struct BlkError : std::runtime_error {
    blk_status code;
    BlkError(blk_status c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define BLK_CUDA(expr)                                                                                              \
    do {                                                                                                            \
        cudaError_t e__ = (expr);                                                                                   \
        if (e__ != cudaSuccess)                                                                                     \
            throw ::blk::BlkError(e__ == cudaErrorMemoryAllocation ? BLK_ERR_OOM : BLK_ERR_CUDA,                    \
                                  std::string(#expr) + ": " + cudaGetErrorString(e__));                             \
    } while (0)

void log_msg(int level, const std::string& s);

struct LayerWeights {
    QMat wq, wk, wv, wo, gate, up, down;
    const float* attn_norm = nullptr;
    const float* ffn_norm = nullptr;
    const float* bq = nullptr;
    const float* bk = nullptr;
    const float* bv = nullptr;
};

// Threshold top-64 of `rows` logits rows (topk_select_kernel, decode_kernels.cuh): the selector's scratch in the layout TopkArgs
// indexes, the device lists and their pinned copies.  Between selections every chunk maximum holds the empty key and both
// counters are zero (the selector restores that after reading).
struct TopkRows {
    int rows = 0;
    int* chunk_max = nullptr; float* cand_l = nullptr; int* cand_i = nullptr; unsigned int* counters = nullptr;
    int32_t* ids = nullptr; float* logits = nullptr;          // device [rows][TOPK_MAX]
    int32_t* h_ids = nullptr; float* h_logits = nullptr;      // pinned [rows][TOPK_MAX]
};

} // namespace blk

// persistent decode kernel: stream copy of the weights + phase table (mega_decode.cuh)
struct blk_mega_model {
    bool ok = false;
    std::vector<blk::MegaPhase> phases;      // host copy (device pointers inside)
    blk::MegaPhase* d_phases = nullptr;
    uint4* d_list = nullptr; int* d_counts = nullptr; int* d_counts_body = nullptr; int list_stride = 0;
    uint8_t* arena = nullptr; size_t arena_bytes = 0;
    int n_cta = 0, slot_bytes = 0, max_items = 0, act_bytes = 0, ts_cap = 0, attn_off = 0;
};

struct blk_model {
    int device = 0;
    blk_mega_model mega;
    std::string arch;
    int n_vocab = 0, n_embd = 0, n_layer = 0, n_head = 0, n_head_kv = 0, d_head = 0, n_ff = 0, n_ctx_train = 0, n_rot = 0;
    float rms_eps = 1e-5f, rope_theta = 10000.0f, theta_scale = 1.0f;
    bool neox = false;
    int tok_bos = -1, tok_eos = -1, tok_eot = -1, tok_eom = -1;
    bool add_bos = false;
    std::vector<blk::LayerWeights> layers;
    blk::QMat tok_embd, output;
    const float* out_norm = nullptr;
    const float* rope_freqs = nullptr;
    std::vector<void*> allocs;
    std::vector<std::string> vocab;
    std::vector<int32_t> token_type;          // tokenizer.ggml.token_type (1 normal, 2 unknown, 3 control, 4 user defined, 5 unused, 6 byte)
    std::vector<std::string> merges;          // tokenizer.ggml.merges ("left right", rank = index)
    std::vector<uint8_t> eog;                 // per token: end-of-generation (ids from the metadata + the token texts llama.cpp recognises)
    bool add_eos = false;
    bool vocab_only = false;                  // metadata + vocabulary only: no device, no weights (Model::Params::vocabOnly)
    std::map<std::string, std::string> meta;
    int64_t weight_bytes_per_token = 0;
    int act_fmt = blk::ACT_F32;       // activation format of the layer mat-vecs
    // Resident bf16 copies ("panels") of the layer matrices for the TMA-fed tcgen05 GEMMs of the multi-token paths (prompt prefill,
    // verify, batched decode): B200 has 180 GB, an 8B model's panels are 14 GB.  Filled once, by the first multi-token pass that
    // wants them, into whatever device memory is free beyond a reserve (BLK_PANEL_CACHE_GB caps it, 0 = off); indexed by GEMM op
    // (gemm_op in engine.cu); nullptr = not resident (streamed through the per-context panels).
    struct PanelCache { std::mutex mu; bool built = false; std::vector<__nv_bfloat16*> op; std::vector<void*> allocs; size_t bytes = 0; int n_resident = 0; } panels;
    ~blk_model();
};

struct blk_ctx {
    blk_model* m = nullptr;
    int n_ctx = 0, n_batch = 0, n_past = 0;   // n_past: cells in the cache = cell index of the next token
    int n_pages = 0, n_split = 1;
    int verify_mode = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t pf_stream = nullptr;      // side stream of the prefill panel fills (one GEMM ahead of the main stream) and the model panel cache
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<void*> allocs;
    std::vector<void*> host_allocs;
    // KV pages
    std::vector<__half*> k_pool, v_pool;
    __half** d_kpools = nullptr; __half** d_vpools = nullptr;      // device arrays of the per-layer pool pointers
    int32_t* page_table = nullptr;
    std::vector<int32_t> page_table_host;                          // host copy of the page table (state save / restore)
    // decode-step state
    int32_t* d_tok = nullptr;
    // KV cell bookkeeping (engine.cu): every path that adds cells goes through begin_cells / end_cells, every reset through
    // reset_cells, and only upload_pos writes d_pos from the host.
    int32_t* d_pos = nullptr;             // device [2]: {n_past, rope_off}; the kernels that add cells advance word 0
    // Self-Extend (llama_kv_self_seq_add / seq_div, reference Session.cpp:348-368): cell positions other than the cell index.
    // Materialised on the first such call; empty = every cell's position is its index (the normal case, nothing is touched).
    std::vector<int32_t> cell_pos, cell_shift;      // position of every cell; rotation delta not yet applied to its K row
    int32_t* d_cell_shift = nullptr;                // device [n_ctx]: cell_shift staged for the K re-rotation
    int rope_off = 0;                               // rotary position of the next token - n_past
    bool shift_pending = false;                     // some cell_shift is non-zero: applied to the K rows before the cache is read
    static constexpr int TOK_RING = 256;
    int32_t* h_tok = nullptr;             // pinned ring [TOK_RING]
    int tok_slot = 0;
    float* x = nullptr;                   // residual stream [d]
    float* qbuf = nullptr;                // [n_head*d_head]
    float* hbuf = nullptr;                // [n_ff]
    float2* rope_cs = nullptr;            // [d_head/2]
    blk::ActBuf act_d, act_q, act_q2, act_ff;
    int attn_cluster = 0, attn_cap = 0;   // cluster size (0 = three-kernel fallback) and tokens per CTA
    float* part_o = nullptr; float* scores = nullptr;
    float* logits = nullptr;              // [n_vocab] of the last decoded token
    blk::TopkRows top;                    // its top-64
    int n_chunks = 0; int chunk_shift = 10; int cand_cap = 2048;      // vocabulary chunks and candidates per row of every selection
    bool have_logits = false;
    cudaGraphExec_t g_full = nullptr, g_body = nullptr, g_loop = nullptr;
    int64_t launches_full = 0, launches_body = 0, launches_loop = 0;
    int64_t launches = 0;
    // per-kernel event timing of one eagerly launched step (blk_profile_step)
    bool profiling = false;
    std::vector<std::pair<const char*, cudaEvent_t>> prof_marks;
    // multi-token prefill workspaces (allocated on first use, sized for pf_cap tokens)
    int pf_cap = 0, pf_logit_rows = 0;
    int32_t* pf_tokens = nullptr; float2* pf_rope = nullptr;
    float* pf_x = nullptr; __nv_bfloat16* pf_xn = nullptr; float* pf_qkv = nullptr; __half* pf_q = nullptr;
    __nv_bfloat16* pf_ao = nullptr; __nv_bfloat16* pf_h = nullptr;
    float* pf_logits = nullptr;
    __half* pf_vt = nullptr; int pf_vt_pad = 0;           // transposed V of one layer for the tcgen05 prefill attention
    float* pf_splitk = nullptr; size_t pf_splitk_elems = 0;               // partial sums of the split-K prefill GEMMs (few-token batches)
    __nv_bfloat16* pf_panel[4] = {nullptr, nullptr, nullptr, nullptr};     // bf16 weight panels of the two-pass GEMM form, one per GEMM kind
    cudaEvent_t pn_filled[4] = {nullptr, nullptr, nullptr, nullptr}, pn_start[4] = {nullptr, nullptr, nullptr, nullptr};
    int panel_min = 257;  // matrices that are NOT resident (model panel cache): streamed two-pass GEMM form from this many tokens per chunk on
                          // (0 = never); measured (tools/prefill_sweep.py): up to one 256-token M tile the fused form wins, beyond it the two-pass form
    bool panel_tried = false;
    int32_t* pf_claimed = nullptr; int32_t* pf_nclaimed = nullptr; float* pf_gath = nullptr; int32_t* pf_topi = nullptr; float* pf_topl = nullptr;
    int prefill_min = 32;                  // blk_decode / blk_verify_prefill use the tcgen05 path from this many tokens on
    // scratch for gather / verify
    int32_t* d_ids = nullptr; float* d_gath = nullptr; int ids_cap = 0;
    void* flush_buf = nullptr; size_t flush_bytes = 0;
    // batched decode step (blk_decode_batch): per-row descriptors (pinned host staging + device copy) and the top-64 of every row
    uint8_t* bd_host = nullptr; uint8_t* bd_dev = nullptr;
    blk::TopkRows bd_top;
    // logit edit pass (blk_*_edited, logit_edit.cuh), allocated on first use for ed_top.rows rows: the edited copies and a selection
    // of their own (the raw selection stays untouched), plus the packed edit lists (pinned staging + device copy)
    float* ed_logits = nullptr;
    blk::TopkRows ed_top;
    uint8_t* ed_stage_h = nullptr; uint8_t* ed_stage_d = nullptr; size_t ed_stage_cap = 0;
    // persistent decode kernel (one cooperative launch per token instead of the per-op graph)
    bool mega_on = false;
    blk::MegaParams mega_params{};
    size_t mega_smem = 0;
    uint32_t mega_seq = 0;
    int* mega_err = nullptr;               // mapped host word the kernel sets when a poll times out
    ~blk_ctx();
};
