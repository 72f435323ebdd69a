// engine.cu -- model loading, context, decode step and the C ABI (include/blama_b200.h).
//
// Replaces, for blama's hot path, what llama.cpp does under llama_model_load_from_file / llama_init_from_model /
// llama_decode / llama_get_logits_ith (reference call sites: Model.cpp:50-53, Instance.cpp:34-48, Session.cpp:388,
// Session.cpp:24).  There is no CPU fallback anywhere in this file: without a device every entry point fails.
#include "engine.hpp"
#include "gemv_kernels.cuh"
#include "gguf.hpp"
#include "prefill.hpp"
#include "prefill_kernels.cuh"
#include "batch_decode.cuh"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <random>
#include <tuple>

using namespace blk;

// ------------------------------------------------------------------------------------------------------------------
// logging / errors
// ------------------------------------------------------------------------------------------------------------------
namespace {
thread_local std::string g_last_error;
blk_log_cb g_log_cb = nullptr;
void* g_log_user = nullptr;
std::once_flag g_init_once;
int g_device_count = 0;

blk_status fail(blk_status code, const std::string& msg) {
    g_last_error = msg;
    log_msg(3, msg);
    return code;
}
template <class F> blk_status guarded(F&& f) {
    try { f(); return BLK_OK; }
    catch (const BlkError& e) { return fail(e.code, e.what()); }
    catch (const std::bad_alloc&) { return fail(BLK_ERR_OOM, "host allocation failed"); }
    catch (const std::exception& e) { return fail(BLK_ERR_FORMAT, e.what()); }
}
} // namespace

void blk::log_msg(int level, const std::string& s) {
    if (g_log_cb) g_log_cb(level, s.c_str(), g_log_user);
    else if (level >= 2) fprintf(stderr, "[blama_b200] %s\n", s.c_str());
}

extern "C" blk_status blk_init(void) {
    std::call_once(g_init_once, [] {
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess) { n = 0; (void)cudaGetLastError(); }
        g_device_count = n;
    });
    if (g_device_count <= 0) return fail(BLK_ERR_NO_DEVICE, "no CUDA device available (blama_b200 has no CPU fallback)");
    return BLK_OK;
}
extern "C" void blk_set_log_callback(blk_log_cb cb, void* user) { g_log_cb = cb; g_log_user = user; }
extern "C" const char* blk_last_error(void) { return g_last_error.c_str(); }
extern "C" int32_t blk_device_count(void) { blk_init(); return g_device_count; }
extern "C" const char* blk_version(void) { return "blama_b200 0.1 (sm_100a)"; }

// ------------------------------------------------------------------------------------------------------------------
// model
// ------------------------------------------------------------------------------------------------------------------
blk_model::~blk_model() {
    if (allocs.empty()) return;          // vocabulary-only models never touched a device
    cudaSetDevice(device);
    for (void* p : allocs) cudaFree(p);
    for (void* p : panels.allocs) cudaFree(p);
}

namespace {

struct Uploader {
    blk_model* m;
    uint8_t* staging = nullptr; size_t staging_bytes = 0;
    uint8_t* arena = nullptr; size_t arena_off = 0, arena_bytes = 0;
    cudaStream_t stream = nullptr;

    uint8_t* take(size_t n) {
        uint8_t* p = arena + arena_off;
        arena_off += (n + 255) & ~size_t(255);
        if (arena_off > arena_bytes) throw BlkError(BLK_ERR_OOM, "weight arena overflow");
        return p;
    }
    static size_t planes_bytes(const GgufTensor& t) {
        // split planes are padded to 256 B each; worst case 4 planes
        return t.nbytes + 4 * 256;
    }
    QMat upload_matrix(const GgufTensor& t) {
        QMat W; W.type = t.type; W.K = (int)t.ne[0]; W.N = (int)t.n_rows(); W.bytes = t.nbytes;
        const int64_t K = W.K, N = W.N;
        if (t.type == GT_F32 || t.type == GT_F16) {
            uint8_t* dst = take(t.nbytes);
            BLK_CUDA(cudaMemcpyAsync(dst, t.data, t.nbytes, cudaMemcpyHostToDevice, stream));
            W.p0 = dst;
            if (K % 8) throw BlkError(BLK_ERR_FORMAT, "row length must be a multiple of 8: " + t.name);
            return W;
        }
        BLK_CUDA(cudaMemcpyAsync(staging, t.data, t.nbytes, cudaMemcpyHostToDevice, stream));
        const int threads = 128;
        if (t.type == GT_Q4_K) {
            const int64_t nb = N * (K / 256);
            uint8_t* qs = take(nb * 128); uint8_t* hdr = take(nb * 16);
            retile_q4k_kernel<<<(unsigned)((nb + threads - 1) / threads), threads, 0, stream>>>(staging, qs, hdr, nb);
            W.p0 = qs; W.p1 = hdr;
        } else if (t.type == GT_Q5_K) {
            const int64_t nb = N * (K / 256);
            uint8_t* qs = take(nb * 128); uint8_t* hdr = take(nb * 16); uint8_t* qh = take(nb * 32);
            retile_q5k_kernel<<<(unsigned)((nb + threads - 1) / threads), threads, 0, stream>>>(staging, qs, hdr, qh, nb);
            W.p0 = qs; W.p1 = hdr; W.p2 = qh;
        } else if (t.type == GT_Q6_K) {
            const int64_t nb = N * (K / 256);
            uint8_t* ql = take(nb * 128); uint8_t* qh = take(nb * 64); uint8_t* sc = take(nb * 16); uint8_t* d = take(nb * 2);
            retile_q6k_kernel<<<(unsigned)((nb + threads - 1) / threads), threads, 0, stream>>>(staging, ql, qh, sc, d, nb);
            W.p0 = ql; W.p1 = qh; W.p2 = sc; W.p3 = d;
        } else if (t.type == GT_Q8_0) {
            const int64_t nb = N * (K / 32);
            uint8_t* qs = take(nb * 32); uint8_t* d = take(nb * 2);
            retile_q80_kernel<<<(unsigned)((nb + threads - 1) / threads), threads, 0, stream>>>(staging, qs, d, nb);
            W.p0 = qs; W.p1 = d;
        } else {
            throw BlkError(BLK_ERR_FORMAT, "unsupported tensor type for " + t.name);
        }
        BLK_CUDA(cudaGetLastError());
        BLK_CUDA(cudaStreamSynchronize(stream));      // staging is reused by the next tensor
        return W;
    }
    const float* upload_f32(const GgufTensor& t) {
        if (t.type != GT_F32) throw BlkError(BLK_ERR_FORMAT, "expected F32 tensor: " + t.name);
        uint8_t* dst = take(t.nbytes);
        BLK_CUDA(cudaMemcpyAsync(dst, t.data, t.nbytes, cudaMemcpyHostToDevice, stream));
        return reinterpret_cast<const float*>(dst);
    }
};

} // namespace


// ------------------------------------------------------------------------------------------------------------------
// persistent decode kernel: plan the stream copy (phases, segments, chunk geometry) from the tensor types
// ------------------------------------------------------------------------------------------------------------------
namespace {
struct MegaHook { int phase, seg, rowmap, ab; };       // where (and how) a GGUF tensor lands in the stream copy
struct MegaPlan {
    bool ok = false;
    std::map<std::string, std::vector<MegaHook>> hooks;
    std::vector<size_t> seg_off[3];                    // arena offsets per phase / segment
    size_t arena_bytes = 0;
};

bool mega_type_ok(int t) { return t == QT_Q4_K || t == QT_Q5_K || t == QT_Q6_K || t == QT_Q8_0; }

// K -> (warps per row pair, lanes per slice, row slices per chunk)
bool mega_geometry(int K, int& W, int& L, int& rpc) {
    if (K <= 0 || K % 256) return false;
    const int halfs = K / 128;
    W = (halfs + 31) / 32;
    L = (halfs + W - 1) / W; L += L & 1;
    rpc = (2 * L <= 32) ? 2 : 1;
    return W <= MG_WARPS;
}

MegaPlan mega_plan(blk_model* m, GgufFile& f, int n_sms) {
    MegaPlan pl;
    blk_mega_model& mg = m->mega;
    { const char* e = getenv("BLK_MEGA"); if (e && e[0] == '0') return pl; }
    const int d = m->n_embd, dh = m->d_head, dq = m->n_head * dh, dkv = m->n_head_kv * dh, ff = m->n_ff, V = m->n_vocab;
    if (V % 2 || dq % 256 || d % 256 || ff % 256 || n_sms < m->n_head_kv) return pl;
    auto ttype = [&](const std::string& n) -> int { const GgufTensor* t = f.find(n); return t ? t->type : -1; };
    const bool tied = f.find("output.weight") == nullptr;
    mg.n_cta = n_sms;
    int max_items = 1, slot = 0, kmax = 0;
    bool bad = false;
    auto add_phase = [&](int layer, int K, int src, std::initializer_list<std::tuple<std::string, int, int, int, int>> segs /*tensor, n_pairs, kind, rowmap, ab*/) {
        MegaPhase ph{};
        if (!mega_geometry(K, ph.W, ph.L, ph.rpc)) { bad = true; return; }
        ph.K = K; ph.src = src; ph.layer = layer; ph.nseg = 0;
        const int NGtot = mg.n_cta * (MG_WARPS / ph.W);
        int items = 0;
        // The segments of a phase occupy consecutive warp groups, starting so that the chain ENDS at the last group: the groups that
        // carry one pair more than the others are the highest CTAs.  CTAs 0 .. n_head_kv * n_split - 1 run the attention stages (and
        // CTAs 0 .. n_head_kv - 1 the split combine), so the extra QKV pairs and the idle groups of Wo keep off the attention's path.
        int64_t total = 0;
        for (auto& sgd : segs) if (!(std::get<2>(sgd) == MK_SWIGLU && std::get<4>(sgd) == 1)) total += std::get<1>(sgd);
        int64_t rot_acc = (NGtot - total % NGtot) % NGtot;          // first group of the chain
        const int pi = (int)mg.phases.size();
        for (auto& sgd : segs) {
            const std::string& name = std::get<0>(sgd);
            const int type = ttype(name);
            if (!mega_type_ok(type)) { bad = true; return; }
            const int kind = std::get<2>(sgd);
            const bool new_seg = !(kind == MK_SWIGLU && std::get<4>(sgd) == 1);     // ffn_up shares the gate segment
            const int si = new_seg ? ph.nseg : ph.nseg - 1;
            if (new_seg) {
                MegaSeg& sg = ph.seg[si];
                sg.type = type; sg.n_pairs = std::get<1>(sgd); sg.kind = kind;
                sg.slice_bytes = mg_slice_bytes(type, ph.L / 2);
                sg.rot = (int)((NGtot - rot_acc % NGtot) % NGtot); rot_acc += sg.n_pairs;     // group gg starts at pair (gg + rot) mod NGtot
                sg.slot0 = items;
                sg.bias = nullptr; sg.base = nullptr;
                pl.seg_off[si].resize(pi + 1, 0);
                pl.seg_off[si][pi] = pl.arena_bytes;
                pl.arena_bytes += (size_t)sg.n_pairs * ph.W * 2 * sg.slice_bytes;
                pl.arena_bytes = (pl.arena_bytes + 255) & ~size_t(255);
                items += (sg.n_pairs + NGtot - 1) / NGtot;
                slot = std::max(slot, sg.slice_bytes * ph.rpc);
                ph.nseg++;
            } else if (type != ph.seg[si].type) { bad = true; return; }
            pl.hooks[name].push_back({pi, si, std::get<3>(sgd), std::get<4>(sgd)});
        }
        ph.act_fmt = act_format_for(ph.seg[0].type);
        for (int s = 1; s < ph.nseg; s++) if (act_format_for(ph.seg[s].type) != ph.act_fmt) bad = true;
        ph.items = items;
        ph.NG = MG_WARPS / ph.W;
        auto ilog2 = [](int v) { int s = 0; while ((1 << s) < v) s++; return (1 << s) == v ? s : -1; };
        ph.wsh = ilog2(ph.W); ph.ngsh = ilog2(ph.NG);
        if (src == MSRC_X && K > 2 * MG_WARPS * 256) bad = true;   // RMS-normed source rows: at most 2 blocks of 256 per warp
        max_items = std::max(max_items, items);
        kmax = std::max(kmax, K);
        mg.phases.push_back(ph);
    };
    const int qk_map = m->neox ? 1 : 0;
    for (int l = 0; l < m->n_layer && !bad; l++) {
        const std::string p = "blk." + std::to_string(l) + ".";
        add_phase(l, d, MSRC_X, {{p + "attn_q.weight", dq / 2, MK_Q, qk_map, 0}, {p + "attn_k.weight", dkv / 2, MK_K, qk_map, 0}, {p + "attn_v.weight", dkv / 2, MK_V, 0, 0}});
        add_phase(l, dq, MSRC_ATTN, {{p + "attn_output.weight", d / 2, MK_RESID, 0, 0}});
        add_phase(l, d, MSRC_X, {{p + "ffn_gate.weight", ff, MK_SWIGLU, 2, 0}, {p + "ffn_up.weight", ff, MK_SWIGLU, 2, 1}});
        add_phase(l, ff, MSRC_H, {{p + "ffn_down.weight", d / 2, MK_RESID, 0, 0}});
    }
    if (!bad) add_phase(m->n_layer, d, MSRC_X, {{tied ? "token_embd.weight" : "output.weight", V / 2, MK_LOGITS, 0, 0}});
    if (bad) { mg.phases.clear(); return pl; }
    const int gq = m->n_head / m->n_head_kv;
    const int act_q = kmax + kmax / 4;
    mg.slot_bytes = (slot + 127) / 128 * 128;
    mg.max_items = max_items;
    MegaParams probe{}; probe.slot_bytes = mg.slot_bytes; probe.max_items = mg.max_items; probe.d_head = dh; probe.n_layer = m->n_layer;
    int limit = 0;
    (void)mega_setup(0, &limit); (void)cudaGetLastError();
    // attention tile: the largest power of two (<= 64 tokens) whose K + V rows fit beside the ring
    mg.ts_cap = 0;
    mg.attn_off = (d + d / 4 + 127) / 128 * 128;       // the tiles sit behind the (small) activations of the QKV phase
    for (int ts = 64; ts >= 8; ts >>= 1) {
        const int act_attn = mg.attn_off + gq * dh * 2 + gq * ts * 4 + std::max(2 * ts * dh * 2, MG_THREADS * gq * 4);
        probe.act_bytes = (std::max(act_q, act_attn) + 127) / 128 * 128;
        if (mega_smem_bytes(probe) <= (size_t)limit) { mg.ts_cap = ts; mg.act_bytes = probe.act_bytes; break; }
    }
    if (!mg.ts_cap || mega_setup(mega_smem_bytes(probe), &limit) != cudaSuccess) {
        (void)cudaGetLastError();
        log_msg(1, "persistent decode kernel disabled: needs " + std::to_string(mega_smem_bytes(probe)) + " B of shared memory");
        mg.phases.clear(); return pl;
    }
    pl.ok = true;
    return pl;
}
} // namespace

namespace {
// hyper-parameters, special tokens and the vocabulary (what llama.cpp's llm_load_hparams / llama_vocab::load read).
// vocab_only: the architecture is not restricted and no tensor geometry is needed.
void load_metadata(blk_model* m, GgufFile& f, bool vocab_only) {
    const std::string* arch = f.str("general.architecture");
    if (!arch) throw BlkError(BLK_ERR_FORMAT, "gguf: no general.architecture");
    m->arch = *arch;
    if (!vocab_only) {
        if (m->arch != "llama" && m->arch != "qwen2") throw BlkError(BLK_ERR_FORMAT, "unsupported architecture: " + m->arch);
        auto hp = [&](const char* k) { return f.num_required(m->arch + "." + k); };
        auto hpd = [&](const char* k, double d) { return f.num(m->arch + "." + k, d); };
        auto pos_int = [&](double v, const char* what, double hi) -> int {
            if (!(v >= 1 && v <= hi) || v != (double)(long long)v) throw BlkError(BLK_ERR_FORMAT, std::string("gguf: bad ") + what);
            return (int)v;
        };
        m->n_embd = pos_int(hp("embedding_length"), "embedding_length", 1 << 20);
        m->n_layer = pos_int(hp("block_count"), "block_count", 4096);
        m->n_ff = pos_int(hp("feed_forward_length"), "feed_forward_length", 1 << 24);
        m->n_head = pos_int(hp("attention.head_count"), "attention.head_count", 4096);
        m->n_head_kv = pos_int(hpd("attention.head_count_kv", m->n_head), "attention.head_count_kv", 4096);
        m->n_ctx_train = pos_int(hp("context_length"), "context_length", 1 << 30);
        m->rms_eps = (float)hpd("attention.layer_norm_rms_epsilon", 1e-5);
        m->rope_theta = (float)hpd("rope.freq_base", 10000.0);
        if (m->n_embd % m->n_head) throw BlkError(BLK_ERR_FORMAT, "gguf: embedding_length is not a multiple of head_count");
        m->d_head = m->n_embd / m->n_head;
        m->n_rot = pos_int(hpd("rope.dimension_count", m->d_head), "rope.dimension_count", 1 << 16);
        m->neox = (m->arch == "qwen2");
        m->theta_scale = powf(m->rope_theta, -2.0f / (float)m->n_rot);
        if (m->n_rot != m->d_head) throw BlkError(BLK_ERR_FORMAT, "partial rotary dimensions are not supported");
        if (m->d_head != 64 && m->d_head != 128) throw BlkError(BLK_ERR_FORMAT, "head size must be 64 or 128");
        if (m->n_head % m->n_head_kv || m->n_head / m->n_head_kv > MAX_GQ) throw BlkError(BLK_ERR_FORMAT, "unsupported GQA ratio");
        if ((m->n_head * m->d_head) % 256 || m->n_embd % 256 || m->n_ff % 256) throw BlkError(BLK_ERR_FORMAT, "model widths must be multiples of 256");
    }
    m->vocab_only = vocab_only;
    m->tok_bos = (int)f.num("tokenizer.ggml.bos_token_id", -1);
    m->tok_eos = (int)f.num("tokenizer.ggml.eos_token_id", -1);
    m->tok_eot = (int)f.num("tokenizer.ggml.eot_token_id", -1);
    m->tok_eom = (int)f.num("tokenizer.ggml.eom_token_id", -1);
    m->add_bos = f.num("tokenizer.ggml.add_bos_token", 0) != 0;
    m->add_eos = f.num("tokenizer.ggml.add_eos_token", 0) != 0;
    if (const auto* v = f.str_array("tokenizer.ggml.tokens")) m->vocab = *v;
    if (const auto* v = f.str_array("tokenizer.ggml.merges")) m->merges = *v;
    if (const auto* v = f.int_array("tokenizer.ggml.token_type")) { m->token_type.resize(v->size()); for (size_t i = 0; i < v->size(); i++) m->token_type[i] = (int32_t)(*v)[i]; }
    if (m->token_type.size() != m->vocab.size()) m->token_type.assign(m->vocab.size(), 1);
    for (const char* k : {"general.name", "general.architecture", "tokenizer.chat_template", "tokenizer.ggml.model", "tokenizer.ggml.pre"})
        if (const std::string* s = f.str(k)) m->meta[k] = *s;
    // End-of-generation set: the metadata ids plus the token texts llama.cpp's vocabulary loader recognises (llama-vocab.cpp,
    // "special_eog_ids"): real Llama-3 / Qwen2 files mark <|eot_id|> / <|im_end|> only through their text.
    m->eog.assign(m->vocab.size(), 0);
    static const char* const eog_texts[] = {"<|eot_id|>", "<|im_end|>", "<|end|>", "<end_of_turn>", "<|endoftext|>", "<|eom_id|>", "<EOT>", "_<EOT>"};
    for (size_t i = 0; i < m->vocab.size(); i++)
        for (const char* t : eog_texts) if (m->vocab[i] == t) { m->eog[i] = 1; if (m->token_type[i] == 1) m->token_type[i] = 3; }
    for (int id : {m->tok_eos, m->tok_eot, m->tok_eom}) if (id >= 0 && (size_t)id < m->eog.size()) m->eog[(size_t)id] = 1;
}
} // namespace

extern "C" blk_model* blk_model_load(const char* path, int32_t device, blk_progress_cb cb, void* user) {
    if (blk_init() != BLK_OK) return nullptr;
    if (device < 0 || device >= g_device_count) { fail(BLK_ERR_ARG, "bad device index"); return nullptr; }
    std::unique_ptr<blk_model> m(new blk_model());
    m->device = device;
    blk_status st = guarded([&] {
        std::unique_ptr<GgufFile> fp;
        try { fp.reset(new GgufFile(path)); }
        catch (const std::exception& e) {
            const std::string w = e.what();
            throw BlkError(w.rfind("gguf:", 0) == 0 ? BLK_ERR_FORMAT : BLK_ERR_IO, w);
        }
        GgufFile& f = *fp;
        load_metadata(m.get(), f, false);

        BLK_CUDA(cudaSetDevice(device));
        Uploader up; up.m = m.get();
        BLK_CUDA(cudaStreamCreateWithFlags(&up.stream, cudaStreamNonBlocking));
        size_t total = 0, biggest = 0;
        for (const GgufTensor& t : f.tensors()) { total += Uploader::planes_bytes(t); biggest = std::max(biggest, t.nbytes); }
        up.arena_bytes = total;
        BLK_CUDA(cudaMalloc(&up.arena, up.arena_bytes)); m->allocs.push_back(up.arena);
        BLK_CUDA(cudaMalloc(&up.staging, biggest)); up.staging_bytes = biggest;
        struct StagingGuard { uint8_t* p; cudaStream_t s; ~StagingGuard() { cudaFree(p); cudaStreamDestroy(s); } } sg{up.staging, up.stream};

        const size_t n_t = f.tensors().size(); size_t done = 0;
        auto progress = [&]() { done++; if (cb && !cb((float)done / (float)n_t, user)) throw BlkError(BLK_ERR_IO, "model load aborted by the progress callback"); };
        auto need = [&](const std::string& n) -> const GgufTensor& { const GgufTensor* t = f.find(n); if (!t) throw BlkError(BLK_ERR_FORMAT, "gguf: missing tensor " + n); return *t; };
        MegaPlan mplan;        // filled once the hyper-parameters are known (below)
        // scatter the raw tensor still sitting in the staging buffer into the stream copy of the persistent decode kernel
        auto mega_scatter = [&](const GgufTensor& t) {
            if (!mplan.ok) return;
            auto it = mplan.hooks.find(t.name);
            if (it == mplan.hooks.end()) return;
            for (const MegaHook& hk : it->second) {
                const MegaPhase& ph = m->mega.phases[hk.phase];
                const MegaSeg& sg = ph.seg[hk.seg];
                BLK_CUDA(mega_build_stream(up.staging, const_cast<uint8_t*>(sg.base), t.type, (int)t.n_rows(), (int)t.ne[0], ph.W, ph.L / 2, sg.slice_bytes,
                                           hk.rowmap, m->d_head, hk.ab, up.stream));
            }
            BLK_CUDA(cudaStreamSynchronize(up.stream));
        };
        auto mat = [&](const std::string& n, int K, int N) {
            const GgufTensor& t = need(n);
            if (t.ne[0] != K || t.n_rows() != N) throw BlkError(BLK_ERR_FORMAT, "gguf: unexpected shape for " + n);
            QMat W = up.upload_matrix(t); mega_scatter(t); progress(); return W;
        };
        auto vec = [&](const std::string& n, int len, bool required) -> const float* {
            const GgufTensor* t = f.find(n);
            if (!t) { if (required) throw BlkError(BLK_ERR_FORMAT, "gguf: missing tensor " + n); return nullptr; }
            if (t->ne[0] != len) throw BlkError(BLK_ERR_FORMAT, "gguf: unexpected shape for " + n);
            const float* p = up.upload_f32(*t); progress(); return p;
        };
        const int d = m->n_embd, dq = m->n_head * m->d_head, dkv = m->n_head_kv * m->d_head, ff = m->n_ff;
        {
            const GgufTensor& te = need("token_embd.weight");
            if (te.ne[0] != d) throw BlkError(BLK_ERR_FORMAT, "gguf: unexpected shape for token_embd.weight");
            m->n_vocab = (int)te.n_rows();
            {   // plan the persistent decode kernel's stream copy (second copy of the weights, laid out per warp chunk)
                int n_sms = 0;
                BLK_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, device));
                mplan = mega_plan(m.get(), f, n_sms);
                if (mplan.ok) {
                    blk_mega_model& mg = m->mega;
                    mg.arena_bytes = mplan.arena_bytes;
                    if (cudaMalloc(&mg.arena, mg.arena_bytes) != cudaSuccess) { (void)cudaGetLastError(); mplan.ok = false; mg.phases.clear(); mg.arena = nullptr; }
                    else {
                        m->allocs.push_back(mg.arena);
                        BLK_CUDA(cudaMemsetAsync(mg.arena, 0, mg.arena_bytes, up.stream));
                        for (size_t pi = 0; pi < mg.phases.size(); pi++)
                            for (int s = 0; s < mg.phases[pi].nseg; s++) mg.phases[pi].seg[s].base = mg.arena + mplan.seg_off[s][pi];
                    }
                }
            }
            m->tok_embd = up.upload_matrix(te); mega_scatter(te); progress();
        }
        m->layers.resize(m->n_layer);
        int64_t wb = 0;
        for (int l = 0; l < m->n_layer; l++) {
            const std::string p = "blk." + std::to_string(l) + ".";
            LayerWeights& L = m->layers[l];
            L.attn_norm = vec(p + "attn_norm.weight", d, true);
            L.wq = mat(p + "attn_q.weight", d, dq); L.wk = mat(p + "attn_k.weight", d, dkv); L.wv = mat(p + "attn_v.weight", d, dkv);
            L.bq = vec(p + "attn_q.bias", dq, false); L.bk = vec(p + "attn_k.bias", dkv, false); L.bv = vec(p + "attn_v.bias", dkv, false);
            L.wo = mat(p + "attn_output.weight", dq, d);
            L.ffn_norm = vec(p + "ffn_norm.weight", d, true);
            L.gate = mat(p + "ffn_gate.weight", d, ff); L.up = mat(p + "ffn_up.weight", d, ff); L.down = mat(p + "ffn_down.weight", ff, d);
            if (L.gate.type != L.up.type) throw BlkError(BLK_ERR_FORMAT, "ffn_gate / ffn_up must share a type");
            const int fam = act_format_for(L.wq.type);
            for (const QMat* W : {&L.wk, &L.wv, &L.wo, &L.gate, &L.up, &L.down})
                if (act_format_for(W->type) != fam) throw BlkError(BLK_ERR_FORMAT, "mixed quantisation families within a model are not supported");
            if (l == 0) m->act_fmt = fam; else if (fam != m->act_fmt) throw BlkError(BLK_ERR_FORMAT, "mixed quantisation families across layers");
            wb += (int64_t)(L.wq.bytes + L.wk.bytes + L.wv.bytes + L.wo.bytes + L.gate.bytes + L.up.bytes + L.down.bytes) + 2 * 4 * d;
            if (L.bq) wb += 4 * (dq + 2 * dkv);
        }
        m->out_norm = vec("output_norm.weight", d, true);
        if (f.find("output.weight")) m->output = mat("output.weight", d, m->n_vocab); else m->output = m->tok_embd;
        m->rope_freqs = vec("rope_freqs.weight", m->d_head / 2, false);
        wb += (int64_t)m->output.bytes + 4 * d;
        m->weight_bytes_per_token = wb;
        if (mplan.ok) {   // norms / biases are known now: finish the phase table, upload it, build the per-warp chunk lists
            blk_mega_model& mg = m->mega;
            for (MegaPhase& ph : mg.phases) {
                if (ph.layer < m->n_layer) {
                    const LayerWeights& L = m->layers[ph.layer];
                    if (ph.seg[0].kind == MK_Q) { ph.norm_w = L.attn_norm; ph.seg[0].bias = L.bq; ph.seg[1].bias = L.bk; ph.seg[2].bias = L.bv; }
                    else if (ph.seg[0].kind == MK_SWIGLU) ph.norm_w = L.ffn_norm;
                } else ph.norm_w = m->out_norm;
            }
            BLK_CUDA(cudaMalloc(&mg.d_phases, mg.phases.size() * sizeof(MegaPhase))); m->allocs.push_back(mg.d_phases);
            BLK_CUDA(cudaMemcpyAsync(mg.d_phases, mg.phases.data(), mg.phases.size() * sizeof(MegaPhase), cudaMemcpyHostToDevice, up.stream));
            const int n_w = mg.n_cta * MG_WARPS;
            BLK_CUDA(cudaMalloc(&mg.d_counts, n_w * sizeof(int))); m->allocs.push_back(mg.d_counts);
            BLK_CUDA(mega_chunk_lists(mg.d_phases, (int)mg.phases.size(), mg.n_cta, nullptr, 0, mg.d_counts, up.stream));
            std::vector<int> counts(n_w);
            BLK_CUDA(cudaMemcpyAsync(counts.data(), mg.d_counts, n_w * sizeof(int), cudaMemcpyDeviceToHost, up.stream));
            BLK_CUDA(cudaStreamSynchronize(up.stream));
            mg.list_stride = std::max(1, *std::max_element(counts.begin(), counts.end()));
            BLK_CUDA(cudaMalloc(&mg.d_list, (size_t)n_w * mg.list_stride * sizeof(uint4))); m->allocs.push_back(mg.d_list);
            BLK_CUDA(mega_chunk_lists(mg.d_phases, (int)mg.phases.size(), mg.n_cta, mg.d_list, mg.list_stride, mg.d_counts, up.stream));
            // a step without the lm_head (prompt tokens fed one by one) must not prefetch the head's chunks
            BLK_CUDA(cudaMalloc(&mg.d_counts_body, n_w * sizeof(int))); m->allocs.push_back(mg.d_counts_body);
            BLK_CUDA(mega_chunk_lists(mg.d_phases, (int)mg.phases.size() - 1, mg.n_cta, nullptr, 0, mg.d_counts_body, up.stream));
            mg.ok = true;
        }
        BLK_CUDA(cudaStreamSynchronize(up.stream));
        if ((int)m->vocab.size() != m->n_vocab) m->vocab.clear();
    });
    if (st != BLK_OK) return nullptr;
    return m.release();
}

// Model::Params::vocabOnly (reference Model.hpp:30, test t-integration.cpp:25-43): metadata + vocabulary, no device, no weights.
extern "C" blk_model* blk_model_load_vocab(const char* path) {
    std::unique_ptr<blk_model> m(new blk_model());
    m->device = -1;
    blk_status st = guarded([&] {
        std::unique_ptr<GgufFile> fp;
        try { fp.reset(new GgufFile(path)); }
        catch (const std::exception& e) {
            const std::string w = e.what();
            throw BlkError(w.rfind("gguf:", 0) == 0 ? BLK_ERR_FORMAT : BLK_ERR_IO, w);
        }
        load_metadata(m.get(), *fp, true);
        m->n_vocab = (int)m->vocab.size();
    });
    if (st != BLK_OK) return nullptr;
    return m.release();
}

extern "C" void blk_model_free(blk_model* m) { delete m; }
extern "C" int32_t blk_model_n_vocab(const blk_model* m) { return m->n_vocab; }
extern "C" int32_t blk_model_n_ctx_train(const blk_model* m) { return m->n_ctx_train; }
extern "C" int32_t blk_model_n_embd(const blk_model* m) { return m->n_embd; }
extern "C" int32_t blk_model_n_layer(const blk_model* m) { return m->n_layer; }
extern "C" int32_t blk_model_token_bos(const blk_model* m) { return m->tok_bos; }
extern "C" int32_t blk_model_token_eos(const blk_model* m) { return m->tok_eos; }
extern "C" int32_t blk_model_is_eog(const blk_model* m, int32_t t) {
    if (t < 0) return 0;
    if ((size_t)t < m->eog.size()) return m->eog[(size_t)t];
    return t == m->tok_eos || t == m->tok_eot || t == m->tok_eom;
}
extern "C" int32_t blk_model_add_eos(const blk_model* m) { return m->add_eos ? 1 : 0; }
extern "C" int32_t blk_model_token_type(const blk_model* m, int32_t t) { return (t >= 0 && (size_t)t < m->token_type.size()) ? m->token_type[(size_t)t] : 0; }
extern "C" int32_t blk_model_n_merges(const blk_model* m) { return (int32_t)m->merges.size(); }
extern "C" int32_t blk_model_merge_text(const blk_model* m, int32_t i, char* buf, int32_t cap) {
    if (i < 0 || (size_t)i >= m->merges.size()) return 0;
    const std::string& s = m->merges[(size_t)i];
    const int n = (int)s.size();
    if (buf && cap > 0) memcpy(buf, s.data(), (size_t)std::min(n, cap));
    return n;
}
extern "C" int32_t blk_model_vocab_only(const blk_model* m) { return m->vocab_only ? 1 : 0; }
extern "C" int32_t blk_model_add_bos(const blk_model* m) { return m->add_bos ? 1 : 0; }
extern "C" int32_t blk_model_device(const blk_model* m) { return m->device; }
extern "C" int64_t blk_model_weight_bytes_per_token(const blk_model* m) { return m->weight_bytes_per_token; }
extern "C" int64_t blk_model_kv_bytes_per_token(const blk_model* m) { return (int64_t)m->n_layer * m->n_head_kv * m->d_head * 2 * 2; }
extern "C" int32_t blk_model_token_text(const blk_model* m, int32_t tok, char* buf, int32_t cap) {
    if (tok < 0 || tok >= (int)m->vocab.size()) return 0;
    const std::string& s = m->vocab[tok];
    const int n = (int)s.size();
    if (buf && cap > 0) memcpy(buf, s.data(), (size_t)std::min(n, cap));
    return n;
}
extern "C" int32_t blk_model_meta_str(const blk_model* m, const char* key, char* buf, int32_t cap) {
    auto it = m->meta.find(key);
    if (it == m->meta.end()) return -1;
    const int n = (int)it->second.size();
    if (buf && cap > 0) memcpy(buf, it->second.data(), (size_t)std::min(n, cap));
    return n;
}

// ------------------------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------------------------
blk_ctx::~blk_ctx() {
    if (m) cudaSetDevice(m->device);
    if (g_full) cudaGraphExecDestroy(g_full);
    if (g_body) cudaGraphExecDestroy(g_body);
    if (g_loop) cudaGraphExecDestroy(g_loop);
    for (void* p : allocs) cudaFree(p);
    for (void* p : host_allocs) cudaFreeHost(p);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    for (int i = 0; i < 4; i++) { if (pn_filled[i]) cudaEventDestroy(pn_filled[i]); if (pn_start[i]) cudaEventDestroy(pn_start[i]); }
    if (pf_stream) cudaStreamDestroy(pf_stream);
    if (stream) cudaStreamDestroy(stream);
}

namespace {

template <class T> T* dalloc(blk_ctx* c, size_t n) {
    void* p = nullptr;
    BLK_CUDA(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
    c->allocs.push_back(p);
    return reinterpret_cast<T*>(p);
}
template <class T> T* halloc(blk_ctx* c, size_t n) {
    void* p = nullptr;
    BLK_CUDA(cudaMallocHost(&p, std::max<size_t>(n, 1) * sizeof(T)));
    c->host_allocs.push_back(p);
    return reinterpret_cast<T*>(p);
}
ActBuf make_act(blk_ctx* c, int K) {
    ActBuf a;
    a.f32 = dalloc<float>(c, K); a.q = dalloc<int8_t>(c, K); a.d = dalloc<float>(c, K / 32 + 8); a.bs = dalloc<int16_t>(c, K / 16 + 8);
    return a;
}

void ensure_kernel_attrs(int device) {
    static std::mutex mu; static bool done[64] = {false};
    std::lock_guard<std::mutex> lk(mu);
    if (device < 0 || device >= 64 || done[device]) return;
    BLK_CUDA(cudaFuncSetAttribute(act_prepare_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    BLK_CUDA(cudaFuncSetAttribute(act_prepare_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    done[device] = true;
}

template <int EPI>
void launch_gemv(blk_ctx* c, GemvArgs& a) {
    cudaError_t e;
    if (EPI == EPI_STORE) e = launch_gemv_store(a, c->stream);
    else if (EPI == EPI_RESID) e = launch_gemv_resid(a, c->stream);
    else if (EPI == EPI_QKV) e = launch_gemv_qkv(a, c->stream);
    else e = launch_gemv_swiglu(a, c->stream);
    if (e == cudaErrorInvalidValue) throw BlkError(BLK_ERR_FORMAT, "no mat-vec kernel for this weight type / row length");
    BLK_CUDA(e);
    c->launches++;
}

void launch_act_prepare(blk_ctx* c, const float* x, const float* w, int K, int fmt, const ActBuf& out, bool norm) {
    const size_t smem = (size_t)K * 4;
    if (smem > 160 * 1024) throw BlkError(BLK_ERR_ARG, "row too long for act_prepare");
    if (norm) BLK_CUDA(launch_pdl(act_prepare_kernel<true>, dim3(1), dim3(512), smem, c->stream, x, w, K, c->m->rms_eps, fmt, out, 0, 0, 0));
    else BLK_CUDA(launch_pdl(act_prepare_kernel<false>, dim3(1), dim3(512), smem, c->stream, x, w, K, c->m->rms_eps, fmt, out, 0, 0, 0));
    BLK_CUDA(cudaGetLastError());
    c->launches++;
}

void prof_mark(blk_ctx* c, const char* name) {
    if (!c->profiling) return;
    cudaEvent_t e; BLK_CUDA(cudaEventCreate(&e));
    BLK_CUDA(cudaEventRecord(e, c->stream));
    c->prof_marks.emplace_back(name, e);
}

// A mat-vec of the decode step: y = epilogue(W . act(in)) where act = (optional RMSNorm * norm_w) then the quantisation the
// weight type needs: a separate act_prepare / act_quant kernel followed by the register-staged kernel of gemv_kernels.cuh.
// (This per-op path serves F32 / F16 weights, shapes the persistent decode kernel does not take, and BLK_MEGA=0.)
template <int EPI>
void matvec(blk_ctx* c, GemvArgs& a, const float* in, const float* norm_w, const ActBuf& scratch, const char* name) {
    const int K = a.seg[0].W.K;
    const int ta = a.seg[0].W.type, tb = (a.nseg > 2) ? a.seg[2].W.type : ta;
    const int fmt = act_format_for(ta);
    a.act_fmt = fmt;
    if (!norm_w && fmt != ACT_F32) {
        // quantise only: every 256-element block is independent -> one warp per block across several CTAs
        BLK_CUDA(launch_pdl(act_quant_kernel, dim3((K / 256 + 7) / 8), dim3(256), 0, c->stream, in, K, fmt, scratch));
        c->launches++;
    } else {
        launch_act_prepare(c, in, norm_w, K, fmt, scratch, norm_w != nullptr);
    }
    prof_mark(c, "act_prepare");
    a.act = scratch;
    if (fmt == ACT_F32 && !norm_w) a.act.f32 = const_cast<float*>(in);
    launch_gemv<EPI>(c, a);
    prof_mark(c, name);
}

// the threshold top-k of the context's own logits row (c->logits -> c->top_ids / c->top_logits)
TopkArgs own_topk_args(const blk_ctx* c) {
    TopkArgs tk{};
    tk.logits = c->logits; tk.n = c->m->n_vocab; tk.chunk_max = c->chunk_max; tk.n_chunks = c->n_chunks;
    tk.cand_l = c->cand_l; tk.cand_i = c->cand_i; tk.cap = c->cand_cap; tk.count = c->counters + 1; tk.done = c->counters + 2;
    tk.out_ids = c->top_ids; tk.out_logits = c->top_logits;
    return tk;
}

// The per-op decode attention form of a context of c->n_pages KV pages (decode_kernels.cuh): the single-kernel cluster form when
// one CTA's share of the scores fits in shared memory and its token slice spans at most ATTN_CLUSTER_PAGES pages, else the
// three-kernel split form.  A slice of cap tokens starting anywhere inside a page spans at most (cap + KV_PAGE - 2) / KV_PAGE + 1
// pages, hence the bound on cap.  form: -1 = that rule, 0 = the split form, 1 = the cluster form (BLK_ERR_ARG when the rule does
// not allow it).  Sets attn_cluster, attn_cap, n_split and the cluster kernels' shared-memory attribute.
void plan_decode_attn(blk_ctx* c, int form = -1) {
    const blk_model* m = c->m;
    const int gq = m->n_head / m->n_head_kv;
    const int cs = 8;
    c->attn_cap = (c->n_pages * KV_PAGE + cs - 1) / cs;
    const size_t smem = (size_t)gq * (c->attn_cap + (ATTN_THREADS / 32) * m->d_head) * sizeof(float);
    const bool fits = smem <= 160 * 1024 && c->attn_cap <= (ATTN_CLUSTER_PAGES - 1) * KV_PAGE + 1;
    if (form == 1 && !fits) throw BlkError(BLK_ERR_ARG, "the cluster attention form does not cover this context");
    c->attn_cluster = (form == -1 ? fits : form == 1) ? cs : 0;
    if (c->attn_cluster) {
        BLK_CUDA(cudaFuncSetAttribute(attn_cluster_kernel<128, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 164 * 1024));
        BLK_CUDA(cudaFuncSetAttribute(attn_cluster_kernel<128, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 164 * 1024));
        BLK_CUDA(cudaFuncSetAttribute(attn_cluster_kernel<64, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 164 * 1024));
        BLK_CUDA(cudaFuncSetAttribute(attn_cluster_kernel<64, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 164 * 1024));
    }
    c->n_split = std::max(1, std::min(32, (2 * 148) / m->n_head_kv));
}

// decode attention of layer l (c->qbuf over the cache at c->d_pos -> c->act_q.f32) in the form plan_decode_attn chose
void launch_decode_attn(blk_ctx* c, int l) {
    const blk_model* m = c->m;
    const int dh = m->d_head, dq = m->n_head * dh, dkv = m->n_head_kv * dh;
    if (c->attn_cluster > 0) {
        AttnClusterArgs ac{};
        ac.q = c->qbuf; ac.k_pool = c->k_pool[l]; ac.v_pool = c->v_pool[l]; ac.page_table = c->page_table; ac.pos = c->d_pos;
        ac.n_head = m->n_head; ac.n_head_kv = m->n_head_kv; ac.kv_dim = dkv; ac.cap = c->attn_cap;
        ac.scale = 1.0f / sqrtf((float)dh); ac.out = c->act_q.f32;
        const size_t smem = (size_t)(m->n_head / m->n_head_kv) * (c->attn_cap + (ATTN_THREADS / 32) * dh) * sizeof(float);
        const dim3 grid(m->n_head_kv * c->attn_cluster), block(ATTN_THREADS);
        const bool g4 = (m->n_head / m->n_head_kv) <= 4;
        if (dh == 128 && g4) BLK_CUDA(launch_pdl_cluster(attn_cluster_kernel<128, 4>, grid, block, smem, c->attn_cluster, c->stream, ac));
        else if (dh == 128) BLK_CUDA(launch_pdl_cluster(attn_cluster_kernel<128, 8>, grid, block, smem, c->attn_cluster, c->stream, ac));
        else if (g4) BLK_CUDA(launch_pdl_cluster(attn_cluster_kernel<64, 4>, grid, block, smem, c->attn_cluster, c->stream, ac));
        else BLK_CUDA(launch_pdl_cluster(attn_cluster_kernel<64, 8>, grid, block, smem, c->attn_cluster, c->stream, ac));
        c->launches++;
        prof_mark(c, "attn_cluster");
        return;
    }
    AttnArgs at{};
    at.q = c->qbuf; at.k_pool = c->k_pool[l]; at.v_pool = c->v_pool[l]; at.page_table = c->page_table; at.pos = c->d_pos;
    at.n_head = m->n_head; at.n_head_kv = m->n_head_kv; at.d_head = dh; at.kv_dim = dkv; at.n_split = c->n_split;
    at.scale = 1.0f / sqrtf((float)dh); at.scores = c->scores; at.score_stride = c->n_pages * KV_PAGE; at.part_o = c->part_o;
    dim3 grid(m->n_head_kv, c->n_split);
    if (dh == 128) {
        BLK_CUDA(launch_pdl(attn_scores_kernel<128>, grid, dim3(128), 0, c->stream, at));
        prof_mark(c, "attn_scores");
        BLK_CUDA(launch_pdl(attn_pv_kernel<128>, grid, dim3(128), 0, c->stream, at));
        prof_mark(c, "attn_pv");
    } else {
        BLK_CUDA(launch_pdl(attn_scores_kernel<64>, grid, dim3(64), 0, c->stream, at));
        prof_mark(c, "attn_scores");
        BLK_CUDA(launch_pdl(attn_pv_kernel<64>, grid, dim3(64), 0, c->stream, at));
        prof_mark(c, "attn_pv");
    }
    c->launches += 2;
    // one CTA per 256 outputs: model widths are multiples of 256; blk_test_decode_attn pads part_o / act_q for narrower shapes
    BLK_CUDA(launch_pdl(attn_combine_kernel, dim3((dq + 255) / 256), dim3(256), 0, c->stream, c->part_o, dh, c->n_split, (int)ACT_F32, c->act_q));
    c->launches++;
    prof_mark(c, "attn_combine");
}

// one decode step on c->stream: token id in c->d_tok, position in c->d_pos.
// Per layer: QKV mat-vec (RMSNorm prologue; +bias, RoPE, KV-page write) | attention | Wo mat-vec (+residual) |
// gate/up mat-vec (RMSNorm prologue; SwiGLU) | down mat-vec (+residual); then final norm + lm_head mat-vec + top-k.
void enqueue_step(blk_ctx* c, bool with_head, bool feedback = false) {
    blk_model* m = c->m;
    const int d = m->n_embd, dh = m->d_head, dq = m->n_head * dh, dkv = m->n_head_kv * dh, ff = m->n_ff;
    if (c->mega_on) {
        // the whole step is one persistent cooperative kernel (mega_decode.cuh) + the top-k selection
        MegaParams P = c->mega_params;
        P.with_head = with_head ? 1 : 0; P.advance_pos = 1;
        P.seq = ++c->mega_seq;
        if (!with_head) P.chunk_counts = m->mega.d_counts_body;
        BLK_CUDA(mega_launch(P, c->mega_smem, c->stream));
        c->launches++;
        prof_mark(c, "mega_decode");
        if (with_head) {
            TopkArgs tk = own_topk_args(c);
            tk.feed_tok = feedback ? c->d_tok : nullptr;
            topk_select_kernel<<<16, 1024, 0, c->stream>>>(tk);
            BLK_CUDA(cudaGetLastError());
            c->launches++;
            prof_mark(c, "topk_select");
            if (!feedback) {
                BLK_CUDA(cudaMemcpyAsync(c->h_top_ids, c->top_ids, TOPK_MAX * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
                BLK_CUDA(cudaMemcpyAsync(c->h_top_logits, c->top_logits, TOPK_MAX * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
            }
        }
        return;
    }
    BLK_CUDA(launch_pdl(embed_kernel, dim3(1), dim3(256), 0, c->stream, m->tok_embd, c->d_tok, c->d_pos, c->x, c->rope_cs, dh / 2, m->theta_scale, m->rope_freqs));
    c->launches++;
    prof_mark(c, "embed");
    for (int l = 0; l < m->n_layer; l++) {
        const LayerWeights& L = m->layers[l];
        {
            GemvArgs a{};
            a.nseg = 3;
            a.seg[0] = {L.wq, L.bq, 0, 0};
            a.seg[1] = {L.wk, L.bk, dq / 2, 1};
            a.seg[2] = {L.wv, L.bv, dq / 2 + dkv / 2, 2};
            a.total_pairs = dq / 2 + dkv;
            a.out = c->qbuf;
            a.d_head = dh; a.neox = m->neox ? 1 : 0; a.rope_cs = c->rope_cs; a.pos = c->d_pos;
            a.k_pool = c->k_pool[l]; a.v_pool = c->v_pool[l]; a.page_table = c->page_table; a.kv_dim = dkv;
            matvec<EPI_QKV>(c, a, c->x, L.attn_norm, c->act_d, "gemv_qkv");
        }
        launch_decode_attn(c, l);
        {
            GemvArgs a{};
            a.nseg = 1; a.seg[0] = {L.wo, nullptr, 0, 0}; a.total_pairs = d / 2; a.out = c->x;
            matvec<EPI_RESID>(c, a, c->act_q.f32, nullptr, c->act_q2, "gemv_wo");
        }
        {
            GemvArgs a{};
            a.nseg = 2; a.seg[0] = {L.gate, nullptr, 0, 0}; a.seg[1] = {L.up, nullptr, 0, 0}; a.total_pairs = ff; a.out = c->hbuf;
            matvec<EPI_SWIGLU>(c, a, c->x, L.ffn_norm, c->act_d, "gemv_gate_up");
        }
        {
            GemvArgs a{};
            a.nseg = 1; a.seg[0] = {L.down, nullptr, 0, 0}; a.total_pairs = d / 2; a.out = c->x;
            matvec<EPI_RESID>(c, a, c->hbuf, nullptr, c->act_ff, "gemv_down");
        }
    }
    if (with_head) {
        GemvArgs a{};
        a.nseg = 1; a.seg[0] = {m->output, nullptr, 0, 0}; a.total_pairs = m->n_vocab / 2; a.out = c->logits;
        a.tail.kind = TAIL_CHUNKMAX; a.tail.chunk_max = c->chunk_max; a.tail.chunk_shift = c->chunk_shift;
        matvec<EPI_STORE>(c, a, c->x, m->out_norm, c->act_d, "gemv_lm_head");
        BLK_CUDA(launch_pdl(topk_select_kernel, dim3(16), dim3(1024), 0, c->stream, own_topk_args(c)));
        c->launches++;
        prof_mark(c, "topk_select");
    }
    BLK_CUDA(launch_pdl(advance_pos_kernel, dim3(1), dim3(32), 0, c->stream, c->d_pos, 1));
    c->launches++;
    if (feedback) {
        BLK_CUDA(launch_pdl(feed_top1_kernel, dim3(1), dim3(32), 0, c->stream, (const int32_t*)c->top_ids, c->d_tok));
        c->launches++;
    } else if (with_head) {
        BLK_CUDA(cudaMemcpyAsync(c->h_top_ids, c->top_ids, TOPK_MAX * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        BLK_CUDA(cudaMemcpyAsync(c->h_top_logits, c->top_logits, TOPK_MAX * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    }
}

} // namespace

// ------------------------------------------------------------------------------------------------------------------
// cell positions other than the cell index (Self-Extend: llama_kv_self_seq_add / seq_div, reference Session.cpp:348-368)
// ------------------------------------------------------------------------------------------------------------------
namespace {
// K rows of cells [cell0, cell0 + n) of every layer rotated IN PLACE by each cell's own position delta (llama.cpp's K-shift after
// llama_kv_self_seq_add / seq_div: ggml rope on the F16 cache).  grid = (n, n_layer), block = 128.
__global__ void __launch_bounds__(128) kv_rerope_kernel(__half* const* __restrict__ k_pools, const int32_t* __restrict__ page_table, int kv_dim, int d_head,
                                                        int neox, int cell0, const int32_t* __restrict__ delta, float theta_scale,
                                                        const float* __restrict__ freq_factors) {
    __shared__ float2 cs[64];
    const int cell = cell0 + (int)blockIdx.x;
    const int dl = delta[cell];
    if (dl == 0) return;
    const int half_rot = d_head / 2;
    rope_table_fill(cs, half_rot, dl, theta_scale, freq_factors);
    __syncthreads();
    __half* k = k_pools[blockIdx.y] + ((size_t)page_table[cell / KV_PAGE] * KV_PAGE + (cell % KV_PAGE)) * kv_dim;
    for (int p = threadIdx.x; p < kv_dim / 2; p += blockDim.x) {
        const int h = p / half_rot, i = p - h * half_rot;
        const int e0 = neox ? h * d_head + i : h * d_head + 2 * i;
        const int e1 = neox ? e0 + half_rot : e0 + 1;
        const float x0 = __half2float(k[e0]), x1 = __half2float(k[e1]);
        const float2 c = cs[i];
        k[e0] = __float2half_rn(__fsub_rn(__fmul_rn(x0, c.x), __fmul_rn(x1, c.y)));
        k[e1] = __float2half_rn(__fadd_rn(__fmul_rn(x0, c.y), __fmul_rn(x1, c.x)));
    }
}

// positions of the cells as a host vector (created on the first Self-Extend call)
void materialise_positions(blk_ctx* c) {
    if (!c->cell_pos.empty() || c->n_past == 0) { if (c->cell_pos.empty()) { c->cell_pos.assign((size_t)c->n_ctx, 0); c->cell_shift.assign((size_t)c->n_ctx, 0); } return; }
    c->cell_pos.resize((size_t)c->n_ctx); c->cell_shift.assign((size_t)c->n_ctx, 0);
    for (int i = 0; i < c->n_ctx; i++) c->cell_pos[(size_t)i] = i;
}
// after a position change: the next token's rotary position is one past the largest cell position (llama_batch_allocr, pos == nullptr)
void refresh_rope_offset(blk_ctx* c) {
    int mx = -1;
    for (int i = 0; i < c->n_past; i++) mx = std::max(mx, c->cell_pos[(size_t)i]);
    c->rope_off = (mx + 1) - c->n_past;
    const int32_t both[2] = {c->n_past, c->rope_off};
    BLK_CUDA(cudaMemcpyAsync(c->d_pos, both, sizeof(both), cudaMemcpyHostToDevice, c->stream));
    BLK_CUDA(cudaStreamSynchronize(c->stream));
}
// new cells [n_past, n_past + n) take the positions the kernels used for them
void note_new_cells(blk_ctx* c, int n) {
    if (c->cell_pos.empty()) return;
    for (int i = 0; i < n; i++) { c->cell_pos[(size_t)(c->n_past + i)] = c->n_past + c->rope_off + i; c->cell_shift[(size_t)(c->n_past + i)] = 0; }
}
// the accumulated position changes reach the K rows before anything reads them (llama.cpp applies its K-shift at the next decode)
void flush_pos_shift(blk_ctx* c) {
    if (!c->shift_pending) return;
    blk_model* m = c->m;
    int32_t* d_delta = nullptr;
    BLK_CUDA(cudaMalloc(&d_delta, (size_t)c->n_past * sizeof(int32_t)));
    cudaError_t e = cudaMemcpyAsync(d_delta, c->cell_shift.data(), (size_t)c->n_past * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        kv_rerope_kernel<<<dim3((unsigned)c->n_past, (unsigned)m->n_layer), 128, 0, c->stream>>>(c->d_kpools, c->page_table, m->n_head_kv * m->d_head, m->d_head,
                                                                                                   m->neox ? 1 : 0, 0, d_delta, m->theta_scale, m->rope_freqs);
        e = cudaGetLastError();
        c->launches++;
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_delta);
    BLK_CUDA(e);
    std::fill(c->cell_shift.begin(), c->cell_shift.begin() + c->n_past, 0);
    c->shift_pending = false;
}
} // namespace

// llama_kv_self_seq_add(ctx, 0, p0, p1, delta) (reference Session.cpp:359, 361): cells whose POSITION lies in [p0, p1) move by delta
extern "C" blk_status blk_kv_seq_add(blk_ctx* c, int32_t p0, int32_t p1, int32_t delta) {
    if (!c || p0 < 0 || p1 < p0) return fail(BLK_ERR_ARG, "blk_kv_seq_add: bad range");
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        if (delta == 0 || p0 == p1) return;
        materialise_positions(c);
        for (int i = 0; i < c->n_past; i++) {
            int32_t& p = c->cell_pos[(size_t)i];
            if (p >= p0 && p < p1) { p += delta; c->cell_shift[(size_t)i] += delta; c->shift_pending = true; if (p < 0) throw BlkError(BLK_ERR_ARG, "blk_kv_seq_add: negative position"); }
        }
        refresh_rope_offset(c);
    });
}
// llama_kv_self_seq_div(ctx, 0, p0, p1, d) (reference Session.cpp:360): positions in [p0, p1) are divided by d
extern "C" blk_status blk_kv_seq_div(blk_ctx* c, int32_t p0, int32_t p1, int32_t d) {
    if (!c || p0 < 0 || p1 < p0 || d <= 0) return fail(BLK_ERR_ARG, "blk_kv_seq_div: bad arguments");
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        if (d == 1 || p0 == p1) return;
        materialise_positions(c);
        for (int i = 0; i < c->n_past; i++) {
            int32_t& p = c->cell_pos[(size_t)i];
            if (p >= p0 && p < p1) { const int32_t old = p; p /= d; c->cell_shift[(size_t)i] += p - old; c->shift_pending = true; }
        }
        refresh_rope_offset(c);
    });
}
// rotary position the next token will get (one past the largest cell position; = n_past unless Self-Extend moved positions)
extern "C" int32_t blk_ctx_next_pos(const blk_ctx* c) { return c->n_past + c->rope_off; }


namespace {

// ------------------------------------------------------------------------------------------------------------------
// multi-token prefill (tcgen05 GEMM path)
// ------------------------------------------------------------------------------------------------------------------
// The GEMMs of a multi-token pass, in pass order: op 4 l + {OP_QKV, OP_WO, OP_GATE_UP, OP_DOWN} of layer l, then the lm_head.
// This index is shared by the model's resident panel cache, the per-context streaming panels and the pass itself.
enum GemmKind { OP_QKV, OP_WO, OP_GATE_UP, OP_DOWN, OP_HEAD };
struct GemmOp {
    GemmKind kind;
    int n_parts;
    GemmPart part[3];                   // OP_GATE_UP: {gate, up}
    const __nv_bfloat16* panel;         // set by GemmSchedule::next: the bf16 panel the GEMM reads (nullptr: fused form)
    size_t panel_elems() const { return prefill_panel_elems(part, n_parts, kind == OP_GATE_UP); }
    // false: the combination takes the fused GEMM form
    bool fill_panel(__nv_bfloat16* p, cudaStream_t st, cudaError_t* err) const { return prefill_panel_fill(part, n_parts, kind == OP_GATE_UP, p, st, err); }
};
int n_gemm_ops(const blk_model* m) { return 4 * m->n_layer + 1; }
GemmOp gemm_op(const blk_model* m, int i) {
    const int l = i / 4;
    if (l == m->n_layer) return {OP_HEAD, 1, {{&m->output, nullptr, 0}}, nullptr};
    const LayerWeights& L = m->layers[l];
    const int dq = m->n_head * m->d_head, dkv = m->n_head_kv * m->d_head;
    switch (i % 4) {
        case OP_QKV: return {OP_QKV, 3, {{&L.wq, L.bq, 0}, {&L.wk, L.bk, dq}, {&L.wv, L.bv, dq + dkv}}, nullptr};
        case OP_WO: return {OP_WO, 1, {{&L.wo, nullptr, 0}}, nullptr};
        case OP_GATE_UP: return {OP_GATE_UP, 2, {{&L.gate, nullptr, 0}, {&L.up, nullptr, 0}}, nullptr};
        default: return {OP_DOWN, 1, {{&L.down, nullptr, 0}}, nullptr};
    }
}
// Per-context streaming panels of the two-pass GEMM form (matrices that are not resident in the model's panel cache): one bf16
// panel per GEMM kind, so the de-quantisation of the NEXT matrix (second stream) runs while the current GEMM does.  The lm_head
// shares the gate+up panel.
int stream_panel(GemmKind k) { return k == OP_HEAD ? OP_GATE_UP : k; }
void ensure_stream_panels(blk_ctx* c) {
    if (c->panel_tried) return;
    c->panel_tried = true;
    blk_model* m = c->m;
    size_t elems[4] = {0, 0, 0, 0};      // each panel holds the largest op of its kind
    for (int i = 0; i < n_gemm_ops(m); i++) {
        const GemmOp g = gemm_op(m, i);
        elems[stream_panel(g.kind)] = std::max(elems[stream_panel(g.kind)], g.panel_elems());
    }
    bool ok = true;
    for (int i = 0; i < 4 && ok; i++) {
        void* p = nullptr;
        ok = cudaMalloc(&p, elems[i] * sizeof(__nv_bfloat16)) == cudaSuccess;
        if (ok) { c->allocs.push_back(p); c->pf_panel[i] = reinterpret_cast<__nv_bfloat16*>(p); }
    }
    if (!ok) { (void)cudaGetLastError(); for (int i = 0; i < 4; i++) c->pf_panel[i] = nullptr; }
    else for (int i = 0; i < 4; i++) {
        BLK_CUDA(cudaEventCreateWithFlags(&c->pn_filled[i], cudaEventDisableTiming));
        BLK_CUDA(cudaEventCreateWithFlags(&c->pn_start[i], cudaEventDisableTiming));
    }
}

// The model's resident panel cache (engine.hpp), built by the first multi-token pass: layer by layer while device memory beyond
// the reserve lasts.  Every later pass only reads it, so nothing but this build needs the lock.
const std::vector<__nv_bfloat16*>& model_panels(blk_ctx* c) {
    blk_model* m = c->m;
    blk_model::PanelCache& pc = m->panels;
    std::lock_guard<std::mutex> lk(pc.mu);
    if (pc.built) return pc.op;
    pc.built = true;
    const int n_ops = n_gemm_ops(m);
    pc.op.assign(n_ops, nullptr);
    double cap_gb = 1e9;
    { const char* e = getenv("BLK_PANEL_CACHE_GB"); if (e) cap_gb = atof(e); }
    if (cap_gb <= 0.0) return pc.op;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { (void)cudaGetLastError(); return pc.op; }
    // reserve: later contexts (KV pages, prefill workspaces) and other users of the device must still find room
    const size_t reserve = std::max((size_t)16 << 30, total_b / 6);
    size_t budget = free_b > reserve ? free_b - reserve : 0;
    budget = (size_t)std::min((double)budget, cap_gb * 1e9);
    cudaStream_t ss = c->pf_stream;
    for (int i = 0; i < n_ops; i++) {
        const GemmOp g = gemm_op(m, i);
        const size_t bytes = g.panel_elems() * sizeof(__nv_bfloat16);
        if (pc.bytes + bytes > budget) break;
        void* p = nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess) { (void)cudaGetLastError(); break; }
        cudaError_t err = cudaSuccess;
        const bool ok = g.fill_panel(reinterpret_cast<__nv_bfloat16*>(p), ss, &err);
        if (!ok || err != cudaSuccess) { (void)cudaGetLastError(); cudaStreamSynchronize(ss); cudaFree(p); if (err != cudaSuccess) break; continue; }   // a type without a panel form: fused GEMM
        pc.allocs.push_back(p); pc.op[i] = reinterpret_cast<__nv_bfloat16*>(p); pc.bytes += bytes; pc.n_resident++;
    }
    BLK_CUDA(cudaStreamSynchronize(ss));
    log_msg(1, "resident bf16 panels: " + std::to_string(pc.n_resident) + " of " + std::to_string(n_ops) + " matrices, " + std::to_string(pc.bytes >> 20) + " MiB");
    return pc.op;
}

// Where each GEMM of a multi-token pass reads its weights from, in pass order (gemm_op):
//  - a resident bf16 panel of the model cache: the TMA-fed GEMM at every batch size;
//  - otherwise, from panel_min tokens on, a streaming panel: the matrix is de-quantised ONCE on pf_stream, one GEMM ahead of the
//    main stream.  The fill of op i+1 starts when GEMM i starts (its panel's previous user, GEMM i-3, is then done), so fills
//    overlap GEMMs, not the small bandwidth-bound kernels;
//  - otherwise the fused form (weights de-quantised inside the GEMM, once per 256 tokens), which moves fewer bytes for few tokens.
class GemmSchedule {
  public:
    // n_ops: the pass runs ops 0 .. n_ops - 1
    GemmSchedule(blk_ctx* c, int n, int n_ops) : c_(c), n_ops_(n_ops), res_(model_panels(c)), filled_(n_ops, 0) {
        bool all_res = true;
        for (int i = 0; i < n_ops; i++) all_res = all_res && resident(i);
        if (!all_res && c->panel_min > 0 && n >= c->panel_min) ensure_stream_panels(c);
        stream_ = !all_res && c->pf_panel[0] && c->panel_min > 0 && n >= c->panel_min;
        if (stream_ && !resident(0)) { BLK_CUDA(cudaEventRecord(c->pn_start[0], c->stream)); BLK_CUDA(cudaStreamWaitEvent(c->pf_stream, c->pn_start[0], 0)); }   // after whatever ran before
        fill(0);
    }
    // main stream, right before the next GEMM of the pass (which must be of this kind): that op, with its panel
    GemmOp next(GemmKind kind) {
        const int i = next_++;
        if (i >= n_ops_) throw BlkError(BLK_ERR_ARG, "multi-token pass: more GEMMs than scheduled");
        GemmOp g = gemm_op(c_->m, i);
        if (g.kind != kind) throw BlkError(BLK_ERR_ARG, "multi-token pass: GEMM op out of order");
        const int b = stream_panel(g.kind);
        const bool next_fill = stream_ && i + 1 < n_ops_ && !resident(i + 1);
        if (next_fill) {
            BLK_CUDA(cudaEventRecord(c_->pn_start[b], c_->stream));                 // GEMM i is about to start ...
            BLK_CUDA(cudaStreamWaitEvent(c_->pf_stream, c_->pn_start[b], 0));       // ... so is the fill of op i + 1 (other panel; its last reader, GEMM i - 3, is done)
        }
        g.panel = resident(i);
        if (!g.panel && stream_) {
            BLK_CUDA(cudaStreamWaitEvent(c_->stream, c_->pn_filled[b], 0));
            g.panel = filled_[i] ? c_->pf_panel[b] : nullptr;
        }
        if (next_fill) fill(i + 1);
        return g;
    }

  private:
    __nv_bfloat16* resident(int i) const { return i < (int)res_.size() ? res_[i] : nullptr; }
    void fill(int i) {      // enqueue the fill of op i on the side stream
        if (!stream_ || i >= n_ops_ || resident(i)) return;
        const GemmOp g = gemm_op(c_->m, i);
        const int b = stream_panel(g.kind);
        cudaError_t err = cudaSuccess;
        const bool ok = g.fill_panel(c_->pf_panel[b], c_->pf_stream, &err);
        BLK_CUDA(err);
        filled_[i] = ok ? 1 : 0;
        BLK_CUDA(cudaEventRecord(c_->pn_filled[b], c_->pf_stream));
        c_->launches += ok ? 2 : 0;
    }
    blk_ctx* c_;
    int n_ops_, next_ = 0;
    bool stream_ = false;
    const std::vector<__nv_bfloat16*>& res_;
    std::vector<char> filled_;
};

void ensure_prefill_bufs(blk_ctx* c, int T) {
    if (T <= c->pf_cap) return;
    blk_model* m = c->m;
    const int d = m->n_embd, dh = m->d_head, dq = m->n_head * dh, dkv = m->n_head_kv * dh, ff = m->n_ff;
    const int cap = std::max(T, std::min(c->n_batch, c->n_ctx));
    const size_t t = (size_t)cap;
    c->pf_tokens = dalloc<int32_t>(c, t); c->pf_rope = dalloc<float2>(c, t * (dh / 2));
    c->pf_x = dalloc<float>(c, t * d);
    c->pf_xn = dalloc<__nv_bfloat16>(c, t * std::max(d, dq));
    c->pf_qkv = dalloc<float>(c, t * (dq + 2 * dkv));
    c->pf_q = dalloc<__half>(c, t * dq);
    c->pf_ao = dalloc<__nv_bfloat16>(c, t * dq);
    c->pf_h = dalloc<__nv_bfloat16>(c, t * ff);
    {   // split-K workspace of the prefill GEMMs (few-token batches): splits * tiles <= SMs, a tile is 256 x 256 f32
        int sms = 0; BLK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device));
        c->pf_splitk_elems = (size_t)sms * 65536;
        c->pf_splitk = dalloc<float>(c, c->pf_splitk_elems);
    }
    c->pf_logit_rows = 512;     // rows of one lm_head chunk: two M tiles share every weight tile through L2
    c->pf_logits = dalloc<float>(c, (size_t)c->pf_logit_rows * m->n_vocab);
    if (prefill_attn_tc_supported(dh, m->n_head, m->n_head_kv)) {      // transposed-V scratch of the tcgen05 attention (one layer at a time)
        c->pf_vt_pad = (c->n_pages * KV_PAGE + 127) / 128 * 128;
        c->pf_vt = dalloc<__half>(c, (size_t)m->n_head_kv * 128 * c->pf_vt_pad);
    }
    c->pf_claimed = dalloc<int32_t>(c, t * 10); c->pf_nclaimed = dalloc<int32_t>(c, t);
    c->pf_gath = dalloc<float>(c, t * 10); c->pf_topi = dalloc<int32_t>(c, t * 10); c->pf_topl = dalloc<float>(c, t * 10);
    c->pf_cap = cap;
    BLK_CUDA(cudaFuncSetAttribute(prefill_attn_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * 64 * (64 + 8) * 2));
}

// top-64 of c->logits through the threshold selector (the row did not come from the decode lm_head mat-vec)
void topk_of_logits(blk_ctx* c) {
    blk_model* m = c->m;
    chunk_max_kernel<<<c->n_chunks, 256, 0, c->stream>>>(c->logits, m->n_vocab, c->chunk_shift, c->chunk_max);
    BLK_CUDA(cudaGetLastError()); c->launches++;
    topk_select_kernel<<<16, 1024, 0, c->stream>>>(own_topk_args(c));
    BLK_CUDA(cudaGetLastError()); c->launches++;
    BLK_CUDA(cudaMemcpyAsync(c->h_top_ids, c->top_ids, TOPK_MAX * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    BLK_CUDA(cudaMemcpyAsync(c->h_top_logits, c->top_logits, TOPK_MAX * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
}

// causal flash attention of a prefill chunk: the query heads of a KV head share a CTA when the GQA ratio is a power of two
template <int DH, int GQ>
void launch_attn_gqa(const PrefillAttnArgs& pa, int n, int n_head_kv, cudaStream_t st) {
    constexpr int smem = prefill_attn_gqa_smem<DH, GQ>();
    // the opt-in is per (function, device) and several worker threads launch concurrently: set it on every launch (host-only, cheap)
    BLK_CUDA(cudaFuncSetAttribute(prefill_attn_gqa_kernel<DH, GQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    constexpr int BQ = 128 / GQ;
    prefill_attn_gqa_kernel<DH, GQ><<<dim3((n + BQ - 1) / BQ, n_head_kv), 256, smem, st>>>(pa);
}
// d_head 128: the tcgen05 kernel (GQA ratio <= 8, pf_vt allocated by ensure_prefill_bufs); d_head 64: the mma.sync kernels
void launch_prefill_attn(blk_ctx* c, const PrefillAttnArgs& pa, int n, cudaStream_t st) {
    const blk_model* m = c->m;
    const int dh = m->d_head, gq = m->n_head / m->n_head_kv;
    if (dh == 128) {
        if (!c->pf_vt || !prefill_attn_tc_supported(dh, m->n_head, m->n_head_kv)) throw BlkError(BLK_ERR_ARG, "prefill attention: no kernel for this head shape");
        // the layer's pools are recovered from the arguments
        BLK_CUDA(prefill_attn_tc(pa.q, pa.k_pool, pa.v_pool, pa.page_table, c->n_pages, pa.pos0, c->n_past, pa.out, c->pf_vt, c->pf_vt_pad, n,
                                 m->n_head, m->n_head_kv, pa.kv_dim, pa.scale, st));
        return;
    }
    if (gq == 4) launch_attn_gqa<64, 4>(pa, n, m->n_head_kv, st);
    else if (gq == 8) launch_attn_gqa<64, 8>(pa, n, m->n_head_kv, st);
    else if (gq == 2) launch_attn_gqa<64, 2>(pa, n, m->n_head_kv, st);
    else prefill_attn_kernel<64><<<dim3((n + 63) / 64, m->n_head), 128, 3 * 64 * (64 + 8) * 2, st>>>(pa);
    BLK_CUDA(cudaGetLastError());
}

// The layers of a multi-token pass over the n rows of c->pf_x: RMSNorm, QKV GEMM, attend(l) (pf_qkv -> pf_ao: RoPE, the new KV
// cache rows and the attention of layer l), Wo GEMM (+residual), RMSNorm, gate+up GEMM (SwiGLU epilogue), down GEMM (+residual).
// Few-token passes fold the split-K reduce of Wo / down into the RMSNorm that follows (pend).  final_norm: the caller runs the
// final RMSNorm with pend after the last layer; otherwise the last down GEMM reduces its own partial sums.
template <class Attend>
void run_layers(blk_ctx* c, int n, GemmSchedule& sched, PendingReduce& pend, bool final_norm, Attend attend) {
    blk_model* m = c->m;
    const int d = m->n_embd, dq = m->n_head * m->d_head, dkv = m->n_head_kv * m->d_head, ff = m->n_ff;
    const long long ldq = dq + 2 * dkv;
    cudaStream_t st = c->stream;
    const SplitKWs sk{c->pf_splitk, c->pf_splitk_elems, &pend};
    SplitKWs sk_last = sk;
    if (!final_norm) sk_last.defer = nullptr;
    for (int l = 0; l < m->n_layer; l++) {
        const LayerWeights& L = m->layers[l];
        rmsnorm_bf16_launch(c->pf_x, L.attn_norm, d, m->rms_eps, c->pf_xn, n, st, &pend);
        BLK_CUDA(cudaGetLastError());
        prof_mark(c, "rmsnorm_bf16");
        GemmOp g = sched.next(OP_QKV);
        BLK_CUDA(prefill_gemm_multi(g.part, g.n_parts, c->pf_xn, n, c->pf_qkv, ldq, st, g.panel, &sk));
        prof_mark(c, "gemm_qkv");
        attend(l);
        g = sched.next(OP_WO);
        BLK_CUDA(prefill_gemm(*g.part[0].W, c->pf_ao, n, c->pf_x, d, nullptr, 1, st, g.panel, &sk));
        prof_mark(c, "gemm_wo");
        rmsnorm_bf16_launch(c->pf_x, L.ffn_norm, d, m->rms_eps, c->pf_xn, n, st, &pend);
        BLK_CUDA(cudaGetLastError());
        prof_mark(c, "rmsnorm_bf16");
        g = sched.next(OP_GATE_UP);
        BLK_CUDA(prefill_gemm_swiglu(*g.part[0].W, *g.part[1].W, c->pf_xn, n, c->pf_h, ff, st, g.panel, &sk));
        prof_mark(c, "gemm_gate_up_swiglu");
        g = sched.next(OP_DOWN);
        BLK_CUDA(prefill_gemm(*g.part[0].W, c->pf_h, n, c->pf_x, d, nullptr, 1, st, g.panel, l + 1 < m->n_layer ? &sk : &sk_last));
        prof_mark(c, "gemm_down");
        c->launches += 6;
    }
    if (pend.ws && !final_norm) throw BlkError(BLK_ERR_CUDA, "multi-token pass: a deferred split-K reduce was left unconsumed");
}

// One causal prefill of n tokens at positions n_past.. .  verify != nullptr: logits of EVERY position go through the
// per-row top-10 + claimed-id gather (never stored beyond a 256-row chunk); otherwise only the last position's logits are
// produced (decode mat-vec on the last row).
struct VerifyIo { const int32_t* claimed; const int32_t* n_claimed; float* gathered; blk_token_data* top; };

void prefill_chunk(blk_ctx* c, const int32_t* tokens, int n, const VerifyIo* verify, int verify_row0) {
    blk_model* m = c->m;
    const int d = m->n_embd, dh = m->d_head, dq = m->n_head * dh, dkv = m->n_head_kv * dh, V = m->n_vocab;
    ensure_prefill_bufs(c, n);
    flush_pos_shift(c);
    note_new_cells(c, n);
    cudaStream_t st = c->stream;
    const ChainPdl chain_scope(n);      // few-token passes: every kernel of the chain is a programmatic dependent of its predecessor
    BLK_CUDA(cudaMemcpyAsync(c->pf_tokens, tokens, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    embed_kernel<<<n, 256, 0, st>>>(m->tok_embd, c->pf_tokens, c->d_pos, c->pf_x, c->pf_rope, dh / 2, m->theta_scale, m->rope_freqs);
    BLK_CUDA(cudaGetLastError()); c->launches++;
    prof_mark(c, "embed");
    // verify without the verifier's own per-position top-10: only the logits at the claimed ids are needed (what the reference's
    // fillCtx reads, Session.cpp:263-282) -> sparse rows of the vocabulary projection instead of the T x V GEMM
    const bool sparse_head = verify && !verify->top && m->output.type != QT_F32 && m->output.type != QT_F16 && (d % 64) == 0;
    GemmSchedule sched(c, n, n_gemm_ops(m) - (verify && !sparse_head ? 0 : 1));
    PendingReduce pend;
    run_layers(c, n, sched, pend, verify != nullptr, [&](int l) {
        QkvPostArgs qa{};
        qa.qkv = c->pf_qkv; qa.ld = dq + 2 * dkv; qa.rope_cs = c->pf_rope; qa.pos0 = c->d_pos; qa.q_out = c->pf_q;
        qa.k_pool = c->k_pool[l]; qa.v_pool = c->v_pool[l]; qa.page_table = c->page_table;
        qa.dq = dq; qa.dkv = dkv; qa.d_head = dh; qa.neox = m->neox ? 1 : 0;
        BLK_CUDA(launch_chain(qkv_post_kernel, dim3(n), dim3(256), 0, st, qa));
        BLK_CUDA(cudaGetLastError());
        prof_mark(c, "qkv_post(rope+kv)");
        PrefillAttnArgs pa{};
        pa.q = c->pf_q; pa.k_pool = c->k_pool[l]; pa.v_pool = c->v_pool[l]; pa.page_table = c->page_table; pa.pos0 = c->d_pos;
        pa.out = c->pf_ao; pa.T = n; pa.n_head = m->n_head; pa.n_head_kv = m->n_head_kv; pa.kv_dim = dkv; pa.scale = 1.0f / sqrtf((float)dh);
        launch_prefill_attn(c, pa, n, st);
        prof_mark(c, "flash_attn");
        c->launches += 6;      // (with the 6 run_layers counts: 12 per layer)
    });
    BLK_CUDA(launch_pdl(advance_pos_kernel, dim3(1), dim3(32), 0, st, c->d_pos, n));
    c->launches++;
    if (verify) {
        BLK_CUDA(cudaMemcpyAsync(c->pf_claimed, verify->claimed + (size_t)verify_row0 * 10, (size_t)n * 10 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        BLK_CUDA(cudaMemcpyAsync(c->pf_nclaimed, verify->n_claimed + verify_row0, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        rmsnorm_bf16_launch(c->pf_x, m->out_norm, d, m->rms_eps, c->pf_xn, n, st, &pend);
        BLK_CUDA(cudaGetLastError()); c->launches++;
        if (sparse_head) {
            BLK_CUDA(prefill_claimed_logits(m->output, c->pf_xn, c->pf_claimed, c->pf_nclaimed, n, c->pf_gath, st));
            c->launches++;
            prof_mark(c, "claimed_logits");
            // the last position's full row (sampling may continue after the fill): decode mat-vec on the last row
            GemvArgs a{};
            a.nseg = 1; a.seg[0] = {m->output, nullptr, 0, 0}; a.total_pairs = V / 2; a.out = c->logits;
            matvec<EPI_STORE>(c, a, c->pf_x + (size_t)(n - 1) * d, m->out_norm, c->act_d, "gemv_lm_head");
        }
        GemmOp head{};
        for (int r0 = 0; r0 < n && !sparse_head; r0 += c->pf_logit_rows) {
            const int rows = std::min(c->pf_logit_rows, n - r0);
            if (r0 == 0) head = sched.next(OP_HEAD);
            BLK_CUDA(prefill_gemm(*head.part[0].W, c->pf_xn + (size_t)r0 * d, rows, c->pf_logits, V, nullptr, 0, st, head.panel));
            prof_mark(c, "gemm_lm_head");
            RowTopkArgs ta{};
            ta.logits = c->pf_logits; ta.ld = V; ta.n_vocab = V; ta.row0 = r0;
            ta.claimed = c->pf_claimed; ta.n_claimed = c->pf_nclaimed; ta.gathered = c->pf_gath;
            ta.top_ids = verify->top ? c->pf_topi : nullptr; ta.top_logits = c->pf_topl;
            row_topk_gather_kernel<<<rows, 256, 0, st>>>(ta);
            BLK_CUDA(cudaGetLastError()); c->launches += 2;
            prof_mark(c, "row_top10_gather");
            if (r0 + rows == n)     // keep the last position's full row for top-k / gather / sampling after the fill
                BLK_CUDA(cudaMemcpyAsync(c->logits, c->pf_logits + (size_t)(rows - 1) * V, (size_t)V * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
        BLK_CUDA(cudaMemcpyAsync(verify->gathered + (size_t)verify_row0 * 10, c->pf_gath, (size_t)n * 10 * sizeof(float), cudaMemcpyDeviceToHost, st));
        topk_of_logits(c);
        BLK_CUDA(cudaStreamSynchronize(st));
        if (verify->top) {
            std::vector<int32_t> ti((size_t)n * 10); std::vector<float> tl((size_t)n * 10);
            BLK_CUDA(cudaMemcpy(ti.data(), c->pf_topi, ti.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
            BLK_CUDA(cudaMemcpy(tl.data(), c->pf_topl, tl.size() * sizeof(float), cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < ti.size(); i++) { verify->top[(size_t)verify_row0 * 10 + i].token = ti[i]; verify->top[(size_t)verify_row0 * 10 + i].logit = tl[i]; }
        }
    } else {
        // only the last position's distribution is needed (llama_get_logits_ith(-1)): decode mat-vec on the last row
        GemvArgs a{};
        a.nseg = 1; a.seg[0] = {m->output, nullptr, 0, 0}; a.total_pairs = V / 2; a.out = c->logits;
        matvec<EPI_STORE>(c, a, c->pf_x + (size_t)(n - 1) * d, m->out_norm, c->act_d, "gemv_lm_head");
        topk_of_logits(c);
    }
    c->n_past += n;
    c->have_logits = true;
}

// tokens per chunk when n tokens do not fit one logical batch: equal chunks (rounded up to whole 64-token tiles) instead of full
// batches plus a small remainder -- a 32-token tail would run the few-token GEMM form and cost as much as a quarter of a full chunk
int balanced_chunk(int n, int n_batch) {
    if (n <= n_batch) return n;
    const int chunks = (n + n_batch - 1) / n_batch;
    const int per = ((n + chunks - 1) / chunks + 63) / 64 * 64;
    return std::min(per, n_batch);
}

void build_graphs(blk_ctx* c) {
    for (int which = 0; which < 3; which++) {
        const bool head = (which != 1);
        cudaGraph_t g = nullptr;
        const int64_t before = c->launches;
        BLK_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        try { enqueue_step(c, head, which == 2); }
        catch (...) { cudaGraph_t tmp = nullptr; cudaStreamEndCapture(c->stream, &tmp); if (tmp) cudaGraphDestroy(tmp); throw; }
        BLK_CUDA(cudaStreamEndCapture(c->stream, &g));
        cudaGraphExec_t ge = nullptr;
        cudaError_t e = cudaGraphInstantiate(&ge, g, 0);
        cudaGraphDestroy(g);
        BLK_CUDA(e);
        (which == 0 ? c->g_full : which == 1 ? c->g_body : c->g_loop) = ge;
        (which == 0 ? c->launches_full : which == 1 ? c->launches_body : c->launches_loop) = c->launches - before;
        c->launches = before;
    }
}

// after a stream synchronisation: did a poll of the persistent decode kernel give up?
void check_mega(blk_ctx* c) {
    if (c->mega_err && *c->mega_err) {
        const int w = *c->mega_err; *c->mega_err = 0;
        throw BlkError(BLK_ERR_CUDA, "persistent decode kernel: a phase never arrived (poll " + std::to_string(w) + " timed out)");
    }
}

void step(blk_ctx* c, int32_t tok, bool with_head) {
    blk_model* m = c->m;
    if (tok < 0 || tok >= m->n_vocab) throw BlkError(BLK_ERR_ARG, "token id out of range");
    if (c->n_past + 1 > c->n_ctx) throw BlkError(BLK_ERR_CTX_FULL, "context is full");
    flush_pos_shift(c);
    note_new_cells(c, 1);
    // pinned ring of token slots: a slot is only rewritten after the stream has drained once per lap
    if (c->tok_slot == 0) BLK_CUDA(cudaStreamSynchronize(c->stream));
    int32_t* slot = c->h_tok + c->tok_slot;
    c->tok_slot = (c->tok_slot + 1) % blk_ctx::TOK_RING;
    *slot = tok;
    BLK_CUDA(cudaMemcpyAsync(c->d_tok, slot, sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    if (c->mega_on) enqueue_step(c, with_head, false);
    else {
        BLK_CUDA(cudaGraphLaunch(with_head ? c->g_full : c->g_body, c->stream));
        c->launches += with_head ? c->launches_full : c->launches_body;
    }
    c->n_past++;
    c->have_logits = with_head;
}

} // namespace

extern "C" int64_t blk_model_panel_bytes(blk_model* m, int32_t* n_resident, int32_t* n_matrices) {
    if (!m) return 0;
    std::lock_guard<std::mutex> lk(m->panels.mu);
    if (n_resident) *n_resident = m->panels.n_resident;
    if (n_matrices) *n_matrices = n_gemm_ops(m);
    return (int64_t)m->panels.bytes;
}

extern "C" blk_ctx* blk_ctx_create(blk_model* m, int32_t n_ctx, int32_t n_batch) {
    if (!m) { fail(BLK_ERR_ARG, "null model"); return nullptr; }
    if (m->vocab_only) { fail(BLK_ERR_ARG, "Failed to create context: the model was loaded vocabulary-only"); return nullptr; }
    std::unique_ptr<blk_ctx> c(new blk_ctx());
    c->m = m;
    blk_status st = guarded([&] {
        BLK_CUDA(cudaSetDevice(m->device));
        ensure_kernel_attrs(m->device);
        c->n_ctx = n_ctx > 0 ? n_ctx : m->n_ctx_train;
        c->n_batch = n_batch > 0 ? n_batch : 2048;
        { const char* e = getenv("BLK_PREFILL_MIN"); if (e) c->prefill_min = std::max(2, atoi(e)); }
        { const char* e = getenv("BLK_PANEL_MIN"); if (e) c->panel_min = atoi(e); }
        BLK_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        BLK_CUDA(cudaEventCreate(&c->ev0)); BLK_CUDA(cudaEventCreate(&c->ev1));
        BLK_CUDA(cudaStreamCreateWithFlags(&c->pf_stream, cudaStreamNonBlocking));
        const int d = m->n_embd, dh = m->d_head, dq = m->n_head * dh, dkv = m->n_head_kv * dh, ff = m->n_ff;
        c->n_pages = (c->n_ctx + KV_PAGE - 1) / KV_PAGE;
        c->k_pool.resize(m->n_layer); c->v_pool.resize(m->n_layer);
        const size_t pool_elems = (size_t)c->n_pages * KV_PAGE * dkv;
        for (int l = 0; l < m->n_layer; l++) { c->k_pool[l] = dalloc<__half>(c.get(), pool_elems); c->v_pool[l] = dalloc<__half>(c.get(), pool_elems); }
        c->page_table = dalloc<int32_t>(c.get(), c->n_pages);
        {   // identity mapping today; every kernel goes through the table so pages can be shared / remapped later
            std::vector<int32_t> pt(c->n_pages);
            for (int i = 0; i < c->n_pages; i++) pt[i] = i;
            BLK_CUDA(cudaMemcpy(c->page_table, pt.data(), pt.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
            c->page_table_host = pt;
        }
        c->d_kpools = dalloc<__half*>(c.get(), m->n_layer); c->d_vpools = dalloc<__half*>(c.get(), m->n_layer);
        BLK_CUDA(cudaMemcpy(c->d_kpools, c->k_pool.data(), m->n_layer * sizeof(__half*), cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(c->d_vpools, c->v_pool.data(), m->n_layer * sizeof(__half*), cudaMemcpyHostToDevice));
        c->d_tok = dalloc<int32_t>(c.get(), 1); c->d_pos = dalloc<int32_t>(c.get(), 2);
        BLK_CUDA(cudaMemset(c->d_pos, 0, 2 * sizeof(int32_t)));
        c->h_tok = halloc<int32_t>(c.get(), blk_ctx::TOK_RING);
        c->x = dalloc<float>(c.get(), d); c->qbuf = dalloc<float>(c.get(), dq); c->hbuf = dalloc<float>(c.get(), ff);
        c->rope_cs = dalloc<float2>(c.get(), dh / 2);
        c->act_d = make_act(c.get(), d); c->act_q = make_act(c.get(), dq); c->act_q2 = make_act(c.get(), dq); c->act_ff = make_act(c.get(), ff);
        plan_decode_attn(c.get());
        c->part_o = dalloc<float>(c.get(), (size_t)m->n_head * c->n_split * dh);
        c->scores = dalloc<float>(c.get(), (size_t)m->n_head * c->n_pages * KV_PAGE);
        c->logits = dalloc<float>(c.get(), m->n_vocab);
        c->chunk_shift = 6;
        while (((m->n_vocab + (1 << c->chunk_shift) - 1) >> c->chunk_shift) > 256) c->chunk_shift++;
        c->n_chunks = (m->n_vocab + (1 << c->chunk_shift) - 1) >> c->chunk_shift;
        c->cand_l = dalloc<float>(c.get(), c->cand_cap); c->cand_i = dalloc<int>(c.get(), c->cand_cap);
        c->chunk_max = dalloc<int>(c.get(), 256);
        {
            std::vector<int> init(256, (int)0x80000000);
            BLK_CUDA(cudaMemcpy(c->chunk_max, init.data(), 256 * sizeof(int), cudaMemcpyHostToDevice));
        }
        c->counters = dalloc<unsigned int>(c.get(), 8 + ff / 256 + 8);
        BLK_CUDA(cudaMemset(c->counters, 0, (8 + ff / 256 + 8) * sizeof(unsigned int)));
        c->top_ids = dalloc<int32_t>(c.get(), TOPK_MAX); c->top_logits = dalloc<float>(c.get(), TOPK_MAX);
        c->h_top_ids = halloc<int32_t>(c.get(), TOPK_MAX); c->h_top_logits = halloc<float>(c.get(), TOPK_MAX);
        c->ids_cap = 4096;
        c->d_ids = dalloc<int32_t>(c.get(), c->ids_cap); c->d_gath = dalloc<float>(c.get(), c->ids_cap);
        if (m->n_vocab % 2) throw BlkError(BLK_ERR_FORMAT, "vocabulary size must be even");
        if (m->mega.ok) {   // persistent decode kernel: per-context parameters
            const blk_mega_model& mg = m->mega;
            MegaParams& P = c->mega_params;
            P.phases = mg.d_phases; P.n_phases = (int)mg.phases.size(); P.n_layer = m->n_layer;
            P.chunk_list = mg.d_list; P.chunk_counts = mg.d_counts; P.list_stride = mg.list_stride;
            P.n_cta = mg.n_cta; P.slot_bytes = mg.slot_bytes; P.max_items = mg.max_items; P.act_bytes = mg.act_bytes; P.ts_cap = mg.ts_cap; P.attn_off = mg.attn_off;
            P.tok_embd = m->tok_embd;
            P.n_embd = d; P.n_head = m->n_head; P.n_head_kv = m->n_head_kv; P.d_head = dh; P.n_ff = ff; P.n_vocab = m->n_vocab; P.neox = m->neox ? 1 : 0;
            P.eps = m->rms_eps; P.theta_scale = m->theta_scale; P.attn_scale = 1.0f / sqrtf((float)dh); P.rope_freqs = m->rope_freqs;
            P.tok = c->d_tok; P.pos = c->d_pos;
            P.max_split = std::max(1, std::min(32, mg.n_cta / m->n_head_kv));
            auto ll = [&](size_t n) { uint2* p = dalloc<uint2>(c.get(), n); BLK_CUDA(cudaMemset(p, 0, n * sizeof(uint2))); return p; };
            P.x2 = ll(d); P.q2 = ll(dq); P.h2 = ll(ff); P.ao2 = ll(dq);
            P.po2 = ll((size_t)P.max_split * dq); P.kvn2 = ll(2 * (size_t)dkv);
            P.st2 = ll((size_t)m->n_head * P.max_split * 2);

            P.k_pools = c->d_kpools; P.v_pools = c->d_vpools; P.page_table = c->page_table; P.kv_dim = dkv;
            P.logits = c->logits; P.chunk_max = c->chunk_max; P.chunk_shift = c->chunk_shift;
            {   // a poll that times out reports here instead of hanging the GPU (mapped pinned host word)
                void* hp = nullptr;
                BLK_CUDA(cudaHostAlloc(&hp, sizeof(int), cudaHostAllocMapped)); c->host_allocs.push_back(hp);
                c->mega_err = reinterpret_cast<int*>(hp); *c->mega_err = 0;
                void* dp = nullptr; BLK_CUDA(cudaHostGetDevicePointer(&dp, hp, 0)); P.err = reinterpret_cast<int*>(dp);
            }
            { const char* tr = getenv("BLK_MEGA_TRACE"); if (tr && (tr[0] == '1' || tr[0] == '2')) { P.trace_cap = 2048; P.trace_global = tr[0] == '2'; P.trace = dalloc<long long>(c.get(), (size_t)P.n_cta * P.trace_cap); } }
            c->mega_smem = mega_smem_bytes(P);
            int limit = 0;
            c->mega_on = mega_setup(c->mega_smem, &limit) == cudaSuccess;
            (void)cudaGetLastError();
        }
        {   // one eager step: loads modules and sets per-function attributes outside of stream capture
            BLK_CUDA(cudaMemsetAsync(c->d_tok, 0, sizeof(int32_t), c->stream));
            if (c->mega_on) {
                try { enqueue_step(c.get(), true, false); BLK_CUDA(cudaStreamSynchronize(c->stream)); check_mega(c.get()); }
                catch (const BlkError& err) {
                    (void)cudaGetLastError();
                    log_msg(2, std::string("persistent decode kernel unavailable (") + err.what() + "); using the per-op graph");
                    c->mega_on = false;
                }
            }
            if (!c->mega_on) { enqueue_step(c.get(), true, false); BLK_CUDA(cudaStreamSynchronize(c->stream)); }
            BLK_CUDA(cudaMemsetAsync(c->d_pos, 0, sizeof(int32_t), c->stream));
            c->launches = 0;
        }
        if (!c->mega_on) build_graphs(c.get());
        BLK_CUDA(cudaStreamSynchronize(c->stream));
    });
    if (st != BLK_OK) { fail(st == BLK_ERR_OOM ? BLK_ERR_OOM : st, std::string("Failed to create context: ") + g_last_error); return nullptr; }
    return c.release();
}
extern "C" void blk_ctx_free(blk_ctx* c) { delete c; }
extern "C" int32_t blk_ctx_n_ctx(const blk_ctx* c) { return c->n_ctx; }
extern "C" int32_t blk_ctx_n_batch(const blk_ctx* c) { return c->n_batch; }
extern "C" int32_t blk_ctx_n_past(const blk_ctx* c) { return c->n_past; }
extern "C" const blk_model* blk_ctx_model(const blk_ctx* c) { return c->m; }
extern "C" int64_t blk_ctx_kernel_launches(const blk_ctx* c) { return c->launches; }
extern "C" int32_t blk_ctx_persistent_decode(const blk_ctx* c) { return c->mega_on ? 1 : 0; }

extern "C" blk_status blk_ctx_set_verify_mode(blk_ctx* c, int32_t mode) {
    if (!c || mode < 0 || mode > 1) return fail(BLK_ERR_ARG, "blk_ctx_set_verify_mode: bad arguments");
    c->verify_mode = mode; return BLK_OK;
}

extern "C" blk_status blk_kv_clear(blk_ctx* c) {
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        BLK_CUDA(cudaMemsetAsync(c->d_pos, 0, 2 * sizeof(int32_t), c->stream));
        c->n_past = 0; c->have_logits = false;
        c->cell_pos.clear(); c->cell_shift.clear(); c->rope_off = 0; c->shift_pending = false;
    });
}
extern "C" blk_status blk_sync(blk_ctx* c) {
    return guarded([&] { BLK_CUDA(cudaSetDevice(c->m->device)); BLK_CUDA(cudaStreamSynchronize(c->stream)); check_mega(c); });
}

// ------------------------------------------------------------------------------------------------------------------
// context shift + state (reference Session.cpp:324-347 llama_kv_self_seq_rm / seq_add; :284-310 llama_state_get/set_data)
// ------------------------------------------------------------------------------------------------------------------
namespace {
// Cache rows [src0, src0 + n) of every layer move to [dst0, dst0 + n) (the two ranges do not overlap within one launch).  K rows are
// re-rotated by `delta` positions the way llama.cpp's K-shift does it (ggml rope on the F16 cache: f16 -> f32, rotate by
// theta_i = delta * theta_scale^i / freq_factor_i, f32 -> f16); V rows are copied.  grid = (n, n_layer), block = 128.
__global__ void __launch_bounds__(128) kv_shift_kernel(__half* const* __restrict__ k_pools, __half* const* __restrict__ v_pools,
                                                       const int32_t* __restrict__ page_table, int kv_dim, int d_head, int neox, int src0, int dst0,
                                                       int delta, float theta_scale, const float* __restrict__ freq_factors) {
    __shared__ float2 cs[64];
    const int half_rot = d_head / 2;
    rope_table_fill(cs, half_rot, delta, theta_scale, freq_factors);
    __syncthreads();
    const int ts = src0 + (int)blockIdx.x, td = dst0 + (int)blockIdx.x;
    const size_t rs = ((size_t)page_table[ts / KV_PAGE] * KV_PAGE + (ts % KV_PAGE)) * kv_dim;
    const size_t rd = ((size_t)page_table[td / KV_PAGE] * KV_PAGE + (td % KV_PAGE)) * kv_dim;
    const __half* ks = k_pools[blockIdx.y] + rs; __half* kd = k_pools[blockIdx.y] + rd;
    const __half* vs = v_pools[blockIdx.y] + rs; __half* vd = v_pools[blockIdx.y] + rd;
    for (int p = threadIdx.x; p < kv_dim / 2; p += blockDim.x) {
        const int h = p / half_rot, i = p - h * half_rot;
        const int e0 = neox ? h * d_head + i : h * d_head + 2 * i;
        const int e1 = neox ? e0 + half_rot : e0 + 1;
        const float x0 = __half2float(ks[e0]), x1 = __half2float(ks[e1]);
        const float2 c = cs[i];
        kd[e0] = __float2half_rn(__fsub_rn(__fmul_rn(x0, c.x), __fmul_rn(x1, c.y)));
        kd[e1] = __float2half_rn(__fadd_rn(__fmul_rn(x0, c.y), __fmul_rn(x1, c.x)));
    }
    for (int e = threadIdx.x; e < kv_dim / 8; e += blockDim.x) reinterpret_cast<uint4*>(vd)[e] = reinterpret_cast<const uint4*>(vs)[e];
}

constexpr uint32_t STATE_MAGIC = 0x534B4C42u;      // "BLKS"
struct StateHeader { uint32_t magic, version; int32_t n_layer, kv_dim, n_vocab, n_past, have_logits, reserved; };
size_t state_bytes(const blk_ctx* c, int n_past, bool with_positions) {
    const blk_model* m = c->m;
    const size_t kv_dim = (size_t)m->n_head_kv * m->d_head;
    return sizeof(StateHeader) + (size_t)m->n_vocab * 4 + TOPK_MAX * 8 + (with_positions ? 4 + (size_t)n_past * 4 : 0) +
           2 * (size_t)m->n_layer * (size_t)n_past * kv_dim * 2;
}
} // namespace

extern "C" blk_status blk_kv_shift(blk_ctx* c, int32_t p0, int32_t p1) {
    if (!c || p0 < 0 || p1 <= p0 || p1 > c->n_past) return fail(BLK_ERR_ARG, "blk_kv_shift: bad range");
    return guarded([&] {
        blk_model* m = c->m;
        BLK_CUDA(cudaSetDevice(m->device));
        if (!c->cell_pos.empty()) throw BlkError(BLK_ERR_ARG, "blk_kv_shift: not available once Self-Extend has moved cell positions (blk_kv_seq_add / blk_kv_seq_div)");
        const int d = p1 - p0, dkv = m->n_head_kv * m->d_head;
        // front to back in chunks of at most d rows: a chunk's destination never overlaps its source, and what it overwrites has been
        // moved already
        for (int t = p1; t < c->n_past; t += d) {
            const int n = std::min(d, c->n_past - t);
            kv_shift_kernel<<<dim3((unsigned)n, (unsigned)m->n_layer), 128, 0, c->stream>>>(c->d_kpools, c->d_vpools, c->page_table, dkv, m->d_head, m->neox ? 1 : 0,
                                                                                                t, t - d, -d, m->theta_scale, m->rope_freqs);
            BLK_CUDA(cudaGetLastError());
            c->launches++;
        }
        c->n_past -= d;
        int32_t np = c->n_past;
        BLK_CUDA(cudaMemcpyAsync(c->d_pos, &np, sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
        BLK_CUDA(cudaStreamSynchronize(c->stream));      // np is a stack variable
    });
}

extern "C" int64_t blk_state_size(const blk_ctx* c) { return c ? (int64_t)state_bytes(c, c->n_past, !c->cell_pos.empty()) : 0; }

extern "C" blk_status blk_state_get(blk_ctx* c, void* dst, int64_t cap, int64_t* written) {
    if (!c || !dst || !written) return fail(BLK_ERR_ARG, "blk_state_get: bad arguments");
    return guarded([&] {
        blk_model* m = c->m;
        BLK_CUDA(cudaSetDevice(m->device));
        const bool with_pos = !c->cell_pos.empty();
        const size_t need = state_bytes(c, c->n_past, with_pos);
        if ((size_t)cap < need) throw BlkError(BLK_ERR_ARG, "blk_state_get: buffer too small");
        flush_pos_shift(c);
        BLK_CUDA(cudaStreamSynchronize(c->stream));
        check_mega(c);
        uint8_t* out = static_cast<uint8_t*>(dst);
        const int kv_dim = m->n_head_kv * m->d_head;
        StateHeader h{STATE_MAGIC, 1u, m->n_layer, kv_dim, m->n_vocab, c->n_past, c->have_logits ? 1 : 0, with_pos ? 1 : 0};
        memcpy(out, &h, sizeof(h)); out += sizeof(h);
        BLK_CUDA(cudaMemcpy(out, c->logits, (size_t)m->n_vocab * 4, cudaMemcpyDeviceToHost)); out += (size_t)m->n_vocab * 4;
        memcpy(out, c->h_top_ids, TOPK_MAX * 4); out += TOPK_MAX * 4;
        memcpy(out, c->h_top_logits, TOPK_MAX * 4); out += TOPK_MAX * 4;
        if (with_pos) {      // Self-Extend moved cell positions: they are part of the state
            const int32_t off = c->rope_off;
            memcpy(out, &off, 4); out += 4;
            memcpy(out, c->cell_pos.data(), (size_t)c->n_past * 4); out += (size_t)c->n_past * 4;
        }
        const size_t row = (size_t)kv_dim * 2;
        for (int l = 0; l < m->n_layer; l++)
            for (const __half* pool : {c->k_pool[l], c->v_pool[l]})
                for (int t0 = 0; t0 < c->n_past; t0 += KV_PAGE) {
                    const int n = std::min(KV_PAGE, c->n_past - t0);
                    BLK_CUDA(cudaMemcpy(out, pool + (size_t)c->page_table_host[t0 / KV_PAGE] * KV_PAGE * kv_dim, n * row, cudaMemcpyDeviceToHost));
                    out += n * row;
                }
        *written = (int64_t)need;
    });
}

extern "C" blk_status blk_state_set(blk_ctx* c, const void* src, int64_t size) {
    if (!c || !src || size < (int64_t)sizeof(StateHeader)) return fail(BLK_ERR_ARG, "blk_state_set: bad arguments");
    return guarded([&] {
        blk_model* m = c->m;
        BLK_CUDA(cudaSetDevice(m->device));
        const uint8_t* in = static_cast<const uint8_t*>(src);
        StateHeader h;
        memcpy(&h, in, sizeof(h)); in += sizeof(h);
        const int kv_dim = m->n_head_kv * m->d_head;
        if (h.magic != STATE_MAGIC || h.version != 1u) throw BlkError(BLK_ERR_FORMAT, "blk_state_set: not a state blob of this engine");
        if (h.n_layer != m->n_layer || h.kv_dim != kv_dim || h.n_vocab != m->n_vocab) throw BlkError(BLK_ERR_FORMAT, "blk_state_set: the state belongs to another model");
        if (h.n_past < 0 || h.n_past > c->n_ctx) throw BlkError(BLK_ERR_CTX_FULL, "blk_state_set: the state does not fit this context");
        if ((size_t)size != state_bytes(c, h.n_past, h.reserved != 0)) throw BlkError(BLK_ERR_FORMAT, "blk_state_set: truncated state");
        BLK_CUDA(cudaStreamSynchronize(c->stream));
        BLK_CUDA(cudaMemcpy(c->logits, in, (size_t)m->n_vocab * 4, cudaMemcpyHostToDevice)); in += (size_t)m->n_vocab * 4;
        memcpy(c->h_top_ids, in, TOPK_MAX * 4); in += TOPK_MAX * 4;
        memcpy(c->h_top_logits, in, TOPK_MAX * 4); in += TOPK_MAX * 4;
        BLK_CUDA(cudaMemcpy(c->top_ids, c->h_top_ids, TOPK_MAX * 4, cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(c->top_logits, c->h_top_logits, TOPK_MAX * 4, cudaMemcpyHostToDevice));
        c->cell_pos.clear(); c->cell_shift.clear(); c->rope_off = 0; c->shift_pending = false;
        if (h.reserved != 0) {
            int32_t off = 0;
            memcpy(&off, in, 4); in += 4;
            c->cell_pos.assign((size_t)c->n_ctx, 0); c->cell_shift.assign((size_t)c->n_ctx, 0);
            memcpy(c->cell_pos.data(), in, (size_t)h.n_past * 4); in += (size_t)h.n_past * 4;
            c->rope_off = off;
        }
        const size_t row = (size_t)kv_dim * 2;
        for (int l = 0; l < m->n_layer; l++)
            for (__half* pool : {c->k_pool[l], c->v_pool[l]})
                for (int t0 = 0; t0 < h.n_past; t0 += KV_PAGE) {
                    const int n = std::min(KV_PAGE, h.n_past - t0);
                    BLK_CUDA(cudaMemcpy(pool + (size_t)c->page_table_host[t0 / KV_PAGE] * KV_PAGE * kv_dim, in, n * row, cudaMemcpyHostToDevice));
                    in += n * row;
                }
        c->n_past = h.n_past; c->have_logits = h.have_logits != 0;
        const int32_t both[2] = {h.n_past, c->rope_off};
        BLK_CUDA(cudaMemcpy(c->d_pos, both, sizeof(both), cudaMemcpyHostToDevice));
    });
}

extern "C" blk_status blk_decode(blk_ctx* c, const int32_t* tokens, int32_t n) {
    if (!c || !tokens || n <= 0) return fail(BLK_ERR_ARG, "blk_decode: bad arguments");
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        if (c->n_past + n > c->n_ctx) throw BlkError(BLK_ERR_CTX_FULL, "context is full");
        for (int i = 0; i < n; i++) if (tokens[i] < 0 || tokens[i] >= c->m->n_vocab) throw BlkError(BLK_ERR_ARG, "token id out of range");
        if (n >= c->prefill_min) {
            const int per = balanced_chunk(n, c->n_batch);
            for (int off = 0; off < n; off += per) prefill_chunk(c, tokens + off, std::min(per, n - off), nullptr, 0);
            return;
        }
        for (int i = 0; i < n; i++) step(c, tokens[i], i == n - 1);
    });
}

// ------------------------------------------------------------------------------------------------------------------
// batched decode step: n sequences, one new token each, ONE pass over the weights (continuous batching, SURVEY.md 8f item 4)
// ------------------------------------------------------------------------------------------------------------------
namespace {
struct BatchDesc {       // layout of blk_ctx::bd_host / bd_dev
    int32_t tokens[BATCH_MAX];
    int32_t pos[BATCH_MAX];          // cell index of the new token
    int32_t rpos[BATCH_MAX];         // its rotary position (differs after Self-Extend)
    const int32_t* page_table[BATCH_MAX];
    __half* const* k_pools[BATCH_MAX];
    __half* const* v_pools[BATCH_MAX];
    int32_t* pos_ptr[BATCH_MAX];
};
} // namespace

extern "C" blk_status blk_decode_batch(blk_ctx* ws, blk_ctx* const* ctxs, const int32_t* tokens, int32_t n, int32_t k, blk_token_data* out) {
    if (!ws || !ctxs || !tokens || !out || n <= 0 || n > BATCH_MAX || k <= 0 || k > TOPK_MAX) return fail(BLK_ERR_ARG, "blk_decode_batch: bad arguments");
    return guarded([&] {
        blk_model* m = ws->m;
        BLK_CUDA(cudaSetDevice(m->device));
        const int d = m->n_embd, dh = m->d_head, dq = m->n_head * dh, dkv = m->n_head_kv * dh, V = m->n_vocab;
        for (int i = 0; i < n; i++) {
            blk_ctx* c = ctxs[i];
            if (!c || c->m != m) throw BlkError(BLK_ERR_ARG, "blk_decode_batch: every context must belong to the workspace's model");
            for (int j = 0; j < i; j++) if (ctxs[j] == c) throw BlkError(BLK_ERR_ARG, "blk_decode_batch: a context appears twice");
            if (tokens[i] < 0 || tokens[i] >= V) throw BlkError(BLK_ERR_ARG, "token id out of range");
            if (c->n_past + 1 > c->n_ctx) throw BlkError(BLK_ERR_CTX_FULL, "context is full");
            BLK_CUDA(cudaStreamSynchronize(c->stream));          // its prompt prefill / previous step ran on its own stream
            flush_pos_shift(c);
        }
        ensure_prefill_bufs(ws, n);
        if (!ws->bd_host) {
            ws->bd_host = reinterpret_cast<uint8_t*>(halloc<BatchDesc>(ws, 1));
            ws->bd_dev = reinterpret_cast<uint8_t*>(dalloc<BatchDesc>(ws, 1));
            ws->bd_top_ids = dalloc<int32_t>(ws, BATCH_MAX * TOPK_MAX); ws->bd_top_logits = dalloc<float>(ws, BATCH_MAX * TOPK_MAX);
            ws->bd_h_top_ids = halloc<int32_t>(ws, BATCH_MAX * TOPK_MAX); ws->bd_h_top_logits = halloc<float>(ws, BATCH_MAX * TOPK_MAX);
            // per-row scratch of the batched threshold selector
            ws->bd_chunk_max = dalloc<int>(ws, BATCH_MAX * 256);
            { std::vector<int> init(BATCH_MAX * 256, (int)0x80000000); BLK_CUDA(cudaMemcpy(ws->bd_chunk_max, init.data(), init.size() * sizeof(int), cudaMemcpyHostToDevice)); }
            ws->bd_cand_l = dalloc<float>(ws, (size_t)BATCH_MAX * ws->cand_cap); ws->bd_cand_i = dalloc<int>(ws, (size_t)BATCH_MAX * ws->cand_cap);
            ws->bd_counters = dalloc<unsigned int>(ws, 2 * BATCH_MAX);
            BLK_CUDA(cudaMemset(ws->bd_counters, 0, 2 * BATCH_MAX * sizeof(unsigned int)));
        }
        cudaStream_t st = ws->stream;
        BLK_CUDA(cudaStreamSynchronize(st));                      // the staging block is reused every step
        BatchDesc* h = reinterpret_cast<BatchDesc*>(ws->bd_host);
        const BatchDesc* dv = reinterpret_cast<const BatchDesc*>(ws->bd_dev);
        for (int i = 0; i < n; i++) {
            h->tokens[i] = tokens[i]; h->pos[i] = ctxs[i]->n_past; h->rpos[i] = ctxs[i]->n_past + ctxs[i]->rope_off; h->page_table[i] = ctxs[i]->page_table;
            note_new_cells(ctxs[i], 1);
            h->k_pools[i] = ctxs[i]->d_kpools; h->v_pools[i] = ctxs[i]->d_vpools; h->pos_ptr[i] = ctxs[i]->d_pos;
        }
        BLK_CUDA(cudaMemcpyAsync(ws->bd_dev, ws->bd_host, sizeof(BatchDesc), cudaMemcpyHostToDevice, st));
        embed_rows_kernel<<<n, 256, 0, st>>>(m->tok_embd, dv->tokens, dv->rpos, ws->pf_x, ws->pf_rope, dh / 2, m->theta_scale, m->rope_freqs);
        BLK_CUDA(cudaGetLastError()); ws->launches++;
        const ChainPdl chain_scope(n);
        // matrices with a resident bf16 panel (model cache) take the TMA-fed GEMM: the step then streams the panels at HBM speed
        // instead of waiting for the de-quantising producers of the fused form (BATCH_MAX rows are below the default panel_min)
        GemmSchedule sched(ws, n, n_gemm_ops(m));
        PendingReduce pend;
        run_layers(ws, n, sched, pend, true, [&](int l) {
            QkvPostBatchArgs qa{};
            qa.base.qkv = ws->pf_qkv; qa.base.ld = dq + 2 * dkv; qa.base.rope_cs = ws->pf_rope; qa.base.q_out = ws->pf_q;
            qa.base.dq = dq; qa.base.dkv = dkv; qa.base.d_head = dh; qa.base.neox = m->neox ? 1 : 0;
            qa.pos = dv->pos; qa.page_table = dv->page_table; qa.k_pools = dv->k_pools; qa.v_pools = dv->v_pools; qa.layer = l;
            BLK_CUDA(launch_chain(qkv_post_batch_kernel, dim3(n), dim3(256), 0, st, qa));
            BatchAttnArgs aa{};
            aa.q = ws->pf_q; aa.pos = dv->pos; aa.page_table = dv->page_table; aa.k_pools = dv->k_pools; aa.v_pools = dv->v_pools; aa.out = ws->pf_ao;
            aa.layer = l; aa.n_head = m->n_head; aa.n_head_kv = m->n_head_kv; aa.kv_dim = dkv; aa.scale = 1.0f / sqrtf((float)dh);
            if (dh == 128) BLK_CUDA(launch_chain(decode_attn_batch_kernel<128>, dim3(m->n_head_kv, n), dim3(256), 0, st, aa));
            else BLK_CUDA(launch_chain(decode_attn_batch_kernel<64>, dim3(m->n_head_kv, n), dim3(256), 0, st, aa));
            BLK_CUDA(cudaGetLastError());
            ws->launches += 2;
        });
        rmsnorm_bf16_launch(ws->pf_x, m->out_norm, d, m->rms_eps, ws->pf_xn, n, st, &pend);
        const GemmOp head = sched.next(OP_HEAD);
        BLK_CUDA(prefill_gemm(*head.part[0].W, ws->pf_xn, n, ws->pf_logits, V, nullptr, 0, st, head.panel));
        ws->launches += 2;
        // threshold top-64 of every row (the selector of the batch-1 path, blockIdx.y = row): two launches for the whole batch
        {
            chunk_max_kernel<<<dim3(ws->n_chunks, n), 256, 0, st>>>(ws->pf_logits, V, ws->chunk_shift, ws->bd_chunk_max, (long long)V);
            TopkArgs tk{};
            tk.logits = ws->pf_logits; tk.n = V; tk.ld = V; tk.chunk_max = ws->bd_chunk_max; tk.n_chunks = ws->n_chunks;
            tk.cand_l = ws->bd_cand_l; tk.cand_i = ws->bd_cand_i; tk.cap = ws->cand_cap; tk.count = ws->bd_counters; tk.done = ws->bd_counters + 1;
            tk.out_ids = ws->bd_top_ids; tk.out_logits = ws->bd_top_logits;
            topk_select_kernel<<<dim3(16, n), 1024, 0, st>>>(tk);
            BLK_CUDA(cudaGetLastError()); ws->launches += 2;
        }
        advance_many_kernel<<<1, BATCH_MAX, 0, st>>>(dv->pos_ptr, n);
        BLK_CUDA(cudaGetLastError()); ws->launches++;
        BLK_CUDA(cudaMemcpyAsync(ws->bd_h_top_ids, ws->bd_top_ids, (size_t)n * TOPK_MAX * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        BLK_CUDA(cudaMemcpyAsync(ws->bd_h_top_logits, ws->bd_top_logits, (size_t)n * TOPK_MAX * sizeof(float), cudaMemcpyDeviceToHost, st));
        BLK_CUDA(cudaStreamSynchronize(st));
        for (int i = 0; i < n; i++) {
            ctxs[i]->n_past++; ctxs[i]->have_logits = false;
            for (int j = 0; j < k; j++) { out[(size_t)i * k + j].token = ws->bd_h_top_ids[i * TOPK_MAX + j]; out[(size_t)i * k + j].logit = ws->bd_h_top_logits[i * TOPK_MAX + j]; }
        }
    });
}

extern "C" blk_status blk_decode_loop(blk_ctx* c, int32_t first_token, int32_t n_steps, int32_t* last_token) {
    if (!c || n_steps <= 0) return fail(BLK_ERR_ARG, "blk_decode_loop: bad arguments");
    return guarded([&] {
        blk_model* m = c->m;
        BLK_CUDA(cudaSetDevice(m->device));
        if (first_token < 0 || first_token >= m->n_vocab) throw BlkError(BLK_ERR_ARG, "token id out of range");
        if (c->n_past + n_steps > c->n_ctx) throw BlkError(BLK_ERR_CTX_FULL, "context is full");
        flush_pos_shift(c);
        note_new_cells(c, n_steps);
        BLK_CUDA(cudaStreamSynchronize(c->stream));
        c->h_tok[0] = first_token; c->tok_slot = 1;
        BLK_CUDA(cudaMemcpyAsync(c->d_tok, c->h_tok, sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
        if (c->mega_on) { for (int i = 0; i < n_steps; i++) enqueue_step(c, true, true); }
        else {
            for (int i = 0; i < n_steps; i++) BLK_CUDA(cudaGraphLaunch(c->g_loop, c->stream));
            c->launches += c->launches_loop * n_steps;
        }
        c->n_past += n_steps;
        BLK_CUDA(cudaMemcpyAsync(c->h_top_ids, c->top_ids, TOPK_MAX * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        BLK_CUDA(cudaMemcpyAsync(c->h_top_logits, c->top_logits, TOPK_MAX * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        c->have_logits = true;
        if (last_token) { BLK_CUDA(cudaStreamSynchronize(c->stream)); *last_token = c->h_top_ids[0]; }
    });
}

extern "C" blk_status blk_topk_last(blk_ctx* c, int32_t k, blk_token_data* out) {
    if (!c || !out || k <= 0 || k > TOPK_MAX) return fail(BLK_ERR_ARG, "blk_topk_last: bad arguments");
    return guarded([&] {
        if (!c->have_logits) throw BlkError(BLK_ERR_ARG, "no logits available: decode first");
        BLK_CUDA(cudaSetDevice(c->m->device));
        BLK_CUDA(cudaStreamSynchronize(c->stream));
        check_mega(c);
        for (int i = 0; i < k; i++) { out[i].token = c->h_top_ids[i]; out[i].logit = c->h_top_logits[i]; }
    });
}

extern "C" blk_status blk_decode_topk(blk_ctx* c, int32_t token, int32_t k, blk_token_data* out) {
    if (!c || !out || k <= 0 || k > TOPK_MAX) return fail(BLK_ERR_ARG, "blk_decode_topk: bad arguments");
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        step(c, token, true);
        BLK_CUDA(cudaStreamSynchronize(c->stream));
        check_mega(c);
        for (int i = 0; i < k; i++) { out[i].token = c->h_top_ids[i]; out[i].logit = c->h_top_logits[i]; }
    });
}

extern "C" blk_status blk_gather_last(blk_ctx* c, const int32_t* ids, int32_t n, float* out) {
    if (!c || !ids || !out || n <= 0 || n > 4096) return fail(BLK_ERR_ARG, "blk_gather_last: bad arguments");
    return guarded([&] {
        if (!c->have_logits) throw BlkError(BLK_ERR_ARG, "no logits available: decode first");
        BLK_CUDA(cudaSetDevice(c->m->device));
        BLK_CUDA(cudaMemcpyAsync(c->d_ids, ids, n * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
        BLK_CUDA(launch_pdl(gather_logits_kernel, dim3((n + 127) / 128), dim3(128), 0, c->stream, c->logits, c->m->n_vocab, c->d_ids, n, c->d_gath));
        BLK_CUDA(cudaGetLastError()); c->launches++;
        BLK_CUDA(cudaMemcpyAsync(out, c->d_gath, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        BLK_CUDA(cudaStreamSynchronize(c->stream));
    });
}

extern "C" blk_status blk_get_logits_last(blk_ctx* c, float* out) {
    if (!c || !out) return fail(BLK_ERR_ARG, "blk_get_logits_last: bad arguments");
    return guarded([&] {
        if (!c->have_logits) throw BlkError(BLK_ERR_ARG, "no logits available: decode first");
        BLK_CUDA(cudaSetDevice(c->m->device));
        BLK_CUDA(cudaMemcpyAsync(out, c->logits, (size_t)c->m->n_vocab * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        BLK_CUDA(cudaStreamSynchronize(c->stream));
    });
}

extern "C" blk_status blk_verify_prefill(blk_ctx* c, const int32_t* tokens, int32_t n, const int32_t* claimed, const int32_t* n_claimed,
                                         float* gathered, blk_token_data* top) {
    if (!c || !tokens || n <= 0 || !claimed || !n_claimed || !gathered) return fail(BLK_ERR_ARG, "blk_verify_prefill: bad arguments");
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        if (c->n_past + n > c->n_ctx) throw BlkError(BLK_ERR_CTX_FULL, "context is full");
        for (int i = 0; i < n; i++) if (tokens[i] < 0 || tokens[i] >= c->m->n_vocab) throw BlkError(BLK_ERR_ARG, "token id out of range");
        if (c->verify_mode == 0 && n >= c->prefill_min) {
            VerifyIo io{claimed, n_claimed, gathered, top};
            const int per = balanced_chunk(n, c->n_batch);
            for (int off = 0; off < n; off += per) prefill_chunk(c, tokens + off, std::min(per, n - off), &io, off);
            return;
        }
        // sequential form of the context fill: one batch-1 decode per response token (Session.cpp:235-241), logits gathered
        // on the device at the claimed ids.  Bit-identical to what blk_decode_topk produced for the prover.
        for (int i = 0; i < n; i++) {
            step(c, tokens[i], true);
            const int nc = std::max(0, std::min(10, n_claimed[i]));
            if (nc > 0) {
                BLK_CUDA(cudaMemcpyAsync(c->d_ids, claimed + (size_t)i * 10, nc * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
                BLK_CUDA(launch_pdl(gather_logits_kernel, dim3(1), dim3(32), 0, c->stream, c->logits, c->m->n_vocab, c->d_ids, nc, c->d_gath));
                BLK_CUDA(cudaGetLastError()); c->launches++;
                BLK_CUDA(cudaMemcpyAsync(gathered + (size_t)i * 10, c->d_gath, nc * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
            }
            BLK_CUDA(cudaStreamSynchronize(c->stream));
            if (top) for (int j = 0; j < 10; j++) { top[(size_t)i * 10 + j].token = c->h_top_ids[j]; top[(size_t)i * 10 + j].logit = c->h_top_logits[j]; }
        }
    });
}

// ------------------------------------------------------------------------------------------------------------------
// measurement
// ------------------------------------------------------------------------------------------------------------------
extern "C" blk_status blk_timer_start(blk_ctx* c) {
    return guarded([&] { BLK_CUDA(cudaSetDevice(c->m->device)); BLK_CUDA(cudaEventRecord(c->ev0, c->stream)); });
}
extern "C" blk_status blk_timer_stop(blk_ctx* c, float* ms) {
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        BLK_CUDA(cudaEventRecord(c->ev1, c->stream));
        BLK_CUDA(cudaEventSynchronize(c->ev1));
        BLK_CUDA(cudaEventElapsedTime(ms, c->ev0, c->ev1));
    });
}
extern "C" blk_status blk_bench_kernel(blk_ctx* c, int32_t which, int32_t iters, float* avg_ms, int64_t* bytes_per_launch) {
    if (!c || iters <= 0 || !avg_ms || !bytes_per_launch || which < 0 || which > 5) return fail(BLK_ERR_ARG, "blk_bench_kernel: bad arguments");
    return guarded([&] {
        blk_model* m = c->m;
        BLK_CUDA(cudaSetDevice(m->device));
        if (which == 5) {
            // the persistent decode kernel alone (no top-k, position held): one launch = one token's whole forward
            if (!c->mega_on) throw BlkError(BLK_ERR_ARG, "blk_bench_kernel(5): this context does not run the persistent decode kernel");
            if (c->n_past + 1 > c->n_ctx) throw BlkError(BLK_ERR_CTX_FULL, "context is full");
            auto one = [&] {
                MegaParams P = c->mega_params;
                P.with_head = 1; P.advance_pos = 0; P.seq = ++c->mega_seq;
                BLK_CUDA(mega_launch(P, c->mega_smem, c->stream));
                c->launches++;
            };
            BLK_CUDA(cudaMemsetAsync(c->d_tok, 0, sizeof(int32_t), c->stream));
            for (int i = 0; i < std::min(iters, 4); i++) one();
            BLK_CUDA(cudaEventRecord(c->ev0, c->stream));
            for (int i = 0; i < iters; i++) one();
            BLK_CUDA(cudaEventRecord(c->ev1, c->stream));
            BLK_CUDA(cudaEventSynchronize(c->ev1));
            check_mega(c);
            float ms = 0.0f;
            BLK_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
            *avg_ms = ms / (float)iters;
            *bytes_per_launch = m->weight_bytes_per_token + (int64_t)(c->n_past + 1) * blk_model_kv_bytes_per_token(m);
            // the launches left chunk maxima behind (no top-k ran): clear them, and forget the logits
            std::vector<int> init(256, (int)0x80000000);
            BLK_CUDA(cudaMemcpyAsync(c->chunk_max, init.data(), 256 * sizeof(int), cudaMemcpyHostToDevice, c->stream));
            BLK_CUDA(cudaStreamSynchronize(c->stream));
            c->have_logits = false;
            return;
        }
        const int d = m->n_embd, dh = m->d_head, dq = m->n_head * dh, dkv = m->n_head_kv * dh, ff = m->n_ff;
        // make the activation buffers hold something sane
        BLK_CUDA(cudaMemsetAsync(c->x, 0, d * sizeof(float), c->stream));
        BLK_CUDA(cudaMemsetAsync(c->hbuf, 0, ff * sizeof(float), c->stream));
        BLK_CUDA(cudaMemsetAsync(c->act_q.f32, 0, dq * sizeof(float), c->stream));
        int64_t bytes = 0;
        auto one = [&](int it, bool count) {
            const LayerWeights& L = m->layers[it % m->n_layer];
            GemvArgs a{};
            switch (which) {
            case 0:
                a.nseg = 2; a.seg[0] = {L.gate, nullptr, 0, 0}; a.seg[1] = {L.up, nullptr, 0, 0}; a.total_pairs = ff; a.out = c->hbuf;
                if (count) bytes += (int64_t)L.gate.bytes + (int64_t)L.up.bytes + d * 8 + ff * 4;
                matvec<EPI_SWIGLU>(c, a, c->x, L.ffn_norm, c->act_d, "bench"); break;
            case 1:
                a.nseg = 1; a.seg[0] = {L.down, nullptr, 0, 0}; a.total_pairs = d / 2; a.out = c->x;
                if (count) bytes += (int64_t)L.down.bytes + ff * 4 + d * 8;
                matvec<EPI_RESID>(c, a, c->hbuf, nullptr, c->act_ff, "bench"); break;
            case 2:
                a.nseg = 3; a.seg[0] = {L.wq, L.bq, 0, 0}; a.seg[1] = {L.wk, L.bk, dq / 2, 1}; a.seg[2] = {L.wv, L.bv, dq / 2 + dkv / 2, 2};
                a.total_pairs = dq / 2 + dkv; a.out = c->qbuf;
                a.d_head = dh; a.neox = m->neox ? 1 : 0; a.rope_cs = c->rope_cs; a.pos = c->d_pos;
                a.k_pool = c->k_pool[it % m->n_layer]; a.v_pool = c->v_pool[it % m->n_layer]; a.page_table = c->page_table; a.kv_dim = dkv;
                if (count) bytes += (int64_t)(L.wq.bytes + L.wk.bytes + L.wv.bytes) + d * 8 + dq * 4 + dkv * 4;
                matvec<EPI_QKV>(c, a, c->x, L.attn_norm, c->act_d, "bench"); break;
            case 3:
                a.nseg = 1; a.seg[0] = {L.wo, nullptr, 0, 0}; a.total_pairs = d / 2; a.out = c->x;
                if (count) bytes += (int64_t)L.wo.bytes + dq * 4 + d * 8;
                matvec<EPI_RESID>(c, a, c->act_q.f32, nullptr, c->act_q2, "bench"); break;
            default:
                a.nseg = 1; a.seg[0] = {m->output, nullptr, 0, 0}; a.total_pairs = m->n_vocab / 2; a.out = c->logits;
                if (count) bytes += (int64_t)m->output.bytes + d * 8 + (int64_t)m->n_vocab * 4;
                matvec<EPI_STORE>(c, a, c->x, m->out_norm, c->act_d, "bench"); break;
            }
        };
        for (int i = 0; i < std::min(iters, 8); i++) one(i, false);          // warm-up
        BLK_CUDA(cudaEventRecord(c->ev0, c->stream));
        for (int i = 0; i < iters; i++) one(i, true);
        BLK_CUDA(cudaEventRecord(c->ev1, c->stream));
        BLK_CUDA(cudaEventSynchronize(c->ev1));
        float ms = 0.0f;
        BLK_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
        *avg_ms = ms / (float)iters;
        *bytes_per_launch = bytes / iters;
        BLK_CUDA(cudaMemsetAsync(c->d_pos, 0, sizeof(int32_t), c->stream));
        c->n_past = 0; c->have_logits = false;
    });
}

namespace {
void prof_report(blk_ctx* c, char* report, int32_t cap) {
    std::map<std::string, std::pair<int, float>> agg;
    float total = 0.0f;
    for (size_t i = 1; i < c->prof_marks.size(); i++) {
        float ms = 0.0f;
        BLK_CUDA(cudaEventElapsedTime(&ms, c->prof_marks[i - 1].second, c->prof_marks[i].second));
        auto& a = agg[c->prof_marks[i].first]; a.first++; a.second += ms; total += ms;
    }
    for (auto& p : c->prof_marks) cudaEventDestroy(p.second);
    c->prof_marks.clear();
    std::string out = "kernel,launches,total_us,avg_us,share\n";
    char line[256];
    for (auto& kv : agg) {
        snprintf(line, sizeof(line), "%s,%d,%.1f,%.2f,%.3f\n", kv.first.c_str(), kv.second.first, kv.second.second * 1e3f,
                 kv.second.second * 1e3f / kv.second.first, kv.second.second / total);
        out += line;
    }
    snprintf(line, sizeof(line), "TOTAL,,%.1f,,1.0\n", total * 1e3f);
    out += line;
    snprintf(report, (size_t)cap, "%s", out.c_str());
}
} // namespace

extern "C" blk_status blk_profile_step(blk_ctx* c, int32_t token, char* report, int32_t cap) {
    if (!c || !report || cap <= 0) return fail(BLK_ERR_ARG, "blk_profile_step: bad arguments");
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        if (c->n_past + 1 > c->n_ctx) throw BlkError(BLK_ERR_CTX_FULL, "context is full");
        BLK_CUDA(cudaStreamSynchronize(c->stream));
        c->h_tok[0] = token; c->tok_slot = 1;
        BLK_CUDA(cudaMemcpyAsync(c->d_tok, c->h_tok, sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
        c->profiling = true; c->prof_marks.clear();
        prof_mark(c, "start");
        enqueue_step(c, true, false);
        c->profiling = false;
        BLK_CUDA(cudaStreamSynchronize(c->stream));
        c->n_past++; c->have_logits = true;
        prof_report(c, report, cap);
    });
}

extern "C" blk_status blk_profile_verify(blk_ctx* c, const int32_t* tokens, int32_t n, char* report, int32_t cap) {
    if (!c || !tokens || n <= 0 || !report || cap <= 0) return fail(BLK_ERR_ARG, "blk_profile_verify: bad arguments");
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        if (c->n_past + n > c->n_ctx || n > c->n_batch) throw BlkError(BLK_ERR_CTX_FULL, "context is full / chunk too large");
        std::vector<int32_t> claimed((size_t)n * 10, 0), ncl((size_t)n, 10);
        std::vector<float> g((size_t)n * 10);
        std::vector<blk_token_data> top((size_t)n * 10);
        VerifyIo io{claimed.data(), ncl.data(), g.data(), top.data()};
        ensure_prefill_bufs(c, n);
        BLK_CUDA(cudaStreamSynchronize(c->stream));
        c->profiling = true; c->prof_marks.clear();
        prof_mark(c, "start");
        prefill_chunk(c, tokens, n, &io, 0);
        c->profiling = false;
        prof_report(c, report, cap);
    });
}

extern "C" blk_status blk_debug_trace(blk_ctx* c, int64_t* out, int32_t cap, int32_t* n_cta, int32_t* per_cta) {
    if (!c || !out || !n_cta || !per_cta) return fail(BLK_ERR_ARG, "blk_debug_trace: bad arguments");
    return guarded([&] {
        if (!c->mega_on || !c->mega_params.trace) throw BlkError(BLK_ERR_ARG, "no trace: set BLK_MEGA_TRACE=1 before creating the context");
        BLK_CUDA(cudaSetDevice(c->m->device));
        BLK_CUDA(cudaStreamSynchronize(c->stream));
        const size_t n = (size_t)c->mega_params.n_cta * c->mega_params.trace_cap;
        if ((size_t)cap < n) throw BlkError(BLK_ERR_ARG, "blk_debug_trace: buffer too small");
        BLK_CUDA(cudaMemcpy(out, c->mega_params.trace, n * sizeof(long long), cudaMemcpyDeviceToHost));
        *n_cta = c->mega_params.n_cta; *per_cta = c->mega_params.trace_cap;
    });
}

extern "C" blk_status blk_flush_l2(blk_ctx* c) {
    return guarded([&] {
        BLK_CUDA(cudaSetDevice(c->m->device));
        if (!c->flush_buf) { c->flush_bytes = 256u << 20; BLK_CUDA(cudaMalloc(&c->flush_buf, c->flush_bytes)); c->allocs.push_back(c->flush_buf); }
        BLK_CUDA(cudaMemsetAsync(c->flush_buf, 0x5a, c->flush_bytes, c->stream));
    });
}

// ------------------------------------------------------------------------------------------------------------------
// unit-level entry points
// ------------------------------------------------------------------------------------------------------------------
namespace {
struct TestMat {
    blk_model holder;       // owns device allocations
    QMat W;
};
void test_upload(TestMat& tm, int device, int type, const void* blocks, int64_t rows, int64_t k) {
    if (blk_init() != BLK_OK) throw BlkError(BLK_ERR_NO_DEVICE, g_last_error);
    BLK_CUDA(cudaSetDevice(device));
    tm.holder.device = device;
    GgufTensor t; t.name = "test"; t.type = type; t.n_dims = 2; t.ne[0] = k; t.ne[1] = rows;
    int blck = 0, bytes = 0;
    if (!ggml_type_geometry(type, blck, bytes) || k % blck) throw BlkError(BLK_ERR_ARG, "bad type / row length");
    if (type != GT_F32 && type != GT_F16 && (k % 256) && type != GT_Q8_0) throw BlkError(BLK_ERR_ARG, "row length must be a multiple of 256");
    t.nbytes = (size_t)(k / blck) * bytes * (size_t)rows; t.data = (const uint8_t*)blocks;
    Uploader up; up.m = &tm.holder;
    BLK_CUDA(cudaStreamCreateWithFlags(&up.stream, cudaStreamNonBlocking));
    up.arena_bytes = Uploader::planes_bytes(t);
    BLK_CUDA(cudaMalloc(&up.arena, up.arena_bytes)); tm.holder.allocs.push_back(up.arena);
    BLK_CUDA(cudaMalloc(&up.staging, t.nbytes)); tm.holder.allocs.push_back(up.staging);
    tm.W = up.upload_matrix(t);
    BLK_CUDA(cudaStreamSynchronize(up.stream));
    cudaStreamDestroy(up.stream);
}
__global__ void test_dequant_kernel(QMat W, float* out) { dequant_row_cta(W, blockIdx.x, out + (size_t)blockIdx.x * W.K); }
} // namespace

extern "C" blk_status blk_test_dequant(int32_t device, int32_t type, const void* blocks, int64_t rows, int64_t k, float* out) {
    return guarded([&] {
        TestMat tm; test_upload(tm, device, type, blocks, rows, k);
        float* d_out = nullptr;
        BLK_CUDA(cudaMalloc(&d_out, (size_t)rows * k * 4)); tm.holder.allocs.push_back(d_out);
        test_dequant_kernel<<<(unsigned)rows, 128>>>(tm.W, d_out);
        BLK_CUDA(cudaGetLastError());
        BLK_CUDA(cudaMemcpy(out, d_out, (size_t)rows * k * 4, cudaMemcpyDeviceToHost));
    });
}

extern "C" blk_status blk_test_gemv(int32_t device, int32_t type, const void* blocks, int64_t rows, int64_t k, const float* x, float* y) {
    return guarded([&] {
        if (rows % 2) throw BlkError(BLK_ERR_ARG, "rows must be even");
        TestMat tm; test_upload(tm, device, type, blocks, rows, k);
        blk_ctx c; c.m = &tm.holder;
        ensure_kernel_attrs(device);
        BLK_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        float* d_x = dalloc<float>(&c, k); float* d_y = dalloc<float>(&c, rows);
        ActBuf act = make_act(&c, (int)k);
        BLK_CUDA(cudaMemcpyAsync(d_x, x, k * 4, cudaMemcpyHostToDevice, c.stream));
        GemvArgs a{};
        a.nseg = 1; a.seg[0] = {tm.W, nullptr, 0, 0}; a.total_pairs = (int)(rows / 2); a.out = d_y;
        matvec<EPI_STORE>(&c, a, d_x, nullptr, act, "test");
        BLK_CUDA(cudaMemcpyAsync(y, d_y, rows * 4, cudaMemcpyDeviceToHost, c.stream));
        BLK_CUDA(cudaStreamSynchronize(c.stream));
    });
}

extern "C" blk_status blk_test_gemm(int32_t device, int32_t type, const void* blocks, int64_t rows, int64_t k, const float* x, int64_t n_tok, float* y) {
    return guarded([&] {
        if (n_tok <= 0) throw BlkError(BLK_ERR_ARG, "n_tok must be positive");
        TestMat tm; test_upload(tm, device, type, blocks, rows, k);
        blk_ctx c; c.m = &tm.holder;
        BLK_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        float* d_x = dalloc<float>(&c, (size_t)n_tok * k);
        __nv_bfloat16* d_xb = dalloc<__nv_bfloat16>(&c, (size_t)n_tok * k);
        float* d_y = dalloc<float>(&c, (size_t)n_tok * rows);
        BLK_CUDA(cudaMemcpyAsync(d_x, x, (size_t)n_tok * k * 4, cudaMemcpyHostToDevice, c.stream));
        BLK_CUDA(convert_f32_to_bf16(d_x, d_xb, (size_t)n_tok * k, c.stream));
        __nv_bfloat16* panel = nullptr;        // BLK_TEST_PANEL=1: the two-pass form (dequantise to a bf16 panel, TMA-fed GEMM)
        const GemmPart part{&tm.W, nullptr, 0};
        { const char* tp = getenv("BLK_TEST_PANEL"); if (tp && tp[0] == '1' && type != GT_F32 && type != GT_F16) panel = dalloc<__nv_bfloat16>(&c, prefill_panel_elems(&part, 1, false)); }
        cudaError_t err = cudaSuccess;
        if (panel && !prefill_panel_fill(&part, 1, false, panel, c.stream, &err)) panel = nullptr;
        BLK_CUDA(err);
        BLK_CUDA(prefill_gemm(tm.W, d_xb, (int)n_tok, d_y, rows, nullptr, 0, c.stream, panel));
        BLK_CUDA(cudaMemcpyAsync(y, d_y, (size_t)n_tok * rows * 4, cudaMemcpyDeviceToHost, c.stream));
        BLK_CUDA(cudaStreamSynchronize(c.stream));
    });
}

extern "C" blk_status blk_bench_gemm(int32_t device, int32_t type, const void* blocks, int64_t rows, int64_t k, int64_t n_tok, int32_t iters, float* avg_ms) {
    return guarded([&] {
        if (n_tok <= 0 || iters <= 0 || !avg_ms) throw BlkError(BLK_ERR_ARG, "blk_bench_gemm: bad arguments");
        TestMat tm; test_upload(tm, device, type, blocks, rows, k);
        blk_ctx c; c.m = &tm.holder;
        BLK_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        BLK_CUDA(cudaEventCreate(&c.ev0)); BLK_CUDA(cudaEventCreate(&c.ev1));
        __nv_bfloat16* d_xb = dalloc<__nv_bfloat16>(&c, (size_t)n_tok * k);
        float* d_y = dalloc<float>(&c, (size_t)n_tok * rows);
        BLK_CUDA(cudaMemsetAsync(d_xb, 0x3c, (size_t)n_tok * k * 2, c.stream));
        __nv_bfloat16* panel = nullptr;        // BLK_TEST_PANEL=1: time the two-pass form (dequantisation pass included)
        const GemmPart part{&tm.W, nullptr, 0};
        { const char* tp = getenv("BLK_TEST_PANEL"); if (tp && tp[0] == '1') panel = dalloc<__nv_bfloat16>(&c, prefill_panel_elems(&part, 1, false)); }
        auto run = [&] {
            cudaError_t err = cudaSuccess;
            const bool filled = panel && prefill_panel_fill(&part, 1, false, panel, c.stream, &err);
            BLK_CUDA(err);
            BLK_CUDA(prefill_gemm(tm.W, d_xb, (int)n_tok, d_y, rows, nullptr, 0, c.stream, filled ? panel : nullptr));
        };
        for (int i = 0; i < 3; i++) run();
        BLK_CUDA(cudaEventRecord(c.ev0, c.stream));
        for (int i = 0; i < iters; i++) run();
        BLK_CUDA(cudaEventRecord(c.ev1, c.stream));
        BLK_CUDA(cudaEventSynchronize(c.ev1));
        float ms = 0.0f;
        BLK_CUDA(cudaEventElapsedTime(&ms, c.ev0, c.ev1));
        *avg_ms = ms / (float)iters;
    });
}

// ---- unit entry points of the non-GEMM prefill kernels (tests/test_gpu_prefill_units.py: float64 numpy on the rounded operands) ----
namespace {
struct Scratch {        // device allocations of one test call
    std::vector<void*> ptrs;
    template <class T> T* get(size_t n) { void* p = nullptr; BLK_CUDA(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T))); ptrs.push_back(p); return reinterpret_cast<T*>(p); }
    ~Scratch() { for (void* p : ptrs) cudaFree(p); }
};
__global__ void f32_to_f16_kernel(const float* x, __half* y, size_t n) { const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) y[i] = __float2half_rn(x[i]); }
__global__ void f16_to_f32_kernel(const __half* x, float* y, size_t n) { const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) y[i] = __half2float(x[i]); }
__global__ void bf16_to_f32_kernel(const __nv_bfloat16* x, float* y, size_t n) { const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) y[i] = __bfloat162float(x[i]); }
__global__ void rope_rows_kernel(float2* rope_cs, int half_rot, int pos0, float theta_scale, const float* ff) {
    rope_table_fill(rope_cs + (size_t)blockIdx.x * half_rot, half_rot, pos0 + (int)blockIdx.x, theta_scale, ff);
}
unsigned grid_of(size_t n) { return (unsigned)((n + 255) / 256); }
// rows [n][dkv] f32 -> f16 cache cells 0 .. n - 1 of a paged pool, through the page table
__global__ void scatter_cells_kernel(const float* x, __half* pool, const int32_t* page_table, int n, int dkv) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n * dkv) return;
    const int t = (int)(i / dkv), e = (int)(i % dkv);
    pool[((size_t)page_table[t / KV_PAGE] * KV_PAGE + (t % KV_PAGE)) * dkv + e] = __float2half_rn(x[i]);
}
// A page table of n_pages entries over a pool of about 1.5 times as many pages: the first n_pages of a seeded random permutation.
// Returns the pool size in pages.
int random_page_table(std::mt19937_64& rng, int n_pages, std::vector<int32_t>& pt) {
    const int pool_pages = n_pages + n_pages / 2 + 1;
    std::vector<int32_t> perm(pool_pages);
    for (int i = 0; i < pool_pages; i++) perm[i] = i;
    std::shuffle(perm.begin(), perm.end(), rng);
    pt.assign(perm.begin(), perm.begin() + n_pages);
    return pool_pages;
}
// Fill a pool with f16 NaN (0xffff), then write rows [n][dkv] into cells 0 .. n - 1 through the table: a read through the wrong
// page, of a cell past n, or of the wrong pool gives NaN.
void fill_pool(__half* pool, size_t pool_elems, const float* staging, const int32_t* d_pt, int n, int dkv, cudaStream_t st) {
    BLK_CUDA(cudaMemsetAsync(pool, 0xff, pool_elems * sizeof(__half), st));
    scatter_cells_kernel<<<grid_of((size_t)n * dkv), 256, 0, st>>>(staging, pool, d_pt, n, dkv);
    BLK_CUDA(cudaGetLastError());
}
} // namespace

// y[t][:] = bf16(rms_norm(x[t][:]) * w) through rmsnorm_bf16_kernel; out as f32 (exactly the bf16 values)
extern "C" blk_status blk_test_rmsnorm(int32_t device, const float* x, const float* w, int32_t T, int32_t K, float eps, float* out) {
    return guarded([&] {
        if (blk_init() != BLK_OK) throw BlkError(BLK_ERR_NO_DEVICE, g_last_error);
        if (T <= 0 || K <= 0 || K % 8 || K > 8192) throw BlkError(BLK_ERR_ARG, "blk_test_rmsnorm: bad shape");
        BLK_CUDA(cudaSetDevice(device));
        Scratch sc;
        float* dx = sc.get<float>((size_t)T * K); float* dw = sc.get<float>(K); float* dout = sc.get<float>((size_t)T * K);
        __nv_bfloat16* dy = sc.get<__nv_bfloat16>((size_t)T * K);
        BLK_CUDA(cudaMemcpy(dx, x, (size_t)T * K * 4, cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(dw, w, (size_t)K * 4, cudaMemcpyHostToDevice));
        rmsnorm_bf16_launch(dx, dw, K, eps, dy, T, nullptr);
        bf16_to_f32_kernel<<<grid_of((size_t)T * K), 256>>>(dy, dout, (size_t)T * K);
        BLK_CUDA(cudaGetLastError());
        BLK_CUDA(cudaMemcpy(out, dout, (size_t)T * K * 4, cudaMemcpyDeviceToHost));
    });
}

// qkv_post_kernel on T rows at positions pos0 .. : q_out [T][dq], k_out / v_out [T][dkv] (the f16 values as f32); freq_factors may be NULL
extern "C" blk_status blk_test_qkv_post(int32_t device, const float* qkv, int32_t T, int32_t n_head, int32_t n_head_kv, int32_t d_head, int32_t neox,
                                        int32_t pos0, float rope_theta, const float* freq_factors, float* q_out, float* k_out, float* v_out) {
    return guarded([&] {
        if (blk_init() != BLK_OK) throw BlkError(BLK_ERR_NO_DEVICE, g_last_error);
        if (T <= 0 || pos0 < 0 || (d_head != 64 && d_head != 128) || n_head <= 0 || n_head_kv <= 0) throw BlkError(BLK_ERR_ARG, "blk_test_qkv_post: bad shape");
        BLK_CUDA(cudaSetDevice(device));
        const int dq = n_head * d_head, dkv = n_head_kv * d_head, ld = dq + 2 * dkv, half = d_head / 2;
        const int n_pages = (pos0 + T + KV_PAGE - 1) / KV_PAGE;
        Scratch sc;
        float* dqkv = sc.get<float>((size_t)T * ld);
        float2* rope = sc.get<float2>((size_t)T * half);
        float* dff = freq_factors ? sc.get<float>(half) : nullptr;
        __half* dq16 = sc.get<__half>((size_t)T * dq);
        __half* kp = sc.get<__half>((size_t)n_pages * KV_PAGE * dkv); __half* vp = sc.get<__half>((size_t)n_pages * KV_PAGE * dkv);
        int32_t* pt = sc.get<int32_t>(n_pages); int32_t* dpos = sc.get<int32_t>(2);
        float* fq = sc.get<float>((size_t)T * dq); float* fk = sc.get<float>((size_t)T * dkv); float* fv = sc.get<float>((size_t)T * dkv);
        // a REVERSED page table: the kernel must go through it
        std::vector<int32_t> hpt(n_pages);
        for (int i = 0; i < n_pages; i++) hpt[i] = n_pages - 1 - i;
        const int32_t hpos[2] = {pos0, 0};
        BLK_CUDA(cudaMemcpy(dqkv, qkv, (size_t)T * ld * 4, cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(pt, hpt.data(), (size_t)n_pages * 4, cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(dpos, hpos, sizeof(hpos), cudaMemcpyHostToDevice));
        if (dff) BLK_CUDA(cudaMemcpy(dff, freq_factors, (size_t)half * 4, cudaMemcpyHostToDevice));
        rope_rows_kernel<<<T, 64>>>(rope, half, pos0, powf(rope_theta, -2.0f / (float)d_head), dff);
        QkvPostArgs qa{};
        qa.qkv = dqkv; qa.ld = ld; qa.rope_cs = rope; qa.pos0 = dpos; qa.q_out = dq16; qa.k_pool = kp; qa.v_pool = vp; qa.page_table = pt;
        qa.dq = dq; qa.dkv = dkv; qa.d_head = d_head; qa.neox = neox ? 1 : 0;
        qkv_post_kernel<<<T, 256>>>(qa);
        BLK_CUDA(cudaGetLastError());
        f16_to_f32_kernel<<<grid_of((size_t)T * dq), 256>>>(dq16, fq, (size_t)T * dq);
        BLK_CUDA(cudaMemcpy(q_out, fq, (size_t)T * dq * 4, cudaMemcpyDeviceToHost));
        for (int t = 0; t < T; t++) {        // rows come back through the same page table
            const int pos = pos0 + t;
            const size_t row = ((size_t)hpt[pos / KV_PAGE] * KV_PAGE + (pos % KV_PAGE)) * dkv;
            f16_to_f32_kernel<<<grid_of(dkv), 256>>>(kp + row, fk + (size_t)t * dkv, dkv);
            f16_to_f32_kernel<<<grid_of(dkv), 256>>>(vp + row, fv + (size_t)t * dkv, dkv);
        }
        BLK_CUDA(cudaGetLastError());
        BLK_CUDA(cudaMemcpy(k_out, fk, (size_t)T * dkv * 4, cudaMemcpyDeviceToHost));
        BLK_CUDA(cudaMemcpy(v_out, fv, (size_t)T * dkv * 4, cudaMemcpyDeviceToHost));
    });
}

// Causal prefill attention of T query rows at positions pos0 .. over a cache of pos0 + T keys: q [T][n_head*dh], k / v [pos0+T][n_head_kv*dh]
// (rounded to f16 on the way in, like the cache); out [T][n_head*dh] = the kernel's bf16 output as f32.  *used_tc = 1 when the tcgen05
// kernel ran (d_head 128), 0 for the mma.sync kernels (d_head 64).  A d_head 128 shape the tcgen05 kernel does not cover is BLK_ERR_ARG.
extern "C" blk_status blk_test_prefill_attn(int32_t device, const float* q, const float* k, const float* v, int32_t T, int32_t pos0, int32_t n_head,
                                            int32_t n_head_kv, int32_t d_head, float* out, int32_t* used_tc) {
    return guarded([&] {
        if (blk_init() != BLK_OK) throw BlkError(BLK_ERR_NO_DEVICE, g_last_error);
        if (T <= 0 || pos0 < 0 || (d_head != 64 && d_head != 128) || n_head <= 0 || n_head_kv <= 0 || n_head % n_head_kv) throw BlkError(BLK_ERR_ARG, "blk_test_prefill_attn: bad shape");
        if (d_head == 128 && !prefill_attn_tc_supported(d_head, n_head, n_head_kv)) throw BlkError(BLK_ERR_ARG, "blk_test_prefill_attn: no kernel for this shape");
        BLK_CUDA(cudaSetDevice(device));
        const int dq = n_head * d_head, dkv = n_head_kv * d_head, n_keys = pos0 + T;
        blk_model mm; mm.device = device; mm.n_head = n_head; mm.n_head_kv = n_head_kv; mm.d_head = d_head;
        blk_ctx c; c.m = &mm;
        BLK_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        c.n_pages = (n_keys + KV_PAGE - 1) / KV_PAGE; c.n_past = pos0;
        const size_t pool = (size_t)c.n_pages * KV_PAGE * dkv;
        float* fq = dalloc<float>(&c, (size_t)T * dq); float* fkv = dalloc<float>(&c, (size_t)n_keys * dkv);
        __half* q16 = dalloc<__half>(&c, (size_t)T * dq); __half* kp = dalloc<__half>(&c, pool); __half* vp = dalloc<__half>(&c, pool);
        __nv_bfloat16* o = dalloc<__nv_bfloat16>(&c, (size_t)T * dq); float* fo = dalloc<float>(&c, (size_t)T * dq);
        c.page_table = dalloc<int32_t>(&c, c.n_pages); c.d_pos = dalloc<int32_t>(&c, 2);
        std::vector<int32_t> hpt(c.n_pages);
        for (int i = 0; i < c.n_pages; i++) hpt[i] = i;
        const int32_t hpos[2] = {pos0, 0};
        BLK_CUDA(cudaMemcpyAsync(c.page_table, hpt.data(), (size_t)c.n_pages * 4, cudaMemcpyHostToDevice, c.stream));
        BLK_CUDA(cudaMemcpyAsync(c.d_pos, hpos, sizeof(hpos), cudaMemcpyHostToDevice, c.stream));
        BLK_CUDA(cudaMemsetAsync(kp, 0, pool * 2, c.stream)); BLK_CUDA(cudaMemsetAsync(vp, 0, pool * 2, c.stream));
        BLK_CUDA(cudaMemcpyAsync(fq, q, (size_t)T * dq * 4, cudaMemcpyHostToDevice, c.stream));
        f32_to_f16_kernel<<<grid_of((size_t)T * dq), 256, 0, c.stream>>>(fq, q16, (size_t)T * dq);
        BLK_CUDA(cudaMemcpyAsync(fkv, k, (size_t)n_keys * dkv * 4, cudaMemcpyHostToDevice, c.stream));
        f32_to_f16_kernel<<<grid_of((size_t)n_keys * dkv), 256, 0, c.stream>>>(fkv, kp, (size_t)n_keys * dkv);
        BLK_CUDA(cudaStreamSynchronize(c.stream));
        BLK_CUDA(cudaMemcpyAsync(fkv, v, (size_t)n_keys * dkv * 4, cudaMemcpyHostToDevice, c.stream));
        f32_to_f16_kernel<<<grid_of((size_t)n_keys * dkv), 256, 0, c.stream>>>(fkv, vp, (size_t)n_keys * dkv);
        const bool tc = d_head == 128;
        if (tc) { c.pf_vt_pad = (c.n_pages * KV_PAGE + 127) / 128 * 128; c.pf_vt = dalloc<__half>(&c, (size_t)n_head_kv * 128 * c.pf_vt_pad); }
        BLK_CUDA(cudaFuncSetAttribute(prefill_attn_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * 64 * (64 + 8) * 2));
        PrefillAttnArgs pa{};
        pa.q = q16; pa.k_pool = kp; pa.v_pool = vp; pa.page_table = c.page_table; pa.pos0 = c.d_pos; pa.out = o; pa.T = T;
        pa.n_head = n_head; pa.n_head_kv = n_head_kv; pa.kv_dim = dkv; pa.scale = 1.0f / sqrtf((float)d_head);
        launch_prefill_attn(&c, pa, T, c.stream);
        bf16_to_f32_kernel<<<grid_of((size_t)T * dq), 256, 0, c.stream>>>(o, fo, (size_t)T * dq);
        BLK_CUDA(cudaGetLastError());
        BLK_CUDA(cudaMemcpyAsync(out, fo, (size_t)T * dq * 4, cudaMemcpyDeviceToHost, c.stream));
        BLK_CUDA(cudaStreamSynchronize(c.stream));
        if (used_tc) *used_tc = tc ? 1 : 0;
    });
}

// Decode attention of one query row q [n_head*dh] (f32, the kernels round it to f16) over the cache cells 0 .. n_kv - 1 of a context of
// n_ctx cells, through plan_decode_attn / launch_decode_attn: k / v [n_kv][n_head_kv*dh] are rounded to f16 into a NaN-filled pool
// behind a seeded random page table.  form: -1 = the plan's choice, 0 / 1 = force the split / cluster form (BLK_ERR_ARG, without a
// launch, when the plan does not allow the cluster form).  out [n_head*dh] f32; *used_form = 1 when the cluster form ran.
extern "C" blk_status blk_test_decode_attn(int32_t device, const float* q, const float* k, const float* v, int32_t n_kv, int32_t n_ctx,
                                           int32_t n_head, int32_t n_head_kv, int32_t d_head, int32_t form, int64_t seed, float* out,
                                           int32_t* used_form) {
    return guarded([&] {
        if (blk_init() != BLK_OK) throw BlkError(BLK_ERR_NO_DEVICE, g_last_error);
        if (n_kv <= 0 || n_ctx < n_kv || (d_head != 64 && d_head != 128) || n_head <= 0 || n_head_kv <= 0 || n_head % n_head_kv ||
            n_head / n_head_kv > MAX_GQ || form < -1 || form > 1)
            throw BlkError(BLK_ERR_ARG, "blk_test_decode_attn: bad shape");
        BLK_CUDA(cudaSetDevice(device));
        const int dq = n_head * d_head, dkv = n_head_kv * d_head;
        const int dq_pad = (dq + 255) / 256 * 256;          // attn_combine_kernel writes whole 256-output blocks
        blk_model mm; mm.device = device; mm.n_head = n_head; mm.n_head_kv = n_head_kv; mm.d_head = d_head;
        blk_ctx c; c.m = &mm;
        c.n_ctx = n_ctx; c.n_pages = (n_ctx + KV_PAGE - 1) / KV_PAGE;
        plan_decode_attn(&c, form);
        BLK_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        std::mt19937_64 rng((uint64_t)seed);
        std::vector<int32_t> hpt;
        const int pool_pages = random_page_table(rng, c.n_pages, hpt);
        const size_t pool = (size_t)pool_pages * KV_PAGE * dkv;
        c.k_pool = {dalloc<__half>(&c, pool)}; c.v_pool = {dalloc<__half>(&c, pool)};
        c.page_table = dalloc<int32_t>(&c, c.n_pages); c.d_pos = dalloc<int32_t>(&c, 2);
        c.qbuf = dalloc<float>(&c, dq); c.act_q.f32 = dalloc<float>(&c, dq_pad);
        c.part_o = dalloc<float>(&c, (size_t)dq_pad * c.n_split);
        BLK_CUDA(cudaMemsetAsync(c.part_o, 0, (size_t)dq_pad * c.n_split * 4, c.stream));
        c.scores = dalloc<float>(&c, (size_t)n_head * c.n_pages * KV_PAGE);
        float* staging = dalloc<float>(&c, (size_t)n_kv * dkv);
        const int32_t hpos[2] = {n_kv - 1, 0};
        BLK_CUDA(cudaMemcpyAsync(c.page_table, hpt.data(), (size_t)c.n_pages * 4, cudaMemcpyHostToDevice, c.stream));
        BLK_CUDA(cudaMemcpyAsync(c.d_pos, hpos, sizeof(hpos), cudaMemcpyHostToDevice, c.stream));
        BLK_CUDA(cudaMemcpyAsync(c.qbuf, q, (size_t)dq * 4, cudaMemcpyHostToDevice, c.stream));
        BLK_CUDA(cudaMemcpyAsync(staging, k, (size_t)n_kv * dkv * 4, cudaMemcpyHostToDevice, c.stream));
        fill_pool(c.k_pool[0], pool, staging, c.page_table, n_kv, dkv, c.stream);
        BLK_CUDA(cudaMemcpyAsync(staging, v, (size_t)n_kv * dkv * 4, cudaMemcpyHostToDevice, c.stream));
        fill_pool(c.v_pool[0], pool, staging, c.page_table, n_kv, dkv, c.stream);
        BLK_CUDA(cudaMemsetAsync(c.act_q.f32, 0xff, (size_t)dq * 4, c.stream));
        launch_decode_attn(&c, 0);
        BLK_CUDA(cudaGetLastError());
        BLK_CUDA(cudaMemcpyAsync(out, c.act_q.f32, (size_t)dq * 4, cudaMemcpyDeviceToHost, c.stream));
        BLK_CUDA(cudaStreamSynchronize(c.stream));
        if (used_form) *used_form = c.attn_cluster > 0 ? 1 : 0;
    });
}

// decode_attn_batch_kernel over n <= BATCH_MAX rows in one launch: row b attends with q [b][n_head*dh] (rounded to f16 like the batch
// step's q) over its own n_kv[b] cells; k / v hold the rows' keys / values one after another ([sum n_kv][n_head_kv*dh], rounded to
// f16).  Every row has its own seeded random page table and two-layer K / V pools, all NaN except the cells 0 .. n_kv[b] - 1 of
// layer 1, which the kernel reads.  out [n][n_head*dh] = the kernel's bf16 output as f32.
extern "C" blk_status blk_test_decode_attn_batch(int32_t device, int32_t n, const float* q, const float* k, const float* v, const int32_t* n_kv,
                                                 int32_t n_head, int32_t n_head_kv, int32_t d_head, int64_t seed, float* out) {
    return guarded([&] {
        if (blk_init() != BLK_OK) throw BlkError(BLK_ERR_NO_DEVICE, g_last_error);
        if (n <= 0 || n > BATCH_MAX || !n_kv || (d_head != 64 && d_head != 128) || n_head <= 0 || n_head_kv <= 0 || n_head % n_head_kv ||
            n_head / n_head_kv > MAX_GQ)
            throw BlkError(BLK_ERR_ARG, "blk_test_decode_attn_batch: bad shape");
        for (int b = 0; b < n; b++) if (n_kv[b] <= 0) throw BlkError(BLK_ERR_ARG, "blk_test_decode_attn_batch: bad n_kv");
        BLK_CUDA(cudaSetDevice(device));
        constexpr int N_LAYER = 2, LAYER = 1;
        const int dq = n_head * d_head, dkv = n_head_kv * d_head;
        std::mt19937_64 rng((uint64_t)seed);
        // per row: its page table, its pool size in pages, where both start, where its keys start
        std::vector<int32_t> pt_all, pos(n);
        std::vector<size_t> pt_off(n), page_off(n), row_off(n);
        size_t total_pages = 0, total_rows = 0;
        for (int b = 0; b < n; b++) {
            std::vector<int32_t> pt;
            const int pool_pages = random_page_table(rng, (n_kv[b] + KV_PAGE - 1) / KV_PAGE, pt);
            pt_off[b] = pt_all.size(); page_off[b] = total_pages; row_off[b] = total_rows;
            pt_all.insert(pt_all.end(), pt.begin(), pt.end());
            total_pages += pool_pages; total_rows += n_kv[b]; pos[b] = n_kv[b] - 1;
        }
        const size_t layer_elems = total_pages * KV_PAGE * dkv;
        Scratch sc;
        __half* kar = sc.get<__half>(N_LAYER * layer_elems); __half* var = sc.get<__half>(N_LAYER * layer_elems);
        int32_t* d_pt = sc.get<int32_t>(pt_all.size()); int32_t* d_pos = sc.get<int32_t>(n);
        float* staging = sc.get<float>(std::max(total_rows * dkv, (size_t)n * dq));
        __half* q16 = sc.get<__half>((size_t)n * dq);
        __nv_bfloat16* o = sc.get<__nv_bfloat16>((size_t)n * dq); float* fo = sc.get<float>((size_t)n * dq);
        // device pointer tables: [b] -> page table, [b] -> [layer] -> pool
        std::vector<const int32_t*> h_pts(n);
        std::vector<__half*> h_kl((size_t)n * N_LAYER), h_vl((size_t)n * N_LAYER);
        const int32_t** d_pts = sc.get<const int32_t*>(n);
        __half** d_kl = sc.get<__half*>((size_t)n * N_LAYER); __half** d_vl = sc.get<__half*>((size_t)n * N_LAYER);
        std::vector<__half* const*> h_kp(n), h_vp(n);
        __half* const** d_kp = sc.get<__half* const*>(n); __half* const** d_vp = sc.get<__half* const*>(n);
        for (int b = 0; b < n; b++) {
            h_pts[b] = d_pt + pt_off[b];
            for (int l = 0; l < N_LAYER; l++) {
                h_kl[(size_t)b * N_LAYER + l] = kar + l * layer_elems + page_off[b] * KV_PAGE * dkv;
                h_vl[(size_t)b * N_LAYER + l] = var + l * layer_elems + page_off[b] * KV_PAGE * dkv;
            }
            h_kp[b] = d_kl + (size_t)b * N_LAYER; h_vp[b] = d_vl + (size_t)b * N_LAYER;
        }
        BLK_CUDA(cudaMemcpy(d_pt, pt_all.data(), pt_all.size() * 4, cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(d_pos, pos.data(), (size_t)n * 4, cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(d_pts, h_pts.data(), (size_t)n * sizeof(void*), cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(d_kl, h_kl.data(), h_kl.size() * sizeof(void*), cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(d_vl, h_vl.data(), h_vl.size() * sizeof(void*), cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(d_kp, h_kp.data(), (size_t)n * sizeof(void*), cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemcpy(d_vp, h_vp.data(), (size_t)n * sizeof(void*), cudaMemcpyHostToDevice));
        BLK_CUDA(cudaMemset(kar, 0xff, N_LAYER * layer_elems * sizeof(__half)));
        BLK_CUDA(cudaMemset(var, 0xff, N_LAYER * layer_elems * sizeof(__half)));
        for (int kv = 0; kv < 2; kv++) {
            BLK_CUDA(cudaMemcpy(staging, kv ? v : k, total_rows * dkv * 4, cudaMemcpyHostToDevice));
            for (int b = 0; b < n; b++)
                scatter_cells_kernel<<<grid_of((size_t)n_kv[b] * dkv), 256>>>(staging + row_off[b] * dkv, (kv ? h_vl : h_kl)[(size_t)b * N_LAYER + LAYER],
                                                                             d_pt + pt_off[b], n_kv[b], dkv);
            BLK_CUDA(cudaGetLastError());
            BLK_CUDA(cudaDeviceSynchronize());
        }
        BLK_CUDA(cudaMemcpy(staging, q, (size_t)n * dq * 4, cudaMemcpyHostToDevice));
        f32_to_f16_kernel<<<grid_of((size_t)n * dq), 256>>>(staging, q16, (size_t)n * dq);
        BLK_CUDA(cudaMemset(o, 0xff, (size_t)n * dq * sizeof(__nv_bfloat16)));
        BatchAttnArgs aa{};
        aa.q = q16; aa.pos = d_pos; aa.page_table = d_pts; aa.k_pools = d_kp; aa.v_pools = d_vp; aa.out = o;
        aa.layer = LAYER; aa.n_head = n_head; aa.n_head_kv = n_head_kv; aa.kv_dim = dkv; aa.scale = 1.0f / sqrtf((float)d_head);
        if (d_head == 128) decode_attn_batch_kernel<128><<<dim3(n_head_kv, n), 256>>>(aa);
        else decode_attn_batch_kernel<64><<<dim3(n_head_kv, n), 256>>>(aa);
        BLK_CUDA(cudaGetLastError());
        bf16_to_f32_kernel<<<grid_of((size_t)n * dq), 256>>>(o, fo, (size_t)n * dq);
        BLK_CUDA(cudaGetLastError());
        BLK_CUDA(cudaMemcpy(out, fo, (size_t)n * dq * 4, cudaMemcpyDeviceToHost));
    });
}
