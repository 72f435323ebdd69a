// host_capi.cpp -- C entry points over the bl::llama host classes so that tests (ctypes) and foreign callers can drive
// the reference-shaped API: Model / Instance / Session / LogitComparer / MetricsAggregator / Sampler.
// Every function returns 0 on success, 1 when the C++ layer threw; blh_last_error() then holds e.what() -- the same
// strings the reference's tests pin (inference/test/t-integration.cpp:137-217).
#include "llama/Errors.hpp"
#include "llama/Init.hpp"
#include "llama/Instance.hpp"
#include "llama/LogitComparer.hpp"
#include "llama/Model.hpp"
#include "llama/Sampler.hpp"
#include "llama/Session.hpp"
#include "server/Http.hpp"
#include "server/Json.hpp"
#include "server/Server.hpp"
#include "server/Wire.hpp"

#include <blama_b200.h>

#include <condition_variable>
#include <cstring>
#include <map>
#include <mutex>
#include <string>

using namespace bl::llama;
namespace json = bl::json;

namespace {
thread_local std::string g_err;
template <class F> int guard(F&& f) {
    try { f(); return 0; }
    catch (const std::exception& e) { g_err = e.what(); return 1; }
    catch (...) { g_err = "unknown error"; return 1; }
}
struct InstanceBox {
    std::unique_ptr<Instance> inst;
    Session* session = nullptr;
};
TokenDataVector toVec(const blk_token_data* p, int32_t n) {
    TokenDataVector v(static_cast<size_t>(n));
    for (int32_t i = 0; i < n; ++i) v[size_t(i)] = {p[i].token, p[i].logit};
    return v;
}
// claimed lists arrive as [n][10] blocks: the count of every position must lie in 0..10 (prover-controlled input)
TokenDataVector claimedVec(const blk_token_data* block, int32_t n_claimed) {
    if (n_claimed < 0 || n_claimed > 10) Raise{} << "n_claimed must be in 0..10, got " << n_claimed;
    return toVec(block, n_claimed);
}

// ---- Server over the C boundary: asynchronous submit -> ticket -> wait ----------------------------------------------------
struct Ticket {
    bool done = false;
    server::Server::CompleteReponse response;
    float score = 0.0f;
};
struct ServerBox {
    std::unique_ptr<server::Server> srv;
    std::unique_ptr<server::HttpFrontEnd> http;
    std::mutex mu;
    std::condition_variable cv;
    std::map<int64_t, std::shared_ptr<Ticket>> tickets;
    int64_t next = 1;
    std::string lastWorkerError;

    std::pair<int64_t, std::shared_ptr<Ticket>> open() {
        std::lock_guard<std::mutex> lk(mu);
        auto t = std::make_shared<Ticket>();
        const int64_t id = next++;
        tickets[id] = t;
        return {id, t};
    }
    void finish(const std::shared_ptr<Ticket>& t) {
        { std::lock_guard<std::mutex> lk(mu); t->done = true; }
        cv.notify_all();
    }
    std::shared_ptr<Ticket> wait(int64_t id) {
        std::unique_lock<std::mutex> lk(mu);
        auto it = tickets.find(id);
        if (it == tickets.end()) Raise{} << "unknown ticket " << id;
        auto t = it->second;
        cv.wait(lk, [&] { return t->done; });
        tickets.erase(id);
        return t;
    }
};
server::Server::CompleteReponse responseOf(const int32_t* toks, int n, const blk_token_data* claimed, const int32_t* n_claimed) {
    server::Server::CompleteReponse resp(static_cast<size_t>(n));
    for (int t = 0; t < n; ++t) {
        if (n_claimed[t] < 0 || n_claimed[t] > 10) Raise{} << "n_claimed must be in 0..10, got " << n_claimed[t];
        resp[size_t(t)].tokenId = uint32_t(toks[t]);
        for (int j = 0; j < n_claimed[t]; ++j) resp[size_t(t)].logits.push_back({uint32_t(claimed[size_t(t) * 10 + size_t(j)].token), claimed[size_t(t) * 10 + size_t(j)].logit});
    }
    return resp;
}
// the logit-bias and repetition-penalty stages of a Sampler::Params from C arrays
void setStages(Sampler::Params& sp, int32_t last_n, float repeat, float freq, float present, const int32_t* bias_ids, const float* bias_vals, int n_bias) {
    sp.repetitionPenalty = {last_n, repeat, freq, present};
    for (int i = 0; i < n_bias; ++i) sp.logitBias[bias_ids[i]] = bias_vals[i];
}
void writeEdits(const Sampler::LogitEdits& e, blk_logit_edit* out, int cap, int32_t* n, float* out3) {
    *n = int32_t(e.edits.size());
    for (size_t j = 0; j < e.edits.size() && int(j) < cap; ++j) out[j] = {e.edits[j].token, e.edits[j].count, e.edits[j].bias};
    out3[0] = e.repeat; out3[1] = e.freq; out3[2] = e.present;
}
} // namespace

extern "C" {

BLK_API const char* blh_last_error(void) { return g_err.c_str(); }
BLK_API void blh_init(void) { initLibrary(); }

BLK_API int blh_model_create(const char* path, int device, int gpu, int prefix_bos, void** out) {
    return guard([&] {
        Model::Params p; p.gpu = gpu != 0; p.device = device; p.prefixInputsWithBos = prefix_bos != 0;
        *out = new Model(path, p);
    });
}
// Model::Params::vocabOnly: tokenizer / detokenizer only, no device needed
BLK_API int blh_model_create_vocab_only(const char* path, void** out) {
    return guard([&] { Model::Params p; p.vocabOnly = true; *out = new Model(path, p); });
}
BLK_API void blh_model_free(void* m) { delete static_cast<Model*>(m); }
BLK_API int blh_model_train_ctx(void* m) { return int(static_cast<Model*>(m)->trainCtxLength()); }
// Vocab::tokenize over n_bytes of text (may contain NULs); returns the token count (may exceed cap), -1 on failure
BLK_API int blh_model_tokenize(void* m, const char* text, int n_bytes, int add_special, int parse_special, int32_t* out, int cap) {
    int n = -1;
    guard([&] {
        auto v = static_cast<Model*>(m)->vocab().tokenize(std::string_view(text, size_t(n_bytes)), add_special != 0, parse_special != 0);
        for (int i = 0; i < int(v.size()) && i < cap; ++i) out[i] = v[size_t(i)];
        n = int(v.size());
    });
    return n;
}
BLK_API int blh_model_token_to_string(void* m, int32_t tok, int special, char* buf, int cap) {
    int n = -1;
    guard([&] {
        auto s = static_cast<Model*>(m)->vocab().tokenToString(tok, special != 0);
        n = int(s.size());
        memcpy(buf, s.data(), size_t(n < cap ? n : cap));
    });
    return n;
}
BLK_API int blh_model_is_eog(void* m, int32_t tok) { return static_cast<Model*>(m)->vocab().isEog(tok) ? 1 : 0; }

BLK_API int blh_instance_create(void* model, uint32_t ctx_size, uint32_t batch_size, void** out) {
    return guard([&] {
        auto box = std::make_unique<InstanceBox>();
        Instance::InitParams ip; ip.ctxSize = ctx_size; if (batch_size) ip.batchSize = batch_size;
        box->inst = std::make_unique<Instance>(*static_cast<Model*>(model), ip);
        *out = box.release();
    });
}
BLK_API void blh_instance_free(void* i) { delete static_cast<InstanceBox*>(i); }
// the C-ABI context behind an Instance (bench.py times it with blk_timer_* / counts its launches)
BLK_API void* blh_instance_ctx(void* i) { return static_cast<InstanceBox*>(i)->inst->lctx(); }
BLK_API int blh_instance_warmup(void* i) { return guard([&] { static_cast<InstanceBox*>(i)->inst->warmup(); }); }

BLK_API int blh_session_start(void* i, uint32_t seed, float temp, float top_p, int sequential_verify) {
    return guard([&] {
        auto* box = static_cast<InstanceBox*>(i);
        Session::InitParams sp; sp.seed = seed; sp.temperature = temp; sp.topP = top_p; sp.sequentialVerify = sequential_verify != 0;
        box->session = &box->inst->startSession(sp);
    });
}
BLK_API void blh_session_stop(void* i) { auto* box = static_cast<InstanceBox*>(i); box->inst->stopSession(); box->session = nullptr; }
BLK_API int blh_session_set_initial_prompt(void* i, const int32_t* toks, int n) {
    return guard([&] { static_cast<InstanceBox*>(i)->session->setInitialPrompt({toks, size_t(n)}); });
}
// out_top10: [max_tokens][10]; out_n_logits[i] = number of valid logits for token i; *out_n = tokens produced
BLK_API int blh_session_complete(void* i, const int32_t* prompt, int n_prompt, int max_tokens, int32_t* out_tokens,
                                 blk_token_data* out_top10, int32_t* out_n_logits, int32_t* out_n) {
    return guard([&] {
        auto preds = static_cast<InstanceBox*>(i)->session->complete({.prompt = {prompt, size_t(n_prompt)}, .suffix = {}, .maxTokens = max_tokens});
        *out_n = int32_t(preds.size());
        for (size_t t = 0; t < preds.size(); ++t) {
            out_tokens[t] = preds[t].token;
            out_n_logits[t] = int32_t(preds[t].logits.size());
            for (size_t j = 0; j < preds[t].logits.size() && j < 10; ++j) out_top10[t * 10 + j] = {preds[t].logits[j].token, preds[t].logits[j].logit};
        }
    });
}
BLK_API int blh_session_stream(void* i, int max_tokens, int32_t* out_tokens, int32_t* out_n) {
    return guard([&] {
        auto gen = static_cast<InstanceBox*>(i)->session->completeStream({.prompt = {}, .suffix = {}, .maxTokens = max_tokens});
        int n = 0;
        while (gen.status() == Session::StreamGenerator::Status::InProgress) {
            auto p = gen.complete();
            if (!p) break;
            out_tokens[n++] = p.token;
        }
        *out_n = n;
    });
}
BLK_API int blh_session_fill_ctx(void* i, const int32_t* toks, int n, const blk_token_data* claimed /*[n][10]*/, const int32_t* n_claimed,
                                 blk_token_data* out /*[n][10]*/, int32_t* out_n) {
    return guard([&] {
        std::vector<TokenPrediction> in(static_cast<size_t>(n));
        for (int t = 0; t < n; ++t) { in[size_t(t)].token = toks[t]; in[size_t(t)].logits = claimedVec(claimed + size_t(t) * 10, n_claimed[t]); }
        auto res = static_cast<InstanceBox*>(i)->session->fillCtx(in);
        for (size_t t = 0; t < res.size(); ++t) {
            out_n[t] = int32_t(res[t].logits.size());
            for (size_t j = 0; j < res[t].logits.size() && j < 10; ++j) out[t * 10 + j] = {res[t].logits[j].token, res[t].logits[j].logit};
        }
    });
}
// Server::verify in one call (reference Server.cpp:127-161 after tokenisation): fillCtx + LogitComparer over every position
BLK_API int blh_session_verify(void* i, const int32_t* toks, int n, const blk_token_data* claimed /*[n][10]*/, const int32_t* n_claimed, float* score) {
    return guard([&] {
        std::vector<TokenPrediction> orig(static_cast<size_t>(n));
        for (int t = 0; t < n; ++t) { orig[size_t(t)].token = toks[t]; orig[size_t(t)].logits = claimedVec(claimed + size_t(t) * 10, n_claimed[t]); }
        auto mine = static_cast<InstanceBox*>(i)->session->fillCtx(orig);
        // The reference pushes the metrics one by one and re-sums its whole history on every push (Server.cpp:153-156, O(n^2));
        // only the value of the LAST push is returned, and that is the in-order double sum over all metrics: one push of the
        // whole span computes exactly that float.
        std::vector<TokenPredictionView> pairs(orig.size());
        for (size_t t = 0; t < orig.size(); ++t) pairs[t] = {&orig[t].logits, &mine[t].logits};
        const std::vector<ComparisonMetrics> ms = compareAll(pairs);
        MetricsAggregator agg;
        *score = ms.empty() ? 0.0f : agg.pushAndVerify(ms);
    });
}
// Session::getState into buf (cap bytes); *size = bytes of the state (call with cap 0 to learn it -- the state is then dropped)
BLK_API int blh_session_get_state(void* i, uint8_t* buf, int64_t cap, int64_t* size) {
    return guard([&] {
        auto st = static_cast<InstanceBox*>(i)->session->getState();
        *size = int64_t(st.size());
        if (buf && cap >= int64_t(st.size())) memcpy(buf, st.data(), st.size());
    });
}
BLK_API int blh_session_set_state(void* i, uint8_t* buf, int64_t size) {
    return guard([&] { (void)static_cast<InstanceBox*>(i)->session->setState({buf, size_t(size < 0 ? 0 : size)}); });
}
// Self-Extend session (Session::InitParams::gaFactor / gaWidth)
BLK_API int blh_session_start_ga(void* i, uint32_t seed, float temp, float top_p, uint32_t ga_factor, uint32_t ga_width) {
    return guard([&] {
        auto* box = static_cast<InstanceBox*>(i);
        Session::InitParams sp; sp.seed = seed; sp.temperature = temp; sp.topP = top_p; sp.gaFactor = ga_factor; sp.gaWidth = ga_width;
        box->session = &box->inst->startSession(sp);
    });
}
BLK_API int blh_session_start_ex(void* i, uint32_t seed, float temp, float top_p, int sequential_verify, int infinite_context) {
    return guard([&] {
        auto* box = static_cast<InstanceBox*>(i);
        Session::InitParams sp; sp.seed = seed; sp.temperature = temp; sp.topP = top_p; sp.sequentialVerify = sequential_verify != 0;
        sp.infiniteContext = infinite_context != 0;
        box->session = &box->inst->startSession(sp);
    });
}

// Session::resetSampler with the reference's chain plus logit bias / repetition penalties (bias_ids / bias_vals: n_bias map entries)
BLK_API int blh_session_reset_sampler(void* i, uint32_t seed, float temp, float top_p, int32_t last_n, float repeat, float freq, float present,
                                      const int32_t* bias_ids, const float* bias_vals, int n_bias) {
    return guard([&] {
        Sampler::Params sp; sp.rngSeed = seed; sp.temp = temp; sp.topP = top_p;
        setStages(sp, last_n, repeat, freq, present, bias_ids, bias_vals, n_bias);
        static_cast<InstanceBox*>(i)->session->resetSampler(sp);
    });
}
// the session sampler's current edit list (Session::logitEdits): *n entries (at most cap written), out3 = repeat, freq, present
BLK_API int blh_session_logit_edits(void* i, blk_logit_edit* out, int cap, int32_t* n, float* out3) {
    return guard([&] { writeEdits(static_cast<InstanceBox*>(i)->session->logitEdits(), out, cap, n, out3); });
}
// Session::samplingCandidates: *n entries, at most cap written
BLK_API int blh_session_candidates(void* i, blk_token_data* out, int cap, int32_t* n) {
    return guard([&] {
        const auto c = static_cast<InstanceBox*>(i)->session->samplingCandidates();
        *n = int32_t(c.size());
        for (size_t j = 0; j < c.size() && int(j) < cap; ++j) out[j] = {c[j].token, c[j].logit};
    });
}

// ---- verdict -------------------------------------------------------------------------------------------------------
BLK_API void blh_lc_compare(const blk_token_data* a, int32_t na, const blk_token_data* b, int32_t nb, float* out3) {
    auto m = compareChecked(toVec(a, na < 0 ? 0 : na), toVec(b, nb < 0 ? 0 : nb));
    out3[0] = m.top1Match; out3[1] = m.distance; out3[2] = m.jsd;
}
BLK_API float blh_lc_similarity(const blk_token_data* a, int32_t na, const blk_token_data* b, int32_t nb) {
    return LogitComparer::logitSimilarity(toVec(a, na), toVec(b, nb));
}
// pushes metrics one at a time (as Server::verify does) and returns the final score
BLK_API float blh_lc_score(const float* metrics3, int32_t n) {
    MetricsAggregator agg; float score = 0;
    for (int32_t i = 0; i < n; ++i) { ComparisonMetrics m{metrics3[i * 3], metrics3[i * 3 + 1], metrics3[i * 3 + 2]}; score = agg.pushAndVerify({&m, 1}); }
    return score;
}

// ---- sampler (host only; no device needed) -------------------------------------------------------------------------
// draws n_draws tokens from the same sorted candidate list with one sampler instance
BLK_API int blh_sampler_draw(uint32_t seed, float temp, float top_p, int32_t top_k, float min_p, int32_t min_keep,
                             const blk_token_data* cand, int32_t n_cand, int32_t sorted, int32_t n_draws, int32_t* out) {
    return guard([&] {
        Sampler::Params sp; sp.rngSeed = seed; sp.temp = temp; sp.topP = top_p; sp.topK = top_k; sp.minP = min_p; sp.minKeep = min_keep;
        Model* none = nullptr;
        Sampler s(*none, sp);
        auto v = toVec(cand, n_cand);
        for (int32_t i = 0; i < n_draws; ++i) out[i] = s.sample(v, sorted != 0);
    });
}

// The full-row path with logit bias and penalties: accepts `history`, then n_draws times edits a copy of the row (n_vocab logits)
// with the window so far, draws from it (unsorted, as Session does with the whole vocabulary) and accepts the draw.
BLK_API int blh_sampler_draw_penalized(uint32_t seed, float temp, float top_p, int32_t top_k, float min_p, int32_t min_keep,
                                       int32_t last_n, float repeat, float freq, float present, const int32_t* bias_ids, const float* bias_vals, int n_bias,
                                       const int32_t* history, int32_t n_history, const float* logits, int32_t n_vocab, int32_t n_draws, int32_t* out) {
    return guard([&] {
        Sampler::Params sp; sp.rngSeed = seed; sp.temp = temp; sp.topP = top_p; sp.topK = top_k; sp.minP = min_p; sp.minKeep = min_keep;
        setStages(sp, last_n, repeat, freq, present, bias_ids, bias_vals, n_bias);
        Model* none = nullptr;
        Sampler s(*none, sp);
        for (int32_t i = 0; i < n_history; ++i) s.accept(history[i], false);
        std::vector<float> row(static_cast<size_t>(n_vocab));
        TokenDataVector all(static_cast<size_t>(n_vocab));
        for (int32_t d = 0; d < n_draws; ++d) {
            row.assign(logits, logits + n_vocab);
            s.applyEdits(row);
            for (int32_t t = 0; t < n_vocab; ++t) all[size_t(t)] = {t, row[size_t(t)]};
            out[d] = s.sample(all, false);
            s.accept(out[d], true);
        }
    });
}
// constructs a Sampler with the given mirostat version / grammar (the stages this build refuses): 0 when it is accepted
BLK_API int blh_sampler_check(int32_t mirostat, const char* grammar) {
    return guard([&] {
        Sampler::Params sp; sp.mirostat.ver = mirostat; sp.grammar = grammar ? grammar : "";
        Model* none = nullptr;
        Sampler s(*none, sp);
    });
}
// Sampler::logitEdits after accepting `history` (and a reset() afterwards when reset_after != 0)
BLK_API int blh_sampler_logit_edits(int32_t last_n, float repeat, float freq, float present, const int32_t* bias_ids, const float* bias_vals, int n_bias,
                                    const int32_t* history, int32_t n_history, int32_t reset_after, int32_t n_vocab,
                                    blk_logit_edit* out, int cap, int32_t* n, float* out3) {
    return guard([&] {
        Sampler::Params sp;
        setStages(sp, last_n, repeat, freq, present, bias_ids, bias_vals, n_bias);
        Model* none = nullptr;
        Sampler s(*none, sp);
        for (int32_t i = 0; i < n_history; ++i) s.accept(history[i], false);
        if (reset_after) s.reset();
        writeEdits(s.logitEdits(n_vocab), out, cap, n, out3);
    });
}

// ---- Server (reference server/code/server/Server.hpp:58-64): N workers = N replicas, requests are whole jobs ----------------------
// models: handles from blh_model_create, one per replica (they stay owned by the caller and must outlive the server)
BLK_API int blh_server_create_ex(void* const* models, int n_models, uint32_t ctx_size, uint32_t batch_size, uint32_t max_batch, void** out);
BLK_API int blh_server_create(void* const* models, int n_models, uint32_t ctx_size, uint32_t batch_size, void** out) {
    return blh_server_create_ex(models, n_models, ctx_size, batch_size, 1, out);
}
// max_batch > 1: continuous batching, up to max_batch /complete requests in flight per replica (Server.hpp)
BLK_API int blh_server_create_ex(void* const* models, int n_models, uint32_t ctx_size, uint32_t batch_size, uint32_t max_batch, void** out) {
    return guard([&] {
        if (n_models <= 0) Raise{} << "a server needs at least one model replica";
        std::vector<std::shared_ptr<Model>> reps;
        for (int i = 0; i < n_models; ++i) reps.emplace_back(static_cast<Model*>(models[i]), [](Model*) {});
        Instance::InitParams ip; ip.ctxSize = ctx_size; if (batch_size) ip.batchSize = batch_size;
        auto box = std::make_unique<ServerBox>();
        if (max_batch > 64) Raise{} << "at most 64 requests per batched step";
        box->srv = std::make_unique<server::Server>(std::move(reps), ip, max_batch < 1 ? 1u : max_batch);
        ServerBox* raw = box.get();
        box->srv->setErrorHandler([raw](const std::string& e) { std::lock_guard<std::mutex> lk(raw->mu); raw->lastWorkerError = e; });
        *out = box.release();
    });
}
BLK_API void blh_server_free(void* s) { delete static_cast<ServerBox*>(s); }
BLK_API int blh_server_workers(void* s) { return int(static_cast<ServerBox*>(s)->srv->workerCount()); }
BLK_API void blh_server_drain(void* s) { static_cast<ServerBox*>(s)->srv->drain(); }
// text of the last exception a worker caught (empty when none)
BLK_API int blh_server_last_worker_error(void* s, char* buf, int cap) {
    auto* box = static_cast<ServerBox*>(s);
    std::lock_guard<std::mutex> lk(box->mu);
    const int n = int(box->lastWorkerError.size());
    if (buf && cap > 0) { memcpy(buf, box->lastWorkerError.data(), size_t(n < cap ? n : cap)); }
    return n;
}
// Server::completeText with the prompt already tokenised; *ticket identifies the pending answer
BLK_API int blh_server_submit_complete(void* s, const int32_t* prompt, int n_prompt, uint32_t max_tokens, uint32_t seed, float temp, float top_p, int64_t* ticket) {
    return guard([&] {
        auto* box = static_cast<ServerBox*>(s);
        auto [id, t] = box->open();
        server::Server::CompleteRequestParams p; p.maxTokens = max_tokens; p.seed = seed; p.temperature = temp; p.topP = top_p;
        box->srv->completeTokens(std::vector<int32_t>(prompt, prompt + n_prompt), std::move(p),
                                 [box, t = t](server::Server::CompleteReponse r) { t->response = std::move(r); box->finish(t); });
        *ticket = id;
    });
}
// the same with the request's logit bias / repetition penalties (CompleteRequestParams extension)
BLK_API int blh_server_submit_complete_ex(void* s, const int32_t* prompt, int n_prompt, uint32_t max_tokens, uint32_t seed, float temp, float top_p,
                                          int32_t last_n, float repeat, float freq, float present, const int32_t* bias_ids, const float* bias_vals,
                                          int n_bias, int64_t* ticket) {
    return guard([&] {
        auto* box = static_cast<ServerBox*>(s);
        server::Server::CompleteRequestParams p; p.maxTokens = max_tokens; p.seed = seed; p.temperature = temp; p.topP = top_p;
        p.repetitionPenalty = {last_n, repeat, freq, present};
        for (int i = 0; i < n_bias; ++i) p.logitBias[bias_ids[i]] = bias_vals[i];
        auto [id, t] = box->open();
        box->srv->completeTokens(std::vector<int32_t>(prompt, prompt + n_prompt), std::move(p),
                                 [box, t = t](server::Server::CompleteReponse r) { t->response = std::move(r); box->finish(t); });
        *ticket = id;
    });
}
// Server::verify with the prompt already tokenised and the response as [n][10] claimed blocks
BLK_API int blh_server_submit_verify(void* s, const int32_t* prompt, int n_prompt, uint32_t seed, float temp, float top_p,
                                     const int32_t* toks, int n, const blk_token_data* claimed, const int32_t* n_claimed, int64_t* ticket) {
    return guard([&] {
        auto* box = static_cast<ServerBox*>(s);
        auto resp = responseOf(toks, n, claimed, n_claimed);
        auto [id, t] = box->open();
        server::Server::CompleteRequestParams p; p.seed = seed; p.temperature = temp; p.topP = top_p;
        box->srv->verifyTokens(std::vector<int32_t>(prompt, prompt + n_prompt), std::move(p), std::move(resp),
                               [box, t = t](float score) { t->score = score; box->finish(t); });
        *ticket = id;
    });
}
// the two HTTP bodies, text in / ticket out: POST /complete (HttpServerMain.cpp:312-318), POST /verify_completion (:328-337)
BLK_API int blh_server_submit_complete_json(void* s, const char* body, int64_t* ticket) {
    return guard([&] {
        auto* box = static_cast<ServerBox*>(s);
        auto params = server::wire::parseCompleteParams(body);
        auto [id, t] = box->open();
        box->srv->completeText(std::move(params), [box, t = t](server::Server::CompleteReponse r) { t->response = std::move(r); box->finish(t); });
        *ticket = id;
    });
}
BLK_API int blh_server_submit_verify_json(void* s, const char* body, int64_t* ticket) {
    return guard([&] {
        auto* box = static_cast<ServerBox*>(s);
        auto vb = server::wire::parseVerifyBody(body);
        auto [id, t] = box->open();
        box->srv->verify(std::move(vb.request), std::move(vb.response), [box, t = t](float score) { t->score = score; box->finish(t); });
        *ticket = id;
    });
}
// blocks until the ticket's request has run.  out_top10: [cap][10]
BLK_API int blh_server_wait_complete(void* s, int64_t ticket, int cap, int32_t* out_tokens, blk_token_data* out_top10, int32_t* out_n_logits, int32_t* out_n) {
    return guard([&] {
        auto t = static_cast<ServerBox*>(s)->wait(ticket);
        const int n = int(std::min<size_t>(t->response.size(), size_t(cap < 0 ? 0 : cap)));
        *out_n = int32_t(t->response.size());
        for (int i = 0; i < n; ++i) {
            const auto& td = t->response[size_t(i)];
            out_tokens[i] = int32_t(td.tokenId);
            out_n_logits[i] = int32_t(td.logits.size());
            for (size_t j = 0; j < td.logits.size() && j < 10; ++j) out_top10[size_t(i) * 10 + j] = {int32_t(td.logits[j].tokenId), td.logits[j].logit};
        }
    });
}
BLK_API int blh_server_wait_verify(void* s, int64_t ticket, float* score) {
    return guard([&] { *score = static_cast<ServerBox*>(s)->wait(ticket)->score; });
}
// the answer as the HTTP body the reference would send ({"text","tokenData"} or {"result"}); returns the length, copies <= cap bytes
BLK_API int blh_server_wait_complete_json(void* s, int64_t ticket, char* buf, int cap, int* len) {
    return guard([&] {
        const std::string js = server::wire::completeResponseJson(static_cast<ServerBox*>(s)->wait(ticket)->response);
        *len = int(js.size());
        if (buf && cap > 0) memcpy(buf, js.data(), size_t(std::min<int>(cap, int(js.size()))));
    });
}
BLK_API int blh_server_wait_verify_json(void* s, int64_t ticket, char* buf, int cap, int* len) {
    return guard([&] {
        const std::string js = server::wire::verifyResponseJson(static_cast<ServerBox*>(s)->wait(ticket)->score);
        *len = int(js.size());
        if (buf && cap > 0) memcpy(buf, js.data(), size_t(std::min<int>(cap, int(js.size()))));
    });
}
BLK_API int blh_server_stats(void* s, int32_t* devices, uint64_t* requests, double* gpu_ms, int cap) {
    const auto st = static_cast<ServerBox*>(s)->srv->workerStats();
    for (size_t i = 0; i < st.size() && int(i) < cap; ++i) { devices[i] = st[i].device; requests[i] = st[i].requests; gpu_ms[i] = st[i].gpuMs; }
    return int(st.size());
}
// HTTP front end on host:port (0 = any free port; the bound one comes back through *out_port)
BLK_API int blh_server_http_start(void* s, const char* host, int port, int io_threads, int* out_port) {
    return guard([&] {
        auto* box = static_cast<ServerBox*>(s);
        if (box->http) Raise{} << "the HTTP front end is already running";
        box->http = std::make_unique<server::HttpFrontEnd>(*box->srv, host ? host : "0.0.0.0", uint16_t(port), io_threads > 0 ? io_threads : 4);
        if (out_port) *out_port = box->http->port();
    });
}
BLK_API void blh_server_http_stop(void* s) { static_cast<ServerBox*>(s)->http.reset(); }

// ---- wire format, no device needed (tests pin the float text and the key order) ------------------------------------------------
// dumps {"result": v}
BLK_API int blh_wire_verify_json(float v, char* buf, int cap) {
    const std::string js = server::wire::verifyResponseJson(v);
    if (buf && cap > 0) memcpy(buf, js.data(), size_t(std::min<int>(cap, int(js.size()))));
    return int(js.size());
}
// parse -> dump of any JSON document (normalises key order and number text exactly as the reference's nlohmann round trip does)
BLK_API int blh_wire_json_roundtrip(const char* text, char* buf, int cap, int* len) {
    return guard([&] {
        const std::string js = json::parse(text).dump();
        *len = int(js.size());
        if (buf && cap > 0) memcpy(buf, js.data(), size_t(std::min<int>(cap, int(js.size()))));
    });
}
// request body -> fields (HttpServerMain.cpp:85-94)
BLK_API int blh_wire_parse_request(const char* body, char* prompt, int prompt_cap, uint32_t* max_tokens, uint32_t* seed, float* temp, float* top_p) {
    return guard([&] {
        const auto p = server::wire::parseCompleteParams(body);
        snprintf(prompt, size_t(prompt_cap), "%s", p.prompt.c_str());
        *max_tokens = p.maxTokens; *seed = p.seed; *temp = p.temperature; *top_p = p.topP;
    });
}
// /verify_completion body -> the response's token ids and claimed logits ([cap][10] blocks); *n = tokens in the response
BLK_API int blh_wire_parse_verify(const char* body, int cap, int32_t* toks, blk_token_data* claimed, int32_t* n_claimed, int32_t* n) {
    return guard([&] {
        const auto vb = server::wire::parseVerifyBody(body);
        *n = int32_t(vb.response.size());
        for (size_t i = 0; i < vb.response.size() && int(i) < cap; ++i) {
            toks[i] = int32_t(vb.response[i].tokenId);
            n_claimed[i] = int32_t(vb.response[i].logits.size());
            for (size_t j = 0; j < vb.response[i].logits.size() && j < 10; ++j) claimed[i * 10 + j] = {int32_t(vb.response[i].logits[j].tokenId), vb.response[i].logits[j].logit};
        }
    });
}
// [n][10] blocks -> the /complete answer body
BLK_API int blh_wire_complete_json(void* model, const int32_t* toks, int n, const blk_token_data* top10, const int32_t* n_logits, char* buf, int cap, int* len) {
    return guard([&] {
        server::Server::CompleteReponse resp = responseOf(toks, n, top10, n_logits);
        if (model) for (auto& td : resp) td.tokenStr = static_cast<Model*>(model)->vocab().tokenToString(Token(td.tokenId));
        const std::string js = server::wire::completeResponseJson(resp);
        *len = int(js.size());
        if (buf && cap > 0) memcpy(buf, js.data(), size_t(std::min<int>(cap, int(js.size()))));
    });
}

} // extern "C"
