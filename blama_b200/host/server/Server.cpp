// Server.cpp -- reference server/code/server/Server.cpp:45-161 with N workers (one per GPU replica).
#include "Server.hpp"

#include "../llama/Instance.hpp"
#include "../llama/LogitComparer.hpp"
#include "../llama/Model.hpp"
#include "../llama/Session.hpp"

#include <blama_b200.h>

#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <deque>
#include <limits>
#include <mutex>
#include <thread>

namespace bl::llama::server {

struct Server::Impl {
    struct Worker {
        std::shared_ptr<Model> model;
        std::unique_ptr<Instance> instance;                 // slot 0; also the workspace of the batched steps
        std::vector<std::unique_ptr<Instance>> extra;       // slots 1 .. maxBatch - 1 (continuous batching)
        std::thread thread;
        uint64_t requests = 0;      // guarded by Impl::mu
        double gpuMs = 0;
        Instance& slot(size_t i) { return i == 0 ? *instance : *extra[i - 1]; }
    };
    struct Job {
        std::function<void(Worker&, size_t)> run;      // (worker, slot): slot 0 unless the worker batches
        std::function<void()> failed;      // delivers the request's "no result" answer to its callback
        // a /complete request in a form the batching worker can advance token by token
        bool isComplete = false;
        std::vector<int32_t> prompt; bool tokenize = false; CompleteRequestParams params;
        std::shared_ptr<std::function<void(CompleteReponse)>> completeCb;
    };
    struct Generation {              // a /complete request in flight on one slot
        size_t slotIndex;
        Session* session;
        uint32_t maxTokens;
        std::vector<TokenPrediction> preds;
        std::shared_ptr<std::function<void(CompleteReponse)>> cb;
    };
    unsigned maxBatch = 1;

    std::vector<std::unique_ptr<Worker>> workers;
    mutable std::mutex mu;
    std::condition_variable cv, idleCv;
    std::deque<Job> queue;
    size_t running = 0;
    bool stopping = false;
    std::function<void(const std::string&)> onError;

    Impl(std::vector<std::shared_ptr<Model>> replicas, Instance::InitParams ip, unsigned batch) : maxBatch(batch < 1 ? 1 : batch) {
        for (auto& r : replicas) {
            auto w = std::make_unique<Worker>();
            w->model = std::move(r);
            w->instance = std::make_unique<Instance>(*w->model, ip);
            w->instance->warmup();
            for (unsigned i = 1; i < maxBatch; ++i) w->extra.push_back(std::make_unique<Instance>(*w->model, ip));
            workers.push_back(std::move(w));
        }
        for (auto& w : workers) w->thread = std::thread([this, wp = w.get()] { if (maxBatch > 1) batchLoop(*wp); else loop(*wp); });
    }
    ~Impl() {
        { std::lock_guard<std::mutex> lk(mu); stopping = true; }
        cv.notify_all();
        for (auto& w : workers) if (w->thread.joinable()) w->thread.join();
    }
    void post(Job j) {
        { std::lock_guard<std::mutex> lk(mu); queue.push_back(std::move(j)); }
        cv.notify_one();
    }
    void loop(Worker& w) {
        for (;;) {
            Job job;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return stopping || !queue.empty(); });
                if (queue.empty()) return;
                job = std::move(queue.front());
                queue.pop_front();
                ++running;
            }
            // CUDA events on the worker's own stream bracket the request: the GPU time of this replica, whatever the host did
            blk_ctx* ctx = w.instance->lctx();
            (void)blk_timer_start(ctx);
            std::string error;
            bool ok = true;
            try { job.run(w, 0); }
            catch (const std::exception& e) { ok = false; error = e.what(); }
            catch (...) { ok = false; error = "unknown error"; }
            float ms = 0.0f;
            (void)blk_timer_stop(ctx, &ms);
            if (!ok) {
                // the reference lets the exception escape its io_context and dies (SURVEY.md section 5); here the session is
                // stopped, the error reported and the request's callback answered, so that nobody waits forever
                w.instance->stopSession();
                std::function<void(const std::string&)> handler;
                { std::lock_guard<std::mutex> lk(mu); handler = onError; }
                try { if (handler) handler(error); } catch (...) {}
                try { if (job.failed) job.failed(); } catch (...) {}
            }
            {
                std::lock_guard<std::mutex> lk(mu);
                w.requests++; w.gpuMs += ms;
                --running;
                if (queue.empty() && running == 0) idleCv.notify_all();
            }
        }
    }
    // ---- continuous batching: up to maxBatch /complete requests advance together, one blk_decode_batch step per token ----
    void reportFailure(const std::string& error) {
        std::function<void(const std::string&)> handler;
        { std::lock_guard<std::mutex> lk(mu); handler = onError; }
        try { if (handler) handler(error); } catch (...) {}
    }
    void finish(Worker& w, Generation& g) {
        auto response = marshal(*w.model, g.preds);
        w.slot(g.slotIndex).stopSession();
        try { (*g.cb)(std::move(response)); } catch (...) {}
        std::lock_guard<std::mutex> lk(mu);
        w.requests++;
    }
    void batchLoop(Worker& w) {
        // BLAMA_SERVER_PROFILE=1: host-side time per part of the loop, printed when the worker stops
        const bool prof = std::getenv("BLAMA_SERVER_PROFILE") != nullptr;
        double tAdmit = 0, tSample = 0, tStep = 0, tAccept = 0, tRetire = 0; uint64_t nSteps = 0, nRows = 0;
        auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        struct Report { bool on; double& a; double& b; double& c; double& d; double& e; uint64_t& n; uint64_t& r;
            ~Report() { if (on) std::fprintf(stderr, "[server profile] steps %llu rows %llu | admit %.1f ms, sample %.1f, step %.1f, accept %.1f, retire %.1f\n",
                                             (unsigned long long)n, (unsigned long long)r, a, b, c, d, e); } } report{prof, tAdmit, tSample, tStep, tAccept, tRetire, nSteps, nRows};
        std::vector<Generation> active;
        std::vector<char> busy(maxBatch, 0);
        blk_ctx* ws = w.instance->lctx();
        for (;;) {
            // 1. admit: block only when nothing is in flight
            std::vector<Job> admitted;
            {
                std::unique_lock<std::mutex> lk(mu);
                if (active.empty()) cv.wait(lk, [&] { return stopping || !queue.empty(); });
                if (queue.empty() && active.empty()) { if (stopping) return; continue; }
                size_t freeSlots = maxBatch - active.size();
                while (!queue.empty()) {
                    if (queue.front().isComplete) { if (freeSlots == 0) break; --freeSlots; }
                    else if (!active.empty() && freeSlots == 0) break;          // a verify needs a slot of its own, too
                    else if (freeSlots > 0) --freeSlots;
                    admitted.push_back(std::move(queue.front()));
                    queue.pop_front();
                    ++running;
                }
            }
            const double ta0 = now();
            for (Job& job : admitted) {
                size_t si = 0;
                while (si < maxBatch && busy[si]) ++si;
                float ms = 0.0f;
                blk_ctx* ctx = w.slot(si).lctx();
                (void)blk_timer_start(ctx);
                try {
                    if (!job.isComplete) {                    // e.g. a verify: one prefill on a free slot, between two steps
                        job.run(w, si);
                    } else {
                        auto& session = startComplete(w.slot(si), job.params);
                        if (job.tokenize) job.prompt = w.model->vocab().tokenize(job.params.prompt, true, true);
                        session.setInitialPrompt(job.prompt);
                        busy[si] = 1;
                        active.push_back({si, &session, job.params.maxTokens, {}, job.completeCb});
                    }
                } catch (const std::exception& e) {
                    w.slot(si).stopSession();
                    reportFailure(e.what());
                    try { if (job.failed) job.failed(); } catch (...) {}
                }
                (void)blk_timer_stop(ctx, &ms);
                std::lock_guard<std::mutex> lk(mu);
                w.gpuMs += ms;
                if (!job.isComplete) { w.requests++; --running; }
            }
            tAdmit += now() - ta0;
            const double tr0 = now();
            // 2. requests that are done (token budget reached) leave
            auto retire = [&](size_t i, bool failed, const std::string& why) {
                Generation g = std::move(active[i]);
                active.erase(active.begin() + long(i));
                busy[g.slotIndex] = 0;
                if (failed) { w.slot(g.slotIndex).stopSession(); reportFailure(why); try { (*g.cb)({}); } catch (...) {} std::lock_guard<std::mutex> lk(mu); w.requests++; }
                else finish(w, g);
                std::lock_guard<std::mutex> lk(mu);
                --running;
                if (queue.empty() && running == 0) idleCv.notify_all();
            };
            for (size_t i = active.size(); i-- > 0;) if (active[i].preds.size() >= active[i].maxTokens) retire(i, false, {});
            tRetire += now() - tr0;
            if (active.empty()) { std::lock_guard<std::mutex> lk(mu); if (queue.empty() && running == 0) idleCv.notify_all(); continue; }
            // 3. one token for everybody in flight
            float ms = 0.0f;
            (void)blk_timer_start(ws);
            if (active.size() == 1) {
                // a lone request: the batch-1 decode kernel (the reference's arithmetic), exactly Session::complete's step
                Generation& g = active[0];
                try {
                    auto preds = g.session->complete({.prompt = {}, .suffix = {}, .maxTokens = 1});
                    if (preds.empty()) g.maxTokens = uint32_t(g.preds.size());        // end of generation
                    else g.preds.push_back(std::move(preds[0]));
                } catch (const std::exception& e) { (void)blk_timer_stop(ws, &ms); retire(0, true, e.what()); continue; }
            } else {
                std::vector<blk_ctx*> ctxs; std::vector<Token> toks; std::vector<size_t> who;
                const double ts0 = now();
                for (size_t i = active.size(); i-- > 0;) {
                    try {
                        const Token t = active[i].session->sampleNext();
                        if (t == Token_Invalid) { active[i].maxTokens = uint32_t(active[i].preds.size()); continue; }      // leaves at the next round
                        ctxs.push_back(w.slot(active[i].slotIndex).lctx()); toks.push_back(t); who.push_back(i);
                    } catch (const std::exception& e) { retire(i, true, e.what()); for (auto& x : who) if (x > i) --x; }
                }
                tSample += now() - ts0;
                if (!ctxs.empty()) {
                    const double tb0 = now();
                    constexpr int32_t K = Sampler::MaxDeviceCandidates;
                    // rows whose sampler edits the logits (bias / penalties, after sampleNext accepted the token) need the edited
                    // top-k too: then one edit pass covers every row; without any, exactly the plain step
                    std::vector<Sampler::LogitEdits> edits(ctxs.size());
                    bool anyEdits = false;
                    for (size_t j = 0; j < who.size(); ++j) { edits[j] = active[who[j]].session->logitEdits(); anyEdits = anyEdits || !edits[j].edits.empty(); }
                    std::vector<blk_token_data> top(ctxs.size() * size_t(K)), edited(anyEdits ? top.size() : 0);
                    std::vector<blk_logit_edits> rows;
                    for (const auto& e : edits) rows.push_back(abiEdits(e));
                    const blk_status st = anyEdits ? blk_decode_batch_edited(ws, ctxs.data(), toks.data(), int32_t(ctxs.size()), K, rows.data(), top.data(), edited.data())
                                                   : blk_decode_batch(ws, ctxs.data(), toks.data(), int32_t(ctxs.size()), K, top.data());
                    if (st != BLK_OK) {
                        const std::string why = std::string("Failed to decode tokens: ") + blk_last_error();
                        (void)blk_timer_stop(ws, &ms);
                        while (!active.empty()) retire(active.size() - 1, true, why);
                        continue;
                    }
                    const double tc0 = now();
                    tStep += tc0 - tb0; nSteps++; nRows += ctxs.size();
                    using LlamaTokenData = bl::llama::TokenData;      // (Server::TokenData is the marshalled form)
                    static_assert(sizeof(LlamaTokenData) == sizeof(blk_token_data));
                    for (size_t j = 0; j < who.size(); ++j) {
                        const LlamaTokenData* cand = reinterpret_cast<const LlamaTokenData*>(top.data() + j * size_t(K));
                        std::span<const LlamaTokenData> ed;
                        if (anyEdits) ed = {reinterpret_cast<const LlamaTokenData*>(edited.data() + j * size_t(K)), size_t(K)};
                        active[who[j]].preds.push_back(active[who[j]].session->acceptDecoded(toks[j], std::span<const LlamaTokenData>(cand, size_t(K)), ed));
                    }
                    tAccept += now() - tc0;
                }
            }
            (void)blk_timer_stop(ws, &ms);
            { std::lock_guard<std::mutex> lk(mu); w.gpuMs += ms; }
        }
    }
    void drain() {
        std::unique_lock<std::mutex> lk(mu);
        idleCv.wait(lk, [&] { return queue.empty() && running == 0; });
    }

    // a /complete session: the reference's sampler, replaced by one with the request's bias / penalties when it asks for them
    static Session& startComplete(Instance& inst, const CompleteRequestParams& p) {
        auto& session = inst.startSession({.seed = p.seed, .temperature = p.temperature, .topP = p.topP});
        const auto& rp = p.repetitionPenalty;
        if (!p.logitBias.empty() || !(rp.repeat == 1.0f && rp.freq == 0.0f && rp.present == 0.0f)) {
            Sampler::Params sp;
            sp.rngSeed = p.seed; sp.topP = p.topP; sp.temp = p.temperature;
            sp.repetitionPenalty = rp;
            sp.logitBias.insert(p.logitBias.begin(), p.logitBias.end());
            session.resetSampler(sp);
        }
        return session;
    }
    static CompleteReponse marshal(const Model& model, const std::vector<TokenPrediction>& preds) {
        CompleteReponse response;
        response.reserve(preds.size());
        for (const auto& p : preds) {
            auto& td = response.emplace_back();
            td.tokenStr = model.vocab().tokenToString(p.token);
            td.tokenId = uint32_t(p.token);
            td.logits.reserve(p.logits.size());
            for (const auto& l : p.logits) td.logits.push_back({uint32_t(l.token), l.logit});
        }
        return response;
    }
    static std::vector<TokenPrediction> unmarshal(const CompleteReponse& resp) {
        std::vector<TokenPrediction> preds;
        preds.reserve(resp.size());
        for (const auto& t : resp) {
            auto& p = preds.emplace_back();
            p.token = Token(t.tokenId);
            p.logits.reserve(t.logits.size());
            for (const auto& l : t.logits) p.logits.push_back({Token(l.tokenId), l.logit});
        }
        return preds;
    }

    void complete(std::vector<int32_t> prompt, bool tokenize, CompleteRequestParams params, std::function<void(CompleteReponse)> cb) {
        auto cbp = std::make_shared<std::function<void(CompleteReponse)>>(std::move(cb));
        Job job;
        job.isComplete = true; job.prompt = prompt; job.tokenize = tokenize; job.params = params; job.completeCb = cbp;
        job.run = [prompt = std::move(prompt), tokenize, params = std::move(params), cbp](Worker& w, size_t) mutable {
            auto& session = startComplete(*w.instance, params);
            if (tokenize) prompt = w.model->vocab().tokenize(params.prompt, true, true);
            session.setInitialPrompt(prompt);
            auto preds = session.complete({.prompt = {}, .suffix = {}, .maxTokens = int32_t(params.maxTokens)});
            auto response = marshal(*w.model, preds);
            w.instance->stopSession();
            (*cbp)(std::move(response));
        };
        job.failed = [cbp] { (*cbp)({}); };
        post(std::move(job));
    }
    void verify(std::vector<int32_t> prompt, bool tokenize, CompleteRequestParams req, CompleteReponse resp, std::function<void(float)> cb) {
        auto cbp = std::make_shared<std::function<void(float)>>(std::move(cb));
        Job job;
        job.run = [prompt = std::move(prompt), tokenize, req = std::move(req), resp = std::move(resp), cbp](Worker& w, size_t slot) mutable {
            Instance& inst = w.slot(slot);
            auto& session = inst.startSession({.seed = req.seed, .temperature = req.temperature, .topP = req.topP});
            if (tokenize) prompt = w.model->vocab().tokenize(req.prompt, true, true);
            auto orig = unmarshal(resp);
            // setInitialPrompt + fillCtx (reference :135, :149) as one causal prefill over [prompt | response]
            auto mine = session.setInitialPromptAndFill(prompt, orig);
            // the reference pushes one metric at a time and re-sums the history on every push (Server.cpp:153-156); only the last
            // push's value is reported, which is the in-order double sum over all metrics: one push of the whole span
            std::vector<TokenPredictionView> pairs(orig.size());
            for (size_t i = 0; i < orig.size(); i++) pairs[i] = {&orig[i].logits, &mine[i].logits};
            const std::vector<ComparisonMetrics> ms = compareAll(pairs);
            MetricsAggregator agg;
            const float score = ms.empty() ? 0.0f : agg.pushAndVerify(ms);
            inst.stopSession();
            (*cbp)(score);
        };
        job.failed = [cbp] { (*cbp)(std::numeric_limits<float>::quiet_NaN()); };
        post(std::move(job));
    }
};

Server::Server(std::shared_ptr<Model> model) : m_impl(std::make_unique<Impl>(std::vector<std::shared_ptr<Model>>{std::move(model)}, Instance::InitParams{}, 1u)) {}
Server::Server(std::vector<std::shared_ptr<Model>> replicas) : m_impl(std::make_unique<Impl>(std::move(replicas), Instance::InitParams{}, 1u)) {}
Server::Server(std::vector<std::shared_ptr<Model>> replicas, Instance::InitParams ip) : m_impl(std::make_unique<Impl>(std::move(replicas), ip, 1u)) {}
Server::Server(std::vector<std::shared_ptr<Model>> replicas, Instance::InitParams ip, unsigned maxBatch) : m_impl(std::make_unique<Impl>(std::move(replicas), ip, maxBatch)) {}
Server::~Server() = default;

void Server::completeText(CompleteRequestParams params, std::function<void(CompleteReponse)> cb) {
    m_impl->complete({}, true, std::move(params), std::move(cb));
}
void Server::verify(CompleteRequestParams req, CompleteReponse resp, std::function<void(float)> cb) {
    m_impl->verify({}, true, std::move(req), std::move(resp), std::move(cb));
}
void Server::completeTokens(std::vector<int32_t> prompt, CompleteRequestParams params, std::function<void(CompleteReponse)> cb) {
    m_impl->complete(std::move(prompt), false, std::move(params), std::move(cb));
}
void Server::verifyTokens(std::vector<int32_t> prompt, CompleteRequestParams req, CompleteReponse resp, std::function<void(float)> cb) {
    m_impl->verify(std::move(prompt), false, std::move(req), std::move(resp), std::move(cb));
}
void Server::setErrorHandler(std::function<void(const std::string&)> handler) {
    std::lock_guard<std::mutex> lk(m_impl->mu);
    m_impl->onError = std::move(handler);
}
std::vector<Server::WorkerStats> Server::workerStats() const {
    std::lock_guard<std::mutex> lk(m_impl->mu);
    std::vector<WorkerStats> out;
    for (const auto& w : m_impl->workers) out.push_back({w->model->params().device, w->requests, w->gpuMs});
    return out;
}
size_t Server::workerCount() const noexcept { return m_impl->workers.size(); }
void Server::drain() { m_impl->drain(); }

} // namespace bl::llama::server
