// Session.cpp -- blama's per-request control loop (reference inference/code/llama/Session.cpp) on the CUDA engine.
//
// What stays: phases, error strings, the "logits attached to token t are those AFTER t was decoded" rule
// (reference :186-189 + :252), EOG handling (:181-184), sampler accept/reset points.
// What changes: one blk_decode_topk per generated token replaces llama_decode + a 513 KB logits copy + two host
// passes + a full std::sort (:23-39, :254-260); fillCtx is one causal prefill instead of N decodes (:235-241).
#include "Session.hpp"
#include "Errors.hpp"
#include "Init.hpp"
#include "Instance.hpp"
#include "Model.hpp"

#include <blama_b200.h>

#include <algorithm>

namespace bl::llama {
namespace {
constexpr int32_t kReportedTop = 10;       // TokenPrediction carries the 10 best logits (Session.cpp:188)
}

Session::Session(Instance& instance, blk_ctx* ctx, InitParams params)
    : m_instance(instance)
    , m_ctx(ctx)
    , m_sampler(new Sampler(instance.model(), [&] {
          Sampler::Params sp;
          sp.rngSeed = params.seed;
          sp.topP = params.topP;
          sp.temp = params.temperature;
          sp.grammar = params.grammar;
          return sp;
      }()))
    , m_params(std::move(params)) {
    throwIfFailed(blk_kv_clear(m_ctx), "kv clear");
    throwIfFailed(blk_sync(m_ctx), "synchronize");
    m_maxTokens = unsigned(blk_ctx_n_ctx(m_ctx)) - 4;   // (#16)
}

Session::~Session() {
    try { flushPendingState(); } catch (...) {}
}

void Session::requireStarted(bool allowStreaming) const {
    if (m_phase == Phase::Generating) return;
    if (allowStreaming && m_phase == Phase::Streaming) return;
    Raise{} << "Session hasn't started yet";
}

void Session::setInitialPrompt(std::span<const Token> initialPrompt) {
    if (m_phase != Phase::Initial) Raise{} << "Session already started";

    Token single;
    const auto ctxLen = blk_ctx_n_ctx(m_ctx);
    m_numKeep = std::min(uint32_t(initialPrompt.size()), m_maxTokens);
    if (initialPrompt.empty()) {
        single = blk_model_token_bos(m_instance.model().lmodel());
        initialPrompt = {&single, 1};
    }
    if (initialPrompt.size() > m_maxTokens)
        Raise{} << "Initial prompt too long. Got " << initialPrompt.size() << " tokens, max: " << ctxLen - 4;
    if (m_params.gaFactor != 1) {
        if (m_params.gaFactor == 0 || m_params.gaWidth % m_params.gaFactor != 0)
            Raise{} << "Group-attention width " << m_params.gaWidth << " must be a multiple of group-attention factor " << m_params.gaFactor;
        logLine(LogLevel::Info, "self-extend: train = " + std::to_string(m_instance.model().trainCtxLength()) + ", gaFactor = " +
                                    std::to_string(m_params.gaFactor) + ", gaWidth = " + std::to_string(m_params.gaWidth));
    }
    doDecode(initialPrompt, Source::InitialPrompt);
    m_phase = Phase::Generating;
}

void Session::pushPrompt(std::span<const Token> prompt, std::span<const Token> postfix) {
    requireStarted(false);
    flushPendingState();
    if (prompt.empty() && postfix.empty()) Raise{} << "Prompt and postfix are empty";
    if (!postfix.empty()) Raise{} << "fill-in-the-middle prompts are not supported by this build";

    auto& model = m_instance.model();
    m_sampler->reset();     // previous inputs must not influence the generation

    std::vector<Token> tokens;
    tokens.reserve(prompt.size() + 1);
    if (model.prefixInputsWithBos()) tokens.push_back(blk_model_token_bos(model.lmodel()));
    tokens.insert(tokens.end(), prompt.begin(), prompt.end());
    if (tokens.size() > m_maxTokens)
        Raise{} << "Prompt too long. Got " << tokens.size() << " tokens, max: " << blk_ctx_n_ctx(m_ctx) - 4;
    doDecode(tokens, Source::InteractivePrompt);
}

TokenPrediction Session::getToken() {
    requireStarted(true);
    flushPendingState();

    // sample from the distribution left by the last decode; the chain only ever looks at its top-k
    const int32_t need = m_sampler->candidatesNeeded();
    if (need > 0) {
        const auto cands = samplingCandidates();
        m_currToken = m_sampler->sample(cands.first(std::min<size_t>(cands.size(), size_t(need))), true);
    } else {
        // top-k disabled or wider than the device list: the whole row is needed (reference behaviour, slow path)
        const int32_t nVocab = blk_model_n_vocab(m_instance.model().lmodel());
        std::vector<float> row(static_cast<size_t>(nVocab));
        throwIfFailed(blk_get_logits_last(m_ctx, row.data()), "get logits");
        m_sampler->applyEdits(row);
        TokenDataVector all(static_cast<size_t>(nVocab));
        for (int32_t i = 0; i < nVocab; ++i) all[size_t(i)] = {i, row[size_t(i)]};
        m_currToken = m_sampler->sample(all, false);
    }

    if (m_instance.model().vocab().isEog(m_currToken)) m_currToken = Token_Invalid;   // EOG is never decoded
    TokenPrediction out;
    out.token = m_currToken;
    out.logits = getLogitsFromCtx(kReportedTop);
    return out;
}

std::vector<TokenPrediction> Session::complete(CompleteParams params) {
    requireStarted(false);
    flushPendingState();
    if (params.prompt.size() || params.suffix.size()) pushPrompt(params.prompt, params.suffix);

    std::vector<TokenPrediction> predictions;
    for (int32_t i = 0; i < params.maxTokens; i++) {
        auto p = getToken();
        if (p.token == Token_Invalid) break;
        predictions.push_back(std::move(p));
    }
    return predictions;
}

Session::StreamGenerator Session::completeStream(CompleteParams params) {
    requireStarted(false);
    flushPendingState();
    if (params.prompt.size() || params.suffix.size()) pushPrompt(params.prompt, params.suffix);
    m_phase = Phase::Streaming;
    return StreamGenerator(*this, params);
}

std::vector<TokenPrediction> Session::fillCtx(std::span<TokenPrediction> tokens) {
    std::vector<TokenPrediction> result;
    result.reserve(tokens.size());
    if (tokens.empty()) return result;

    // the device gathers at most 10 ids per position in the batched form; the reference accepts any number of claimed logits
    bool wide = false;
    for (const auto& token : tokens) wide = wide || token.logits.size() > 10;
    // a fill that does not fit the context shifts it token by token exactly like the reference's loop
    const bool overflows = m_numPast + tokens.size() >= uint32_t(blk_ctx_n_ctx(m_ctx));
    if (m_instance.model().prefixInputsWithBos() || wide || overflows || m_params.gaFactor != 1) {      // (Self-Extend regroups between tokens)
        // every pushPrompt would insert a BOS before its token (reference :129-132) / more than 10 claimed ids somewhere:
        // keep the reference's literal per-token loop
        for (const auto& token : tokens) {
            pushPrompt({&token.token, 1}, {});
            result.push_back({token.token, getLogitsFromCtx(token.logits)});
        }
        return result;
    }

    requireStarted(false);
    flushPendingState();
    m_sampler->reset();

    const size_t n = tokens.size();
    std::vector<Token> ids(n);
    std::vector<int32_t> claimed(n * 10, 0), nClaimed(n, 0);
    for (size_t i = 0; i < n; ++i) {
        ids[i] = tokens[i].token;
        // distinct claimed ids in ascending order: what the reference's vocabulary walk would visit (:271-275)
        std::vector<Token> uniq;
        for (const auto& td : tokens[i].logits) uniq.push_back(td.token);
        std::sort(uniq.begin(), uniq.end());
        uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
        const int32_t nVocab = blk_model_n_vocab(m_instance.model().lmodel());
        uniq.erase(std::remove_if(uniq.begin(), uniq.end(), [&](Token t) { return t < 0 || t >= nVocab; }), uniq.end());
        nClaimed[i] = int32_t(uniq.size());
        std::copy(uniq.begin(), uniq.end(), claimed.begin() + long(i * 10));
    }
    // the reference pushes every response token as a prompt of its own (reset, then accept): its last one is what remains
    m_sampler->accept(ids.back(), false);
    std::vector<float> gathered(n * 10, 0.0f);
    throwIfFailed(blk_ctx_set_verify_mode(m_ctx, m_params.sequentialVerify ? 1 : 0), "verify mode");
    // the per-position top-10 of the verifier is not needed here (only the claimed ids are compared): nullptr skips that pass
    const int st = blk_verify_prefill(m_ctx, ids.data(), int32_t(n), claimed.data(), nClaimed.data(), gathered.data(), nullptr);
    if (st != BLK_OK) Raise{} << "Failed to decode tokens";
    m_numPast += uint32_t(n);
    m_haveRow = true;

    for (size_t i = 0; i < n; ++i) {
        TokenDataVector v(size_t(nClaimed[i]));
        for (int32_t j = 0; j < nClaimed[i]; ++j) v[size_t(j)] = {claimed[i * 10 + size_t(j)], gathered[i * 10 + size_t(j)]};
        std::sort(v.begin(), v.end(), [](const TokenData& a, const TokenData& b) { return a.logit > b.logit; });
        result.push_back({ids[i], std::move(v)});
    }
    // the verifier's own candidates (last position) for whoever continues generating after the fill
    refreshCandidates();
    return result;
}

std::vector<TokenPrediction> Session::setInitialPromptAndFill(std::span<const Token> prompt, std::span<TokenPrediction> tokens) {
    if (m_phase != Phase::Initial) Raise{} << "Session already started";
    bool wide = false;
    for (const auto& token : tokens) wide = wide || token.logits.size() > 10;
    const size_t total = std::max<size_t>(prompt.size(), 1) + tokens.size();
    const bool batched = !tokens.empty() && !m_instance.model().prefixInputsWithBos() && !wide && !m_params.sequentialVerify &&
                         m_params.gaFactor == 1 && total < m_maxTokens && total < size_t(blk_ctx_n_ctx(m_ctx));
    if (!batched) {
        setInitialPrompt(prompt);
        return fillCtx(tokens);
    }
    Token single;
    m_numKeep = std::min(uint32_t(prompt.size()), m_maxTokens);
    if (prompt.empty()) {
        single = blk_model_token_bos(m_instance.model().lmodel());
        prompt = {&single, 1};
    }
    const size_t np = prompt.size(), n = tokens.size();
    std::vector<Token> ids(np + n);
    std::vector<int32_t> claimed((np + n) * 10, 0), nClaimed(np + n, 0);
    for (size_t i = 0; i < np; ++i) { ids[i] = prompt[i]; m_sampler->accept(prompt[i], false); }
    // fillCtx pushes every response token as a prompt of its own (reset, then accept): only the last one remains
    m_sampler->reset();
    m_sampler->accept(tokens[n - 1].token, false);
    const int32_t nVocab = blk_model_n_vocab(m_instance.model().lmodel());
    for (size_t i = 0; i < n; ++i) {
        ids[np + i] = tokens[i].token;
        std::vector<Token> uniq;
        for (const auto& td : tokens[i].logits) uniq.push_back(td.token);
        std::sort(uniq.begin(), uniq.end());
        uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
        uniq.erase(std::remove_if(uniq.begin(), uniq.end(), [&](Token t) { return t < 0 || t >= nVocab; }), uniq.end());
        nClaimed[np + i] = int32_t(uniq.size());
        std::copy(uniq.begin(), uniq.end(), claimed.begin() + long((np + i) * 10));
    }
    std::vector<float> gathered((np + n) * 10, 0.0f);
    throwIfFailed(blk_ctx_set_verify_mode(m_ctx, 0), "verify mode");
    if (blk_verify_prefill(m_ctx, ids.data(), int32_t(np + n), claimed.data(), nClaimed.data(), gathered.data(), nullptr) != BLK_OK)
        Raise{} << "Failed to decode tokens";
    m_numPast += uint32_t(np + n);
    m_haveRow = true;
    m_phase = Phase::Generating;
    std::vector<TokenPrediction> result;
    result.reserve(n);
    for (size_t i = np; i < np + n; ++i) {
        TokenDataVector v(size_t(nClaimed[i]));
        for (int32_t j = 0; j < nClaimed[i]; ++j) v[size_t(j)] = {claimed[i * 10 + size_t(j)], gathered[i * 10 + size_t(j)]};
        std::sort(v.begin(), v.end(), [](const TokenData& a, const TokenData& b) { return a.logit > b.logit; });
        result.push_back({ids[i], std::move(v)});
    }
    refreshCandidates();
    return result;
}

Token Session::sampleNext() {
    requireStarted(true);
    flushPendingState();
    const int32_t need = m_sampler->candidatesNeeded();
    if (need <= 0) Raise{} << "batched decoding needs a sampler chain that starts with top-k (the device returns the top " << Sampler::MaxDeviceCandidates << ")";
    const auto cands = samplingCandidates();
    const Token t = m_sampler->sample(cands.first(std::min<size_t>(cands.size(), size_t(need))), true);
    if (m_instance.model().vocab().isEog(t)) return Token_Invalid;
    ensureRoom(1);
    m_sampler->accept(t, true);
    return t;
}

TokenPrediction Session::acceptDecoded(Token token, std::span<const TokenData> candidates, std::span<const TokenData> edited) {
    m_numPast += 1;
    m_candidates.assign(candidates.begin(), candidates.end());
    m_edited.assign(edited.begin(), edited.end());
    m_useEdited = !edited.empty();
    m_haveRow = false;
    TokenPrediction out;
    out.token = token;
    out.logits.assign(m_candidates.begin(), m_candidates.begin() + std::min<size_t>(m_candidates.size(), size_t(kReportedTop)));
    return out;
}

void Session::refreshCandidates() {
    m_candidates.resize(size_t(Sampler::MaxDeviceCandidates));
    static_assert(sizeof(TokenData) == sizeof(blk_token_data));
    throwIfFailed(blk_topk_last(m_ctx, Sampler::MaxDeviceCandidates, reinterpret_cast<blk_token_data*>(m_candidates.data())), "top-k");
    refreshEdited();
}

// the edited top-k of the kept row for the current sampler (nothing to do, and no launch, when it has no edits)
void Session::refreshEdited() {
    const Sampler::LogitEdits edits = logitEdits();
    m_useEdited = !edits.edits.empty();
    if (!m_useEdited) return;
    if (!m_haveRow) Raise{} << "logit bias and repetition penalties need the last logits row, which a batched decode step does not keep";
    const blk_logit_edits e = abiEdits(edits);
    m_edited.resize(size_t(Sampler::MaxDeviceCandidates));
    throwIfFailed(blk_topk_last_edited(m_ctx, Sampler::MaxDeviceCandidates, &e, reinterpret_cast<blk_token_data*>(m_edited.data())), "edited top-k");
}

std::span<const TokenData> Session::samplingCandidates() const { return m_useEdited ? m_edited : m_candidates; }

Sampler::LogitEdits Session::logitEdits() const { return m_sampler->logitEdits(nVocab()); }

int32_t Session::nVocab() const { return blk_model_n_vocab(m_instance.model().lmodel()); }

TokenDataVector Session::getLogitsFromCtx(int32_t topK) {
    requireStarted(true);
    flushPendingState();
    if (topK < 0) topK = 0;
    if (size_t(topK) <= m_candidates.size()) return TokenDataVector(m_candidates.begin(), m_candidates.begin() + topK);
    // more than the device list holds: fetch the row and sort on the host exactly like the reference (:254-260)
    const int32_t nVocab = blk_model_n_vocab(m_instance.model().lmodel());
    std::vector<float> row(static_cast<size_t>(nVocab));
    throwIfFailed(blk_get_logits_last(m_ctx, row.data()), "get logits");
    TokenDataVector all(static_cast<size_t>(nVocab));
    for (int32_t i = 0; i < nVocab; ++i) all[size_t(i)] = {i, row[size_t(i)]};
    std::sort(all.begin(), all.end(), [](const TokenData& a, const TokenData& b) { return a.logit > b.logit; });
    all.resize(size_t(std::min(topK, nVocab)));
    return all;
}

TokenDataVector Session::getLogitsFromCtx(TokenDataVector tokens) {
    requireStarted(true);
    flushPendingState();
    std::vector<Token> uniq;
    for (const auto& td : tokens) uniq.push_back(td.token);
    std::sort(uniq.begin(), uniq.end());
    uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
    const int32_t nVocab = blk_model_n_vocab(m_instance.model().lmodel());
    uniq.erase(std::remove_if(uniq.begin(), uniq.end(), [&](Token t) { return t < 0 || t >= nVocab; }), uniq.end());
    TokenDataVector res(uniq.size());
    if (uniq.empty()) return res;
    std::vector<float> vals(uniq.size());
    throwIfFailed(blk_gather_last(m_ctx, uniq.data(), int32_t(uniq.size()), vals.data()), "gather logits");
    for (size_t i = 0; i < uniq.size(); ++i) res[i] = {uniq[i], vals[i]};
    std::sort(res.begin(), res.end(), [](const TokenData& a, const TokenData& b) { return a.logit > b.logit; });
    return res;
}

std::vector<uint8_t> Session::getState() {
    requireStarted(false);
    flushPendingState();
    const auto size = blk_state_size(m_ctx);
    std::vector<uint8_t> state(static_cast<size_t>(size));
    int64_t written = 0;
    if (blk_state_get(m_ctx, state.data(), size, &written) != BLK_OK || written != size) Raise{} << "Failed to get state";
    return state;
}

bool Session::setState(std::span<uint8_t> state) {
    if (m_phase != Phase::Initial) Raise{} << "Session already started";
    if (blk_state_set(m_ctx, state.data(), int64_t(state.size())) != BLK_OK) Raise{} << "Failed to set state";
    // llama.cpp keeps the positions inside its context; here the session's counters follow the restored cache
    m_numPast = uint32_t(blk_ctx_next_pos(m_ctx));
    m_numKeep = std::min(m_numPast, m_maxTokens);
    m_haveRow = true;
    refreshCandidates();
    m_phase = Phase::Generating;
    return true;
}

void Session::ensureRoom(size_t nTokens) {
    if (m_params.gaFactor != 1) {
        // context extension via Self-Extend (reference :348-368): whenever a whole group-attention window lies behind gaIndex, its
        // positions are divided by gaFactor and everything after it moves up close -- positions only, the cells stay; the engine
        // re-rotates the K rows by the position change (llama.cpp's K-shift) before the next decode
        const int gaFactor = int(m_params.gaFactor), gaWidth = int(m_params.gaWidth);
        while (int(m_numPast) >= int(m_gaIndex) + gaWidth) {
            const int ib = (gaFactor * int(m_gaIndex)) / gaWidth;
            const int bd = (gaWidth / gaFactor) * (gaFactor - 1);
            const int dd = (gaWidth / gaFactor) - ib * bd - gaWidth;
            logLine(LogLevel::Debug, "Group attention shift: ib = " + std::to_string(ib) + ", bd = " + std::to_string(bd) + ", dd = " + std::to_string(dd));
            throwIfFailed(blk_kv_seq_add(m_ctx, int32_t(m_gaIndex), int32_t(m_numPast), ib * bd), "group attention shift");
            throwIfFailed(blk_kv_seq_div(m_ctx, int32_t(m_gaIndex) + ib * bd, int32_t(m_gaIndex) + ib * bd + gaWidth, gaFactor), "group attention shift");
            throwIfFailed(blk_kv_seq_add(m_ctx, int32_t(m_gaIndex) + ib * bd + gaWidth, int32_t(m_numPast) + ib * bd, dd), "group attention shift");
            m_numPast -= uint32_t(bd);
            m_gaIndex += uint32_t(gaWidth / gaFactor);
            logLine(LogLevel::Info, "Context full mitigation performed: past = " + std::to_string(m_numPast) + ", tokens = " + std::to_string(nTokens));
        }
        return;
    }
    const auto ctxLen = uint32_t(blk_ctx_n_ctx(m_ctx));
    if (m_numPast + nTokens >= ctxLen) {
        // infinite text generation via context shifting (reference :324-347): keep the first numKeep tokens (the initial prompt),
        // drop half of the rest, move what remains down -- blk_kv_shift re-rotates the K rows like llama.cpp's K-shift
        if (!m_params.infiniteContext) Raise{} << "context limit of " << ctxLen << " reached";
        const auto numLeft = m_numPast - m_numKeep;
        const int numDiscard = int(numLeft / 2);
        if (numDiscard <= 0) Raise{} << "context limit of " << ctxLen << " reached";
        logLine(LogLevel::Debug, "Context is full. Swapping: past = " + std::to_string(m_numPast) + ", numLeft: " + std::to_string(numLeft) +
                                     ", ctxLen: " + std::to_string(ctxLen) + ", numKeep: " + std::to_string(m_numKeep) + ", numDiscard: " + std::to_string(numDiscard));
        throwIfFailed(blk_kv_shift(m_ctx, int32_t(m_numKeep), int32_t(m_numKeep) + numDiscard), "context shift");
        m_numPast -= uint32_t(numDiscard);
        logLine(LogLevel::Info, "Context full mitigation performed: past = " + std::to_string(m_numPast) + ", tokens = " + std::to_string(nTokens));
    }
}

void Session::doDecode(std::span<const Token> tokens, Source src) {
    if (tokens.size() > m_maxTokens) {
        const auto skipped = tokens.size() - m_maxTokens;
        tokens = tokens.first(m_maxTokens);
        logLine(LogLevel::Warning, "Input too long. Skipping " + std::to_string(skipped) + " tokens");
    }
    ensureRoom(tokens.size());
    for (auto t : tokens) m_sampler->accept(t, src == Source::Generated);

    if (tokens.size() == 1) {
        m_candidates.resize(size_t(Sampler::MaxDeviceCandidates));
        auto* raw = reinterpret_cast<blk_token_data*>(m_candidates.data());
        // the edits of the history that now ends with this token: with none, exactly the plain decode
        const Sampler::LogitEdits edits = logitEdits();
        m_useEdited = !edits.edits.empty();
        int st;
        if (!m_useEdited) {
            st = blk_decode_topk(m_ctx, tokens[0], Sampler::MaxDeviceCandidates, raw);
        } else {
            const blk_logit_edits e = abiEdits(edits);
            m_edited.resize(size_t(Sampler::MaxDeviceCandidates));
            st = blk_decode_topk_edited(m_ctx, tokens[0], Sampler::MaxDeviceCandidates, &e, raw, reinterpret_cast<blk_token_data*>(m_edited.data()));
        }
        if (st != BLK_OK) Raise{} << "Failed to decode tokens";
        m_numPast += 1;
        m_haveRow = true;
        return;
    }
    const auto batchSize = size_t(blk_ctx_n_batch(m_ctx));
    while (!tokens.empty()) {
        auto batch = tokens.size() > batchSize ? tokens.first(batchSize) : tokens;
        tokens = tokens.subspan(batch.size());
        if (blk_decode(m_ctx, batch.data(), int32_t(batch.size())) != BLK_OK) Raise{} << "Failed to decode tokens";
        m_numPast += uint32_t(batch.size());
    }
    m_haveRow = true;
    refreshCandidates();
}

void Session::flushPendingState() {
    if (m_currToken != Token_Invalid) {
        const Token t = m_currToken;
        m_currToken = Token_Invalid;
        doDecode({&t, 1}, Source::Generated);
    }
}

void Session::resetSampler(const Sampler::Params& params) {
    m_sampler.reset(new Sampler(m_instance.model(), params));
    if (m_phase == Phase::Initial) return;      // no row yet: the first decode selects with the new sampler's edits
    refreshEdited();
}

TokenPrediction Session::StreamGenerator::complete() {
    if (m_session.m_phase != Session::Phase::Streaming || m_status != Status::InProgress) return {Token_Invalid, {}};
    auto p = m_session.getToken();
    if (p.token == Token_Invalid) {
        m_session.m_phase = Session::Phase::Generating;
        m_status = Status::Completed;
        return p;
    }
    m_genTokens++;
    if (m_genTokens >= m_params.maxTokens) {
        m_session.m_phase = Session::Phase::Generating;
        m_status = Status::Completed;
    }
    return p;
}

void Session::StreamGenerator::abort() { m_status = Status::Aborted; }

} // namespace bl::llama
