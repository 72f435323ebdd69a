// Session.hpp -- per-request state machine (mirror of reference inference/code/llama/Session.hpp:29-137).
//
// Same public surface and error strings as the reference; underneath, every llama.cpp call is replaced by the C ABI:
//   llama_decode(1 token) + llama_get_logits_ith + host sort   ->  blk_decode_topk (one graph launch, 512 B back)
//   fillCtx's N single-token decodes + V-long host gather     ->  blk_verify_prefill (one causal prefill)
#pragma once
#include "Sampler.hpp"
#include "Token.hpp"

#include <blama_b200.h>

#include <memory>
#include <span>
#include <string>
#include <vector>

namespace bl::llama {

class Instance;

// a sampler's edit list as the C ABI takes it (valid while `e` lives)
inline blk_logit_edits abiEdits(const Sampler::LogitEdits& e) {
    static_assert(sizeof(Sampler::LogitEdit) == sizeof(blk_logit_edit));
    return {e.repeat, e.freq, e.present, reinterpret_cast<const blk_logit_edit*>(e.edits.data()), int32_t(e.edits.size())};
}

struct TokenPrediction {
    Token token;
    TokenDataVector logits;      // top-10 {id, logit} of the distribution AFTER `token` was decoded
    operator bool() const { return token != Token_Invalid; }
};

class Session {
public:
    struct InitParams {
        uint32_t gaFactor = 1;          // group-attention (Self-Extend) factor
        uint32_t gaWidth = 512;         // group-attention width (a multiple of gaFactor)
        bool infiniteContext = true;    // a full context drops half of the non-prompt past and shifts the rest (false: throws)
        uint32_t seed = 0;
        std::string grammar;
        float temperature = 0.80f;
        float topP = 0.95f;
        // extension: false = fillCtx runs one causal prefill (fast, fp tolerance); true = N single-token decodes,
        // bit-identical to complete() (what the reference does, t-integration.cpp:219-248)
        bool sequentialVerify = false;
    };

    Session(Instance& instance, blk_ctx* ctx, InitParams params);
    Session(const Session&) = delete;
    Session& operator=(const Session&) = delete;
    ~Session();

    // Prompt prefill (Session.cpp:65-107): BOS is prepended when the model asks for it; >= BLK_PREFILL_MIN tokens take the tcgen05
    // prefill path, the last position's logits come from the decode mat-vec.  Throws "Session already started" /
    // "Initial prompt too long. Got N tokens, max: M" with the reference's texts.
    void setInitialPrompt(std::span<const Token> prompt);
    // Context save / restore (Session.cpp:284-310): the KV rows, the pending logits and their top-k as one blob; the sampler's
    // RNG is not part of it (as in the reference).  Same state checks and texts ("Session already started" / "Session hasn't
    // started yet" / "Failed to set state").
    bool setState(std::span<uint8_t> state);

    struct CompleteParams {
        std::span<const Token> prompt;
        std::span<const Token> suffix;
        int32_t maxTokens = 0;
    };
    // The /complete loop (Session.cpp:192-213): one persistent-kernel launch per token (blk_decode_topk), the sampler chain on
    // the 64 device candidates, top-10 of the NEXT distribution attached to every token; stops at an end-of-generation token.
    std::vector<TokenPrediction> complete(CompleteParams params);

    class StreamGenerator {
    public:
        enum class Status { InProgress, Completed, Aborted };
        StreamGenerator(Session& session, CompleteParams params)
            : m_session(session), m_params(params), m_genTokens(0), m_status(Status::InProgress) {}
        TokenPrediction complete();
        void abort();
        Status status() const { return m_status; }
    private:
        Session& m_session;
        CompleteParams m_params;
        int32_t m_genTokens;
        Status m_status;
    };
    // Token-at-a-time form of complete() (Session.cpp:215-229, 407-432); only one generator may be active.
    StreamGenerator completeStream(CompleteParams params);

    // The /verify_completion context fill (Session.cpp:231-244): decodes the claimed tokens and returns, per position, this
    // model's logits at the claimed ids sorted by logit.  ONE causal prefill here (or N single-token decodes when
    // InitParams::sequentialVerify is set: bit-identical to complete()).
    std::vector<TokenPrediction> fillCtx(std::span<TokenPrediction> tokens);
    // Extension for Server::verify: setInitialPrompt(prompt) followed by fillCtx(tokens) as ONE causal prefill over [prompt | response]
    // (a short prompt run on its own streams every weight once for a handful of tokens: 7 ms of a 35 ms request on the 8B model).
    // Same checks, texts and results layout as the two calls; falls back to them whenever fillCtx itself would not batch.
    std::vector<TokenPrediction> setInitialPromptAndFill(std::span<const Token> prompt, std::span<TokenPrediction> tokens);
    // Extension for a batching server (SURVEY.md 8f item 4): the two halves of getToken() around a decode that somebody else runs
    // for several sessions at once (blk_decode_batch).  sampleNext() draws from the current distribution (Token_Invalid at an
    // end-of-generation token; shifts the context first when it is full, like doDecode); acceptDecoded() records that `token` has
    // been decoded into this session's cache and installs the new distribution's top-k.  Returns what getToken() would have.
    // sampleNext() also accepts the drawn token into the sampler (as the reference does right before decoding it), so that
    // logitEdits() then describes the edits of the row the decode produces: with logit bias or penalties active the batch runs
    // blk_decode_batch_edited and acceptDecoded receives that row's edited top-k as well (empty = the raw list is sampled).
    Token sampleNext();
    TokenPrediction acceptDecoded(Token token, std::span<const TokenData> candidates, std::span<const TokenData> edited = {});
    Sampler::LogitEdits logitEdits() const;
    // what the next draw samples from: the device top-k of the current row after the sampler's edits (the raw top-k without any)
    std::span<const TokenData> samplingCandidates() const;
    std::vector<uint8_t> getState();
    // New sampler chain for the rest of the session (Session.cpp:403-405); the KV cache is kept.  With logit bias active the edited
    // top-k of the current row is recomputed, which needs that row: after a batched step (acceptDecoded) it is gone and this throws.
    void resetSampler(const Sampler::Params& params);

private:
    friend class StreamGenerator;
    enum class Source { InitialPrompt, InteractivePrompt, Generated };
    enum class Phase { Initial, Generating, Streaming };

    void pushPrompt(std::span<const Token> prompt, std::span<const Token> postfix = {});
    TokenPrediction getToken();
    void doDecode(std::span<const Token> tokens, Source src);
    void ensureRoom(size_t nTokens);      // context shift when nTokens more do not fit (reference :324-347)
    void flushPendingState();
    TokenDataVector getLogitsFromCtx(int32_t topK);
    TokenDataVector getLogitsFromCtx(TokenDataVector tokens);
    void requireStarted(bool allowStreaming) const;
    void refreshCandidates();
    void refreshEdited();
    int32_t nVocab() const;

    Instance& m_instance;
    blk_ctx* m_ctx;
    std::unique_ptr<Sampler> m_sampler;
    InitParams m_params;

    Phase m_phase = Phase::Initial;
    Token m_currToken = Token_Invalid;      // sampled but not yet decoded
    unsigned m_maxTokens = 0;
    unsigned m_numKeep = 0;
    uint32_t m_numPast = 0;                 // position of the next token (= cells in the cache unless Self-Extend regrouped positions)
    uint32_t m_gaIndex = 0;                 // number of grouped KV tokens (only used if gaFactor > 1)
    TokenDataVector m_candidates;           // device top-k of the current logits, descending (what is reported)
    TokenDataVector m_edited;               // device top-k of the current logits after logit bias + penalties (what is sampled)
    bool m_useEdited = false;               // m_edited is current: the sampler had edits for the current row
    bool m_haveRow = false;                 // the context keeps the current logits row (not after a batched step)
};

} // namespace bl::llama
