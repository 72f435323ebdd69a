// Sampler.hpp -- host-side sampler chain (mirror of reference inference/code/llama/Sampler.hpp:22-115).
//
// The reference builds a llama.cpp chain: logit-bias -> penalties -> top-k 40 -> typical -> top-p -> min-p -> temp ->
// dist(seed) (Sampler.cpp:30-95) and feeds it all n_vocab logits (Sampler.cpp:110-123: a 513 KB device->host copy and
// a 1.5 MB host fill per token).  Because the chain STARTS with top-k, nothing outside the k best logits can influence
// the draw while bias and penalties are at their defaults; this implementation therefore consumes the device's
// top-k list (<= 64 entries, already sorted) and restates the remaining stages exactly: same float operations,
// std::discrete_distribution over std::mt19937 as llama-sampling.cpp's llama_sample_dist.
// The two stages ahead of top-k (logit bias, repetition penalties) are handed to the device as an edit list (logitEdits):
// it applies them to a copy of the row and selects that copy's top-k, so the shortcut stays exact with them active.
#pragma once
#include "Token.hpp"

#include <deque>
#include <map>
#include <random>
#include <span>
#include <string>
#include <vector>

namespace bl::llama {

class Model;

class Sampler {
public:
    enum class SamplingType { Top_K, Top_P, Min_P, Typical_P, Temperature, XTC, Infill };

    struct Params {
        uint32_t rngSeed = 0;
        int32_t minKeep = 0;
        int32_t topK = 40;        // <= 0 to use vocab size
        float topP = 0.95f;       // 1.0 = disabled
        float minP = 0.05f;       // 0.0 = disabled
        float tfsZ = 1.00f;
        float typicalP = 1.00f;   // 1.0 = disabled
        float temp = 0.80f;       // <= 0.0 to sample greedily
        float tempRange = 0.00f;
        float tempExp = 1.00f;
        struct RepetitionPenalty { int32_t numTokens = 64; float repeat = 1.00f; float freq = 0.00f; float present = 0.00f; } repetitionPenalty;
        struct Mirostat { int32_t ver = 0; float tau = 5.00f; float eta = 0.10f; } mirostat;
        struct XTC { float probability = 0.00f; float threshold = 0.10f; } xtc;
        std::vector<SamplingType> samplerSequence = {SamplingType::Top_K, SamplingType::Typical_P, SamplingType::Top_P,
                                                     SamplingType::Min_P, SamplingType::Temperature};
        std::string grammar;
        std::map<Token, float> logitBias;
    };

    // largest candidate list the device hands over in one decode (blk_decode_topk)
    static constexpr int32_t MaxDeviceCandidates = 64;

    explicit Sampler(Model& model, const Params& params);
    ~Sampler();
    Sampler(const Sampler&) = delete;
    Sampler& operator=(const Sampler&) = delete;

    // One edited id of the logit-bias + penalties stages (layout of blk_logit_edit): logit += bias (when bias != 0), then with
    // count > 0 the repetition penalty of an id seen count times in the window.
    struct LogitEdit { Token token; int32_t count; float bias; };
    struct LogitEdits { float repeat = 1.0f, freq = 0.0f, present = 0.0f; std::vector<LogitEdit> edits; };

    void reset();        // re-seeds the RNG and empties the penalty window (llama_sampler_reset on every stage of the chain)
    void perfReset() {}

    // how many of the best logits sample() needs (top-k clipped to the device limit; 0 = the whole vocabulary)
    int32_t candidatesNeeded() const noexcept;
    // draw from candidates sorted by logit descending (the device's top-k list, or the whole vocabulary sorted/unsorted)
    Token sample(std::span<const TokenData> candidates, bool sorted = true);
    // pushes id into the penalty window of the last repetitionPenalty.numTokens accepted ids (llama_sampler_penalties_accept)
    void accept(Token id, bool acceptGrammar);

    // The bias map merged with the window's counts, one entry per id in [0, nVocab), ascending: what the two stages change in
    // a logits row (empty = they change nothing).  Window counts are left out while the penalty stage is a no-op.
    LogitEdits logitEdits(int32_t nVocab) const;
    // the two stages applied to a whole row of nVocab logits (the full-row path: candidatesNeeded() == 0)
    void applyEdits(std::span<float> row) const;
    // one edited logit, in the float operations llama.cpp uses (the device's edit kernel repeats them bit for bit)
    static float editLogit(float logit, int32_t count, float bias, float repeat, float freq, float present);

private:
    struct Cand { Token id; float logit; float p; };
    void softmax(size_t size, bool& sorted);
    bool penaltiesActive() const noexcept;
    Params m_params;
    std::mt19937 m_rng;
    std::vector<Cand> m_cur;
    std::deque<Token> m_prev;           // penalty window, oldest first
    std::map<Token, int32_t> m_counts;  // occurrences of every id in m_prev
};

} // namespace bl::llama
