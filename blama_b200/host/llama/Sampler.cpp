// Sampler.cpp -- restatement of the llama.cpp sampler stages blama configures (reference Sampler.cpp:15-97,126-173;
// upstream src/llama-sampling.cpp top_k / top_p / min_p / temp / dist) over a short candidate list.
#include "Sampler.hpp"
#include "Errors.hpp"
#include "Model.hpp"

#include <algorithm>
#include <cmath>

namespace bl::llama {

Sampler::Sampler(Model& /*model*/, const Params& params) : m_params(params), m_rng(params.rngSeed) {
    // stages that need a grammar engine or adapt to the draws are outside the hot path this build covers
    if (!params.grammar.empty()) Raise{} << "grammar-constrained sampling is not supported by this build";
    if (params.mirostat.ver != 0) {
        if (params.mirostat.ver > 2) throw std::runtime_error("Unsupported mirostat version");
        Raise{} << "mirostat sampling is not supported by this build";
    }
    // -inf bans an id; NaN and +inf would poison the row (the reference passes them through unchecked)
    for (const auto& [id, bias] : params.logitBias)
        if (std::isnan(bias) || bias == INFINITY) Raise{} << "logit bias of token " << id << " must not be NaN or +inf";
    const auto& rp = params.repetitionPenalty;
    if (!(rp.repeat == 1.0f && rp.freq == 0.0f && rp.present == 0.0f)) {
        // whether llama_sampler_init_penalties clamps a negative window to 0 could not be confirmed, so it is refused
        if (rp.numTokens < 0) Raise{} << "repetition penalty window must not be negative, got " << rp.numTokens;
        if (!(std::isfinite(rp.repeat) && rp.repeat > 0.0f) || !std::isfinite(rp.freq) || !std::isfinite(rp.present))
            Raise{} << "repetition penalties must be finite, and the repeat penalty > 0";
    }
    for (auto t : params.samplerSequence)
        if (t == SamplingType::XTC || t == SamplingType::Infill) throw std::runtime_error("Unsupported sampler type");
    if (params.typicalP < 1.0f) Raise{} << "typical sampling is not supported by this build";
    if (params.tempRange > 0.0f) Raise{} << "dynamic temperature is not supported by this build";
}

Sampler::~Sampler() = default;

void Sampler::reset() {
    m_rng.seed(m_params.rngSeed);
    m_prev.clear();
    m_counts.clear();
}

void Sampler::accept(Token id, bool) {
    const int32_t window = m_params.repetitionPenalty.numTokens;
    if (window <= 0) return;
    m_counts[id]++;
    if (m_prev.size() >= size_t(window)) {
        const Token old = m_prev.front();
        m_prev.pop_front();
        if (--m_counts[old] == 0) m_counts.erase(old);
    }
    m_prev.push_back(id);
}

bool Sampler::penaltiesActive() const noexcept {
    const auto& rp = m_params.repetitionPenalty;
    return rp.numTokens > 0 && !(rp.repeat == 1.0f && rp.freq == 0.0f && rp.present == 0.0f);
}

Sampler::LogitEdits Sampler::logitEdits(int32_t nVocab) const {
    LogitEdits out;
    const bool penalties = penaltiesActive();
    if (penalties) {
        out.repeat = m_params.repetitionPenalty.repeat;
        out.freq = m_params.repetitionPenalty.freq;
        out.present = m_params.repetitionPenalty.present;
    }
    // both maps are ordered by id: merge them
    auto b = m_params.logitBias.lower_bound(0);
    auto c = penalties ? m_counts.lower_bound(0) : m_counts.end();
    const auto bEnd = m_params.logitBias.lower_bound(nVocab);
    const auto cEnd = penalties ? m_counts.lower_bound(nVocab) : m_counts.end();
    while (b != bEnd || c != cEnd) {
        const Token id = (c == cEnd || (b != bEnd && b->first < c->first)) ? b->first : c->first;
        LogitEdit e{id, 0, 0.0f};
        if (b != bEnd && b->first == id) { e.bias = b->second; ++b; }
        if (c != cEnd && c->first == id) { e.count = c->second; ++c; }
        if (e.bias != 0.0f || e.count > 0) out.edits.push_back(e);
    }
    return out;
}

float Sampler::editLogit(float logit, int32_t count, float bias, float repeat, float freq, float present) {
    if (bias != 0.0f) logit += bias;
    if (count > 0) {
        logit = logit <= 0.0f ? logit * repeat : logit / repeat;
        logit -= float(count) * freq + present;
    }
    return logit;
}

void Sampler::applyEdits(std::span<float> row) const {
    const LogitEdits e = logitEdits(int32_t(row.size()));
    for (const auto& d : e.edits) row[size_t(d.token)] = editLogit(row[size_t(d.token)], d.count, d.bias, e.repeat, e.freq, e.present);
}

int32_t Sampler::candidatesNeeded() const noexcept {
    const bool hasTopK = std::find(m_params.samplerSequence.begin(), m_params.samplerSequence.end(), SamplingType::Top_K) != m_params.samplerSequence.end()
                         && m_params.samplerSequence.front() == SamplingType::Top_K;
    if (!hasTopK || m_params.topK <= 0 || m_params.topK > MaxDeviceCandidates) return 0;
    return m_params.topK;
}

// llama_sampler_softmax_impl: sort descending if needed, p = exp(logit - max) / sum
void Sampler::softmax(size_t size, bool& sorted) {
    if (!sorted) {
        std::sort(m_cur.begin(), m_cur.begin() + size, [](const Cand& a, const Cand& b) { return a.logit > b.logit; });
        sorted = true;
    }
    const float maxLogit = m_cur[0].logit;
    float cum = 0.0f;
    for (size_t i = 0; i < size; ++i) {
        const float p = expf(m_cur[i].logit - maxLogit);
        m_cur[i].p = p;
        cum += p;
    }
    for (size_t i = 0; i < size; ++i) m_cur[i].p /= cum;
}

Token Sampler::sample(std::span<const TokenData> candidates, bool sorted) {
    if (candidates.empty()) throw std::runtime_error("no selected token during sampling - check your sampling configuration");
    m_cur.resize(candidates.size());
    for (size_t i = 0; i < candidates.size(); ++i) m_cur[i] = {candidates[i].token, candidates[i].logit, 0.0f};
    size_t size = m_cur.size();
    const size_t minKeep = size_t(m_params.minKeep);

    for (auto stage : m_params.samplerSequence) {
        switch (stage) {
        case SamplingType::Top_K: {
            int k = m_params.topK;
            if (k <= 0) k = int(size);
            k = std::min(k, int(size));
            if (!sorted) {
                std::partial_sort(m_cur.begin(), m_cur.begin() + k, m_cur.begin() + size,
                                  [](const Cand& a, const Cand& b) { return a.logit > b.logit; });
                sorted = true;
            }
            size = size_t(k);
            break;
        }
        case SamplingType::Typical_P:
            break;                       // p >= 1: llama_sampler_typical_apply returns immediately
        case SamplingType::Top_P: {
            if (m_params.topP >= 1.0f) break;
            softmax(size, sorted);
            float cum = 0.0f;
            size_t last = size;
            for (size_t i = 0; i < size; ++i) {
                cum += m_cur[i].p;
                if (cum >= m_params.topP && i + 1 >= minKeep) { last = i + 1; break; }
            }
            size = last;
            break;
        }
        case SamplingType::Min_P: {
            if (m_params.minP <= 0.0f || size == 0) break;
            bool applied = false;
            if (!sorted) {               // unsorted branch of llama_sampler_min_p_apply
                float maxLogit = -INFINITY;
                for (size_t i = 0; i < size; ++i) maxLogit = std::max(maxLogit, m_cur[i].logit);
                const float minLogit = maxLogit + logf(m_params.minP);
                std::vector<Cand> kept;
                for (size_t i = 0; i < size; ++i) if (m_cur[i].logit >= minLogit) kept.push_back(m_cur[i]);
                if (!kept.empty() && kept.size() >= minKeep) {
                    std::copy(kept.begin(), kept.end(), m_cur.begin());
                    size = kept.size();
                    applied = true;
                }
            }
            if (!applied) {
                if (!sorted) {
                    std::sort(m_cur.begin(), m_cur.begin() + size, [](const Cand& a, const Cand& b) { return a.logit > b.logit; });
                    sorted = true;
                }
                const float minLogit = m_cur[0].logit + logf(m_params.minP);
                size_t i = 1;
                for (; i < size; ++i) if (m_cur[i].logit < minLogit && i >= minKeep) break;
                size = i;
            }
            break;
        }
        case SamplingType::Temperature: {
            if (m_params.temp <= 0.0f) {     // greedy: keep only the arg-max alive
                size_t best = 0;
                for (size_t i = 1; i < size; ++i) if (m_cur[i].logit > m_cur[best].logit) best = i;
                for (size_t i = 0; i < size; ++i) if (i != best) m_cur[i].logit = -INFINITY;
            } else {
                for (size_t i = 0; i < size; ++i) m_cur[i].logit /= m_params.temp;
            }
            break;
        }
        default:
            throw std::runtime_error("Unsupported sampler type");
        }
    }

    // dist: softmax then one draw of std::discrete_distribution (llama_sample_dist)
    softmax(size, sorted);
    std::vector<double> probs(size);
    for (size_t i = 0; i < size; ++i) probs[i] = m_cur[i].p;
    std::discrete_distribution<int> dist(probs.begin(), probs.end());
    return m_cur[size_t(dist(m_rng))].id;
}

} // namespace bl::llama
