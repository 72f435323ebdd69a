// Server.hpp -- request-level façade (mirror of reference server/code/server/Server.hpp:17-69).
//
// The reference owns ONE Instance and ONE inference thread (Server.cpp:23-43): requests are serialised.  Requests are
// independent (fresh session + KV clear each), so this build partitions them across GPUs: one full model replica,
// one Instance and one worker thread per GPU, all pulling whole requests from a shared queue.  No collective is
// involved (SURVEY.md section 8e).
#pragma once
#include "../llama/Instance.hpp"
#include "../llama/Sampler.hpp"

#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

namespace bl::llama {
class Model;
namespace server {

class Server {
public:
    explicit Server(std::shared_ptr<Model> model);                      // reference signature: one replica
    explicit Server(std::vector<std::shared_ptr<Model>> replicas);      // one replica per GPU
    // extension: the Instance parameters of every worker (the reference passes {}: KV cache sized for the training context)
    Server(std::vector<std::shared_ptr<Model>> replicas, Instance::InitParams instanceParams);
    // extension (SURVEY.md 8f item 4, continuous batching): every worker keeps up to maxBatch /complete requests in flight and
    // advances them together, one blk_decode_batch step per token (weights streamed once for all of them); requests join and leave
    // between steps.  1 = the reference's behaviour (a worker serves one request at a time, batch-1 decode kernel).  With more than
    // one request in flight a step runs in the bf16 arithmetic of the verify prefill; a lone request runs the batch-1 kernel.
    Server(std::vector<std::shared_ptr<Model>> replicas, Instance::InitParams instanceParams, unsigned maxBatch);
    ~Server();
    Server(const Server&) = delete;
    Server& operator=(const Server&) = delete;

    struct CompleteRequestParams {
        std::string prompt;
        uint32_t maxTokens = 0;
        uint32_t seed = 0;
        std::string suffix;           // parsed by the HTTP layer but never forwarded (reference Server.cpp:53-56)
        float temperature = 0.8f;
        float topP = 0.95f;
        // extension, off by default (the HTTP body does not carry them): the logit-bias and repetition-penalty stages of the
        // reference's sampler chain (Sampler::Params::logitBias / repetitionPenalty), applied through Session::resetSampler
        Sampler::Params::RepetitionPenalty repetitionPenalty;
        std::map<int32_t, float> logitBias;
    };
    struct TokenData {
        std::string tokenStr;
        uint32_t tokenId = 0;
        struct LogitData { uint32_t tokenId = 0; float logit = 0; };
        std::vector<LogitData> logits;
    };
    using CompleteReponse = std::vector<TokenData>;

    // POST /complete (Server.cpp:45-77): tokenize, fresh session on the worker's replica, Session::complete, token strings + top-10
    // per token to the callback (called on the worker thread).
    void completeText(CompleteRequestParams params, std::function<void(CompleteReponse)> cb);
    // POST /verify_completion (Server.cpp:127-161): re-fill the context with the response's tokens (one batched prefill), compare the
    // claimed logits with this replica's through LogitComparer, aggregate with MetricsAggregator; the callback gets the score.
    void verify(CompleteRequestParams req, CompleteReponse resp, std::function<void(float)> cb);

    // extension used by the benchmark harness: prompts given as token ids (no tokenizer on the path)
    void completeTokens(std::vector<int32_t> prompt, CompleteRequestParams params, std::function<void(CompleteReponse)> cb);
    void verifyTokens(std::vector<int32_t> prompt, CompleteRequestParams req, CompleteReponse resp, std::function<void(float)> cb);

    // A request that throws (malformed response, context overflow, ...) terminates the reference process (the exception escapes
    // its io_context, SURVEY.md section 5).  Here the worker survives: the request's callback is still invoked -- with an empty
    // response / a NaN score -- after the handler set here has received the exception text (called on the worker thread).
    void setErrorHandler(std::function<void(const std::string&)> handler);

    // what a worker did, for the dispatcher benchmark: requests served and the CUDA-event time its GPU spent inside them
    struct WorkerStats { int device = 0; uint64_t requests = 0; double gpuMs = 0; };
    std::vector<WorkerStats> workerStats() const;

    size_t workerCount() const noexcept;
    void drain();     // blocks until every queued request has run

private:
    struct Impl;
    std::unique_ptr<Impl> m_impl;
};

} // namespace server
} // namespace bl::llama
