// pool.cu — the utterance-batching scheduler across the GPUs of one box.
//
// The reference has no batching layer: `speech transcribe-batch` is a serial loop over files
// (/root/reference/Sources/AudioCLILib/TranscribeBatchCommand.swift:82-125).  Here every utterance is an
// independent unit (transcribe builds a fresh cache per call, Qwen3ASR.swift:246-251), so the pool
// replicates the weights on each GPU, deals utterances longest-processing-time-first to the least loaded
// GPU, lets one worker thread per GPU run its share in length-sorted sub-batches, and gathers the ids on
// the host.  No collective touches the data path.
#include <algorithm>
#include <atomic>
#include <mutex>
#include <numeric>
#include <thread>

#include "model.h"

using namespace q3;

struct q3asr_pool {
    std::vector<q3asr_handle*> handles;
    std::string last_error;
    std::mutex run_mu;  // one batch at a time on the pool's handles (submitted jobs queue on it in submission order of their threads)
    std::atomic<int> continuous{0};  // q3asr_pool_set_continuous: each worker's share runs as one continuous batch
};

// an asynchronous q3asr_pool_transcribe_ids_opts call: the worker thread owns the result buffers until q3asr_job_wait copies them out
struct q3asr_job {
    std::thread worker;
    std::atomic<int> done{0};
    int rc = Q3ASR_OK;
    int batch = 0, max_tokens = 0;
    std::vector<int32_t> ids;
    std::vector<int> lens;
    std::vector<q3asr_prompt> prompts;
    std::vector<int> rates;
    bool has_sampling = false;
    q3asr_sampling sampling{};
    bool has_lp = false;     // submitted through q3asr_pool_submit_lp
    bool waited = false;     // q3asr_job_wait returned Q3ASR_OK
    std::vector<float> lp;   // [batch, max_tokens] log-probabilities (has_lp only)
    std::string error;
};

namespace {
thread_local std::string g_create_error;  // q3asr_pool_last_error(NULL): why the last q3asr_pool_create on this thread failed

// the continuous schedule is greedy only (the sampler indexes generated ids by row and keys its noise by slot)
bool greedy_sampling(const q3asr_sampling* s) {
    return s == nullptr || (s->repetition_penalty == 1.0f && s->no_repeat_ngram_size == 0 && s->temperature == 0.0f && s->force_device_sampler == 0);
}

// One batch over the pool's handles (arguments checked by the caller, p->run_mu held).  May throw from its own host allocations or
// thread creation; workers already started are joined first.
int pool_run(q3asr_pool* p, const float* const* pcm, const size_t* n_in, const int* sample_rates, int batch, const q3asr_prompt* prompts,
             const q3asr_sampling* sampling, int max_tokens, int stop_on_eos, int max_batch_per_gpu, int32_t* ids_out, int* lens_out,
             float* lp_out) {
    const int G = (int)p->handles.size();
    if (max_batch_per_gpu <= 0) max_batch_per_gpu = 256;  // the widest batch the weight-streaming decode kernels take (512 x 30 s on one GPU, two workers: 11 460 audio-s/s against 10 840 at 128 and 9 390 at 64)
    // the scheduler's cost model and the length sort work on 16 kHz-equivalent lengths
    std::vector<size_t> n16(n_in, n_in + batch);
    if (sample_rates)
        for (int i = 0; i < batch; i++) n16[i] = q3asr_resample_len(n_in[i], sample_rates[i], 16000);
    const size_t* n_samples = n16.data();
    std::vector<int> gpu(batch);
    q3asr_schedule(n_samples, batch, G, gpu.data());
    std::vector<int> rc(G, Q3ASR_OK);
    std::vector<std::string> host_err(G);  // failures of the worker's own host code (the handle keeps the message of a failed call)
    const bool continuous = p->continuous.load() != 0;
    auto work = [&](int g) {
        try {  // nothing may escape a std::thread
            std::vector<int> mine;
            for (int i = 0; i < batch; i++)
                if (gpu[i] == g) mine.push_back(i);
            // similar lengths together: prefill rows and decode steps stay homogeneous
            std::stable_sort(mine.begin(), mine.end(), [&](int a, int b) { return n_samples[a] > n_samples[b]; });
            // continuous: the whole share is one request, max_batch_per_gpu rows resident at a time
            const size_t step = continuous ? std::max<size_t>(mine.size(), 1) : (size_t)max_batch_per_gpu;
            for (size_t s = 0; s < mine.size(); s += step) {
                const int nb = (int)std::min<size_t>(step, mine.size() - s);
                std::vector<const float*> pp(nb);
                std::vector<size_t> nn(nb);
                std::vector<int> rr(nb, 16000);
                std::vector<q3asr_prompt> pr(nb);
                for (int j = 0; j < nb; j++) {
                    pp[j] = pcm[mine[s + j]];
                    nn[j] = n_in[mine[s + j]];
                    if (sample_rates) rr[j] = sample_rates[mine[s + j]];
                    if (prompts) pr[j] = prompts[mine[s + j]];
                }
                std::vector<int32_t> ids((size_t)nb * max_tokens);
                std::vector<int> lens(nb);
                std::vector<float> lp(lp_out ? (size_t)nb * max_tokens : 0);
                if (continuous)
                    rc[g] = q3asr_transcribe_ids_continuous(p->handles[g], pp.data(), nn.data(), sample_rates ? rr.data() : nullptr, nb,
                                                            prompts ? pr.data() : nullptr, max_tokens, stop_on_eos, max_batch_per_gpu,
                                                            ids.data(), lens.data(), lp_out ? lp.data() : nullptr);
                else
                    rc[g] = q3asr_transcribe_ids_lp(p->handles[g], pp.data(), nn.data(), sample_rates ? rr.data() : nullptr, nb,
                                                    prompts ? pr.data() : nullptr, sampling, max_tokens, stop_on_eos, ids.data(), lens.data(),
                                                    lp_out ? lp.data() : nullptr);
                if (rc[g] != Q3ASR_OK) break;
                for (int j = 0; j < nb; j++) {  // host-side result gather, original order
                    const int i = mine[s + j];
                    lens_out[i] = lens[j];
                    std::copy(ids.begin() + (size_t)j * max_tokens, ids.begin() + (size_t)j * max_tokens + lens[j],
                              ids_out + (size_t)i * max_tokens);
                    if (lp_out)  // the whole row: the entries past lens[j] are zeros
                        std::copy(lp.begin() + (size_t)j * max_tokens, lp.begin() + (size_t)(j + 1) * max_tokens, lp_out + (size_t)i * max_tokens);
                }
            }
        } catch (const std::bad_alloc&) {
            rc[g] = Q3ASR_ERR_NOMEM;
            host_err[g] = "out of host memory";
        } catch (const std::exception& e) {
            rc[g] = Q3ASR_ERR_STATE;
            host_err[g] = e.what();
        }
    };
    std::vector<std::thread> workers;
    workers.reserve(G);
    try {
        for (int g = 0; g < G; g++) workers.emplace_back(work, g);
    } catch (...) {
        for (auto& t : workers) t.join();
        throw;
    }
    for (auto& t : workers) t.join();
    for (int g = 0; g < G; g++)
        if (rc[g] != Q3ASR_OK) {
            p->last_error = std::string("gpu worker ") + std::to_string(g) + ": " +
                            (host_err[g].empty() ? q3asr_last_error(p->handles[g]) : host_err[g].c_str());
            return rc[g];
        }
    return Q3ASR_OK;
}

int pool_transcribe_locked(q3asr_pool* p, const float* const* pcm, const size_t* n_in, const int* sample_rates, int batch,
                           const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos,
                           int max_batch_per_gpu, int32_t* ids_out, int* lens_out, float* lp_out) {
    if (pcm == nullptr || n_in == nullptr || ids_out == nullptr || lens_out == nullptr || batch <= 0 || max_tokens <= 0) {
        p->last_error = "pool_transcribe: null argument, empty batch or max_tokens <= 0";
        return Q3ASR_ERR_INVALID;
    }
    if (sample_rates)
        for (int i = 0; i < batch; i++)
            if (sample_rates[i] <= 0) {
                p->last_error = "pool_transcribe: sample rate <= 0";
                return Q3ASR_ERR_INVALID;
            }
    if (p->continuous.load() && !greedy_sampling(sampling)) {
        p->last_error = "pool_transcribe: a continuous pool decodes greedily only (no decoder knobs)";
        return Q3ASR_ERR_INVALID;
    }
    try {
        return pool_run(p, pcm, n_in, sample_rates, batch, prompts, sampling, max_tokens, stop_on_eos, max_batch_per_gpu, ids_out, lens_out,
                        lp_out);
    } catch (const std::bad_alloc&) {
        p->last_error = "pool_transcribe: out of host memory";
        return Q3ASR_ERR_NOMEM;
    } catch (const std::exception& e) {  // std::system_error: no thread to be had
        p->last_error = std::string("pool_transcribe: ") + e.what();
        return Q3ASR_ERR_STATE;
    }
}

// The blocking call; *err (may be NULL) receives the message of a failure while the pool is still locked, so a job's message cannot be
// overwritten by the next job's.
int pool_transcribe(q3asr_pool* p, const float* const* pcm, const size_t* n_in, const int* sample_rates, int batch,
                    const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos, int max_batch_per_gpu,
                    int32_t* ids_out, int* lens_out, float* lp_out, std::string* err) {
    if (p == nullptr) return Q3ASR_ERR_INVALID;
    std::lock_guard<std::mutex> run_lock(p->run_mu);
    const int rc = pool_transcribe_locked(p, pcm, n_in, sample_rates, batch, prompts, sampling, max_tokens, stop_on_eos, max_batch_per_gpu,
                                          ids_out, lens_out, lp_out);
    if (rc != Q3ASR_OK && err) *err = p->last_error;
    return rc;
}
}  // namespace

extern "C" {

int q3asr_schedule(const size_t* n_samples, int batch, int n_gpus, int* gpu_out) {
    if (n_samples == nullptr || gpu_out == nullptr || batch < 0 || n_gpus <= 0) return Q3ASR_ERR_INVALID;
    std::vector<int> order(batch);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return n_samples[a] > n_samples[b]; });
    std::vector<unsigned long long> load(n_gpus, 0);
    for (int i : order) {
        int best = 0;
        for (int g = 1; g < n_gpus; g++)
            if (load[g] < load[best]) best = g;
        gpu_out[i] = best;
        // cost model: encoder/prefill/decode work all grow with the audio length; the constant stands for
        // the fixed prompt and decode cost of an utterance
        load[best] += (unsigned long long)n_samples[i] + 16000ull;
    }
    return Q3ASR_OK;
}

int q3asr_pool_create(const q3asr_config* cfg, const int* devices, int n_devices, uint64_t random_seed, const char* weights_dir,
                      q3asr_pool** out) {
    if (out) *out = nullptr;
    if (cfg == nullptr || devices == nullptr || n_devices <= 0 || out == nullptr) {
        g_create_error = "pool_create: null argument or no devices";
        return Q3ASR_ERR_INVALID;
    }
    q3asr_pool* p = new q3asr_pool();
    for (int i = 0; i < n_devices; i++) {
        q3asr_handle* h = nullptr;
        int rc = q3asr_create(cfg, devices[i], &h);
        if (rc == Q3ASR_OK) rc = weights_dir ? q3asr_load_safetensors(h, weights_dir) : q3asr_init_random(h, random_seed);
        if (rc != Q3ASR_OK) {
            g_create_error = std::string("device ") + std::to_string(devices[i]) + ": " + q3asr_last_error(h);
            if (h) q3asr_destroy(h);
            q3asr_pool_destroy(p);
            return rc;
        }
        p->handles.push_back(h);
    }
    *out = p;
    return Q3ASR_OK;
}

void q3asr_pool_destroy(q3asr_pool* p) {
    if (p == nullptr) return;
    for (q3asr_handle* h : p->handles) q3asr_destroy(h);
    delete p;
}

int q3asr_pool_set_continuous(q3asr_pool* p, int enable) {
    if (p == nullptr) return Q3ASR_ERR_INVALID;
    std::lock_guard<std::mutex> run_lock(p->run_mu);  // not in the middle of a batch
    p->continuous.store(enable != 0 ? 1 : 0);
    return Q3ASR_OK;
}

const char* q3asr_pool_last_error(const q3asr_pool* p) { return p ? p->last_error.c_str() : g_create_error.c_str(); }

int q3asr_pool_transcribe_ids(q3asr_pool* p, const float* const* pcm, const size_t* n_samples, int batch, const q3asr_prompt* prompts,
                              int max_tokens, int stop_on_eos, int max_batch_per_gpu, int32_t* ids_out, int* lens_out) {
    return q3asr_pool_transcribe_ids_opts(p, pcm, n_samples, nullptr, batch, prompts, nullptr, max_tokens, stop_on_eos, max_batch_per_gpu,
                                          ids_out, lens_out);
}

int q3asr_pool_transcribe_ids_opts(q3asr_pool* p, const float* const* pcm, const size_t* n_in, const int* sample_rates, int batch,
                                   const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos,
                                   int max_batch_per_gpu, int32_t* ids_out, int* lens_out) {
    return pool_transcribe(p, pcm, n_in, sample_rates, batch, prompts, sampling, max_tokens, stop_on_eos, max_batch_per_gpu, ids_out, lens_out,
                           nullptr, nullptr);
}

int q3asr_pool_transcribe_ids_lp(q3asr_pool* p, const float* const* pcm, const size_t* n_in, const int* sample_rates, int batch,
                                 const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos,
                                 int max_batch_per_gpu, int32_t* ids_out, int* lens_out, float* logprobs_out) {
    return pool_transcribe(p, pcm, n_in, sample_rates, batch, prompts, sampling, max_tokens, stop_on_eos, max_batch_per_gpu, ids_out, lens_out,
                           logprobs_out, nullptr);
}

// ---- submit / wait: the blocking call on a thread of its own, so the caller can load the next files meanwhile (SURVEY.md 8b) ----
namespace {
int pool_submit(q3asr_pool* p, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch, const q3asr_prompt* prompts,
                const q3asr_sampling* sampling, int max_tokens, int stop_on_eos, int max_batch_per_gpu, bool want_lp, q3asr_job** out) {
    if (out) *out = nullptr;
    if (p == nullptr || pcm == nullptr || n_samples == nullptr || batch <= 0 || max_tokens <= 0 || out == nullptr) return Q3ASR_ERR_INVALID;
    if (p->continuous.load() && !greedy_sampling(sampling)) return Q3ASR_ERR_INVALID;  // (see pool_transcribe_locked)
    q3asr_job* j = nullptr;
    try {
        j = new q3asr_job();
        j->batch = batch;
        j->max_tokens = max_tokens;
        j->ids.assign((size_t)batch * max_tokens, 0);
        j->lens.assign((size_t)batch, 0);
        j->has_lp = want_lp;
        if (want_lp) j->lp.assign((size_t)batch * max_tokens, 0.f);
        if (prompts) j->prompts.assign(prompts, prompts + batch);  // the id arrays they point to stay the caller's, like the samples
        if (sample_rates) j->rates.assign(sample_rates, sample_rates + batch);
        if (sampling) {
            j->has_sampling = true;
            j->sampling = *sampling;
        }
        std::vector<const float*> pp(pcm, pcm + batch);
        std::vector<size_t> nn(n_samples, n_samples + batch);
        // starting the worker is the last thing that can throw: on failure the job is still this thread's alone
        j->worker = std::thread([p, j, pp = std::move(pp), nn = std::move(nn), stop_on_eos, max_batch_per_gpu]() {
            j->rc = pool_transcribe(p, pp.data(), nn.data(), j->rates.empty() ? nullptr : j->rates.data(), j->batch,
                                    j->prompts.empty() ? nullptr : j->prompts.data(), j->has_sampling ? &j->sampling : nullptr,
                                    j->max_tokens, stop_on_eos, max_batch_per_gpu, j->ids.data(), j->lens.data(),
                                    j->has_lp ? j->lp.data() : nullptr, &j->error);
            j->done.store(1, std::memory_order_release);
        });
    } catch (const std::exception&) {  // bad_alloc for the result buffers, or no thread to be had
        delete j;
        return Q3ASR_ERR_NOMEM;
    }
    *out = j;
    return Q3ASR_OK;
}
}  // namespace

int q3asr_pool_submit(q3asr_pool* p, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                      const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos, int max_batch_per_gpu,
                      q3asr_job** out) {
    return pool_submit(p, pcm, n_samples, sample_rates, batch, prompts, sampling, max_tokens, stop_on_eos, max_batch_per_gpu, false, out);
}
int q3asr_pool_submit_lp(q3asr_pool* p, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                         const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos, int max_batch_per_gpu,
                         q3asr_job** out) {
    return pool_submit(p, pcm, n_samples, sample_rates, batch, prompts, sampling, max_tokens, stop_on_eos, max_batch_per_gpu, true, out);
}

int q3asr_job_done(const q3asr_job* j) { return j != nullptr && j->done.load(std::memory_order_acquire) != 0; }

int q3asr_job_wait(q3asr_job* j, int32_t* ids_out, int* lens_out) {
    if (j == nullptr || ids_out == nullptr || lens_out == nullptr) return Q3ASR_ERR_INVALID;
    if (j->worker.joinable()) j->worker.join();
    if (j->rc != Q3ASR_OK) return j->rc;
    std::copy(j->ids.begin(), j->ids.end(), ids_out);
    std::copy(j->lens.begin(), j->lens.end(), lens_out);
    j->waited = true;
    return Q3ASR_OK;
}

int q3asr_job_logprobs(const q3asr_job* j, float* out) {
    if (j == nullptr || out == nullptr || !j->has_lp || !j->waited) return Q3ASR_ERR_INVALID;
    std::copy(j->lp.begin(), j->lp.end(), out);
    return Q3ASR_OK;
}

const char* q3asr_job_last_error(const q3asr_job* j) { return j ? j->error.c_str() : ""; }

void q3asr_job_free(q3asr_job* j) {
    if (j == nullptr) return;
    if (j->worker.joinable()) j->worker.join();
    delete j;
}

}  // extern "C"
