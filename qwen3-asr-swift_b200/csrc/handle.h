// handle.h — the object behind q3asr_handle: device, stream, constant tables, weights, work buffers.
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/q3asr.h"
#include "common.cuh"
#include "mel.cuh"

namespace q3 {

// growable device buffer (capacity only ever grows; contents are scratch)
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    size_t* total = nullptr;  // accounting (bytes held by the handle)
    void reserve(size_t bytes) {
        if (bytes <= cap) return;
        if (p) {
            Q3_CUDA(cudaFree(p));
            if (total) *total -= cap;
            p = nullptr;
            cap = 0;
        }
        bytes = (bytes + 255) & ~size_t(255);
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            p = nullptr;
            throw Error(Q3ASR_ERR_NOMEM, std::string("cudaMalloc(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
        }
        cap = bytes;
        if (total) *total += cap;
    }
    void release() {
        if (p) {
            cudaFree(p);
            if (total) *total -= cap;
        }
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

// pinned host staging buffer
struct HostBuf {
    void* p = nullptr;
    size_t cap = 0;
    void reserve(size_t bytes) {
        if (bytes <= cap) return;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMallocHost(&p, bytes);
        if (e != cudaSuccess) {
            p = nullptr;
            throw Error(Q3ASR_ERR_NOMEM, std::string("cudaMallocHost(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
        }
        cap = bytes;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

struct Tensor {
    std::string name;
    std::vector<int64_t> shape;
    size_t numel = 0;
    bf16* d = nullptr;  // canonical copy, bf16, device
};

// polyphase filter of one (input rate, output rate) pair (audio_io.cu)
struct ResampleTab {
    int L = 1, M = 1, K = 0;
    DevBuf taps;  // [L][2K + 2] fp32
};

struct Model;      // weights in kernel-ready layouts (model.cu)
struct BatchState; // resident batch: plan + activations (model.cu)

struct Handle {
    q3asr_config cfg;
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    // Samples travel host -> device on their own stream, one event per clip: the mel kernel of a group of clips waits only for that
    // group's copies, so the first groups' mel + convolution work overlaps the rest of the upload (forward.cu batch_upload / run_mel).
    cudaStream_t copy_stream = nullptr;
    std::vector<cudaEvent_t> copy_ev;
    std::string last_error;
    size_t dev_bytes = 0;          // bytes held in DevBufs + tensors
    unsigned long long launches = 0;  // kernels launched by this handle (non-GEMM; GEMMs are counted in gemm.cu)
    unsigned long long gemm_base = 0;

    MelTables mel_tables{};
    bool mel_ready = false;
    // mel scratch
    DevBuf mel_pcm, mel_out, mel_clips, mel_gmax, mel_tmin;
    HostBuf mel_stage;

    std::vector<Tensor> tensors;            // canonical named weights
    std::map<std::string, int> tensor_index;
    bool loaded = false;
    std::unique_ptr<Model> model;
    std::unique_ptr<BatchState> batch;
    // continuous batching: the admission groups, two so the next group's samples are staged while the current one is admitted
    std::unique_ptr<BatchState> adm[2];

    // optional per-kernel-family profiling (q3asr_profile): CUDA events around tagged launches
    struct ProfRec {
        const char* tag;
        cudaEvent_t a, b;
        double flops, bytes;
    };
    bool prof_on = false;
    std::vector<ProfRec> prof;
    size_t prof_used = 0;

    bool decode_warm = false;  // a decode step has run eagerly on this handle (function attributes set): later batches go straight to the step graph
    cudaEvent_t timer[16] = {nullptr};
    float stage_ms[4] = {0, 0, 0, 0};
    DevBuf flush_buf;
    // sample-rate conversion (audio_io.cu): filter tables per rate pair, scratch of q3asr_resample
    std::map<std::pair<int, int>, ResampleTab> resample_tabs;
    DevBuf rs_in, rs_out;
    HostBuf rs_stage;

    Handle() {
        for (DevBuf* b : {&mel_pcm, &mel_out, &mel_clips, &mel_gmax, &mel_tmin, &flush_buf, &rs_in, &rs_out}) b->total = &dev_bytes;
    }
};

// RAII tag around one or more launches; no-op unless profiling is enabled on the handle
struct ProfScope {
    Handle* h;
    size_t idx = (size_t)-1;
    ProfScope(Handle* hh, const char* tag, double flops, double bytes) : h(hh) {
        if (!h->prof_on) return;
        if (h->prof_used == h->prof.size()) {
            Handle::ProfRec r{tag, nullptr, nullptr, 0, 0};
            Q3_CUDA(cudaEventCreate(&r.a));
            Q3_CUDA(cudaEventCreate(&r.b));
            h->prof.push_back(r);
        }
        idx = h->prof_used++;
        h->prof[idx].tag = tag;
        h->prof[idx].flops = flops;
        h->prof[idx].bytes = bytes;
        cudaEventRecord(h->prof[idx].a, h->stream);
    }
    ~ProfScope() {
        if (idx != (size_t)-1) cudaEventRecord(h->prof[idx].b, h->stream);
    }
};

struct DeviceGuard {
    int prev = 0;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) Q3_CUDA(cudaSetDevice(dev));
    }
    ~DeviceGuard() { cudaSetDevice(prev); }
};

// ---- mel front (frontend.cu) ----
struct MelPlan {
    std::vector<MelClip> clips;
    long long pcm_floats = 0, out_floats = 0;
    int total_tiles = 0;
};
MelPlan mel_plan(const size_t* n_samples, int batch);
int mel_frames_for(size_t n);

// ---- model (model.cu) ----
void model_tensor_specs(const q3asr_config& c, std::vector<std::pair<std::string, std::vector<int64_t>>>* out);
void model_init_random(Handle* h, uint64_t seed);
void model_set_tensor(Handle* h, const char* name, const void* data, int dtype, const int64_t* shape, int ndim);
void model_get_tensor(const Handle* h, const char* name, float* out, size_t n);
void model_commit(Handle* h);
void model_unload(Handle* h);
void model_load_safetensors(Handle* h, const char* dir);
// the forced aligner's word splitter (csrc/text.cu; TextPreprocessing.swift:97-115, 163-243): surface keeps the punctuation, cleaned
// is what the tokenizer sees
struct WordPair {
    std::string surface, cleaned;
};
std::vector<WordPair> split_into_word_pairs(const std::string& text, const std::string& language);
// validated tensor index of a checkpoint directory as text (name \t dtype \t shape \t bytes per line); host only
std::string checkpoint_list(const char* dir);
int encoder_tokens_for(int frames);
// chat-template ids around `ntok` audio placeholders; *audio_at = index of the first placeholder (Qwen3ASR.swift:196-233)
void build_prompt(const q3asr_config& c, const q3asr_prompt* pr, int ntok, std::vector<int32_t>* ids, int* audio_at);

// rates: per-clip sample rates or null (all 16 kHz); other rates are converted on the device (audio_io.cu)
// defer_join: the staging threads keep running after the call returns (the caller's sample buffers stay borrowed) until
// finish_upload; only for callers that run the batch inside the same API call (q3asr_transcribe_ids*)
void batch_upload(Handle* h, const float* const* pcm, const size_t* n, int batch, const q3asr_prompt* prompts, const int* rates = nullptr,
                  bool defer_join = false);
struct BatchState;
void finish_upload(BatchState* bs);
void batch_set_sampling(Handle* h, const q3asr_sampling* opts);
void pick_next_token(Handle* h, const float* logits, int vocab, const int32_t* generated, int n_generated, const q3asr_sampling* opts,
                     int draw, int32_t* token);
void batch_run(Handle* h, int stages, int max_tokens, int stop_on_eos);
void batch_download(Handle* h, int32_t* ids, int max_tokens, int* lens);
void batch_set_logprobs(Handle* h, int enable);
void batch_download_logprobs(Handle* h, float* out, int max_tokens);
// continuous batching (q3asr_transcribe_ids_continuous): the whole request through one resident batch of at most max_rows rows
void transcribe_continuous(Handle* h, const float* const* pcm, const size_t* n, const int* rates, int batch, const q3asr_prompt* prompts,
                           int max_tokens, int stop_on_eos, int max_rows, int32_t* ids_out, int* lens_out, float* lp_out);
void encode_one(Handle* h, const float* mel, int frames, float* out, int* tokens);
void decode_forced(Handle* h, const float* pcm, size_t n, const q3asr_prompt* prompt, const int32_t* forced, int n_forced,
                   int32_t* argmax_out, float* top_out, const float* audio_embeds = nullptr, int n_audio_tokens = 0);
void prefill_logits(Handle* h, const float* pcm, size_t n, const q3asr_prompt* prompt, float* logits);
void config_validate(const q3asr_config& c);
void align_indices(Handle* h, const float* const* pcm, const size_t* n, const int* rates, int batch, const int32_t* const* slotted_ids,
                   const int* n_slotted, const int* const* positions, const int* n_positions, int32_t* const* raw_out);

// ---- front door (audio_io.cu) ----
size_t wav_parse(const uint8_t* data, size_t size, float* out, size_t cap, int* sample_rate);
size_t resample_len(size_t n, int in_rate, int out_rate);
void resample_design(int in_rate, int out_rate, int* L, int* M, int* K, std::vector<float>* taps);
void resample_device(Handle* h, const float* d_in, size_t n, int in_rate, int out_rate, float* d_out, size_t n_out, cudaStream_t st);
void resample_host(Handle* h, const float* in, size_t n, int in_rate, int out_rate, float* out, size_t cap, size_t* n_out);
int longform_plan(size_t n, size_t window, size_t min_tail, size_t* starts, size_t* lens, int cap);

}  // namespace q3
