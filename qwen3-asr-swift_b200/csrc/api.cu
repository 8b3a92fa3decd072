// api.cu — the extern "C" surface declared in include/q3asr.h.  Every entry point catches, records the
// message on the handle and returns a status code; nothing aborts (SURVEY.md §8b error contract).
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <mutex>

#include "gemm.cuh"
#include "model.h"

using namespace q3;

struct q3asr_handle {
    Handle h;
};

namespace {

thread_local std::string g_create_error;  // q3asr_last_error(NULL): the calling thread's last failed q3asr_create

template <typename F>
int guarded(q3asr_handle* hh, F&& fn) {
    if (hh == nullptr) return Q3ASR_ERR_INVALID;
    try {
        DeviceGuard g(hh->h.device);
        fn(hh->h);
        return Q3ASR_OK;
    } catch (const Error& e) {
        hh->h.last_error = e.what();
        return e.code > 0 ? e.code : Q3ASR_ERR_CUDA;
    } catch (const std::bad_alloc&) {
        hh->h.last_error = "out of host memory";
        return Q3ASR_ERR_NOMEM;
    } catch (const std::exception& e) {
        hh->h.last_error = e.what();
        return Q3ASR_ERR_INVALID;
    }
}

void set_common_tokens(q3asr_config* c) {
    c->tok_im_start = 151644;
    c->tok_im_end = 151645;
    c->tok_audio_start = 151669;
    c->tok_audio_end = 151670;
    c->tok_audio_pad = 151676;
    c->tok_asr_text = 151704;
    c->tok_newline = 198;
    c->tok_system = 8948;
    c->tok_user = 872;
    c->tok_assistant = 77091;
    c->tok_eos = Q3ASR_EOS_TOKEN;
    c->tok_timestamp = 151705;
}

// the device buffers of one debug-hook call, freed on every exit path
struct DebugAllocs {
    std::vector<void*> p;
    template <typename T>
    T* get(size_t n) {
        void* q = nullptr;
        Q3_CUDA(cudaMalloc(&q, n * sizeof(T)));
        p.push_back(q);
        return static_cast<T*>(q);
    }
    ~DebugAllocs() {
        for (void* q : p) cudaFree(q);
    }
};

}  // namespace

extern "C" {

const char* q3asr_version(void) { return "q3asr-b200 0.1.0 (sm_100a)"; }

int q3asr_config_preset(const char* name, q3asr_config* c) {
    if (name == nullptr || c == nullptr) return Q3ASR_ERR_INVALID;
    memset(c, 0, sizeof(*c));
    c->enc_conv_ch = 480;
    c->enc_n_window = 50;
    c->enc_n_window_infer = 800;
    c->enc_ln_eps = 1e-5f;
    c->dec_vocab = 151936;
    c->dec_layers = 28;
    c->dec_heads = 16;
    c->dec_kv_heads = 8;
    c->dec_head_dim = 128;
    c->dec_rope_theta = 1000000.0f;
    c->dec_rms_eps = 1e-6f;
    set_common_tokens(c);
    const std::string n(name);
    if (n == "0.6B" || n == "small") {
        c->enc_d_model = 896; c->enc_heads = 14; c->enc_ffn = 3584; c->enc_layers = 18; c->enc_out_dim = 1024;
        c->dec_hidden = 1024; c->dec_inter = 3072;
    } else if (n == "1.7B" || n == "large") {
        c->enc_d_model = 1024; c->enc_heads = 16; c->enc_ffn = 4096; c->enc_layers = 24; c->enc_out_dim = 2048;
        c->dec_hidden = 2048; c->dec_inter = 6144;
    } else if (n == "aligner") {  // Qwen3AudioEncoderConfig.forcedAligner (AudioEncoder.swift:71-88) + TextDecoderConfig.small + 5000 classes
        c->enc_d_model = 1024; c->enc_heads = 16; c->enc_ffn = 4096; c->enc_layers = 24; c->enc_out_dim = 1024;
        c->dec_hidden = 1024; c->dec_inter = 3072;
        c->classify_num = 5000;
    } else if (n == "tiny" || n == "tiny-aligner") {
        // small enough for the CPU oracle to finish in seconds; same graph, same kernels
        c->enc_d_model = 128; c->enc_heads = 2; c->enc_ffn = 256; c->enc_layers = 2; c->enc_out_dim = 128;
        c->enc_conv_ch = 32;
        c->dec_vocab = 2048; c->dec_hidden = 128; c->dec_layers = 2; c->dec_heads = 4; c->dec_kv_heads = 2;
        c->dec_inter = 256;
        c->tok_im_start = 2001; c->tok_im_end = 2002; c->tok_audio_start = 2003; c->tok_audio_end = 2004;
        c->tok_audio_pad = 2005; c->tok_asr_text = 2006; c->tok_newline = 198; c->tok_system = 1948; c->tok_user = 872;
        c->tok_assistant = 1091; c->tok_eos = 2002; c->tok_timestamp = 2007;
        if (n == "tiny-aligner") c->classify_num = 70;  // not a multiple of the GEMM tile: exercises the padded head
    } else {
        return Q3ASR_ERR_INVALID;
    }
    return Q3ASR_OK;
}

const char* q3asr_last_error(const q3asr_handle* h) {
    if (h == nullptr) return g_create_error.c_str();
    return h->h.last_error.c_str();
}

int q3asr_create(const q3asr_config* cfg, int device, q3asr_handle** out) {
    if (cfg == nullptr || out == nullptr) return Q3ASR_ERR_INVALID;
    *out = nullptr;
    q3asr_handle* hh = nullptr;
    try {
        config_validate(*cfg);
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0)
            throw Error(Q3ASR_ERR_CUDA, std::string("no CUDA device: libq3asr has no CPU fallback (") + cudaGetErrorString(e) + ")");
        Q3_CHECK(device >= 0 && device < ndev, Q3ASR_ERR_INVALID, "device index out of range");
        DeviceGuard g(device);
        hh = new q3asr_handle();
        Handle& h = hh->h;
        h.cfg = *cfg;
        h.device = device;
        gemm_init(device);
        cudaDeviceProp prop;
        Q3_CUDA(cudaGetDeviceProperties(&prop, device));
        h.num_sms = prop.multiProcessorCount;
        Q3_CUDA(cudaStreamCreateWithFlags(&h.stream, cudaStreamNonBlocking));
        Q3_CUDA(cudaStreamCreateWithFlags(&h.copy_stream, cudaStreamNonBlocking));
        mel_tables_create(&h.mel_tables);
        h.mel_ready = true;
        for (int i = 0; i < 16; i++) Q3_CUDA(cudaEventCreate(&h.timer[i]));
        h.gemm_base = gemm_launch_count();
        *out = hh;
        return Q3ASR_OK;
    } catch (const std::exception& e) {
        g_create_error = e.what();
        const Error* qe = dynamic_cast<const Error*>(&e);
        if (hh) q3asr_destroy(hh);
        return qe ? qe->code : Q3ASR_ERR_INVALID;
    }
}

void q3asr_destroy(q3asr_handle* hh) {
    if (hh == nullptr) return;
    Handle& h = hh->h;
    try {
        DeviceGuard g(h.device);
        if (h.copy_stream) cudaStreamSynchronize(h.copy_stream);
        if (h.stream) cudaStreamSynchronize(h.stream);
        model_unload(&h);
        if (h.mel_ready) mel_tables_destroy(&h.mel_tables);
        for (DevBuf* b : {&h.mel_pcm, &h.mel_out, &h.mel_clips, &h.mel_gmax, &h.mel_tmin, &h.flush_buf, &h.rs_in, &h.rs_out}) b->release();
        for (auto& kv : h.resample_tabs) kv.second.taps.release();
        h.rs_stage.release();
        h.mel_stage.release();
        for (int i = 0; i < 16; i++)
            if (h.timer[i]) cudaEventDestroy(h.timer[i]);
        for (auto& r : h.prof) {
            cudaEventDestroy(r.a);
            cudaEventDestroy(r.b);
        }
        for (cudaEvent_t e : h.copy_ev) cudaEventDestroy(e);
        if (h.copy_stream) cudaStreamDestroy(h.copy_stream);
        if (h.stream) cudaStreamDestroy(h.stream);
    } catch (...) {
    }
    delete hh;
}

// ---- weights ----
int q3asr_init_random(q3asr_handle* h, uint64_t seed) {
    return guarded(h, [&](Handle& x) { model_init_random(&x, seed); });
}
int q3asr_tensor_count(const q3asr_handle* h) { return h ? (int)h->h.tensors.size() : 0; }
int q3asr_tensor_info(const q3asr_handle* h, int index, char* name, int name_cap, int64_t* shape4, int* ndim) {
    if (h == nullptr || index < 0 || index >= (int)h->h.tensors.size()) return Q3ASR_ERR_INVALID;
    const Tensor& t = h->h.tensors[index];
    if (name && name_cap > 0) {
        strncpy(name, t.name.c_str(), name_cap - 1);
        name[name_cap - 1] = 0;
    }
    if (shape4)
        for (int i = 0; i < 4; i++) shape4[i] = i < (int)t.shape.size() ? t.shape[i] : 1;
    if (ndim) *ndim = (int)t.shape.size();
    return Q3ASR_OK;
}
int q3asr_set_tensor(q3asr_handle* h, const char* name, const void* data, int dtype, const int64_t* shape, int ndim) {
    return guarded(h, [&](Handle& x) { model_set_tensor(&x, name, data, dtype, shape, ndim); });
}
int q3asr_get_tensor(const q3asr_handle* h, const char* name, float* out, size_t n) {
    return guarded(const_cast<q3asr_handle*>(h), [&](Handle& x) { model_get_tensor(&x, name, out, n); });
}
int q3asr_commit_weights(q3asr_handle* h) {
    return guarded(h, [&](Handle& x) { model_commit(&x); });
}
int q3asr_load_safetensors(q3asr_handle* h, const char* dir) {
    return guarded(h, [&](Handle& x) { model_load_safetensors(&x, dir); });
}
int q3asr_checkpoint_list(const char* dir, char* buf, size_t cap, size_t* needed) {
    static thread_local std::string err;
    try {
        const std::string s = checkpoint_list(dir);
        if (needed) *needed = s.size() + 1;
        if (buf == nullptr) return needed ? Q3ASR_OK : Q3ASR_ERR_INVALID;
        if (cap < s.size() + 1) return Q3ASR_ERR_NOMEM;
        memcpy(buf, s.c_str(), s.size() + 1);
        return Q3ASR_OK;
    } catch (const Error& e) {
        err = e.what();
    } catch (const std::exception& e) {
        err = e.what();
    }
    // the message instead of the list, as far as it fits
    if (needed) *needed = err.size() + 1;
    if (buf && cap > 0) {
        const size_t n = std::min(cap - 1, err.size());
        memcpy(buf, err.data(), n);
        buf[n] = 0;
    }
    return Q3ASR_ERR_IO;
}
int q3asr_is_loaded(const q3asr_handle* h) { return h != nullptr && h->h.loaded ? 1 : 0; }
int q3asr_unload(q3asr_handle* h) {
    return guarded(h, [&](Handle& x) { model_unload(&x); });
}
size_t q3asr_memory_footprint(const q3asr_handle* h) { return h ? h->h.dev_bytes : 0; }

// ---- mel ----
int q3asr_mel_frames(size_t n) { return mel_frames_for(n); }

int q3asr_mel_batch(q3asr_handle* hh, const float* const* pcm, const size_t* n, int batch, float* const* out, int* frames) {
    return guarded(hh, [&](Handle& h) {
        Q3_CHECK(pcm != nullptr && n != nullptr && out != nullptr && batch > 0, Q3ASR_ERR_INVALID, "mel: null argument / empty batch");
        for (int b = 0; b < batch; b++)
            Q3_CHECK(pcm[b] != nullptr && n[b] > 0 && n[b] < (size_t)1 << 30, Q3ASR_ERR_INVALID, "mel: empty or oversized clip");
        MelPlan plan = mel_plan(n, batch);
        h.mel_pcm.reserve(sizeof(float) * (plan.pcm_floats + 64));
        h.mel_out.reserve(sizeof(float) * std::max<long long>(plan.out_floats, 1));
        h.mel_clips.reserve(sizeof(MelClip) * batch);
        h.mel_gmax.reserve(sizeof(int) * batch);
        h.mel_tmin.reserve(sizeof(float) * 2 * plan.total_tiles);  // per-tile minimum + per-tile clip
        h.mel_stage.reserve(sizeof(float) * std::max<long long>(plan.pcm_floats, plan.out_floats));
        float* stage = h.mel_stage.as<float>();
        for (int b = 0; b < batch; b++) memcpy(stage + plan.clips[b].in_off, pcm[b], sizeof(float) * n[b]);
        Q3_CUDA(cudaMemcpyAsync(h.mel_pcm.p, stage, sizeof(float) * plan.pcm_floats, cudaMemcpyHostToDevice, h.stream));
        Q3_CUDA(cudaMemcpyAsync(h.mel_clips.p, plan.clips.data(), sizeof(MelClip) * batch, cudaMemcpyHostToDevice, h.stream));
        mel_launch(h.mel_tables, h.mel_pcm.as<float>(), h.mel_out.as<float>(), h.mel_clips.as<MelClip>(), batch, plan.total_tiles,
                   h.mel_gmax.as<int>(), h.mel_tmin.as<float>(), h.num_sms, h.stream);
        h.launches += 3;
        Q3_CUDA(cudaStreamSynchronize(h.stream));  // staging buffer is reused for the way back
        if (plan.out_floats > 0)
            Q3_CUDA(cudaMemcpyAsync(stage, h.mel_out.p, sizeof(float) * plan.out_floats, cudaMemcpyDeviceToHost, h.stream));
        Q3_CUDA(cudaStreamSynchronize(h.stream));
        for (int b = 0; b < batch; b++) {
            const MelClip& c = plan.clips[b];
            if (c.frames > 0) memcpy(out[b], stage + c.out_off, sizeof(float) * (size_t)MEL_BINS * c.frames);
            if (frames) frames[b] = c.frames;
        }
    });
}

int q3asr_mel(q3asr_handle* h, const float* pcm, size_t n, float* out, int* frames) {
    const float* pp[1] = {pcm};
    float* oo[1] = {out};
    return q3asr_mel_batch(h, pp, &n, 1, oo, frames);
}

int q3asr_encoder_tokens(int frames) { return encoder_tokens_for(frames); }

int q3asr_prompt_ids(const q3asr_config* cfg, int n_audio_tokens, const q3asr_prompt* prompt, int32_t* ids_out, int cap, int* n_ids,
                     int* audio_at) {
    if (!cfg || n_audio_tokens < 0 || !n_ids || cap < 0 || (cap > 0 && !ids_out)) return Q3ASR_ERR_INVALID;
    if (prompt && ((prompt->n_context > 0 && !prompt->context_ids) || (prompt->n_language > 0 && !prompt->language_ids) ||
                   prompt->n_context < 0 || prompt->n_language < 0))
        return Q3ASR_ERR_INVALID;
    if (n_audio_tokens > (1 << 24)) return Q3ASR_ERR_INVALID;  // 120 000 frames give 15 600 tokens (AudioPreprocessing.swift:304)
    try {
        std::vector<int32_t> ids;
        int at = 0;
        build_prompt(*cfg, prompt, n_audio_tokens, &ids, &at);
        *n_ids = (int)ids.size();
        if (audio_at) *audio_at = at;
        if ((int)ids.size() > cap) return Q3ASR_ERR_INVALID;  // *n_ids says how much room is needed
        std::copy(ids.begin(), ids.end(), ids_out);
        return Q3ASR_OK;
    } catch (const std::exception&) {  // host allocation failure: nothing may cross the C boundary
        return Q3ASR_ERR_NOMEM;
    }
}

int q3asr_encode(q3asr_handle* h, const float* mel, int frames, float* out, int* tokens) {
    return guarded(h, [&](Handle& x) { encode_one(&x, mel, frames, out, tokens); });
}

// ---- transcription ----
int q3asr_batch_upload(q3asr_handle* h, const float* const* pcm, const size_t* n, int batch, const q3asr_prompt* prompts) {
    return guarded(h, [&](Handle& x) { batch_upload(&x, pcm, n, batch, prompts); });
}
namespace {
// joins a deferred upload on every way out of a transcribe call (errors of the threads were either reported by batch_run or
// are secondary to the exception already in flight)
struct UploadGuard {
    Handle* h;
    ~UploadGuard() {
        try {
            finish_upload(h->batch.get());
        } catch (...) {
        }
    }
};
}  // namespace
namespace {
// A request larger than the decode step's row capacity (SKINNY_MAX_ROWS = 256 token rows) is served as equal sub-batches one after
// the other: above it the decode falls back to the general GEMMs (measured at the former capacity of 128: 160 clips in one batch
// 6 500 audio-s/s against 9 400 for 128; ids within bf16 noise of, but not bit-identical to, the weight-streaming path), so an
// utterance's ids would depend on the size of the request it arrived in.  Utterances are independent; outputs land at their own
// offsets; stage times are summed over the sub-batches.
void transcribe_chunked(Handle& x, const float* const* pcm, const size_t* n, const int* rates, int batch, const q3asr_prompt* prompts,
                        const q3asr_sampling* sampling, bool set_sampling, int max_tokens, int stop_on_eos, int32_t* ids_out, int* lens_out,
                        float* lp_out = nullptr) {
    Q3_CHECK(ids_out != nullptr && lens_out != nullptr, Q3ASR_ERR_INVALID, "transcribe: null output");
    const int chunks = batch <= SKINNY_MAX_ROWS ? 1 : (batch + SKINNY_MAX_ROWS - 1) / SKINNY_MAX_ROWS;
    const int per = chunks == 1 ? batch : (batch + chunks - 1) / chunks;  // batch <= 0 is refused by batch_upload below
    float stage_sum[4] = {0.f, 0.f, 0.f, 0.f};
    int b0 = 0;
    do {
        const int nb = std::min(per, batch - b0);
        UploadGuard ug{&x};  // the staging threads never outlive this call (they read the caller's buffers)
        batch_upload(&x, pcm + b0, n + b0, nb, prompts ? prompts + b0 : nullptr, rates ? rates + b0 : nullptr, true);
        if (set_sampling) batch_set_sampling(&x, sampling);
        if (lp_out) batch_set_logprobs(&x, 1);
        batch_run(&x, Q3ASR_STAGE_ALL, max_tokens, stop_on_eos);
        batch_download(&x, ids_out + (size_t)b0 * max_tokens, max_tokens, lens_out + b0);
        if (lp_out) batch_download_logprobs(&x, lp_out + (size_t)b0 * max_tokens, max_tokens);
        for (int i = 0; i < 4; i++) stage_sum[i] += x.stage_ms[i];
        b0 += nb;
    } while (b0 < batch);
    for (int i = 0; i < 4; i++) x.stage_ms[i] = stage_sum[i];
}
}  // namespace
int q3asr_batch_run(q3asr_handle* h, int stages, int max_tokens, int stop_on_eos) {
    return guarded(h, [&](Handle& x) { batch_run(&x, stages, max_tokens, stop_on_eos); });
}
int q3asr_batch_download(q3asr_handle* h, int32_t* ids, int max_tokens, int* lens) {
    return guarded(h, [&](Handle& x) { batch_download(&x, ids, max_tokens, lens); });
}
int q3asr_transcribe_ids(q3asr_handle* h, const float* const* pcm, const size_t* n, int batch, const q3asr_prompt* prompts,
                         int max_tokens, int stop_on_eos, int32_t* ids_out, int* lens_out) {
    return guarded(h, [&](Handle& x) { transcribe_chunked(x, pcm, n, nullptr, batch, prompts, nullptr, false, max_tokens, stop_on_eos, ids_out, lens_out); });
}
int q3asr_batch_upload_sr(q3asr_handle* h, const float* const* pcm, const size_t* n, const int* sample_rates, int batch,
                          const q3asr_prompt* prompts) {
    return guarded(h, [&](Handle& x) { batch_upload(&x, pcm, n, batch, prompts, sample_rates); });
}
int q3asr_transcribe_ids_sr(q3asr_handle* h, const float* const* pcm, const size_t* n, const int* sample_rates, int batch,
                            const q3asr_prompt* prompts, int max_tokens, int stop_on_eos, int32_t* ids_out, int* lens_out) {
    return guarded(h, [&](Handle& x) { transcribe_chunked(x, pcm, n, sample_rates, batch, prompts, nullptr, false, max_tokens, stop_on_eos, ids_out, lens_out); });
}
int q3asr_batch_set_sampling(q3asr_handle* h, const q3asr_sampling* opts) {
    return guarded(h, [&](Handle& x) { batch_set_sampling(&x, opts); });
}
int q3asr_transcribe_ids_opts(q3asr_handle* h, const float* const* pcm, const size_t* n, const int* sample_rates, int batch,
                              const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos,
                              int32_t* ids_out, int* lens_out) {
    return q3asr_transcribe_ids_lp(h, pcm, n, sample_rates, batch, prompts, sampling, max_tokens, stop_on_eos, ids_out, lens_out, nullptr);
}
int q3asr_transcribe_ids_lp(q3asr_handle* h, const float* const* pcm, const size_t* n, const int* sample_rates, int batch,
                            const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos,
                            int32_t* ids_out, int* lens_out, float* logprobs_out) {
    return guarded(h, [&](Handle& x) {
        transcribe_chunked(x, pcm, n, sample_rates, batch, prompts, sampling, true, max_tokens, stop_on_eos, ids_out, lens_out, logprobs_out);
    });
}
int q3asr_transcribe_ids_continuous(q3asr_handle* h, const float* const* pcm, const size_t* n, const int* sample_rates, int batch,
                                    const q3asr_prompt* prompts, int max_tokens, int stop_on_eos, int max_rows, int32_t* ids_out, int* lens_out,
                                    float* logprobs_out) {
    return guarded(h, [&](Handle& x) {
        Q3_CHECK(max_rows <= SKINNY_MAX_ROWS && batch > 0 && max_tokens >= 0, Q3ASR_ERR_INVALID,
                 "transcribe_continuous: max_rows > 256, empty batch or max_tokens < 0");
        if (max_tokens == 0) {  // nothing is decoded: the static path validates the clips and returns empty utterances
            transcribe_chunked(x, pcm, n, sample_rates, batch, prompts, nullptr, false, 0, stop_on_eos, ids_out, lens_out, logprobs_out);
            return;
        }
        transcribe_continuous(&x, pcm, n, sample_rates, batch, prompts, max_tokens, stop_on_eos, max_rows, ids_out, lens_out, logprobs_out);
    });
}
int q3asr_batch_set_logprobs(q3asr_handle* h, int enable) {
    return guarded(h, [&](Handle& x) { batch_set_logprobs(&x, enable); });
}
int q3asr_batch_download_logprobs(q3asr_handle* h, float* out, int max_tokens) {
    return guarded(h, [&](Handle& x) { batch_download_logprobs(&x, out, max_tokens); });
}
int q3asr_pick_next_token(q3asr_handle* h, const float* logits, int vocab, const int32_t* generated, int n_generated,
                          const q3asr_sampling* opts, int draw, int32_t* token) {
    return guarded(h, [&](Handle& x) { pick_next_token(&x, logits, vocab, generated, n_generated, opts, draw, token); });
}
int q3asr_align_indices(q3asr_handle* h, const float* const* pcm, const size_t* n, const int* sample_rates, int batch,
                        const int32_t* const* slotted_ids, const int* n_slotted, const int* const* positions, const int* n_positions,
                        int32_t* const* raw_out) {
    return guarded(h, [&](Handle& x) { align_indices(&x, pcm, n, sample_rates, batch, slotted_ids, n_slotted, positions, n_positions, raw_out); });
}
int q3asr_resample(q3asr_handle* h, const float* in, size_t n, int in_rate, int out_rate, float* out, size_t cap, size_t* n_out) {
    return guarded(h, [&](Handle& x) { resample_host(&x, in, n, in_rate, out_rate, out, cap, n_out); });
}
int q3asr_decode_forced(q3asr_handle* h, const float* pcm, size_t n, const q3asr_prompt* prompt, const int32_t* forced, int n_forced,
                        int32_t* argmax_out, float* top_out) {
    return guarded(h, [&](Handle& x) { decode_forced(&x, pcm, n, prompt, forced, n_forced, argmax_out, top_out); });
}
int q3asr_decode_forced_embeds(q3asr_handle* h, const float* pcm, size_t n, const q3asr_prompt* prompt, const float* audio_embeds,
                               int n_audio_tokens, const int32_t* forced, int n_forced, int32_t* argmax_out, float* top_out) {
    return guarded(h, [&](Handle& x) {
        Q3_CHECK(audio_embeds != nullptr && n_audio_tokens > 0, Q3ASR_ERR_INVALID, "decode_forced_embeds: null embeddings");
        decode_forced(&x, pcm, n, prompt, forced, n_forced, argmax_out, top_out, audio_embeds, n_audio_tokens);
    });
}
int q3asr_prefill_logits(q3asr_handle* h, const float* pcm, size_t n, const q3asr_prompt* prompt, float* logits) {
    return guarded(h, [&](Handle& x) { prefill_logits(&x, pcm, n, prompt, logits); });
}

int q3asr_sync(q3asr_handle* h) {
    return guarded(h, [&](Handle& x) { Q3_CUDA(cudaStreamSynchronize(x.stream)); });
}
int q3asr_timer_record(q3asr_handle* h, int slot) {
    return guarded(h, [&](Handle& x) {
        Q3_CHECK(slot >= 0 && slot < 16, Q3ASR_ERR_INVALID, "timer slot");
        Q3_CUDA(cudaEventRecord(x.timer[slot], x.stream));
    });
}
int q3asr_timer_elapsed_ms(q3asr_handle* h, int a, int b, float* ms) {
    return guarded(h, [&](Handle& x) {
        Q3_CHECK(a >= 0 && a < 16 && b >= 0 && b < 16 && ms != nullptr, Q3ASR_ERR_INVALID, "timer slot");
        Q3_CUDA(cudaEventSynchronize(x.timer[b]));
        Q3_CUDA(cudaEventElapsedTime(ms, x.timer[a], x.timer[b]));
    });
}
int q3asr_stage_ms(q3asr_handle* h, float* ms4) {
    if (h == nullptr || ms4 == nullptr) return Q3ASR_ERR_INVALID;
    for (int i = 0; i < 4; i++) ms4[i] = h->h.stage_ms[i];
    return Q3ASR_OK;
}
uint64_t q3asr_launch_count(const q3asr_handle* h) {
    if (h == nullptr) return 0;
    return h->h.launches + (gemm_launch_count() - h->h.gemm_base);
}
int q3asr_decode_stats(const q3asr_handle* h, uint64_t* out4) {
    if (h == nullptr || out4 == nullptr) return Q3ASR_ERR_INVALID;
    const BatchState* bs = h->h.batch.get();
    out4[0] = bs ? bs->stat_steps : 0;
    out4[1] = bs ? bs->stat_row_steps : 0;
    out4[2] = bs ? bs->stat_compactions : 0;
    out4[3] = bs ? (uint64_t)bs->dec_rows : 0;
    return Q3ASR_OK;
}
int q3asr_decode_admissions(const q3asr_handle* h, uint64_t* out2) {
    if (h == nullptr || out2 == nullptr) return Q3ASR_ERR_INVALID;
    const BatchState* bs = h->h.batch.get();
    out2[0] = bs ? bs->stat_admissions : 0;
    out2[1] = bs ? bs->stat_admitted : 0;
    return Q3ASR_OK;
}
int q3asr_profile(q3asr_handle* h, int enable) {
    return guarded(h, [&](Handle& x) {
        Q3_CUDA(cudaStreamSynchronize(x.stream));
        x.prof_on = enable != 0;
        x.prof_used = 0;
    });
}
int q3asr_profile_report(q3asr_handle* h, char* buf, size_t cap) {
    return guarded(h, [&](Handle& x) {
        Q3_CHECK(buf != nullptr && cap > 0, Q3ASR_ERR_INVALID, "profile_report: null buffer");
        Q3_CUDA(cudaStreamSynchronize(x.stream));
        struct Agg { double ms = 0, flops = 0, bytes = 0; long n = 0; };
        std::vector<std::pair<std::string, Agg>> agg;
        for (size_t i = 0; i < x.prof_used; i++) {
            float ms = 0.f;
            Q3_CUDA(cudaEventElapsedTime(&ms, x.prof[i].a, x.prof[i].b));
            size_t k = 0;
            for (; k < agg.size(); k++)
                if (agg[k].first == x.prof[i].tag) break;
            if (k == agg.size()) agg.emplace_back(x.prof[i].tag, Agg());
            agg[k].second.ms += ms;
            agg[k].second.flops += x.prof[i].flops;
            agg[k].second.bytes += x.prof[i].bytes;
            agg[k].second.n++;
        }
        std::string out;
        char line[256];
        for (auto& kv : agg) {
            snprintf(line, sizeof(line), "%s,%ld,%.6f,%.6e,%.6e\n", kv.first.c_str(), kv.second.n, kv.second.ms, kv.second.flops,
                     kv.second.bytes);
            out += line;
        }
        Q3_CHECK(out.size() + 1 <= cap, Q3ASR_ERR_INVALID, "profile_report: buffer too small");
        memcpy(buf, out.c_str(), out.size() + 1);
        x.prof_used = 0;
    });
}
int q3asr_flush_l2(q3asr_handle* h) {
    return guarded(h, [&](Handle& x) {
        const size_t bytes = (size_t)256 << 20;
        x.flush_buf.reserve(bytes);
        Q3_CUDA(cudaMemsetAsync(x.flush_buf.p, 0, bytes, x.stream));
    });
}

// ---- debug hooks ----
int q3asr_debug_gemm(q3asr_handle* hh, const uint16_t* A, const uint16_t* W, const uint16_t* bias, const uint16_t* resid, int M, int N,
                     int K, int epi, int gelu, int bn, int use_simt, void* out) {
    return guarded(hh, [&](Handle& h) {
        Q3_CHECK(A && W && out && M > 0 && N > 0 && K > 0, Q3ASR_ERR_INVALID, "debug_gemm: bad argument");
        // 8 / 9: the LM-head kernel / EPI_ARGMAX with the per-tile sums of exp(z - tile max) -> int32 ids [M], then fp32 logprobs [M]
        const bool lp = epi == 8 || epi == 9;
        if (epi == 9) epi = EPI_ARGMAX;
        if (epi == 7 || epi == 8) {  // decode-step LM head (lmhead.cuh): int32 argmax ids [M]
            bf16 *dA, *dW;
            float *dv, *ds = nullptr, *dlp = nullptr;
            int* di;
            int32_t* dtok;
            const int tiles = lmhead_tiles(N);
            Q3_CUDA(cudaMalloc(&dA, 2 * (size_t)M * K));
            Q3_CUDA(cudaMalloc(&dW, 2 * (size_t)N * K));
            Q3_CUDA(cudaMalloc(&dv, sizeof(float) * (size_t)M * tiles));
            Q3_CUDA(cudaMalloc(&di, sizeof(int) * (size_t)M * tiles));
            Q3_CUDA(cudaMalloc(&dtok, sizeof(int32_t) * (size_t)M));
            if (lp) {
                Q3_CUDA(cudaMalloc(&ds, sizeof(float) * (size_t)M * tiles));
                Q3_CUDA(cudaMalloc(&dlp, sizeof(float) * (size_t)M));
            }
            cudaError_t se = cudaSuccess;
            auto release = [&]() { cudaFree(dA); cudaFree(dW); cudaFree(dv); cudaFree(di); cudaFree(dtok); cudaFree(ds); cudaFree(dlp); };
            try {
                Q3_H2D_SYNC(dA, A, 2 * (size_t)M * K);
                Q3_H2D_SYNC(dW, W, 2 * (size_t)N * K);
                lmhead_argmax(dA, K, M, K, dW, N, dv, di, h.stream, ds);
                if (lp) argmax_lse_reduce(dv, di, ds, nullptr, nullptr, 0, M, tiles, dtok, nullptr, dlp, h.stream);
                else argmax_reduce(dv, di, M, tiles, dtok, nullptr, h.stream);
                se = cudaStreamSynchronize(h.stream);
                if (se == cudaSuccess) se = cudaMemcpy(out, dtok, sizeof(int32_t) * (size_t)M, cudaMemcpyDeviceToHost);
                if (se == cudaSuccess && lp) se = cudaMemcpy(reinterpret_cast<int32_t*>(out) + M, dlp, sizeof(float) * (size_t)M, cudaMemcpyDeviceToHost);
            } catch (...) {
                release();
                throw;
            }
            release();
            Q3_CUDA(se);
            return;
        }
        if (epi >= 4) {  // decode-step weight-streaming kernel (skinny.cuh): 4 split-K partials (summed here), 5 store
            Q3_CHECK(epi <= 5, Q3ASR_ERR_INVALID, "debug_gemm: bad epilogue");
            const int sk = epi - 4;
            const int splits = gemm_skinny_splits(N, K, sk);
            bf16 *dA, *dW;
            void* dO;
            const size_t out_elems = (size_t)M * N;
            const size_t dev_bytes = sk == SK_PARTIAL ? sizeof(float) * out_elems * splits : 2 * out_elems;
            Q3_CUDA(cudaMalloc(&dA, 2 * (size_t)M * K));
            Q3_CUDA(cudaMalloc(&dW, 2 * (size_t)N * K));
            Q3_CUDA(cudaMalloc(&dO, dev_bytes));
            Q3_H2D_SYNC(dA, A, 2 * (size_t)M * K);
            Q3_H2D_SYNC(dW, W, 2 * (size_t)N * K);
            std::vector<float> part;
            cudaError_t se = cudaSuccess;
            try {
                gemm_skinny(dA, K, M, K, dW, N, sk, dO, N, h.stream);
                se = cudaStreamSynchronize(h.stream);
                if (se == cudaSuccess) {
                    if (sk == SK_PARTIAL) {
                        part.resize(out_elems * splits);
                        se = cudaMemcpy(part.data(), dO, dev_bytes, cudaMemcpyDeviceToHost);
                        float* o = reinterpret_cast<float*>(out);
                        for (size_t i = 0; i < out_elems; i++) {
                            float a = part[i];
                            for (int sp = 1; sp < splits; sp++) a += part[(size_t)sp * out_elems + i];
                            o[i] = a;
                        }
                    } else {
                        se = cudaMemcpy(out, dO, dev_bytes, cudaMemcpyDeviceToHost);
                    }
                }
            } catch (...) {
                cudaFree(dA); cudaFree(dW); cudaFree(dO);
                throw;
            }
            cudaFree(dA); cudaFree(dW); cudaFree(dO);
            Q3_CUDA(se);
            return;
        }
        bf16 *dA, *dW, *dB = nullptr, *dR = nullptr;
        void* dO;
        float *dv = nullptr, *ds = nullptr, *dlp = nullptr;
        int* di = nullptr;
        int32_t* dtok = nullptr;
        const int bnn = bn ? bn : gemm_pick_bn(N, epi, cdiv(M, GEMM_BM));
        const int tiles_n = N / bnn;
        const size_t out_bytes = epi == EPI_F32 ? sizeof(float) * (size_t)M * N
                                 : epi == EPI_SWIGLU ? 2 * (size_t)M * (N / 2)
                                 : epi == EPI_ARGMAX ? sizeof(int32_t) * (size_t)M
                                                     : 2 * (size_t)M * N;
        Q3_CUDA(cudaMalloc(&dA, 2 * (size_t)M * K));
        Q3_CUDA(cudaMalloc(&dW, 2 * (size_t)N * K));
        Q3_CUDA(cudaMalloc(&dO, std::max<size_t>(out_bytes, 2 * (size_t)M * N)));
        Q3_H2D_SYNC(dA, A, 2 * (size_t)M * K);
        Q3_H2D_SYNC(dW, W, 2 * (size_t)N * K);
        if (bias) {
            Q3_CUDA(cudaMalloc(&dB, 2 * (size_t)N));
            Q3_H2D_SYNC(dB, bias, 2 * (size_t)N);
        }
        if (resid) {
            Q3_CUDA(cudaMalloc(&dR, 2 * (size_t)M * N));
            Q3_H2D_SYNC(dR, resid, 2 * (size_t)M * N);
        }
        GemmEpiArgs e;
        e.epi = epi;
        e.out = dO;
        e.ldo = epi == EPI_SWIGLU ? N / 2 : N;
        e.bias = dB;
        e.resid = dR;
        e.ldr = N;
        e.gelu = gelu;
        if (epi == EPI_ARGMAX) {
            Q3_CUDA(cudaMalloc(&dv, sizeof(float) * (size_t)M * tiles_n));
            Q3_CUDA(cudaMalloc(&di, sizeof(int) * (size_t)M * tiles_n));
            Q3_CUDA(cudaMalloc(&dtok, sizeof(int32_t) * (size_t)M));
            e.amax_val = dv;
            e.amax_idx = di;
            if (lp) {
                Q3_CUDA(cudaMalloc(&ds, sizeof(float) * (size_t)M * tiles_n));
                Q3_CUDA(cudaMalloc(&dlp, sizeof(float) * (size_t)M));
                e.amax_sum = ds;
            }
        }
        gemm(dA, K, M, K, dW, N, e, h.stream, use_simt != 0, bnn);
        if (epi == EPI_ARGMAX && lp) {
            argmax_lse_reduce(dv, di, ds, nullptr, nullptr, 0, M, tiles_n, dtok, nullptr, dlp, h.stream);
            Q3_CUDA(cudaMemcpyAsync(out, dtok, out_bytes, cudaMemcpyDeviceToHost, h.stream));
            Q3_CUDA(cudaMemcpyAsync(reinterpret_cast<int32_t*>(out) + M, dlp, sizeof(float) * (size_t)M, cudaMemcpyDeviceToHost, h.stream));
        } else if (epi == EPI_ARGMAX) {
            argmax_reduce(dv, di, M, tiles_n, dtok, nullptr, h.stream);
            Q3_CUDA(cudaMemcpyAsync(out, dtok, out_bytes, cudaMemcpyDeviceToHost, h.stream));
        } else {
            Q3_CUDA(cudaMemcpyAsync(out, dO, out_bytes, cudaMemcpyDeviceToHost, h.stream));
        }
        cudaError_t se = cudaStreamSynchronize(h.stream);
        cudaFree(dA); cudaFree(dW); cudaFree(dO); cudaFree(dB); cudaFree(dR); cudaFree(dv); cudaFree(di); cudaFree(dtok); cudaFree(ds); cudaFree(dlp);
        Q3_CUDA(se);
    });
}

int q3asr_debug_conv(q3asr_handle* hh, const uint16_t* in, const uint16_t* w, const uint16_t* bias, int B, int H, int W, int C, int O,
                     int box_w, int box_h, int box_b, int use_simt, uint16_t* out) {
    return guarded(hh, [&](Handle& h) {
        Q3_CHECK(in && w && out && B > 0 && H > 0 && W > 0 && C > 0 && O > 0, Q3ASR_ERR_INVALID, "debug_conv: bad argument");
        const int OH = (H - 1) / 2 + 1, OW = (W - 1) / 2 + 1;
        bf16 *dI, *dW, *dB = nullptr, *dO;
        const size_t in_n = (size_t)B * H * W * C, w_n = (size_t)O * 9 * C, out_n = (size_t)B * OH * OW * O;
        Q3_CUDA(cudaMalloc(&dI, 2 * in_n));
        Q3_CUDA(cudaMalloc(&dW, 2 * w_n));
        Q3_CUDA(cudaMalloc(&dO, 2 * out_n));
        Q3_H2D_SYNC(dI, in, 2 * in_n);
        Q3_H2D_SYNC(dW, w, 2 * w_n);
        if (bias) {
            Q3_CUDA(cudaMalloc(&dB, 2 * (size_t)O));
            Q3_H2D_SYNC(dB, bias, 2 * (size_t)O);
        }
        GemmA a;
        a.ptr = dI; a.C = C; a.W = W; a.H = H; a.B = B;
        a.sW = C; a.sH = (long)W * C; a.sB = (long)H * W * C;
        GemmShape s;
        s.Wb = box_w; s.Hb = box_h; s.Bb = box_b;
        s.OW = OW; s.OH = OH; s.OB = B;
        s.sw = 2; s.sh = 2;
        s.taps = 9;
        for (int t = 0; t < 9; t++) { s.tap_dw[t] = (signed char)(t % 3 - 1); s.tap_dh[t] = (signed char)(t / 3 - 1); }
        GemmEpiArgs e;
        e.out = dO; e.ldo = O; e.bias = dB; e.gelu = 1;
        gemm_conv(a, s, dW, O, e, h.stream, use_simt != 0, 0);
        Q3_CUDA(cudaMemcpyAsync(out, dO, 2 * out_n, cudaMemcpyDeviceToHost, h.stream));
        cudaError_t se = cudaStreamSynchronize(h.stream);
        cudaFree(dI); cudaFree(dW); cudaFree(dO); cudaFree(dB);
        Q3_CUDA(se);
    });
}

int q3asr_debug_attention(q3asr_handle* hh, const uint16_t* q, const uint16_t* k, const uint16_t* v, int rows, int heads, int group,
                          int head_dim, const int* seg_row0, const int* seg_len, int n_segs, int causal, float scale, int kernel,
                          uint16_t* out) {
    return guarded(hh, [&](Handle& h) {
        Q3_CHECK(q && k && v && out && seg_row0 && seg_len && rows > 0 && heads > 0 && group > 0 && heads % group == 0 && n_segs > 0,
                 Q3ASR_ERR_INVALID, "debug_attention: bad argument");
        const size_t nq = (size_t)rows * heads * head_dim, nk = (size_t)rows * (heads / group) * head_dim;
        bf16 *dq, *dk, *dv, *dout;
        int* dseg;
        Q3_CUDA(cudaMalloc(&dq, 2 * nq));
        Q3_CUDA(cudaMalloc(&dk, 2 * nk));
        Q3_CUDA(cudaMalloc(&dv, 2 * nk));
        Q3_CUDA(cudaMalloc(&dout, 2 * nq));
        Q3_CUDA(cudaMalloc(&dseg, sizeof(int) * 2 * n_segs));
        Q3_H2D_SYNC(dq, q, 2 * nq);
        Q3_H2D_SYNC(dk, k, 2 * nk);
        Q3_H2D_SYNC(dv, v, 2 * nk);
        Q3_H2D_SYNC(dseg, seg_row0, sizeof(int) * n_segs);
        Q3_H2D_SYNC(dseg + n_segs, seg_len, sizeof(int) * n_segs);
        Q3_CUDA(cudaMemset(dout, 0, 2 * nq));
        int max_len = 0;
        for (int i = 0; i < n_segs; i++) max_len = std::max(max_len, seg_len[i]);
        AttnSegs segs{dseg, dseg + n_segs, n_segs, max_len};
        cudaError_t se = cudaSuccess;
        try {
            const int ldq = heads * head_dim, ldk = (heads / group) * head_dim;
            if (kernel == 0)
                flash_attn_tc_launch(dq, ldq, dk, ldk, dv, ldk, dout, ldq, segs, rows, heads, group, head_dim, causal != 0, scale, h.stream);
            else
                flash_attn_launch(dq, ldq, dk, ldk, dv, ldk, dout, ldq, segs, heads, group, head_dim, causal != 0, scale, h.stream);
            se = cudaStreamSynchronize(h.stream);
            if (se == cudaSuccess) se = cudaMemcpy(out, dout, 2 * nq, cudaMemcpyDeviceToHost);
        } catch (...) {
            cudaFree(dq); cudaFree(dk); cudaFree(dv); cudaFree(dout); cudaFree(dseg);
            throw;
        }
        cudaFree(dq); cudaFree(dk); cudaFree(dv); cudaFree(dout); cudaFree(dseg);
        Q3_CUDA(se);
    });
}

int q3asr_debug_decode_attention(q3asr_handle* hh, const float* qkv_part, int splits, int n_seqs, int heads, int kv_heads,
                                 const uint16_t* q_norm, const uint16_t* k_norm, float eps, float scale, const int* kv_len,
                                 const int* page_table, int max_pages, uint16_t* pool, int n_pages, int layers, int layer, int variant,
                                 int launches, uint16_t* out) {
    return guarded(hh, [&](Handle& h) {
        Q3_CHECK(h.loaded && h.model, Q3ASR_ERR_STATE, "debug_decode_attention: no model loaded (the RoPE frequencies come from it)");
        Q3_CHECK(qkv_part && q_norm && k_norm && kv_len && page_table && pool && out && splits >= 1 && n_seqs >= 1 && kv_heads >= 1 &&
                     heads >= 1 && max_pages >= 1 && n_pages >= 1 && layers >= 1 && layer >= 0 && layer < layers && launches >= 1,
                 Q3ASR_ERR_INVALID, "debug_decode_attention: bad argument");
        Q3_CHECK(variant == -1 || variant == 0 || variant == 1 || variant == 2 || variant == 4 || variant == 8 || variant == 16,
                 Q3ASR_ERR_INVALID, "debug_decode_attention: variant must be -1, 0, 1, 2, 4, 8 or 16");
        Q3_CHECK(variant == -1 ? (heads == kv_heads || heads == 2 * kv_heads) : heads == 2 * kv_heads, Q3ASR_ERR_INVALID,
                 "debug_decode_attention: the fused kernels take 2 query heads per kv head, the general path 1 or 2");
        for (size_t i = 0; i < (size_t)n_seqs * max_pages; i++)
            Q3_CHECK(page_table[i] >= 0 && page_table[i] < n_pages, Q3ASR_ERR_INVALID, "debug_decode_attention: page-table entry out of range");
        for (int s = 0; s < n_seqs; s++)
            Q3_CHECK(kv_len[s] >= 1 && kv_len[s] <= max_pages * KV_PAGE, Q3ASR_ERR_INVALID, "debug_decode_attention: kv_len out of range");
        const int nqkv = (heads + 2 * kv_heads) * 128, n_pos = max_pages * KV_PAGE;
        const size_t part_n = (size_t)splits * n_seqs * nqkv, out_n = (size_t)n_seqs * heads * 128;
        const size_t pool_n = (size_t)n_pages * layers * 2 * kv_heads * KV_PAGE * 128;
        DebugAllocs a;
        std::vector<int> pos(n_seqs), row_seq(n_seqs);
        for (int s = 0; s < n_seqs; s++) { pos[s] = kv_len[s] - 1; row_seq[s] = s; }
        float* dpart = a.get<float>(part_n);
        bf16 *dqw = a.get<bf16>(128), *dkw = a.get<bf16>(128), *dpool = a.get<bf16>(pool_n), *dout = a.get<bf16>(out_n * launches);
        int *dlen = a.get<int>(n_seqs), *dpos = a.get<int>(n_seqs), *dpt = a.get<int>((size_t)n_seqs * max_pages);
        float2* drope = a.get<float2>((size_t)n_pos * 64);
        Q3_H2D_SYNC(dpart, qkv_part, sizeof(float) * part_n);
        Q3_H2D_SYNC(dqw, q_norm, 2 * 128);
        Q3_H2D_SYNC(dkw, k_norm, 2 * 128);
        Q3_H2D_SYNC(dpool, pool, 2 * pool_n);
        Q3_H2D_SYNC(dlen, kv_len, sizeof(int) * n_seqs);
        Q3_H2D_SYNC(dpos, pos.data(), sizeof(int) * n_seqs);
        Q3_H2D_SYNC(dpt, page_table, sizeof(int) * (size_t)n_seqs * max_pages);
        rope_table_launch(h.model->inv_freq, n_pos, drope, nullptr, h.stream);
        const KvCache cache{dpool, dpt, max_pages, layers, kv_heads, 128};
        if (variant == -1) {  // the general path: the product's bf16 rounding of q|k|v, then the separate norm + RoPE + append kernel
            std::vector<bf16> qkv((size_t)n_seqs * nqkv);
            for (size_t i = 0; i < qkv.size(); i++) {
                float acc = 0.f;
                for (int sp = 0; sp < splits; sp++) acc += qkv_part[(size_t)sp * n_seqs * nqkv + i];
                qkv[i] = __float2bfloat16_rn(acc);
            }
            bf16 *dqkv = a.get<bf16>(qkv.size()), *dq = a.get<bf16>(out_n);
            int* drow = a.get<int>(n_seqs);
            Q3_H2D_SYNC(dqkv, qkv.data(), 2 * qkv.size());
            Q3_H2D_SYNC(drow, row_seq.data(), sizeof(int) * n_seqs);
            for (int i = 0; i < launches; i++) {
                qknorm_rope_kv_launch(dqkv, nqkv, dqw, dkw, dpos, drow, n_seqs, heads, kv_heads, eps, drope, dq, nullptr, nullptr, cache, layer,
                                      h.stream);
                decode_attn_launch(dq, cache, layer, dlen, n_seqs, heads, scale, dout + i * out_n, h.stream);
            }
        } else {  // the fused kernels; the split variant's counters start at zero, as reserve_decoder leaves them
            float* dsplit = a.get<float>(decode_attn_split_floats(n_seqs, kv_heads));
            int* dcnt = a.get<int>((size_t)n_seqs * kv_heads);
            Q3_CUDA(cudaMemsetAsync(dcnt, 0, sizeof(int) * n_seqs * kv_heads, h.stream));
            struct PdlOn {  // back-to-back launches overlap as in the decode step: each one's prefetch runs ahead of the previous launch's end
                bool prev = pdl_enabled();
                PdlOn() { pdl_enabled() = true; }
                ~PdlOn() { pdl_enabled() = prev; }
            } pdl;
            for (int i = 0; i < launches; i++)
                decode_attn_fused_launch(dpart, splits, (long long)n_seqs * nqkv, nqkv, dqw, dkw, dpos, eps, drope, cache, layer, dlen, n_seqs,
                                         heads, scale, dout + i * out_n, h.num_sms, h.stream, dsplit, dcnt, variant);
        }
        Q3_CUDA(cudaStreamSynchronize(h.stream));
        Q3_CUDA(cudaMemcpy(out, dout, 2 * out_n * launches, cudaMemcpyDeviceToHost));
        Q3_CUDA(cudaMemcpy(pool, dpool, 2 * pool_n, cudaMemcpyDeviceToHost));
    });
}

int q3asr_debug_prefill_attention(q3asr_handle* hh, const uint16_t* x, const uint16_t* w, int rows, int hidden, int heads, int kv_heads,
                                  const uint16_t* q_norm, const uint16_t* k_norm, float eps, float scale, const int* seg_row0,
                                  const int* seg_len, const int* seg_table_row, int n_segs, const int* page_table, int table_rows,
                                  int max_pages, uint16_t* pool, int n_pages, int layers, int layer, int qkv_variant, int bn,
                                  int attn_variant, uint16_t* q_out, uint16_t* k_out, uint16_t* qkv_out, uint16_t* att_out) {
    return guarded(hh, [&](Handle& h) {
        Q3_CHECK(h.loaded && h.model, Q3ASR_ERR_STATE, "debug_prefill_attention: no model loaded (the RoPE frequencies come from it)");
        Q3_CHECK(x && w && q_norm && k_norm && seg_row0 && seg_len && seg_table_row && page_table && pool && q_out && k_out && qkv_out &&
                     att_out && rows >= 1 && hidden >= 64 && hidden % 64 == 0 && heads >= 1 && kv_heads >= 1 && heads % kv_heads == 0 &&
                     n_segs >= 1 && table_rows >= 1 && max_pages >= 1 && n_pages >= 1 && layers >= 1 && layer >= 0 && layer < layers,
                 Q3ASR_ERR_INVALID, "debug_prefill_attention: bad argument");
        const int nq = heads * 128, nkv = kv_heads * 128, nqkv = nq + 2 * nkv, n_pos = max_pages * KV_PAGE;
        Q3_CHECK(qkv_variant == 0 || qkv_variant == -1, Q3ASR_ERR_INVALID, "debug_prefill_attention: qkv_variant must be 0 or -1");
        Q3_CHECK(bn == 0 || ((bn == 128 || bn == 256) && nqkv % bn == 0), Q3ASR_ERR_INVALID,
                 "debug_prefill_attention: bn must be 0, or 128 / 256 dividing (heads + 2 kv_heads) * 128");
        Q3_CHECK(attn_variant >= -1 && attn_variant <= 1, Q3ASR_ERR_INVALID, "debug_prefill_attention: attn_variant must be -1, 0 or 1");
        for (size_t i = 0; i < (size_t)table_rows * max_pages; i++)
            Q3_CHECK(page_table[i] >= 0 && page_table[i] < n_pages, Q3ASR_ERR_INVALID, "debug_prefill_attention: page-table entry out of range");
        // the segments tile the rows back to back, as the batch plan packs the prompts
        std::vector<int> pos(rows), row_seq(rows);
        int next = 0, max_len = 0;
        for (int s = 0; s < n_segs; s++) {
            Q3_CHECK(seg_row0[s] == next && seg_len[s] >= 1 && seg_len[s] <= n_pos && seg_len[s] <= rows - next, Q3ASR_ERR_INVALID,
                     "debug_prefill_attention: segments must be packed back to back, each within the table's positions");
            Q3_CHECK(seg_table_row[s] >= 0 && seg_table_row[s] < table_rows, Q3ASR_ERR_INVALID,
                     "debug_prefill_attention: segment table row out of range");
            for (int i = 0; i < seg_len[s]; i++) {
                pos[next + i] = i;
                row_seq[next + i] = seg_table_row[s];
            }
            next += seg_len[s];
            max_len = std::max(max_len, seg_len[s]);
        }
        Q3_CHECK(next == rows, Q3ASR_ERR_INVALID, "debug_prefill_attention: the segments must cover the rows");
        const size_t pool_n = (size_t)n_pages * layers * 2 * kv_heads * KV_PAGE * 128;
        DebugAllocs a;
        bf16 *dx = a.get<bf16>((size_t)rows * hidden), *dw = a.get<bf16>((size_t)nqkv * hidden), *dqw = a.get<bf16>(128),
             *dkw = a.get<bf16>(128), *dpool = a.get<bf16>(pool_n), *dqkv = a.get<bf16>((size_t)rows * nqkv), *dq = a.get<bf16>((size_t)rows * nq),
             *dk = a.get<bf16>((size_t)rows * nkv), *datt = a.get<bf16>((size_t)rows * nq);
        int *dpt = a.get<int>((size_t)table_rows * max_pages), *dpos = a.get<int>(rows), *drow = a.get<int>(rows), *dseg = a.get<int>(2 * (size_t)n_segs);
        float2 *drope = a.get<float2>((size_t)n_pos * 64), *drope_t = a.get<float2>((size_t)n_pos * 64);
        Q3_H2D_SYNC(dx, x, 2 * (size_t)rows * hidden);
        Q3_H2D_SYNC(dw, w, 2 * (size_t)nqkv * hidden);
        Q3_H2D_SYNC(dqw, q_norm, 2 * 128);
        Q3_H2D_SYNC(dkw, k_norm, 2 * 128);
        Q3_H2D_SYNC(dpool, pool, 2 * pool_n);
        Q3_H2D_SYNC(dpt, page_table, sizeof(int) * (size_t)table_rows * max_pages);
        Q3_H2D_SYNC(dpos, pos.data(), sizeof(int) * rows);
        Q3_H2D_SYNC(drow, row_seq.data(), sizeof(int) * rows);
        Q3_H2D_SYNC(dseg, seg_row0, sizeof(int) * n_segs);
        Q3_H2D_SYNC(dseg + n_segs, seg_len, sizeof(int) * n_segs);
        // every output element the call does not write reads back as bf16 NaN (0xFFFF)
        Q3_CUDA(cudaMemsetAsync(dqkv, 0xFF, 2 * (size_t)rows * nqkv, h.stream));
        Q3_CUDA(cudaMemsetAsync(dq, 0xFF, 2 * (size_t)rows * nq, h.stream));
        Q3_CUDA(cudaMemsetAsync(dk, 0xFF, 2 * (size_t)rows * nkv, h.stream));
        Q3_CUDA(cudaMemsetAsync(datt, 0xFF, 2 * (size_t)rows * nq, h.stream));
        rope_table_launch(h.model->inv_freq, n_pos, drope, drope_t, h.stream);
        const PrefillAttn pa{dx, dw, dqw, dkw, rows, hidden, heads, kv_heads, eps, scale, dpos, drow, AttnSegs{dseg, dseg + n_segs, n_segs, max_len},
                             drope, drope_t, n_pos, KvCache{dpool, dpt, max_pages, layers, kv_heads, 128}, layer, dqkv, dq, dk, datt};
        prefill_attention(&h, pa, qkv_variant == 0, bn, attn_variant, 0.0);
        Q3_CUDA(cudaStreamSynchronize(h.stream));
        Q3_CUDA(cudaMemcpy(q_out, dq, 2 * (size_t)rows * nq, cudaMemcpyDeviceToHost));
        Q3_CUDA(cudaMemcpy(k_out, dk, 2 * (size_t)rows * nkv, cudaMemcpyDeviceToHost));
        Q3_CUDA(cudaMemcpy(qkv_out, dqkv, 2 * (size_t)rows * nqkv, cudaMemcpyDeviceToHost));
        Q3_CUDA(cudaMemcpy(att_out, datt, 2 * (size_t)rows * nq, cudaMemcpyDeviceToHost));
        Q3_CUDA(cudaMemcpy(pool, dpool, 2 * pool_n, cudaMemcpyDeviceToHost));
    });
}

}  // extern "C"
