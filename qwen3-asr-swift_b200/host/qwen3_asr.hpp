// qwen3_asr.hpp — C++ host-side mirror of the reference's Swift API for the batch-transcription path,
// written above the C ABI (include/q3asr.h).  The reference's own language (Swift) has no toolchain in
// this image, so this header plays the role the Swift shim (swift/Qwen3ASRB200.swift) plays on a Mac/Linux
// box with Swift: same type and method names, same defaults, same error behaviour.
//
//   Qwen3DecodingOptions                     Sources/Qwen3ASR/Qwen3ASR.swift:13-51
//   ASRModelSize / detect                    Sources/Qwen3ASR/Qwen3ASR.swift:541-586
//   MelFeatures / WhisperFeatureExtractor    Sources/Qwen3ASR/AudioPreprocessing.swift:8-18, 347
//   Qwen3ASRModel::fromPretrained            Sources/Qwen3ASR/Qwen3ASR.swift:608-668  (load: throws)
//   Qwen3ASRModel::transcribe (2 overloads)  Sources/Qwen3ASR/Qwen3ASR.swift:107-164  (inference: never throws)
//   isLoaded / unload / memoryFootprint      Sources/Qwen3ASR/Qwen3ASR+Memory.swift:3-17
//   inputSampleRate                          Sources/Qwen3ASR/Qwen3ASR+Protocols.swift:5-11
//   AudioFileLoader::loadWAV / resample      Sources/AudioCommon/AudioFileLoader.swift:70-213 (AudioLoadError :216-234)
//   TranscriptionSegment                     Sources/Qwen3ASR/StreamingASR.swift:7-21 (long-form windows instead of VAD segments)
// Header-only; link with -lq3asr.  Not thread-safe per instance (Qwen3ASR.swift:67).
#pragma once
#include <algorithm>
#include <cctype>
#include <cstdint>
#include <functional>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/q3asr.h"

namespace qwen3asr {

struct Qwen3DecodingOptions {
    int maxTokens = 448;
    std::optional<std::string> language;
    std::optional<std::string> context;
    float repetitionPenalty = 1.0f;
    int noRepeatNgramSize = 0;
    float temperature = 0.0f;
    uint64_t seed = 0;  // keys the reproducible Gumbel noise stream of the device sampler (the reference uses the system RNG)
    bool isGreedyFastPath() const {  // Qwen3ASR.swift:300-304
        return temperature == 0.0f && repetitionPenalty == 1.0f && noRepeatNgramSize == 0;
    }
};

enum class ASRModelSize { small, large };
inline ASRModelSize detectModelSize(const std::string& modelId) {  // Qwen3ASR.swift:581-586: "1.7B"/"1.7b" in the id -> large
    std::string s = modelId;
    std::transform(s.begin(), s.end(), s.begin(), [](unsigned char c) { return (char)std::tolower(c); });
    return s.find("1.7b") != std::string::npos ? ASRModelSize::large : ASRModelSize::small;
}
// Qwen3ASR.swift:588-600: "8bit"/"8-bit" or "4bit"/"4-bit" in the id, else 4 for the small model and 8 for the large one.  The
// loader itself reads the packing from the tensor shapes (csrc/safetensors.cu); this is the id convention of the reference.
inline int detectModelBits(const std::string& modelId) {
    std::string s = modelId;
    std::transform(s.begin(), s.end(), s.begin(), [](unsigned char c) { return (char)std::tolower(c); });
    if (s.find("8bit") != std::string::npos || s.find("8-bit") != std::string::npos) return 8;
    if (s.find("4bit") != std::string::npos || s.find("4-bit") != std::string::npos) return 4;
    return detectModelSize(modelId) == ASRModelSize::large ? 8 : 4;
}

// The preset a checkpoint directory holds, from its validated tensor index (q3asr_checkpoint_list, host only): "aligner" when it
// carries lm_head.*, else "0.6B" / "1.7B" by the width of model.norm.weight; "" when the index does not say.
inline std::string detectPresetFromCheckpoint(const std::string& dir) {
    size_t need = 0;
    if (q3asr_checkpoint_list(dir.c_str(), nullptr, 0, &need) != Q3ASR_OK || need == 0) return "";
    std::string list(need, '\0');
    if (q3asr_checkpoint_list(dir.c_str(), &list[0], list.size(), &need) != Q3ASR_OK) return "";
    if (list.find("\nlm_head.weight\t") != std::string::npos || list.compare(0, 15, "lm_head.weight\t") == 0) return "aligner";
    const size_t at = list.find("model.norm.weight\t");
    if (at == std::string::npos || (at != 0 && list[at - 1] != '\n')) return "";
    const size_t shape = list.find('\t', list.find('\t', at) + 1) + 1;  // name \t dtype \t shape \t bytes
    const std::string dims = list.substr(shape, list.find('\t', shape) - shape);
    return dims == "1024" ? "0.6B" : dims == "2048" ? "1.7B" : "";
}

struct MelFeatures {  // row-major [melBins, timeFrames]
    std::vector<float> data;
    int melBins = 128;
    int timeFrames = 0;
};

struct AudioModelError : std::runtime_error {  // AudioCommon/AudioModelError.swift:4-34 (modelLoadFailed / weightLoadingFailed)
    int code;
    AudioModelError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

// token-id <-> text: any pair of functions, or the library's own byte-level BPE tokenizer (Qwen3Tokenizer,
// AudioCommon/Tokenizer.swift) loaded from the checkpoint directory's vocab.json / tokenizer_config.json / merges.txt
struct Tokenizer {
    std::function<std::vector<int32_t>(const std::string&)> encode;
    std::function<std::string(const std::vector<int32_t>&)> decode;

    static Tokenizer fromDirectory(const std::string& dir) {
        q3asr_tokenizer* raw = nullptr;
        const int rc = q3asr_tokenizer_load(dir.c_str(), &raw);
        std::shared_ptr<q3asr_tokenizer> t(raw, q3asr_tokenizer_destroy);
        if (rc != Q3ASR_OK) throw AudioModelError(rc, std::string("tokenizer: ") + q3asr_tokenizer_last_error(raw));
        Tokenizer out;
        out.encode = [t](const std::string& text) {
            int n = 0;
            q3asr_tokenizer_encode(t.get(), text.c_str(), nullptr, 0, &n);
            std::vector<int32_t> ids((size_t)std::max(n, 1));
            q3asr_tokenizer_encode(t.get(), text.c_str(), ids.data(), (int)ids.size(), &n);
            ids.resize((size_t)n);
            return ids;
        };
        out.decode = [t](const std::vector<int32_t>& ids) {
            size_t need = 0;
            q3asr_tokenizer_decode(t.get(), ids.data(), (int)ids.size(), nullptr, 0, &need);
            std::string s(need, '\0');
            q3asr_tokenizer_decode(t.get(), ids.data(), (int)ids.size(), &s[0], need, nullptr);
            s.resize(need ? need - 1 : 0);
            return s;
        };
        return out;
    }
};

struct AudioLoadError : std::runtime_error {  // AudioFileLoader.swift:216-234
    int code;
    AudioLoadError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

struct TranscriptionSegment {  // StreamingASR.swift:7-21
    std::string text;
    float startTime = 0.f, endTime = 0.f;
    bool isFinal = true;
    int segmentIndex = 0;
    float avgLogprob = 0.f;  // transcribeLong(..., withConfidence = true) only: mean token log-probability of the window
};

// a transcript with its score: mean token log-probability (EOS included, include/q3asr.h); confidence = exp(avgLogprob)
struct ScoredTranscript {
    std::string text;
    float avgLogprob = 0.f;
};

class Qwen3ASRModel;

struct AudioFileLoader {
    struct Wav {
        std::vector<float> samples;
        int sampleRate = 0;
    };
    // AudioFileLoader.loadWAV: 16-bit PCM, first channel; throws AudioLoadError like the reference
    static Wav loadWAV(const std::string& path) {
        Wav w;
        size_t n = 0;
        int rc = q3asr_wav_load(path.c_str(), nullptr, 0, &n, &w.sampleRate);
        if (rc != Q3ASR_OK) throw AudioLoadError(rc, q3asr_io_last_error());
        w.samples.assign(n, 0.f);
        rc = q3asr_wav_load(path.c_str(), w.samples.data(), n, &n, &w.sampleRate);
        if (rc != Q3ASR_OK) throw AudioLoadError(rc, q3asr_io_last_error());
        return w;
    }
    // AudioFileLoader.resample: returns the input unchanged when the conversion cannot run (the reference's own fallback, :175, :207)
    static std::vector<float> resample(const Qwen3ASRModel& model, const std::vector<float>& samples, int from, int to);
};

struct WAVWriter {  // Sources/AudioCommon/WAVWriter.swift:11-47: mono 16-bit PCM; throws AudioLoadError when the file cannot be written
    static void write(const std::vector<float>& samples, int sampleRate, const std::string& path) {
        const int rc = q3asr_wav_write(path.c_str(), samples.data(), samples.size(), sampleRate);
        if (rc != Q3ASR_OK) throw AudioLoadError(rc, q3asr_io_last_error());
    }
};

class WhisperFeatureExtractor {
  public:
    static constexpr int sampleRate = 16000, nFFT = 400, hopLength = 160, nMels = 128;  // AudioPreprocessing.swift:24-30
    MelFeatures extractFeaturesRaw(const std::vector<float>& audio) const {
        MelFeatures m;
        m.timeFrames = q3asr_mel_frames(audio.size());
        m.data.assign((size_t)128 * std::max(m.timeFrames, 0), 0.f);
        int frames = 0;
        if (q3asr_mel(h_, audio.data(), audio.size(), m.data.data(), &frames) != Q3ASR_OK) {
            m.timeFrames = 0;
            m.data.clear();
        } else {
            m.timeFrames = frames;
        }
        return m;
    }

  private:
    friend class Qwen3ASRModel;
    q3asr_handle* h_ = nullptr;
};

class Qwen3ASRModel {
  public:
    WhisperFeatureExtractor featureExtractor;
    static constexpr int inputSampleRate = 16000;

    // modelDir: a directory holding the checkpoint's *.safetensors (the reference resolves it from the HF cache);
    // modelId decides the size like ASRModelSize.detect unless the checkpoint's own tensor index says otherwise.  Throws
    // AudioModelError on load failure.
    static std::unique_ptr<Qwen3ASRModel> fromPretrained(const std::string& modelId, const std::string& modelDir, int device = 0,
                                                         std::function<void(double, const std::string&)> progressHandler = nullptr) {
        if (progressHandler) progressHandler(0.0, "Loading model...");
        ASRModelSize size = detectModelSize(modelId);
        const std::string held = detectPresetFromCheckpoint(modelDir);  // what the files say wins over the name
        if (held == "1.7B") size = ASRModelSize::large;
        else if (held == "0.6B") size = ASRModelSize::small;
        std::unique_ptr<Qwen3ASRModel> m(new Qwen3ASRModel(size, device));
        int rc = q3asr_load_safetensors(m->h_, modelDir.c_str());
        if (rc != Q3ASR_OK) throw AudioModelError(rc, std::string("weightLoadingFailed: ") + q3asr_last_error(m->h_));
        try {  // Qwen3ASR.swift:643-649: the tokenizer is optional (ids are returned as text without it, :288-289)
            m->tok_ = Tokenizer::fromDirectory(modelDir);
        } catch (const AudioModelError&) {
        }
        if (progressHandler) progressHandler(1.0, "Ready");
        return m;
    }
    // random-init weights of the right architecture (weights are not available offline; parity / bench runs)
    static std::unique_ptr<Qwen3ASRModel> randomInit(ASRModelSize size, uint64_t seed = 20260418, int device = 0) {
        std::unique_ptr<Qwen3ASRModel> m(new Qwen3ASRModel(size, device));
        int rc = q3asr_init_random(m->h_, seed);
        if (rc != Q3ASR_OK) throw AudioModelError(rc, std::string("modelLoadFailed: ") + q3asr_last_error(m->h_));
        return m;
    }
    ~Qwen3ASRModel() { q3asr_destroy(h_); }
    Qwen3ASRModel(const Qwen3ASRModel&) = delete;
    Qwen3ASRModel& operator=(const Qwen3ASRModel&) = delete;

    void setTokenizer(Tokenizer t) { tok_ = std::move(t); }

    // Qwen3ASR.swift:131-137.  Other sample rates are converted to 16 kHz on the device first (AudioPreprocessing.swift:323-337).
    // Never throws.
    std::string transcribe(const std::vector<float>& audio, int sampleRate = 16000, const std::optional<std::string>& language = {},
                           int maxTokens = 448, const std::optional<std::string>& context = {}) {
        return transcribeBatch({&audio}, language, maxTokens, context, {sampleRate})[0];
    }
    // Qwen3ASR.swift:107-111
    std::string transcribe(const std::vector<float>& audio, int sampleRate, const Qwen3DecodingOptions& options) {
        // the decoder knobs (repetition penalty, no-repeat n-gram, temperature) run as a device kernel (Qwen3ASR.swift:396-520)
        return transcribeBatch({&audio}, options.language, options.maxTokens, options.context, {sampleRate}, &options)[0];
    }
    // SpeechRecognitionModel.transcribe(audio:sampleRate:language:)
    std::string transcribe(const std::vector<float>& audio, int sampleRate, const std::optional<std::string>& language) {
        return transcribe(audio, sampleRate, language, 448);
    }

    // the batched entry the utterance scheduler enables; ids per utterance (EOS included when hit, like the reference loop)
    std::vector<std::vector<int32_t>> transcribeIds(const std::vector<const std::vector<float>*>& audio, int maxTokens = 448,
                                                    bool stopOnEos = true, const std::vector<int32_t>& contextIds = {},
                                                    const std::vector<int32_t>& languageIds = {}, std::string* error = nullptr,
                                                    const std::vector<int>& sampleRates = {}, const Qwen3DecodingOptions* options = nullptr,
                                                    std::vector<std::vector<float>>* logprobs = nullptr) {
        const int n = (int)audio.size();
        if (logprobs) logprobs->assign(n, {});
        if (!sampleRates.empty() && (int)sampleRates.size() != n) {
            if (error) *error = "sampleRates must have one entry per utterance";
            return std::vector<std::vector<int32_t>>(n);
        }
        std::vector<const float*> pcm(n);
        std::vector<size_t> len(n);
        for (int i = 0; i < n; i++) {
            pcm[i] = audio[i]->data();
            len[i] = audio[i]->size();
        }
        q3asr_prompt pr{contextIds.data(), (int)contextIds.size(), languageIds.data(), (int)languageIds.size()};
        std::vector<q3asr_prompt> prompts(n, pr);
        std::vector<int32_t> ids((size_t)n * maxTokens);
        std::vector<int> lens(n);
        std::vector<std::vector<int32_t>> out(n);
        q3asr_sampling samp{1.0f, 0, 0.0f, 0, 0};
        if (options) samp = q3asr_sampling{options->repetitionPenalty, options->noRepeatNgramSize, options->temperature, options->seed, 0};
        std::vector<float> lp(logprobs ? (size_t)n * maxTokens : 0);
        int rc = q3asr_transcribe_ids_lp(h_, pcm.data(), len.data(), sampleRates.empty() ? nullptr : sampleRates.data(), n, prompts.data(),
                                         options ? &samp : nullptr, maxTokens, stopOnEos ? 1 : 0, ids.data(), lens.data(),
                                         logprobs ? lp.data() : nullptr);
        if (rc != Q3ASR_OK) {
            if (error) *error = q3asr_last_error(h_);
            return out;
        }
        for (int i = 0; i < n; i++) {
            out[i].assign(ids.begin() + (size_t)i * maxTokens, ids.begin() + (size_t)i * maxTokens + lens[i]);
            if (logprobs) (*logprobs)[i].assign(lp.begin() + (size_t)i * maxTokens, lp.begin() + (size_t)i * maxTokens + lens[i]);
        }
        return out;
    }

    std::vector<std::string> transcribeBatch(const std::vector<const std::vector<float>*>& audio, const std::optional<std::string>& language = {},
                                             int maxTokens = 448, const std::optional<std::string>& context = {},
                                             const std::vector<int>& sampleRates = {}, const Qwen3DecodingOptions* options = nullptr) {
        std::vector<std::string> out;
        for (ScoredTranscript& t : run(audio, language, maxTokens, context, sampleRates, options, false)) out.push_back(std::move(t.text));
        return out;
    }

    // transcribeBatch plus each utterance's mean token log-probability (0 for an utterance without tokens or after an error)
    std::vector<ScoredTranscript> transcribeBatchWithConfidence(const std::vector<const std::vector<float>*>& audio,
                                                                const std::optional<std::string>& language = {}, int maxTokens = 448,
                                                                const std::optional<std::string>& context = {},
                                                                const std::vector<int>& sampleRates = {},
                                                                const Qwen3DecodingOptions* options = nullptr) {
        return run(audio, language, maxTokens, context, sampleRates, options, true);
    }

    // trimmingCharacters(in: .whitespaces): Unicode space separators (Zs) and TAB at either end, not line breaks
    static std::string trimSwiftWhitespaces(const std::string& s) {
        static const char* const ws[] = {" ", "\t", "\xC2\xA0", "\xE1\x9A\x80", "\xE2\x80\x80", "\xE2\x80\x81", "\xE2\x80\x82", "\xE2\x80\x83",
                                         "\xE2\x80\x84", "\xE2\x80\x85", "\xE2\x80\x86", "\xE2\x80\x87", "\xE2\x80\x88", "\xE2\x80\x89",
                                         "\xE2\x80\x8A", "\xE2\x80\xAF", "\xE2\x81\x9F", "\xE3\x80\x80"};
        size_t a = 0, b = s.size();
        for (bool again = true; again;) {
            again = false;
            for (const char* w : ws) {
                const size_t n = strlen(w);
                if (b - a >= n && s.compare(a, n, w) == 0) { a += n; again = true; }
                if (b - a >= n && s.compare(b - n, n, w) == 0) { b -= n; again = true; }
            }
        }
        return s.substr(a, b - a);
    }

    // generated ids -> transcript (Qwen3ASR.swift:283-289): decode, keep what follows "<asr_text>", trim; without a tokenizer the ids
    // joined by spaces (the reference's own fallback)
    static std::string textFromIds(const Tokenizer& tok, const std::vector<int32_t>& t) {
        std::string out;
        if (tok.decode) {
            std::string raw = tok.decode(t);
            const size_t at = raw.find("<asr_text>");
            if (at != std::string::npos) raw = raw.substr(at + 10);
            out = trimSwiftWhitespaces(raw);
        } else {
            for (size_t j = 0; j < t.size(); j++) out += (j ? " " : "") + std::to_string(t[j]);
        }
        return out;
    }

    // Long-form audio (BASELINE config 5): fixed windows of windowSeconds, each an independent utterance, `batch` windows per pass.
    std::vector<TranscriptionSegment> transcribeLong(const std::vector<float>& audio, int sampleRate = 16000, float windowSeconds = 30.f,
                                                     int maxTokens = 448, int batch = 64, const std::optional<std::string>& language = {},
                                                     bool withConfidence = false) {
        std::vector<TranscriptionSegment> out;
        const size_t window = (size_t)((double)windowSeconds * sampleRate + 0.5);
        const size_t minTail = std::max<size_t>(160, ((size_t)160 * sampleRate + 15999) / 16000);
        int count = 0;
        if (window == 0 || q3asr_longform_plan(audio.size(), window, minTail, nullptr, nullptr, 0, &count) != Q3ASR_OK || count == 0) return out;
        std::vector<size_t> starts((size_t)count), lens((size_t)count);
        q3asr_longform_plan(audio.size(), window, minTail, starts.data(), lens.data(), count, &count);
        for (int b0 = 0; b0 < count; b0 += std::max(batch, 1)) {
            const int nb = std::min(std::max(batch, 1), count - b0);
            std::vector<std::vector<float>> clips((size_t)nb);
            std::vector<const std::vector<float>*> ptrs((size_t)nb);
            for (int i = 0; i < nb; i++) {
                clips[i].assign(audio.begin() + starts[b0 + i], audio.begin() + starts[b0 + i] + lens[b0 + i]);
                ptrs[i] = &clips[i];
            }
            auto texts = run(ptrs, language, maxTokens, {}, std::vector<int>((size_t)nb, sampleRate), nullptr, withConfidence);
            for (int i = 0; i < nb; i++) {
                TranscriptionSegment seg;
                seg.text = texts[i].text;
                seg.avgLogprob = texts[i].avgLogprob;
                seg.startTime = (float)((double)starts[b0 + i] / sampleRate);
                seg.endTime = (float)((double)(starts[b0 + i] + lens[b0 + i]) / sampleRate);
                seg.segmentIndex = b0 + i;
                out.push_back(seg);
            }
        }
        return out;
    }

    // ModelMemoryManageable
    bool isLoaded() const { return q3asr_is_loaded(h_) != 0; }
    void unload() { q3asr_unload(h_); }
    size_t memoryFootprint() const { return q3asr_memory_footprint(h_); }
    q3asr_handle* handle() const { return h_; }

  private:
    std::vector<ScoredTranscript> run(const std::vector<const std::vector<float>*>& audio, const std::optional<std::string>& language,
                                      int maxTokens, const std::optional<std::string>& context, const std::vector<int>& sampleRates,
                                      const Qwen3DecodingOptions* options, bool scored) {
        const size_t n = audio.size();
        if (!isLoaded()) return std::vector<ScoredTranscript>(n, {"[Audio encoded] - Text decoder not loaded", 0.f});  // Qwen3ASR.swift:116-119
        std::vector<int32_t> ctx, lang;
        if (tok_.encode) {
            if (context) ctx = tok_.encode(*context);                  // Qwen3ASR.swift:203-206
            if (language) lang = tok_.encode("language " + *language);  // Qwen3ASR.swift:228-232
        }
        std::string err;
        std::vector<std::vector<float>> lp;
        auto ids = transcribeIds(audio, maxTokens, true, ctx, lang, &err, sampleRates, options, scored ? &lp : nullptr);
        std::vector<ScoredTranscript> out(n);
        for (size_t i = 0; i < n; i++) {
            if (!err.empty()) {
                out[i].text = "[Qwen3-ASR B200 error: " + err + "]";
                continue;
            }
            out[i].text = textFromIds(tok_, ids[i]);
            if (scored && !lp[i].empty()) {
                double sum = 0;
                for (float v : lp[i]) sum += v;
                out[i].avgLogprob = (float)(sum / lp[i].size());
            }
        }
        return out;
    }

    Qwen3ASRModel(ASRModelSize size, int device) {
        q3asr_config cfg;
        q3asr_config_preset(size == ASRModelSize::large ? "1.7B" : "0.6B", &cfg);
        int rc = q3asr_create(&cfg, device, &h_);
        if (rc != Q3ASR_OK) throw AudioModelError(rc, std::string("modelLoadFailed: ") + q3asr_last_error(nullptr));
        featureExtractor.h_ = h_;
    }
    q3asr_handle* h_ = nullptr;
    Tokenizer tok_;
};

struct AlignedWord {  // AudioCommon/Protocols.swift (AlignedWord)
    std::string text;
    float startTime = 0.f, endTime = 0.f;
};

// Qwen3ForcedAligner (ForcedAligner.swift:50-331) over q3asr_align_indices.  Word splitting: the whitespace path of
// TextPreprocessor.splitIntoWordPairs (TextPreprocessing.swift: letters, digits and the ASCII apostrophe are kept, other ASCII
// punctuation is stripped from the form the tokenizer sees; non-ASCII bytes are kept as they are).  The Japanese / Korean / per-Han
// paths of the reference need Apple's NaturalLanguage framework and are not reproduced.
class Qwen3ForcedAligner {
  public:
    static constexpr float timestampSegmentTime = 0.08f;  // Configuration.swift:133
    static std::unique_ptr<Qwen3ForcedAligner> randomInit(uint64_t seed = 20260418, int device = 0, const char* preset = "aligner") {
        std::unique_ptr<Qwen3ForcedAligner> m(new Qwen3ForcedAligner(preset, device));
        if (q3asr_init_random(m->h_, seed) != Q3ASR_OK) throw AudioModelError(1, std::string("modelLoadFailed: ") + q3asr_last_error(m->h_));
        return m;
    }
    static std::unique_ptr<Qwen3ForcedAligner> fromPretrained(const std::string& modelDir, int device = 0) {
        std::unique_ptr<Qwen3ForcedAligner> m(new Qwen3ForcedAligner("aligner", device));
        int rc = q3asr_load_safetensors(m->h_, modelDir.c_str());
        if (rc != Q3ASR_OK) throw AudioModelError(rc, std::string("weightLoadingFailed: ") + q3asr_last_error(m->h_));
        m->tok_ = Tokenizer::fromDirectory(modelDir);  // the aligner cannot work without one (ForcedAligner.swift:232-235)
        return m;
    }
    ~Qwen3ForcedAligner() { q3asr_destroy(h_); }
    Qwen3ForcedAligner(const Qwen3ForcedAligner&) = delete;
    Qwen3ForcedAligner& operator=(const Qwen3ForcedAligner&) = delete;
    void setTokenizer(Tokenizer t) { tok_ = std::move(t); }
    int timestampTokenId = 151705;  // Qwen3ASR.swift:62 (the tests' tiny vocabulary overrides it)

    struct WordPair { std::string surface, cleaned; };
    // TextPreprocessor.splitIntoWordPairs (TextPreprocessing.swift:97-115) through the library's Unicode-aware splitter.  Throws
    // AudioModelError for the languages the reference hands to NLTokenizer (Japanese, Korean, Thai, ...).
    static std::vector<WordPair> splitIntoWordPairs(const std::string& text, const std::string& language = "English") {
        size_t need = 0;
        int n = 0;
        int rc = q3asr_text_word_pairs(text.c_str(), language.c_str(), nullptr, 0, &need, &n);
        std::string flat(need, '\0');
        if (rc == Q3ASR_OK && need) rc = q3asr_text_word_pairs(text.c_str(), language.c_str(), &flat[0], flat.size(), &need, &n);
        if (rc != Q3ASR_OK) throw AudioModelError(rc, std::string("text: ") + q3asr_text_last_error());
        std::vector<WordPair> out;
        const char* p = flat.data();
        for (int i = 0; i < n; i++) {
            WordPair w;
            w.surface = p;
            p += w.surface.size() + 1;
            w.cleaned = p;
            p += w.cleaned.size() + 1;
            out.push_back(std::move(w));
        }
        return out;
    }

    // ForcedAligner.swift:226-331.  Returns [] when no tokenizer is set or the text has no words (like the reference).
    std::vector<AlignedWord> align(const std::vector<float>& audio, const std::string& text, int sampleRate = 16000,
                                   const std::string& language = "English") {
        std::vector<AlignedWord> out;
        if (!tok_.encode) return out;
        std::vector<int32_t> ids;
        std::vector<int> pos;
        std::vector<std::string> words;
        for (const WordPair& w : splitIntoWordPairs(text, language)) {  // TextPreprocessing.swift:48-80: <timestamp> word tokens <timestamp>
            const std::vector<int32_t> t = tok_.encode(w.cleaned);
            if (t.empty()) {
                if (!words.empty()) words.back() += w.surface;
                continue;
            }
            pos.push_back((int)ids.size());
            ids.push_back(timestampTokenId);
            ids.insert(ids.end(), t.begin(), t.end());
            pos.push_back((int)ids.size());
            ids.push_back(timestampTokenId);
            words.push_back(w.surface);
        }
        if (words.empty()) return out;
        const float* pcm = audio.data();
        const size_t n = audio.size();
        const int32_t* sl = ids.data();
        const int nsl = (int)ids.size(), np = (int)pos.size();
        const int* pp = pos.data();
        std::vector<int32_t> raw((size_t)np);
        int32_t* rp = raw.data();
        if (q3asr_align_indices(h_, &pcm, &n, &sampleRate, 1, &sl, &nsl, &pp, &np, &rp) != Q3ASR_OK) return out;
        std::vector<int> r(raw.begin(), raw.end()), fixed((size_t)np);
        q3asr_enforce_monotonicity(r.data(), np, fixed.data());
        for (size_t w = 0; w < words.size(); w++) {
            const float st = (float)fixed[2 * w] * timestampSegmentTime, en = (float)fixed[2 * w + 1] * timestampSegmentTime;
            out.push_back(AlignedWord{words[w], st, std::max(en, st)});
        }
        return out;
    }

    // ForcedAligner.swift:104-176: re-align the remainder when the tail of a long recording collapses onto one timestamp
    std::vector<AlignedWord> alignLong(const std::vector<float>& audio, const std::string& text, int sampleRate = 16000,
                                       const std::string& language = "English") {
        const float bypassThresholdSeconds = 240.f, minChunkSeconds = 5.f, plateauTolerance = 0.1f;
        const int plateauMinWords = 5;
        std::vector<AlignedWord> all;
        std::vector<float> remAudio = audio;
        std::string remText = text;
        float offset = 0.f;
        for (int pass = 1; !remAudio.empty() && !remText.empty() && pass <= 10; pass++) {
            const float duration = (float)remAudio.size() / (float)sampleRate;
            std::vector<AlignedWord> a = align(remAudio, remText, sampleRate, language);
            if (a.empty()) break;
            auto append = [&](size_t count) {
                for (size_t i = 0; i < count; i++) all.push_back(AlignedWord{a[i].text, a[i].startTime + offset, a[i].endTime + offset});
            };
            if (duration <= bypassThresholdSeconds || (int)a.size() < plateauMinWords * 2) { append(a.size()); break; }
            std::vector<float> starts;
            for (const AlignedWord& w : a) starts.push_back(w.startTime);
            const int plateau = q3asr_trailing_plateau_start(starts.data(), (int)starts.size(), plateauTolerance, plateauMinWords);
            if (plateau == (int)a.size()) { append(a.size()); break; }
            if (plateau == 0) break;
            append((size_t)plateau);
            const float splitTime = a[(size_t)plateau - 1].endTime;
            const size_t splitSample = (size_t)(splitTime * (float)sampleRate);
            if (splitSample >= remAudio.size()) break;
            std::vector<float> next(remAudio.begin() + splitSample, remAudio.end());
            if ((float)next.size() / (float)sampleRate < minChunkSeconds) break;
            std::vector<std::string> wordsAll;  // the reference splits the text on the space character only (:161)
            for (size_t i = 0; i < remText.size();) {
                const size_t j = std::min(remText.find(' ', i), remText.size());
                if (j > i) wordsAll.push_back(remText.substr(i, j - i));
                i = j + 1;
            }
            if (plateau >= (int)wordsAll.size()) break;
            std::string nextText;
            for (size_t i = (size_t)plateau; i < wordsAll.size(); i++) nextText += (i > (size_t)plateau ? " " : "") + wordsAll[i];
            remAudio.swap(next);
            remText.swap(nextText);
            offset += splitTime;
        }
        return all;
    }
    q3asr_handle* handle() const { return h_; }

  private:
    Qwen3ForcedAligner(const char* preset, int device) {
        q3asr_config cfg;
        if (q3asr_config_preset(preset, &cfg) != Q3ASR_OK) throw AudioModelError(1, "modelLoadFailed: unknown aligner preset");
        timestampTokenId = cfg.tok_timestamp;
        int rc = q3asr_create(&cfg, device, &h_);
        if (rc != Q3ASR_OK) throw AudioModelError(rc, std::string("modelLoadFailed: ") + q3asr_last_error(nullptr));
    }
    q3asr_handle* h_ = nullptr;
    Tokenizer tok_;
};

inline std::vector<float> AudioFileLoader::resample(const Qwen3ASRModel& model, const std::vector<float>& samples, int from, int to) {
    if (from == to || samples.empty()) return samples;
    size_t n = q3asr_resample_len(samples.size(), from, to);
    std::vector<float> out(n);
    if (q3asr_resample(model.handle(), samples.data(), samples.size(), from, to, out.data(), out.size(), &n) != Q3ASR_OK) return samples;
    out.resize(n);
    return out;
}

}  // namespace qwen3asr
