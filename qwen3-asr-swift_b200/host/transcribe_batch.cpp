// transcribe_batch.cpp — the `speech transcribe-batch` front door over the batched B200 path
// (/root/reference/Sources/AudioCLILib/TranscribeBatchCommand.swift:45-139, 217-243): walks a directory, loads every WAV
// (AudioFileLoader.loadWAV) and — unlike the reference's serial per-file loop (:82-125) — hands the files to the utterance-batching
// pool in groups: the utterances of a group share every kernel launch, the groups are dealt over the GPUs named by --devices, and
// while one group runs (q3asr_pool_submit) the next group's files are read and parsed.  Files at other sample rates are converted
// on the device; recordings longer than --window-seconds are cut into windows (each an independent utterance) and their texts
// joined.  Output lines follow the reference: JSONL {"file","text","time","rtf","duration"} or the bracketed progress lines, then the
// aggregate block.  A file's "time" is its share (by audio duration) of the group it ran in.
//
//   transcribe_batch <inputDir> [--output-dir D] [--model 0.6B|1.7B] [--model-dir DIR] [--language L] [--extensions wav]
//                    [--jsonl] [--batch N] [--max-tokens N] [--window-seconds S] [--devices 0,1,...] [--workers-per-gpu W] [--list]
//                    [--confidence] [--continuous]
// --confidence adds each file's average token log-probability (over all its windows, EOS included: include/q3asr.h) to its JSONL
// record ("avg_logprob") and progress line — the score a caller uses to flag hallucinated or low-quality output.
// --continuous runs each worker's share of a group as one continuous batch of at most --batch rows (<= 256): rows freed by EOS are
// refilled with the waiting utterances (q3asr_pool_set_continuous).  The output is the same as without it.
// Two pool workers per GPU by default: the decode steps of two batches in flight on one GPU interleave (each is a chain of
// latency-bound launches), which measured +24 % aggregate throughput over one batch at a time (tools/pool_concurrency.py).
// Without --model-dir the weights are random-init (this repo has no checkpoint offline); --list only prints the files.
#include <chrono>
#include <cstdio>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <set>

#include "qwen3_asr.hpp"

using namespace qwen3asr;
namespace fs = std::filesystem;

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static std::string json_escape(const std::string& s) {  // TranscribeBatchCommand.swift:101-103 (+ control characters)
    std::string o;
    for (unsigned char c : s) {
        if (c == '\\') o += "\\\\";
        else if (c == '"') o += "\\\"";
        else if (c == '\n') o += "\\n";
        else if (c == '\r') o += "\\r";
        else if (c == '\t') o += "\\t";
        else if (c < 0x20) { char b[8]; snprintf(b, sizeof b, "\\u%04x", c); o += b; }
        else o += (char)c;
    }
    return o;
}

static std::vector<std::string> split_commas(const std::string& s) {
    std::vector<std::string> out;
    size_t a = 0;
    while (a <= s.size()) {
        size_t b = s.find(',', a);
        if (b == std::string::npos) b = s.size();
        if (b > a) out.push_back(s.substr(a, b - a));
        a = b + 1;
    }
    return out;
}

// TranscribeBatchCommand.swift:217-234: regular files with a listed extension, hidden entries skipped, sorted by file name
static std::vector<fs::path> find_audio_files(const std::string& dir, const std::string& extensions) {
    std::set<std::string> exts;
    for (std::string e : split_commas(extensions)) {
        std::transform(e.begin(), e.end(), e.begin(), [](unsigned char c) { return (char)std::tolower(c); });
        exts.insert(e);
    }
    std::vector<fs::path> files;
    std::error_code ec;
    for (fs::recursive_directory_iterator it(dir, fs::directory_options::skip_permission_denied, ec), end; !ec && it != end; it.increment(ec)) {
        const std::string name = it->path().filename().string();
        if (!name.empty() && name[0] == '.') {
            if (it->is_directory(ec)) it.disable_recursion_pending();
            continue;
        }
        if (!it->is_regular_file(ec)) continue;
        std::string e = it->path().extension().string();
        if (!e.empty()) e = e.substr(1);
        std::transform(e.begin(), e.end(), e.begin(), [](unsigned char c) { return (char)std::tolower(c); });
        if (exts.count(e)) files.push_back(it->path());
    }
    std::sort(files.begin(), files.end(), [](const fs::path& x, const fs::path& y) { return x.filename().string() < y.filename().string(); });
    return files;
}

struct Item {
    std::string name, error, text;
    double duration = 0, time = 0;
    double lp_sum = 0;  // --confidence: sum and count of the token log-probabilities of the file's windows
    long lp_n = 0;
};
struct Unit { size_t item; std::vector<float> samples; int rate; };

// one group of utterances in flight on the pool
struct Group {
    std::vector<Unit> units;
    std::vector<const float*> pcm;
    std::vector<size_t> n;
    std::vector<int> rates;
    std::vector<q3asr_prompt> prompts;
    q3asr_job* job = nullptr;
    double t0 = 0;
};

int main(int argc, char** argv) {
    std::string inputDir, outputDir, model = "0.6B", modelDir, extensions = "wav,flac,mp3", devicesArg = "0";
    std::optional<std::string> language;
    bool jsonl = false, listOnly = false, confidence = false, continuous = false;
    int batch = 256, maxTokens = 448, workersPerGpu = 2;
    float windowSeconds = 30.f;
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto val = [&]() -> std::string { return i + 1 < argc ? argv[++i] : ""; };
        if (a == "--output-dir") outputDir = val();
        else if (a == "--model" || a == "-m") model = val();
        else if (a == "--model-dir") modelDir = val();
        else if (a == "--language") language = val();
        else if (a == "--extensions") extensions = val();
        else if (a == "--jsonl") jsonl = true;
        else if (a == "--list") listOnly = true;
        else if (a == "--confidence") confidence = true;
        else if (a == "--continuous") continuous = true;
        else if (a == "--batch") batch = std::max(1, atoi(val().c_str()));
        else if (a == "--max-tokens") maxTokens = std::max(1, atoi(val().c_str()));
        else if (a == "--window-seconds") windowSeconds = (float)atof(val().c_str());
        else if (a == "--devices" || a == "--device") devicesArg = val();
        else if (a == "--workers-per-gpu") workersPerGpu = std::max(1, atoi(val().c_str()));
        else if (!a.empty() && a[0] != '-' && inputDir.empty()) inputDir = a;
        else { fprintf(stderr, "unknown argument %s\n", a.c_str()); return 2; }
    }
    if (inputDir.empty()) { fprintf(stderr, "usage: transcribe_batch <inputDir> [options]\n"); return 2; }
    const auto files = find_audio_files(inputDir, extensions);
    if (files.empty()) { printf("No audio files found in %s\n", inputDir.c_str()); return 0; }
    printf("Found %zu audio files\n", files.size());
    if (listOnly) {
        for (const auto& f : files) printf("%s\n", f.filename().string().c_str());
        return 0;
    }
    std::vector<int> devices;
    for (const std::string& d : split_commas(devicesArg))
        for (int w = 0; w < workersPerGpu; w++) devices.push_back(atoi(d.c_str()));
    if (devices.empty()) devices.push_back(0);
    const ASRModelSize size = detectModelSize(model);
    printf("Loading model (%s): %s, %zu pool worker(s)\n", size == ASRModelSize::large ? "1.7B" : "0.6B",
           modelDir.empty() ? "random-init weights" : modelDir.c_str(), devices.size());
    const double loadStart = now_s();
    q3asr_config cfg;
    q3asr_config_preset(size == ASRModelSize::large ? "1.7B" : "0.6B", &cfg);
    q3asr_pool* pool = nullptr;
    if (q3asr_pool_create(&cfg, devices.data(), (int)devices.size(), 20260418, modelDir.empty() ? nullptr : modelDir.c_str(), &pool) != Q3ASR_OK) {
        fprintf(stderr, "Error: modelLoadFailed: %s\n", q3asr_last_error(nullptr));
        return 1;
    }
    if (continuous) {
        batch = std::min(batch, 256);  // the resident rows of a continuous batch
        q3asr_pool_set_continuous(pool, 1);
    }
    Tokenizer tok;
    if (!modelDir.empty()) {
        try { tok = Tokenizer::fromDirectory(modelDir); } catch (const AudioModelError&) {}  // optional, Qwen3ASR.swift:643-649
    }
    std::vector<int32_t> langIds;
    if (language && tok.encode) langIds = tok.encode("language " + *language);  // Qwen3ASR.swift:228-232
    const double loadTime = now_s() - loadStart;
    printf("  Model loaded in %.2fs\n", loadTime);
    if (!outputDir.empty()) fs::create_directories(outputDir);

    std::vector<Item> items(files.size());
    const size_t group_units = (size_t)batch * devices.size();
    size_t next_file = 0;
    // reads files until a group is full (a file's windows stay together); a file that fails is reported in its place and skipped
    // (TranscribeBatchCommand.swift:118-124)
    auto load_group = [&]() {
        Group* g = new Group();
        while (next_file < files.size() && g->units.size() < group_units) {
            const size_t i = next_file++;
            items[i].name = files[i].stem().string();
            try {
                AudioFileLoader::Wav w = AudioFileLoader::loadWAV(files[i].string());
                if (w.sampleRate <= 0 || q3asr_resample_len(w.samples.size(), w.sampleRate, 16000) < 160)
                    throw AudioLoadError(1, "audio shorter than one mel frame");
                items[i].duration = (double)w.samples.size() / w.sampleRate;
                const size_t window = std::max<size_t>((size_t)((double)windowSeconds * w.sampleRate + 0.5), 1);
                const size_t minTail = std::max<size_t>(160, ((size_t)160 * w.sampleRate + 15999) / 16000);
                int count = 0;
                q3asr_longform_plan(w.samples.size(), window, minTail, nullptr, nullptr, 0, &count);
                std::vector<size_t> st((size_t)count), ln((size_t)count);
                q3asr_longform_plan(w.samples.size(), window, minTail, st.data(), ln.data(), count, &count);
                for (int k = 0; k < count; k++)
                    g->units.push_back(Unit{i, std::vector<float>(w.samples.begin() + st[k], w.samples.begin() + st[k] + ln[k]), w.sampleRate});
            } catch (const std::exception& e) {
                items[i].error = e.what();
            }
        }
        for (const Unit& u : g->units) {
            g->pcm.push_back(u.samples.data());
            g->n.push_back(u.samples.size());
            g->rates.push_back(u.rate);
            g->prompts.push_back(q3asr_prompt{nullptr, 0, langIds.empty() ? nullptr : langIds.data(), (int)langIds.size(), 0});
        }
        return g;
    };
    auto submit = [&](Group* g, int tokens) {
        g->t0 = now_s();
        if (g->units.empty()) return true;
        return (confidence ? q3asr_pool_submit_lp : q3asr_pool_submit)(pool, g->pcm.data(), g->n.data(), g->rates.data(), (int)g->units.size(),
                                                                      g->prompts.data(), nullptr, tokens, 1, batch, &g->job) == Q3ASR_OK;
    };
    double totalInference = 0;
    std::vector<int32_t> ids;
    std::vector<int> lens;
    std::vector<float> lps;
    auto finish = [&](Group* g, int tokens, bool record) {
        if (g->job != nullptr) {
            ids.assign(g->units.size() * (size_t)tokens, 0);
            lens.assign(g->units.size(), 0);
            int rc = q3asr_job_wait(g->job, ids.data(), lens.data());
            if (rc == Q3ASR_OK && confidence) {
                lps.assign(g->units.size() * (size_t)tokens, 0.f);
                rc = q3asr_job_logprobs(g->job, lps.data());
            }
            const double elapsed = now_s() - g->t0;
            if (record) {
                totalInference += elapsed;
                double audio = 0;
                for (const Unit& u : g->units) audio += (double)u.samples.size() / u.rate;
                for (size_t k = 0; k < g->units.size(); k++) {
                    Item& it = items[g->units[k].item];
                    if (rc != Q3ASR_OK) {
                        it.error = std::string("[Qwen3-ASR B200 error: ") + q3asr_job_last_error(g->job) + "]";
                        continue;
                    }
                    std::vector<int32_t> t(ids.begin() + k * (size_t)tokens, ids.begin() + k * (size_t)tokens + lens[k]);
                    if (confidence)
                        for (int s = 0; s < lens[k]; s++) { it.lp_sum += lps[k * (size_t)tokens + s]; it.lp_n++; }
                    if (!t.empty() && t.back() == Q3ASR_EOS_TOKEN) t.pop_back();
                    if (!it.text.empty()) it.text += " ";
                    it.text += Qwen3ASRModel::textFromIds(tok, t);
                    it.time += elapsed * ((double)g->units[k].samples.size() / g->units[k].rate) / std::max(audio, 1e-9);
                }
            }
            q3asr_job_free(g->job);
        }
        delete g;
    };

    // warm-up (TranscribeBatchCommand.swift:68-75): the first group once with a short decode, results discarded
    const double warmStart = now_s();
    Group* cur = load_group();
    {
        Group* warm = new Group();
        if (!cur->units.empty()) {
            warm->units.push_back(Unit{cur->units[0].item, cur->units[0].samples, cur->units[0].rate});
            warm->pcm.push_back(warm->units[0].samples.data());
            warm->n.push_back(warm->units[0].samples.size());
            warm->rates.push_back(warm->units[0].rate);
            warm->prompts.push_back(q3asr_prompt{nullptr, 0, nullptr, 0, 0});
        }
        submit(warm, std::min(maxTokens, 4));
        finish(warm, std::min(maxTokens, 4), false);
    }
    const double warmupTime = now_s() - warmStart;
    printf("  Warmup: %.2fs\n", warmupTime);

    const double batchStart = now_s();
    while (cur != nullptr) {
        submit(cur, maxTokens);
        Group* nxt = next_file < files.size() ? load_group() : nullptr;  // file I/O and parsing overlap the GPU work
        finish(cur, maxTokens, true);
        cur = nxt;
    }
    const double batchTime = now_s() - batchStart;
    double totalAudio = 0;
    for (size_t i = 0; i < items.size(); i++) {
        const Item& it = items[i];
        if (!it.error.empty()) {
            if (jsonl) printf("{\"file\":\"%s\",\"error\":\"%s\"}\n", json_escape(it.name).c_str(), json_escape(it.error).c_str());
            else printf("  [%zu/%zu] %s: ERROR - %s\n", i + 1, items.size(), it.name.c_str(), it.error.c_str());
            continue;
        }
        totalAudio += it.duration;
        const double rtf = it.time / std::max(it.duration, 0.001);
        const double avg_lp = it.lp_n ? it.lp_sum / it.lp_n : 0.0;
        if (jsonl && confidence)
            printf("{\"file\":\"%s\",\"text\":\"%s\",\"time\":%.3f,\"rtf\":%.4f,\"duration\":%.2f,\"avg_logprob\":%.6f}\n",
                   json_escape(it.name).c_str(), json_escape(it.text).c_str(), it.time, rtf, it.duration, avg_lp);
        else if (jsonl)
            printf("{\"file\":\"%s\",\"text\":\"%s\",\"time\":%.3f,\"rtf\":%.4f,\"duration\":%.2f}\n", json_escape(it.name).c_str(),
                   json_escape(it.text).c_str(), it.time, rtf, it.duration);
        else if (confidence)
            printf("  [%zu/%zu] (%.0f%%) %s: %s  (%.2fs, RTF=%.3f, avg_logprob=%.3f)\n", i + 1, items.size(), 100.0 * (i + 1) / items.size(),
                   it.name.c_str(), it.text.c_str(), it.time, rtf, avg_lp);
        else
            printf("  [%zu/%zu] (%.0f%%) %s: %s  (%.2fs, RTF=%.3f)\n", i + 1, items.size(), 100.0 * (i + 1) / items.size(), it.name.c_str(),
                   it.text.c_str(), it.time, rtf);
        if (!outputDir.empty()) {
            std::ofstream f(fs::path(outputDir) / (it.name + ".txt"));
            f << it.text;
        }
    }
    printf("\nBatch complete: %zu files, %.1fs audio\n", files.size(), totalAudio);
    printf("  Total inference: %.2fs, Aggregate RTF: %.4f\n", totalInference, totalInference / std::max(totalAudio, 0.001));
    printf("  Wall time: %.2fs (includes I/O)\n", batchTime);
    printf("  Model load: %.2fs, Warmup: %.2fs\n", loadTime, warmupTime);
    q3asr_pool_destroy(pool);
    return 0;
}
