// Qwen3ASRB200.swift — the Swift side of the drop-in boundary.  NOT compiled in this repository's CI
// (no Swift toolchain in the build image); it is the binding a maintainer of qwen3-asr-swift adds next
// to Sources/Qwen3ASR so that the batch-transcription hot path runs on libq3asr.so (B200, sm_100a).
//
// It keeps the reference's public surface for this path:
//   Qwen3ASRModel.fromPretrained(modelId:cacheDir:offlineMode:progressHandler:)   Qwen3ASR.swift:608-613
//   transcribe(audio:sampleRate:language:maxTokens:context:) -> String             Qwen3ASR.swift:131-137
//   transcribe(audio:sampleRate:options:) -> String                                Qwen3ASR.swift:107-111
//   SpeechRecognitionModel / ModelMemoryManageable conformances                    Qwen3ASR+Protocols.swift, +Memory.swift
//   WhisperFeatureExtractor.extractFeaturesRaw(_:) -> MelFeatures                  AudioPreprocessing.swift:347
// and adds the batched entry point the new scheduler enables (transcribeBatch).
// The tokenizer (Qwen3Tokenizer, AudioCommon/Tokenizer.swift) stays in Swift: the C ABI deals in token ids.
import AudioCommon
import CQ3ASR
import Foundation

public enum Q3ASRB200Error: Error, CustomStringConvertible {
    case library(code: Int32, message: String)
    public var description: String {
        switch self { case .library(let c, let m): return "q3asr error \(c): \(m)" }
    }
}

/// Same container as the reference's MelFeatures (AudioPreprocessing.swift:8-18).
public struct B200MelFeatures {
    public let data: [Float]      // row-major [melBins, timeFrames]
    public let melBins: Int
    public let timeFrames: Int
}

#if os(Linux)
/// On Linux (no MLX / Metal) the reference's type names resolve to the B200 implementation, so code written against
/// `Qwen3ASRModel` / `Qwen3ForcedAligner` (Qwen3ASR.swift:67, ForcedAligner.swift:226) builds and runs unchanged.
public typealias Qwen3ASRModel = Qwen3ASRB200Model
public typealias Qwen3ForcedAligner = Qwen3ForcedAlignerB200
#endif

public final class Qwen3ASRB200Model {
    private var handle: OpaquePointer?
    private let tokenizer: Qwen3Tokenizer?
    public let modelSize: ASRModelSize

    private init(handle: OpaquePointer?, tokenizer: Qwen3Tokenizer?, size: ASRModelSize) {
        self.handle = handle
        self.tokenizer = tokenizer
        self.modelSize = size
    }

    deinit { if let h = handle { q3asr_destroy(h) } }

    private static func check(_ rc: Int32, _ h: OpaquePointer?) throws {
        if rc != Q3ASR_OK {
            throw Q3ASRB200Error.library(code: rc, message: String(cString: q3asr_last_error(h)))
        }
    }

    /// Mirrors Qwen3ASRModel.fromPretrained: resolves / downloads the checkpoint directory with the
    /// reference's HuggingFaceDownloader, then hands the directory to the library (fp16/bf16/fp32 safetensors).
    /// Same parameter names, order and defaults as the reference (Qwen3ASR.swift:608-613); `device` is the one addition and comes
    /// last with a default, so every existing call site compiles unchanged.  The default model id is the reference's
    /// (an MLX 4-bit checkpoint: the loader dequantises it to bf16, csrc/safetensors.cu).
    public static func fromPretrained(
        modelId: String = "aufklarer/Qwen3-ASR-0.6B-MLX-4bit",
        cacheDir: URL? = nil,
        offlineMode: Bool = false,
        progressHandler: ((Double, String) -> Void)? = nil,
        device: Int32 = 0
    ) async throws -> Qwen3ASRB200Model {
        progressHandler?(0.0, "Downloading model...")
        let size = ASRModelSize.detect(from: modelId)
        let dir = try cacheDir ?? HuggingFaceDownloader.getCacheDirectory(for: modelId)
        try await HuggingFaceDownloader.downloadWeights(modelId: modelId, to: dir, offlineMode: offlineMode) { p in
            progressHandler?(p * 0.8, "Downloading weights...")
        }
        var cfg = q3asr_config()
        try check(q3asr_config_preset(size == .large ? "1.7B" : "0.6B", &cfg), nil)
        var h: OpaquePointer?
        try check(q3asr_create(&cfg, device, &h), nil)
        progressHandler?(0.85, "Loading weights onto the GPU...")
        do { try check(q3asr_load_safetensors(h, dir.path), h) } catch { q3asr_destroy(h); throw error }
        let tok = try? Qwen3Tokenizer(vocabURL: dir.appendingPathComponent("vocab.json"))
        progressHandler?(1.0, "Ready")
        return Qwen3ASRB200Model(handle: h, tokenizer: tok, size: size)
    }

    // MARK: stages (parity surface)

    public func extractFeaturesRaw(_ audio: [Float]) -> B200MelFeatures {
        let frames = Int(q3asr_mel_frames(audio.count))
        var out = [Float](repeating: 0, count: 128 * max(frames, 0))
        var got: Int32 = 0
        let rc = audio.withUnsafeBufferPointer { a in
            out.withUnsafeMutableBufferPointer { o in q3asr_mel(handle, a.baseAddress, audio.count, o.baseAddress, &got) }
        }
        precondition(rc == Q3ASR_OK, String(cString: q3asr_last_error(handle)))
        return B200MelFeatures(data: out, melBins: 128, timeFrames: Int(got))
    }

    // MARK: transcription

    private func promptIds(language: String?, context: String?) -> (ctx: [Int32], lang: [Int32]) {
        // Qwen3ASR.swift:203-206 (context in the system turn), :228-232 ("language <name>" before <asr_text>)
        let ctx = context.flatMap { c in tokenizer?.encode(c).map(Int32.init) } ?? []
        let lang = language.flatMap { l in tokenizer?.encode("language \(l)").map(Int32.init) } ?? []
        return (ctx, lang)
    }

    /// Batched greedy transcription: utterances are independent, the library batches them on the GPU.
    public func transcribeBatch(audio: [[Float]], language: String? = nil, maxTokens: Int = 448, context: String? = nil,
                                sampleRates: [Int]? = nil, options: Qwen3DecodingOptions? = nil) -> [String] {
        return run(audio: audio, language: language, maxTokens: maxTokens, context: context, sampleRates: sampleRates, options: options,
                   scored: false).map { $0.text }
    }

    /// transcribeBatch plus each utterance's confidence = exp(mean token log-probability, EOS included) — the value the reference's
    /// C bridge carries in sc_transcription_result_t.confidence (VoicePipeline.swift:374-411); 0 for an utterance without tokens.
    public func transcribeBatchWithConfidence(audio: [[Float]], language: String? = nil, maxTokens: Int = 448, context: String? = nil,
                                              sampleRates: [Int]? = nil, options: Qwen3DecodingOptions? = nil)
        -> [(text: String, confidence: Float)] {
        return run(audio: audio, language: language, maxTokens: maxTokens, context: context, sampleRates: sampleRates, options: options,
                   scored: true)
    }

    private func run(audio: [[Float]], language: String?, maxTokens: Int, context: String?, sampleRates: [Int]?,
                     options: Qwen3DecodingOptions?, scored: Bool) -> [(text: String, confidence: Float)] {
        guard q3asr_is_loaded(handle) != 0 else {
            return audio.map { _ in ("[Audio encoded] - Text decoder not loaded", 0) }   // Qwen3ASR.swift:116-119
        }
        let n = audio.count
        let (ctx, lang) = promptIds(language: language, context: context)
        var ids = [Int32](repeating: 0, count: n * maxTokens)
        var lens = [Int32](repeating: 0, count: n)
        var lp = [Float](repeating: 0, count: scored ? n * maxTokens : 0)
        var sizes = audio.map { $0.count }
        // borrow every clip's storage for the duration of the call
        var ptrs = [UnsafePointer<Float>?](repeating: nil, count: n)
        func withAll(_ i: Int, _ body: () -> Int32) -> Int32 {
            if i == n { return body() }
            return audio[i].withUnsafeBufferPointer { b in ptrs[i] = b.baseAddress; return withAll(i + 1, body) }
        }
        let rc: Int32 = ctx.withUnsafeBufferPointer { c in
            lang.withUnsafeBufferPointer { l in
                var prompts = [q3asr_prompt](repeating: q3asr_prompt(context_ids: c.baseAddress, n_context: Int32(c.count),
                                                                    language_ids: l.baseAddress, n_language: Int32(l.count),
                                                                    raw_suffix: 0), count: n)
                // clips at other sample rates are converted to 16 kHz on the device (AudioPreprocessing.swift:323-337); the decoder
                // knobs of Qwen3DecodingOptions run as a device kernel (pickNextToken, Qwen3ASR.swift:449-520)
                var rates = (sampleRates ?? [Int](repeating: 16000, count: n)).map(Int32.init)
                var samp = q3asr_sampling(repetition_penalty: options?.repetitionPenalty ?? 1.0,
                                          no_repeat_ngram_size: Int32(options?.noRepeatNgramSize ?? 0),
                                          temperature: options?.temperature ?? 0.0,
                                          seed: UInt64.random(in: 0 ... UInt64.max), force_device_sampler: 0)
                return lp.withUnsafeMutableBufferPointer { lpb in
                    withAll(0) {
                        q3asr_transcribe_ids_lp(handle, &ptrs, &sizes, &rates, Int32(n), &prompts, &samp, Int32(maxTokens), 1, &ids, &lens,
                                                scored ? lpb.baseAddress : nil)
                    }
                }
            }
        }
        if rc != Q3ASR_OK {
            let msg = String(cString: q3asr_last_error(handle))
            return audio.map { _ in ("[Qwen3-ASR B200 error: \(msg)]", 0) }             // cf. CoreMLASRModel.swift:299-305
        }
        return (0..<n).map { i in
            let len = Int(lens[i])
            let conf: Float = scored && len > 0 ? exp(lp[(i * maxTokens)..<(i * maxTokens + len)].reduce(0, +) / Float(len)) : 0
            var toks = Array(ids[(i * maxTokens)..<(i * maxTokens + len)]).map(Int.init)
            if toks.last == Int(Q3ASR_EOS_TOKEN) { toks.removeLast() }
            guard let tokenizer = tokenizer else { return (toks.map(String.init).joined(separator: " "), conf) } // id-string fallback, Qwen3ASR.swift:283-289
            let raw = tokenizer.decode(tokens: toks)
            if let r = raw.range(of: "<asr_text>") { return (String(raw[r.upperBound...]).trimmingCharacters(in: .whitespaces), conf) }
            return (raw.trimmingCharacters(in: .whitespaces), conf)
        }
    }

    public func transcribe(audio: [Float], sampleRate: Int = 16000, language: String? = nil, maxTokens: Int = 448,
                           context: String? = nil) -> String {
        return transcribeBatch(audio: [audio], language: language, maxTokens: maxTokens, context: context, sampleRates: [sampleRate])[0]
    }

    public func transcribe(audio: [Float], sampleRate: Int = 16000, options: Qwen3DecodingOptions) -> String {
        return transcribeBatch(audio: [audio], language: options.language, maxTokens: options.maxTokens, context: options.context,
                               sampleRates: [sampleRate], options: options)[0]
    }
}

extension Qwen3ASRB200Model: SpeechRecognitionModel {
    public var inputSampleRate: Int { 16000 }
    public func transcribe(audio: [Float], sampleRate: Int, language: String?) -> String {
        transcribe(audio: audio, sampleRate: sampleRate, language: language, maxTokens: 448)
    }
}

extension Qwen3ASRB200Model: ModelMemoryManageable {
    public var isLoaded: Bool { q3asr_is_loaded(handle) != 0 }
    public func unload() { _ = q3asr_unload(handle) }
    public var memoryFootprint: Int { Int(q3asr_memory_footprint(handle)) }
}

// Because Qwen3ASRB200Model is a SpeechRecognitionModel, the reference's own C bridge takes it unchanged: VoicePipeline's
// STTBridge(model:) -> makeSTTVtable (Sources/SpeechCore/VoicePipeline.swift:374-411) wraps any SpeechRecognitionModel into a
// sc_stt_vtable_t, and keeps the "pointers valid until the next transcribe call" ownership on the bridge object.

/// Qwen3ForcedAligner (Sources/Qwen3ASR/ForcedAligner.swift:50-331) over q3asr_align_indices.  The text side stays the reference's
/// own Swift: TextPreprocessor.prepareForAlignment (NLTokenizer for Japanese / Korean / Thai ..., TextPreprocessing.swift:48-160)
/// produces the slotted ids and the <timestamp> positions; the library runs mel -> encoder -> one prefill over the aligner template ->
/// classification head -> first-maximum class at those positions; TimestampCorrection finishes on the host (either the Swift
/// original or q3asr_enforce_monotonicity, which restates it line by line).
public final class Qwen3ForcedAlignerB200 {
    private var handle: OpaquePointer?
    private let tokenizer: Qwen3Tokenizer
    public static let timestampSegmentTime: Float = 0.08   // Configuration.swift:133

    private init(handle: OpaquePointer?, tokenizer: Qwen3Tokenizer) {
        self.handle = handle
        self.tokenizer = tokenizer
    }

    deinit { if let h = handle { q3asr_destroy(h) } }

    /// `dir`: the snapshot directory the reference's downloader filled (ForcedAligner.swift:394-452): *.safetensors with the
    /// thinker.* / lm_head.* keys (MLX 4-bit or bf16), vocab.json, merges.txt, tokenizer_config.json.
    public static func fromPretrained(directory dir: URL, device: Int32 = 0) throws -> Qwen3ForcedAlignerB200 {
        var cfg = q3asr_config()
        guard q3asr_config_preset("aligner", &cfg) == Q3ASR_OK else {
            throw Q3ASRB200Error.library(code: 1, message: "unknown preset")
        }
        var h: OpaquePointer?
        var rc = q3asr_create(&cfg, device, &h)
        guard rc == Q3ASR_OK else { throw Q3ASRB200Error.library(code: rc, message: String(cString: q3asr_last_error(nil))) }
        rc = q3asr_load_safetensors(h, dir.path)
        guard rc == Q3ASR_OK else {
            let msg = String(cString: q3asr_last_error(h))
            q3asr_destroy(h)
            throw Q3ASRB200Error.library(code: rc, message: msg)
        }
        let tok = Qwen3Tokenizer()
        try tok.load(from: dir.appendingPathComponent("vocab.json"))
        return Qwen3ForcedAlignerB200(handle: h, tokenizer: tok)
    }

    /// ForcedAligner.swift:226-331, same signature and the same empty result when the text has no words.
    public func align(audio: [Float], text: String, sampleRate: Int = 16000, language: String = "English") -> [AlignedWord] {
        let slotted = TextPreprocessor.prepareForAlignment(text: text, tokenizer: tokenizer, language: language)
        guard !slotted.words.isEmpty else { return [] }
        let ids = slotted.tokenIds.map { Int32($0) }
        let pos = slotted.timestampPositions.map { Int32($0) }
        var raw = [Int32](repeating: 0, count: pos.count)
        let rc: Int32 = audio.withUnsafeBufferPointer { a in
            ids.withUnsafeBufferPointer { i in
                pos.withUnsafeBufferPointer { p in
                    raw.withUnsafeMutableBufferPointer { r in
                        var pcm: UnsafePointer<Float>? = a.baseAddress
                        var n = audio.count
                        var rate = Int32(sampleRate)
                        var idp: UnsafePointer<Int32>? = i.baseAddress
                        var nid = Int32(ids.count)
                        var pp: UnsafePointer<Int32>? = p.baseAddress
                        var np = Int32(pos.count)
                        var out: UnsafeMutablePointer<Int32>? = r.baseAddress
                        return q3asr_align_indices(handle, &pcm, &n, &rate, 1, &idp, &nid, &pp, &np, &out)
                    }
                }
            }
        }
        guard rc == Q3ASR_OK else {
            print("Error: \(String(cString: q3asr_last_error(handle)))")   // the reference prints and returns [] (:232-235)
            return []
        }
        let corrected = TimestampCorrection.enforceMonotonicity(raw.map { Int($0) })
        var words: [AlignedWord] = []
        for (w, word) in slotted.words.enumerated() where 2 * w + 1 < corrected.count {
            let start = Float(corrected[2 * w]) * Self.timestampSegmentTime
            let end = Float(corrected[2 * w + 1]) * Self.timestampSegmentTime
            words.append(AlignedWord(text: word, startTime: start, endTime: max(end, start)))
        }
        return words
    }
    // alignLong (ForcedAligner.swift:100-181) is host logic over align(): the reference's body applies unchanged.
}

extension Qwen3ForcedAlignerB200: ForcedAlignmentModel {   // AudioCommon/Protocols.swift:170-173
    public func align(audio: [Float], text: String, sampleRate: Int, language: String?) -> [AlignedWord] {
        align(audio: audio, text: text, sampleRate: sampleRate, language: language ?? "English")
    }
}
