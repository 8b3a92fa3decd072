/*
 * q3asr.h — C ABI of libq3asr.so, the B200-native (sm_100a) implementation of the Qwen3-ASR batch
 * transcription hot path: log-mel -> audio encoder -> Qwen3 decoder prefill -> greedy decode.
 *
 * This is the drop-in boundary for the reference's Swift API (paths relative to /root/reference):
 *   Qwen3ASRModel.fromPretrained            Sources/Qwen3ASR/Qwen3ASR.swift:608-668   -> q3asr_create + q3asr_load_safetensors
 *   Qwen3ASRModel.transcribe(audio:...)     Sources/Qwen3ASR/Qwen3ASR.swift:107-164   -> q3asr_transcribe_ids (ids; the tokenizer stays in Swift)
 *   WhisperFeatureExtractor.extractFeaturesRaw  Sources/Qwen3ASR/AudioPreprocessing.swift:347-470 -> q3asr_mel / q3asr_mel_batch
 *   Qwen3AudioEncoder.callAsFunction        Sources/Qwen3ASR/AudioEncoder.swift:362-511 -> q3asr_encode
 *   ModelMemoryManageable                   Sources/Qwen3ASR/Qwen3ASR+Memory.swift:3-17 -> q3asr_is_loaded / q3asr_unload / q3asr_memory_footprint
 *   sc_stt_vtable_t (the reference's own C bridge)  Sources/SpeechCore/VoicePipeline.swift:374-411 -> q3asr_transcribe_ids has the same shape
 *
 * Conventions: every function returns 0 (Q3ASR_OK) or a positive error code; q3asr_last_error() gives
 * the message.  Nothing aborts.  Input pointers are borrowed for the duration of the call; outputs are
 * written into caller-provided buffers.  A handle is single-caller (the reference's model classes are
 * documented as not thread-safe, Qwen3ASR.swift:67); use one handle per GPU, or a q3asr_pool.
 * There is no CPU fallback: without a Blackwell GPU q3asr_create fails.
 */
#ifndef Q3ASR_H
#define Q3ASR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define Q3ASR_OK 0
#define Q3ASR_ERR_INVALID 1 /* bad argument */
#define Q3ASR_ERR_STATE 2   /* e.g. weights not loaded (the reference returns a placeholder string, Qwen3ASR.swift:116-119) */
#define Q3ASR_ERR_CUDA 3
#define Q3ASR_ERR_NOMEM 4
#define Q3ASR_ERR_IO 5

#define Q3ASR_EOS_TOKEN 151645 /* <|im_end|>, Qwen3ASR.swift:59 */

typedef struct q3asr_handle q3asr_handle;
typedef struct q3asr_pool q3asr_pool;

/* Model dimensions.  Presets mirror Qwen3AudioEncoderConfig (AudioEncoder.swift:28-68) and
 * TextDecoderConfig (Configuration.swift:47-100). */
typedef struct q3asr_config {
    /* audio encoder */
    int enc_d_model;     /* 896 / 1024 */
    int enc_heads;       /* 14 / 16 (head dim must be 64) */
    int enc_ffn;         /* 3584 / 4096 */
    int enc_layers;      /* 18 / 24 */
    int enc_out_dim;     /* 1024 / 2048 */
    int enc_conv_ch;     /* 480 (downsampleHiddenSize) */
    int enc_n_window;    /* 50  -> conv chunks of 100 frames */
    int enc_n_window_infer; /* 800 -> attention windows of 13*8 tokens */
    float enc_ln_eps;    /* 1e-5 */
    /* text decoder */
    int dec_vocab;       /* 151936 */
    int dec_hidden;      /* 1024 / 2048 */
    int dec_layers;      /* 28 */
    int dec_heads;       /* 16 */
    int dec_kv_heads;    /* 8 */
    int dec_head_dim;    /* 128 */
    int dec_inter;       /* 3072 / 6144 */
    float dec_rope_theta; /* 1e6 */
    float dec_rms_eps;   /* 1e-6 */
    /* prompt token ids (Qwen3ASR.swift:181-195); only the tests' tiny vocabulary changes them */
    int32_t tok_im_start, tok_im_end, tok_audio_start, tok_audio_end, tok_audio_pad, tok_asr_text, tok_newline, tok_system,
        tok_user, tok_assistant, tok_eos;
    /* forced aligner (ForcedAligner.swift:57-85, Configuration.swift:132-133): > 0 adds the timestamp classification head
     * lm_head.{weight,bias} [classify_num, dec_hidden]; 0 for the ASR models */
    int classify_num;     /* 5000 */
    int32_t tok_timestamp; /* <|timestamp|> 151705, Qwen3ASR.swift:62 */
} q3asr_config;

/* name: "0.6B", "1.7B", "aligner" (Qwen3-ForcedAligner-0.6B: the large encoder projecting to the 1024-wide decoder, 5000 classes),
 * or "tiny" / "tiny-aligner" (small configurations used by the parity tests) */
int q3asr_config_preset(const char* name, q3asr_config* cfg);

/* library identification (no reference equivalent; the Swift shim logs it next to the model id) */
const char* q3asr_version(void);
/* message of the last failed call on this handle (handle may be NULL: the calling thread's last failed q3asr_create) — the text the
 * Swift shim puts into AudioModelError.modelLoadFailed / weightLoadingFailed (Sources/AudioCommon/AudioModelError.swift:4-34) */
const char* q3asr_last_error(const q3asr_handle* h);

/* Qwen3ASRModel.init(audioConfig:textConfig:) (Qwen3ASR.swift:82-91): an empty model of the given dimensions on one GPU, weights to
 * follow; q3asr_destroy is its deinit.  Fails with Q3ASR_ERR_CUDA when there is no sm_100 device (no CPU fallback). */
int q3asr_create(const q3asr_config* cfg, int device, q3asr_handle** out);
void q3asr_destroy(q3asr_handle* h);

/* ---- weights (names are the reference's safetensors keys, WeightLoading.swift:17-126, 235-323) ---- */
/* deterministic random initialisation: bf16(0.02 * approx-normal) keyed by (seed, tensor name); norm weights 1.  No reference
 * equivalent: it stands in for the checkpoints (no network here), SURVEY.md 8d; oracle/weights.py generates the same values. */
int q3asr_init_random(q3asr_handle* h, uint64_t seed);
/* the tensors of the model by the reference's key names — what Qwen3ASRWeightLoader.loadWeights walks (WeightLoading.swift:17-126):
 * enumerate, set one by one (any of the dtypes MLX.loadArrays yields), read back, then commit */
int q3asr_tensor_count(const q3asr_handle* h);
int q3asr_tensor_info(const q3asr_handle* h, int index, char* name, int name_cap, int64_t* shape4, int* ndim);
/* dtype: 0 = fp32, 1 = bf16, 2 = fp16; converted to bf16 on upload */
int q3asr_set_tensor(q3asr_handle* h, const char* name, const void* data, int dtype, const int64_t* shape, int ndim);
int q3asr_get_tensor(const q3asr_handle* h, const char* name, float* out, size_t out_elems);
/* builds the fused / permuted device layouts from the named tensors; required after q3asr_set_tensor */
int q3asr_commit_weights(q3asr_handle* h);
/* Qwen3ASRWeightLoader.loadWeights / CommonWeightLoader.loadAllSafetensors (WeightLoading.swift:17-126, MLXCommon/WeightLoading.swift:
 * 9-11, 48-95): reads every *.safetensors in dir (audio_tower.* and model.* keys, the aligner's thinker.* / lm_head.*; fp32/fp16/bf16
 * and MLX U32-packed 4-/8-bit tensors, dequantised; conv weights in MLX [O,kH,kW,I] or PyTorch [O,I,kH,kW] layout) and commits */
int q3asr_load_safetensors(q3asr_handle* h, const char* dir);
/* Host-only (no GPU): the tensors q3asr_load_safetensors would see in dir after validating every header against its file —
 * one line per tensor, "name\tdtype\tshape\tbytes\n" (shape as 1024x128; U32 = MLX-packed, WeightLoading.swift:17-126).  buf == NULL
 * sizes the buffer through *needed.  On Q3ASR_ERR_IO the buffer holds the reason instead (malformed header, offsets outside the
 * file, oversized dimensions, unreadable directory). */
int q3asr_checkpoint_list(const char* dir, char* buf, size_t cap, size_t* needed);
int q3asr_is_loaded(const q3asr_handle* h);
int q3asr_unload(q3asr_handle* h);
size_t q3asr_memory_footprint(const q3asr_handle* h);

/* ---- stages (parity surface) ---- */
/* frames kept for n samples at 16 kHz: min(n / 160, 120000) (AudioPreprocessing.swift:195, 296, 304) */
int q3asr_mel_frames(size_t n_samples);
/* out: [128, frames] fp32 row-major (mel-major), the layout of MelFeatures.data */
int q3asr_mel(q3asr_handle* h, const float* pcm, size_t n_samples, float* out, int* frames);
int q3asr_mel_batch(q3asr_handle* h, const float* const* pcm, const size_t* n_samples, int batch, float* const* out,
                    int* frames);
/* audio tokens produced for `frames` mel frames (AudioEncoder.swift:287-303) */
int q3asr_encoder_tokens(int frames);
/* mel: [128, frames] fp32 (host).  out: [tokens, enc_out_dim] fp32 (converted from the bf16 result) */
int q3asr_encode(q3asr_handle* h, const float* mel, int frames, float* out, int* tokens);

/* per-utterance prompt extras (token ids from the Swift tokenizer; either may be NULL/0):
 * context goes into the system turn, language ("language xx") before <asr_text>  (Qwen3ASR.swift:203-232) */
typedef struct q3asr_prompt {
    const int32_t* context_ids;
    int n_context;
    const int32_t* language_ids;
    int n_language;
    /* != 0: language_ids are appended verbatim after "<|im_start|>assistant\n" and the <asr_text> token is NOT added — the forced
     * aligner's template (ForcedAligner.swift:338-378), whose suffix is the timestamp-slotted text */
    int raw_suffix;
} q3asr_prompt;

/* Host-only: TextPreprocessor.splitIntoWordPairs, default path (TextPreprocessing.swift:97-115, 163-243, 262-306) — split UTF-8 text on
 * Unicode white space, one word per Han ideograph, punctuation kept on the surface form only.  buf receives n_pairs records
 * "surface\0cleaned\0"; *needed = bytes required (call with buf == NULL to size).  language NULL = "English".  Japanese, Korean, Thai,
 * Lao, Khmer, Burmese and Tibetan return Q3ASR_ERR_INVALID: the reference segments them with Apple's NLTokenizer (:101-160), which
 * stays on the Swift side.  Errors: q3asr_text_last_error(). */
int q3asr_text_word_pairs(const char* text, const char* language, char* buf, size_t cap, size_t* needed, int* n_pairs);
const char* q3asr_text_last_error(void);

/* Host-only (no GPU work): the chat-template ids the prefill runs on for an utterance with n_audio_tokens audio tokens —
 * <|im_start|>system\n[context]<|im_end|>\n<|im_start|>user\n<|audio_start|><|audio_pad|>*n<|audio_end|><|im_end|>\n
 * <|im_start|>assistant\n[language]<asr_text>  (Qwen3ASR.swift:196-233; raw_suffix: ForcedAligner.swift:338-378).
 * *n_ids = ids needed, *audio_at = index of the first <|audio_pad|> (may be NULL).  Q3ASR_ERR_INVALID with *n_ids set when
 * cap is too small (call with cap 0 to size the buffer). */
int q3asr_prompt_ids(const q3asr_config* cfg, int n_audio_tokens, const q3asr_prompt* prompt, int32_t* ids_out, int cap, int* n_ids,
                     int* audio_at);

/* Batched greedy transcription.  ids_out: [batch, max_tokens] int32; lens_out: [batch].
 * stop_on_eos != 0 reproduces the reference loop (EOS appended, then stop, Qwen3ASR.swift:378-379);
 * stop_on_eos == 0 decodes exactly max_tokens ids (fixed-length parity runs).  prompts may be NULL.
 * Any batch size: more than 256 utterances are served as equal sub-batches of at most 256 one after the other (the decode
 * step's row capacity), so an utterance's ids do not depend on the size of the request; q3asr_stage_ms sums over them. */
int q3asr_transcribe_ids(q3asr_handle* h, const float* const* pcm, const size_t* n_samples, int batch,
                         const q3asr_prompt* prompts, int max_tokens, int stop_on_eos, int32_t* ids_out, int* lens_out);

/* Decoder knobs of Qwen3DecodingOptions (Qwen3ASR.swift:13-51).  The default values are the greedy fast path
 * (isGreedyFastPath, Qwen3ASR.swift:300-304: the fused argmax epilogue); anything else runs pickNextToken
 * (Qwen3ASR.swift:449-520) as a device kernel over the full logits: sign-aware repetition penalty on the tokens generated so far,
 * no-repeat-n-gram mask, logits / temperature + Gumbel(0,1) noise, first maximum.  The reference draws its noise from the system
 * RNG; here it is a counter-based stream keyed by (seed, sequence, step, vocabulary index), so runs are reproducible. */
typedef struct q3asr_sampling {
    float repetition_penalty;  /* 1.0 = off */
    int no_repeat_ngram_size;  /* 0 = off */
    float temperature;         /* 0 = argmax */
    uint64_t seed;
    int force_device_sampler;  /* != 0: run the sampling kernel even for the greedy configuration (parity tests) */
} q3asr_sampling;
/* q3asr_transcribe_ids_sr with decoder knobs (one setting for the whole batch; sampling == NULL is greedy) */
int q3asr_transcribe_ids_opts(q3asr_handle* h, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                              const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos,
                              int32_t* ids_out, int* lens_out);
/* resident-batch form: call between q3asr_batch_upload and the prefill stage */
int q3asr_batch_set_sampling(q3asr_handle* h, const q3asr_sampling* sampling);

/* Per-token log-probabilities (the score behind sc_transcription_result_t.confidence, VoicePipeline.swift:374-411).  For the token t
 * emitted at step s of utterance i:
 *     logprob[i][s] = z[t] - logsumexp(z)
 * z = the model's bf16-rounded logits over the whole vocabulary (the values the argmax ranks), the sum evaluated in fp32 with max
 * subtraction on the device, in the LM head's epilogue.  Step 0 is the token chosen at the prefill position (like top_out of
 * q3asr_decode_forced).  With decoder knobs z is the UNMODIFIED model logits — before repetition penalty, n-gram mask, temperature
 * and noise (Whisper's convention), so the number means the same on both paths.  Entries at and beyond lens_out[i] are 0.
 * An utterance's log-probabilities do not depend on the size of the request or the sub-batch it lands in.
 * Utterance score (host side): avg_logprob = mean(logprob[i][0 .. lens_out[i])) (an emitted EOS counts, as in Whisper),
 * confidence = exp(avg_logprob).
 * q3asr_transcribe_ids_lp: q3asr_transcribe_ids_opts plus logprobs_out [batch, max_tokens] (may be NULL: no extra work). */
int q3asr_transcribe_ids_lp(q3asr_handle* h, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                            const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos,
                            int32_t* ids_out, int* lens_out, float* logprobs_out);
/* Continuous batching: the whole request runs as ONE resident decode batch of at most max_rows rows (max_rows <= 0: 256).  The
 * first max_rows utterances are prefilled together; whenever a poll of the decode loop (every 16 steps) finds at least
 * max(4, max_rows / 4) rows finished (or none active), the finished rows leave the batch and the next waiting utterances, in request
 * order, go through mel -> encoder -> prefill as a group whose KV cache is written into the freed page blocks; they join the
 * decode rows at once.  The call returns when no utterance waits and no row is active.  Greedy only (there is no sampling
 * argument).  ids_out [batch, max_tokens], lens_out [batch] and logprobs_out [batch, max_tokens] (may be NULL) are in request order
 * and equal, bit for bit, what q3asr_transcribe_ids_lp returns for the same utterances: only the schedule changes.  The next
 * group's samples are staged on the copy stream while the decode runs.  q3asr_stage_ms: mel / encoder / prefill summed over the
 * first group and every admission, decode = the rest; q3asr_decode_stats covers the whole call (a partition of the decode rows
 * counts as a compaction).  Q3ASR_ERR_INVALID: max_rows > 256, batch <= 0 or > 65536. */
int q3asr_transcribe_ids_continuous(q3asr_handle* h, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                                    const q3asr_prompt* prompts, int max_tokens, int stop_on_eos, int max_rows, int32_t* ids_out,
                                    int* lens_out, float* logprobs_out);
/* resident-batch form: enable != 0 between q3asr_batch_upload and the prefill stage (every upload starts with them off), then
 * q3asr_batch_download_logprobs after the run: out [batch, max_tokens], the layout of q3asr_batch_download's ids.
 * Q3ASR_ERR_STATE when they were not enabled for the batch. */
int q3asr_batch_set_logprobs(q3asr_handle* h, int enable);
int q3asr_batch_download_logprobs(q3asr_handle* h, float* out, int max_tokens);
/* pickNextToken on caller-provided logits ([vocab] fp32; the reference's own unit tests drive it this way,
 * Tests/Qwen3ASRTests/Qwen3DecodingOptionsTests.swift:47-235).  draw selects the noise draw (the decode step). */
int q3asr_pick_next_token(q3asr_handle* h, const float* logits, int vocab, const int32_t* generated, int n_generated,
                          const q3asr_sampling* sampling, int draw, int32_t* token);

/* ---- forced aligner (SURVEY.md 8f rank 4; Qwen3ForcedAligner.align, ForcedAligner.swift:226-331) ---- */
/* One prefill pass per utterance over "<system><user><audio><assistant>" + slotted text, no decode loop: the classification head
 * (bf16 logits = h W^T + b over classify_num classes) is applied at the given positions of the slotted text (indices into
 * slotted_ids, normally the <|timestamp|> slots) and the argmax class (lowest index on ties) is written to
 * raw_indices_out[i][0..n_positions[i]).  Needs a configuration with classify_num > 0.  Time = index * 0.08 s after
 * q3asr_enforce_monotonicity. */
int q3asr_align_indices(q3asr_handle* h, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                        const int32_t* const* slotted_ids, const int* n_slotted, const int* const* positions, const int* n_positions,
                        int32_t* const* raw_indices_out);
/* TimestampCorrection (Sources/Qwen3ASR/TimestampCorrection.swift:15-145), host only: LIS anchors, nearest-neighbour / linear
 * fill of the other positions, final non-decreasing pass.  Pinned by the reference's ForcedAlignerTests.swift:213-259. */
int q3asr_enforce_monotonicity(const int* raw, int n, int* corrected);
int q3asr_lis_positions(const int* values, int n, int* positions, int* count);
/* Qwen3ForcedAligner.findTrailingPlateauStart (ForcedAligner.swift:191-216): first word of the trailing run of >= min_size words
 * whose start times differ by < tolerance, or n when there is none */
int q3asr_trailing_plateau_start(const float* start_times, int n, float tolerance, int min_size);

/* Teacher-forced scoring (parity on a prescribed token stream): the decoder consumes forced[0..n) as its
 * own outputs; argmax_out[i] / top_out[i] are the argmax id and its bf16 logit at step i (i = 0 is the
 * prefill position), n_forced + 1 entries. */
int q3asr_decode_forced(q3asr_handle* h, const float* pcm, size_t n_samples, const q3asr_prompt* prompt,
                        const int32_t* forced, int n_forced, int32_t* argmax_out, float* top_out);
/* The same with the audio encoder's output replaced by audio_embeds [n_audio_tokens, enc_out_dim] fp32 (rounded to bf16, like the
 * splice of Qwen3ASR.swift:236-244 casts them): isolates the decoder in parity tests — both sides of a comparison then start
 * from identical audio embeddings instead of two encoder outputs that differ by bf16 rounding noise.  n_audio_tokens must equal
 * q3asr_encoder_tokens of the clip's frame count. */
int q3asr_decode_forced_embeds(q3asr_handle* h, const float* pcm, size_t n_samples, const q3asr_prompt* prompt,
                               const float* audio_embeds, int n_audio_tokens, const int32_t* forced, int n_forced,
                               int32_t* argmax_out, float* top_out);
/* full logits of the prefill's last position, [vocab] fp32 (debug / parity) */
int q3asr_prefill_logits(q3asr_handle* h, const float* pcm, size_t n_samples, const q3asr_prompt* prompt, float* logits);

/* ---- resident-batch interface (what q3asr_transcribe_ids is made of; lets a caller time the stages
 * with inputs already in HBM).  upload = the audio hand-over of transcribe (Qwen3ASR.swift:131-141), run = featureExtractor.process ->
 * audioEncoder -> generateText (:141-164, 181-390) by stage, download = the generated ids (:283-293).  The timing / profiling / L2
 * helpers below have no reference equivalent: they exist for bench.py (SURVEY.md 8d). ---- */
int q3asr_batch_upload(q3asr_handle* h, const float* const* pcm, const size_t* n_samples, int batch,
                       const q3asr_prompt* prompts);
/* stages: bit 0 mel, bit 1 encoder, bit 2 prefill (+ first token), bit 3 greedy decode */
#define Q3ASR_STAGE_MEL 1
#define Q3ASR_STAGE_ENCODER 2
#define Q3ASR_STAGE_PREFILL 4
#define Q3ASR_STAGE_DECODE 8
#define Q3ASR_STAGE_ALL 15
int q3asr_batch_run(q3asr_handle* h, int stages, int max_tokens, int stop_on_eos);
int q3asr_batch_download(q3asr_handle* h, int32_t* ids_out, int max_tokens, int* lens_out);
int q3asr_sync(q3asr_handle* h);
/* device-side timing on the handle's stream: record slot (0..15), elapsed between two recorded slots */
int q3asr_timer_record(q3asr_handle* h, int slot);
int q3asr_timer_elapsed_ms(q3asr_handle* h, int slot_a, int slot_b, float* ms);
/* per-stage device time of the last q3asr_batch_run: [mel, encoder, prefill, decode] in ms */
int q3asr_stage_ms(q3asr_handle* h, float* ms4);
/* kernels launched by this handle so far */
uint64_t q3asr_launch_count(const q3asr_handle* h);
/* the decode loop of the last q3asr_batch_run / q3asr_transcribe_ids*: out4 = {decode steps run, sum over the steps of the rows
 * decoded in that step, compactions of the decode batch, rows at the end}.  With stop_on_eos the finished utterances leave the
 * decode batch (the reference stops each utterance at EOS, Qwen3ASR.swift:378-379), so row-steps follow the tokens actually
 * generated instead of batch x longest utterance. */
int q3asr_decode_stats(const q3asr_handle* h, uint64_t* out4);
/* the last q3asr_transcribe_ids_continuous: out2 = {admissions (groups prefilled after the first), utterances admitted after the first
 * group}; {0, 0} after any other run */
int q3asr_decode_admissions(const q3asr_handle* h, uint64_t* out2);
/* per-kernel-family device timing (CUDA events around tagged launches of the encoder / prefill / decode stages).
 * report: one line per tag "tag,launches,total_ms,algorithmic_flops,algorithmic_bytes"; reading it resets the log. */
int q3asr_profile(q3asr_handle* h, int enable);
int q3asr_profile_report(q3asr_handle* h, char* buf, size_t cap);
/* L2 flush helper for benchmarks: overwrites a >L2-sized scratch buffer on the handle's stream */
int q3asr_flush_l2(q3asr_handle* h);

/* ---- utterance-batching scheduler over several GPUs of one box (one worker thread + handle per GPU,
 * weights replicated, utterances dealt longest-first; no collective on the data path).  Replaces the serial file loop of
 * `speech transcribe-batch` (Sources/AudioCLILib/TranscribeBatchCommand.swift:82-125); every utterance is independent because
 * transcribe builds a fresh cache per call (Qwen3ASR.swift:246-251). ---- */
int q3asr_pool_create(const q3asr_config* cfg, const int* devices, int n_devices, uint64_t random_seed, const char* weights_dir,
                      q3asr_pool** out);
void q3asr_pool_destroy(q3asr_pool* p);
/* message of the last failed call on this pool; p == NULL: why the last q3asr_pool_create on the calling thread failed */
const char* q3asr_pool_last_error(const q3asr_pool* p);
/* max_batch_per_gpu <= 0 picks the default sub-batch (256 utterances).  The device list of q3asr_pool_create may name a GPU more than
 * once: every entry is a worker with its own handle and stream, and two workers per GPU interleave the latency-bound decode steps of
 * their batches (+24 % aggregate throughput measured). */
int q3asr_pool_transcribe_ids(q3asr_pool* p, const float* const* pcm, const size_t* n_samples, int batch,
                              const q3asr_prompt* prompts, int max_tokens, int stop_on_eos, int max_batch_per_gpu,
                              int32_t* ids_out, int* lens_out);
/* the same with per-utterance sample rates (NULL = 16 kHz) and decoder knobs (NULL = greedy); the noise stream of a sampled run is
 * keyed by the position inside the sub-batch an utterance lands in, so sampled output depends on the schedule */
int q3asr_pool_transcribe_ids_opts(q3asr_pool* p, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                                   const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos,
                                   int max_batch_per_gpu, int32_t* ids_out, int* lens_out);
/* the same plus per-token log-probabilities (see q3asr_transcribe_ids_lp), logprobs_out [batch, max_tokens] (may be NULL) */
int q3asr_pool_transcribe_ids_lp(q3asr_pool* p, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                                 const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos,
                                 int max_batch_per_gpu, int32_t* ids_out, int* lens_out, float* logprobs_out);
/* Submit / wait form of the call above (the "optional submit/poll pair" of the scheduler): the batch runs on a thread of the
 * library while the caller prepares the next one.  The sample, prompt-id and sample-rate arrays are borrowed until q3asr_job_wait
 * returns (the pointer tables themselves are copied); jobs of one pool run one after the other.  q3asr_job_wait blocks, copies
 * ids [batch, max_tokens] / lens [batch] out and may be called once; q3asr_job_free joins if needed. */
/* enable != 0: every q3asr_pool_transcribe_ids* / q3asr_pool_submit* call runs each worker's whole length-sorted share through
 * q3asr_transcribe_ids_continuous with max_batch_per_gpu as max_rows, instead of sub-batches one after the other.  Same ids.  A call
 * with non-greedy decoder knobs on a continuous pool returns Q3ASR_ERR_INVALID. */
int q3asr_pool_set_continuous(q3asr_pool* p, int enable);
typedef struct q3asr_job q3asr_job;
int q3asr_pool_submit(q3asr_pool* p, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                      const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos, int max_batch_per_gpu,
                      q3asr_job** job);
int q3asr_job_done(const q3asr_job* job);
int q3asr_job_wait(q3asr_job* job, int32_t* ids_out, int* lens_out);
/* q3asr_pool_submit that also records per-token log-probabilities; after a successful q3asr_job_wait, q3asr_job_logprobs copies them
 * out ([batch, max_tokens]).  Q3ASR_ERR_INVALID for a job submitted without them or not yet waited for. */
int q3asr_pool_submit_lp(q3asr_pool* p, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                         const q3asr_prompt* prompts, const q3asr_sampling* sampling, int max_tokens, int stop_on_eos, int max_batch_per_gpu,
                         q3asr_job** job);
int q3asr_job_logprobs(const q3asr_job* job, float* logprobs_out);
const char* q3asr_job_last_error(const q3asr_job* job);
void q3asr_job_free(q3asr_job* job);
/* the scheduler's assignment alone (host logic; no GPU needed): gpu_out[i] = GPU of utterance i */
int q3asr_schedule(const size_t* n_samples, int batch, int n_gpus, int* gpu_out);

/* ---- tokenizer (host only; replaces Qwen3Tokenizer, Sources/AudioCommon/Tokenizer.swift:17-328) ---- */
typedef struct q3asr_tokenizer q3asr_tokenizer;
/* path: a directory holding vocab.json (+ optional tokenizer_config.json, merges.txt) or the vocab.json itself (Tokenizer.swift:38-62).
 * *out is set even on failure (read q3asr_tokenizer_last_error, then destroy). */
int q3asr_tokenizer_load(const char* path, q3asr_tokenizer** out);
/* the reference's test-only initialiser (Tokenizer.swift:31-35): explicit id -> token pairs, no merges */
int q3asr_tokenizer_from_pairs(const int32_t* ids, const char* const* tokens, int n, q3asr_tokenizer** out);
/* appends one merge rule (rank = number of rules so far); tests build small BPE tables with it */
int q3asr_tokenizer_add_merge(q3asr_tokenizer* t, const char* first, const char* second);
void q3asr_tokenizer_destroy(q3asr_tokenizer* t);
const char* q3asr_tokenizer_last_error(const q3asr_tokenizer* t);
int q3asr_tokenizer_size(const q3asr_tokenizer* t, int* n_tokens, int* n_merges);
/* ids -> UTF-8 text (Tokenizer.swift:111-142).  out may be NULL to query *needed (bytes incl. the terminator). */
int q3asr_tokenizer_decode(const q3asr_tokenizer* t, const int32_t* ids, int n, char* out, size_t cap, size_t* needed);
/* UTF-8 text -> ids (Tokenizer.swift:195-278).  ids may be NULL to query *n. */
int q3asr_tokenizer_encode(const q3asr_tokenizer* t, const char* text, int32_t* ids, int cap, int* n);
/* id of a token string, or -1 (Tokenizer.swift:281-283) */
int q3asr_tokenizer_token_id(const q3asr_tokenizer* t, const char* token);

/* Host-only: TextPreprocessor.prepareForAlignment (TextPreprocessing.swift:48-87) — q3asr_text_word_pairs, then per word
 * <timestamp> tokens(cleaned) <timestamp>; a word the tokenizer cannot encode hands its surface form to the previous word.
 * ids[0..*n_ids) is the slotted text q3asr_align_indices takes, positions[0..*n_positions) the indices of the <timestamp> slots in it
 * (two per word), words receives *n_positions / 2 NUL-terminated surface forms (*words_needed bytes).  All three buffers NULL =
 * sizing call.  timestamp_id: q3asr_config.tok_timestamp.  Errors: q3asr_text_last_error(). */
int q3asr_text_prepare_for_alignment(const q3asr_tokenizer* tok, const char* text, const char* language, int32_t timestamp_id, int32_t* ids,
                                     int ids_cap, int* n_ids, int* positions, int pos_cap, int* n_positions, char* words, size_t words_cap,
                                     size_t* words_needed);

/* ---- front door of the batched path: WAV, sample-rate conversion, long-form windows (SURVEY.md 8f rank 3) ---- */
/* message of the last failed q3asr_wav_* / q3asr_resample_design / q3asr_longform_plan call on this thread */
const char* q3asr_io_last_error(void);
/* AudioFileLoader.loadWAV (Sources/AudioCommon/AudioFileLoader.swift:70-157): RIFF/WAVE, PCM, 16-bit, any channel count (first
 * channel kept), samples / 32768.  Same rejections, in the same order, as the reference ("Invalid WAV file format",
 * "Unsupported audio format: Not PCM format" / "Not 16-bit").  samples may be NULL to query *n_samples (frames). */
int q3asr_wav_parse(const uint8_t* data, size_t size, float* samples, size_t cap, size_t* n_samples, int* sample_rate);
int q3asr_wav_load(const char* path, float* samples, size_t cap, size_t* n_samples, int* sample_rate);
/* WAVWriter.write(samples:sampleRate:to:) (Sources/AudioCommon/WAVWriter.swift:11-47), the writer on the other side of this format:
 * mono 16-bit PCM, 44-byte header, samples clamped to [-1, 1] and truncated toward zero after * 32767.  Host only. */
int q3asr_wav_write(const char* path, const float* samples, size_t n_samples, int sample_rate);
/* AudioFileLoader.resample (AudioFileLoader.swift:159-213).  Output length floor(n * out / in) as the reference computes it
 * (:190-191); the filter is a polyphase Kaiser-windowed sinc (csrc/audio_io.cu states the design; AVAudioConverter's own filter is
 * not part of the reference), evaluated on the GPU.  out may be NULL to query *n_out. */
size_t q3asr_resample_len(size_t n_samples, int in_rate, int out_rate);
int q3asr_resample(q3asr_handle* h, const float* in, size_t n_samples, int in_rate, int out_rate, float* out, size_t cap, size_t* n_out);
/* the filter bank itself (host only; parity tests): L = out/g, M = in/g, K, taps [L][2K+2] */
int q3asr_resample_design(int in_rate, int out_rate, int* L, int* M, int* K, float* taps, size_t cap, size_t* n_taps);
/* Qwen3ASRModel.transcribe(audio:sampleRate:...) resamples to 16 kHz first (AudioPreprocessing.swift:323-337; the reference's
 * batch command feeds 24 kHz, TranscribeBatchCommand.swift:73, 92): sample_rates[i] != 16000 clips are converted on the device,
 * straight into the packed sample buffer.  sample_rates may be NULL (all 16 kHz). */
int q3asr_batch_upload_sr(q3asr_handle* h, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                          const q3asr_prompt* prompts);
int q3asr_transcribe_ids_sr(q3asr_handle* h, const float* const* pcm, const size_t* n_samples, const int* sample_rates, int batch,
                            const q3asr_prompt* prompts, int max_tokens, int stop_on_eos, int32_t* ids_out, int* lens_out);
/* Long-form audio (BASELINE config 5): windows [k*window, min((k+1)*window, n)), each an independent utterance for the scheduler;
 * a tail shorter than min_tail samples joins the previous window.  starts/lens may be NULL (or cap too small) to query *count. */
int q3asr_longform_plan(size_t n_samples, size_t window, size_t min_tail, size_t* starts, size_t* lens, int cap, int* count);

/* ---- debug / test hooks (exercise single kernels through the C ABI) ---- */
/* C[M,N] = A[M,K] W[N,K]^T with bf16 (uint16) host operands; epi: 0 store(+bias,+gelu), 1 swiglu (W rows alternate
 * 32 gate / 32 up rows), 2 fp32, 3 argmax.
 * use_simt != 0 runs the CUDA-core checker kernel instead of tcgen05.  out: bf16 as uint16 (epi 0,1: [M,N] / [M,N/2]),
 * fp32 (epi 2) or int32 argmax ids [M] (epi 3). bn = 0 picks the tile width.
 * epi 4,5 run the decode-step weight-streaming kernel (M <= 128): 4 split-K fp32 partials summed -> fp32 [M,N]; 5 bf16 [M,N];
 * epi 7 runs the decode-step LM-head kernel (M <= 256): int32 argmax ids [M].  epi 8 (the LM-head kernel) and 9 (epi 3) also reduce
 * the log-sum-exp: int32 ids [M] followed by fp32 log-probabilities of those ids [M] (q3asr_transcribe_ids_lp's definition). */
int q3asr_debug_gemm(q3asr_handle* h, const uint16_t* A, const uint16_t* W, const uint16_t* bias, const uint16_t* resid, int M,
                     int N, int K, int epi, int gelu, int bn, int use_simt, void* out);
/* 3x3 stride-2 pad-1 NHWC convolution as implicit GEMM: in [B,H,W,C] bf16, w [O,3,3,C] bf16, out [B,OH,OW,O] bf16 (+bias, GELU) */
int q3asr_debug_conv(q3asr_handle* h, const uint16_t* in, const uint16_t* w, const uint16_t* bias, int B, int H, int W, int C, int O,
                     int box_w, int box_h, int box_b, int use_simt, uint16_t* out);

/* Segment-packed attention: q [rows, heads*hd], k/v [rows, (heads/group)*hd] bf16 (uint16), segments (row0, len) independent;
 * kernel: 0 = tcgen05/TMEM (attention_tc.cu, the product path), 1 = mma.sync checker (attention.cu).  out: [rows, heads*hd] bf16. */
int q3asr_debug_attention(q3asr_handle* h, const uint16_t* q, const uint16_t* k, const uint16_t* v, int rows, int heads, int group,
                          int head_dim, const int* seg_row0, const int* seg_len, int n_segs, int causal, float scale, int kernel,
                          uint16_t* out);

/* Decode-step attention of one layer for n_seqs sequences, as the decode step runs it (head_dim 128; needs a loaded model, whose
 * RoPE frequencies are used).  qkv_part: fp32 split-K partials of the QKV product [splits][n_seqs][(heads + 2*kv_heads)*128];
 * q_norm / k_norm: bf16 [128]; kv_len[s] includes the new token, whose position is kv_len[s] - 1; page_table [n_seqs][max_pages],
 * every entry in [0, n_pages); pool [n_pages][layers][2][kv_heads][32][128] bf16, in/out (the new k and v are appended at `layer`).
 * variant: 0 = the decode step's own choice, 1 / 2 / 8 = the tensor-core kernel (1: two single-warp CTAs per item), 4 / 16 = the
 * SIMT kernel's 4 / 16 warps (these need heads == 2*kv_heads); -1 = the general path (partials summed on the host in split order,
 * rounded to bf16, then the separate norm + RoPE + append kernel and the paged attention kernel; heads / kv_heads 1 or 2).
 * The same launch runs `launches` times back to back on the same buffers.  out: [launches][n_seqs][heads*128] bf16. */
int q3asr_debug_decode_attention(q3asr_handle* h, const float* qkv_part, int splits, int n_seqs, int heads, int kv_heads,
                                 const uint16_t* q_norm, const uint16_t* k_norm, float eps, float scale, const int* kv_len,
                                 const int* page_table, int max_pages, uint16_t* pool, int n_pages, int layers, int layer, int variant,
                                 int launches, uint16_t* out);

/* One decoder layer's prefill attention block for packed prompts, through the same host function as the prefill (head_dim 128;
 * needs a loaded model, whose RoPE frequencies are tabulated for max_pages*32 positions).  x: the normed hidden states
 * [rows][hidden] bf16; w: the fused weight [(heads + 2*kv_heads)*128][hidden] bf16 in q | k | v row order; q_norm / k_norm: bf16
 * [128].  Segment s holds rows seg_row0[s] .. + seg_len[s] - 1 at positions 0 .. seg_len[s] - 1, and its KV pages are
 * page_table row seg_table_row[s]; the segments are packed back to back from row 0 and cover the rows.  page_table
 * [table_rows][max_pages], every entry in [0, n_pages); pool [n_pages][layers][2][kv_heads][32][128] bf16, in/out (k and v are
 * written at `layer`).  qkv_variant: 0 = norm, RoPE and cache write in the product's epilogue (the prefill's path), -1 = the plain
 * product + the separate norm / RoPE / cache kernel.  bn: the product's tile width, 0 = the prefill's choice, or 128 / 256.
 * attn_variant: 0 = the tcgen05 kernel (the prefill's), 1 = the mma.sync kernel, -1 = none.  Outputs (bf16): q_out [rows][heads*128],
 * k_out [rows][kv_heads*128], qkv_out [rows][(heads + 2*kv_heads)*128] (under qkv_variant 0 only its v columns are written),
 * att_out [rows][heads*128]; whatever the call does not write reads back as NaN. */
int q3asr_debug_prefill_attention(q3asr_handle* h, const uint16_t* x, const uint16_t* w, int rows, int hidden, int heads, int kv_heads,
                                  const uint16_t* q_norm, const uint16_t* k_norm, float eps, float scale, const int* seg_row0,
                                  const int* seg_len, const int* seg_table_row, int n_segs, const int* page_table, int table_rows,
                                  int max_pages, uint16_t* pool, int n_pages, int layers, int layer, int qkv_variant, int bn,
                                  int attn_variant, uint16_t* q_out, uint16_t* k_out, uint16_t* qkv_out, uint16_t* att_out);

#ifdef __cplusplus
}
#endif
#endif /* Q3ASR_H */
