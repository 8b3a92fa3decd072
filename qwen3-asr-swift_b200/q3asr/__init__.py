"""ctypes binding of libq3asr.so — the Python host side above the C ABI (include/q3asr.h).

The reference's host language is Swift (no toolchain in this image); this module mirrors the reference's
operator interface for the path so the parity tests read like the reference's own:

    Qwen3ASRModel.fromPretrained / transcribe      /root/reference/Sources/Qwen3ASR/Qwen3ASR.swift:107-164, 608-668
    WhisperFeatureExtractor.extractFeaturesRaw     /root/reference/Sources/Qwen3ASR/AudioPreprocessing.swift:347-470
    Qwen3AudioEncoder.callAsFunction               /root/reference/Sources/Qwen3ASR/AudioEncoder.swift:362-511

There is no CPU fallback and nothing here imports oracle/: if the shared library is missing, or no
Blackwell GPU is present, construction fails loudly.
"""
import ctypes
import os

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG, "lib", "libq3asr.so")

OK = 0
STAGE_MEL, STAGE_ENCODER, STAGE_PREFILL, STAGE_DECODE, STAGE_ALL = 1, 2, 4, 8, 15
EPI_NORMAL, EPI_SWIGLU, EPI_F32, EPI_ARGMAX = 0, 1, 2, 3
EPI_SKINNY_PARTIAL, EPI_SKINNY_STORE = 4, 5  # decode-step weight-streaming kernel


class Q3Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"q3asr error {code}: {msg}")
        self.code = code


class Config(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in (
        "enc_d_model", "enc_heads", "enc_ffn", "enc_layers", "enc_out_dim", "enc_conv_ch", "enc_n_window",
        "enc_n_window_infer")] + [("enc_ln_eps", ctypes.c_float)] + [(n, ctypes.c_int) for n in (
            "dec_vocab", "dec_hidden", "dec_layers", "dec_heads", "dec_kv_heads", "dec_head_dim", "dec_inter")] + [
                ("dec_rope_theta", ctypes.c_float), ("dec_rms_eps", ctypes.c_float)] + [(n, ctypes.c_int32) for n in (
                    "tok_im_start", "tok_im_end", "tok_audio_start", "tok_audio_end", "tok_audio_pad", "tok_asr_text",
                    "tok_newline", "tok_system", "tok_user", "tok_assistant", "tok_eos")] + [
                        ("classify_num", ctypes.c_int), ("tok_timestamp", ctypes.c_int32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class Prompt(ctypes.Structure):
    _fields_ = [("context_ids", ctypes.POINTER(ctypes.c_int32)), ("n_context", ctypes.c_int),
                ("language_ids", ctypes.POINTER(ctypes.c_int32)), ("n_language", ctypes.c_int), ("raw_suffix", ctypes.c_int)]


class Sampling(ctypes.Structure):
    """q3asr_sampling: the decoder knobs of Qwen3DecodingOptions (Qwen3ASR.swift:13-51)."""
    _fields_ = [("repetition_penalty", ctypes.c_float), ("no_repeat_ngram_size", ctypes.c_int), ("temperature", ctypes.c_float),
                ("seed", ctypes.c_uint64), ("force_device_sampler", ctypes.c_int)]


class Qwen3DecodingOptions:
    """Qwen3DecodingOptions (Qwen3ASR.swift:13-51), same names and defaults; `seed` keys the reproducible Gumbel noise stream."""

    def __init__(self, max_tokens=448, language=None, context=None, repetition_penalty=1.0, no_repeat_ngram_size=0, temperature=0.0,
                 seed=0):
        self.max_tokens, self.language, self.context = max_tokens, language, context
        self.repetition_penalty, self.no_repeat_ngram_size, self.temperature, self.seed = repetition_penalty, no_repeat_ngram_size, temperature, seed

    @property
    def is_greedy_fast_path(self):  # Qwen3ASR.swift:300-304
        return self.repetition_penalty == 1.0 and self.no_repeat_ngram_size == 0 and self.temperature == 0.0

    def c_struct(self, force_device_sampler=False):
        return Sampling(float(self.repetition_penalty), int(self.no_repeat_ngram_size), float(self.temperature), int(self.seed),
                        int(bool(force_device_sampler)))


# every symbol include/q3asr.h declares (tests/test_abi.py checks the library exports all of them)
EXPORTS = [
    "q3asr_config_preset", "q3asr_version", "q3asr_last_error", "q3asr_create", "q3asr_destroy", "q3asr_init_random",
    "q3asr_tensor_count", "q3asr_tensor_info", "q3asr_set_tensor", "q3asr_get_tensor", "q3asr_commit_weights",
    "q3asr_load_safetensors", "q3asr_checkpoint_list", "q3asr_is_loaded", "q3asr_unload", "q3asr_memory_footprint", "q3asr_mel_frames", "q3asr_mel",
    "q3asr_mel_batch", "q3asr_encoder_tokens", "q3asr_prompt_ids", "q3asr_text_word_pairs", "q3asr_text_last_error", "q3asr_text_prepare_for_alignment", "q3asr_encode", "q3asr_transcribe_ids", "q3asr_decode_forced", "q3asr_decode_forced_embeds",
    "q3asr_prefill_logits", "q3asr_batch_upload", "q3asr_batch_run", "q3asr_batch_download", "q3asr_sync",
    "q3asr_timer_record", "q3asr_timer_elapsed_ms", "q3asr_stage_ms", "q3asr_launch_count", "q3asr_decode_stats", "q3asr_flush_l2",
    "q3asr_profile", "q3asr_profile_report",
    "q3asr_pool_create", "q3asr_pool_destroy", "q3asr_pool_last_error", "q3asr_pool_transcribe_ids", "q3asr_schedule",
    "q3asr_debug_gemm", "q3asr_debug_conv", "q3asr_debug_attention", "q3asr_debug_decode_attention", "q3asr_debug_prefill_attention",
    "q3asr_tokenizer_load", "q3asr_tokenizer_from_pairs", "q3asr_tokenizer_add_merge", "q3asr_tokenizer_destroy",
    "q3asr_tokenizer_last_error", "q3asr_tokenizer_size", "q3asr_tokenizer_decode", "q3asr_tokenizer_encode", "q3asr_tokenizer_token_id",
    "q3asr_io_last_error", "q3asr_wav_parse", "q3asr_wav_load", "q3asr_wav_write", "q3asr_resample_len", "q3asr_resample", "q3asr_resample_design",
    "q3asr_batch_upload_sr", "q3asr_transcribe_ids_sr", "q3asr_longform_plan",
    "q3asr_transcribe_ids_opts", "q3asr_batch_set_sampling", "q3asr_pick_next_token",
    "q3asr_align_indices", "q3asr_enforce_monotonicity", "q3asr_lis_positions", "q3asr_trailing_plateau_start",
    "q3asr_pool_transcribe_ids_opts", "q3asr_pool_submit", "q3asr_job_done", "q3asr_job_wait", "q3asr_job_last_error", "q3asr_job_free",
    "q3asr_transcribe_ids_lp", "q3asr_batch_set_logprobs", "q3asr_batch_download_logprobs", "q3asr_pool_transcribe_ids_lp",
    "q3asr_pool_submit_lp", "q3asr_job_logprobs",
    "q3asr_transcribe_ids_continuous", "q3asr_decode_admissions", "q3asr_pool_set_continuous",
]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Q3Error(-1, f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        vp, ci, cs = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
        L.q3asr_version.restype = ctypes.c_char_p
        L.q3asr_last_error.restype = ctypes.c_char_p
        L.q3asr_last_error.argtypes = [vp]
        L.q3asr_pool_last_error.restype = ctypes.c_char_p
        L.q3asr_pool_last_error.argtypes = [vp]
        L.q3asr_config_preset.argtypes = [ctypes.c_char_p, ctypes.POINTER(Config)]
        L.q3asr_create.argtypes = [ctypes.POINTER(Config), ci, ctypes.POINTER(vp)]
        L.q3asr_destroy.argtypes = [vp]
        L.q3asr_destroy.restype = None
        L.q3asr_init_random.argtypes = [vp, ctypes.c_uint64]
        L.q3asr_tensor_count.argtypes = [vp]
        L.q3asr_tensor_info.argtypes = [vp, ci, ctypes.c_char_p, ci, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ci)]
        L.q3asr_set_tensor.argtypes = [vp, ctypes.c_char_p, vp, ci, ctypes.POINTER(ctypes.c_int64), ci]
        L.q3asr_get_tensor.argtypes = [vp, ctypes.c_char_p, vp, cs]
        L.q3asr_commit_weights.argtypes = [vp]
        L.q3asr_load_safetensors.argtypes = [vp, ctypes.c_char_p]
        L.q3asr_checkpoint_list.argtypes = [ctypes.c_char_p, ctypes.c_char_p, cs, ctypes.POINTER(cs)]
        L.q3asr_is_loaded.argtypes = [vp]
        L.q3asr_unload.argtypes = [vp]
        L.q3asr_memory_footprint.argtypes = [vp]
        L.q3asr_memory_footprint.restype = cs
        L.q3asr_mel_frames.argtypes = [cs]
        L.q3asr_mel.argtypes = [vp, vp, cs, vp, ctypes.POINTER(ci)]
        L.q3asr_mel_batch.argtypes = [vp, vp, vp, ci, vp, vp]
        L.q3asr_encoder_tokens.argtypes = [ci]
        L.q3asr_text_word_pairs.argtypes = [ctypes.c_char_p, ctypes.c_char_p, vp, cs, ctypes.POINTER(cs), ctypes.POINTER(ci)]
        L.q3asr_text_last_error.restype = ctypes.c_char_p
        L.q3asr_text_prepare_for_alignment.argtypes = [vp, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int32, vp, ci, ctypes.POINTER(ci), vp, ci,
                                                       ctypes.POINTER(ci), vp, cs, ctypes.POINTER(cs)]
        L.q3asr_prompt_ids.argtypes = [vp, ci, vp, vp, ci, ctypes.POINTER(ci), ctypes.POINTER(ci)]
        L.q3asr_encode.argtypes = [vp, vp, ci, vp, ctypes.POINTER(ci)]
        L.q3asr_transcribe_ids.argtypes = [vp, vp, vp, ci, vp, ci, ci, vp, vp]
        L.q3asr_decode_forced.argtypes = [vp, vp, cs, vp, vp, ci, vp, vp]
        L.q3asr_decode_forced_embeds.argtypes = [vp, vp, cs, vp, vp, ci, vp, ci, vp, vp]
        L.q3asr_prefill_logits.argtypes = [vp, vp, cs, vp, vp]
        L.q3asr_batch_upload.argtypes = [vp, vp, vp, ci, vp]
        L.q3asr_batch_run.argtypes = [vp, ci, ci, ci]
        L.q3asr_batch_download.argtypes = [vp, vp, ci, vp]
        L.q3asr_sync.argtypes = [vp]
        L.q3asr_timer_record.argtypes = [vp, ci]
        L.q3asr_timer_elapsed_ms.argtypes = [vp, ci, ci, ctypes.POINTER(ctypes.c_float)]
        L.q3asr_stage_ms.argtypes = [vp, vp]
        L.q3asr_launch_count.argtypes = [vp]
        L.q3asr_launch_count.restype = ctypes.c_uint64
        L.q3asr_decode_stats.argtypes = [vp, vp]
        L.q3asr_flush_l2.argtypes = [vp]
        L.q3asr_profile.argtypes = [vp, ci]
        L.q3asr_profile_report.argtypes = [vp, ctypes.c_char_p, cs]
        L.q3asr_pool_create.argtypes = [ctypes.POINTER(Config), vp, ci, ctypes.c_uint64, ctypes.c_char_p, ctypes.POINTER(vp)]
        L.q3asr_pool_destroy.argtypes = [vp]
        L.q3asr_pool_destroy.restype = None
        L.q3asr_pool_transcribe_ids.argtypes = [vp, vp, vp, ci, vp, ci, ci, ci, vp, vp]
        L.q3asr_schedule.argtypes = [vp, ci, ci, vp]
        L.q3asr_pool_submit.argtypes = [vp, vp, vp, vp, ci, vp, ctypes.POINTER(Sampling), ci, ci, ci, ctypes.POINTER(vp)]
        L.q3asr_job_done.argtypes = [vp]
        L.q3asr_job_wait.argtypes = [vp, vp, vp]
        L.q3asr_job_last_error.argtypes = [vp]
        L.q3asr_job_last_error.restype = ctypes.c_char_p
        L.q3asr_job_free.argtypes = [vp]
        L.q3asr_job_free.restype = None
        L.q3asr_pool_transcribe_ids_opts.argtypes = [vp, vp, vp, vp, ci, vp, ctypes.POINTER(Sampling), ci, ci, ci, vp, vp]
        L.q3asr_debug_gemm.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, vp]
        L.q3asr_debug_conv.argtypes = [vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, ci, ci, vp]
        L.q3asr_debug_attention.argtypes = [vp, vp, vp, vp, ci, ci, ci, ci, vp, vp, ci, ci, ctypes.c_float, ci, vp]
        L.q3asr_debug_decode_attention.argtypes = [vp, vp, ci, ci, ci, ci, vp, vp, ctypes.c_float, ctypes.c_float, vp, vp, ci, vp, ci, ci,
                                                   ci, ci, ci, vp]
        L.q3asr_debug_prefill_attention.argtypes = [vp, vp, vp, ci, ci, ci, ci, vp, vp, ctypes.c_float, ctypes.c_float, vp, vp, vp, ci, vp,
                                                    ci, ci, vp, ci, ci, ci, ci, ci, ci, vp, vp, vp, vp]
        L.q3asr_tokenizer_load.argtypes = [ctypes.c_char_p, ctypes.POINTER(vp)]
        L.q3asr_tokenizer_from_pairs.argtypes = [vp, vp, ci, ctypes.POINTER(vp)]
        L.q3asr_tokenizer_add_merge.argtypes = [vp, ctypes.c_char_p, ctypes.c_char_p]
        L.q3asr_tokenizer_destroy.argtypes = [vp]
        L.q3asr_tokenizer_destroy.restype = None
        L.q3asr_tokenizer_last_error.argtypes = [vp]
        L.q3asr_tokenizer_last_error.restype = ctypes.c_char_p
        L.q3asr_tokenizer_size.argtypes = [vp, ctypes.POINTER(ci), ctypes.POINTER(ci)]
        L.q3asr_tokenizer_decode.argtypes = [vp, vp, ci, ctypes.c_char_p, cs, ctypes.POINTER(cs)]
        L.q3asr_tokenizer_encode.argtypes = [vp, ctypes.c_char_p, vp, ci, ctypes.POINTER(ci)]
        L.q3asr_tokenizer_token_id.argtypes = [vp, ctypes.c_char_p]
        L.q3asr_io_last_error.restype = ctypes.c_char_p
        L.q3asr_wav_parse.argtypes = [vp, cs, vp, cs, ctypes.POINTER(cs), ctypes.POINTER(ci)]
        L.q3asr_wav_write.argtypes = [ctypes.c_char_p, vp, cs, ci]
        L.q3asr_wav_load.argtypes = [ctypes.c_char_p, vp, cs, ctypes.POINTER(cs), ctypes.POINTER(ci)]
        L.q3asr_resample_len.argtypes = [cs, ci, ci]
        L.q3asr_resample_len.restype = cs
        L.q3asr_resample.argtypes = [vp, vp, cs, ci, ci, vp, cs, ctypes.POINTER(cs)]
        L.q3asr_resample_design.argtypes = [ci, ci, ctypes.POINTER(ci), ctypes.POINTER(ci), ctypes.POINTER(ci), vp, cs, ctypes.POINTER(cs)]
        L.q3asr_batch_upload_sr.argtypes = [vp, vp, vp, vp, ci, vp]
        L.q3asr_transcribe_ids_sr.argtypes = [vp, vp, vp, vp, ci, vp, ci, ci, vp, vp]
        L.q3asr_longform_plan.argtypes = [cs, cs, cs, vp, vp, ci, ctypes.POINTER(ci)]
        L.q3asr_transcribe_ids_opts.argtypes = [vp, vp, vp, vp, ci, vp, ctypes.POINTER(Sampling), ci, ci, vp, vp]
        L.q3asr_batch_set_sampling.argtypes = [vp, ctypes.POINTER(Sampling)]
        L.q3asr_align_indices.argtypes = [vp, vp, vp, vp, ci, vp, vp, vp, vp, vp]
        L.q3asr_enforce_monotonicity.argtypes = [vp, ci, vp]
        L.q3asr_lis_positions.argtypes = [vp, ci, vp, ctypes.POINTER(ci)]
        L.q3asr_trailing_plateau_start.argtypes = [vp, ci, ctypes.c_float, ci]
        L.q3asr_pick_next_token.argtypes = [vp, vp, ci, vp, ci, ctypes.POINTER(Sampling), ci, ctypes.POINTER(ctypes.c_int32)]
        L.q3asr_transcribe_ids_lp.argtypes = [vp, vp, vp, vp, ci, vp, ctypes.POINTER(Sampling), ci, ci, vp, vp, vp]
        L.q3asr_batch_set_logprobs.argtypes = [vp, ci]
        L.q3asr_batch_download_logprobs.argtypes = [vp, vp, ci]
        L.q3asr_pool_transcribe_ids_lp.argtypes = [vp, vp, vp, vp, ci, vp, ctypes.POINTER(Sampling), ci, ci, ci, vp, vp, vp]
        L.q3asr_pool_submit_lp.argtypes = [vp, vp, vp, vp, ci, vp, ctypes.POINTER(Sampling), ci, ci, ci, ctypes.POINTER(vp)]
        L.q3asr_job_logprobs.argtypes = [vp, vp]
        L.q3asr_transcribe_ids_continuous.argtypes = [vp, vp, vp, vp, ci, vp, ci, ci, ci, vp, vp, vp]
        L.q3asr_decode_admissions.argtypes = [vp, vp]
        L.q3asr_pool_set_continuous.argtypes = [vp, ci]
        _lib = L
    return _lib


def version():
    return lib().q3asr_version().decode()


def preset(name):
    c = Config()
    rc = lib().q3asr_config_preset(name.encode(), ctypes.byref(c))
    if rc != OK:
        raise Q3Error(rc, f"unknown preset {name!r}")
    return c


def mel_frames(n):
    return lib().q3asr_mel_frames(int(n))


def encoder_tokens(frames):
    return lib().q3asr_encoder_tokens(int(frames))


def prompt_ids(config, n_audio_tokens, context=None, language=None, raw_suffix=False):
    """The chat-template ids the prefill runs on (Qwen3ASR.swift:196-233) and the index of the first <|audio_pad|>; host logic,
    no GPU needed."""
    pack = _PromptPack([{"context": context, "language": language, "raw_suffix": raw_suffix}], 1)
    n, at = ctypes.c_int(0), ctypes.c_int(0)
    cfg = ctypes.byref(config)
    rc = lib().q3asr_prompt_ids(cfg, int(n_audio_tokens), pack.ptr, None, 0, ctypes.byref(n), ctypes.byref(at))
    if n.value == 0:
        raise ValueError(f"q3asr_prompt_ids: invalid argument (code {rc})")
    out = np.empty(n.value, dtype=np.int32)
    rc = lib().q3asr_prompt_ids(cfg, int(n_audio_tokens), pack.ptr, out.ctypes.data, out.size, ctypes.byref(n), ctypes.byref(at))
    if rc != 0:
        raise ValueError(f"q3asr_prompt_ids failed with code {rc}")
    return out, at.value


def schedule(n_samples, n_gpus):
    """The scheduler's utterance -> GPU assignment (host logic, no GPU needed)."""
    n = np.ascontiguousarray(n_samples, dtype=np.uint64)
    out = np.zeros(n.size, dtype=np.int32)
    rc = lib().q3asr_schedule(n.ctypes.data, n.size, int(n_gpus), out.ctypes.data)
    if rc != OK:
        raise Q3Error(rc, "schedule: bad argument")
    return out


class AudioLoadError(Q3Error):
    """AudioLoadError of the reference (AudioFileLoader.swift:216-234): invalidWAVFile / unsupportedFormat."""


class AudioFileLoader:
    """AudioFileLoader.loadWAV / resample of the reference (Sources/AudioCommon/AudioFileLoader.swift:70-213)."""

    @staticmethod
    def _finish(rc):
        if rc != OK:
            raise AudioLoadError(rc, lib().q3asr_io_last_error().decode())

    @staticmethod
    def parse_wav(data):
        """bytes of a RIFF/WAVE PCM16 file -> (float32 samples of the first channel, sample rate)."""
        buf = np.frombuffer(bytes(data), dtype=np.uint8)
        n, rate = ctypes.c_size_t(), ctypes.c_int()
        ptr = buf.ctypes.data if buf.size else None
        AudioFileLoader._finish(lib().q3asr_wav_parse(ptr, buf.size, None, 0, ctypes.byref(n), ctypes.byref(rate)))
        out = np.empty(n.value, dtype=np.float32)
        AudioFileLoader._finish(lib().q3asr_wav_parse(ptr, buf.size, out.ctypes.data, out.size, ctypes.byref(n), ctypes.byref(rate)))
        return out, int(rate.value)

    @staticmethod
    def load_wav(path):
        with open(path, "rb") as f:
            return AudioFileLoader.parse_wav(f.read())

    @staticmethod
    def write_wav(path, samples, sample_rate=24000):
        """WAVWriter.write (Sources/AudioCommon/WAVWriter.swift:11-47): mono PCM16."""
        x = np.ascontiguousarray(samples, dtype=np.float32)
        AudioFileLoader._finish(lib().q3asr_wav_write(os.fsencode(path), x.ctypes.data if x.size else None, x.size, int(sample_rate)))

    @staticmethod
    def resample_len(n, in_rate, out_rate):
        return int(lib().q3asr_resample_len(int(n), int(in_rate), int(out_rate)))

    @staticmethod
    def resample_design(in_rate, out_rate):
        """(L, M, K, taps [L, 2K+2]) of the polyphase converter (csrc/audio_io.cu)."""
        L, M, K, nt = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_size_t()
        AudioFileLoader._finish(lib().q3asr_resample_design(int(in_rate), int(out_rate), ctypes.byref(L), ctypes.byref(M), ctypes.byref(K),
                                                            None, 0, ctypes.byref(nt)))
        taps = np.empty(nt.value, dtype=np.float32)
        AudioFileLoader._finish(lib().q3asr_resample_design(int(in_rate), int(out_rate), ctypes.byref(L), ctypes.byref(M), ctypes.byref(K),
                                                            taps.ctypes.data, taps.size, ctypes.byref(nt)))
        return L.value, M.value, K.value, taps.reshape(L.value, 2 * K.value + 2)


def enforce_monotonicity(raw_indices):
    """TimestampCorrection.enforceMonotonicity (TimestampCorrection.swift:15-98)."""
    a = np.ascontiguousarray(raw_indices, dtype=np.int32)
    out = np.empty_like(a)
    rc = lib().q3asr_enforce_monotonicity(a.ctypes.data if a.size else None, a.size, out.ctypes.data if a.size else None)
    if rc != OK:
        raise Q3Error(rc, "enforce_monotonicity: bad argument")
    return out.tolist()


def lis_positions(values):
    """TimestampCorrection.longestIncreasingSubsequencePositions (TimestampCorrection.swift:101-144)."""
    a = np.ascontiguousarray(values, dtype=np.int32)
    out = np.empty(max(a.size, 1), dtype=np.int32)
    cnt = ctypes.c_int()
    rc = lib().q3asr_lis_positions(a.ctypes.data if a.size else None, a.size, out.ctypes.data, ctypes.byref(cnt))
    if rc != OK:
        raise Q3Error(rc, "lis_positions: bad argument")
    return out[:cnt.value].tolist()


def trailing_plateau_start(start_times, tolerance=0.1, min_size=5):
    """Qwen3ForcedAligner.findTrailingPlateauStart (ForcedAligner.swift:191-216)."""
    a = np.ascontiguousarray(start_times, dtype=np.float32)
    return int(lib().q3asr_trailing_plateau_start(a.ctypes.data if a.size else None, a.size, float(tolerance), int(min_size)))


def longform_plan(n_samples, window, min_tail=160):
    """[(start, length)] windows of a long recording (each an independent utterance for the scheduler)."""
    cnt = ctypes.c_int()
    rc = lib().q3asr_longform_plan(int(n_samples), int(window), int(min_tail), None, None, 0, ctypes.byref(cnt))
    if rc != OK:
        raise Q3Error(rc, lib().q3asr_io_last_error().decode())
    starts = np.zeros(max(cnt.value, 1), dtype=np.uint64)
    lens = np.zeros(max(cnt.value, 1), dtype=np.uint64)
    rc = lib().q3asr_longform_plan(int(n_samples), int(window), int(min_tail), starts.ctypes.data, lens.ctypes.data, cnt.value, ctypes.byref(cnt))
    if rc != OK:
        raise Q3Error(rc, lib().q3asr_io_last_error().decode())
    return [(int(starts[i]), int(lens[i])) for i in range(cnt.value)]


def avg_logprob(logprobs):
    """Utterance score of one utterance's per-token log-probabilities (include/q3asr.h): their mean, EOS included; exp() of it is
    the confidence.  An empty utterance scores 0."""
    lp = np.asarray(logprobs, dtype=np.float64)
    return float(lp.mean()) if lp.size else 0.0


def f32_to_bf16_bits(x):
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    return r


def bf16_bits_to_f32(b):
    return (np.ascontiguousarray(b, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)


def _ptr_array(arrs):
    return (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])


def text_word_pairs(text, language="English"):
    """TextPreprocessor.splitIntoWordPairs through the library (csrc/text.cu): [(surface, cleaned)].  `text` may be str or UTF-8 bytes."""
    raw = text.encode("utf-8") if isinstance(text, str) else bytes(text)
    if b"\0" in raw:
        raise ValueError("text_word_pairs: embedded NUL")
    need, n = ctypes.c_size_t(), ctypes.c_int()
    lang = language.encode("utf-8") if language is not None else None
    rc = lib().q3asr_text_word_pairs(raw, lang, None, 0, ctypes.byref(need), ctypes.byref(n))
    if rc != OK:
        raise Q3Error(rc, lib().q3asr_text_last_error().decode("utf-8", "replace"))
    buf = ctypes.create_string_buffer(max(need.value, 1))
    rc = lib().q3asr_text_word_pairs(raw, lang, buf, need.value, ctypes.byref(need), ctypes.byref(n))
    if rc != OK:
        raise Q3Error(rc, lib().q3asr_text_last_error().decode("utf-8", "replace"))
    parts = buf.raw[:need.value].split(b"\0")[:2 * n.value]
    dec = (lambda b: b.decode("utf-8")) if isinstance(text, str) else (lambda b: b)
    return [(dec(parts[2 * i]), dec(parts[2 * i + 1])) for i in range(n.value)]


def text_prepare_for_alignment(tokenizer, text, language="English", timestamp_token_id=151705):
    """TextPreprocessor.prepareForAlignment through the library: (token_ids, timestamp_positions, words), the tuple q3asr.text's
    pure-Python twin returns.  `tokenizer` is a Qwen3Tokenizer (the native one)."""
    n_ids, n_pos, need = ctypes.c_int(), ctypes.c_int(), ctypes.c_size_t()
    raw = text.encode("utf-8")
    lang = language.encode("utf-8") if language is not None else None

    def call(ids, pos, words):
        rc = lib().q3asr_text_prepare_for_alignment(tokenizer._t, raw, lang, int(timestamp_token_id), ids.ctypes.data if ids is not None else None,
                                                    ids.size if ids is not None else 0, ctypes.byref(n_ids),
                                                    pos.ctypes.data if pos is not None else None, pos.size if pos is not None else 0,
                                                    ctypes.byref(n_pos), words, len(words) if words is not None else 0, ctypes.byref(need))
        if rc != OK:
            raise Q3Error(rc, lib().q3asr_text_last_error().decode("utf-8", "replace"))

    call(None, None, None)
    ids, pos = np.zeros(max(n_ids.value, 1), dtype=np.int32), np.zeros(max(n_pos.value, 1), dtype=np.int32)
    words = ctypes.create_string_buffer(max(need.value, 1))
    call(ids, pos, words)
    surf = [w.decode("utf-8") for w in words.raw[:need.value].split(b"\0")[:n_pos.value // 2]]
    return [int(v) for v in ids[:n_ids.value]], [int(v) for v in pos[:n_pos.value]], surf


def checkpoint_list(model_dir):
    """[(name, dtype, shape, bytes)] of the tensors q3asr_load_safetensors would read from model_dir (host only; raises Q3Error with
    the loader's message when a header is malformed or points outside its file)."""
    need = ctypes.c_size_t()
    d = os.fsencode(model_dir)
    rc = lib().q3asr_checkpoint_list(d, None, 0, ctypes.byref(need))
    buf = ctypes.create_string_buffer(max(need.value, 1))
    rc = lib().q3asr_checkpoint_list(d, buf, len(buf), ctypes.byref(need))
    if rc != OK:
        raise Q3Error(rc, buf.value.decode("utf-8", "replace"))
    out = []
    for line in buf.value.decode("utf-8", "replace").splitlines():
        name, dtype, shape, nbytes = line.split("\t")
        out.append((name, dtype, tuple(int(v) for v in shape.split("x")), int(nbytes)))
    return out


def detect_preset_from_checkpoint(model_dir):
    """The preset a checkpoint directory holds, read from its tensor index (host only): "aligner" when it carries the classification
    head (lm_head.*, WeightLoading.swift:177-179), else "0.6B" / "1.7B" by the decoder width (model.norm.weight: 1024 / 2048,
    Configuration.swift:47-100).  None when the index does not say (the caller falls back to the model id, like the reference)."""
    shapes = {name: shape for name, _, shape, _ in checkpoint_list(model_dir)}
    if "lm_head.weight" in shapes:
        return "aligner"
    return {(1024,): "0.6B", (2048,): "1.7B"}.get(shapes.get("model.norm.weight"))


def detect_model_size(model_id):
    """ASRModelSize.detect (Qwen3ASR.swift:581-586): the preset name for a model id."""
    return "1.7B" if ("1.7B" in model_id or "1.7b" in model_id) else "0.6B"


def detect_bits(model_id):
    """ASRModelSize.detectBits (Qwen3ASR.swift:588-600).  The loader reads the packing from the tensor shapes; this is the reference's
    id convention, kept for callers that pick a checkpoint directory by id."""
    low = model_id.lower()
    if "8bit" in low or "8-bit" in low:
        return 8
    if "4bit" in low or "4-bit" in low:
        return 4
    return 8 if detect_model_size(model_id) == "1.7B" else 4


_SWIFT_WHITESPACES = " \t\u00a0\u1680\u2000\u2001\u2002\u2003\u2004\u2005\u2006\u2007\u2008\u2009\u200a\u202f\u205f\u3000"  # CharacterSet.whitespaces


class _PromptPack:
    """Keeps the numpy arrays behind an array of q3asr_prompt alive."""

    def __init__(self, prompts, batch):
        self.keep = []
        self.arr = None
        if prompts is None:
            return
        assert len(prompts) == batch
        self.arr = (Prompt * batch)()
        for i, p in enumerate(prompts):
            ctx, lang = (p or {}).get("context"), (p or {}).get("language")
            for key, ids in (("context", ctx), ("language", lang)):
                if ids is not None and len(ids):
                    a = np.ascontiguousarray(ids, dtype=np.int32)
                    self.keep.append(a)
                    setattr(self.arr[i], f"{key}_ids", a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)))
                    setattr(self.arr[i], f"n_{key}", a.size)
            self.arr[i].raw_suffix = int(bool((p or {}).get("raw_suffix", False)))

    @property
    def ptr(self):
        return ctypes.cast(self.arr, ctypes.c_void_p) if self.arr is not None else None


class Qwen3ASRModel:
    """Mirror of the reference's Qwen3ASRModel for the transcription path (ids instead of text: the
    tokenizer stays on the Swift side, and with no tokenizer the reference itself returns the ids joined by
    spaces, Qwen3ASR.swift:290-293)."""

    def __init__(self, size="0.6B", device=0, config=None):
        self.cfg = config if config is not None else preset(size)
        self._h = ctypes.c_void_p()
        rc = lib().q3asr_create(ctypes.byref(self.cfg), int(device), ctypes.byref(self._h))
        if rc != OK:
            raise Q3Error(rc, lib().q3asr_last_error(None).decode())

    # -- lifecycle ---------------------------------------------------------------------------
    @classmethod
    def from_pretrained(cls, model_dir, size=None, device=0):
        """size None: decided from the checkpoint's own tensor index, else from the directory name like ASRModelSize.detect does from
        the model id (Qwen3ASR.swift:615)."""
        if size is None:  # what the files say first, then the directory name
            size = detect_preset_from_checkpoint(model_dir) or detect_model_size(os.path.basename(os.path.normpath(os.fspath(model_dir))))
        m = cls(size=size, device=device)
        m._ck(lib().q3asr_load_safetensors(m._h, os.fspath(model_dir).encode()))
        if os.path.exists(os.path.join(model_dir, "vocab.json")):  # Qwen3ASR.swift:643-649
            m.tokenizer = Qwen3Tokenizer(path=os.fspath(model_dir))
        return m

    @classmethod
    def random_init(cls, size="0.6B", seed=20260418, device=0, config=None):
        m = cls(size=size, device=device, config=config)
        m._ck(lib().q3asr_init_random(m._h, int(seed)))
        return m

    def close(self):
        if self._h:
            lib().q3asr_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != OK:
            raise Q3Error(rc, lib().q3asr_last_error(self._h).decode())

    @property
    def is_loaded(self):
        return bool(lib().q3asr_is_loaded(self._h))

    def unload(self):
        self._ck(lib().q3asr_unload(self._h))

    @property
    def memory_footprint(self):
        return int(lib().q3asr_memory_footprint(self._h))

    @property
    def launch_count(self):
        return int(lib().q3asr_launch_count(self._h))

    def decode_stats(self):
        """{steps, row_steps, compactions, rows} of the last decode loop (q3asr_decode_stats)."""
        out = np.zeros(4, dtype=np.uint64)
        self._ck(lib().q3asr_decode_stats(self._h, out.ctypes.data))
        return dict(steps=int(out[0]), row_steps=int(out[1]), compactions=int(out[2]), rows=int(out[3]))

    def decode_admissions(self):
        """{admissions, admitted} of the last continuous-batching call (q3asr_decode_admissions): groups prefilled after the first
        one, and the utterances in them."""
        out = np.zeros(2, dtype=np.uint64)
        self._ck(lib().q3asr_decode_admissions(self._h, out.ctypes.data))
        return dict(admissions=int(out[0]), admitted=int(out[1]))

    # -- weights -----------------------------------------------------------------------------
    def tensor_names(self):
        out = []
        name = ctypes.create_string_buffer(256)
        shape = (ctypes.c_int64 * 4)()
        nd = ctypes.c_int()
        for i in range(lib().q3asr_tensor_count(self._h)):
            self._ck(lib().q3asr_tensor_info(self._h, i, name, 256, shape, ctypes.byref(nd)))
            out.append((name.value.decode(), tuple(shape[j] for j in range(nd.value))))
        return out

    def get_tensor(self, name, shape):
        out = np.empty(int(np.prod(shape)), dtype=np.float32)
        self._ck(lib().q3asr_get_tensor(self._h, name.encode(), out.ctypes.data, out.size))
        return out.reshape(shape)

    def set_tensor(self, name, array):
        a = np.ascontiguousarray(array, dtype=np.float32)
        shape = (ctypes.c_int64 * a.ndim)(*a.shape)
        self._ck(lib().q3asr_set_tensor(self._h, name.encode(), a.ctypes.data, 0, shape, a.ndim))

    def commit_weights(self):
        self._ck(lib().q3asr_commit_weights(self._h))

    def state_dict(self):
        return {n: self.get_tensor(n, s) for n, s in self.tensor_names()}

    # -- stages ------------------------------------------------------------------------------
    def extract_features(self, audio):
        """WhisperFeatureExtractor.extractFeaturesRaw: float32 [n] at 16 kHz -> [128, n // 160]."""
        return self.extract_features_batch([audio])[0]

    def extract_features_batch(self, clips):
        clips = [np.ascontiguousarray(c, dtype=np.float32) for c in clips]
        n = np.array([c.size for c in clips], dtype=np.uint64)
        outs = [np.empty((128, mel_frames(c.size)), dtype=np.float32) for c in clips]
        frames = np.zeros(len(clips), dtype=np.int32)
        self._ck(lib().q3asr_mel_batch(self._h, ctypes.cast(_ptr_array(clips), ctypes.c_void_p), n.ctypes.data, len(clips),
                                       ctypes.cast(_ptr_array(outs), ctypes.c_void_p), frames.ctypes.data))
        return outs

    def encode(self, mel):
        """Qwen3AudioEncoder: mel float32 [128, T] -> [tokens, out_dim] float32."""
        mel = np.ascontiguousarray(mel, dtype=np.float32)
        T = mel.shape[1]
        out = np.empty((encoder_tokens(T) + 16, self.cfg.enc_out_dim), dtype=np.float32)
        ntok = ctypes.c_int()
        self._ck(lib().q3asr_encode(self._h, mel.ctypes.data, T, out.ctypes.data, ctypes.byref(ntok)))
        return out[:ntok.value].copy()

    def transcribe_ids(self, clips, max_tokens=448, stop_on_eos=True, prompts=None, sample_rates=None, options=None,
                       force_device_sampler=False, return_logprobs=False, continuous_rows=None):
        """Batched transcription -> list of int32 id arrays (EOS included when it stops the loop).  sample_rates: per-clip
        rates; clips not at 16 kHz are converted on the device (AudioPreprocessing.swift:323-337).  options: a
        Qwen3DecodingOptions whose decoder knobs (repetition penalty, no-repeat n-gram, temperature) run as a device kernel.
        return_logprobs: (ids, logprobs) lists instead, logprobs[i] the float32 log-probability of every id (q3asr_transcribe_ids_lp).
        continuous_rows: continuous batching (q3asr_transcribe_ids_continuous) — the request runs as one resident decode batch of at
        most that many rows (0: 256), refilled with the waiting clips as rows finish; the same ids, greedy only."""
        clips = [np.ascontiguousarray(c, dtype=np.float32) for c in clips]
        n = np.array([c.size for c in clips], dtype=np.uint64)
        ids = np.zeros((len(clips), max_tokens), dtype=np.int32)
        lens = np.zeros(len(clips), dtype=np.int32)
        pp = _PromptPack(prompts, len(clips))
        if continuous_rows is not None:
            if options is not None:
                raise ValueError("continuous_rows: greedy decoding only (no decoder options)")
            sr = None if sample_rates is None else np.ascontiguousarray(sample_rates, dtype=np.int32)
            lp = np.zeros((len(clips), max_tokens), dtype=np.float32) if return_logprobs else None
            self._ck(lib().q3asr_transcribe_ids_continuous(self._h, ctypes.cast(_ptr_array(clips), ctypes.c_void_p), n.ctypes.data,
                                                           sr.ctypes.data if sr is not None else None, len(clips), pp.ptr, int(max_tokens),
                                                           int(bool(stop_on_eos)), int(continuous_rows), ids.ctypes.data, lens.ctypes.data,
                                                           lp.ctypes.data if lp is not None else None))
            out = [ids[i, :lens[i]].copy() for i in range(len(clips))]
            return (out, [lp[i, :lens[i]].copy() for i in range(len(clips))]) if return_logprobs else out
        if return_logprobs:
            lp = np.zeros((len(clips), max_tokens), dtype=np.float32)
            sr = None if sample_rates is None else np.ascontiguousarray(sample_rates, dtype=np.int32)
            samp = None if options is None else options.c_struct(force_device_sampler)
            self._ck(lib().q3asr_transcribe_ids_lp(self._h, ctypes.cast(_ptr_array(clips), ctypes.c_void_p), n.ctypes.data,
                                                   sr.ctypes.data if sr is not None else None, len(clips), pp.ptr,
                                                   ctypes.byref(samp) if samp is not None else None, int(max_tokens),
                                                   int(bool(stop_on_eos)), ids.ctypes.data, lens.ctypes.data, lp.ctypes.data))
            return ([ids[i, :lens[i]].copy() for i in range(len(clips))], [lp[i, :lens[i]].copy() for i in range(len(clips))])
        if options is not None:
            sr = None if sample_rates is None else np.ascontiguousarray(sample_rates, dtype=np.int32)
            samp = options.c_struct(force_device_sampler)
            self._ck(lib().q3asr_transcribe_ids_opts(self._h, ctypes.cast(_ptr_array(clips), ctypes.c_void_p), n.ctypes.data,
                                                     sr.ctypes.data if sr is not None else None, len(clips), pp.ptr, ctypes.byref(samp),
                                                     int(max_tokens), int(bool(stop_on_eos)), ids.ctypes.data, lens.ctypes.data))
        elif sample_rates is None:
            self._ck(lib().q3asr_transcribe_ids(self._h, ctypes.cast(_ptr_array(clips), ctypes.c_void_p), n.ctypes.data, len(clips), pp.ptr,
                                                int(max_tokens), int(bool(stop_on_eos)), ids.ctypes.data, lens.ctypes.data))
        else:
            sr = np.ascontiguousarray(sample_rates, dtype=np.int32)
            assert sr.size == len(clips)
            self._ck(lib().q3asr_transcribe_ids_sr(self._h, ctypes.cast(_ptr_array(clips), ctypes.c_void_p), n.ctypes.data, sr.ctypes.data,
                                                   len(clips), pp.ptr, int(max_tokens), int(bool(stop_on_eos)), ids.ctypes.data,
                                                   lens.ctypes.data))
        return [ids[i, :lens[i]].copy() for i in range(len(clips))]

    def pick_next_token(self, logits, generated_so_far, options, draw=0):
        """Qwen3ASRModel.pickNextToken (Qwen3ASR.swift:449-520) through the device kernel, on caller-provided logits."""
        lg = np.ascontiguousarray(logits, dtype=np.float32).reshape(-1)
        gen = np.ascontiguousarray(generated_so_far, dtype=np.int32).reshape(-1)
        samp = options.c_struct(True)
        tok = ctypes.c_int32()
        self._ck(lib().q3asr_pick_next_token(self._h, lg.ctypes.data, lg.size, gen.ctypes.data if gen.size else None, gen.size,
                                             ctypes.byref(samp), int(draw), ctypes.byref(tok)))
        return int(tok.value)

    TIMESTAMP_SEGMENT_TIME = 0.08  # Configuration.swift:133

    def align_indices(self, clips, slotted_ids, positions, sample_rates=None):
        """Qwen3ForcedAligner.align, steps 1-7 (ForcedAligner.swift:226-299), batched: one prefill per clip over the aligner template
        ending in slotted_ids[i]; the classification head's argmax at positions[i] (indices into slotted_ids[i])."""
        clips = [np.ascontiguousarray(c, dtype=np.float32) for c in clips]
        B = len(clips)
        n = np.array([c.size for c in clips], dtype=np.uint64)
        sl = [np.ascontiguousarray(x, dtype=np.int32) for x in slotted_ids]
        ps = [np.ascontiguousarray(x, dtype=np.int32) for x in positions]
        outs = [np.zeros(max(p.size, 1), dtype=np.int32) for p in ps]
        nsl = np.array([x.size for x in sl], dtype=np.int32)
        nps = np.array([x.size for x in ps], dtype=np.int32)
        sr = None if sample_rates is None else np.ascontiguousarray(sample_rates, dtype=np.int32)
        self._ck(lib().q3asr_align_indices(self._h, ctypes.cast(_ptr_array(clips), ctypes.c_void_p), n.ctypes.data,
                                           sr.ctypes.data if sr is not None else None, B, ctypes.cast(_ptr_array(sl), ctypes.c_void_p),
                                           nsl.ctypes.data, ctypes.cast(_ptr_array(ps), ctypes.c_void_p), nps.ctypes.data,
                                           ctypes.cast(_ptr_array(outs), ctypes.c_void_p)))
        return [o[:p.size].copy() for o, p in zip(outs, ps)]

    def align(self, audio, word_token_ids, words=None, sample_rate=16000):
        """Qwen3ForcedAligner.align for text already split into words and tokenised (the reference's word splitter needs Apple's
        NaturalLanguage framework, TextPreprocessing.swift:2): <|timestamp|> slots around every word (TextPreprocessing.swift:48-80),
        argmax classes, LIS fix-up, 0.08 s per class, end >= start (ForcedAligner.swift:301-330).
        Returns [dict(text, start_time, end_time)]."""
        ts = int(self.cfg.tok_timestamp)
        ids, pos = [], []
        for w in word_token_ids:
            pos.append(len(ids)); ids.append(ts)
            ids.extend(int(t) for t in w)
            pos.append(len(ids)); ids.append(ts)
        raw = self.align_indices([audio], [ids], [pos], None if sample_rate == 16000 else [sample_rate])[0]
        fixed = enforce_monotonicity(raw)
        out = []
        for i in range(len(word_token_ids)):
            st = np.float32(fixed[2 * i]) * np.float32(self.TIMESTAMP_SEGMENT_TIME)
            en = np.float32(fixed[2 * i + 1]) * np.float32(self.TIMESTAMP_SEGMENT_TIME)
            out.append(dict(text=words[i] if words else "", start_time=float(st), end_time=float(max(en, st))))
        return out

    def align_text(self, audio, text, language="English", sample_rate=16000):
        """Qwen3ForcedAligner.align(audio:text:sampleRate:language:) (ForcedAligner.swift:226-331): word splitting and timestamp slots
        by q3asr.text (TextPreprocessing.swift), the rest by `align`.  [] without a tokenizer or without words, like the reference."""
        from . import text as _text
        if self.tokenizer is None:
            return []
        st = _text.prepare_for_alignment(text, self.tokenizer, language, int(self.cfg.tok_timestamp))
        if not st.words:
            return []
        raw = self.align_indices([audio], [st.token_ids], [st.timestamp_positions], None if sample_rate == 16000 else [sample_rate])[0]
        fixed = enforce_monotonicity(raw)
        seg = np.float32(self.TIMESTAMP_SEGMENT_TIME)
        out = []
        for i, w in enumerate(st.words):
            a, b = np.float32(fixed[2 * i]) * seg, np.float32(fixed[2 * i + 1]) * seg
            out.append(dict(text=w, start_time=float(a), end_time=float(max(a, b))))
        return out

    @staticmethod
    def offset_words(words, seconds):
        """Qwen3ForcedAligner.offsetWords (ForcedAligner.swift:183-188), float32 arithmetic like the reference's Float."""
        if seconds == 0:
            return words
        sec = np.float32(seconds)
        return [dict(text=w["text"], start_time=float(np.float32(w["start_time"]) + sec), end_time=float(np.float32(w["end_time"]) + sec))
                for w in words]

    def align_long(self, audio, text, language="English", sample_rate=16000, progress=None):
        """Qwen3ForcedAligner.alignLong (ForcedAligner.swift:100-181): align everything, find the trailing plateau (the words the
        monotonicity pass collapsed onto one timestamp once the classification head saturates), keep the reliable prefix, re-align the
        remaining audio and words, offset.  One `align_text` pass for recordings up to 240 s."""
        bypass_s, min_chunk_s, tol, min_words = np.float32(240.0), np.float32(5.0), 0.1, 5
        x = np.ascontiguousarray(audio, dtype=np.float32)
        out, rem_text, offset, npass = [], text, np.float32(0.0), 1
        while x.size and rem_text:
            duration = np.float32(x.size) / np.float32(sample_rate)
            aligned = self.align_text(x, rem_text, language, sample_rate)
            if not aligned:
                break
            if duration <= bypass_s or len(aligned) < 2 * min_words:
                out += self.offset_words(aligned, offset)
                break
            plateau = trailing_plateau_start([w["start_time"] for w in aligned], tol, min_words)
            if plateau == len(aligned):
                out += self.offset_words(aligned, offset)
                break
            if plateau == 0:  # the reference force-unwraps the last reliable word here; nothing reliable means nothing to keep
                break
            split_time = np.float32(aligned[plateau - 1]["end_time"])
            out += self.offset_words(aligned[:plateau], offset)
            split_sample = int(split_time * np.float32(sample_rate))
            if split_sample >= x.size:
                break
            nxt = x[split_sample:]
            remaining = np.float32(nxt.size) / np.float32(sample_rate)
            if remaining < min_chunk_s:
                break
            words_all = [w for w in rem_text.split(" ") if w]  # the reference splits on the space character only (:161)
            if plateau >= len(words_all):
                break
            if progress is not None:
                progress(f"Audio {duration:.1f}s saturated after word {plateau} ({split_time:.1f}s); chunking remaining "
                         f"{remaining:.1f}s (pass {npass + 1})")
            x, rem_text = nxt, " ".join(words_all[plateau:])
            offset = np.float32(offset + split_time)
            npass += 1
            if npass > 10:
                break
        return out

    def resample(self, samples, in_rate, out_rate):
        """AudioFileLoader.resample (AudioFileLoader.swift:159-213) on the GPU: float32 [n] -> float32 [floor(n * out / in)]."""
        x = np.ascontiguousarray(samples, dtype=np.float32)
        out = np.empty(AudioFileLoader.resample_len(x.size, in_rate, out_rate), dtype=np.float32)
        n_out = ctypes.c_size_t()
        self._ck(lib().q3asr_resample(self._h, x.ctypes.data, x.size, int(in_rate), int(out_rate), out.ctypes.data, out.size,
                                      ctypes.byref(n_out)))
        return out[:n_out.value]

    def _text_of(self, ids):
        tok = self.tokenizer
        if tok is None:
            return " ".join(str(int(t)) for t in ids)
        raw = tok.decode([int(t) for t in ids])
        # trimmingCharacters(in: .whitespaces) (Qwen3ASR.swift:286): Unicode space separators and TAB, not line breaks
        return raw.split("<asr_text>", 1)[1].strip(_SWIFT_WHITESPACES) if "<asr_text>" in raw else raw

    def transcribe_long(self, audio, sample_rate=16000, window_seconds=30.0, max_tokens=448, batch=64, language_ids=None, context_ids=None):
        """Long-form transcription (BASELINE config 5): fixed windows, each an independent utterance, `batch` windows per pass.
        Returns [dict(text, ids, start_time, end_time, segment_index)] in the shape of the reference's TranscriptionSegment
        (StreamingASR.swift:7-21); " ".join of the texts is the transcript."""
        x = np.ascontiguousarray(audio, dtype=np.float32)
        wins = longform_plan(x.size, int(round(window_seconds * sample_rate)), min_tail=max(160, (160 * sample_rate + 15999) // 16000))
        segs = []
        for b0 in range(0, len(wins), batch):
            part = wins[b0:b0 + batch]
            clips = [x[s:s + ln] for s, ln in part]
            pr = [{"context": context_ids, "language": language_ids}] * len(part)
            out = self.transcribe_ids(clips, max_tokens=max_tokens, stop_on_eos=True, prompts=pr,
                                      sample_rates=None if sample_rate == 16000 else [sample_rate] * len(part))
            for (s, ln), ids in zip(part, out):
                segs.append(dict(text=self._text_of(ids), ids=ids, start_time=s / sample_rate, end_time=(s + ln) / sample_rate,
                                 segment_index=len(segs)))
        return segs

    tokenizer = None  # a Qwen3Tokenizer; set by from_pretrained when the checkpoint directory has a vocab.json

    def transcribe(self, audio, sample_rate=16000, language=None, max_tokens=448, context=None, language_ids=None, context_ids=None,
                   options=None):
        """Qwen3ASRModel.transcribe(audio:sampleRate:language:maxTokens:context:) (Qwen3ASR.swift:131-164, 181-289): with a tokenizer
        the text after "<asr_text>", else the ids joined by spaces (the reference's own fallback)."""
        tok = self.tokenizer
        if options is not None:  # transcribe(audio:sampleRate:options:), Qwen3ASR.swift:107-111
            language, context, max_tokens = options.language, options.context, options.max_tokens
        if tok is not None:
            if context is not None and context_ids is None:
                context_ids = tok.encode(context)                    # Qwen3ASR.swift:203-206
            if language is not None and language_ids is None:
                language_ids = tok.encode("language " + language)    # Qwen3ASR.swift:228-232
        pr = [{"context": context_ids, "language": language_ids}]
        ids = self.transcribe_ids([audio], max_tokens=max_tokens, stop_on_eos=True, prompts=pr,
                                  sample_rates=None if sample_rate == 16000 else [sample_rate],
                                  options=None if options is None or options.is_greedy_fast_path else options)[0]
        return self._text_of(ids)

    def decode_forced(self, audio, forced, prompt=None):
        audio = np.ascontiguousarray(audio, dtype=np.float32)
        forced = np.ascontiguousarray(forced, dtype=np.int32)
        am = np.zeros(forced.size + 1, dtype=np.int32)
        top = np.zeros(forced.size + 1, dtype=np.float32)
        pp = _PromptPack([prompt] if prompt else None, 1)
        self._ck(lib().q3asr_decode_forced(self._h, audio.ctypes.data, audio.size, pp.ptr, forced.ctypes.data, forced.size,
                                           am.ctypes.data, top.ctypes.data))
        return am, top

    def decode_forced_embeds(self, audio, audio_embeds, forced, prompt=None):
        """decode_forced with the encoder's output replaced by audio_embeds [tokens, enc_out_dim] (parity hook: isolates the decoder)."""
        audio = np.ascontiguousarray(audio, dtype=np.float32)
        emb = np.ascontiguousarray(audio_embeds, dtype=np.float32)
        forced = np.ascontiguousarray(forced, dtype=np.int32)
        am = np.zeros(forced.size + 1, dtype=np.int32)
        top = np.zeros(forced.size + 1, dtype=np.float32)
        pp = _PromptPack([prompt] if prompt else None, 1)
        self._ck(lib().q3asr_decode_forced_embeds(self._h, audio.ctypes.data, audio.size, pp.ptr, emb.ctypes.data, emb.shape[0],
                                                  forced.ctypes.data, forced.size, am.ctypes.data, top.ctypes.data))
        return am, top

    def prefill_logits(self, audio, prompt=None):
        audio = np.ascontiguousarray(audio, dtype=np.float32)
        out = np.empty(self.cfg.dec_vocab, dtype=np.float32)
        pp = _PromptPack([prompt] if prompt else None, 1)
        self._ck(lib().q3asr_prefill_logits(self._h, audio.ctypes.data, audio.size, pp.ptr, out.ctypes.data))
        return out

    # -- resident batch (benchmarks) -----------------------------------------------------------
    def batch_upload(self, clips, prompts=None):
        self._clips = [np.ascontiguousarray(c, dtype=np.float32) for c in clips]
        n = np.array([c.size for c in self._clips], dtype=np.uint64)
        pp = _PromptPack(prompts, len(self._clips))
        self._ck(lib().q3asr_batch_upload(self._h, ctypes.cast(_ptr_array(self._clips), ctypes.c_void_p), n.ctypes.data,
                                          len(self._clips), pp.ptr))

    def batch_run(self, stages=STAGE_ALL, max_tokens=128, stop_on_eos=False):
        self._ck(lib().q3asr_batch_run(self._h, int(stages), int(max_tokens), int(bool(stop_on_eos))))

    def batch_set_logprobs(self, enable=True):
        self._ck(lib().q3asr_batch_set_logprobs(self._h, int(bool(enable))))

    def batch_download_logprobs(self, batch, max_tokens):
        """[batch, max_tokens] float32, zeros past each utterance's length"""
        lp = np.zeros((batch, max(max_tokens, 1)), dtype=np.float32)
        self._ck(lib().q3asr_batch_download_logprobs(self._h, lp.ctypes.data, int(max_tokens)))
        return lp[:, :max_tokens]

    def batch_download(self, batch, max_tokens):
        ids = np.zeros((batch, max(max_tokens, 1)), dtype=np.int32)
        lens = np.zeros(batch, dtype=np.int32)
        self._ck(lib().q3asr_batch_download(self._h, ids.ctypes.data, int(max_tokens), lens.ctypes.data))
        return [ids[i, :lens[i]].copy() for i in range(batch)]

    def sync(self):
        self._ck(lib().q3asr_sync(self._h))

    def timer_record(self, slot):
        self._ck(lib().q3asr_timer_record(self._h, slot))

    def timer_ms(self, a, b):
        ms = ctypes.c_float()
        self._ck(lib().q3asr_timer_elapsed_ms(self._h, a, b, ctypes.byref(ms)))
        return float(ms.value)

    def stage_ms(self):
        out = np.zeros(4, dtype=np.float32)
        self._ck(lib().q3asr_stage_ms(self._h, out.ctypes.data))
        return out

    def profile(self, enable=True):
        self._ck(lib().q3asr_profile(self._h, int(bool(enable))))

    def profile_report(self):
        """{tag: dict(launches, ms, flops, bytes)} for the launches since profiling was enabled / last read."""
        buf = ctypes.create_string_buffer(1 << 16)
        self._ck(lib().q3asr_profile_report(self._h, buf, len(buf)))
        out = {}
        for line in buf.value.decode().splitlines():
            tag, n, ms, fl, by = line.split(",")
            out[tag] = dict(launches=int(n), ms=float(ms), flops=float(fl), bytes=float(by))
        return out

    def flush_l2(self):
        self._ck(lib().q3asr_flush_l2(self._h))

    # -- debug hooks -----------------------------------------------------------------------------
    def debug_gemm(self, A, W, bias=None, resid=None, epi=EPI_NORMAL, gelu=False, bn=0, simt=False):
        """A [M,K], W [N,K] float32 holding bf16-representable values."""
        M, K = A.shape
        N = W.shape[0]
        a, w = f32_to_bf16_bits(A), f32_to_bf16_bits(W)
        b = f32_to_bf16_bits(bias) if bias is not None else None
        r = f32_to_bf16_bits(resid) if resid is not None else None
        if epi in (EPI_F32, EPI_SKINNY_PARTIAL):
            out = np.empty((M, N), dtype=np.float32)
        elif epi in (EPI_ARGMAX, 7):  # 7: the decode-step LM-head kernel (lmhead.cuh)
            out = np.empty(M, dtype=np.int32)
        elif epi in (8, 9):  # 8 / 9: the LM-head kernel / EPI_ARGMAX with the log-sum-exp: ids [M], then float32 logprobs [M]
            out = np.empty(2 * M, dtype=np.int32)
        elif epi == EPI_SWIGLU:
            out = np.empty((M, N // 2), dtype=np.uint16)
        else:
            out = np.empty((M, N), dtype=np.uint16)
        self._ck(lib().q3asr_debug_gemm(self._h, a.ctypes.data, w.ctypes.data, b.ctypes.data if b is not None else None,
                                        r.ctypes.data if r is not None else None, M, N, K, int(epi), int(bool(gelu)), int(bn),
                                        int(bool(simt)), out.ctypes.data))
        if epi in (8, 9):
            return out[:M].copy(), out[M:].view(np.float32).copy()
        return bf16_bits_to_f32(out) if out.dtype == np.uint16 else out

    def debug_attention(self, q, k, v, segs, heads, group, causal, scale, kernel=0):
        """q [rows, heads*hd], k/v [rows, heads/group*hd] float32 holding bf16 values; segs: list of (row0, len)."""
        rows = q.shape[0]
        hd = q.shape[1] // heads
        qb, kb, vb = f32_to_bf16_bits(q), f32_to_bf16_bits(k), f32_to_bf16_bits(v)
        r0 = np.ascontiguousarray([s[0] for s in segs], dtype=np.int32)
        ln = np.ascontiguousarray([s[1] for s in segs], dtype=np.int32)
        out = np.empty((rows, heads * hd), dtype=np.uint16)
        self._ck(lib().q3asr_debug_attention(self._h, qb.ctypes.data, kb.ctypes.data, vb.ctypes.data, rows, heads, group, hd,
                                             r0.ctypes.data, ln.ctypes.data, len(segs), int(bool(causal)), ctypes.c_float(scale),
                                             int(kernel), out.ctypes.data))
        return bf16_bits_to_f32(out)

    def debug_decode_attention(self, qkv_part, heads, kv_heads, q_norm, k_norm, kv_len, page_table, pool, layer, variant=0, launches=1,
                               eps=1e-6, scale=None):
        """One layer's decode-step attention (q3asr_debug_decode_attention).  qkv_part float32 [splits, n_seqs, (heads + 2*kv_heads)*128];
        q_norm / k_norm float32 [128] holding bf16 values; kv_len [n_seqs] (new token included); page_table [n_seqs, max_pages];
        pool uint16 (bf16 bits) [n_pages, layers, 2, kv_heads, 32, 128].  Returns (out float32 [launches, n_seqs, heads*128],
        the pool after the calls, uint16)."""
        part = np.ascontiguousarray(qkv_part, dtype=np.float32)
        splits, n_seqs, nqkv = part.shape
        assert nqkv == (heads + 2 * kv_heads) * 128
        qw, kw = f32_to_bf16_bits(np.asarray(q_norm, np.float32)), f32_to_bf16_bits(np.asarray(k_norm, np.float32))
        lens = np.ascontiguousarray(kv_len, dtype=np.int32)
        pt = np.ascontiguousarray(page_table, dtype=np.int32)
        pool = np.array(pool, dtype=np.uint16, order="C")  # a copy: the call writes the appended k / v into it
        n_pages, layers = pool.shape[0], pool.shape[1]
        assert pool.shape[2:] == (2, kv_heads, 32, 128) and pt.shape[0] == n_seqs and lens.shape == (n_seqs,)
        if scale is None:
            scale = 1.0 / np.sqrt(128.0)
        out = np.empty((launches, n_seqs, heads * 128), dtype=np.uint16)
        self._ck(lib().q3asr_debug_decode_attention(self._h, part.ctypes.data, splits, n_seqs, heads, kv_heads, qw.ctypes.data, kw.ctypes.data,
                                                    ctypes.c_float(eps), ctypes.c_float(scale), lens.ctypes.data, pt.ctypes.data, pt.shape[1],
                                                    pool.ctypes.data, n_pages, layers, int(layer), int(variant), int(launches),
                                                    out.ctypes.data))
        return bf16_bits_to_f32(out), pool

    def debug_prefill_attention(self, x, w, heads, kv_heads, q_norm, k_norm, segs, seg_table_rows, page_table, pool, layer, qkv_variant=0,
                                bn=0, attn_variant=0, eps=1e-6, scale=None):
        """One decoder layer's prefill attention block (q3asr_debug_prefill_attention).  x [rows, hidden], w [(heads + 2*kv_heads)*128,
        hidden], q_norm / k_norm [128]: float32 holding bf16 values; segs: (row0, len) packed back to back; seg_table_rows: the
        page-table row of every segment; page_table [table_rows, max_pages]; pool uint16 (bf16 bits) [n_pages, layers, 2, kv_heads,
        32, 128].  Returns (q, k, qkv, att) float32 (NaN where the call wrote nothing) and the pool after the call, uint16."""
        xb, wb = f32_to_bf16_bits(np.asarray(x, np.float32)), f32_to_bf16_bits(np.asarray(w, np.float32))
        rows, hidden = xb.shape
        nq, nkv = heads * 128, kv_heads * 128
        assert wb.shape == (nq + 2 * nkv, hidden)
        qw, kw = f32_to_bf16_bits(np.asarray(q_norm, np.float32)), f32_to_bf16_bits(np.asarray(k_norm, np.float32))
        r0 = np.ascontiguousarray([s[0] for s in segs], dtype=np.int32)
        ln = np.ascontiguousarray([s[1] for s in segs], dtype=np.int32)
        tr = np.ascontiguousarray(seg_table_rows, dtype=np.int32)
        pt = np.ascontiguousarray(page_table, dtype=np.int32)
        pool = np.array(pool, dtype=np.uint16, order="C")  # a copy: the call writes k and v into it
        n_pages, layers = pool.shape[0], pool.shape[1]
        assert pool.shape[2:] == (2, kv_heads, 32, 128) and pt.ndim == 2 and tr.shape == r0.shape
        if scale is None:
            scale = 1.0 / np.sqrt(128.0)
        q = np.empty((rows, nq), dtype=np.uint16)
        k = np.empty((rows, nkv), dtype=np.uint16)
        qkv = np.empty((rows, nq + 2 * nkv), dtype=np.uint16)
        att = np.empty((rows, nq), dtype=np.uint16)
        self._ck(lib().q3asr_debug_prefill_attention(self._h, xb.ctypes.data, wb.ctypes.data, rows, hidden, heads, kv_heads, qw.ctypes.data,
                                                     kw.ctypes.data, ctypes.c_float(eps), ctypes.c_float(scale), r0.ctypes.data, ln.ctypes.data,
                                                     tr.ctypes.data, len(r0), pt.ctypes.data, pt.shape[0], pt.shape[1], pool.ctypes.data,
                                                     n_pages, layers, int(layer), int(qkv_variant), int(bn), int(attn_variant), q.ctypes.data,
                                                     k.ctypes.data, qkv.ctypes.data, att.ctypes.data))
        return bf16_bits_to_f32(q), bf16_bits_to_f32(k), bf16_bits_to_f32(qkv), bf16_bits_to_f32(att), pool

    def debug_conv(self, x, w, bias, box=(0, 0, 0), simt=False):
        """x [B,H,W,C], w [O,3,3,C] float32 (bf16-representable) -> gelu(conv3x3 s2 p1 + bias) [B,OH,OW,O]."""
        B, H, Wd, C = x.shape
        O = w.shape[0]
        OH, OW = (H - 1) // 2 + 1, (Wd - 1) // 2 + 1
        bw, bh, bb = box
        if bw == 0:
            bw, bh, bb = OW, 1, max(1, 128 // OW)
        out = np.empty((B, OH, OW, O), dtype=np.uint16)
        xb, wb, bbias = f32_to_bf16_bits(x), f32_to_bf16_bits(w), f32_to_bf16_bits(bias)
        self._ck(lib().q3asr_debug_conv(self._h, xb.ctypes.data, wb.ctypes.data, bbias.ctypes.data, B, H, Wd, C, O, bw, bh, bb,
                                        int(bool(simt)), out.ctypes.data))
        return bf16_bits_to_f32(out)


class Qwen3Tokenizer:
    """Mirror of the reference's Qwen3Tokenizer (Sources/AudioCommon/Tokenizer.swift) over q3asr_tokenizer_*."""

    def __init__(self, path=None, id_to_token=None, merges=()):
        self._t = ctypes.c_void_p()
        if path is not None:
            rc = lib().q3asr_tokenizer_load(os.fsencode(path), ctypes.byref(self._t))
            if rc != OK:
                msg = lib().q3asr_tokenizer_last_error(self._t).decode("utf-8", "replace")
                lib().q3asr_tokenizer_destroy(self._t)
                self._t = ctypes.c_void_p()
                raise Q3Error(rc, msg)
        else:
            items = sorted((id_to_token or {}).items())
            ids = np.ascontiguousarray([k for k, _ in items], dtype=np.int32)
            toks = (ctypes.c_char_p * len(items))(*[v.encode("utf-8") for _, v in items])
            rc = lib().q3asr_tokenizer_from_pairs(ids.ctypes.data, ctypes.cast(toks, ctypes.c_void_p), len(items), ctypes.byref(self._t))
            if rc != OK:
                raise Q3Error(rc, "tokenizer_from_pairs failed")
        for a, b in merges:
            lib().q3asr_tokenizer_add_merge(self._t, a.encode("utf-8"), b.encode("utf-8"))

    def close(self):
        if self._t:
            lib().q3asr_tokenizer_destroy(self._t)
            self._t = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def size(self):
        a, b = ctypes.c_int(), ctypes.c_int()
        lib().q3asr_tokenizer_size(self._t, ctypes.byref(a), ctypes.byref(b))
        return a.value, b.value

    def decode(self, tokens):
        ids = np.ascontiguousarray(tokens, dtype=np.int32)
        need = ctypes.c_size_t()
        lib().q3asr_tokenizer_decode(self._t, ids.ctypes.data, ids.size, None, 0, ctypes.byref(need))
        buf = ctypes.create_string_buffer(need.value)
        rc = lib().q3asr_tokenizer_decode(self._t, ids.ctypes.data, ids.size, buf, need.value, None)
        if rc != OK:
            raise Q3Error(rc, "tokenizer decode failed")
        return buf.value.decode("utf-8")

    def encode(self, text):
        n = ctypes.c_int()
        raw = text.encode("utf-8")
        lib().q3asr_tokenizer_encode(self._t, raw, None, 0, ctypes.byref(n))
        out = np.zeros(max(n.value, 1), dtype=np.int32)
        rc = lib().q3asr_tokenizer_encode(self._t, raw, out.ctypes.data, out.size, ctypes.byref(n))
        if rc != OK:
            raise Q3Error(rc, "tokenizer encode failed")
        return out[:n.value].tolist()

    def token_id(self, token):
        v = lib().q3asr_tokenizer_token_id(self._t, token.encode("utf-8"))
        return None if v < 0 else v


class Pool:
    """Utterance-batching scheduler over several GPUs of one process (q3asr_pool_*)."""

    def __init__(self, size="0.6B", devices=(0,), seed=20260418, weights_dir=None, config=None, continuous=False):
        """continuous: each worker runs its whole share as one continuous batch of max_batch_per_gpu rows
        (q3asr_pool_set_continuous); greedy decoding only."""
        self.cfg = config if config is not None else preset(size)
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        self._p = ctypes.c_void_p()
        rc = lib().q3asr_pool_create(ctypes.byref(self.cfg), dev.ctypes.data, dev.size, int(seed),
                                     os.fspath(weights_dir).encode() if weights_dir else None, ctypes.byref(self._p))
        if rc != OK:
            raise Q3Error(rc, "pool_create failed: " + lib().q3asr_pool_last_error(None).decode())
        if continuous:
            rc = lib().q3asr_pool_set_continuous(self._p, 1)
            if rc != OK:
                self.close()
                raise Q3Error(rc, "pool_set_continuous failed")

    def transcribe_ids(self, clips, max_tokens=448, stop_on_eos=True, max_batch_per_gpu=64, sample_rates=None, options=None,
                       return_logprobs=False):
        clips = [np.ascontiguousarray(c, dtype=np.float32) for c in clips]
        n = np.array([c.size for c in clips], dtype=np.uint64)
        ids = np.zeros((len(clips), max_tokens), dtype=np.int32)
        lens = np.zeros(len(clips), dtype=np.int32)
        sr = None if sample_rates is None else np.ascontiguousarray(sample_rates, dtype=np.int32)
        samp = None if options is None else options.c_struct()
        args = (self._p, ctypes.cast(_ptr_array(clips), ctypes.c_void_p), n.ctypes.data, sr.ctypes.data if sr is not None else None, len(clips),
                None, ctypes.byref(samp) if samp is not None else None, int(max_tokens), int(bool(stop_on_eos)), int(max_batch_per_gpu),
                ids.ctypes.data, lens.ctypes.data)
        if return_logprobs:
            lp = np.zeros((len(clips), max_tokens), dtype=np.float32)
            rc = lib().q3asr_pool_transcribe_ids_lp(*args, lp.ctypes.data)
        else:
            rc = lib().q3asr_pool_transcribe_ids_opts(*args)
        if rc != OK:
            raise Q3Error(rc, lib().q3asr_pool_last_error(self._p).decode())
        out = [ids[i, :lens[i]].copy() for i in range(len(clips))]
        return (out, [lp[i, :lens[i]].copy() for i in range(len(clips))]) if return_logprobs else out

    def submit(self, clips, max_tokens=448, stop_on_eos=True, max_batch_per_gpu=64, sample_rates=None, options=None, return_logprobs=False):
        """Asynchronous transcribe_ids: returns a PoolJob whose wait() gives the ids (and log-probabilities with return_logprobs);
        the clips are kept alive by the job."""
        return PoolJob(self, clips, max_tokens, stop_on_eos, max_batch_per_gpu, sample_rates, options, return_logprobs)

    def close(self):
        if self._p:
            lib().q3asr_pool_destroy(self._p)
            self._p = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PoolJob:
    """q3asr_pool_submit / q3asr_job_wait: a batch running on the library's own thread."""

    def __init__(self, pool, clips, max_tokens, stop_on_eos, max_batch_per_gpu, sample_rates, options, return_logprobs=False):
        self._clips = [np.ascontiguousarray(c, dtype=np.float32) for c in clips]
        self._n = np.array([c.size for c in self._clips], dtype=np.uint64)
        self._sr = None if sample_rates is None else np.ascontiguousarray(sample_rates, dtype=np.int32)
        self._samp = None if options is None else options.c_struct()
        self._max_tokens = int(max_tokens)
        self._lp = bool(return_logprobs)
        self._j = ctypes.c_void_p()
        submit = lib().q3asr_pool_submit_lp if self._lp else lib().q3asr_pool_submit
        rc = submit(pool._p, ctypes.cast(_ptr_array(self._clips), ctypes.c_void_p), self._n.ctypes.data,
                                     self._sr.ctypes.data if self._sr is not None else None, len(self._clips), None,
                                     ctypes.byref(self._samp) if self._samp is not None else None, self._max_tokens, int(bool(stop_on_eos)),
                                     int(max_batch_per_gpu), ctypes.byref(self._j))
        if rc != OK:
            raise Q3Error(rc, "pool_submit: bad argument")

    @property
    def done(self):
        return bool(lib().q3asr_job_done(self._j))

    def wait(self):
        ids = np.zeros((len(self._clips), self._max_tokens), dtype=np.int32)
        lens = np.zeros(len(self._clips), dtype=np.int32)
        rc = lib().q3asr_job_wait(self._j, ids.ctypes.data, lens.ctypes.data)
        if rc != OK:
            msg = lib().q3asr_job_last_error(self._j).decode()
            self.free()
            raise Q3Error(rc, msg)
        if self._lp:
            lp = np.zeros((len(self._clips), self._max_tokens), dtype=np.float32)
            rc = lib().q3asr_job_logprobs(self._j, lp.ctypes.data)
            self.free()
            if rc != OK:
                raise Q3Error(rc, "job_logprobs failed")
        self.free()
        out = [ids[i, :lens[i]].copy() for i in range(len(self._clips))]
        return (out, [lp[i, :lens[i]].copy() for i in range(len(self._clips))]) if self._lp else out

    def free(self):
        if self._j:
            lib().q3asr_job_free(self._j)
            self._j = ctypes.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
