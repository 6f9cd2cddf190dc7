"""ctypes binding of libwkb200.so (the C ABI in include/wkb200.h).

This is the binding a reference-side host would write (Swift: `@_silgen_name` / module map; here: ctypes).
Loading fails loudly when the shared library has not been built - there is no Python or CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libwkb200.so")

WK_DTYPE_F32, WK_DTYPE_F16, WK_DTYPE_BF16, WK_DTYPE_I32 = 0, 1, 2, 3

STATUS_NAMES = {
    0: "ok", -1: "invalidArgument", -2: "modelsUnavailable", -3: "audioProcessingFailed",
    -4: "prepareDecoderInputsFailed", -5: "decodingLogitsFailed", -6: "decodingFailed",
    -7: "transcriptionFailed", -8: "cudaError",
}


class WhisperError(RuntimeError):
    """Mirrors WhisperError (Sources/WhisperKit/Utilities/WhisperError.swift:6-19)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {message}")
        self.status = status
        self.case = STATUS_NAMES.get(status, str(status))


class wk_model_config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_mels", "d_model", "n_heads", "enc_layers", "dec_layers", "vocab",
                                         "n_audio_ctx", "n_text_ctx", "dtype", "max_batch")]


class wk_model_info(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_mels", "n_audio_ctx", "d_model", "n_heads", "enc_layers", "dec_layers",
                                         "vocab", "kv_embed_dim", "kv_max_len", "window_samples",
                                         "has_alignment_heads", "is_multilingual", "dtype", "max_batch")]


class wk_special_tokens(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("end_token", "english_token", "no_speech_token", "no_timestamps_token",
                                         "special_token_begin", "start_of_previous_token",
                                         "start_of_transcript_token", "time_token_begin", "transcribe_token",
                                         "translate_token", "whitespace_token")]


class wk_decode_opts(C.Structure):
    _fields_ = [
        ("task_translate", C.c_int32), ("language_token", C.c_int32), ("temperature", C.c_float),
        ("sample_length", C.c_int32), ("top_k", C.c_int32), ("use_prefill_prompt", C.c_int32),
        ("without_timestamps", C.c_int32), ("suppress_blank", C.c_int32),
        ("suppress_tokens", C.POINTER(C.c_int32)), ("n_suppress_tokens", C.c_int32),
        ("prompt_tokens", C.POINTER(C.c_int32)), ("n_prompt_tokens", C.c_int32),
        ("prefix_tokens", C.POINTER(C.c_int32)), ("n_prefix_tokens", C.c_int32),
        ("has_compression_ratio_threshold", C.c_int32), ("compression_ratio_threshold", C.c_float),
        ("has_logprob_threshold", C.c_int32), ("logprob_threshold", C.c_float),
        ("has_first_token_logprob_threshold", C.c_int32), ("first_token_logprob_threshold", C.c_float),
        ("has_no_speech_threshold", C.c_int32), ("no_speech_threshold", C.c_float),
        ("seed", C.c_uint64),
        ("temperature_fallback_count", C.c_int32), ("temperature_increment_on_fallback", C.c_float),
        ("word_timestamps", C.c_int32),
        ("beam_size", C.c_int32), ("beam_patience", C.c_float),
        ("detect_language", C.c_int32),
    ]


class wk_decode_result(C.Structure):
    _fields_ = [
        ("n_tokens", C.c_int32), ("tokens", C.c_int32 * 226), ("token_logprobs", C.c_float * 226),
        ("avg_logprob", C.c_float), ("compression_ratio", C.c_float), ("temperature", C.c_float),
        ("needs_fallback", C.c_int32), ("fallback_reason", C.c_int32), ("first_token_logprob_too_low", C.c_int32),
        ("n_current_tokens", C.c_int32), ("steps", C.c_int32),
    ]


PROGRESS_FN = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_float)


class wk_batch_opts(C.Structure):
    _fields_ = [("opts", C.POINTER(wk_decode_opts)), ("n_opts", C.c_int32),
                ("prompts", C.POINTER(C.POINTER(C.c_int32))), ("prompt_lens", C.POINTER(C.c_int32)),
                ("prompt", C.POINTER(C.c_int32)), ("n_prompt", C.c_int32),
                ("progress", PROGRESS_FN), ("progress_user", C.c_void_p), ("progress_every", C.c_int32),
                ("status", C.POINTER(C.c_int32)), ("encoder_chunk", C.c_int32)]


class wk_segment(C.Structure):
    _fields_ = [("stream", C.c_int32), ("id", C.c_int32), ("seek", C.c_int64), ("start", C.c_float), ("end", C.c_float),
                ("token_offset", C.c_int64), ("n_tokens", C.c_int32), ("temperature", C.c_float), ("avg_logprob", C.c_float),
                ("compression_ratio", C.c_float), ("no_speech_prob", C.c_float)]


class wk_word(C.Structure):
    _fields_ = [("word", C.c_char_p), ("tokens", C.POINTER(C.c_int32)), ("n_tokens", C.c_int32), ("start", C.c_float), ("end", C.c_float),
                ("probability", C.c_float), ("segment", C.c_int32)]


SPLIT_FN = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_char), C.c_int32, C.POINTER(C.c_int32), C.c_int32)
DECODE_FN = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_char), C.c_int32)


class wk_tokenizer_hooks(C.Structure):
    _fields_ = [("split_to_word_tokens", SPLIT_FN), ("decode", DECODE_FN), ("user", C.c_void_p)]


# every symbol include/wkb200.h declares: (name, restype, argtypes)
P = C.c_void_p
I32, I64, F32 = C.c_int32, C.c_int64, C.c_float
PI32, PI64, PF32 = C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_float)
SYMBOLS = [
    ("wk_last_error", C.c_char_p, []),
    ("wk_version", C.c_char_p, []),
    ("wk_device_available", I32, []),
    ("wk_default_config", None, [C.c_char_p, C.POINTER(wk_model_config)]),
    ("wk_model_create", I32, [C.POINTER(wk_model_config), I32, C.POINTER(P)]),
    ("wk_model_set_tensor", I32, [P, C.c_char_p, P, I32, PI64, I32]),
    ("wk_model_finalize", I32, [P]),
    ("wk_model_load", I32, [C.c_char_p, I32, I32, I32, C.POINTER(P)]),
    ("wk_model_init_random", I32, [P, C.c_uint64, F32]),
    ("wk_model_info_get", I32, [P, C.POINTER(wk_model_info)]),
    ("wk_model_free", None, [P]),
    ("wk_tensor_shape", I32, [P, PI64, PI32, PI32]),
    ("wk_tensor_to_host", I32, [P, P, I64]),
    ("wk_tensor_to_host_strided", I32, [P, P, I64, I64, I64, I64]),
    ("wk_tensor_free", None, [P]),
    ("wk_mel", I32, [P, P, I64, I64, PI32, C.POINTER(P)]),
    ("wk_encode", I32, [P, P, C.POINTER(P)]),
    ("wk_session_create", I32, [P, I32, C.POINTER(P)]),
    ("wk_session_free", None, [P]),
    ("wk_session_set_encoder_output", I32, [P, P]),
    ("wk_session_reset", I32, [P]),
    ("wk_build_prompt", I32, [P, C.POINTER(wk_special_tokens), C.POINTER(wk_decode_opts), I32, PI32, I32, PI32]),
    ("wk_decode_step", I32, [P, PI32, PI32, P]),
    ("wk_detect_language", I32, [P, C.POINTER(wk_special_tokens), PI32, I32, F32, PI32, PF32]),
    ("wk_filter_sample", I32, [P, C.POINTER(wk_special_tokens), C.POINTER(wk_decode_opts), I32, P, I32, I32, P, I32, P,
                               I32, I32, P, I32, I32, P, P, P]),
    ("wk_decode_text", I32, [P, C.POINTER(wk_special_tokens), C.POINTER(wk_decode_opts), PI32, I32,
                             C.POINTER(wk_decode_result)]),
    ("wk_session_last_logits", I32, [P, P]),
    ("wk_session_stats", I32, [P, PI64]),
    ("wk_session_set_language_tokens", I32, [P, PI32, I32]),
    ("wk_session_languages", I32, [P, I64, PI32, PF32]),
    ("wk_decode_text_ex", I32, [P, C.POINTER(wk_special_tokens), C.POINTER(wk_batch_opts), C.POINTER(wk_decode_result)]),
    ("wk_transcribe_windows_ex", I32, [P, P, P, I64, I64, PI32, C.POINTER(wk_special_tokens), C.POINTER(wk_batch_opts),
                                       C.POINTER(wk_decode_result)]),
    ("wk_transcribe_windows", I32, [P, P, P, I64, I64, PI32, C.POINTER(wk_special_tokens), C.POINTER(wk_decode_opts),
                                    PI32, I32, C.POINTER(wk_decode_result)]),
    ("wk_comm_shard_bounds", None, [I64, I32, I32, PI64, PI64]),
    ("wk_comm_unique_id", I32, [P]),
    ("wk_comm_create", I32, [P, I32, I32, I32, C.POINTER(P)]),
    ("wk_comm_free", None, [P]),
    ("wk_comm_scatter_windows", I32, [P, P, I64, I64, I32, P, PI64]),
    ("wk_comm_gather_results", I32, [P, C.POINTER(wk_decode_result), I64, I64, I32, C.POINTER(wk_decode_result)]),
    ("wk_transcribe_windows_sharded", I32, [P, P, P, P, I64, I64, I32, C.POINTER(wk_special_tokens), C.POINTER(wk_batch_opts),
                                            C.POINTER(wk_decode_result)]),
    ("wk_comm_last_stage_ms", I32, [P, PF32]),
    ("wk_find_seek_point_and_segments", I32, [PI32, PF32, I32, F32, F32, F32, F32, C.POINTER(wk_decode_opts), I32, I64, I64, I32, I32,
                                              PI64, C.POINTER(wk_segment), I32, PI32]),
    ("wk_prepare_seek_clips", I32, [PF32, I32, I64, PI64, I32, PI32]),
    ("wk_vad_voice_activity", I32, [P, I64, I32, I32, F32, P, I64, PI64]),
    ("wk_vad_find_longest_silence", I32, [P, I64, PI64, PI64]),
    ("wk_vad_active_chunks", I32, [P, I64, I32, I32, F32, PI64, I32, PI32]),
    ("wk_vad_chunk_all", I32, [P, I64, I64, PF32, I32, I64, I32, I32, F32, PI64, I32, PI32]),
    ("wk_transcribe_streams", I32, [P, P, C.POINTER(P), PI64, I32, C.POINTER(wk_special_tokens), C.POINTER(wk_decode_opts), PI32, I32,
                                    PF32, I32, F32, I64, I32, C.POINTER(wk_tokenizer_hooks), C.POINTER(P)]),
    ("wk_transcription_segment_count", I32, [P]),
    ("wk_transcription_window_count", I32, [P]),
    ("wk_transcription_token_count", I64, [P]),
    ("wk_transcription_segments", I32, [P, C.POINTER(wk_segment), I32]),
    ("wk_transcription_tokens", I32, [P, PI32, PF32, I64]),
    ("wk_transcription_word_count", I32, [P]),
    ("wk_transcription_word", I32, [P, I32, C.POINTER(wk_word)]),
    ("wk_transcription_language", I32, [P, I32, PI32, PF32]),
    ("wk_transcription_free", None, [P]),
    ("wk_model_set_alignment_heads", I32, [P, PI32, I32]),
    ("wk_session_alignment_weights", I32, [P, I32, I32, P]),
    ("wk_session_alignment_weights_f16", I32, [P, I32, I32, P, I32]),
    ("wk_words_count", I32, [P]),
    ("wk_words_get", I32, [P, I32, C.POINTER(wk_word)]),
    ("wk_words_free", None, [P]),
    ("wk_dtw", I32, [P, I32, I32, I32, I64, PI32, PI32, I32, PI32]),
    ("wk_find_alignment", I32, [C.POINTER(wk_word), I32, P, I32, I32, I32, I64, PF32, I32, C.POINTER(P)]),
    ("wk_merge_punctuations", I32, [C.POINTER(wk_word), I32, C.c_char_p, C.c_char_p, C.POINTER(P)]),
    ("wk_word_duration_constraints", I32, [C.POINTER(wk_word), I32, PF32, PF32]),
    ("wk_truncate_long_words", I32, [C.POINTER(wk_word), I32, F32, C.POINTER(P)]),
    ("wk_update_segments_with_word_timings", I32, [C.POINTER(wk_segment), I32, PI32, C.POINTER(wk_word), I32, I64, F32, F32, F32, I32,
                                                   C.POINTER(wk_tokenizer_hooks), C.POINTER(P)]),
    ("wk_add_word_timestamps", I32, [C.POINTER(wk_segment), I32, PI32, PF32, P, I32, I32, I32, I64, C.POINTER(wk_tokenizer_hooks), I64, F32, I32,
                                     C.c_char_p, C.c_char_p, C.POINTER(P)]),
    ("wk_detect_variant", I32, [I32, I32, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), PI32]),
    ("wk_tokenizer_load", I32, [C.c_char_p, C.POINTER(P)]),
    ("wk_tokenizer_create", I32, [C.POINTER(C.c_char_p), PI32, C.POINTER(C.c_uint8), I32, I32, C.POINTER(P)]),
    ("wk_tokenizer_free", None, [P]),
    ("wk_tokenizer_vocab_size", I32, [P]),
    ("wk_tokenizer_token_to_id", I32, [P, C.c_char_p]),
    ("wk_tokenizer_decode", I32, [P, PI32, I32, I32, C.POINTER(C.c_char), I32]),
    ("wk_tokenizer_encode", I32, [P, C.c_char_p, PI32, I32]),
    ("wk_tokenizer_set_merges", I32, [P, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), I32]),
    ("wk_tokenizer_special_tokens", I32, [P, C.POINTER(wk_special_tokens)]),
    ("wk_tokenizer_split_to_word_tokens", I32, [P, PI32, I32, C.POINTER(C.c_char), I32, PI32, I32]),
    ("wk_tokenizer_language_tokens", I32, [P, PI32, I32]),
    ("wk_tokenizer_hooks_init", I32, [P, C.POINTER(wk_tokenizer_hooks)]),
    ("wk_format_time", I32, [F32, I32, C.c_char_p, C.POINTER(C.c_char), I32]),
    ("wk_write_srt", I32, [PF32, PF32, C.POINTER(C.c_char_p), I32, C.POINTER(C.c_char), I32]),
    ("wk_write_vtt", I32, [PF32, PF32, C.POINTER(C.c_char_p), I32, C.POINTER(C.c_char), I32]),
    ("wk_kernel_launch_count", I64, [I32]),
    ("wk_last_timings", I32, [P, PF32]),
    ("wk_model_stream", P, [P]),
    ("wk_test_gemm", I32, [P, P, P, P, P, I32, I32, I32, I32, I32, I32]),
    ("wk_test_cross_attention", I32, [P, P, P, P, P, I32, I32, I32, I32, P]),
    ("wk_test_cross_attention_shared", I32, [P, P, P, P, P, I32, I32, I32, I32, P, I32]),
    ("wk_test_self_attention", I32, [P, P, P, P, P, P, I32, I32, I32, P]),
    ("wk_test_gemm_residual", I32, [P, P, P, P, P, I32, I32, I32, I32]),
    ("wk_test_gemm_splitk", I32, [P, P, P, P, I32, I32, I32, I32, I32]),
    ("wk_test_attention", I32, [P, P, P, I32, I32, I32, I32]),
    ("wk_debug_read", I32, [P, P, I32, I64, P, I64]),
    ("wk_bench_kernel", I32, [P, P, I32, I32, I32, PF32, C.POINTER(C.c_double)]),
]

_lib = None


def load() -> C.CDLL:
    """dlopen libwkb200.so and attach prototypes.  Raises if the library is missing (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not built: run `python -m whisperkit_b200.build` (needs nvcc). "
            "whisperkit_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the ABI and the header ever diverge
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        raise WhisperError(status, load().wk_last_error().decode("utf-8", "replace"))
