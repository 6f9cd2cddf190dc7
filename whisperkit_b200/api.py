"""Host-side mirror of the reference's protocol surface over the C ABI (ctypes).

Class / method names follow WhisperKit so parity tests read like the reference's own tests:

  FeatureExtractor.logMelSpectrogram      Sources/WhisperKit/Core/FeatureExtractor.swift:13-17,40-56
  AudioEncoder.encodeFeatures             Sources/WhisperKit/Core/AudioEncoder.swift:10-18,50-63
  TextDecoder.{prepareDecoderInputs,      Sources/WhisperKit/Core/TextDecoder.swift:60-105
     prefillDecoderInputs, predictLogits, decodeText}
  DecodingOptions                         Sources/WhisperKit/Core/Configurations.swift:155-247
  SpecialTokens                           Sources/WhisperKit/Core/Models.swift:1111-1149
  WhisperKit.transcribe(audioArrays:)     Sources/WhisperKit/Core/WhisperKit.swift:667-812

All arithmetic happens in libwkb200.so (sm_100a kernels); this module only marshals arguments.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import (PROGRESS_FN, WK_DTYPE_BF16, WK_DTYPE_F16, WK_DTYPE_F32, WhisperError, check, wk_batch_opts, wk_decode_opts,
                   wk_decode_result, wk_model_config, wk_model_info, wk_special_tokens)

MAX_TOKEN_CONTEXT = 224  # Constants.maxTokenContext (Models.swift:1334)
WINDOW_SAMPLES = 480000  # Constants.defaultWindowSamples (Models.swift:1457)
FALLBACK_REASONS = {0: None, 1: "firstTokenLogProbThreshold", 2: "silence", 3: "compressionRatioThreshold",
                    4: "logProbThreshold"}


def _ptr(x):
    """Raw address of a numpy array or torch tensor (host or device)."""
    if x is None:
        return None
    if hasattr(x, "data_ptr"):
        return C.c_void_p(x.data_ptr())
    return C.c_void_p(x.ctypes.data)


@dataclass
class SpecialTokens:
    endToken: int = 50257
    englishToken: int = 50259
    noSpeechToken: int = 50362
    noTimestampsToken: int = 50363
    specialTokenBegin: int = 50257
    startOfPreviousToken: int = 50361
    startOfTranscriptToken: int = 50258
    timeTokenBegin: int = 50364
    transcribeToken: int = 50359
    translateToken: int = 50358
    whitespaceToken: int = 220

    def to_c(self) -> wk_special_tokens:
        return wk_special_tokens(self.endToken, self.englishToken, self.noSpeechToken, self.noTimestampsToken,
                                 self.specialTokenBegin, self.startOfPreviousToken, self.startOfTranscriptToken,
                                 self.timeTokenBegin, self.transcribeToken, self.translateToken, self.whitespaceToken)

    @staticmethod
    def from_any(o) -> "SpecialTokens":
        return SpecialTokens(**{k: getattr(o, k) for k in SpecialTokens().__dict__})


@dataclass
class DecodingOptions:
    task: str = "transcribe"
    language: Optional[str] = None
    languageToken: Optional[int] = None  # id of "<|language|>" (tokenizer lookup is the host's job)
    temperature: float = 0.0
    temperatureIncrementOnFallback: float = 0.2
    temperatureFallbackCount: int = 5
    sampleLength: int = MAX_TOKEN_CONTEXT
    topK: int = 5
    usePrefillPrompt: bool = True
    skipSpecialTokens: bool = False
    withoutTimestamps: bool = False
    maxInitialTimestamp: Optional[float] = None
    promptTokens: Optional[List[int]] = None
    prefixTokens: Optional[List[int]] = None
    suppressBlank: bool = False
    suppressTokens: List[int] = field(default_factory=list)
    compressionRatioThreshold: Optional[float] = 2.4
    logProbThreshold: Optional[float] = -1.0
    firstTokenLogProbThreshold: Optional[float] = -1.5
    noSpeechThreshold: Optional[float] = 0.6
    concurrentWorkerCount: int = 16
    wordTimestamps: bool = False
    seed: int = 0
    beamSize: int = 1                 # extension: the reference's BeamSearchTokenSampler is an unimplemented stub (TokenSampler.swift:254-290)
    beamPatience: float = 1.0
    detectLanguage: Optional[bool] = None   # None = !usePrefillPrompt (Configurations.swift:222)

    def to_c(self):
        """Returns (struct, keepalive) - keepalive holds the int arrays the struct points into."""
        keep = []

        def arr(v):
            if v is None:
                return None, -1
            a = (C.c_int32 * max(1, len(v)))(*v)
            keep.append(a)
            return C.cast(a, C.POINTER(C.c_int32)), len(v)

        sup, nsup = arr(list(self.suppressTokens))
        pr, npr = arr(self.promptTokens)
        pf, npf = arr(self.prefixTokens)

        def opt(v):
            return (0, 0.0) if v is None else (1, float(v))

        o = wk_decode_opts()
        o.task_translate = 1 if self.task == "translate" else 0
        o.language_token = -1 if self.languageToken is None else int(self.languageToken)
        o.temperature = float(self.temperature)
        o.sample_length = int(self.sampleLength)
        o.top_k = int(self.topK)
        o.use_prefill_prompt = int(self.usePrefillPrompt)
        o.without_timestamps = int(self.withoutTimestamps)
        o.suppress_blank = int(self.suppressBlank)
        o.suppress_tokens, o.n_suppress_tokens = sup, max(nsup, 0)
        o.prompt_tokens, o.n_prompt_tokens = pr, npr
        o.prefix_tokens, o.n_prefix_tokens = pf, npf
        o.has_compression_ratio_threshold, o.compression_ratio_threshold = opt(self.compressionRatioThreshold)
        o.has_logprob_threshold, o.logprob_threshold = opt(self.logProbThreshold)
        o.has_first_token_logprob_threshold, o.first_token_logprob_threshold = opt(self.firstTokenLogProbThreshold)
        o.has_no_speech_threshold, o.no_speech_threshold = opt(self.noSpeechThreshold)
        o.seed = int(self.seed)
        o.temperature_fallback_count = int(self.temperatureFallbackCount)
        o.temperature_increment_on_fallback = float(self.temperatureIncrementOnFallback)
        o.word_timestamps = int(self.wordTimestamps)
        o.beam_size = int(self.beamSize)
        o.beam_patience = float(self.beamPatience)
        o.detect_language = int(not self.usePrefillPrompt if self.detectLanguage is None else self.detectLanguage)
        return o, keep


@dataclass
class DecodingFallback:
    needsFallback: bool
    fallbackReason: str


@dataclass
class DecodingResult:
    """Models.swift:383-439 (token-level fields; text needs the host tokenizer)."""
    tokens: List[int]
    tokenLogProbs: List[float]
    avgLogProb: float
    compressionRatio: float
    temperature: float
    fallback: Optional[DecodingFallback]
    currentTokenCount: int = 0
    steps: int = 0
    isFirstTokenLogProbTooLow: bool = False
    languageToken: Optional[int] = None        # set by WhisperKit.transcribe (wk_session_languages)
    languageProbs: Dict[object, float] = field(default_factory=dict)   # {language (code, or token id without a tokenizer): log-probability}
    language: Optional[str] = None             # the code ("en"), when the WhisperKit has a tokenizer

    @staticmethod
    def from_c(r: wk_decode_result) -> "DecodingResult":
        n = r.n_tokens
        reason = FALLBACK_REASONS.get(r.fallback_reason)
        fb = DecodingFallback(bool(r.needs_fallback), reason) if reason else None
        return DecodingResult(list(r.tokens[:n]), list(r.token_logprobs[:n]), r.avg_logprob, r.compression_ratio,
                              r.temperature, fb, r.n_current_tokens, r.steps, bool(r.first_token_logprob_too_low))


_DT = {"f32": WK_DTYPE_F32, "f16": WK_DTYPE_F16, "bf16": WK_DTYPE_BF16}


class Model:
    """Owns a wk_model (weights + encoder workspaces on one GPU)."""

    def __init__(self, variant: str = "large-v3", device: int = 0, max_batch: int = 16, dtype: str = "bf16",
                 config: Optional[dict] = None):
        self.lib = _lib.load()
        cfg = wk_model_config()
        self.lib.wk_default_config(variant.encode(), C.byref(cfg))
        if config:
            for k, v in config.items():
                setattr(cfg, k, v)
        cfg.max_batch = max_batch
        cfg.dtype = _DT[dtype]
        self.cfg = cfg
        self.handle = C.c_void_p()
        check(self.lib.wk_model_create(C.byref(cfg), device, C.byref(self.handle)))
        self.variant = variant
        self.device = device

    @classmethod
    def from_pretrained(cls, weights_dir: str, device: int = 0, max_batch: int = 16, dtype: str = "bf16") -> "Model":
        """HuggingFace checkpoint directory (config.json + *.safetensors)."""
        self = cls.__new__(cls)
        self.lib = _lib.load()
        self.handle = C.c_void_p()
        check(self.lib.wk_model_load(weights_dir.encode(), device, max_batch, _DT[dtype], C.byref(self.handle)))
        info = wk_model_info()
        check(self.lib.wk_model_info_get(self.handle, C.byref(info)))
        cfg = wk_model_config()
        for f in ("n_mels", "d_model", "n_heads", "enc_layers", "dec_layers", "vocab", "n_audio_ctx", "dtype", "max_batch"):
            setattr(cfg, f, getattr(info, f))
        self.cfg, self.variant, self.device = cfg, os.path.basename(weights_dir.rstrip("/")), device
        return self

    def set_tensor(self, name: str, t) -> None:
        if hasattr(t, "data_ptr"):
            import torch
            t = t.contiguous()
            dt = {torch.float32: WK_DTYPE_F32, torch.float16: WK_DTYPE_F16, torch.bfloat16: WK_DTYPE_BF16}[t.dtype]
            shape = list(t.shape)
        else:
            t = np.ascontiguousarray(t)
            dt = {np.dtype("float32"): WK_DTYPE_F32, np.dtype("float16"): WK_DTYPE_F16}[t.dtype]
            shape = list(t.shape)
        shp = (C.c_int64 * len(shape))(*shape)
        check(self.lib.wk_model_set_tensor(self.handle, name.encode(), _ptr(t), dt, shp, len(shape)))

    def load_state_dict(self, weights: Dict[str, object]) -> None:
        for k, v in weights.items():
            self.set_tensor(k, v)
        check(self.lib.wk_model_finalize(self.handle))

    def setAlignmentHeads(self, pairs: Sequence[Sequence[int]]) -> None:
        """(layer, head) pairs averaged into `alignment_heads_weights`; [] restores the default (all heads of the last half of the layers)."""
        flat = [int(v) for p in pairs for v in p]
        arr = (C.c_int32 * max(1, len(flat)))(*flat)
        check(self.lib.wk_model_set_alignment_heads(self.handle, arr, len(flat) // 2))

    def init_random(self, seed: int = 0, std: float = 0.02) -> None:
        check(self.lib.wk_model_init_random(self.handle, seed, std))

    @property
    def info(self) -> wk_model_info:
        i = wk_model_info()
        check(self.lib.wk_model_info_get(self.handle, C.byref(i)))
        return i

    @property
    def stream(self) -> int:
        return int(self.lib.wk_model_stream(self.handle) or 0)

    def last_timings(self) -> dict:
        a = (C.c_float * 6)()
        check(self.lib.wk_last_timings(self.handle, a))
        return dict(zip(("logmels", "encoding", "crossKV", "decodingLoop", "h2d", "d2h"), [float(x) for x in a]))

    def close(self):
        if getattr(self, "handle", None) and self.handle.value:
            self.lib.wk_model_free(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceTensor:
    """Opaque device buffer handed between mel -> encoder -> decoder (the reference's marker protocols
    FeatureExtractorOutputType / AudioEncoderOutputType allow exactly this, FeatureExtractor.swift:10-11).  Owns its buffer, like the
    MLMultiArray the reference returns: released with the object."""

    def __init__(self, model: Model, handle):
        self.model, self.handle = model, handle

    def close(self):
        if getattr(self, "handle", None) and self.handle.value and getattr(self.model, "handle", None) and self.model.handle.value:
            self.model.lib.wk_tensor_free(self.handle)
        self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def shape(self):
        shp = (C.c_int64 * 4)()
        nd, dt = C.c_int32(), C.c_int32()
        check(self.model.lib.wk_tensor_shape(self.handle, shp, C.byref(nd), C.byref(dt)))
        return tuple(shp[: nd.value])

    def numpy(self, row_pad: int = 0) -> np.ndarray:
        """Reference layout, f32: mel [B, nMels, 3000]; encoder output [B, d, 1500].  row_pad > 0 reads back through explicit element
        strides into rows padded by that many elements (how an IOSurface-backed MLMultiArray lays its rows out)."""
        b, c, _, t = self.shape
        if row_pad:
            buf = np.zeros((b, c, t + row_pad), dtype=np.float32)
            check(self.model.lib.wk_tensor_to_host_strided(self.handle, _ptr(buf), c * (t + row_pad), t + row_pad, 1, buf.size))
            return buf[:, :, :t]
        out = np.empty((b, c, t), dtype=np.float32)
        check(self.model.lib.wk_tensor_to_host(self.handle, _ptr(out), out.size))
        return out


class FeatureExtractor:
    def __init__(self, model: Model):
        self.model = model

    @property
    def melCount(self) -> int:
        return self.model.info.n_mels

    @property
    def windowSamples(self) -> int:
        return self.model.info.window_samples

    def logMelSpectrogram(self, audio, samples_per_window: Optional[Sequence[int]] = None) -> DeviceTensor:
        """audio: [B, stride] (or [stride]) float32, numpy or torch (host or CUDA)."""
        if not hasattr(audio, "data_ptr"):
            audio = np.ascontiguousarray(audio, dtype=np.float32)
        if audio.ndim == 1:
            audio = audio[None]
        n, stride = int(audio.shape[0]), int(audio.shape[1])
        spw = None
        if samples_per_window is not None:
            spw = (C.c_int32 * n)(*[int(v) for v in samples_per_window])
        out = C.c_void_p()
        check(self.model.lib.wk_mel(self.model.handle, _ptr(audio), n, stride, spw, C.byref(out)))
        return DeviceTensor(self.model, out)


class AudioEncoder:
    def __init__(self, model: Model):
        self.model = model

    @property
    def embedSize(self) -> int:
        return self.model.info.d_model

    @property
    def sequenceLength(self) -> int:
        return self.model.info.n_audio_ctx

    def encodeFeatures(self, features: DeviceTensor) -> DeviceTensor:
        out = C.c_void_p()
        check(self.model.lib.wk_encode(self.model.handle, features.handle, C.byref(out)))
        return DeviceTensor(self.model, out)


class TextDecoder:
    """One decoding session (per-worker DecodingInputs + device KV caches)."""

    def __init__(self, model: Model, max_batch: Optional[int] = None):
        self.model = model
        self.lib = model.lib
        self.max_batch = max_batch or model.cfg.max_batch
        self.handle = C.c_void_p()
        check(self.lib.wk_session_create(model.handle, self.max_batch, C.byref(self.handle)))
        self.batch = 0

    # properties the reference reads off the CoreML model (TextDecoder.swift:313-331)
    @property
    def logitsSize(self) -> int:
        return self.model.info.vocab

    @property
    def kvCacheEmbedDim(self) -> int:
        return self.model.info.kv_embed_dim

    @property
    def kvCacheMaxSequenceLength(self) -> int:
        return self.model.info.kv_max_len

    @property
    def windowSize(self) -> int:
        return self.model.info.n_audio_ctx

    @property
    def embedSize(self) -> int:
        return self.model.info.d_model

    @property
    def isModelMultilingual(self) -> bool:
        return bool(self.model.info.is_multilingual)

    def prepareDecoderInputs(self) -> None:
        check(self.lib.wk_session_reset(self.handle))

    def prefillDecoderInputs(self, options: Optional[DecodingOptions], specialTokens: SpecialTokens) -> List[int]:
        st = specialTokens.to_c()
        o, keep = (options or DecodingOptions()).to_c()
        out = (C.c_int32 * MAX_TOKEN_CONTEXT)()
        n = C.c_int32()
        check(self.lib.wk_build_prompt(self.model.handle, C.byref(st), C.byref(o), 1 if options is not None else 0, out,
                                       MAX_TOKEN_CONTEXT, C.byref(n)))
        return list(out[: n.value])

    def bindEncoderOutput(self, enc: DeviceTensor) -> None:
        check(self.lib.wk_session_set_encoder_output(self.handle, enc.handle))
        self.batch = enc.shape[0]

    def predictLogits(self, inputIds: Sequence[int], cacheLength: Sequence[int]) -> np.ndarray:
        b = self.batch
        ids = (C.c_int32 * b)(*[int(v) for v in inputIds])
        cl = (C.c_int32 * b)(*[int(v) for v in cacheLength])
        out = np.empty((b, self.logitsSize), dtype=np.float32)
        check(self.lib.wk_decode_step(self.handle, ids, cl, _ptr(out)))
        return out

    def decodeText(self, encoderOutput: Optional[DeviceTensor], prompt, options, specialTokens: SpecialTokens,
                   callback=None, callbackEvery: int = 0) -> List[DecodingResult]:
        """decodeText for every bound window.  `prompt` / `options` may be one shared value or one per window;
        callback(window, tokens, avgLogprob) -> bool is the TranscriptionCallback (False = stop that window early)."""
        if encoderOutput is not None:
            self.bindEncoderOutput(encoderOutput)
        st = specialTokens.to_c()
        n = self.batch
        bo, keep = make_batch_opts(n, options, prompt, callback, callbackEvery, None)
        res = (wk_decode_result * n)()
        check(self.lib.wk_decode_text_ex(self.handle, C.byref(st), C.byref(bo), res))
        return [DecodingResult.from_c(r) for r in res]

    def detectLanguage(self, encoderOutput: Optional[DeviceTensor], specialTokens: SpecialTokens, allLanguageTokens: Sequence[int],
                       temperature: float = 0.0):
        """TextDecoder.detectLanguage: returns (language_token[B], logprob[B])."""
        if encoderOutput is not None:
            self.bindEncoderOutput(encoderOutput)
        st = specialTokens.to_c()
        lang = (C.c_int32 * len(allLanguageTokens))(*[int(v) for v in allLanguageTokens])
        tok = (C.c_int32 * self.batch)()
        lp = (C.c_float * self.batch)()
        check(self.lib.wk_detect_language(self.handle, C.byref(st), lang, len(allLanguageTokens), float(temperature), tok, lp))
        return list(tok), list(lp)

    def setLanguageTokens(self, tokens: Sequence[int]) -> None:
        """allLanguageTokens of this session (detectLanguage's choices); [] restores the special tokens' language block."""
        arr = (C.c_int32 * max(1, len(tokens)))(*[int(t) for t in tokens])
        check(self.lib.wk_session_set_language_tokens(self.handle, arr, len(tokens)))

    def languages(self, n: int):
        """[(language token, log-probability)] of the first n windows of the last transcribe call (wk_session_languages)."""
        tok = (C.c_int32 * max(1, n))()
        lp = (C.c_float * max(1, n))()
        check(self.lib.wk_session_languages(self.handle, n, tok, lp))
        return [(int(tok[i]), float(lp[i])) for i in range(n)]

    def alignmentWeights(self, window: int, rows: int = MAX_TOKEN_CONTEXT) -> np.ndarray:
        """DecodingResult.cache.alignmentWeights of one window of the last decodeText(wordTimestamps: true): [rows, 1500] (Float16 values)."""
        out = np.empty((rows, self.model.info.n_audio_ctx), dtype=np.float32)
        check(self.lib.wk_session_alignment_weights(self.handle, window, rows, _ptr(out)))
        return out

    def stats(self) -> dict:
        """Scheduler counters of the last batched call (decode steps launched, live-row steps, admissions, ladder re-admissions)."""
        a = (C.c_int64 * 4)()
        check(self.lib.wk_session_stats(self.handle, a))
        return dict(zip(("steps", "row_steps", "admissions", "ladder"), [int(v) for v in a]))

    def lastLogits(self) -> np.ndarray:
        out = np.empty((self.batch, self.logitsSize), dtype=np.float32)
        check(self.lib.wk_session_last_logits(self.handle, _ptr(out)))
        return out

    def close(self):
        if getattr(self, "handle", None) and self.handle.value:
            self.lib.wk_session_free(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def make_batch_opts(n: int, options, prompt, callback=None, callbackEvery: int = 0, status=None, encoderChunk: int = 0):
    """wk_batch_opts for n windows.  options: DecodingOptions or a list of n; prompt: None (built per window from the options), one token
    list, or a list of n token lists.  Returns (struct, keepalive)."""
    keep = []
    bo = wk_batch_opts()
    opt_list = list(options) if isinstance(options, (list, tuple)) else [options]
    if len(opt_list) not in (1, n):
        raise ValueError(f"{len(opt_list)} DecodingOptions for {n} windows")
    arr = (wk_decode_opts * len(opt_list))()
    for i, o in enumerate(opt_list):
        c, k = o.to_c()
        arr[i] = c
        keep.append(k)
    keep.append(arr)
    bo.opts, bo.n_opts = arr, len(opt_list)
    if prompt is not None and len(prompt) > 0 and isinstance(prompt[0], (list, tuple, np.ndarray)):
        if len(prompt) != n:
            raise ValueError(f"{len(prompt)} prompts for {n} windows")
        rows = [(C.c_int32 * max(1, len(p)))(*[int(v) for v in p]) for p in prompt]
        ptrs = (C.POINTER(C.c_int32) * n)(*[C.cast(r, C.POINTER(C.c_int32)) for r in rows])
        lens = (C.c_int32 * n)(*[len(p) for p in prompt])
        keep += [rows, ptrs, lens]
        bo.prompts, bo.prompt_lens = ptrs, lens
    elif prompt is not None:
        p = (C.c_int32 * max(1, len(prompt)))(*[int(v) for v in prompt])
        keep.append(p)
        bo.prompt, bo.n_prompt = p, len(prompt)
    if callback is not None:
        def tramp(user, window, tokens, n_tokens, avg):
            try:
                return 1 if callback(int(window), [int(tokens[i]) for i in range(n_tokens)], float(avg)) is not False else 0
            except Exception:
                return 0
        fn = PROGRESS_FN(tramp)
        keep.append(fn)
        bo.progress = fn
    bo.progress_every = int(callbackEvery)
    if status is not None:
        bo.status = status
    bo.encoder_chunk = int(encoderChunk)
    return bo, keep


def filter_and_sample(model: Model, logits: np.ndarray, tokens: Sequence[Sequence[int]], specialTokens: SpecialTokens,
                      options: Optional[DecodingOptions] = None, isModelMultilingual: bool = True,
                      timestampSampleBegin: Optional[int] = None, blankSampleBegin: Optional[int] = None,
                      languageTokens: Optional[Sequence[int]] = None, languageSampleBegin: int = 0):
    """LogitsFiltering chain (SuppressBlank, SuppressTokens, TimestampRules, Language) + GreedyTokenSampler.update on
    the device, stateless.  Returns (token[B], logprob[B], filtered_logits[B, V])."""
    lib = model.lib
    logits = np.ascontiguousarray(logits, dtype=np.float32)
    if logits.ndim == 1:
        logits = logits[None]
    b, v = logits.shape
    ld = max(1, max((len(t) for t in tokens), default=1))
    tk = np.zeros((b, ld), dtype=np.int32)
    nt = np.zeros(b, dtype=np.int32)
    for i, t in enumerate(tokens):
        tk[i, : len(t)] = t
        nt[i] = len(t)
    st = specialTokens.to_c()
    o, keep = (options or DecodingOptions()).to_c()
    tok = np.zeros(b, dtype=np.int32)
    lp = np.zeros(b, dtype=np.float32)
    filt = np.zeros((b, v), dtype=np.float32)
    lang = np.asarray(list(languageTokens), dtype=np.int32) if languageTokens is not None else None
    check(lib.wk_filter_sample(model.handle, C.byref(st), C.byref(o), int(isModelMultilingual), _ptr(logits), b, v,
                               _ptr(tk), ld, _ptr(nt), -1 if timestampSampleBegin is None else timestampSampleBegin,
                               -1 if blankSampleBegin is None else blankSampleBegin, _ptr(lang),
                               0 if lang is None else len(lang), languageSampleBegin, _ptr(tok), _ptr(lp), _ptr(filt)))
    return tok, lp, filt


@dataclass
class WhisperKitConfig:
    """Configurations.swift:7-121, fields meaningful on this backend."""
    model: str = "large-v3"
    device: int = 0
    maxBatch: int = 16
    dtype: str = "bf16"
    specialTokens: Optional[SpecialTokens] = None
    weights: Optional[Dict[str, object]] = None  # HF-named tensors; None -> seeded random weights
    seed: int = 0
    modelFolder: Optional[str] = None            # HuggingFace checkpoint directory: config.json + *.safetensors (+ tokenizer.json / vocab.json)


class WhisperKit:
    """Orchestrator: transcribe(audioArrays:) fans a batch of <=30 s windows through mel -> encoder -> decoder on the
    GPU (WhisperKit.swift:667-812 + the per-window body of TranscribeTask.run, TranscribeTask.swift:116-278)."""

    def __init__(self, config: WhisperKitConfig):
        self.config = config
        self.tokenizer = None
        if config.modelFolder is not None:
            # loadModels + loadTokenizer from a local folder (WhisperKit.swift:358-470): weights through the safetensors loader, the
            # decode-side tokenizer when the folder carries tokenizer.json or vocab.json
            self.model = Model.from_pretrained(config.modelFolder, config.device, config.maxBatch, config.dtype)
            if any(os.path.exists(os.path.join(config.modelFolder, f)) for f in ("tokenizer.json", "vocab.json")):
                from .tokenizer import WhisperTokenizer
                self.tokenizer = WhisperTokenizer(config.modelFolder)
        else:
            self.model = Model(config.model, config.device, config.maxBatch, config.dtype)
            if config.weights is not None:
                self.model.load_state_dict(config.weights)
            else:
                self.model.init_random(config.seed)
        self.featureExtractor = FeatureExtractor(self.model)
        self.audioEncoder = AudioEncoder(self.model)
        self.textDecoder = TextDecoder(self.model, config.maxBatch)
        if self.tokenizer is not None:   # allLanguageTokens from the tokenizer's vocabulary (Models.swift:1219)
            self.textDecoder.setLanguageTokens(self.tokenizer.allLanguageTokens)
        info = self.model.info
        if config.specialTokens is not None:
            self.specialTokens = config.specialTokens
        elif self.tokenizer is not None:
            self.specialTokens = self.tokenizer.specialTokens
        elif info.vocab == 51866:
            self.specialTokens = SpecialTokens(endToken=50257, englishToken=50259, noSpeechToken=50363,
                                               noTimestampsToken=50364, specialTokenBegin=50257,
                                               startOfPreviousToken=50362, startOfTranscriptToken=50258,
                                               timeTokenBegin=50365, transcribeToken=50360, translateToken=50359)
        elif info.vocab == 51864:
            self.specialTokens = SpecialTokens(endToken=50256, englishToken=50258, noSpeechToken=50361,
                                               noTimestampsToken=50362, specialTokenBegin=50256,
                                               startOfPreviousToken=50360, startOfTranscriptToken=50257,
                                               timeTokenBegin=50363, transcribeToken=50358, translateToken=50357)
        else:
            self.specialTokens = SpecialTokens()

    def resolveLanguage(self, opts: DecodingOptions) -> DecodingOptions:
        """DecodingOptions.language -> the "<|xx|>" token id through the tokenizer, as prefillDecoderInputs does with
        tokenizer.convertTokenToId (TextDecoder.swift:181-186).  No tokenizer = an error, never a silent <|en|>."""
        if opts.language is None or opts.languageToken is not None or not self.textDecoder.isModelMultilingual:
            return opts
        if self.tokenizer is None:
            raise WhisperError(-4, f"DecodingOptions.language={opts.language!r} needs a tokenizer to resolve <|{opts.language}|> (or set languageToken)")
        tok = self.tokenizer.convertTokenToId(f"<|{opts.language}|>")
        if tok is None or tok < 0:
            raise WhisperError(-4, f"the tokenizer has no <|{opts.language}|> token")
        import dataclasses
        return dataclasses.replace(opts, languageToken=int(tok))

    def transcribe(self, audioArrays, decodeOptions=None, samplesPerWindow: Optional[Sequence[int]] = None, callback=None,
                   callbackEvery: int = 0, returnErrors: bool = False, encoderChunk: int = 0):
        """audioArrays: host float32 [N, stride<=480000-padded] (numpy, or pinned torch CPU tensor).  decodeOptions: one DecodingOptions
        or one per window (transcribeWithOptions' decodeOptionsArray, WhisperKit.swift:716-735).  One DecodingResult per window, in order;
        with returnErrors a window that failed yields its WhisperError instead of failing the call (the reference's Result<>, :775-790)."""
        a = audioArrays
        if not hasattr(a, "data_ptr"):
            a = np.ascontiguousarray(a, dtype=np.float32)
        if a.ndim == 1:
            a = a[None]
        n, stride = int(a.shape[0]), int(a.shape[1])
        if isinstance(decodeOptions, (list, tuple)):
            opts = [self.resolveLanguage(o or DecodingOptions()) for o in decodeOptions]
        else:
            opts = self.resolveLanguage(decodeOptions or DecodingOptions())
        st = self.specialTokens.to_c()
        status = (C.c_int32 * n)() if returnErrors else None
        bo, keep = make_batch_opts(n, opts, None, callback, callbackEvery, status, encoderChunk)
        spw = None
        if samplesPerWindow is not None:
            spw = (C.c_int32 * n)(*[int(v) for v in samplesPerWindow])
        res = (wk_decode_result * n)()
        # the prompt of every window is built inside the library from that window's options (prefillDecoderInputs); decodeWithFallback
        # (TranscribeTask.swift:316-411) runs there too: a window whose DecodingFallback asks for it is decoded again at the next temperature
        check(self.model.lib.wk_transcribe_windows_ex(self.model.handle, self.textDecoder.handle, _ptr(a), n, stride, spw, C.byref(st),
                                                      C.byref(bo), res))
        self.textDecoder.batch = min(n, self.config.maxBatch)
        langs = self.textDecoder.languages(n)
        out = []
        for i, r in enumerate(res):
            if returnErrors and status[i] != 0:
                out.append(WhisperError(int(status[i]), f"window {i} failed"))
            else:
                d = DecodingResult.from_c(r)
                d.languageToken, lp = langs[i]
                d.language = self.languageCode(d.languageToken)
                d.languageProbs = {d.language if d.language is not None else d.languageToken: lp}
                out.append(d)
        return out

    def languageCode(self, token: int) -> Optional[str]:
        """Language token -> code through the tokenizer ("<|de|>" -> "de"); None without a tokenizer."""
        if self.tokenizer is None:
            return None
        return self.tokenizer.decode([int(token)]).removeprefix("<|").removesuffix("|>")
