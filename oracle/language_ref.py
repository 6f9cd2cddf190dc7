"""Language-detection oracle (test infrastructure; see oracle/__init__.py).

CPU restatement of the reference's host logic around detectLanguage:
  * TextDecoding.detectLanguage       Sources/WhisperKit/Core/TextDecoder.swift:420-539
  * decodeWithFallback                Sources/WhisperKit/Core/TranscribeTask.swift:316-411 (detect, re-prefill, decode, ladder,
                                      detectedLanguage bookkeeping)
  * language inferred from the tokens Sources/WhisperKit/Core/TextDecoder.swift:804-822
  * TranscriptionResult.language      TranscribeTask.swift:341-376 (per window), TranscriptionUtilities.swift:103 (chunked audio)
  * allLanguageTokens                 Sources/WhisperKit/Core/Models.swift:1219

Languages are token ids here; the reference's strings are `tokenizer.decode([token])` with "<|" / "|>" trimmed.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from . import decode_ref as D

Language = Tuple[int, float]   # (token, log-probability)


def default_language_tokens(st: D.SpecialTokens) -> List[int]:
    """The language block of a Whisper vocabulary: ids strictly between <|startoftranscript|> and min(<|translate|>, <|transcribe|>)."""
    return list(range(st.startOfTranscriptToken + 1, min(st.translateToken, st.transcribeToken)))


def rung_temperatures(options: D.DecodingOptions) -> List[float]:
    """Float16(temperature) + Float16(i) * Float16(increment), i = 0 ... fallbackCount (TranscribeTask.swift:323-328)."""
    f16 = np.float16
    out = [float(options.temperature)]
    for i in range(1, options.temperatureFallbackCount + 1):
        out.append(float(f16(f16(options.temperature) + f16(f16(i) * f16(options.temperatureIncrementOnFallback)))))
    return out


def detect_language(predict_logits: Callable[[int, int], np.ndarray], st: D.SpecialTokens, allLanguageTokens: Sequence[int],
                    sampler: D.GreedyTokenSampler) -> Language:
    """One decoder step on [SOT] at position 0, LanguageLogitsFilter, the rung's sampler (TextDecoder.swift:420-539)."""
    logits = np.array(predict_logits(st.startOfTranscriptToken, 0), dtype=np.float32).reshape(-1)
    logits = D.LanguageLogitsFilter(allLanguageTokens, len(logits), 0).filterLogits(logits, [st.startOfTranscriptToken])
    return sampler._sample(logits)


def result_language(result: D.DecodingResult, languageToken: Optional[int], allLanguageTokens: Sequence[int],
                    st: D.SpecialTokens) -> Language:
    """DecodingResult.language / languageProbs of decodeText (TextDecoder.swift:804-822): the option's language (0), else the first
    language token of the filtered tokens with its log-probability, else English (0)."""
    if languageToken is not None:
        return languageToken, 0.0
    langs = set(allLanguageTokens)
    for i, t in enumerate(result.tokens):
        if t in langs:
            return t, float(result.tokenLogProbs[i])
    return st.englishToken, 0.0


def decode_with_fallback(predict_logits: Callable[[int, int], np.ndarray], options: D.DecodingOptions, st: D.SpecialTokens,
                         isModelMultilingual: bool, allLanguageTokens: Sequence[int], languageToken: Optional[int] = None,
                         detectLanguage: bool = False, initialPrompt: Optional[Sequence[int]] = None,
                         rng=None) -> Tuple[D.DecodingResult, Language]:
    """decodeWithFallback (TranscribeTask.swift:316-411) for one window.  `predict_logits(token, tokenIndex)` writes its own KV cache at
    tokenIndex, so every decode (and every detection) restarts at 0.  `initialPrompt` = a caller's prompt (usePrefillPrompt false): the
    detection then only reports.  Returns the kept result and the window's language (detectedLanguage ?? defaultLanguageCode)."""
    detected: Optional[Language] = None
    result = None
    for i, temp in enumerate(rung_temperatures(options)):
        sampler = D.GreedyTokenSampler(temp, st.endToken, options, rng=rng)
        lang = languageToken
        if isModelMultilingual and languageToken is None and detectLanguage:   # :339-365
            detected = detect_language(predict_logits, st, allLanguageTokens, sampler)
            lang = detected[0]
        prompt = D.prefill_prompt(options, st, isModelMultilingual, lang) if initialPrompt is None else list(initialPrompt)
        result = D.decode_text(predict_logits, prompt, options, st, isModelMultilingual, sampler=sampler)
        needs = result.fallback is not None and result.fallback.needsFallback
        if not needs or i == options.temperatureFallbackCount:
            break
    if detected is not None:
        return result, detected
    return result, result_language(result, languageToken, allLanguageTokens, st)


def stream_language(units: Sequence[Sequence[Language]], detecting: bool, englishToken: int) -> Language:
    """TranscriptionResult.language of one audio stream.  `units`: the per-window languages of each unit in order (one unit for plain
    audio, one per VAD chunk).  A unit's language is its last window's when the task detects (detectedLanguage is reassigned every window,
    TranscribeTask.swift:352) and its first window's otherwise (:376); a chunked stream takes its first chunk's
    (TranscriptionUtilities.swift:103); no window at all means English."""
    if not units or not units[0]:
        return englishToken, 0.0
    first = units[0]
    return first[-1] if detecting else first[0]
