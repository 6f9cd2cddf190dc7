"""Host mirror of the reference's long-form pieces over the C ABI (SURVEY section 8f rows 1 and 3): SegmentSeeker,
EnergyVAD / VADAudioChunker, prepareSeekClips and the batched seek loop (`transcribe_streams`).  All logic lives in
libwkb200.so (csrc/longform.cu); everything except `transcribe_streams` works without a GPU."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import check, wk_segment
from .api import DecodingOptions, SpecialTokens


@dataclass
class TranscriptionSegment:
    """Models.swift TranscriptionSegment, token-level fields (text needs the host tokenizer)."""
    stream: int
    id: int
    seek: int
    start: float
    end: float
    tokens: List[int]
    tokenLogProbs: List[float]
    temperature: float
    avgLogprob: float
    compressionRatio: float
    noSpeechProb: float
    words: Optional[list] = None
    text: str = ""


def _segs(raw, n, tokens, lps, rel=0) -> List[TranscriptionSegment]:
    out = []
    for i in range(n):
        g = raw[i]
        a, b = g.token_offset - rel, g.token_offset - rel + g.n_tokens
        out.append(TranscriptionSegment(g.stream, g.id, g.seek, g.start, g.end, [int(t) for t in tokens[a:b]], [float(v) for v in lps[a:b]],
                                        g.temperature, g.avg_logprob, g.compression_ratio, g.no_speech_prob))
    return out


class SegmentSeeker:
    """SegmentSeeking.findSeekPointAndSegments (SegmentSeeker.swift:41-189)."""

    def findSeekPointAndSegments(self, tokens: Sequence[int], tokenLogProbs: Sequence[float], avgLogProb: float, compressionRatio: float,
                                 temperature: float, options: DecodingOptions, allSegmentsCount: int, currentSeek: int, segmentSize: int,
                                 sampleRate: int, timeToken: int, noSpeechProb: float = 0.0) -> Tuple[int, Optional[List[TranscriptionSegment]]]:
        lib = _lib.load()
        n = len(tokens)
        tk = (C.c_int32 * max(1, n))(*[int(t) for t in tokens])
        lp = (C.c_float * max(1, n))(*[float(v) for v in tokenLogProbs])
        o, keep = options.to_c()
        raw = (wk_segment * 128)()
        ns, seek = C.c_int32(), C.c_int64()
        check(lib.wk_find_seek_point_and_segments(tk, lp, n, noSpeechProb, avgLogProb, compressionRatio, temperature, C.byref(o),
                                                  allSegmentsCount, currentSeek, segmentSize, sampleRate, timeToken, C.byref(seek), raw, 128,
                                                  C.byref(ns)))
        if ns.value < 0:
            return int(seek.value), None
        return int(seek.value), _segs(raw, ns.value, list(tokens), list(tokenLogProbs))


def prepareSeekClips(clipTimestamps: Sequence[float], contentFrames: int) -> List[Tuple[int, int]]:
    lib = _lib.load()
    n = len(clipTimestamps)
    ts = (C.c_float * max(1, n))(*[float(v) for v in clipTimestamps])
    cap = n // 2 + 2
    clips = (C.c_int64 * (2 * cap))()
    nc = C.c_int32()
    check(lib.wk_prepare_seek_clips(ts, n, contentFrames, clips, cap, C.byref(nc)))
    return [(int(clips[2 * i]), int(clips[2 * i + 1])) for i in range(nc.value)]


class EnergyVAD:
    """EnergyVAD / VoiceActivityDetector (EnergyVAD.swift, VoiceActivityDetector.swift)."""

    def __init__(self, sampleRate: int = 16000, frameLength: float = 0.1, frameOverlap: float = 0.0, energyThreshold: float = 0.02,
                 frameLengthSamples: Optional[int] = None, frameOverlapSamples: Optional[int] = None):
        self.sampleRate = sampleRate
        self.frameLengthSamples = frameLengthSamples if frameLengthSamples is not None else int(np.float32(frameLength) * np.float32(sampleRate))
        self.frameOverlapSamples = frameOverlapSamples if frameOverlapSamples is not None else int(np.float32(frameOverlap) * np.float32(sampleRate))
        self.energyThreshold = float(energyThreshold)
        self.lib = _lib.load()

    def voiceActivity(self, waveform) -> List[bool]:
        x = np.ascontiguousarray(waveform, dtype=np.float32)
        cap = len(x) // self.frameLengthSamples + 2
        out = np.zeros(cap, np.uint8)
        n = C.c_int64()
        check(self.lib.wk_vad_voice_activity(C.c_void_p(x.ctypes.data), len(x), self.frameLengthSamples, self.frameOverlapSamples,
                                             self.energyThreshold, C.c_void_p(out.ctypes.data), cap, C.byref(n)))
        return [bool(v) for v in out[: n.value]]

    def findLongestSilence(self, vad: Sequence[bool]) -> Optional[Tuple[int, int]]:
        v = np.ascontiguousarray(np.asarray(vad, dtype=np.uint8))
        s, e = C.c_int64(), C.c_int64()
        check(self.lib.wk_vad_find_longest_silence(C.c_void_p(v.ctypes.data) if len(v) else None, len(v), C.byref(s), C.byref(e)))
        return None if s.value < 0 else (int(s.value), int(e.value))

    def calculateActiveChunks(self, waveform) -> List[Tuple[int, int]]:
        x = np.ascontiguousarray(waveform, dtype=np.float32)
        cap = len(x) // self.frameLengthSamples + 2
        ch = (C.c_int64 * (2 * cap))()
        n = C.c_int32()
        check(self.lib.wk_vad_active_chunks(C.c_void_p(x.ctypes.data), len(x), self.frameLengthSamples, self.frameOverlapSamples,
                                            self.energyThreshold, ch, cap, C.byref(n)))
        return [(int(ch[2 * i]), int(ch[2 * i + 1])) for i in range(n.value)]

    def voiceActivityIndexToAudioSampleIndex(self, i: int) -> int:
        return i * self.frameLengthSamples

    def calculateNonSilentSeekClips(self, waveform) -> List[Tuple[int, int]]:
        ts = []
        for s, e in self.calculateActiveChunks(waveform):
            ts += [float(np.float32(s) / np.float32(self.sampleRate)), float(np.float32(e) / np.float32(self.sampleRate))]
        return prepareSeekClips(ts, len(waveform))


class VADAudioChunker:
    """VADAudioChunker.chunkAll (AudioChunker.swift:53-107) -> [(seekOffsetIndex, endIndex)]."""

    def __init__(self, windowPadding: int = 16000, vad: Optional[EnergyVAD] = None):
        self.windowPadding = windowPadding
        self.vad = vad or EnergyVAD()

    def chunkAll(self, audioArray, maxChunkLength: int, clipTimestamps: Sequence[float] = ()) -> List[Tuple[int, int]]:
        x = np.ascontiguousarray(audioArray, dtype=np.float32)
        n = len(clipTimestamps)
        ts = (C.c_float * max(1, n))(*[float(v) for v in clipTimestamps])
        cap = len(x) // max(1, maxChunkLength // 2) + n + 8
        ch = (C.c_int64 * (2 * cap))()
        nc = C.c_int32()
        check(self.vad.lib.wk_vad_chunk_all(C.c_void_p(x.ctypes.data), len(x), maxChunkLength, ts, n, self.windowPadding,
                                            self.vad.frameLengthSamples, self.vad.frameOverlapSamples, self.vad.energyThreshold, ch, cap,
                                            C.byref(nc)))
        return [(int(ch[2 * i]), int(ch[2 * i + 1])) for i in range(nc.value)]


def transcribe_streams(kit, audioArrays: Sequence[np.ndarray], options: Optional[DecodingOptions] = None,
                       clipTimestamps: Sequence[float] = (), windowClipTime: float = 1.0, maxWindowSeek: Optional[int] = None,
                       chunkingStrategy: Optional[str] = None, split_to_word_tokens=None, decode=None, hooks=None, languages: Optional[list] = None):
    """TranscribeTask.run's seek loop for many audio arrays at once (TranscribeTask.swift:98-279; `chunkingStrategy="vad"`
    = WhisperKit.swift:878-911).  Returns (segments per stream, number of 30 s windows decoded).  A `languages` list receives each
    stream's TranscriptionResult.language as (token, log-probability) (wk_transcription_language)."""
    opts = kit.resolveLanguage(options or DecodingOptions())   # DecodingOptions.language -> <|xx|> through the tokenizer
    lib = kit.model.lib
    arrs = [np.ascontiguousarray(a, dtype=np.float32) for a in audioArrays]
    ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
    lens = (C.c_int64 * len(arrs))(*[len(a) for a in arrs])
    prompt = kit.textDecoder.prefillDecoderInputs(opts if opts.usePrefillPrompt else None, kit.specialTokens)
    st = kit.specialTokens.to_c()
    o, keep = opts.to_c()
    p = (C.c_int32 * len(prompt))(*prompt)
    n = len(clipTimestamps)
    ts = (C.c_float * max(1, n))(*[float(v) for v in clipTimestamps])
    h = C.c_void_p()
    from .wordtiming import WordTiming, make_hooks
    native = hooks                      # a wk_tokenizer_hooks struct (WhisperTokenizer.hooks()): the library's own tokenizer, no host callbacks
    if native is None:
        hooks, keep_hooks = make_hooks(split_to_word_tokens, decode)
    check(lib.wk_transcribe_streams(kit.model.handle, kit.textDecoder.handle, ptrs, lens, len(arrs), C.byref(st), C.byref(o), p, len(prompt),
                                    ts, n, windowClipTime, -1 if maxWindowSeek is None else maxWindowSeek,
                                    1 if chunkingStrategy == "vad" else 0, C.byref(hooks) if (split_to_word_tokens is not None or native is not None) else None,
                                    C.byref(h)))
    try:
        ns, nt = lib.wk_transcription_segment_count(h), lib.wk_transcription_token_count(h)
        raw = (wk_segment * max(1, ns))()
        check(lib.wk_transcription_segments(h, raw, max(1, ns)))
        tk = (C.c_int32 * max(1, nt))()
        lp = (C.c_float * max(1, nt))()
        check(lib.wk_transcription_tokens(h, tk, lp, max(1, nt)))
        segs = _segs(raw, ns, tk, lp)
        if opts.wordTimestamps:
            for g in segs:
                g.words = []
            w = _lib.wk_word()
            for i in range(lib.wk_transcription_word_count(h)):
                check(lib.wk_transcription_word(h, i, C.byref(w)))
                segs[w.segment].words.append(WordTiming(w.word.decode("utf-8"), [int(w.tokens[k]) for k in range(w.n_tokens)], float(w.start),
                                                        float(w.end), float(w.probability), int(w.segment)))
        windows = lib.wk_transcription_window_count(h)
        if languages is not None:
            tok, lp = C.c_int32(), C.c_float()
            for i in range(len(arrs)):
                check(lib.wk_transcription_language(h, i, C.byref(tok), C.byref(lp)))
                languages.append((int(tok.value), float(lp.value)))
    finally:
        lib.wk_transcription_free(h)
    per_stream = [[g for g in segs if g.stream == i] for i in range(len(arrs))]
    return per_stream, windows


@dataclass
class TranscriptionResult:
    """Models.swift TranscriptionResult, the fields this backend produces."""
    text: str
    segments: List[TranscriptionSegment]
    windows: int = 0
    languageToken: Optional[int] = None
    languageLogProb: float = 0.0
    language: Optional[str] = None      # the code, with a tokenizer


def transcribe_audio(kit, audioArrays: Sequence[np.ndarray], options: Optional[DecodingOptions] = None, tokenizer=None,
                     chunkingStrategy: Optional[str] = None, clipTimestamps: Sequence[float] = ()) -> List[TranscriptionResult]:
    """WhisperKit.transcribe(audioArrays:) for audio of any length (WhisperKit.swift:667-812 over TranscribeTask.run): every array runs the
    seek loop, all arrays share the GPU batches.  With a `whisperkit_b200.tokenizer.WhisperTokenizer` the segment and result texts are
    filled the way the reference does it (segment text: SegmentSeeker.swift:118-121,160-165 - all tokens unless skipSpecialTokens;
    result text: TranscribeTask.finalizeTranscriptionResult, :299-311 - text tokens only, trimmed) and word timestamps need no callbacks."""
    opts = options or DecodingOptions()
    if tokenizer is None and opts.wordTimestamps:
        raise _lib.WhisperError(-1, "wordTimestamps needs a tokenizer")
    native = tokenizer.hooks() if (tokenizer is not None and opts.wordTimestamps and hasattr(tokenizer, "hooks")) else None
    split = tokenizer.splitToWordTokens if (tokenizer is not None and opts.wordTimestamps and native is None) else None
    langs = []
    per_stream, windows = transcribe_streams(kit, audioArrays, opts, clipTimestamps=clipTimestamps, chunkingStrategy=chunkingStrategy,
                                             split_to_word_tokens=split, decode=tokenizer.decode if split is not None else None, hooks=native,
                                             languages=langs)
    sb = kit.specialTokens.specialTokenBegin
    out = []
    for segs, (ltok, llp) in zip(per_stream, langs):
        text = ""
        if tokenizer is not None:
            for g in segs:
                g.text = tokenizer.decode([t for t in g.tokens if t < sb] if opts.skipSpecialTokens else g.tokens)
            text = tokenizer.decode([t for g in segs for t in g.tokens if t < sb]).strip(" \t               　")
        code = tokenizer.decode([ltok]).removeprefix("<|").removesuffix("|>") if tokenizer is not None else None
        out.append(TranscriptionResult(text, segs, windows, ltok, llp, code))
    return out
