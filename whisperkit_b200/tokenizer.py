"""Host mirror of the decode side of the reference tokenizer over the C ABI (SURVEY section 8f row 4): WhisperTokenizer.decode,
convertTokenToId, specialTokens and splitToWordTokens (Models.swift:1165-1306).  All logic lives in libwkb200.so
(csrc/tokenizer.cu) and runs without a GPU."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

from . import _lib
from ._lib import check, wk_special_tokens, wk_tokenizer_hooks
from .api import SpecialTokens


class WhisperTokenizer:
    def __init__(self, path: Optional[str] = None, tokens: Optional[Sequence[str]] = None, ids: Optional[Sequence[int]] = None,
                 flags: Optional[Sequence[int]] = None, cleanUpTokenizationSpaces: bool = True):
        self.lib = _lib.load()
        self.handle = C.c_void_p()
        if path is not None:
            check(self.lib.wk_tokenizer_load(path.encode("utf-8"), C.byref(self.handle)))
        else:
            n = len(tokens)
            arr = (C.c_char_p * max(1, n))(*[t.encode("utf-8") for t in tokens])
            idv = (C.c_int32 * max(1, n))(*[int(i) for i in ids])
            fl = (C.c_uint8 * max(1, n))(*[int(f) for f in (flags or [0] * n)])
            check(self.lib.wk_tokenizer_create(arr, idv, fl, n, int(cleanUpTokenizationSpaces), C.byref(self.handle)))

    @property
    def vocabSize(self) -> int:
        return self.lib.wk_tokenizer_vocab_size(self.handle)

    def convertTokenToId(self, token: str) -> Optional[int]:
        i = self.lib.wk_tokenizer_token_to_id(self.handle, token.encode("utf-8"))
        return None if i < 0 else i

    def decode(self, tokens: Sequence[int], skipSpecialTokens: bool = False) -> str:
        n = len(tokens)
        arr = (C.c_int32 * max(1, n))(*[int(t) for t in tokens])
        cap = 64 * n + 64
        for _ in range(2):
            buf = C.create_string_buffer(cap)
            r = self.lib.wk_tokenizer_decode(self.handle, arr, n, int(skipSpecialTokens), buf, cap)
            if r >= 0:
                return buf.raw[:r].decode("utf-8")
            cap = -r + 1
        raise _lib.WhisperError(-1, "wk_tokenizer_decode failed")

    def encode(self, text: str) -> List[int]:
        """encode(text:) without the post-processor (no special-token template)."""
        b = text.encode("utf-8")
        cap = 4 * len(b) + 16
        for _ in range(2):
            ids = (C.c_int32 * cap)()
            n = self.lib.wk_tokenizer_encode(self.handle, b, ids, cap)
            if n >= 0:
                return [int(v) for v in ids[:n]]
            if n == -1:
                break
            cap = -n
        raise _lib.WhisperError(-1, "wk_tokenizer_encode failed")

    @property
    def specialTokens(self) -> SpecialTokens:
        st = wk_special_tokens()
        check(self.lib.wk_tokenizer_special_tokens(self.handle, C.byref(st)))
        return SpecialTokens(endToken=st.end_token, englishToken=st.english_token, noSpeechToken=st.no_speech_token,
                             noTimestampsToken=st.no_timestamps_token, specialTokenBegin=st.special_token_begin,
                             startOfPreviousToken=st.start_of_previous_token, startOfTranscriptToken=st.start_of_transcript_token,
                             timeTokenBegin=st.time_token_begin, transcribeToken=st.transcribe_token, translateToken=st.translate_token,
                             whitespaceToken=st.whitespace_token)

    @property
    def allLanguageTokens(self) -> List[int]:
        """WhisperTokenizerWrapper.allLanguageTokens (Models.swift:1219): the "<|xx|>" / "<|xxx|>" ids of the vocabulary, ascending."""
        n = self.lib.wk_tokenizer_language_tokens(self.handle, None, 0)
        if n == 0:
            return []
        arr = (C.c_int32 * -n)()
        n = self.lib.wk_tokenizer_language_tokens(self.handle, arr, -n)
        if n < 0:
            raise _lib.WhisperError(-1, "wk_tokenizer_language_tokens failed")
        return [int(v) for v in arr[:n]]

    def splitToWordTokens(self, tokenIds: Sequence[int]) -> Tuple[List[str], List[List[int]]]:
        n = len(tokenIds)
        arr = (C.c_int32 * max(1, n))(*[int(t) for t in tokenIds])
        cap = 64 * n + 256
        text = C.create_string_buffer(cap)
        counts = (C.c_int32 * (n + 1))()
        nw = self.lib.wk_tokenizer_split_to_word_tokens(self.handle, arr, n, text, cap, counts, n + 1)
        if nw < 0:
            raise _lib.WhisperError(-1, f"wk_tokenizer_split_to_word_tokens failed ({nw})")
        words, groups, off, k = [], [], 0, 0
        raw = text.raw
        for i in range(nw):
            end = raw.index(b"\0", off)
            words.append(raw[off:end].decode("utf-8"))
            off = end + 1
            groups.append([int(t) for t in tokenIds[k:k + counts[i]]])
            k += counts[i]
        return words, groups

    def hooks(self) -> wk_tokenizer_hooks:
        """wk_tokenizer_hooks bound to this tokenizer (for wk_transcribe_streams / wk_add_word_timestamps)."""
        h = wk_tokenizer_hooks()
        check(self.lib.wk_tokenizer_hooks_init(self.handle, C.byref(h)))
        return h

    def close(self):
        if getattr(self, "handle", None) and self.handle.value:
            self.lib.wk_tokenizer_free(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass
