"""Language detection, the parts that run without a GPU: the tokenizer's allLanguageTokens through the C ABI, the default language
block, the ABI layout of DecodingOptions.detectLanguage, and the oracle's decodeWithFallback / per-stream language rules."""
import ctypes as C

import numpy as np

from oracle import decode_ref as D
from oracle import language_ref as LR
from whisperkit_b200 import _lib
from whisperkit_b200.api import DecodingOptions
from whisperkit_b200.tokenizer import WhisperTokenizer


def _tokenizer():
    # text, timestamps and every kind of special token, in no particular id order
    toks = ["a", "b", "Ġc", "<|endoftext|>", "<|startoftranscript|>", "<|en|>", "<|de|>", "<|haw|>", "<|yue|>", "<|translate|>",
            "<|transcribe|>", "<|startoftranscript|>x", "<|startofprev|>", "<|nospeech|>", "<|notimestamps|>", "<|0.00|>", "<|0.02|>",
            "<|EN|>", "<|e|>", "<|abcd|>", "<|z9|>"]
    ids = [10, 11, 12, 50, 51, 58, 52, 60, 53, 54, 55, 70, 56, 57, 59, 61, 62, 63, 64, 65, 66]
    flags = [0, 0, 0] + [3] * (len(toks) - 3)
    return WhisperTokenizer(tokens=toks, ids=ids, flags=flags), dict(zip(toks, ids))


def test_tokenizer_language_tokens_from_the_vocabulary():
    tk, ids = _tokenizer()
    want = sorted(ids[t] for t in ("<|en|>", "<|de|>", "<|haw|>", "<|yue|>"))
    assert tk.allLanguageTokens == want
    lib = _lib.load()
    out = (C.c_int32 * 8)()
    assert lib.wk_tokenizer_language_tokens(tk.handle, out, 2) == -len(want)      # -(needed): nothing written past cap
    assert lib.wk_tokenizer_language_tokens(tk.handle, None, 0) == -len(want)
    assert lib.wk_tokenizer_language_tokens(tk.handle, out, 8) == len(want) and list(out[:len(want)]) == want
    plain = WhisperTokenizer(tokens=["<|en|>", "x"], ids=[0, 1], flags=[0, 0])    # not an added token: no language
    assert plain.allLanguageTokens == []


def test_default_language_block():
    assert len(LR.default_language_tokens(D.SpecialTokens.large_v3())) == 100
    assert len(LR.default_language_tokens(D.SpecialTokens.english_only())) == 99
    assert LR.default_language_tokens(D.SpecialTokens.large_v3())[0] == D.SpecialTokens.large_v3().englishToken


def test_decode_result_layout_and_detect_field():
    assert C.sizeof(_lib.wk_decode_result) == 4 + 226 * 4 + 226 * 4 + 8 * 4
    f = _lib.wk_decode_opts
    assert f.detect_language.offset == f.beam_patience.offset + 4
    assert DecodingOptions().to_c()[0].detect_language == 0
    assert DecodingOptions(usePrefillPrompt=False).to_c()[0].detect_language == 1        # detectLanguage ?? !usePrefillPrompt
    assert DecodingOptions(usePrefillPrompt=False, detectLanguage=False).to_c()[0].detect_language == 0
    assert DecodingOptions(detectLanguage=True).to_c()[0].detect_language == 1


class _FakeDecoder:
    """predict_logits over a toy vocabulary: at position 0 the language logits follow `lang_pref`, later positions favour EOT after a few
    tokens; every call is logged."""

    def __init__(self, st, V, lang_pref):
        self.st, self.V, self.lang_pref, self.calls = st, V, lang_pref, []

    def __call__(self, tok, idx):
        self.calls.append((tok, idx))
        x = np.full(self.V, -5.0, np.float32)
        if idx == 0:
            for t, v in self.lang_pref.items():
                x[t] = v
        x[5 + (idx % 7)] = 3.0
        if idx >= 6:
            x[self.st.endToken] = 10.0
        return x


def test_decode_with_fallback_detects_and_reprefills():
    st = D.SpecialTokens.toy(128)
    langs = [st.englishToken, 40, 7]
    fake = _FakeDecoder(st, 128, {40: 2.0, st.englishToken: 1.0, 7: 0.5})
    o = D.DecodingOptions(firstTokenLogProbThreshold=None, logProbThreshold=None, compressionRatioThreshold=None, withoutTimestamps=True,
                          temperatureFallbackCount=0)
    res, (tok, lp) = LR.decode_with_fallback(fake, o, st, True, langs, detectLanguage=True)
    assert tok == 40 and res.tokens[:2] == [st.startOfTranscriptToken, 40]           # decoded in the detected language
    want = 2.0 - np.log(np.exp(2.0) + np.exp(1.0) + np.exp(0.5))
    assert abs(lp - want) < 1e-5
    assert fake.calls[0] == (st.startOfTranscriptToken, 0) and fake.calls[1] == (st.startOfTranscriptToken, 0)
    # an explicit language is never detected; without detection the language comes from the tokens, else English
    fake.calls.clear()
    _, lang = LR.decode_with_fallback(fake, o, st, True, langs, languageToken=7, detectLanguage=True)
    assert lang == (7, 0.0) and [i for _, i in fake.calls].count(0) == 1
    res2, lang2 = LR.decode_with_fallback(fake, o, st, True, langs, detectLanguage=False)
    assert lang2 == (st.englishToken, res2.tokenLogProbs[1])                         # the prompt's <|en|> is the first language token
    res3, lang3 = LR.decode_with_fallback(fake, o, st, True, [41], detectLanguage=False)
    assert lang3 == (st.englishToken, 0.0)
    # English-only model: no detection even when asked
    _, lang4 = LR.decode_with_fallback(fake, o, st, False, langs, detectLanguage=True)
    assert lang4[0] != 40


def test_decode_with_fallback_detects_again_at_every_rung():
    st = D.SpecialTokens.toy(128)
    langs = [st.englishToken, 40, 7]
    fake = _FakeDecoder(st, 128, {40: 2.0, st.englishToken: 1.9, 7: 1.8})
    o = D.DecodingOptions(firstTokenLogProbThreshold=None, logProbThreshold=1.0, compressionRatioThreshold=None, withoutTimestamps=True,
                          temperatureFallbackCount=3, topK=3)
    res, (tok, _) = LR.decode_with_fallback(fake, o, st, True, langs, detectLanguage=True, rng=np.random.default_rng(5))
    assert [t for t, i in fake.calls if i == 0].count(st.startOfTranscriptToken) == 2 * 4       # detection + decode per rung
    assert abs(res.temperature - LR.rung_temperatures(o)[-1]) < 1e-3 and res.tokens[1] == tok  # kept = last rung, in its own language
    assert LR.rung_temperatures(o) == [0.0, float(np.float16(0.2)), float(np.float16(np.float16(2) * np.float16(0.2))),
                                       float(np.float16(np.float16(3) * np.float16(0.2)))]


def test_stream_language_first_versus_last_window():
    en = 2
    units = [[(10, -0.1), (11, -0.2), (12, -0.3)], [(13, -0.4)]]
    assert LR.stream_language(units, detecting=True, englishToken=en) == (12, -0.3)     # detectedLanguage reassigned every window
    assert LR.stream_language(units, detecting=False, englishToken=en) == (10, -0.1)    # set once, by the first window
    assert LR.stream_language([[], [(13, -0.4)]], detecting=True, englishToken=en) == (en, 0.0)
    assert LR.stream_language([], detecting=False, englishToken=en) == (en, 0.0)
