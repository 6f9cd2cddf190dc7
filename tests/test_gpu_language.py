"""DecodingOptions.detectLanguage inside the batched decode loop (TranscribeTask.swift:339-365): the detection rides on step 0 of SOT-first
prompts and takes one pre-step for <|startofprev|> prompts.  Checked against the two-pass route (wk_detect_language, then a decode with
the detected language), against the oracle's decodeWithFallback on the GPU's own logits, and for cost in passes and launches."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import whisperkit_b200 as wk  # noqa: E402
from oracle import decode_ref as D  # noqa: E402
from oracle import language_ref as LR  # noqa: E402
from oracle import mel_ref  # noqa: E402

ST_O = D.SpecialTokens.toy(1024)
ST = wk.SpecialTokens.from_any(ST_O)
# English plus ids in the text and special ranges of the toy vocabulary (text < 512 <= special < 521 <= timestamps)
LANGS = [ST_O.englishToken, 517, 7, 300, 45]
FIELDS = ("tokens", "tokenLogProbs", "avgLogProb", "compressionRatio", "temperature", "fallback", "currentTokenCount", "steps",
          "isFirstTokenLogProbTooLow")


def kit_for(slots, seed=7, model="toy", st=ST, langs=LANGS):
    kit = wk.WhisperKit(wk.WhisperKitConfig(model=model, maxBatch=slots, seed=seed, specialTokens=st))
    if langs is not None:
        kit.textDecoder.setLanguageTokens(langs)
    return kit


def pcm_batch(n, base=70):
    return np.stack([mel_ref.synthetic_pcm(base + i) for i in range(n)])


def same(a, b):
    return all(getattr(a, f) == getattr(b, f) for f in FIELDS)


def base(**kw):
    d = dict(firstTokenLogProbThreshold=None, temperatureFallbackCount=0, sampleLength=16)
    d.update(kw)
    return wk.DecodingOptions(**d)


MIXED = [dict(detectLanguage=True), dict(detectLanguage=True, withoutTimestamps=True), dict(detectLanguage=True, promptTokens=[10, 11, 12]),
         dict(detectLanguage=True, promptTokens=[5], prefixTokens=[20, 21]), dict(detectLanguage=True, promptTokens=[9, 8], withoutTimestamps=True),
         dict(detectLanguage=True, prefixTokens=[30])]
QUIET = [dict(languageToken=517, detectLanguage=True), dict(detectLanguage=False, promptTokens=[4])]   # never detect


def detect_two_pass(kit, pcm, langs, st=ST):
    """wk_detect_language on the encoder output of the same windows (a separate session)."""
    n = len(pcm)
    dec = wk.TextDecoder(kit.model, n)
    e = kit.audioEncoder.encodeFeatures(kit.featureExtractor.logMelSpectrogram(pcm))
    tok, lp = dec.detectLanguage(e, st, langs)
    return dec, e, tok, lp


def check_equivalence(kit, pcm, opts, langs, st=ST, oracle=False):
    n = len(pcm)
    res = kit.transcribe(pcm, [base(**o) for o in opts])
    got = kit.textDecoder.languages(n)
    dec, e, tok, lp = detect_two_pass(kit, pcm, langs, st)
    for w, o in enumerate(opts):
        if o.get("detectLanguage") and "languageToken" not in o:
            assert got[w][0] == tok[w] and np.float32(got[w][1]) == np.float32(lp[w]), (w, got[w], tok[w], lp[w])
            assert res[w].languageToken == tok[w]
    # the second pass: every detecting window decoded with its detected language, detection off
    opts2 = [dict(o, languageToken=tok[w], detectLanguage=False) if o.get("detectLanguage") and "languageToken" not in o else o
             for w, o in enumerate(opts)]
    res2 = kit.transcribe(pcm, [base(**o) for o in opts2])
    for w in range(n):
        assert same(res[w], res2[w]), (w, res[w].tokens, res2[w].tokens)
    if oracle:   # the oracle's decodeWithFallback (detect, re-prefill, decode) on the GPU decoder's own logits
        dec.bindEncoderOutput(e)
        for w, o in enumerate(opts):
            ko = {k: v for k, v in o.items() if k in ("withoutTimestamps", "promptTokens", "prefixTokens")}
            oo = D.DecodingOptions(firstTokenLogProbThreshold=None, temperatureFallbackCount=0, sampleLength=16, **ko)

            def predict(t, i, w=w):
                return dec.predictLogits([t] * n, [i] * n)[w]
            r, lang = LR.decode_with_fallback(predict, oo, ST_O, True, langs, languageToken=o.get("languageToken"),
                                              detectLanguage=bool(o.get("detectLanguage")))
            assert r.tokens == res[w].tokens and lang[0] == got[w][0], (w, r.tokens, res[w].tokens, lang, got[w])
    dec.close()
    return res, got


def test_detection_equals_the_two_pass_route_and_the_oracle():
    """Tests 1-3: mixed prompts (SOT-first, <|startofprev|>, prefix, with / without timestamps) at T = 0; windows that do not detect in
    the same call are unaffected; the oracle loop on the GPU's logits agrees."""
    kit = kit_for(8)
    pcm = pcm_batch(8)
    check_equivalence(kit, pcm, MIXED + QUIET, LANGS, oracle=True)
    # no cross-talk: the quiet windows equal a call in which no window detects
    mixed = kit.transcribe(pcm, [base(**o) for o in MIXED + QUIET])
    none = kit.transcribe(pcm, [base(**dict(o, detectLanguage=False)) for o in MIXED] + [base(**o) for o in QUIET])
    for w in (6, 7):
        assert same(mixed[w], none[w])
    assert kit.textDecoder.languages(8)[6] == (517, 0.0)


def test_ladder_detects_at_every_rung():
    """Test 4: random weights walk the whole ladder; the kept rung's detection is in its prompt and among its top-k languages."""
    kit = kit_for(4, seed=6)
    pcm = pcm_batch(3, base=60)
    o = wk.DecodingOptions(firstTokenLogProbThreshold=None, sampleLength=10, compressionRatioThreshold=None, detectLanguage=True, seed=3, topK=2)
    res = kit.transcribe(pcm, o)
    langs = kit.textDecoder.languages(3)
    assert all(abs(r.temperature - 1.0) < 1e-3 for r in res)
    dec, e, _, _ = detect_two_pass(kit, pcm, LANGS)
    dec.bindEncoderOutput(e)
    lg = dec.predictLogits([ST.startOfTranscriptToken] * 3, [0] * 3)
    for w in range(3):
        assert res[w].tokens[1] == langs[w][0]
        top = sorted(LANGS, key=lambda t: -lg[w][t])[:o.topK]
        assert langs[w][0] in top
    res2 = kit.transcribe(pcm, o)
    assert all(same(a, b) for a, b in zip(res, res2)) and kit.textDecoder.languages(3) == langs
    dec.close()


def test_no_op_cases():
    """Test 5: an English-only model and an explicit language ignore the flag."""
    m = wk.WhisperKit(wk.WhisperKitConfig(model="tiny.en", maxBatch=2, seed=31))
    st_en = m.specialTokens
    pcm = pcm_batch(2, base=90)
    a = m.transcribe(pcm, base(detectLanguage=True))
    la = m.textDecoder.languages(2)
    b = m.transcribe(pcm, base(detectLanguage=False))
    assert all(same(x, y) for x, y in zip(a, b)) and la == m.textDecoder.languages(2)
    block = LR.default_language_tokens(ST_O.english_only())
    for r, (t, lp) in zip(a, la):
        first = next(((x, p) for x, p in zip(r.tokens, r.tokenLogProbs) if x in block), (st_en.englishToken, 0.0))
        assert (t, np.float32(lp)) == (first[0], np.float32(first[1]))
    kit = kit_for(2)
    pcm = pcm_batch(2)
    a = kit.transcribe(pcm, base(languageToken=300, detectLanguage=True))
    b = kit.transcribe(pcm, base(languageToken=300))
    assert all(same(x, y) for x, y in zip(a, b)) and kit.textDecoder.languages(2) == [(300, 0.0)] * 2


def test_beam_with_detection_is_rejected():
    kit = kit_for(8)
    with pytest.raises(wk.WhisperError) as ei:
        kit.transcribe(pcm_batch(1), base(beamSize=5, detectLanguage=True))
    assert ei.value.case == "invalidArgument"


def test_word_timestamps_after_a_pre_step():
    """Test 7: with promptTokens the pre-step leaves no alignment row; the tensor equals the two-pass run's."""
    kit = kit_for(4)
    pcm = pcm_batch(2, base=80)
    o = dict(detectLanguage=True, promptTokens=[10, 11], wordTimestamps=True)
    res = kit.transcribe(pcm, base(**o))
    langs = kit.textDecoder.languages(2)
    a = [kit.textDecoder.alignmentWeights(w, 224) for w in range(2)]
    res2 = kit.transcribe(pcm, [base(**dict(o, detectLanguage=False, languageToken=langs[w][0])) for w in range(2)])
    for w in range(2):
        assert same(res[w], res2[w])
        b = kit.textDecoder.alignmentWeights(w, 224)
        np.testing.assert_array_equal(a[w], b)
        assert np.all(a[w][0] == 0)


def test_streams_decode_each_window_in_its_own_language():
    """Test 8: wk_transcribe_streams, plain and VAD-chunked, against the oracle seek loop driven window by window through the same GPU
    decode; the per-stream language follows the first / last window rule."""
    from oracle import seek_ref as S
    from whisperkit_b200 import longform as L
    kit = kit_for(4, seed=9)
    for detect in (True, False):
        o = wk.DecodingOptions(firstTokenLogProbThreshold=None, logProbThreshold=None, compressionRatioThreshold=None, sampleLength=24,
                               temperatureFallbackCount=0, detectLanguage=detect)
        lens = [480000 * 2 + 12345, 300000, 0]
        streams = [np.concatenate([mel_ref.synthetic_pcm(400 + 10 * i + k) for k in range(3)])[:n].astype(np.float32) for i, n in enumerate(lens)]

        def oracle_stream(x):
            seen = []

            def decode_window(seek, size):
                w = np.zeros(480000, np.float32)
                w[:size] = x[seek:seek + size]
                r = kit.transcribe(w[None], o, samplesPerWindow=[size])[0]
                seen.append((r.languageToken, next(iter(r.languageProbs.values()))))
                if detect:
                    assert r.tokens[1] == r.languageToken          # decoded in its own detected language
                return r
            ref, _ = S.seek_loop(len(x), decode_window, timeToken=ST_O.timeTokenBegin, noSpeechThreshold=o.noSpeechThreshold,
                                 logProbThreshold=o.logProbThreshold)
            return ref, seen
        langs = []
        got, _ = L.transcribe_streams(kit, streams, o, languages=langs)
        for i, x in enumerate(streams):
            ref, seen = oracle_stream(x)
            assert [g.tokens for g in got[i]] == [r.tokens for r in ref]
            want = LR.stream_language([seen], detect, ST.englishToken)
            assert langs[i][0] == want[0] and np.float32(langs[i][1]) == np.float32(want[1]), (i, detect, langs[i], want)
        # VAD chunks: each chunk is a unit; the stream takes its first chunk's language
        x = streams[0].copy()
        x[500000:520000] = 0
        langs = []
        L.transcribe_streams(kit, [x], o, chunkingStrategy="vad", languages=langs)
        chunks = S.vad_chunk_all(x, 480000)
        units = [oracle_stream(x[a:b])[1] for a, b in chunks]
        want = LR.stream_language(units, detect, ST.englishToken)
        assert langs[0][0] == want[0] and np.float32(langs[0][1]) == np.float32(want[1])


def test_cost_in_passes_and_launches():
    """Test 9: SOT-first detection adds no decoder pass and no launch per step; a <|startofprev|> prompt adds one row-pass per window."""
    kit = kit_for(4)
    pcm = pcm_batch(4)
    lib = kit.model.lib

    def run(opts):
        lib.wk_kernel_launch_count(1)
        res = kit.transcribe(pcm, opts, callbackEvery=1)      # poll every step: the counters count single passes
        launches = lib.wk_kernel_launch_count(0)
        st4 = (C.c_int64 * 4)()
        wk._lib.check(lib.wk_session_stats(kit.textDecoder.handle, st4))
        return res, list(st4), launches, kit.textDecoder.languages(4)

    for extra, kw in ((0, {}), (1, dict(promptTokens=[10, 11, 12]))):
        run(base(**kw, detectLanguage=True))                  # warm: graphs captured
        r1, s1, l1, langs = run(base(**kw, detectLanguage=True))
        run([base(**kw, languageToken=t) for t, _ in langs])
        r2, s2, l2, _ = run([base(**kw, languageToken=t) for t, _ in langs])
        assert all(same(a, b) for a, b in zip(r1, r2))
        assert s1[1] - s2[1] == extra * 4 and s1[2:] == s2[2:]
        if extra == 0:
            assert s1[0] == s2[0] and l1 == l2


def test_large_v3_shape():
    """Test 10: large-v3 dims with the default 100-token language block, 64 windows; test 1's equalities."""
    st_o = D.SpecialTokens.large_v3()
    st = wk.SpecialTokens.from_any(st_o)
    kit = kit_for(64, model="large-v3", seed=1, st=st, langs=None)
    pcm = pcm_batch(64, base=500)
    opts = [dict(detectLanguage=True, sampleLength=24) if w % 4 else dict(detectLanguage=True, sampleLength=24, promptTokens=[100 + w, 200])
            for w in range(64)]
    check_equivalence(kit, pcm, opts, LR.default_language_tokens(st_o), st=st)
