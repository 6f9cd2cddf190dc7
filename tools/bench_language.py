"""Cost of DecodingOptions.detectLanguage in the batched decode loop, on the GPU.

Workload: large-v3 dims with seeded random weights, 64 seeded 30 s windows, sampleLength 224 (the full context), one greedy pass per
window (temperature ladder off, first-token threshold off, as bench.py).  Four arms, alternated over the repeats:
  off          detection off (English prompt)
  sot          detection on, SOT-first prompts: the detection rides on step 0
  prompt       detection on, prompts with promptTokens (<|startofprev|> first): one pre-step per window
  two_pass     the host-side alternative: encode, bind, wk_detect_language, then wk_decode_text_ex with the per-window languages
Prints one JSON line: audio seconds per second per arm (median and spread over the repeats), the decoder passes per arm (steps launched
and row-passes, wk_session_stats), the card name and power limit read in the same run.

    python tools/bench_language.py [--repeats 5] [--windows 64] [--sample-length 224]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, limit = [v.strip() for v in out.split(",")]
        return name, limit
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--windows", type=int, default=64)
    ap.add_argument("--sample-length", type=int, default=224)
    args = ap.parse_args()
    import torch
    import whisperkit_b200 as wk
    from oracle import decode_ref as D
    from whisperkit_b200._lib import check, wk_decode_result
    from whisperkit_b200.api import make_batch_opts

    assert torch.cuda.is_available(), "bench_language.py measures on the GPU"
    W = args.windows
    model = wk.Model("large-v3", max_batch=W, dtype="bf16")
    model.init_random(seed=1234)
    dec = wk.TextDecoder(model, W)
    fe, enc = wk.FeatureExtractor(model), wk.AudioEncoder(model)
    lib = model.lib
    st = wk.SpecialTokens.from_any(D.SpecialTokens.large_v3())
    st_c = st.to_c()
    rng = np.random.default_rng(2024)
    pcm = torch.from_numpy((0.1 * rng.standard_normal((W, 480000))).astype(np.float32)).pin_memory()
    base = dict(firstTokenLogProbThreshold=None, temperatureFallbackCount=0, sampleLength=args.sample_length)
    prompt_tokens = [int(t) for t in rng.integers(100, 20000, size=8)]
    langs = list(range(st.startOfTranscriptToken + 1, min(st.translateToken, st.transcribeToken)))
    lang_arr = (C.c_int32 * len(langs))(*langs)
    res = (wk_decode_result * W)()

    def stats():
        s4 = (C.c_int64 * 4)()
        check(lib.wk_session_stats(dec.handle, s4))
        return int(s4[0]), int(s4[1])

    def windows_arm(opts):
        bo, keep = make_batch_opts(W, opts, None)

        def run():
            check(lib.wk_transcribe_windows_ex(model.handle, dec.handle, C.c_void_p(pcm.data_ptr()), W, 480000, None, C.byref(st_c),
                                               C.byref(bo), res))
            return stats()
        return run

    def two_pass():
        e = enc.encodeFeatures(fe.logMelSpectrogram(pcm))
        dec.bindEncoderOutput(e)
        tok = (C.c_int32 * W)()
        check(lib.wk_detect_language(dec.handle, C.byref(st_c), lang_arr, len(langs), 0.0, tok, None))
        opts = [wk.DecodingOptions(languageToken=int(tok[w]), **base) for w in range(W)]
        prompts = [dec.prefillDecoderInputs(o, st) for o in opts]
        bo, keep = make_batch_opts(W, opts, prompts)
        check(lib.wk_decode_text_ex(dec.handle, C.byref(st_c), C.byref(bo), res))
        steps, rows = stats()
        return steps + 1, rows + W   # + the detection pass

    arms = {
        "off": windows_arm(wk.DecodingOptions(**base)),
        "sot": windows_arm(wk.DecodingOptions(detectLanguage=True, **base)),
        "prompt": windows_arm(wk.DecodingOptions(detectLanguage=True, promptTokens=prompt_tokens, **base)),
        "two_pass": two_pass,
    }
    times = {k: [] for k in arms}
    passes = {}
    for k, fn in arms.items():   # warm-up: modules, graphs, workspaces
        fn()
    torch.cuda.synchronize()
    for _ in range(args.repeats):
        for k, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            passes[k] = fn()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    name, limit = card()
    audio_s = W * 30.0
    out = {"metric": "detect_language_cost", "card": name, "power_limit": limit, "variant": "large-v3", "windows": W,
           "sample_length": args.sample_length, "repeats": args.repeats, "arms": {}}
    for k, ts in times.items():
        rates = [audio_s / t for t in ts]
        out["arms"][k] = {"audio_s_per_s_median": round(float(np.median(rates)), 1), "audio_s_per_s_min": round(min(rates), 1),
                          "audio_s_per_s_max": round(max(rates), 1), "seconds": [round(t, 4) for t in ts],
                          "decode_steps": passes[k][0], "row_passes": passes[k][1]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
