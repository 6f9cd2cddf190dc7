#!/usr/bin/env python
"""bench.py - RTFx (audio-seconds per second) of the WhisperKit hot path on B200.

One "step" = one pass of the whole hot path (PCM -> log-mel -> encoder -> cross-KV -> KV-cached greedy decode with
TimestampRules filter + sampler -> token IDs) over one batch of synthetic 30 s windows, whisper-large-v3 shapes,
seeded random weights (no checkpoints offline), bf16 storage / f32 accumulate.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # own arm (CUDA engine, libwkb200.so)
  python bench.py --impl reference [--steps K] [--warmup W]      # CPU restatement of the reference pipeline
  torchrun --nproc-per-node N bench.py --gpus N ...              # one rank per GPU (weak scaling: B windows per GPU)
  python bench.py ... --dump-outputs DIR                         # also write the last timed step's per-window results to DIR/*.npy

`value`  : device-timed RTFx with the PCM already resident in HBM.
`e2e`    : the same metric through the public API with HOST buffers: pinned PCM -> (N>1: NCCL scatter) -> GPU ->
           token IDs -> (N>1: NCCL gather) -> host, copies inside the timed region.
`roofline`: the dominant kernel (chosen by measured share of the step), timed live with CUDA events on the
           library stream, against MEASURED_PEAKS.json.
`cpu_baseline`: the CPU oracle (a restatement of the reference's scheduling: one decoder call per token, batch 1)
           on the host cores, on one 30 s window of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

AUDIO_SECONDS_PER_WINDOW = 30.0
_T0 = time.perf_counter()


def log(msg):
    sys.stderr.write(f"[bench +{time.perf_counter() - _T0:7.1f}s] {msg}\n")
    sys.stderr.flush()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--variant", default="large-v3")
    ap.add_argument("--batch", type=int, default=64, help="30 s windows per GPU per step")
    ap.add_argument("--sample-length", type=int, default=224, help="DecodingOptions.sampleLength (reference default 224)")
    ap.add_argument("--dtype", default="bf16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-second-dtype", action="store_true", help="skip the extra timed passes under the other 16-bit storage policy")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--cpu-windows", type=int, default=1)
    ap.add_argument("--profile-pass", action="store_true", help="one untimed pass of the hot path and exit (for ncu)")
    ap.add_argument("--windows", type=int, default=0, help="30 s windows per GPU per step (default: --batch, i.e. one window per decode slot)")
    ap.add_argument("--eot-profile", action="store_true",
                    help="windows end at their own length: per-window sampleLength drawn (seeded) from a speech-like distribution instead of "
                         "the worst-case 223 steps for every window; with --windows > --batch the freed slots take the next windows")
    ap.add_argument("--encoder-chunk", type=int, default=0, help="windows per mel+encoder pass (default: the model's max_batch)")
    ap.add_argument("--enc-batch", type=int, default=0, help="mel/encoder workspace size in windows (default: min(--batch, windows, 64))")
    ap.add_argument("--beam", type=int, default=1, help="beam search width (BASELINE configs[2]: 5); --batch counts decode ROWS, windows in flight = batch / beam")
    ap.add_argument("--longform", action="store_true",
                    help="BASELINE configs[4] shape: long audio streams through wk_transcribe_streams (seek loop per stream, all streams share the "
                         "GPU batches), word timestamps on; --streams per GPU, --stream-seconds each")
    ap.add_argument("--streams", type=int, default=16)
    ap.add_argument("--stream-seconds", type=float, default=300.0)
    ap.add_argument("--no-word-timestamps", action="store_true")
    ap.add_argument("--chunking", default="vad", choices=["vad", "none"],
                    help="long-form: 'vad' = chunkingStrategy .vad (every stream is cut into independent <= 30 s chunks, WhisperKit.swift:878-911: the "
                         "'chunked to 30 s windows' of BASELINE configs[4]); 'none' = one sequential seek loop per stream")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the per-window decode results of the last device-resident step as DIR/<field>.npy "
                         "(float32 / float64, at most 64 MB in all) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "own" or args.longform or args.profile_pass):
        ap.error("--dump-outputs covers the windowed GPU path only (not --impl reference, --longform or --profile-pass)")
    return args


def eot_profile_lengths(n: int, seed: int = 4321) -> np.ndarray:
    """Decoder steps per 30 s window for the --eot-profile mode.  No checkpoint is available offline, so the lengths come from a seeded
    log-normal fit of what 30 s of speech turns into with Whisper's tokenizer (4 prompt tokens + ~2.5 words/s x ~1.3 tokens/word plus
    timestamp pairs: median ~95 tokens), with 8 % near-silent windows, clipped to [6, 223]."""
    rng = np.random.default_rng(seed)
    x = np.exp(rng.normal(np.log(95.0), 0.45, size=n))
    silent = rng.random(n) < 0.08
    x[silent] = rng.integers(6, 20, size=n)[silent]
    return np.clip(np.round(x), 6, 223).astype(np.int64)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                    "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured"}
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=5)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def synthetic_windows(first_idx: int, n: int) -> np.ndarray:
    from whisperkit_b200.synthetic import synthetic_pcm
    return np.stack([synthetic_pcm(first_idx + i) for i in range(n)])


def special_tokens_for(vocab: int):
    import whisperkit_b200 as wk
    if vocab == 51866:
        return wk.SpecialTokens(endToken=50257, englishToken=50259, noSpeechToken=50363, noTimestampsToken=50364,
                                specialTokenBegin=50257, startOfPreviousToken=50362, startOfTranscriptToken=50258,
                                timeTokenBegin=50365, transcribeToken=50360, translateToken=50359)
    if vocab == 51864:
        return wk.SpecialTokens(endToken=50256, englishToken=50258, noSpeechToken=50361, noTimestampsToken=50362,
                                specialTokenBegin=50256, startOfPreviousToken=50360, startOfTranscriptToken=50257,
                                timeTokenBegin=50363, transcribeToken=50358, translateToken=50357)
    return wk.SpecialTokens()


# ------------------------------------------------------------------------------------------------ CPU restatement
_ORACLE_CACHE = {}


def cpu_restatement(variant: str, sample_length: int, n_windows: int, threads: int, first_idx: int = 0):
    """Times the CPU oracle: log-mel + fp32 Whisper + the reference's decode loop (one decoder call per token,
    batch 1 per stream - exactly how the reference schedules CoreML).  Returns (rtfx, seconds, steps, threads_used).
    The encoder runs on all `threads`; the token loop (GEMV-sized ops) runs on the thread count that a short
    calibration finds fastest (intra-op parallelism over >32 threads slows M=1 decoding down)."""
    import torch
    from oracle import decode_ref as D, mel_ref, model_ref as M
    dims = M.VARIANTS[variant]
    if variant not in _ORACLE_CACHE:  # weight generation (1.5 G parameters for large-v3) is setup, not timed work
        log(f"CPU restatement: generating {variant} fp32 weights")
        torch.set_num_threads(min(threads, 32))
        orc = M.WhisperOracle(dims, M.random_weights(dims, seed=1234, policy="fp32", pool_size=1 << 24), "fp32")
        cands = sorted({t for t in (4, 8, 16, 32, 64, threads) if t <= threads})
        best, best_t = cands[0], float("inf")
        with torch.no_grad():
            enc = torch.zeros(1, dims.n_audio_ctx, dims.d_model)
            cross = orc.cross_kv(enc)
            for t in cands:
                torch.set_num_threads(t)
                cache = orc.new_cache(1)
                t0 = time.perf_counter()
                orc.decode_step(torch.tensor([1]), 0, cache, cross)
                if time.perf_counter() - t0 > 5 * best_t / 3 + 0.5:
                    log(f"  decode calibration: {t} threads slower than {best} - stopping")
                    break
                t0 = time.perf_counter()
                for i in range(1, 4):
                    orc.decode_step(torch.tensor([1]), i, cache, cross)
                dt = time.perf_counter() - t0
                log(f"  decode calibration: {t} threads -> {dt / 3 * 1000:.1f} ms/step")
                if dt < best_t:
                    best, best_t = t, dt
                elif dt > 2 * best_t:
                    break
            # encoder-sized work (one layer's FFN on 1500 rows): same search, separately
            xx = torch.randn(1, dims.n_audio_ctx, dims.d_model)
            w1, w2 = orc.w["model.encoder.layers.0.fc1.weight"], orc.w["model.encoder.layers.0.fc2.weight"]
            ebest, ebest_t = cands[0], float("inf")
            for t in cands:
                torch.set_num_threads(t)
                t0 = time.perf_counter()
                for _ in range(2):
                    torch.nn.functional.linear(torch.nn.functional.gelu(torch.nn.functional.linear(xx, w1)), w2)
                dt = time.perf_counter() - t0
                log(f"  encoder calibration: {t} threads -> {dt / 2 * 1000:.1f} ms/FFN")
                if dt < ebest_t:
                    ebest, ebest_t = t, dt
                elif dt > 2 * ebest_t:
                    break
        _ORACLE_CACHE[variant] = (orc, best, ebest)
    orc, dec_threads, enc_threads = _ORACLE_CACHE[variant]
    threads = enc_threads
    st = D.SpecialTokens.large_v3() if dims.vocab == 51866 else (D.SpecialTokens.english_only() if dims.vocab == 51864 else D.SpecialTokens())
    opts = D.DecodingOptions(firstTokenLogProbThreshold=None, sampleLength=sample_length)
    multilingual = dims.vocab != 51864
    prompt = D.prefill_prompt(opts, st, multilingual)
    pcm = synthetic_windows(first_idx, n_windows)
    steps = 0
    t0 = time.perf_counter()
    with torch.no_grad():
        for i in range(n_windows):
            torch.set_num_threads(threads)
            mel = mel_ref.log_mel(pcm[i], dims.n_mels, dtype=np.float32).astype(np.float16).astype(np.float32)
            enc = orc.encode(torch.from_numpy(mel)[None])
            cross = orc.cross_kv(enc)
            cache = orc.new_cache(1)
            torch.set_num_threads(dec_threads)

            def predict(tok, idx):
                return orc.decode_step(torch.tensor([tok]), idx, cache, cross)[0].numpy()

            r = D.decode_text(predict, prompt, opts, st, multilingual)
            steps += r.steps
    dt = time.perf_counter() - t0
    return n_windows * AUDIO_SECONDS_PER_WINDOW / dt, dt, steps, (threads, dec_threads)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    metric = "RTFx (audio-sec/s) whisper-large-v3 greedy" if args.variant == "large-v3" else f"RTFx (audio-sec/s) whisper-{args.variant} greedy"
    times = []
    warm = min(args.warmup, 1)  # CPU warm-up = first-touch of the weights; one pass is enough
    for i in range(warm):
        cpu_restatement(args.variant, args.sample_length, args.cpu_windows, threads)
    done = 0
    used = (threads, threads)
    for i in range(args.steps):
        rtfx, dt, _, used = cpu_restatement(args.variant, args.sample_length, args.cpu_windows, threads, first_idx=i)
        log(f"reference step {i}: {dt:.1f} s")
        times.append(dt)
        done += 1
    total = sum(times)
    value = done * args.cpu_windows * AUDIO_SECONDS_PER_WINDOW / total
    line = {
        "impl": "reference", "metric": metric, "value": value, "unit": "audio-sec/s", "n_gpus": args.gpus, "steps": done,
        "warmup": warm, "ms_per_step": 1000.0 * total / done, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic 16 kHz PCM, seeded random weights",
        "config": {"workload": f"whisper-{args.variant} greedy, {args.cpu_windows} x 30 s window per step (bounded CPU sample of the "
                               f"batch={args.batch} x 30 s GPU workload), sampleLength={args.sample_length}, timestamps on",
                   "sample_length": args.sample_length},
        "cpu_baseline": {"value": value, "unit": "audio-sec/s", "cores": max(used), "host_cores": threads, "kind": "port",
                         "sample": f"{args.cpu_windows} window(s) x 30 s per step, full pipeline, fp32 PyTorch CPU restatement of the "
                                   f"WhisperKit pipeline (the Swift/CoreML reference cannot run on Linux); encoder on {used[0]} "
                                   f"threads, token loop on {used[1]} threads (calibrated fastest)"},
        "e2e": {"value": value, "unit": "audio-sec/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ own arm
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, res, first_window: int, limit: int = DUMP_LIMIT_BYTES, suffix: str = "") -> None:
    """Writes what a caller of wk_transcribe_windows_ex receives (one wk_decode_result per window) as out_dir/<field><suffix>.npy,
    one row per window, plus window_index (the window's number in the seeded PCM sequence).  Integer fields are stored as float64
    (exact), float fields as float32.  Token slots past a window's n_tokens are not written by the library, so they are stored as
    -1 (ids) and 0 (log-probs).  When the whole output exceeds `limit` bytes, a fixed seeded sample of windows is written."""
    a = np.ctypeslib.as_array(res).copy()
    n = len(a)
    valid = np.arange(a.dtype["tokens"].shape[0])[None, :] < a["n_tokens"][:, None]
    fields = {"window_index": np.arange(first_window, first_window + n, dtype=np.float64)}
    for name in a.dtype.names:
        v = a[name]
        if name == "tokens":
            v = np.where(valid, v, -1)
        elif name == "token_logprobs":
            v = np.where(valid, v, 0)
        fields[name] = v.astype(np.float32 if v.dtype.kind == "f" else np.float64)
    row_bytes = sum(v.nbytes // n for v in fields.values())
    if n * row_bytes > limit:
        keep = np.sort(np.random.default_rng(0).choice(n, limit // row_bytes, replace=False))
        fields = {k: v[keep] for k, v in fields.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, v in fields.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), v)
    log(f"wrote {len(fields)} arrays ({len(fields['window_index'])} of {n} windows) to {out_dir}")


def run_own_arm(args):
    import torch
    import whisperkit_b200 as wk
    from whisperkit_b200._lib import check, wk_decode_result
    from whisperkit_b200.api import make_batch_opts

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    B = args.batch                       # decode slots per GPU
    W = args.windows or B                # windows per GPU per step
    beam = max(1, args.beam)
    enc_batch = args.enc_batch or min(B, W, 64)
    log(f"rank {rank}/{world}: creating model {args.variant}: encoder workspace {enc_batch} windows, {B} decode rows" + (f", beam {beam}" if beam > 1 else ""))
    model = wk.Model(args.variant, device=local_rank, max_batch=enc_batch, dtype=args.dtype)
    model.init_random(seed=1234)
    dec = wk.TextDecoder(model, B)
    log("model + session ready; generating synthetic PCM")
    lib = model.lib
    info = model.info
    st = special_tokens_for(info.vocab)
    # one greedy pass per window: with random-init weights avgLogProb is always below logProbThreshold, so the temperature
    # fallback ladder (retries, not part of the metric) is switched off; the CPU arm decodes one pass as well
    base = dict(firstTokenLogProbThreshold=None, temperatureFallbackCount=0, beamSize=beam)
    if args.eot_profile:
        lens = eot_profile_lengths(world * W)[rank * W:(rank + 1) * W]
        opts = [wk.DecodingOptions(sampleLength=int(v), **base) for v in lens]
        expected_steps = int(lens.sum())
    else:
        opts = wk.DecodingOptions(sampleLength=args.sample_length, **base)
        expected_steps = W * min(args.sample_length, 223)
    st_c = st.to_c()
    bo, keep = make_batch_opts(W, opts, None, encoderChunk=args.encoder_chunk)
    res = (wk_decode_result * W)()
    ext = torch.cuda.ExternalStream(model.stream, device=torch.device("cuda", local_rank))

    pcm_np = synthetic_windows(rank * W, W)
    pcm_host = torch.from_numpy(pcm_np).pin_memory()
    pcm_dev = pcm_host.cuda(non_blocking=False)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def transcribe(ptr, n, result_array, batch_opts):
        check(lib.wk_transcribe_windows_ex(model.handle, dec.handle, C.c_void_p(ptr), n, 480000, None, C.byref(st_c), C.byref(batch_opts), result_array))

    def step_device():
        transcribe(pcm_dev.data_ptr(), W, res, bo)

    # e2e: host PCM in, token IDs on the host out.  N > 1: rank 0 owns all N*W windows in pinned memory, copies them
    # to its GPU, NCCL scatters shards over NVLink, every rank transcribes, NCCL gathers token IDs back to rank 0.
    e2e_stages = {}
    if world > 1:
        # the edges run inside libwkb200 (csrc/comm.cu: ncclSend / ncclRecv); torch.distributed only carried the NCCL id
        from whisperkit_b200 import distributed as WD
        comm = WD.Comm(lib, rank, world, local_rank)
        all_host = torch.from_numpy(synthetic_windows(0, world * W)).pin_memory() if rank == 0 else None
        shard_dev = torch.empty(W, 480000, dtype=torch.float32, device=torch.device("cuda", local_rank))
        all_res = (wk_decode_result * (world * W))() if rank == 0 else None
    d2h_bytes = W * (224 * 8 + 16)

    def step_e2e():
        if world == 1:
            transcribe(pcm_host.data_ptr(), W, res, bo)
            return
        t0 = time.perf_counter()
        comm.scatter_windows(all_host.data_ptr() if rank == 0 else None, world * W, 480000, shard_dev.data_ptr())
        t1 = time.perf_counter()
        transcribe(shard_dev.data_ptr(), W, res, bo)
        t2 = time.perf_counter()
        comm.gather_results(res, W, world * W, all_res)
        t3 = time.perf_counter()
        for k, v in (("scatter_h2d_send", t1 - t0), ("transcribe", t2 - t1), ("gather_d2h", t3 - t2)):
            e2e_stages[k] = e2e_stages.get(k, 0.0) + v * 1000.0
        e2e_stages["_calls"] = e2e_stages.get("_calls", 0) + 1
        if rank == 0:
            assert all_res[world * W - 1].n_tokens > 0

    def timed(fn, steps, warmup, sample_clocks):
        for _ in range(warmup):
            fn()
        e2e_stages.clear()      # per-stage wall clock of the timed calls only (the first call also builds the NCCL communicator's channels)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler = ClockSampler(local_rank) if sample_clocks else None
        lib.wk_kernel_launch_count(1)
        if sampler:
            sampler.__enter__()
        e0.record(ext)
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        e1.record(ext)
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1000.0
        if sampler:
            sampler.__exit__()
        ms = max(e0.elapsed_time(e1), 0.0)
        launches = int(lib.wk_kernel_launch_count(0))
        if world > 1:
            t = torch.tensor([ms, wall_ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall_ms = float(t[0].item()), float(t[1].item())
            lt = torch.tensor([launches], device="cuda", dtype=torch.int64)
            dist.all_reduce(lt, op=dist.ReduceOp.SUM)
            launches = int(lt.item())
        return ms, launches, (sampler.summary() if sampler else None), wall_ms

    log("PCM ready; first (untimed) pass")
    t_first = time.perf_counter()
    step_device()
    log(f"first pass took {time.perf_counter() - t_first:.2f} s, stage ms {model.last_timings()}")
    if args.profile_pass:
        step_device()
        log(f"profile pass done, launches {int(lib.wk_kernel_launch_count(0))}")
        return
    ms, launches, clocks, _ = timed(step_device, args.steps, max(args.warmup, 3), True)
    log(f"device-resident arm: {ms / args.steps:.1f} ms/step")
    if args.dump_outputs:   # before the e2e and other-dtype passes reuse `res`
        dump_outputs(args.dump_outputs, res, rank * W, DUMP_LIMIT_BYTES // world, f"_rank{rank}" if world > 1 else "")
    steps_run = [r.steps for r in res]
    timings = model.last_timings()
    # the e2e region ends when the token IDs are on the host: the library call returns with them, so the wall clock of the calls is the
    # honest end (the event on the model stream cannot see the session's streams)
    ms_e2e, _, _, wall_e2e = timed(step_e2e, args.steps, 1, False)
    log(f"e2e arm: {ms_e2e / args.steps:.1f} ms/step")
    audio = world * W * AUDIO_SECONDS_PER_WINDOW * args.steps
    value = audio / (ms / 1000.0)
    e2e_value = audio / (ms_e2e / 1000.0)
    ms_per_step = ms / args.steps
    name = "whisper-large-v3" if args.variant == "large-v3" else f"whisper-{args.variant}"
    cfg_name = {"large-v3": "BASELINE configs[1]", "large-v3-turbo": "BASELINE configs[3] shape, one GPU's share", "distil-large-v3": "distil decoder"}.get(args.variant, "")
    workload = (f"{name} greedy {args.dtype}, {W} x 30 s windows per GPU through {B} decode slots ({cfg_name}), DecodingOptions defaults except "
                f"firstTokenLogProbThreshold=nil and temperatureFallbackCount=0 (one greedy pass; random-init weights would otherwise always retry); ")
    if args.eot_profile:
        workload += (f"--eot-profile: per-window sampleLength from a seeded speech-like distribution (decode steps per window "
                     f"{min(steps_run)}..{max(steps_run)}, mean {sum(steps_run) / len(steps_run):.0f}); ended windows retire, freed slots take the next windows; ")
    else:
        workload += f"sampleLength={args.sample_length} (decode steps per window: {min(steps_run)}..{max(steps_run)} - the worst case: real speech ends at EOT far earlier); "
    workload += "timestamps on (TimestampRulesFilter active)"

    line = {
        "metric": f"RTFx (audio-sec/s) {name} greedy",
        "value": value, "unit": "audio-sec/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
        "data": f"synthetic 16 kHz PCM (seeded noise + gated tones), seeded random weights of the {args.variant} architecture",
        "config": {"workload": workload,
                   "windows_per_gpu": W, "decode_slots": B, "sample_length": args.sample_length, "decode_steps": max(steps_run),
                   "decode_steps_total_per_gpu": int(sum(steps_run)), "eot_profile": bool(args.eot_profile),
                   "parallelism": f"dp{world} (windows sharded, weights replicated)",
                   "l2": "inputs_larger_than_L2 (decoder weights + cross-KV of every live window streamed every step; no flush needed)",
                   "stage_ms": timings, "scheduler": dec.stats()},
        "e2e": {"value": e2e_value, "unit": "audio-sec/s", "h2d_bytes_per_step": world * W * 480000 * 4,
                "d2h_bytes_per_step": world * d2h_bytes, "ms_per_step": ms_e2e / args.steps,
                "wall_ms_per_step": wall_e2e / args.steps,
                "path": "wk_transcribe_windows_ex(host pinned PCM)" if world == 1 else
                        "wk_comm_scatter_windows (pinned host PCM on rank 0 -> ncclSend/ncclRecv) + wk_transcribe_windows_ex + wk_comm_gather_results"},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if world > 1 and e2e_stages:
        mine = torch.tensor([e2e_stages.get(k, 0.0) / max(1, e2e_stages.get("_calls", 1)) for k in ("scatter_h2d_send", "transcribe", "gather_d2h")], device="cuda")
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        if rank == 0:   # host wall clock per stage and rank, mean over the timed calls: where the end-to-end time goes
            line["e2e"]["stage_ms_per_rank"] = {k: [round(float(a[i]), 2) for a in allr] for i, k in enumerate(("scatter_h2d_send", "transcribe", "gather_d2h"))}
    assert sum(steps_run) <= expected_steps

    if rank == 0 and not args.no_roofline:
        peaks = measured_peaks()
        f = C.c_float()
        wk_ = C.c_double()
        kernels = {}
        L, Ld = info.enc_layers, info.dec_layers
        d, H = info.d_model, info.n_heads
        sched = dec.stats()                       # of the last step: decode steps launched, admissions ...
        nsteps = max(1, sched["steps"])
        live_frac = min(1.0, int(sum(steps_run)) / (nsteps * B))   # share of the slot-steps that carried a live window
        # kernel id -> (name, bound, launches per step of the workload)
        table = {
            0: ("decoder_cross_attention_kernel", "hbm", Ld * nsteps),
            1: (f"gemm_tcgen05_kernel[enc FC1+GELU M=B*1500,N={4 * d},K={d}]", "tensor", L * (W / B)),
            2: ("mel_pass1+pass2", "hbm", W / B),
            3: ("encoder_attention_tcgen05_kernel", "tensor", L * (W / B)),
            4: (f"gemm_tcgen05_kernel[dec QKV swap-AB N={3 * d},K={d},split-K] (L2-warm)", "hbm", 0),
            5: (f"gemm_tcgen05_kernel[enc QKV M=B*1500,N={3 * d},K={d}]", "tensor", L * (W / B)),
            9: ("decoder_self_attention_kernel[pos 100]", "hbm", Ld * nsteps),
            14: (f"gemm_tcgen05_kernel[dec d x d swap-AB split-K, HBM-cold] (x3 per layer)", "hbm", 3 * Ld * nsteps),
            15: (f"gemm_tcgen05_kernel[dec FC1 swap-AB split-K, HBM-cold]", "hbm", Ld * nsteps),
            16: (f"gemm_tcgen05_kernel[dec FC2 swap-AB split-K, HBM-cold]", "hbm", Ld * nsteps),
            17: (f"gemm_tcgen05_kernel[dec QKV swap-AB split-K, HBM-cold]", "hbm", Ld * nsteps),
            8: ("decoder_reduce_resid_ln_kernel (x3 per layer)", "hbm", 3 * Ld * nsteps),
        }
        for which, (kname, bound, per_step) in table.items():
            kb = min(B, enc_batch) if which in (1, 2, 3, 5) else B      # encoder-side kernels run on one encoder chunk
            if which in (1, 2, 3, 5):
                per_step = per_step * B / kb
            check(lib.wk_bench_kernel(model.handle, dec.handle, which, kb, 20 if which != 2 else 5, C.byref(f), C.byref(wk_)))
            t_ms, work = float(f.value), float(wk_.value)
            if bound == "hbm":
                ach, peak, unit = work / (t_ms * 1e-3) / 1e9, peaks["hbm_gbs"], "GB/s"
            else:
                ach, peak, unit = work / (t_ms * 1e-3) / 1e12, peaks["bf16_tflops"], "TFLOP/s"
            kernels[kname] = {"bound": bound, "ms": t_ms, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                              "algorithmic_work": work, "launches_per_step": per_step,
                              "share_of_step": per_step * t_ms * (live_frac if which in (0, 9) else 1.0) / ms_per_step}
        log("per-kernel timings done")
        traffic_file = os.path.join(ROOT, "profiles", "r02_traffic.json")
        tj = {}
        try:
            tj = json.load(open(traffic_file))
        except Exception:
            pass
        roles = tj.get("by_bench_kernel_prefix", {})
        for kname, k in kernels.items():   # DRAM bytes per launch from the committed ncu --set full captures (tools/ncu_traffic.py)
            ent = next((v for pre, v in roles.items() if kname.startswith(pre)), None)
            same_shape = args.variant in ("large-v3", "large-v3-turbo", "distil-large-v3") and (B == 64 or not kname.startswith("decoder"))
            k["traffic"] = ent["bytes"] if ent and same_shape else None
            if ent and same_shape and ent.get("tensor_pipe_pct") and k["bound"] == "tensor":
                k["ncu_tensor_pipe_pct"] = ent["tensor_pipe_pct"]
        dom = max(kernels.items(), key=lambda kv: kv[1]["share_of_step"])
        line["roofline"] = {"kernel": dom[0], "bound": dom[1]["bound"], "achieved": dom[1]["achieved"], "peak": dom[1]["peak"],
                            "unit": dom[1]["unit"], "frac": dom[1]["frac"], "traffic": dom[1]["traffic"],
                            "peak_source": peaks["source"] + " (MEASURED_PEAKS.json burst figures; kernel timed alone)",
                            "share_of_step": dom[1]["share_of_step"]}
        line["kernels"] = kernels
        # whole decode step against HBM: what one step MUST stream = decoder weights (tied embedding included) once + the cross K/V of
        # every live window + the self K/V read so far and the new rows written (SURVEY 8d "K6 decode step")
        V = info.vocab
        w_bytes = Ld * 12 * d * d * 2 + V * d * 2
        cross_bytes = Ld * 2 * 1500 * d * 2
        mean_pos = (max(steps_run) - 1) / 2.0
        self_bytes = Ld * (2 * mean_pos * d * 2 + 2 * d * 2)
        live = B * live_frac
        step_bytes = w_bytes + live * (cross_bytes + self_bytes)
        step_ms = timings["decodingLoop"] / max(1, nsteps)
        line["roofline_step"] = {"bound": "hbm", "bytes_per_step": step_bytes, "ms_per_decode_step": step_ms,
                                 "achieved": step_bytes / (step_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs_sustained"] if "hbm_gbs_sustained" in peaks else peaks["hbm_gbs"],
                                 "unit": "GB/s", "live_rows": live,
                                 "what": "decoder weights once + cross K/V and self K/V of the live windows, divided by the measured decode-loop time per step"}
        line["roofline_step"]["frac"] = line["roofline_step"]["achieved"] / line["roofline_step"]["peak"]
        enc_flops = W * (2 * info.n_mels * 3 * d * 3000 + 2 * d * 3 * d * 1500 + L * (8 * 1500 * d * d + 4 * 1500 * 1500 * d + 16 * 1500 * d * d))
        line["roofline_encoder"] = {"bound": "tensor", "flops": enc_flops, "ms": timings["encoding"],
                                    "achieved": enc_flops / (timings["encoding"] * 1e-3) / 1e12 if timings["encoding"] else None,
                                    "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s"}
        if line["roofline_encoder"]["achieved"]:
            line["roofline_encoder"]["frac"] = line["roofline_encoder"]["achieved"] / peaks["bf16_tflops_sustained"]

    if world == 1 and not args.no_second_dtype and not args.eot_profile and beam == 1 and args.dtype in ("bf16", "f16"):
        # the same workload under the other storage policy.  BASELINE names bf16; the reference itself is Float16 end to end
        # (ArgmaxCore/FloatType.swift:9-13) and only f16 meets north_star's 1e-3 logits tolerance (tests/test_gpu_large.py: 7.1e-4 vs
        # 5.2e-3 for bf16 at 32 decoder layers), so both are timed here, device-resident PCM, same steps
        other = "f16" if args.dtype == "bf16" else "bf16"
        dec.close(); model.close()
        model2 = wk.Model(args.variant, device=local_rank, max_batch=enc_batch, dtype=other)
        model2.init_random(seed=1234)
        dec2 = wk.TextDecoder(model2, B)
        ext2 = torch.cuda.ExternalStream(model2.stream, device=torch.device("cuda", local_rank))

        def step2():
            check(lib.wk_transcribe_windows_ex(model2.handle, dec2.handle, C.c_void_p(pcm_dev.data_ptr()), W, 480000, None, C.byref(st_c), C.byref(bo), res))
        for _ in range(4):
            step2()
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(ext2)
        for _ in range(args.steps):
            step2()
        a1.record(ext2)
        torch.cuda.synchronize()
        ms2 = a0.elapsed_time(a1) / args.steps
        line["other_dtype"] = {"dtype": other, "value": W * AUDIO_SECONDS_PER_WINDOW / (ms2 / 1000.0), "unit": "audio-sec/s", "ms_per_step": ms2,
                               "steps": args.steps, "logits_rel_err_vs_oracle": {"f16": "7.1e-4 (meets 1e-3)", "bf16": "5.2e-3 (does not meet 1e-3)"},
                               "note": "same workload, device-resident PCM; parity figures from tests/test_gpu_large.py on B200"}
        log(f"{other}: {ms2:.1f} ms/step")
        dec2.close(); model2.close()

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        log(f"CPU restatement on {threads} threads")
        rtfx, dt, nst, used = cpu_restatement(args.variant, args.sample_length, args.cpu_windows, threads)
        log(f"CPU restatement: {dt:.1f} s")
        line["cpu_baseline"] = {"value": rtfx, "unit": "audio-sec/s", "cores": max(used), "host_cores": threads, "kind": "port",
                                "sample": f"{args.cpu_windows} window(s) x 30 s, full pipeline ({nst} decoder steps), {dt:.1f} s of CPU "
                                          "work; fp32 PyTorch CPU restatement of the WhisperKit pipeline (one decoder call per token, "
                                          f"batch 1; encoder on {used[0]} threads, token loop on {used[1]} threads) - the Swift/CoreML reference "
                                          "cannot run on Linux"}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ long-form arm
def synthetic_tokenizer(vocab: int, st):
    """A byte-level vocabulary of Whisper's size for the word-timestamp path (splitToWordTokens needs token strings; no tokenizer files are
    available offline): ids 0..255 the GPT-2 byte alphabet, then two-letter merges up to specialTokenBegin, then <|...|> specials."""
    from whisperkit_b200.tokenizer import WhisperTokenizer
    bs = list(range(33, 127)) + list(range(161, 173)) + list(range(174, 256))
    cs = bs[:]
    n = 0
    for b in range(256):
        if b not in bs:
            bs.append(b); cs.append(256 + n); n += 1
    alphabet = {b: chr(c) for b, c in zip(bs, cs)}
    sb = st.specialTokenBegin
    toks, ids, flags = [], [], []
    for b in range(256):
        toks.append(alphabet[b]); ids.append(b); flags.append(0)
    letters = " etaoinshrdlucmfwypvbgkqjxz"
    for i in range(256, sb):
        a, c, e = letters[(i * 7) % len(letters)], letters[(i * 3 + 1) % len(letters)], letters[(i // 27) % len(letters)]
        toks.append("".join(alphabet[ord(ch)] for ch in (a + c + e if i % 3 else a + c))); ids.append(i); flags.append(0)
    names = {st.endToken: "<|endoftext|>", st.startOfTranscriptToken: "<|startoftranscript|>", st.englishToken: "<|en|>", st.translateToken: "<|translate|>",
             st.transcribeToken: "<|transcribe|>", st.startOfPreviousToken: "<|startofprev|>", st.noSpeechToken: "<|nospeech|>",
             st.noTimestampsToken: "<|notimestamps|>"}
    for i in range(sb, vocab):
        toks.append(names.get(i, f"<|{(i - st.timeTokenBegin) * 0.02:.2f}|>" if i >= st.timeTokenBegin else f"<|lang{i}|>")); ids.append(i); flags.append(3)
    return WhisperTokenizer(tokens=toks, ids=ids, flags=flags)


def run_longform_arm(args):
    """BASELINE configs[4] shape on this rank's share: `--streams` long audio streams, each run through TranscribeTask.run's seek loop
    (windows of one stream are sequentially dependent; the streams share the GPU batches), word timestamps on (alignment heads -> DTW ->
    word timings on host threads).  One step = every stream transcribed once.  RTFx = audio seconds / time."""
    import torch
    import whisperkit_b200 as wk
    from whisperkit_b200._lib import check, wk_segment

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    B = args.batch
    model = wk.Model(args.variant, device=local_rank, max_batch=min(B, 64), dtype=args.dtype)
    model.init_random(seed=1234)
    dec = wk.TextDecoder(model, B)
    lib, info = model.lib, model.info
    st = special_tokens_for(info.vocab)
    words = not args.no_word_timestamps
    opts = wk.DecodingOptions(firstTokenLogProbThreshold=None, temperatureFallbackCount=0, sampleLength=args.sample_length, wordTimestamps=words,
                              logProbThreshold=None, compressionRatioThreshold=None, noSpeechThreshold=None)
    prompt = dec.prefillDecoderInputs(opts, st)
    tok = synthetic_tokenizer(info.vocab, st) if words else None
    hooks = tok.hooks() if words else None
    n_samples = int(args.stream_seconds * 16000)
    log(f"rank {rank}: generating {args.streams} synthetic streams of {args.stream_seconds:.0f} s")
    base = synthetic_windows(rank * 8, 8).reshape(-1)
    streams = []
    for i in range(args.streams):
        off = (i * 123457) % (len(base) - 16000)
        x = np.concatenate([base[off:], base[:off]])
        reps = int(np.ceil((n_samples + i * 8000) / len(x)))          # streams of slightly different lengths
        streams.append(np.ascontiguousarray(np.tile(x, reps)[: n_samples + i * 8000], dtype=np.float32))
    ptrs = (C.c_void_p * len(streams))(*[a.ctypes.data for a in streams])
    lens = (C.c_int64 * len(streams))(*[len(a) for a in streams])
    st_c = st.to_c()
    o_c, keep = opts.to_c()
    p_c = (C.c_int32 * len(prompt))(*prompt)
    ext = torch.cuda.ExternalStream(model.stream, device=torch.device("cuda", local_rank))
    stats = {}

    def step():
        h = C.c_void_p()
        check(lib.wk_transcribe_streams(model.handle, dec.handle, ptrs, lens, len(streams), C.byref(st_c), C.byref(o_c), p_c, len(prompt), None, 0,
                                        1.0, -1, 1 if args.chunking == "vad" else 0, C.byref(hooks) if hooks is not None else None, C.byref(h)))
        stats["windows"] = lib.wk_transcription_window_count(h)
        stats["segments"] = lib.wk_transcription_segment_count(h)
        stats["words"] = lib.wk_transcription_word_count(h)
        lib.wk_transcription_free(h)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    log("first (untimed) pass")
    t0 = time.perf_counter()
    step()
    log(f"first pass {time.perf_counter() - t0:.2f} s: {stats}")
    for _ in range(max(args.warmup, 3) - 1):
        step()
    barrier()
    lib.wk_kernel_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as sampler:
        e0.record(ext)
        for _ in range(args.steps):
            step()
        e1.record(ext)
        barrier()
    ms = e0.elapsed_time(e1)
    launches = int(lib.wk_kernel_launch_count(0))
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    audio_s = world * sum(len(a) for a in streams) / 16000.0 * args.steps
    value = audio_s / (ms / 1000.0)
    name = "whisper-large-v3" if args.variant == "large-v3" else f"whisper-{args.variant}"
    line = {
        "metric": f"RTFx (audio-sec/s) {name} long-form" + (" word-timestamps" if words else ""),
        "value": value, "unit": "audio-sec/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
        "data": f"synthetic 16 kHz PCM streams, seeded random weights of the {args.variant} architecture, synthetic byte-level vocabulary of Whisper's size",
        "config": {"workload": f"{name} long-form (BASELINE configs[4] shape, one GPU's share): {args.streams} streams x ~{args.stream_seconds:.0f} s per GPU through "
                               f"wk_transcribe_streams (chunking={args.chunking}: " + ("streams cut into independent <= 30 s VAD chunks" if args.chunking == "vad" else "one sequential seek loop per stream")
                               + f", {B} decode slots shared by all streams), wordTimestamps={words}, "
                               f"sampleLength={args.sample_length}, greedy, no temperature fallback; host PCM in, segments"
                               + (" + word timings" if words else "") + " out (this IS the end-to-end path)",
                   "streams_per_gpu": args.streams, "stream_seconds": args.stream_seconds, "decode_slots": B,
                   "windows_decoded_per_step": stats["windows"], "segments": stats["segments"], "words": stats["words"],
                   "l2": "inputs_larger_than_L2", "parallelism": f"dp{world} (streams sharded, weights replicated)"},
        "e2e": {"value": value, "unit": "audio-sec/s", "h2d_bytes_per_step": int(stats["windows"]) * 480000 * 4 * world,
                "d2h_bytes_per_step": int(stats["windows"]) * (224 * 8 + 16 + (224 * 1500 * 2 if words else 0)) * world, "ms_per_step": ms / args.steps,
                "path": "wk_transcribe_streams(host PCM) - the long-form entry has no device-resident variant"},
        "gpu_launches": launches, "clocks": sampler.summary(),
    }
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_JSON_OUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, on the process's original stdout."""
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    print(json.dumps(line), file=out, flush=True)


def main():
    global _JSON_OUT
    args = parse_args()
    # Libraries may write to file descriptor 1 (NCCL prints its version banner there when NCCL_DEBUG asks for it): keep the original
    # stdout for the JSON line only and send everything else written to fd 1 to stderr.
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.longform:
        run_longform_arm(args)
    else:
        run_own_arm(args)


if __name__ == "__main__":
    main()
