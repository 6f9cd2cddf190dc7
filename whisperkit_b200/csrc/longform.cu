// Long-form windowing: the host-side logic around the hot path (SURVEY section 8f rows 1 and 3), in C++ because the
// reference's is compiled Swift.  Pure host code: every function except wk_transcribe_streams works without a GPU.
//   findSeekPointAndSegments   Sources/WhisperKit/Core/Text/SegmentSeeker.swift:41-189
//   prepareSeekClips           Sources/WhisperKit/Utilities/Extensions+Internal.swift:111-130
//   EnergyVAD / chunk helpers  Sources/WhisperKit/Core/Audio/{EnergyVAD,VoiceActivityDetector,AudioChunker}.swift
//   the seek loop              Sources/WhisperKit/Core/TranscribeTask.swift:98-279, batched over streams
#include <math.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <atomic>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "kernels.h"

using namespace wk;

static constexpr int kSampleRate = 16000;         // WhisperKit.sampleRate
static constexpr float kSecondsPerTimeToken = 0.02f;  // WhisperKit.secondsPerTimeToken
static constexpr int64_t kWindow = 480000;

extern "C" {

wk_status wk_find_seek_point_and_segments(const int32_t* tokens, const float* lps, int32_t n, float no_speech_prob, float avg_logprob,
                                          float compression_ratio, float temperature, const wk_decode_opts* o, int32_t all_segments_count,
                                          int64_t current_seek, int64_t segment_size, int32_t sample_rate, int32_t time_token,
                                          int64_t* new_seek, wk_segment* segs, int32_t cap, int32_t* n_segs) {
    if (!tokens || !lps || !o || !new_seek || !n_segs || n < 0) { set_error("wk_find_seek_point_and_segments: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    int64_t seek = current_seek;
    const float time_offset = (float)seek / (float)sample_rate;
    if (o->has_no_speech_threshold) {
        bool should_skip = no_speech_prob > o->no_speech_threshold;
        if (o->has_logprob_threshold && avg_logprob > o->logprob_threshold) should_skip = false;
        if (should_skip) { *new_seek = seek + segment_size; *n_segs = -1; return WK_OK; }
    }
    auto is_ts = [&](int i) { return tokens[i] >= time_token; };
    bool single_ts_ending = false, no_ts_ending = false;
    if (n >= 3) {
        single_ts_ending = !is_ts(n - 3) && is_ts(n - 2) && !is_ts(n - 1);
        no_ts_ending = !is_ts(n - 3) && !is_ts(n - 2) && !is_ts(n - 1);
    }
    std::vector<int> slices;
    bool prev = false;
    for (int i = 0; i < n; ++i) {
        const bool c = is_ts(i);
        if (prev && c) slices.push_back(i);
        prev = c;
    }
    int count = 0;
    auto emit = [&](int from, int to, float start, float end) -> bool {
        if (count >= cap || !segs) return false;
        wk_segment& g = segs[count];
        memset(&g, 0, sizeof(g));
        g.id = all_segments_count + count; g.seek = seek; g.start = start; g.end = end;
        g.token_offset = from; g.n_tokens = to - from;
        g.temperature = temperature; g.avg_logprob = avg_logprob; g.compression_ratio = compression_ratio; g.no_speech_prob = no_speech_prob;
        ++count;
        return true;
    };
    if (!slices.empty()) {
        if (single_ts_ending) {
            int last = -1;
            for (int i = 0; i < n; ++i) if (is_ts(i)) last = i;
            slices.push_back(last + 1);
        } else if (no_ts_ending) {
            slices.push_back(n);
        }
        int last_slice_start = 0;
        for (int end_i : slices) {
            int first_ts = -1, last_ts = -1;
            for (int i = last_slice_start; i < end_i; ++i)
                if (is_ts(i)) { if (first_ts < 0) first_ts = tokens[i]; last_ts = tokens[i]; }
            const float start_s = (float)(first_ts - time_token) * kSecondsPerTimeToken;
            const float end_s = (float)(last_ts - time_token) * kSecondsPerTimeToken;
            if (!emit(last_slice_start, end_i, time_offset + start_s, time_offset + end_s)) { set_error("segment capacity %d too small", cap); return WK_ERR_INVALID_ARGUMENT; }
            last_slice_start = end_i;
        }
        if (!no_ts_ending) {
            const int last_ts_token = tokens[last_slice_start - (single_ts_ending ? 1 : 0)] - time_token;
            const float last_ts_seconds = (float)last_ts_token * kSecondsPerTimeToken;
            seek += (int64_t)(last_ts_seconds * (float)sample_rate);
        } else {
            seek += segment_size;
        }
    } else {
        float duration = (float)segment_size / (float)sample_rate;
        int last_ts = -1;
        for (int i = 0; i < n; ++i) if (tokens[i] > time_token) last_ts = tokens[i];
        if (last_ts >= 0) duration = (float)(last_ts - time_token) * kSecondsPerTimeToken;
        if (!emit(0, n, time_offset, time_offset + duration)) { set_error("segment capacity %d too small", cap); return WK_ERR_INVALID_ARGUMENT; }
        seek += segment_size;
    }
    *new_seek = seek;
    *n_segs = count;
    return WK_OK;
}

wk_status wk_prepare_seek_clips(const float* ts, int32_t n, int64_t content_frames, int64_t* clips, int32_t cap, int32_t* n_clips) {
    if (!clips || !n_clips || n < 0 || (n > 0 && !ts)) { set_error("wk_prepare_seek_clips: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    std::vector<int64_t> pts;
    for (int i = 0; i < n; ++i) pts.push_back((int64_t)roundf(ts[i] * (float)kSampleRate));   // round(): half away from zero, like Swift
    if (pts.empty()) pts.push_back(0);
    if (pts.size() % 2 == 1) pts.push_back(content_frames);
    const int k = (int)pts.size() / 2;
    if (k > cap) { set_error("wk_prepare_seek_clips: capacity %d < %d", cap, k); return WK_ERR_INVALID_ARGUMENT; }
    for (int i = 0; i < k; ++i) { clips[2 * i] = pts[2 * i]; clips[2 * i + 1] = pts[2 * i + 1]; }
    *n_clips = k;
    return WK_OK;
}

static void vad_frames(const float* x, int64_t n, int frame_len, int overlap, float thr, std::vector<uint8_t>& out) {
    out.clear();
    if (n <= 0 || frame_len <= 0) return;
    const int64_t count = (n + frame_len - 1) / frame_len;
    for (int64_t i = 0; i < count; ++i) {
        const int64_t s = i * frame_len, e = std::min<int64_t>(s + frame_len + overlap, n);
        double acc = 0.0;
        for (int64_t j = s; j < e; ++j) acc += (double)x[j] * (double)x[j];
        const float rms = e > s ? (float)sqrt(acc / (double)(e - s)) : 0.f;   // vDSP_rmsqv
        out.push_back(rms > thr ? 1 : 0);
    }
}

wk_status wk_vad_voice_activity(const float* wav, int64_t n, int32_t frame_len, int32_t overlap, float thr, uint8_t* out, int64_t cap, int64_t* n_frames) {
    if ((n > 0 && !wav) || !n_frames || frame_len <= 0) { set_error("wk_vad_voice_activity: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    std::vector<uint8_t> v;
    vad_frames(wav, n, frame_len, overlap, thr, v);
    if ((int64_t)v.size() > cap) { set_error("wk_vad_voice_activity: capacity too small"); return WK_ERR_INVALID_ARGUMENT; }
    if (!v.empty()) memcpy(out, v.data(), v.size());
    *n_frames = (int64_t)v.size();
    return WK_OK;
}

static bool longest_silence(const uint8_t* vad, int64_t n, int64_t* start, int64_t* end) {
    int64_t best_s = -1, best_e = -1, best = 0, i = 0;
    while (i < n) {
        if (vad[i]) { ++i; continue; }
        int64_t e = i;
        while (e < n && !vad[e]) ++e;
        if (e - i > best) { best = e - i; best_s = i; best_e = e; }
        i = e;
    }
    *start = best_s; *end = best_e;
    return best_s >= 0;
}

wk_status wk_vad_find_longest_silence(const uint8_t* vad, int64_t n, int64_t* start, int64_t* end) {
    if ((n > 0 && !vad) || !start || !end) return WK_ERR_INVALID_ARGUMENT;
    longest_silence(vad, n, start, end);
    return WK_OK;
}

wk_status wk_vad_active_chunks(const float* wav, int64_t n, int32_t frame_len, int32_t overlap, float thr, int64_t* chunks, int32_t cap, int32_t* n_chunks) {
    if ((n > 0 && !wav) || !n_chunks || frame_len <= 0) return WK_ERR_INVALID_ARGUMENT;
    std::vector<uint8_t> v;
    vad_frames(wav, n, frame_len, overlap, thr, v);
    std::vector<int64_t> res;
    bool open = false;
    for (size_t i = 0; i < v.size(); ++i) {
        if (v[i]) {
            const int64_t s = (int64_t)i * frame_len, e = std::min<int64_t>(s + frame_len, n);
            if (open) res.back() = e;
            else { open = true; res.push_back(s); res.push_back(e); }
        } else {
            open = false;
        }
    }
    if ((int)res.size() / 2 > cap) { set_error("wk_vad_active_chunks: capacity too small"); return WK_ERR_INVALID_ARGUMENT; }
    for (size_t i = 0; i < res.size(); ++i) chunks[i] = res[i];
    *n_chunks = (int)res.size() / 2;
    return WK_OK;
}

static wk_status chunk_all(const float* wav, int64_t n, int64_t max_len, const float* cts, int n_cts, int64_t pad, int frame_len, int overlap,
                           float thr, std::vector<int64_t>& out) {
    out.clear();
    if (n <= max_len) { out.push_back(0); out.push_back(n); return WK_OK; }
    std::vector<int64_t> clips(2 * (n_cts / 2 + 2));
    int nc = 0;

    {
        wk_status st = wk_prepare_seek_clips(cts, n_cts, n, clips.data(), (int)clips.size() / 2, &nc);
        if (st != WK_OK) return st;
    }
    std::vector<uint8_t> v;
    for (int c = 0; c < nc; ++c) {
        int64_t start = clips[2 * c];
        const int64_t clip_end = clips[2 * c + 1];
        while (start < clip_end - pad) {
            if (start < 0 || start >= n) { set_error("startIndex is outside the buffer size"); return WK_ERR_AUDIO_PROCESSING_FAILED; }
            int64_t end = clip_end;
            if (start + max_len < end) {
                const int64_t e2 = std::min<int64_t>(n, start + max_len);
                const int64_t mid = start + (e2 - start) / 2;
                vad_frames(wav + mid, e2 - mid, frame_len, overlap, thr, v);
                int64_t ss, se;
                if (longest_silence(v.data(), (int64_t)v.size(), &ss, &se)) end = mid + (ss + (se - ss) / 2) * frame_len;
                else end = e2;
            }
            if (end <= start) break;
            out.push_back(start); out.push_back(end);
            start = end;
        }
    }
    return WK_OK;
}

wk_status wk_vad_chunk_all(const float* wav, int64_t n, int64_t max_chunk_len, const float* cts, int32_t n_cts, int64_t window_padding,
                           int32_t frame_len, int32_t overlap, float thr, int64_t* chunks, int32_t cap, int32_t* n_chunks) {
    if ((n > 0 && !wav) || !chunks || !n_chunks || frame_len <= 0 || max_chunk_len <= 0) { set_error("wk_vad_chunk_all: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    std::vector<int64_t> out;
    wk_status st = chunk_all(wav, n, max_chunk_len, cts, n_cts, window_padding, frame_len, overlap, thr, out);
    if (st != WK_OK) return st;
    if ((int)out.size() / 2 > cap) { set_error("wk_vad_chunk_all: capacity too small"); return WK_ERR_INVALID_ARGUMENT; }
    for (size_t i = 0; i < out.size(); ++i) chunks[i] = out[i];
    *n_chunks = (int)out.size() / 2;
    return WK_OK;
}

}  // extern "C"

// =====================================================================================================
// batched seek loop
// =====================================================================================================
struct OutWord {
    std::string word;
    std::vector<int32_t> tokens;
    float start, end, probability;
    int segment;
};

struct wk_transcription {
    std::vector<wk_segment> segments;
    std::vector<OutWord> words;   // .segment indexes `segments`
    std::vector<int32_t> tokens;
    std::vector<float> logprobs;
    int windows = 0;
    std::vector<int32_t> lang_tok;   // per stream: TranscriptionResult.language
    std::vector<float> lang_lp;
};

namespace {
struct Unit {                 // one independently advancing cursor: a stream, or one VAD chunk of a stream
    int stream;
    const float* audio;       // start of the unit's samples
    int64_t n;                // samples in the unit
    int64_t offset;           // unit start inside the stream (seekOffsetIndex)
    std::vector<int64_t> clips;
    int clip = 0;
    int64_t seek = 0;
    bool done = false;
    std::vector<wk_segment> segs;
    std::vector<OutWord> words;   // word timings; .segment indexes `segs`
    int windows = 0;
    int32_t lang_tok = -1; float lang_lp = 0.f;   // the unit's detectedLanguage (first or last window's, see wk_transcription_language)
};
}  // namespace

namespace {
constexpr int kRoundCap = 256;   // windows per round of the stream loop (host staging: 256 x 1.92 MB pinned)

// pinned host staging, kept for the life of the thread that transcribes (allocation of half a gigabyte of pinned memory costs ~0.1 s)
struct HostStage {
    float* pcm = nullptr; size_t pcm_bytes = 0;
    uint16_t* align = nullptr; size_t align_bytes = 0;
    wk_status ensure(size_t need_pcm, size_t need_align) {
        if (need_pcm > pcm_bytes) {
            if (pcm) cudaFreeHost(pcm);
            pcm = nullptr; pcm_bytes = 0;
            if (cudaHostAlloc((void**)&pcm, need_pcm, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); set_error("pinned staging of %zu bytes failed", need_pcm); return WK_ERR_CUDA; }
            pcm_bytes = need_pcm;
        }
        if (need_align > align_bytes) {
            if (align) cudaFreeHost(align);
            align = nullptr; align_bytes = 0;
            if (cudaHostAlloc((void**)&align, need_align, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); set_error("pinned staging of %zu bytes failed", need_align); return WK_ERR_CUDA; }
            align_bytes = need_align;
        }
        return WK_OK;
    }
    ~HostStage() { if (pcm) cudaFreeHost(pcm); if (align) cudaFreeHost(align); }
};
HostStage& host_stage() { static thread_local HostStage hs; return hs; }

// fn(i) for i in [0, n) on up to n_threads host threads; the first failing status wins, its thread-local message is handed back
template <typename F>
wk_status parallel_for(int n, int n_threads, F fn, std::string* err) {
    if (n <= 0) return WK_OK;
    const int nt = std::max(1, std::min(n_threads, n));
    if (nt == 1) {
        for (int i = 0; i < n; ++i) { wk_status r = fn(i); if (r != WK_OK) { if (err) *err = wk_last_error(); return r; } }
        return WK_OK;
    }
    std::atomic<int> next{0};
    std::atomic<int> status{WK_OK};
    std::mutex mu;
    auto work = [&]() {
        for (;;) {
            const int i = next.fetch_add(1);
            if (i >= n || status.load() != WK_OK) return;
            const wk_status r = fn(i);
            if (r != WK_OK) {
                std::lock_guard<std::mutex> lock(mu);
                if (status.load() == WK_OK) { status.store(r); if (err) *err = wk_last_error(); }
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; ++t) pool.emplace_back(work);
    work();
    for (auto& th : pool) th.join();
    return (wk_status)status.load();
}
}  // namespace

extern "C" {

wk_status wk_transcribe_streams(wk_model* m, wk_session* s, const float* const* audio, const int64_t* n_samples, int32_t n_streams,
                                const wk_special_tokens* st, const wk_decode_opts* o, const int32_t* prompt, int32_t n_prompt,
                                const float* cts, int32_t n_cts, float window_clip_time, int64_t max_window_seek, int32_t chunking_vad,
                                const wk_tokenizer_hooks* hooks, wk_transcription** out) {
    if (!m || !s || !audio || !n_samples || n_streams < 1 || !st || !o || !prompt || !out) { set_error("wk_transcribe_streams: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    if (o->word_timestamps && (!hooks || !hooks->split_to_word_tokens)) { set_error("wk_transcribe_streams: wordTimestamps needs the tokenizer's split_to_word_tokens hook"); return WK_ERR_INVALID_ARGUMENT; }
    wk_model_info info;
    wk_status rc = wk_model_info_get(m, &info);
    if (rc != WK_OK) return rc;
    const int max_batch = info.max_batch;
    const int64_t window_padding = (int64_t)(window_clip_time * (float)kSampleRate);
    std::vector<Unit> units;
    for (int i = 0; i < n_streams; ++i) {
        if (n_samples[i] < 0 || (n_samples[i] > 0 && !audio[i])) { set_error("wk_transcribe_streams: stream %d invalid", i); return WK_ERR_AUDIO_PROCESSING_FAILED; }
        std::vector<int64_t> chunks;
        // WhisperKit.transcribe(audioArray:) takes the VAD route only for (isChunkable, .vad) with isChunkable = count > windowSamples
        // (WhisperKit.swift:876-878); shorter audio goes to runTranscribeTask with the caller's options, clipTimestamps included (:912-919)
        const bool vad_stream = chunking_vad && n_samples[i] > kWindow;
        if (vad_stream) {
            // chunkingStrategy .vad (WhisperKit.swift:878-911): EnergyVAD defaults
            rc = chunk_all(audio[i], n_samples[i], kWindow, cts, n_cts, kSampleRate, 1600, 0, 0.02f, chunks);
            if (rc != WK_OK) return rc;
        } else {
            chunks = {0, n_samples[i]};
        }
        for (size_t c = 0; c + 1 < chunks.size(); c += 2) {
            Unit u;
            u.stream = i; u.audio = audio[i] + chunks[c]; u.n = chunks[c + 1] - chunks[c]; u.offset = chunks[c];
            // chunks are transcribed as whole arrays (clip timestamps were consumed by the chunker); plain streams use them directly
            u.clips.resize(2 * (n_cts / 2 + 2));
            int nc = 0;
            rc = wk_prepare_seek_clips(vad_stream ? nullptr : cts, vad_stream ? 0 : n_cts, u.n, u.clips.data(), (int)u.clips.size() / 2, &nc);
            if (rc != WK_OK) return rc;
            u.clips.resize(2 * nc);
            // a clip is live while seek < clipEnd - windowPadding (TranscribeTask.swift:118) and, as a guard the reference lacks (it would
            // pad a negative-length window), while the seek is still inside the audio
            u.seek = u.clips[0];
            u.done = !(u.seek < u.clips[1] - window_padding && u.seek < u.n);
            while (u.done && u.clip + 1 < nc) { ++u.clip; u.seek = u.clips[2 * u.clip]; u.done = !(u.seek < u.clips[2 * u.clip + 1] - window_padding && u.seek < u.n); }
            units.push_back(std::move(u));
        }
    }
    wk_transcription* T = new wk_transcription();
    // One round = the next window of EVERY unfinished unit (up to kRoundCap): the window scheduler behind wk_transcribe_windows keeps the
    // session's decode slots full and runs the mel + encoder pass of the following windows under the running decode, so a round is not
    // limited to one slot-load.  Host staging is pinned and kept across calls; the per-window host work that follows a round (segment
    // search, DTW, word timing) runs on a pool of host threads.
    const int round_cap = std::max(max_batch, kRoundCap);
    HostStage& hs = host_stage();
    rc = hs.ensure((size_t)round_cap * kWindow * sizeof(float), o->word_timestamps ? (size_t)round_cap * info.kv_max_len * info.n_audio_ctx * 2 : 0);
    if (rc != WK_OK) { delete T; return rc; }
    float* batch = hs.pcm;
    std::vector<int32_t> valid(round_cap);
    std::vector<wk_decode_result> res(round_cap);
    std::vector<int32_t> win_lang(round_cap);
    std::vector<float> win_lang_lp(round_cap);
    // detectedLanguage is reassigned every window when the task detects (TranscribeTask.swift:352), set once otherwise (:376)
    const bool detecting = info.is_multilingual && o->detect_language && o->language_token < 0;
    std::vector<int> active;
    std::vector<std::vector<int32_t>> unit_tokens(units.size());
    std::vector<std::vector<float>> unit_lps(units.size());
    const int n_threads = (int)std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    for (;;) {
        active.clear();
        for (size_t i = 0; i < units.size() && (int)active.size() < round_cap; ++i)
            if (!units[i].done) active.push_back((int)i);
        if (active.empty()) break;
        std::vector<int64_t> seg_size(active.size());
        parallel_for((int)active.size(), n_threads, [&](int k) {
            Unit& u = units[active[k]];
            const int64_t clip_end = u.clips[2 * u.clip + 1];
            const int64_t sz = std::min<int64_t>({kWindow, u.n - u.seek, clip_end - u.seek});   // TranscribeTask.swift:121
            seg_size[k] = sz;
            valid[k] = (int32_t)sz;
            memcpy(batch + (size_t)k * kWindow, u.audio + u.seek, (size_t)sz * sizeof(float));   // padOrTrim (zero fill happens in the mel kernel via `valid`)
            return WK_OK;
        }, nullptr);
        rc = wk_transcribe_windows(m, s, batch, (int64_t)active.size(), kWindow, valid.data(), st, o, prompt, n_prompt, res.data());
        if (rc != WK_OK) { delete T; return rc; }
        T->windows += (int)active.size();
        rc = wk_session_languages(s, (int64_t)active.size(), win_lang.data(), win_lang_lp.data());
        if (rc != WK_OK) { delete T; return rc; }
        for (size_t k = 0; k < active.size(); ++k) {
            Unit& u = units[active[k]];
            if (u.windows++ == 0 || detecting) { u.lang_tok = win_lang[k]; u.lang_lp = win_lang_lp[k]; }
        }
        const int cols = info.n_audio_ctx;
        if (o->word_timestamps) {   // every window's alignment rows back in one burst (Float16, as the reference's alignmentWeights)
            for (size_t k = 0; k < active.size(); ++k) {
                const int have = std::min(res[k].n_tokens, info.kv_max_len);
                rc = wk_session_alignment_weights_f16(s, (int32_t)k, have, hs.align + (size_t)k * info.kv_max_len * cols, k + 1 == active.size() ? 1 : 0);
                if (rc != WK_OK) { delete T; return rc; }
            }
        }
        std::string worker_error;
        rc = parallel_for((int)active.size(), n_threads, [&](int k) -> wk_status {
            Unit& u = units[active[k]];
            const wk_decode_result& r = res[k];
            wk_status rc2;
            wk_segment segs[128];
            int nseg = 0;
            int64_t new_seek = u.seek;
            rc2 = wk_find_seek_point_and_segments(r.tokens, r.token_logprobs, r.n_tokens, 0.f, r.avg_logprob, r.compression_ratio, r.temperature, o,
                                                  (int32_t)u.segs.size(), u.seek, seg_size[k], kSampleRate, st->time_token_begin, &new_seek, segs, 128, &nseg);
            if (rc2 != WK_OK) return rc2;
            const int64_t prev = u.seek;
            u.seek = std::max(u.seek, new_seek);
            if (max_window_seek >= 0) u.seek = std::min(u.seek, prev + max_window_seek);
            std::vector<OutWord> new_words;
            if (o->word_timestamps) {
                // addWordTimestamps on this window (TranscribeTask.swift:197-239): rows = window tokens, zero rows past the tensor's 224
                const int n_tok = r.n_tokens, have = std::min(n_tok, info.kv_max_len);
                const uint16_t* rows16 = hs.align + (size_t)k * info.kv_max_len * cols;
                std::vector<uint16_t> padded;
                if (n_tok > have || n_tok < 1) {   // (226-token results: the rows past the tensor read as zeros)
                    padded.assign((size_t)std::max(n_tok, 1) * cols, 0);
                    memcpy(padded.data(), rows16, (size_t)have * cols * 2);
                    rows16 = padded.data();
                }
                wk_words* wh = nullptr;
                const int n_in = std::max(nseg, 0);
                rc2 = wk_add_word_timestamps(segs, n_in, r.tokens, r.token_logprobs, rows16, WK_DTYPE_F16, std::max(n_tok, 1), cols, cols, hooks, prev,
                                             (float)((double)prev / (double)kSampleRate), st->special_token_begin, nullptr, nullptr, &wh);
                if (rc2 != WK_OK) return rc2;
                // drop zero-length segments (:214), remap the words' segment index, and let the last word end pull the seek forward (:217-219)
                std::vector<int> remap((size_t)n_in, -1);
                int kept = 0;
                for (int g = 0; g < n_in; ++g)
                    if (segs[g].end > segs[g].start) { remap[g] = kept; segs[kept++] = segs[g]; }
                for (int i = 0; i < wk_words_count(wh); ++i) {
                    wk_word w;
                    wk_words_get(wh, i, &w);
                    if (w.segment < 0 || remap[w.segment] < 0) continue;
                    OutWord ow;
                    ow.word = w.word; ow.tokens.assign(w.tokens, w.tokens + w.n_tokens);
                    ow.start = w.start; ow.end = w.end; ow.probability = w.probability; ow.segment = remap[w.segment];
                    new_words.push_back(std::move(ow));
                }
                wk_words_free(wh);
                if (nseg >= 0) nseg = kept;
                if (kept > 0) u.seek = std::max(u.seek, (int64_t)(segs[kept - 1].end * (float)kSampleRate));
                if (max_window_seek >= 0) u.seek = std::min(u.seek, prev + max_window_seek);
            }
            // termination guard (not in the reference, which can spin when a window decodes to <|0.00|><|0.00|>): always move on
            if (u.seek <= prev) u.seek = prev + seg_size[k];
            for (OutWord& w : new_words) { w.segment += (int)u.segs.size(); u.words.push_back(std::move(w)); }
            for (int g = 0; g < nseg; ++g) {
                wk_segment sg = segs[g];
                const int64_t base = (int64_t)unit_tokens[active[k]].size();
                for (int t = 0; t < sg.n_tokens; ++t) {
                    unit_tokens[active[k]].push_back(r.tokens[sg.token_offset + t]);
                    unit_lps[active[k]].push_back(r.token_logprobs[sg.token_offset + t]);
                }
                sg.token_offset = base;
                sg.stream = u.stream;
                u.segs.push_back(sg);
            }
            const int nclips = (int)u.clips.size() / 2;
            while (!(u.seek < u.clips[2 * u.clip + 1] - window_padding && u.seek < u.n)) {
                if (u.clip + 1 >= nclips) { u.done = true; break; }
                ++u.clip;
                u.seek = u.clips[2 * u.clip];
            }
            return WK_OK;
        }, &worker_error);
        if (rc != WK_OK) { set_error("%s", worker_error.c_str()); delete T; return rc; }
    }
    // flatten: streams in order, units (chunks) in order, chunk offsets applied (updateSegmentTimings, AudioChunker.swift:14-39)
    std::vector<int> next_id(n_streams, 0);
    // a stream's language is its first unit's: a plain stream has one, a VAD-chunked stream takes its first chunk's
    // (TranscriptionUtilities.swift:103); a stream without a window reports English
    T->lang_tok.assign(n_streams, st->english_token);
    T->lang_lp.assign(n_streams, 0.f);
    std::vector<uint8_t> lang_set(n_streams, 0);
    for (const Unit& u : units)
        if (!lang_set[u.stream]) {
            lang_set[u.stream] = 1;
            if (u.windows > 0) { T->lang_tok[u.stream] = u.lang_tok; T->lang_lp[u.stream] = u.lang_lp; }
        }
    for (size_t i = 0; i < units.size(); ++i) {
        Unit& u = units[i];
        const float seek_time = (float)u.offset / (float)kSampleRate;
        const int64_t base = (int64_t)T->tokens.size();
        T->tokens.insert(T->tokens.end(), unit_tokens[i].begin(), unit_tokens[i].end());
        T->logprobs.insert(T->logprobs.end(), unit_lps[i].begin(), unit_lps[i].end());
        const int seg_base = (int)T->segments.size();
        for (OutWord w : u.words) {
            w.start += seek_time; w.end += seek_time; w.segment += seg_base;
            T->words.push_back(std::move(w));
        }
        for (wk_segment sg : u.segs) {
            sg.id = next_id[u.stream]++;
            sg.seek += u.offset;
            sg.start += seek_time;
            sg.end += seek_time;
            sg.token_offset += base;
            T->segments.push_back(sg);
        }
    }
    *out = T;
    return WK_OK;
}

int32_t wk_transcription_segment_count(const wk_transcription* t) { return t ? (int32_t)t->segments.size() : 0; }
int32_t wk_transcription_window_count(const wk_transcription* t) { return t ? t->windows : 0; }
int64_t wk_transcription_token_count(const wk_transcription* t) { return t ? (int64_t)t->tokens.size() : 0; }
wk_status wk_transcription_segments(const wk_transcription* t, wk_segment* segs, int32_t cap) {
    if (!t || !segs || cap < (int32_t)t->segments.size()) { set_error("wk_transcription_segments: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    if (!t->segments.empty()) memcpy(segs, t->segments.data(), t->segments.size() * sizeof(wk_segment));
    return WK_OK;
}
wk_status wk_transcription_tokens(const wk_transcription* t, int32_t* tokens, float* logprobs, int64_t cap) {
    if (!t || cap < (int64_t)t->tokens.size()) { set_error("wk_transcription_tokens: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    if (tokens && !t->tokens.empty()) memcpy(tokens, t->tokens.data(), t->tokens.size() * 4);
    if (logprobs && !t->logprobs.empty()) memcpy(logprobs, t->logprobs.data(), t->logprobs.size() * 4);
    return WK_OK;
}
int32_t wk_transcription_word_count(const wk_transcription* t) { return t ? (int32_t)t->words.size() : 0; }
wk_status wk_transcription_word(const wk_transcription* t, int32_t i, wk_word* out) {
    if (!t || !out || i < 0 || i >= (int32_t)t->words.size()) { set_error("wk_transcription_word: index out of range"); return WK_ERR_INVALID_ARGUMENT; }
    const OutWord& w = t->words[i];
    out->word = w.word.c_str(); out->tokens = w.tokens.data(); out->n_tokens = (int32_t)w.tokens.size();
    out->start = w.start; out->end = w.end; out->probability = w.probability; out->segment = w.segment;
    return WK_OK;
}
wk_status wk_transcription_language(const wk_transcription* t, int32_t stream, int32_t* token, float* logprob) {
    if (!t || !token || stream < 0 || stream >= (int32_t)t->lang_tok.size()) { set_error("wk_transcription_language: stream out of range"); return WK_ERR_INVALID_ARGUMENT; }
    *token = t->lang_tok[stream];
    if (logprob) *logprob = t->lang_lp[stream];
    return WK_OK;
}
void wk_transcription_free(wk_transcription* t) { delete t; }

}  // extern "C"
