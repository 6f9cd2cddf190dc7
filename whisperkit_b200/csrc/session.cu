// libwkb200 decode sessions: per-worker decoder state (TextDecoding.prepareDecoderInputs, TextDecoder.swift:109-161), one decoder
// forward (predictLogits, :361-418), the device-resident token loop (decodeText, :541-855) and the window scheduler behind
// wk_transcribe_windows (the per-window body of TranscribeTask.run, TranscribeTask.swift:116-278, fanned out like
// WhisperKit.transcribeWithOptions, WhisperKit.swift:716-812, with decodeWithFallback's temperature ladder, TranscribeTask.swift:316-411).
//
// Scheduling model.  A session owns `max_batch` decode SLOTS.  Every slot carries its own position, prompt and options on the device
// (DecodeState / RowParams), so one CUDA graph of the step serves any mix of windows; a slot whose window has ended is skipped by every
// kernel of the step (no cross-KV stream, no cache traffic, no logits row).  The host polls the done flags every few steps, finalises the
// windows that ended (sampler.finalize, slicing, avgLogProb, compressionRatio, DecodingFallback) and hands their slots to the next
// encoded windows - or back to the same window at the next ladder temperature.  The mel + encoder pass of the next chunk runs on a
// second stream while the current slots decode (tensor-bound under HBM-bound).
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <zlib.h>

#include <algorithm>
#include <string>
#include <vector>

#include "common.cuh"
#include "engine.h"

using namespace wk;

struct wk_session {
    wk_model* m = nullptr;
    int max_batch = 0;        // decode slots
    int batch = 0;            // rows the step runs over: slots [0, batch) (x beam rows per slot with beam search)
    int bound_windows = 0;    // windows bound by wk_session_set_encoder_output (cross K/V blocks 0 .. bound_windows - 1)
    int bp = 16;              // batch padded to the UMMA N granule
    cudaStream_t stream = nullptr;      // decode stream
    cudaStream_t enc_stream = nullptr;  // mel + encoder of the batched entry
    EncWorkspace ws;                    // this session's mel / encoder activations (allocated on first use)
    void* cross_kv = nullptr;   // [2L][S][H][T][64]
    void* self_k = nullptr;     // [L][S][H][224][64]
    void* self_v = nullptr;
    float* partial = nullptr; size_t partial_elems = 0;
    float* x = nullptr; void* xn = nullptr; void* attn = nullptr; void* ffn = nullptr;
    float* logits = nullptr;
    DecodeState st;
    RowParams* rp_dev = nullptr;
    int32_t* pos_dev = nullptr; int32_t* lang_dev = nullptr;
    int32_t* suppress_dev = nullptr; size_t suppress_cap = 0;
    // slot admission staging (pinned host + device)
    int32_t *h_adm_slots = nullptr, *h_adm_prompts = nullptr; RowParams* h_adm_rp = nullptr;
    int32_t *d_adm_slots = nullptr, *d_adm_prompts = nullptr; RowParams* d_adm_rp = nullptr;
    // pinned readback of the decode state
    int32_t *h_tokens = nullptr, *h_n_tokens = nullptr, *h_done = nullptr, *h_first_low = nullptr, *h_steps = nullptr, *h_error = nullptr;
    float* h_logprobs = nullptr;
    // step graph, cached across calls: the step depends on the call only through the rows it covers, the alignment export and the
    // special-token ids baked into the sampler's parameters
    cudaGraphExec_t graph_exec = nullptr, graph_exec_live = nullptr;   // the step with / without the ended-row checks in the attention kernels
    int graph_batch = 0; bool graph_align = false, graph_fused = false; wk_special_tokens graph_st; long long launches_per_step = 0;
    bool warmed = false;
    // word timestamps: per-head softmax rows of the current step, the [S][224][T] Float16 alignmentWeights of the slots, and the per-window
    // copies handed out by wk_session_alignment_weights
    float* align_scratch = nullptr; void* align_w = nullptr; int align_slots = 0; bool align_on = false;
    void* align_store = nullptr; int64_t align_store_cap = 0, align_store_n = 0;
    unsigned int* chain_counters = nullptr;
    cudaEvent_t ev_enc = nullptr, ev_adm = nullptr, ev_stage = nullptr, ev_t[10];
    bool knob_fused = false, knob_graph = true;
    // beam search (allocated on the first call that asks for it)
    BeamState bs = BeamState(); int bs_cap_rows = 0;
    int32_t *h_n_fin = nullptr, *h_fin_len = nullptr, *h_fin_tokens = nullptr; float *h_fin_score = nullptr, *h_fin_lps = nullptr, *h_sum_lp = nullptr;
    int graph_beam = 1;
    std::vector<int> slot_window, slot_try;
    int64_t stats[4] = {0, 0, 0, 0};   // of the last batched call: step launches, sum of live rows over them, admissions, ladder re-admissions
    // language detection: the session's allLanguageTokens (empty = the special tokens' language block), the list length baked into the
    // step graphs, the pinned readback of the rows' detections and the language of every window of the last wk_transcribe_windows(_ex)
    std::vector<int32_t> lang_list;
    int graph_lang_n = 0, loop_lang_n = 0;
    int32_t* h_lang_tok = nullptr; float* h_lang_lp = nullptr;
    std::vector<int32_t> win_lang_tok; std::vector<float> win_lang_lp;
};

namespace wk {

// ---------------------------------------------------------------------------------------------- decoder schedule
static wk_status dec_gemm(wk_session* s, const void* w, int N, int K, const void* act, int* splits_out) {
    wk_model* m = s->m;
    GemmDesc g;
    memset(&g, 0, sizeof(g));
    // swap-AB: A = weights [N, K] (128 output features per tile), B = activations [Bp, K]
    g.a = w; g.a_rows = N; g.a_cols = K; g.a_ld = K; g.a_batches = 1;
    g.b = act; g.b_rows = s->bp; g.b_ld = K; g.in_dtype = m->cfg.dtype;
    g.m_rows_per_batch = N; g.n = s->bp; g.k = K; g.taps = 1; g.bn = s->bp;
    const int tiles = (N + 127) / 128;
    g.splits = choose_splits(tiles, K / 64, m->num_sms);
    g.mode = GEMM_OUT_PARTIAL_T; g.out = s->partial; g.ld_out = N; g.out_rows_per_batch = N; g.partial_cols = s->bp;
    g.pdl = 1; g.a_static = 1;
    if ((size_t)g.splits * s->bp * N > s->partial_elems) { set_error("partial workspace too small"); return WK_ERR_DECODING_FAILED; }
    *splits_out = g.splits;
    return gemm_tcgen05(g, m->num_sms, s->stream);
}

// The fused phase chains hold every SM with a CTA that waits on grid-wide barriers.  Two such grids from different sessions could each
// take half of the machine and wait for the other half forever, so a session only uses them while it is the model's sole live session.
static bool use_fused(const wk_session* s) { return s->knob_fused && s->m->live_sessions.load(std::memory_order_relaxed) == 1; }

// one decoder forward for every row of the step.  explicit_pos == nullptr: loop mode (token / position from DecodeState, ended rows skipped)
static wk_status decoder_forward(wk_session* s, int ts_begin, int sot, const int32_t* explicit_pos, bool fused, bool check_done = true) {
    wk_model* m = s->m;
    const wk_model_config& c = m->cfg;
    const int d = c.d_model, H = c.n_heads, dt = c.dtype, B = s->batch, Bp = s->bp, T = c.n_audio_ctx;
    cudaStream_t st = s->stream;
    const size_t self_layer = (size_t)s->max_batch * H * kKvMaxLen * 64 * 2;   // bytes per layer
    const size_t cross_block = (size_t)s->max_batch * H * T * 64 * 2;          // bytes per (layer, k|v)
    const int32_t* pos = explicit_pos ? explicit_pos : s->st.steps;
    // ended rows are skipped by the attention kernels; a burst that starts with every slot live runs the variant without the checks (a
    // row that ends inside it just keeps computing until the next poll, as harmlessly as before it ended)
    const int32_t* done = (explicit_pos || !check_done) ? nullptr : s->st.done;
    const bool beam_rows = !explicit_pos && s->bs.beam > 1;   // rows are beams: cache ancestry + one cross K/V block per `beam` rows
    const int n_layers = c.dec_layers;
    int sp = 1;
    WK_CHECK(decoder_embed_ln(m->emb, m->dec_pos, m->dec[0].ln1.g, m->dec[0].ln1.b, s->st, c.vocab, ts_begin, sot, s->x, s->xn, B, d, dt, explicit_pos, st));
    auto self_attn = [&](int li, const DecLayer& l) {
        return decoder_self_attention(s->partial, sp, Bp, l.bq, l.bv, (char*)s->self_k + li * self_layer, (char*)s->self_v + li * self_layer, pos, done,
                                      s->attn, B, H, kKvMaxLen, dt, st, beam_rows ? s->bs.anc : nullptr);
    };
    auto cross_attn = [&](int li, const DecLayer& l) {
        const bool align = s->align_on && !explicit_pos && m->align_mask[li] != 0;
        return decoder_cross_attention(s->partial, sp, Bp, l.bcq, (char*)s->cross_kv + (size_t)(2 * li) * cross_block,
                                       (char*)s->cross_kv + (size_t)(2 * li + 1) * cross_block, s->attn, B, H, T, dt, st, done,
                                       align ? s->align_scratch + (size_t)m->align_base[li] * B * T : nullptr, align ? m->align_mask[li] : 0u,
                                       beam_rows ? s->bs.beam : 1);
    };
    if (fused) {
        // per layer: self-attention -> chain B (out-proj, reduce+LN, cross-Q) -> cross-attention -> chain C (cross-out, reduce+LN, FC1,
        // reduce+GELU, FC2, reduce+LN, next layer's QKV): phases of one persistent kernel separated by grid barriers (fused_chain.cu)
        const int kWords = 8;
        auto gemm_phase = [&](const void* w, int N, int K, const void* act) {
            ChainPhaseDesc ph; memset(&ph, 0, sizeof(ph));
            ph.kind = 0; ph.w = w; ph.n = N; ph.k = K; ph.act = act; ph.splits = choose_splits((N + 127) / 128, K / 64, m->num_sms);
            return ph;
        };
        auto ln_phase = [&](const float* bias, const LayerNormW& ln) {
            ChainPhaseDesc ph; memset(&ph, 0, sizeof(ph));
            ph.kind = 1; ph.bias = bias; ph.gamma = ln.g; ph.beta = ln.b; ph.out16 = s->xn;
            return ph;
        };
        auto chain_base = [&](int li, int which) {
            ChainDesc cd; memset(&cd, 0, sizeof(cd));
            cd.partial = s->partial; cd.x = s->x; cd.B = B; cd.Bp = Bp; cd.d = d; cd.dtype = dt; cd.pdl = 1;
            cd.counters = s->chain_counters + ((size_t)li * 2 + which) * kWords;
            cd.reset_counters = s->chain_counters + ((size_t)li * 2 + (which ^ 1)) * kWords;   // the sibling chain re-arms this one's words
            return cd;
        };
        WK_CHECK(dec_gemm(s, m->dec[0].wqkv, 3 * d, d, s->xn, &sp));
        for (int li = 0; li < n_layers; ++li) {
            DecLayer& l = m->dec[li];
            WK_CHECK(self_attn(li, l));
            ChainDesc cb = chain_base(li, 0);
            cb.ph[0] = gemm_phase(l.wo, d, d, s->attn);
            cb.ph[1] = ln_phase(l.bo, l.lnx);
            cb.ph[2] = gemm_phase(l.wcq, d, d, s->xn);
            cb.n_phases = 3;
            WK_CHECK(decoder_chain(cb, m->num_sms, st));
            sp = cb.ph[2].splits;
            WK_CHECK(cross_attn(li, l));
            ChainDesc cc = chain_base(li, 1);
            const LayerNormW& nxt = (li + 1 < n_layers) ? m->dec[li + 1].ln1 : m->dec_ln;
            cc.ph[0] = gemm_phase(l.wco, d, d, s->attn);
            cc.ph[1] = ln_phase(l.bco, l.ln3);
            cc.ph[2] = gemm_phase(l.w1, 4 * d, d, s->xn);
            cc.ph[3].kind = 2; cc.ph[3].bias = l.b1; cc.ph[3].out16 = s->ffn;
            cc.ph[4] = gemm_phase(l.w2, d, 4 * d, s->ffn);
            cc.ph[5] = ln_phase(l.b2, nxt);
            cc.n_phases = 6;
            if (li + 1 < n_layers) { cc.ph[6] = gemm_phase(m->dec[li + 1].wqkv, 3 * d, d, s->xn); cc.n_phases = 7; sp = cc.ph[6].splits; }
            WK_CHECK(decoder_chain(cc, m->num_sms, st));
        }
    } else {
        for (int li = 0; li < n_layers; ++li) {
            DecLayer& l = m->dec[li];
            WK_CHECK(dec_gemm(s, l.wqkv, 3 * d, d, s->xn, &sp));
            WK_CHECK(self_attn(li, l));
            WK_CHECK(dec_gemm(s, l.wo, d, d, s->attn, &sp));
            WK_CHECK(decoder_reduce_resid_ln(s->partial, sp, Bp, l.bo, l.lnx.g, l.lnx.b, s->x, s->xn, B, d, dt, st));
            WK_CHECK(dec_gemm(s, l.wcq, d, d, s->xn, &sp));
            WK_CHECK(cross_attn(li, l));
            WK_CHECK(dec_gemm(s, l.wco, d, d, s->attn, &sp));
            WK_CHECK(decoder_reduce_resid_ln(s->partial, sp, Bp, l.bco, l.ln3.g, l.ln3.b, s->x, s->xn, B, d, dt, st));
            WK_CHECK(dec_gemm(s, l.w1, 4 * d, d, s->xn, &sp));
            WK_CHECK(decoder_reduce_bias_gelu(s->partial, sp, Bp, l.b1, s->ffn, B, 4 * d, dt, st));
            WK_CHECK(dec_gemm(s, l.w2, d, 4 * d, s->ffn, &sp));
            const LayerNormW& nxt = (li + 1 < n_layers) ? m->dec[li + 1].ln1 : m->dec_ln;
            WK_CHECK(decoder_reduce_resid_ln(s->partial, sp, Bp, l.b2, nxt.g, nxt.b, s->x, s->xn, B, d, dt, st));
        }
    }
    // logits = xn . E^T  (tied embedding), written [B][V] f32 by the transposed-store epilogue (splits = 1)
    {
        GemmDesc g;
        memset(&g, 0, sizeof(g));
        g.a = m->emb; g.a_rows = c.vocab; g.a_cols = d; g.a_ld = d; g.a_batches = 1;
        g.b = s->xn; g.b_rows = Bp; g.b_ld = d; g.in_dtype = dt;
        g.m_rows_per_batch = c.vocab; g.n = Bp; g.k = d; g.taps = 1; g.bn = Bp; g.splits = 1;
        g.mode = GEMM_OUT_PARTIAL_T; g.out = s->logits; g.ld_out = c.vocab; g.out_rows_per_batch = c.vocab; g.partial_cols = B;
        g.pdl = 1; g.a_static = 1;
        WK_CHECK(gemm_tcgen05(g, m->num_sms, st));
    }
    return WK_OK;
}

static SamplerParams loop_sampler_params(wk_session* s, const wk_special_tokens* st) {
    SamplerParams p;
    memset(&p, 0, sizeof(p));
    p.st = *st;
    p.vocab = s->m->cfg.vocab;
    p.is_multilingual = s->m->cfg.vocab != 51864;
    p.loop_mode = 1;
    p.suppress = s->suppress_dev;
    p.max_ctx = kKvMaxLen;
    p.beam = s->bs;
    p.language_tokens = s->lang_dev; p.n_language_tokens = s->loop_lang_n;
    return p;
}

// TextUtilities.compressionRatio(of: [Int]) (TextUtilities.swift:14-28): raw DEFLATE of the Int32 LE bytes
static float compression_ratio(const std::vector<int32_t>& toks) {
    if (toks.empty()) return INFINITY;
    const uLong n = (uLong)toks.size() * 4;
    z_stream zs;
    memset(&zs, 0, sizeof(zs));
    if (deflateInit2(&zs, 5, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) return INFINITY;
    std::vector<unsigned char> out(deflateBound(&zs, n) + 64);
    zs.next_in = (Bytef*)toks.data(); zs.avail_in = n;
    zs.next_out = out.data(); zs.avail_out = (uInt)out.size();
    const int r = deflate(&zs, Z_FINISH);
    const uLong clen = zs.total_out;
    deflateEnd(&zs);
    if (r != Z_STREAM_END || clen == 0) return INFINITY;
    return (float)n / (float)clen;
}

// finalisation of one window on the host: finalize + slicing + averages (TextDecoder.swift:776-853)
static void finalize_result(wk_decode_result& r, const int32_t* tokens, const float* lps, int n_tok, int steps, int first_low,
                            const wk_special_tokens* st, const wk_decode_opts* o, float temperature) {
    memset(&r, 0, sizeof(r));
    std::vector<int32_t> seg(tokens, tokens + n_tok);
    std::vector<float> slp(lps, lps + n_tok);
    r.n_current_tokens = n_tok;
    r.steps = steps;
    r.first_token_logprob_too_low = first_low;
    if (seg.empty() || seg.back() != st->end_token) { seg.push_back(st->end_token); slp.push_back(0.f); }  // sampler.finalize
    size_t start = 0, end = seg.size();
    for (size_t i = 0; i < seg.size(); ++i) if (seg[i] == st->start_of_transcript_token) { start = i; break; }
    for (size_t i = 0; i < seg.size(); ++i) if (seg[i] == st->end_token) { end = i; break; }
    if (end >= seg.size()) end = seg.size() - 1;
    if (end < start) start = 0;
    float sum = 0.f;
    std::vector<int32_t> words;
    r.n_tokens = 0;
    for (size_t i = start; i <= end && r.n_tokens < 226; ++i) {
        r.tokens[r.n_tokens] = seg[i];
        r.token_logprobs[r.n_tokens] = slp[i];
        sum += slp[i];
        if (seg[i] < st->special_token_begin) words.push_back(seg[i]);
        ++r.n_tokens;
    }
    r.avg_logprob = sum / (float)r.n_tokens;
    r.compression_ratio = compression_ratio(words);
    r.temperature = roundf(temperature * 1000.f) / 1000.f;
    // DecodingFallback (Models.swift:357-381); noSpeechProb is always 0 in the reference (TextDecoder.swift:802)
    r.needs_fallback = 0; r.fallback_reason = 0;
    if (first_low) { r.needs_fallback = 1; r.fallback_reason = 1; }
    else if (o->has_no_speech_threshold && 0.f > o->no_speech_threshold) { r.needs_fallback = 0; r.fallback_reason = 2; }
    else if (o->has_compression_ratio_threshold && r.compression_ratio > o->compression_ratio_threshold) { r.needs_fallback = 1; r.fallback_reason = 3; }
    else if (o->has_logprob_threshold && r.avg_logprob < o->logprob_threshold) { r.needs_fallback = 1; r.fallback_reason = 4; }
}

// prefillDecoderInputs (TextDecoder.swift:163-216)
static wk_status build_prompt(const wk_model* m, const wk_special_tokens* st, const wk_decode_opts* o, int use_options, std::vector<int32_t>& p) {
    p.clear();
    p.push_back(st->start_of_transcript_token);
    if (use_options && o) {
        const bool multilingual = m->cfg.vocab != 51864;
        if (multilingual) {
            p.push_back(o->language_token >= 0 ? o->language_token : st->english_token);
            p.push_back(o->task_translate ? st->translate_token : st->transcribe_token);
        }
        p.push_back(o->without_timestamps ? st->no_timestamps_token : st->time_token_begin);
        if (o->n_prompt_tokens >= 0 && (o->prompt_tokens || o->n_prompt_tokens == 0)) {
            const int maxlen = kKvMaxLen / 2 - 1;
            std::vector<int32_t> q;
            const int start = o->n_prompt_tokens > maxlen ? o->n_prompt_tokens - maxlen : 0;
            q.push_back(st->start_of_previous_token);
            for (int i = start; i < o->n_prompt_tokens; ++i)
                if (o->prompt_tokens[i] < st->special_token_begin) q.push_back(o->prompt_tokens[i]);
            q.insert(q.end(), p.begin(), p.end());
            p.swap(q);
        }
        if (o->n_prefix_tokens >= 0 && (o->prefix_tokens || o->n_prefix_tokens == 0)) {
            const int maxlen = kKvMaxLen / 2;
            const int start = o->n_prefix_tokens > maxlen ? o->n_prefix_tokens - maxlen : 0;
            for (int i = start; i < o->n_prefix_tokens; ++i)
                if (o->prefix_tokens[i] < st->special_token_begin) p.push_back(o->prefix_tokens[i]);
        }
    }
    return WK_OK;
}

// ---------------------------------------------------------------------------------------------- the step and its graph
static wk_status enqueue_step(wk_session* s, const wk_special_tokens* st, bool fused, bool check_done) {
    wk_model* m = s->m;
    WK_CHECK(decoder_forward(s, st->time_token_begin, st->start_of_transcript_token, nullptr, fused, check_done));
    WK_CHECK(sampler_filter_sample(s->logits, m->cfg.vocab, loop_sampler_params(s, st), s->st, nullptr, 0, nullptr, nullptr, nullptr, nullptr, s->batch, s->stream));
    if (s->bs.beam > 1) WK_CHECK(beam_update(s->st, s->bs, *st, kKvMaxLen, s->batch / s->bs.beam, s->stream));
    if (s->align_on)
        WK_CHECK(decoder_align_mean(s->align_scratch, m->n_align_slots, s->st.steps, s->st.done, s->align_w, s->batch, m->cfg.n_audio_ctx, kKvMaxLen, s->stream));
    return WK_OK;
}

// runs `n` decode steps on the session stream (CUDA graph replay; the first step of a session runs eagerly so that lazily loaded
// kernels and function attributes exist before a capture)
static wk_status run_steps(wk_session* s, const wk_special_tokens* st, int n, bool all_live) {
    const bool fused = use_fused(s);
    const bool check_done = !all_live;
    int done = 0;
    if (!s->knob_graph || !s->warmed) {
        const int eager = s->knob_graph ? 1 : n;
        for (; done < eager && done < n; ++done) WK_CHECK(enqueue_step(s, st, fused, check_done));
        s->warmed = true;
    }
    if (done >= n) return WK_OK;
    const int beam_key = std::max(1, s->bs.beam) * 16 + s->bs.max_candidates;
    const bool stale = s->graph_batch != s->batch || s->graph_align != s->align_on || s->graph_fused != fused || s->graph_beam != beam_key ||
                       s->graph_lang_n != s->loop_lang_n || memcmp(&s->graph_st, st, sizeof(*st)) != 0;
    if (stale) {
        if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }
        if (s->graph_exec_live) { cudaGraphExecDestroy(s->graph_exec_live); s->graph_exec_live = nullptr; }
        s->graph_batch = s->batch; s->graph_align = s->align_on; s->graph_fused = fused; s->graph_st = *st; s->graph_beam = beam_key;
        s->graph_lang_n = s->loop_lang_n;
    }
    cudaGraphExec_t& exec = check_done ? s->graph_exec : s->graph_exec_live;
    if (!exec) {
        for (int attempt = 0; attempt < 2; ++attempt) {
            cudaGraph_t graph = nullptr;
            const long long before = launch_counter_load();
            WK_CUDA_CHECK(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
            wk_status r = enqueue_step(s, st, fused, check_done);
            cudaError_t e = cudaStreamEndCapture(s->stream, &graph);
            s->launches_per_step = launch_counter_load() - before;
            launch_counter_sub(s->launches_per_step);  // captured, not executed
            if (r != WK_OK) { if (graph) cudaGraphDestroy(graph); return r; }
            if (e != cudaSuccess) { set_error("graph capture failed: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
            e = cudaGraphInstantiate(&exec, graph, 0);
            cudaGraphDestroy(graph);
            if (e == cudaSuccess) break;
            exec = nullptr;
            if (attempt == 0 && pdl_enabled()) {   // programmatic edges rejected by this driver: plain serialisation, capture again
                cudaGetLastError();
                pdl_disable();
                continue;
            }
            set_error("graph instantiate failed: %s", cudaGetErrorString(e));
            return WK_ERR_CUDA;
        }
    }
    for (; done < n; ++done) {
        WK_CUDA_CHECK(cudaGraphLaunch(exec, s->stream));
        count_launch((int)s->launches_per_step);
    }
    return WK_OK;
}

// ---------------------------------------------------------------------------------------------- the window scheduler
struct CoreArgs {
    const float* pcm; int64_t n; int64_t stride; const int32_t* spw;   // pcm == nullptr: windows are the session's bound rows (decodeText)
    const wk_special_tokens* st; const wk_batch_opts* bo; wk_decode_result* results;
    bool ladder;
};

static const wk_decode_opts& opts_of(const wk_batch_opts* bo, int64_t w) { return bo->n_opts == 1 ? bo->opts[0] : bo->opts[w]; }

static wk_status ensure_align(wk_session* s, int64_t n_windows) {
    wk_model* m = s->m;
    const size_t T = m->cfg.n_audio_ctx;
    if (!s->align_w) WK_CUDA_CHECK(cudaMalloc(&s->align_w, (size_t)s->max_batch * kKvMaxLen * T * 2));
    if (!s->align_scratch || s->align_slots != m->n_align_slots) {
        if (s->align_scratch) { WK_CUDA_CHECK(cudaStreamSynchronize(s->stream)); cudaFree(s->align_scratch); s->align_scratch = nullptr; }
        WK_CUDA_CHECK(cudaMalloc((void**)&s->align_scratch, (size_t)std::max(1, m->n_align_slots) * s->max_batch * T * 4));
        s->align_slots = m->n_align_slots;
        if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }   // the scratch pointer is baked into the graphs
        if (s->graph_exec_live) { cudaGraphExecDestroy(s->graph_exec_live); s->graph_exec_live = nullptr; }
    }
    if (s->align_store_cap < n_windows) {
        if (s->align_store) { WK_CUDA_CHECK(cudaStreamSynchronize(s->stream)); cudaFree(s->align_store); s->align_store = nullptr; }
        WK_CUDA_CHECK(cudaMalloc(&s->align_store, (size_t)n_windows * kKvMaxLen * T * 2));
        s->align_store_cap = n_windows;
    }
    s->align_store_n = n_windows;
    return WK_OK;
}

static wk_status ensure_beam(wk_session* s) {
    if (s->bs_cap_rows >= s->max_batch) return WK_OK;
    const int S = s->max_batch, G = S / 2 + 1;
    WK_CHECK(dmalloc(&s->bs.sum_lp, S));
    WK_CHECK(dmalloc(&s->bs.cand_tok, (size_t)S * (kMaxBeam + 1)));
    WK_CHECK(dmalloc(&s->bs.cand_lp, (size_t)S * (kMaxBeam + 1)));
    WK_CHECK(dmalloc(&s->bs.anc, (size_t)S * kKvMaxLen));
    WK_CHECK(dmalloc(&s->bs.fin_tokens, (size_t)G * kMaxCand * kKvMaxLen));
    WK_CHECK(dmalloc(&s->bs.fin_lps, (size_t)G * kMaxCand * kKvMaxLen));
    WK_CHECK(dmalloc(&s->bs.fin_len, (size_t)G * kMaxCand));
    WK_CHECK(dmalloc(&s->bs.fin_score, (size_t)G * kMaxCand));
    WK_CHECK(dmalloc(&s->bs.n_fin, G));
    auto pinned = [&](void** p, size_t bytes) -> wk_status {
        cudaError_t e = cudaHostAlloc(p, bytes, cudaHostAllocDefault);
        if (e != cudaSuccess) { set_error("cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return WK_ERR_CUDA; }
        return WK_OK;
    };
    WK_CHECK(pinned((void**)&s->h_n_fin, (size_t)G * 4));
    WK_CHECK(pinned((void**)&s->h_fin_len, (size_t)G * kMaxCand * 4));
    WK_CHECK(pinned((void**)&s->h_fin_score, (size_t)G * kMaxCand * 4));
    WK_CHECK(pinned((void**)&s->h_fin_tokens, (size_t)G * kMaxCand * kKvMaxLen * 4));
    WK_CHECK(pinned((void**)&s->h_fin_lps, (size_t)G * kMaxCand * kKvMaxLen * 4));
    WK_CHECK(pinned((void**)&s->h_sum_lp, (size_t)S * 4));
    s->bs_cap_rows = S;
    return WK_OK;
}

// allLanguageTokens of a call (Models.swift:1219): the session's list, else the ids strictly between <|startoftranscript|> and
// min(<|translate|>, <|transcribe|>) - the language block of every Whisper vocabulary (99 ids, 100 in large-v3)
static std::vector<int32_t> language_list(const wk_session* s, const wk_special_tokens* st) {
    if (!s->lang_list.empty()) return s->lang_list;
    std::vector<int32_t> v;
    const int hi = std::min(st->translate_token, st->transcribe_token);
    for (int t = std::max(st->start_of_transcript_token + 1, 0); t < hi && t < s->m->cfg.vocab; ++t) v.push_back(t);
    return v;
}

static wk_status transcribe_core(wk_session* s, const CoreArgs& a) {
    wk_model* m = s->m;
    const wk_model_config& c = m->cfg;
    const wk_batch_opts* bo = a.bo;
    const wk_special_tokens* st = a.st;
    const bool bound = a.pcm == nullptr;
    const int64_t n = a.n;
    const int d = c.d_model, T = c.n_audio_ctx;
    const int poll = bo->progress_every > 0 ? bo->progress_every : 16;
    // beam search: every window takes `beam` consecutive decode rows; one setting per call (it shapes the step graph)
    const int beam = bo->opts[0].beam_size > 1 ? bo->opts[0].beam_size : 1;
    for (int i = 0; i < bo->n_opts; ++i)
        if ((bo->opts[i].beam_size > 1 ? bo->opts[i].beam_size : 1) != beam || (beam > 1 && bo->opts[i].beam_patience != bo->opts[0].beam_patience)) {
            set_error("beam size / patience must be the same for every window of a call"); return WK_ERR_INVALID_ARGUMENT;
        }
    int max_cand = 0;
    if (beam > 1) {
        const float patience = bo->opts[0].beam_patience > 0.f ? bo->opts[0].beam_patience : 1.f;
        max_cand = (int)((float)beam * patience);                                  // TokenSampler.swift:266
        if (beam > kMaxBeam || max_cand < 1 || max_cand > kMaxCand || s->max_batch < beam) {
            set_error("beam size %d / patience %.2f unsupported (beam <= %d, candidates in [1, %d], session rows %d)", beam, patience, kMaxBeam, kMaxCand, s->max_batch);
            return WK_ERR_INVALID_ARGUMENT;
        }
        for (int i = 0; i < bo->n_opts; ++i)
            if (bo->opts[i].word_timestamps) { set_error("wordTimestamps with beam search is not supported"); return WK_ERR_INVALID_ARGUMENT; }
        WK_CHECK(ensure_beam(s));
    }
    // detectLanguage (TranscribeTask.swift:339-365) runs in decodeWithFallback only (the entry points with the ladder), for a multilingual
    // model and a window without an explicit language
    const std::vector<int32_t> langs = language_list(s, st);
    auto detects = [&](const wk_decode_opts& o) { return a.ladder && c.vocab != 51864 && o.detect_language != 0 && o.language_token < 0; };
    auto is_language = [&](int32_t t) { return std::find(langs.begin(), langs.end(), t) != langs.end(); };
    bool any_detect = false;
    for (int i = 0; i < bo->n_opts; ++i) any_detect |= detects(bo->opts[i]);
    if (any_detect && beam > 1) { set_error("detectLanguage with beam search is not supported"); return WK_ERR_INVALID_ARGUMENT; }
    if (any_detect && (langs.empty() || langs.size() > 4096)) {
        set_error("detectLanguage: %zu language tokens (the list must hold 1 .. 4096 ids)", langs.size()); return WK_ERR_INVALID_ARGUMENT;
    }
    s->bs.beam = beam; s->bs.max_candidates = max_cand;
    const int S = s->max_batch / beam;     // decode slots (windows in flight)
    if (bound && n > S) { set_error("wk_decode_text: %lld bound windows x beam %d exceed the session's %d rows", (long long)n, beam, s->max_batch); return WK_ERR_PREPARE_DECODER_INPUTS; }
    std::vector<wk_status> st_local((size_t)n, WK_OK);
    wk_status* status = bo->status ? bo->status : st_local.data();
    for (int64_t w = 0; w < n; ++w) status[w] = WK_OK;
    std::string first_err;
    auto fail_window = [&](int64_t w, wk_status code) {
        status[w] = code;
        if (first_err.empty()) first_err = last_error_cstr();
        memset(&a.results[w], 0, sizeof(wk_decode_result));
    };
    // ---- per-window prompts, options, suppress lists (validated up front: a bad item fails alone, WhisperKit.swift:775-790)
    std::vector<std::vector<int32_t>> prompts((size_t)(bo->prompts || bo->prompt ? 0 : (bo->n_opts == 1 ? 1 : n)));
    std::vector<int32_t> shared_built;
    auto prompt_of = [&](int64_t w, const int32_t** p, int* np) {
        if (bo->prompts) { *p = bo->prompts[w]; *np = bo->prompt_lens[w]; }
        else if (bo->prompt) { *p = bo->prompt; *np = bo->n_prompt; }
        else { const auto& v = prompts[bo->n_opts == 1 ? 0 : (size_t)w]; *p = v.data(); *np = (int)v.size(); }
    };
    if (!bo->prompts && !bo->prompt)
        for (size_t i = 0; i < prompts.size(); ++i) {
            const wk_decode_opts& o = opts_of(bo, (int64_t)i);
            build_prompt(m, st, &o, o.use_prefill_prompt, prompts[i]);
        }
    bool any_words = false;
    std::vector<int32_t> sup_pool;
    std::vector<int> sup_off((size_t)bo->n_opts), sup_n((size_t)bo->n_opts);
    for (int i = 0; i < bo->n_opts; ++i) {
        const wk_decode_opts& o = bo->opts[i];
        any_words |= o.word_timestamps != 0;
        sup_off[i] = (int)sup_pool.size();
        for (int k = 0; k < o.n_suppress_tokens; ++k)   // SuppressTokensFilter gets the (< specialTokenBegin) ids only (TextDecoder.swift:876-879)
            if (o.suppress_tokens[k] >= 0 && o.suppress_tokens[k] < st->special_token_begin) sup_pool.push_back(o.suppress_tokens[k]);
        sup_n[i] = (int)sup_pool.size() - sup_off[i];
    }
    for (int64_t w = 0; w < n; ++w) {
        const int32_t* p; int np;
        prompt_of(w, &p, &np);
        if (!p || np < 1 || np >= kKvMaxLen) { set_error("window %lld: prompt length %d out of range", (long long)w, np); fail_window(w, WK_ERR_PREPARE_DECODER_INPUTS); continue; }
        bool ok = true;
        for (int i = 0; i < np && ok; ++i)
            if (p[i] < 0 || p[i] >= c.vocab) { set_error("window %lld: prompt token %d out of range", (long long)w, p[i]); ok = false; }
        if (!ok) { fail_window(w, WK_ERR_PREPARE_DECODER_INPUTS); continue; }
        if (!bound && a.spw && (a.spw[w] < 0 || a.spw[w] > kWindowSamples)) {
            set_error("window %lld: samples_per_window %d out of range", (long long)w, a.spw[w]);
            fail_window(w, WK_ERR_AUDIO_PROCESSING_FAILED);
        }
    }
    if (!bound && a.stride < kWindowSamples && !a.spw) { set_error("wk_transcribe_windows: stride < 480000 requires samples_per_window"); return WK_ERR_AUDIO_PROCESSING_FAILED; }
    if (!bo->status)
        for (int64_t w = 0; w < n; ++w) if (status[w] != WK_OK) { set_error("%s", first_err.c_str()); return status[w]; }
    if (sup_pool.size() > s->suppress_cap) {
        WK_CUDA_CHECK(cudaStreamSynchronize(s->stream));
        if (s->suppress_dev) cudaFree(s->suppress_dev);
        s->suppress_cap = std::max<size_t>(4096, sup_pool.size() * 2);
        WK_CHECK(dmalloc(&s->suppress_dev, s->suppress_cap));
        if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }   // pool pointer is baked into the graphs
        if (s->graph_exec_live) { cudaGraphExecDestroy(s->graph_exec_live); s->graph_exec_live = nullptr; }
    }
    if (!sup_pool.empty()) WK_CUDA_CHECK(cudaMemcpyAsync(s->suppress_dev, sup_pool.data(), sup_pool.size() * 4, cudaMemcpyHostToDevice, s->stream));
    if (any_detect) {   // (wk_detect_language shares the buffer: the list goes up again with every call that detects)
        WK_CUDA_CHECK(cudaMemcpyAsync(s->lang_dev, langs.data(), langs.size() * 4, cudaMemcpyHostToDevice, s->stream));
        s->loop_lang_n = (int)langs.size();
    }
    WK_CUDA_CHECK(cudaStreamSynchronize(s->stream));   // sup_pool is pageable: the copy must land before it goes out of scope paths below reuse it
    s->align_on = any_words;
    if (any_words) WK_CHECK(ensure_align(s, n));

    // ---- slots
    const int Brun = (int)std::min<int64_t>(S, n);     // slots in use; the step covers Brun * beam rows
    s->batch = Brun * beam;
    s->bp = round_up(s->batch, 16);
    const int rows = s->batch;
    s->slot_window.assign(S, -1);
    s->slot_try.assign(S, 0);
    {   // every slot starts free: done = 1 keeps its rows out of the step until a window is admitted
        std::vector<int32_t> ones(s->max_batch, 1);
        WK_CUDA_CHECK(cudaMemcpyAsync(s->st.done, ones.data(), s->max_batch * 4, cudaMemcpyHostToDevice, s->stream));
        WK_CUDA_CHECK(cudaStreamSynchronize(s->stream));
    }
    // temperature of ladder rung i, computed in Float16 like the reference (TranscribeTask.swift:327)
    auto rung_temperature = [&](const wk_decode_opts& o, int i) -> float {
        if (i == 0) return o.temperature;
        const float f16_t = __half2float(__float2half(o.temperature));
        const float f16_step = __half2float(__float2half(__half2float(__float2half((float)i)) * __half2float(__float2half(o.temperature_increment_on_fallback))));
        return __half2float(__float2half(f16_t + f16_step));
    };
    int n_adm = 0;
    auto stage_admission = [&](int slot, int64_t w, int rung) {
        const wk_decode_opts& o = opts_of(bo, w);
        const int oi = bo->n_opts == 1 ? 0 : (int)w;
        const int32_t* p; int np;
        prompt_of(w, &p, &np);
        RowParams R;
        memset(&R, 0, sizeof(R));
        R.prompt_len = np;
        // createLogitsFilters (TextDecoder.swift:857-899): SuppressBlank(sampleBegin = prefilledIndex = 0), TimestampRules(sampleBegin = initialPrompt.count)
        R.sample_begin_ts = o.without_timestamps ? -1 : np;
        R.sample_begin_blank = o.suppress_blank ? 0 : -1;
        R.max_steps = std::max(1, std::min(o.sample_length, kKvMaxLen - 1));   // TextDecoder.swift:566
        R.temperature = rung_temperature(o, rung); R.top_k = o.top_k;
        R.has_first_thr = o.has_first_token_logprob_threshold; R.first_thr = o.first_token_logprob_threshold;
        R.seed = o.seed + (uint64_t)rung;
        R.suppress_off = sup_off[oi]; R.n_suppress = sup_n[oi];
        // the language slot: the position after the first SOT, when it holds a language token; without one the detection only reports
        R.lang_slot = -1; R.lang_flags = 0;
        if (detects(o)) {
            R.lang_flags = p[0] == st->start_of_transcript_token ? kLangDetect : kLangPreStep;
            for (int i = 0; i < np; ++i)
                if (p[i] == st->start_of_transcript_token) { if (i + 1 < np && is_language(p[i + 1])) R.lang_slot = i + 1; break; }
        }
        if (n_adm == 0) cudaEventSynchronize(s->ev_stage);   // the previous round's copies out of the pinned staging have landed
        for (int j = 0; j < beam; ++j) {                     // beam search: `beam` identical rows start the window
            s->h_adm_slots[n_adm] = slot * beam + j;
            memset(s->h_adm_prompts + (size_t)n_adm * kKvMaxLen, 0, kKvMaxLen * 4);
            memcpy(s->h_adm_prompts + (size_t)n_adm * kKvMaxLen, p, (size_t)np * 4);
            s->h_adm_rp[n_adm] = R;
            ++n_adm;
        }
        s->slot_window[slot] = (int)w;
        s->slot_try[slot] = rung;
    };
    auto prompt_len_of = [&](int64_t w) -> int { const int32_t* p; int np; prompt_of(w, &p, &np); return np; };
    auto flush_admissions = [&]() -> wk_status {
        if (n_adm == 0) return WK_OK;
        WK_CUDA_CHECK(cudaMemcpyAsync(s->d_adm_slots, s->h_adm_slots, (size_t)n_adm * 4, cudaMemcpyHostToDevice, s->stream));
        WK_CUDA_CHECK(cudaMemcpyAsync(s->d_adm_prompts, s->h_adm_prompts, (size_t)n_adm * kKvMaxLen * 4, cudaMemcpyHostToDevice, s->stream));
        WK_CUDA_CHECK(cudaMemcpyAsync(s->d_adm_rp, s->h_adm_rp, (size_t)n_adm * sizeof(RowParams), cudaMemcpyHostToDevice, s->stream));
        if (s->align_on)
            for (int i = 0; i < n_adm; ++i)   // row 0 and unreached rows of alignmentWeights stay 0
                WK_CUDA_CHECK(cudaMemsetAsync((char*)s->align_w + (size_t)s->h_adm_slots[i] * kKvMaxLen * T * 2, 0, (size_t)kKvMaxLen * T * 2, s->stream));
        WK_CHECK(decode_slots_init(s->st, s->rp_dev, s->d_adm_slots, s->d_adm_prompts, s->d_adm_rp, n_adm, s->stream, s->bs));
        WK_CUDA_CHECK(cudaEventRecord(s->ev_stage, s->stream));
        n_adm = 0;
        return WK_OK;
    };

    // ---- encoder pipeline state
    const int Ec = bound ? 0 : std::max(1, std::min(bo->encoder_chunk > 0 ? bo->encoder_chunk : c.max_batch, c.max_batch));
    int64_t enc_next = 0, chunk_w0 = 0, chunk_n = 0, chunk_adm = 0;
    bool chunk_waited = true;
    float acc[6] = {0, 0, 0, 0, 0, 0};
    struct EncTiming { bool pending = false; } et;
    if (!bound) WK_CHECK(enc_ws_ensure(m, &s->ws, c.max_batch));
    auto launch_encode = [&]() -> wk_status {
        const int64_t nc = std::min<int64_t>(Ec, n - enc_next);
        std::vector<int32_t> spw_fixed;
        const int32_t* spw = a.spw ? a.spw + enc_next : nullptr;
        if (a.spw) {   // windows that already failed validation are encoded as silence: they never reach a slot
            bool any_bad = false;
            for (int64_t i = 0; i < nc; ++i) any_bad |= status[enc_next + i] != WK_OK;
            if (any_bad) {
                spw_fixed.assign(a.spw + enc_next, a.spw + enc_next + nc);
                for (int64_t i = 0; i < nc; ++i) if (status[enc_next + i] != WK_OK) spw_fixed[i] = 0;
                spw = spw_fixed.data();
            }
        }
        cudaStream_t es = s->enc_stream;
        WK_CUDA_CHECK(cudaStreamWaitEvent(es, s->ev_adm, 0));   // the previous chunk's cross-KV projections have read enc_out
        WK_CUDA_CHECK(cudaEventRecord(s->ev_t[0], es));
        const float* src = a.pcm + enc_next * a.stride;
        cudaPointerAttributes pat;
        const bool on_dev = cudaPointerGetAttributes(&pat, src) == cudaSuccess && pat.type == cudaMemoryTypeDevice;
        cudaGetLastError();
        if (!on_dev || a.stride < kWindowSamples) {   // stage here so that the copy is timed apart from the mel kernel
            if (a.stride < kWindowSamples) WK_CUDA_CHECK(cudaMemsetAsync(s->ws.pcm_dev, 0, (size_t)nc * kWindowSamples * 4, es));
            WK_CUDA_CHECK(cudaMemcpy2DAsync(s->ws.pcm_dev, kWindowSamples * 4, src, a.stride * 4, std::min<int64_t>(a.stride, kWindowSamples) * 4, nc,
                                            cudaMemcpyDefault, es));
            src = s->ws.pcm_dev;
        }
        const int64_t src_stride = (!on_dev || a.stride < kWindowSamples) ? kWindowSamples : a.stride;
        WK_CUDA_CHECK(cudaEventRecord(s->ev_t[1], es));
        WK_CHECK(mel_run(m, &s->ws, src, nc, src_stride, spw, s->ws.mel, es));
        WK_CUDA_CHECK(cudaEventRecord(s->ev_t[2], es));
        WK_CHECK(encode_chunk(m, &s->ws, s->ws.mel, (int)nc, s->ws.enc_out, es));
        WK_CUDA_CHECK(cudaEventRecord(s->ev_t[3], es));
        WK_CUDA_CHECK(cudaEventRecord(s->ev_enc, es));
        chunk_w0 = enc_next; chunk_n = nc; chunk_adm = 0; enc_next += nc; chunk_waited = false;
        et.pending = true;
        return WK_OK;
    };
    auto collect_enc_timing = [&]() {
        if (!et.pending || cudaEventQuery(s->ev_t[3]) != cudaSuccess) return;
        float t;
        cudaEventElapsedTime(&t, s->ev_t[0], s->ev_t[1]); acc[4] += t;
        cudaEventElapsedTime(&t, s->ev_t[1], s->ev_t[2]); acc[0] += t;
        cudaEventElapsedTime(&t, s->ev_t[2], s->ev_t[3]); acc[1] += t;
        et.pending = false;
    };
    // cross-attention K/V of windows [w0, w0+cnt) of the encoded chunk into slots [q0, q0+cnt)
    auto project_cross_kv = [&](int64_t w0, int q0, int cnt) -> wk_status {
        if (!chunk_waited) { WK_CUDA_CHECK(cudaStreamWaitEvent(s->stream, s->ev_enc, 0)); chunk_waited = true; }
        const char* src = (const char*)s->ws.enc_out + (size_t)(w0 - chunk_w0) * T * d * 2;
        GemmDesc g = plain_gemm(src, (int64_t)cnt * T, d, m->wckv, 2 * c.dec_layers * d, c.dtype, GEMM_OUT_T16_HEADS,
                                (char*)s->cross_kv + (size_t)q0 * c.n_heads * T * 64 * 2, 0, m->bckv, 0);
        g.heads_T = T; g.heads_B = s->max_batch; g.heads_H = c.n_heads; g.heads_dmodel = d;
        return gemm_tcgen05(g, m->num_sms, s->stream);
    };

    // TranscriptionResult.language of every window: detectedLanguage ?? defaultLanguageCode (TranscribeTask.swift:341-376) - the kept rung's
    // detection, else the explicit language, else the first language token of the result (TextDecoder.swift:804-822), else English
    if (a.ladder) { s->win_lang_tok.assign((size_t)n, st->english_token); s->win_lang_lp.assign((size_t)n, 0.f); }
    auto record_language = [&](int64_t w, const wk_decode_result& r, int r0) {
        if (!a.ladder) return;
        const wk_decode_opts& o = opts_of(bo, w);
        int32_t tok = st->english_token; float lp = 0.f;
        if (detects(o)) { tok = s->h_lang_tok[r0]; lp = s->h_lang_lp[r0]; }
        else if (o.language_token >= 0) tok = o.language_token;
        else
            for (int i = 0; i < r.n_tokens; ++i)
                if (is_language(r.tokens[i])) { tok = r.tokens[i]; lp = r.token_logprobs[i]; break; }
        s->win_lang_tok[(size_t)w] = tok; s->win_lang_lp[(size_t)w] = lp;
    };

    int64_t finished = 0;
    for (int64_t w = 0; w < n; ++w) if (status[w] != WK_OK) ++finished;
    memset(s->stats, 0, sizeof(s->stats));
    int live = 0;
    bool ckv_timing = false;
    if (bound) {
        // decodeText on the bound rows: window w sits in slot w with its cross K/V already projected
        for (int64_t w = 0; w < n; ++w)
            if (status[w] == WK_OK) { stage_admission((int)w, w, 0); ++live; ++s->stats[2]; }
        WK_CHECK(flush_admissions());
    }
    while (finished < n) {
        // (A) next chunk through mel + encoder as soon as the previous chunk has left enc_out
        if (!bound && chunk_adm == chunk_n && enc_next < n) WK_CHECK(launch_encode());
        // (B) admit encoded windows into free slots; consecutive windows going to consecutive slots share one projection GEMM
        if (!bound && chunk_adm < chunk_n) {
            int run_q0 = -1, run_cnt = 0; int64_t run_w0 = 0;
            bool first_gemm = true;
            auto flush_run = [&]() -> wk_status {
                if (run_cnt == 0) return WK_OK;
                if (first_gemm && !ckv_timing) {
                    if (!chunk_waited) { WK_CUDA_CHECK(cudaStreamWaitEvent(s->stream, s->ev_enc, 0)); chunk_waited = true; }   // timed region starts once the encoder output exists
                    WK_CUDA_CHECK(cudaEventRecord(s->ev_t[4], s->stream));
                }
                first_gemm = false;
                wk_status r = project_cross_kv(run_w0, run_q0, run_cnt);
                run_cnt = 0;
                return r;
            };
            for (int q = 0; q < Brun && chunk_adm < chunk_n; ++q) {
                if (s->slot_window[q] >= 0) { WK_CHECK(flush_run()); continue; }
                while (chunk_adm < chunk_n && status[chunk_w0 + chunk_adm] != WK_OK) { WK_CHECK(flush_run()); ++chunk_adm; }
                if (chunk_adm >= chunk_n) break;
                const int64_t w = chunk_w0 + chunk_adm;
                if (run_cnt > 0 && (q != run_q0 + run_cnt || w != run_w0 + run_cnt)) WK_CHECK(flush_run());
                if (run_cnt == 0) { run_q0 = q; run_w0 = w; }
                ++run_cnt;
                stage_admission(q, w, 0);
                ++live; ++s->stats[2];
                ++chunk_adm;
            }
            WK_CHECK(flush_run());
            while (chunk_adm < chunk_n && status[chunk_w0 + chunk_adm] != WK_OK) ++chunk_adm;
            if (!first_gemm && !ckv_timing) { WK_CUDA_CHECK(cudaEventRecord(s->ev_t[5], s->stream)); ckv_timing = true; }
            if (chunk_adm == chunk_n) WK_CUDA_CHECK(cudaEventRecord(s->ev_adm, s->stream));
            WK_CHECK(flush_admissions());
        }
        if (live == 0) {
            if (!bound && (chunk_adm < chunk_n || enc_next < n)) continue;
            break;
        }
        // (C) a burst of decode steps, then the state comes back in one go
        WK_CUDA_CHECK(cudaEventRecord(s->ev_t[6], s->stream));
        WK_CHECK(run_steps(s, st, poll, live == Brun));
        s->stats[0] += poll; s->stats[1] += (int64_t)poll * live;
        WK_CUDA_CHECK(cudaEventRecord(s->ev_t[7], s->stream));
        WK_CUDA_CHECK(cudaMemcpyAsync(s->h_done, s->st.done, rows * 4, cudaMemcpyDeviceToHost, s->stream));
        WK_CUDA_CHECK(cudaMemcpyAsync(s->h_n_tokens, s->st.n_tokens, rows * 4, cudaMemcpyDeviceToHost, s->stream));
        WK_CUDA_CHECK(cudaMemcpyAsync(s->h_steps, s->st.steps, rows * 4, cudaMemcpyDeviceToHost, s->stream));
        WK_CUDA_CHECK(cudaMemcpyAsync(s->h_first_low, s->st.first_low, rows * 4, cudaMemcpyDeviceToHost, s->stream));
        WK_CUDA_CHECK(cudaMemcpyAsync(s->h_error, s->st.error, rows * 4, cudaMemcpyDeviceToHost, s->stream));
        WK_CUDA_CHECK(cudaMemcpyAsync(s->h_tokens, s->st.tokens, (size_t)rows * kKvMaxLen * 4, cudaMemcpyDeviceToHost, s->stream));
        WK_CUDA_CHECK(cudaMemcpyAsync(s->h_logprobs, s->st.logprobs, (size_t)rows * kKvMaxLen * 4, cudaMemcpyDeviceToHost, s->stream));
        if (any_detect) {
            WK_CUDA_CHECK(cudaMemcpyAsync(s->h_lang_tok, s->st.lang_tok, rows * 4, cudaMemcpyDeviceToHost, s->stream));
            WK_CUDA_CHECK(cudaMemcpyAsync(s->h_lang_lp, s->st.lang_lp, rows * 4, cudaMemcpyDeviceToHost, s->stream));
        }
        if (beam > 1) {
            WK_CUDA_CHECK(cudaMemcpyAsync(s->h_sum_lp, s->bs.sum_lp, rows * 4, cudaMemcpyDeviceToHost, s->stream));
            WK_CUDA_CHECK(cudaMemcpyAsync(s->h_n_fin, s->bs.n_fin, Brun * 4, cudaMemcpyDeviceToHost, s->stream));
            WK_CUDA_CHECK(cudaMemcpyAsync(s->h_fin_len, s->bs.fin_len, (size_t)Brun * kMaxCand * 4, cudaMemcpyDeviceToHost, s->stream));
            WK_CUDA_CHECK(cudaMemcpyAsync(s->h_fin_score, s->bs.fin_score, (size_t)Brun * kMaxCand * 4, cudaMemcpyDeviceToHost, s->stream));
            WK_CUDA_CHECK(cudaMemcpyAsync(s->h_fin_tokens, s->bs.fin_tokens, (size_t)Brun * kMaxCand * kKvMaxLen * 4, cudaMemcpyDeviceToHost, s->stream));
            WK_CUDA_CHECK(cudaMemcpyAsync(s->h_fin_lps, s->bs.fin_lps, (size_t)Brun * kMaxCand * kKvMaxLen * 4, cudaMemcpyDeviceToHost, s->stream));
        }
        {
            cudaError_t e = cudaStreamSynchronize(s->stream);
            if (e != cudaSuccess) { set_error("decode loop: %s", cudaGetErrorString(e)); return WK_ERR_DECODING_FAILED; }
        }
        {
            float t;
            cudaEventElapsedTime(&t, s->ev_t[6], s->ev_t[7]); acc[3] += t;
            if (ckv_timing) { cudaEventElapsedTime(&t, s->ev_t[4], s->ev_t[5]); acc[2] += t; ckv_timing = false; }
            collect_enc_timing();
        }
        // (D) retire ended windows; progress callback / early stop for the live ones
        for (int q = 0; q < Brun; ++q) {
            const int w = s->slot_window[q];
            if (w < 0) continue;
            const int r0 = q * beam;                  // first decode row of the slot (the only one without beam search)
            const wk_decode_opts& o = opts_of(bo, w);
            bool ended = s->h_done[r0] != 0, stopped = false;
            if (!ended && bo->progress) {
                const int nt = s->h_n_tokens[r0];
                float sum = 0.f;
                for (int i = 0; i < nt; ++i) sum += s->h_logprobs[(size_t)r0 * kKvMaxLen + i];
                if (!bo->progress(bo->progress_user, w, s->h_tokens + (size_t)r0 * kKvMaxLen, nt, nt > 0 ? sum / nt : 0.f)) {
                    // callback -> false: the reference's early-stop flag ends the loop at the next token (TextDecoder.swift:733-762)
                    std::vector<int32_t> ones(beam, 1);
                    WK_CUDA_CHECK(cudaMemcpyAsync(s->st.done + r0, ones.data(), beam * 4, cudaMemcpyHostToDevice, s->stream));
                    WK_CUDA_CHECK(cudaStreamSynchronize(s->stream));
                    stopped = true;              // an early-stopped window does not walk the ladder
                    ended = true;
                }
            }
            if (!ended) continue;
            wk_decode_result r;
            const int rung = s->slot_try[q];
            const int32_t* seq_tok = s->h_tokens + (size_t)r0 * kKvMaxLen;
            const float* seq_lp = s->h_logprobs + (size_t)r0 * kKvMaxLen;
            int seq_n = s->h_n_tokens[r0];
            std::vector<int32_t> btok; std::vector<float> blp;
            if (beam > 1) {
                // BeamSearchDecoder.finalize + MaximumLikelihoodRanker (oracle/beam_ref.py): the finished list, topped up with the live beams
                // (best sum first) to `beam` entries; the winner maximises sum_logprob / sampled tokens
                struct Cand { const int32_t* tok; const float* lp; int len; float score; bool live; };
                std::vector<Cand> cands;
                const int nf = std::min(s->h_n_fin[q], kMaxCand);
                for (int f = 0; f < nf; ++f) {
                    const size_t slot = (size_t)q * kMaxCand + f;
                    cands.push_back(Cand{s->h_fin_tokens + slot * kKvMaxLen, s->h_fin_lps + slot * kKvMaxLen, s->h_fin_len[slot], s->h_fin_score[slot], false});
                }
                if ((int)cands.size() < beam) {
                    std::vector<int> order(beam);
                    for (int j = 0; j < beam; ++j) order[j] = j;
                    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return s->h_sum_lp[r0 + x] > s->h_sum_lp[r0 + y]; });
                    for (int j : order) {
                        const int rr = r0 + j;
                        cands.push_back(Cand{s->h_tokens + (size_t)rr * kKvMaxLen, s->h_logprobs + (size_t)rr * kKvMaxLen, s->h_n_tokens[rr] + 1, s->h_sum_lp[rr], true});
                        if ((int)cands.size() >= beam) break;
                    }
                }
                const int P = prompt_len_of(w);
                int best = 0; float best_rank = -INFINITY;
                for (size_t i = 0; i < cands.size(); ++i) {
                    const float rk = cands[i].score / (float)std::max(cands[i].len - P - 1, 1);
                    if (i == 0 || rk > best_rank) { best = (int)i; best_rank = rk; }
                }
                const Cand& cd = cands[best];
                const int body = cd.live ? cd.len - 1 : cd.len;      // live beams carry no EOT yet: finalize_result appends it
                btok.assign(cd.tok, cd.tok + body); blp.assign(cd.lp, cd.lp + body);
                seq_tok = btok.data(); seq_lp = blp.data(); seq_n = body;
            }
            finalize_result(r, seq_tok, seq_lp, seq_n, s->h_steps[r0], s->h_first_low[r0], st, &o, rung_temperature(o, rung));
            if (s->h_error[r0]) {
                set_error("window %d: no finite logit at decoder step %d", w, s->h_steps[r0] - 1);
                fail_window(w, WK_ERR_DECODING_LOGITS_FAILED);
            } else if (a.ladder && beam == 1 && !stopped && r.needs_fallback && s->slot_try[q] < o.temperature_fallback_count) {
                // decodeWithFallback (TranscribeTask.swift:316-411): same encoder output (the slot keeps its cross K/V), next temperature
                stage_admission(q, w, s->slot_try[q] + 1);
                ++s->stats[3];
                continue;
            } else {
                a.results[w] = r;
                record_language(w, r, r0);
            }
            if (s->align_on && status[w] == WK_OK)
                WK_CUDA_CHECK(cudaMemcpyAsync((char*)s->align_store + (size_t)w * kKvMaxLen * T * 2, (char*)s->align_w + (size_t)q * kKvMaxLen * T * 2,
                                              (size_t)kKvMaxLen * T * 2, cudaMemcpyDeviceToDevice, s->stream));
            s->slot_window[q] = -1;
            --live;
            ++finished;
        }
        WK_CHECK(flush_admissions());   // ladder re-admissions
    }
    WK_CUDA_CHECK(cudaStreamSynchronize(s->stream));
    if (!bound) {
        WK_CUDA_CHECK(cudaStreamSynchronize(s->enc_stream));
        collect_enc_timing();
        memcpy(m->timings, acc, sizeof(acc));
    }
    if (!bo->status)
        for (int64_t w = 0; w < n; ++w) if (status[w] != WK_OK) { set_error("%s", first_err.c_str()); return status[w]; }
    return WK_OK;
}

}  // namespace wk

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

wk_status wk_session_create(wk_model* m, int32_t max_batch, wk_session** out) {
    if (!m || !out || max_batch < 1 || max_batch > 256) { set_error("wk_session_create: bad arguments (max_batch %d, limit 256)", max_batch); return WK_ERR_INVALID_ARGUMENT; }
    WK_CUDA_CHECK(cudaSetDevice(m->device));
    const wk_model_config& c = m->cfg;
    const int d = c.d_model, H = c.n_heads, L = c.dec_layers, T = c.n_audio_ctx, S = max_batch;
    wk_session* s = new wk_session();
    s->m = m;
    s->max_batch = S;
    // A/B switches, read once per session (never on the step path).  WKB200_FUSED=1 runs the decoder's GEMM / reduce phases as persistent
    // chains with grid barriers (fused_chain.cu): bit-identical, but measured SLOWER on B200 than one PDL-chained launch per phase
    // (64 windows: 1252 vs 1198 ms per pass; a phase costs ~4.5 us of dependent L2 round trips either way and a grid barrier is no
    // cheaper than a programmatic kernel boundary), so it is off by default.  WKB200_NO_GRAPH=1 replays nothing.
    if (const char* e = getenv("WKB200_FUSED")) s->knob_fused = atoi(e) != 0;
    s->knob_graph = getenv("WKB200_NO_GRAPH") == nullptr;
    WK_CUDA_CHECK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    WK_CUDA_CHECK(cudaStreamCreateWithFlags(&s->enc_stream, cudaStreamNonBlocking));
    const int bpm = round_up(S, 16);
    WK_CHECK(alloc16(&s->cross_kv, (size_t)2 * L * S * H * T * 64));
    WK_CHECK(alloc16(&s->self_k, (size_t)L * S * H * kKvMaxLen * 64));
    WK_CHECK(alloc16(&s->self_v, (size_t)L * S * H * kKvMaxLen * 64));
    // split-K partial workspace: max over the decoder GEMM shapes of splits * N
    size_t pe = 0;
    const int shapes[4][2] = {{3 * d, d}, {d, d}, {4 * d, d}, {d, 4 * d}};
    for (auto& sh : shapes) {
        const int sp = choose_splits((sh[0] + 127) / 128, sh[1] / 64, m->num_sms);
        pe = std::max(pe, (size_t)sp * sh[0]);
    }
    s->partial_elems = pe * bpm;
    WK_CHECK(dmalloc(&s->partial, s->partial_elems));
    WK_CHECK(dmalloc(&s->x, (size_t)bpm * d));
    WK_CHECK(alloc16(&s->xn, (size_t)bpm * d));
    WK_CHECK(alloc16(&s->attn, (size_t)bpm * d));
    WK_CHECK(alloc16(&s->ffn, (size_t)bpm * 4 * d));
    WK_CHECK(dmalloc(&s->logits, (size_t)S * c.vocab));
    WK_CHECK(dmalloc(&s->st.tokens, (size_t)S * kKvMaxLen));
    WK_CHECK(dmalloc(&s->st.n_tokens, S));
    WK_CHECK(dmalloc(&s->st.logprobs, (size_t)S * kKvMaxLen));
    WK_CHECK(dmalloc(&s->st.next_token, S));
    WK_CHECK(dmalloc(&s->st.done, S));
    WK_CHECK(dmalloc(&s->st.first_low, S));
    WK_CHECK(dmalloc(&s->st.steps, S));
    WK_CHECK(dmalloc(&s->st.input_ids, S));
    WK_CHECK(dmalloc(&s->st.error, S));
    WK_CHECK(dmalloc(&s->st.lang_tok, S));
    WK_CHECK(dmalloc(&s->st.lang_lp, S));
    WK_CHECK(dmalloc(&s->rp_dev, S));
    s->st.rp = s->rp_dev;
    WK_CHECK(dmalloc(&s->pos_dev, S));
    WK_CHECK(dmalloc(&s->lang_dev, 4096));
    s->suppress_cap = 4096;
    WK_CHECK(dmalloc(&s->suppress_dev, s->suppress_cap));
    WK_CHECK(dmalloc(&s->d_adm_slots, S));
    WK_CHECK(dmalloc(&s->d_adm_prompts, (size_t)S * kKvMaxLen));
    WK_CHECK(dmalloc(&s->d_adm_rp, S));
    WK_CHECK(dmalloc(&s->chain_counters, (size_t)L * 2 * 8));
    auto pinned = [&](void** p, size_t bytes) -> wk_status {
        cudaError_t e = cudaHostAlloc(p, bytes, cudaHostAllocDefault);
        if (e != cudaSuccess) { set_error("cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return WK_ERR_CUDA; }
        memset(*p, 0, bytes);
        return WK_OK;
    };
    WK_CHECK(pinned((void**)&s->h_adm_slots, (size_t)S * 4));
    WK_CHECK(pinned((void**)&s->h_adm_prompts, (size_t)S * kKvMaxLen * 4));
    WK_CHECK(pinned((void**)&s->h_adm_rp, (size_t)S * sizeof(RowParams)));
    WK_CHECK(pinned((void**)&s->h_tokens, (size_t)S * kKvMaxLen * 4));
    WK_CHECK(pinned((void**)&s->h_logprobs, (size_t)S * kKvMaxLen * 4));
    WK_CHECK(pinned((void**)&s->h_n_tokens, (size_t)S * 4));
    WK_CHECK(pinned((void**)&s->h_done, (size_t)S * 4));
    WK_CHECK(pinned((void**)&s->h_first_low, (size_t)S * 4));
    WK_CHECK(pinned((void**)&s->h_steps, (size_t)S * 4));
    WK_CHECK(pinned((void**)&s->h_error, (size_t)S * 4));
    WK_CHECK(pinned((void**)&s->h_lang_tok, (size_t)S * 4));
    WK_CHECK(pinned((void**)&s->h_lang_lp, (size_t)S * 4));
    WK_CUDA_CHECK(cudaEventCreateWithFlags(&s->ev_enc, cudaEventDisableTiming));
    WK_CUDA_CHECK(cudaEventCreateWithFlags(&s->ev_adm, cudaEventDisableTiming));
    WK_CUDA_CHECK(cudaEventCreateWithFlags(&s->ev_stage, cudaEventDisableTiming));
    for (auto& e : s->ev_t) WK_CUDA_CHECK(cudaEventCreate(&e));
    WK_CUDA_CHECK(cudaDeviceSynchronize());  // setup memsets ran on the legacy default stream
    WK_CUDA_CHECK(cudaEventRecord(s->ev_adm, s->stream));
    WK_CUDA_CHECK(cudaEventRecord(s->ev_stage, s->stream));
    s->slot_window.assign(S, -1);
    s->slot_try.assign(S, 0);
    m->live_sessions.fetch_add(1);
    *out = s;
    return WK_OK;
}

void wk_session_free(wk_session* s) {
    if (!s) return;
    cudaSetDevice(s->m->device);
    cudaStreamSynchronize(s->stream);
    cudaStreamSynchronize(s->enc_stream);
    s->m->live_sessions.fetch_sub(1);
    if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
    if (s->graph_exec_live) cudaGraphExecDestroy(s->graph_exec_live);
    void* ptrs[] = {s->cross_kv, s->self_k, s->self_v, s->partial, s->x, s->xn, s->attn, s->ffn, s->logits, s->st.tokens, s->st.n_tokens,
                    s->st.logprobs, s->st.next_token, s->st.done, s->st.first_low, s->st.steps, s->st.input_ids, s->st.error, s->rp_dev,
                    s->pos_dev, s->lang_dev, s->suppress_dev, s->d_adm_slots, s->d_adm_prompts, s->d_adm_rp, s->align_scratch, s->align_w,
                    s->align_store, s->chain_counters, s->st.lang_tok, s->st.lang_lp};
    for (void* p : ptrs) if (p) cudaFree(p);
    void* hptrs[] = {s->h_adm_slots, s->h_adm_prompts, s->h_adm_rp, s->h_tokens, s->h_logprobs, s->h_n_tokens, s->h_done, s->h_first_low, s->h_steps, s->h_error,
                     s->h_lang_tok, s->h_lang_lp};
    for (void* p : hptrs) if (p) cudaFreeHost(p);
    enc_ws_free(&s->ws);
    cudaEventDestroy(s->ev_enc); cudaEventDestroy(s->ev_adm); cudaEventDestroy(s->ev_stage);
    for (auto& e : s->ev_t) cudaEventDestroy(e);
    cudaStreamDestroy(s->stream);
    cudaStreamDestroy(s->enc_stream);
    delete s;
}

wk_status wk_session_reset(wk_session* s) {
    if (!s) return WK_ERR_INVALID_ARGUMENT;
    WK_CUDA_CHECK(cudaSetDevice(s->m->device));
    const wk_model_config& c = s->m->cfg;
    const size_t n = (size_t)c.dec_layers * s->max_batch * c.n_heads * kKvMaxLen * 64 * 2;
    WK_CUDA_CHECK(cudaMemsetAsync(s->self_k, 0, n, s->stream));
    WK_CUDA_CHECK(cudaMemsetAsync(s->self_v, 0, n, s->stream));
    return WK_OK;
}

wk_status wk_session_set_encoder_output(wk_session* s, const wk_tensor* enc) {
    if (!s || !enc) { set_error("wk_session_set_encoder_output: null argument"); return WK_ERR_INVALID_ARGUMENT; }
    wk_model* m = s->m;
    if (enc->kind != 1 || enc->owner != m) { set_error("encoder output does not belong to this model"); return WK_ERR_INVALID_ARGUMENT; }
    if (enc->batch < 1 || enc->batch > s->max_batch) { set_error("encoder batch %lld exceeds session max_batch %d", (long long)enc->batch, s->max_batch); return WK_ERR_PREPARE_DECODER_INPUTS; }
    WK_CUDA_CHECK(cudaSetDevice(m->device));
    const wk_model_config& c = m->cfg;
    const int d = c.d_model, T = c.n_audio_ctx;
    s->batch = (int)enc->batch;
    s->bound_windows = s->batch;
    s->bs.beam = 1;
    s->bp = round_up(s->batch, 16);
    // the encoder ran on the model stream; the projection reads its output on the session stream and the tensor remembers the reader
    std::lock_guard<std::mutex> lock(m->api_mu);
    for (cudaEvent_t e : enc->events) WK_CUDA_CHECK(cudaStreamWaitEvent(s->stream, e, 0));
    GemmDesc g = plain_gemm(enc->data, (int64_t)s->batch * T, d, m->wckv, 2 * c.dec_layers * d, c.dtype, GEMM_OUT_T16_HEADS, s->cross_kv, 0, m->bckv, 0);
    g.heads_T = T; g.heads_B = s->max_batch; g.heads_H = c.n_heads; g.heads_dmodel = d;
    WK_CHECK(gemm_tcgen05(g, m->num_sms, s->stream));
    cudaEvent_t ev;
    WK_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    WK_CUDA_CHECK(cudaEventRecord(ev, s->stream));
    const_cast<wk_tensor*>(enc)->events.push_back(ev);
    return WK_OK;
}

wk_status wk_build_prompt(const wk_model* m, const wk_special_tokens* st, const wk_decode_opts* o, int32_t use_options, int32_t* out, int32_t cap, int32_t* n) {
    if (!m || !st || !out || !n) return WK_ERR_INVALID_ARGUMENT;
    std::vector<int32_t> p;
    WK_CHECK(build_prompt(m, st, o, use_options, p));
    if ((int)p.size() > cap) { set_error("wk_build_prompt: capacity %d < %zu", cap, p.size()); return WK_ERR_PREPARE_DECODER_INPUTS; }
    memcpy(out, p.data(), p.size() * 4);
    *n = (int)p.size();
    return WK_OK;
}

wk_status wk_decode_step(wk_session* s, const int32_t* input_ids, const int32_t* cache_length, float* logits_out) {
    if (!s || !input_ids || !cache_length) { set_error("wk_decode_step: null argument"); return WK_ERR_INVALID_ARGUMENT; }
    wk_model* m = s->m;
    if (s->batch < 1) { set_error("wk_decode_step: no encoder output bound"); return WK_ERR_PREPARE_DECODER_INPUTS; }
    WK_CUDA_CHECK(cudaSetDevice(m->device));
    for (int i = 0; i < s->batch; ++i) {
        if (cache_length[i] < 0 || cache_length[i] >= kKvMaxLen) { set_error("wk_decode_step: cache_length[%d]=%d out of range", i, cache_length[i]); return WK_ERR_DECODING_LOGITS_FAILED; }
        if (input_ids[i] < 0 || input_ids[i] >= m->cfg.vocab) { set_error("wk_decode_step: input_ids[%d]=%d out of range", i, input_ids[i]); return WK_ERR_DECODING_LOGITS_FAILED; }
    }
    WK_CUDA_CHECK(cudaMemcpyAsync(s->st.input_ids, input_ids, s->batch * 4, cudaMemcpyHostToDevice, s->stream));
    WK_CUDA_CHECK(cudaMemcpyAsync(s->pos_dev, cache_length, s->batch * 4, cudaMemcpyHostToDevice, s->stream));
    WK_CHECK(decoder_forward(s, 0, 0, s->pos_dev, use_fused(s)));
    if (logits_out)
        WK_CUDA_CHECK(cudaMemcpyAsync(logits_out, s->logits, (size_t)s->batch * m->cfg.vocab * 4, cudaMemcpyDeviceToHost, s->stream));
    cudaError_t e = cudaStreamSynchronize(s->stream);
    if (e != cudaSuccess) { set_error("wk_decode_step: %s", cudaGetErrorString(e)); return WK_ERR_DECODING_LOGITS_FAILED; }
    return WK_OK;
}

wk_status wk_session_last_logits(wk_session* s, float* logits_out) {
    if (!s || !logits_out) return WK_ERR_INVALID_ARGUMENT;
    WK_CUDA_CHECK(cudaSetDevice(s->m->device));
    WK_CUDA_CHECK(cudaMemcpyAsync(logits_out, s->logits, (size_t)s->batch * s->m->cfg.vocab * 4, cudaMemcpyDeviceToHost, s->stream));
    WK_CUDA_CHECK(cudaStreamSynchronize(s->stream));
    return WK_OK;
}

// TextDecoder.detectLanguage (TextDecoder.swift:420-539): one decoder step on [SOT] at position 0, LanguageLogitsFilter
// (keep only the language tokens), GreedyTokenSampler -> language token id + logprob for every bound window.
wk_status wk_detect_language(wk_session* s, const wk_special_tokens* st, const int32_t* language_tokens, int32_t n_language_tokens,
                             float temperature, int32_t* token_out, float* logprob_out) {
    if (!s || !st || !language_tokens || n_language_tokens < 1 || n_language_tokens > 4096 || !token_out) {
        set_error("wk_detect_language: bad arguments");
        return WK_ERR_INVALID_ARGUMENT;
    }
    wk_model* m = s->m;
    if (s->batch < 1) { set_error("wk_detect_language: no encoder output bound"); return WK_ERR_PREPARE_DECODER_INPUTS; }
    WK_CUDA_CHECK(cudaSetDevice(m->device));
    const int B = s->batch;
    std::vector<int32_t> ids(B, st->start_of_transcript_token), zeros(B, 0), ones(B, 1);
    WK_CUDA_CHECK(cudaMemcpyAsync(s->st.input_ids, ids.data(), B * 4, cudaMemcpyHostToDevice, s->stream));
    WK_CUDA_CHECK(cudaMemcpyAsync(s->pos_dev, zeros.data(), B * 4, cudaMemcpyHostToDevice, s->stream));
    WK_CHECK(decoder_forward(s, 0, 0, s->pos_dev, use_fused(s)));
    // currentTokens = [SOT] for every window: reuse the decode-state arrays as the stateless token history
    WK_CUDA_CHECK(cudaMemcpyAsync(s->st.tokens, ids.data(), B * 4, cudaMemcpyHostToDevice, s->stream));   // ld_tokens = 1
    WK_CUDA_CHECK(cudaMemcpyAsync(s->st.n_tokens, ones.data(), B * 4, cudaMemcpyHostToDevice, s->stream));
    WK_CUDA_CHECK(cudaMemcpyAsync(s->lang_dev, language_tokens, n_language_tokens * 4, cudaMemcpyHostToDevice, s->stream));
    SamplerParams p;
    memset(&p, 0, sizeof(p));
    p.st = *st; p.vocab = m->cfg.vocab; p.is_multilingual = 1; p.loop_mode = 0;
    p.sample_begin_ts = -1; p.sample_begin_blank = -1;
    p.language_tokens = s->lang_dev; p.n_language_tokens = n_language_tokens; p.language_sample_begin = 0;
    p.temperature = temperature; p.top_k = 5; p.seed = 0;
    p.max_ctx = kKvMaxLen;
    DecodeState none;
    memset(&none, 0, sizeof(none));
    WK_CHECK(sampler_filter_sample(s->logits, m->cfg.vocab, p, none, s->st.tokens, 1, s->st.n_tokens, s->st.next_token, s->st.logprobs, nullptr, B, s->stream));
    WK_CUDA_CHECK(cudaMemcpyAsync(token_out, s->st.next_token, B * 4, cudaMemcpyDeviceToHost, s->stream));
    if (logprob_out) WK_CUDA_CHECK(cudaMemcpyAsync(logprob_out, s->st.logprobs, B * 4, cudaMemcpyDeviceToHost, s->stream));
    cudaError_t e = cudaStreamSynchronize(s->stream);
    if (e != cudaSuccess) { set_error("wk_detect_language: %s", cudaGetErrorString(e)); return WK_ERR_DECODING_FAILED; }
    return WK_OK;
}

wk_status wk_decode_text_ex(wk_session* s, const wk_special_tokens* st, const wk_batch_opts* bo, wk_decode_result* results) {
    if (!s || !st || !bo || !bo->opts || bo->n_opts < 1 || !results) { set_error("wk_decode_text: null argument"); return WK_ERR_INVALID_ARGUMENT; }
    if (s->bound_windows < 1) { set_error("wk_decode_text: no encoder output bound"); return WK_ERR_PREPARE_DECODER_INPUTS; }
    if (bo->n_opts != 1 && bo->n_opts != s->bound_windows) { set_error("wk_decode_text: %d option sets for %d windows", bo->n_opts, s->bound_windows); return WK_ERR_INVALID_ARGUMENT; }
    WK_CUDA_CHECK(cudaSetDevice(s->m->device));
    CoreArgs a{nullptr, s->bound_windows, 0, nullptr, st, bo, results, false};
    return transcribe_core(s, a);
}

wk_status wk_decode_text(wk_session* s, const wk_special_tokens* st, const wk_decode_opts* o, const int32_t* prompt, int32_t n_prompt,
                         wk_decode_result* results) {
    if (!s || !st || !o || !prompt || !results) { set_error("wk_decode_text: null argument"); return WK_ERR_INVALID_ARGUMENT; }
    wk_batch_opts bo;
    memset(&bo, 0, sizeof(bo));
    bo.opts = o; bo.n_opts = 1; bo.prompt = prompt; bo.n_prompt = n_prompt;
    return wk_decode_text_ex(s, st, &bo, results);
}

wk_status wk_transcribe_windows_ex(wk_model* m, wk_session* s, const float* pcm_host, int64_t n_windows, int64_t stride,
                                   const int32_t* samples_per_window, const wk_special_tokens* st, const wk_batch_opts* bo,
                                   wk_decode_result* results) {
    if (!m || !s || !pcm_host || !st || !bo || !bo->opts || bo->n_opts < 1 || !results || n_windows < 1) { set_error("wk_transcribe_windows: null argument"); return WK_ERR_INVALID_ARGUMENT; }
    if (s->m != m) { set_error("wk_transcribe_windows: session belongs to another model"); return WK_ERR_INVALID_ARGUMENT; }
    if (bo->n_opts != 1 && bo->n_opts != n_windows) { set_error("wk_transcribe_windows: %d option sets for %lld windows", bo->n_opts, (long long)n_windows); return WK_ERR_INVALID_ARGUMENT; }
    if (bo->prompts && !bo->prompt_lens) { set_error("wk_transcribe_windows: prompts without prompt_lens"); return WK_ERR_INVALID_ARGUMENT; }
    if (!m->finalized) { set_error("wk_transcribe_windows: model weights not finalized"); return WK_ERR_MODELS_UNAVAILABLE; }
    WK_CUDA_CHECK(cudaSetDevice(m->device));
    CoreArgs a{pcm_host, n_windows, stride, samples_per_window, st, bo, results, true};
    return transcribe_core(s, a);
}

wk_status wk_transcribe_windows(wk_model* m, wk_session* s, const float* pcm_host, int64_t n_windows, int64_t stride,
                                const int32_t* samples_per_window, const wk_special_tokens* st, const wk_decode_opts* opts,
                                const int32_t* prompt, int32_t n_prompt, wk_decode_result* results) {
    if (!opts || !prompt) { set_error("wk_transcribe_windows: null argument"); return WK_ERR_INVALID_ARGUMENT; }
    wk_batch_opts bo;
    memset(&bo, 0, sizeof(bo));
    bo.opts = opts; bo.n_opts = 1; bo.prompt = prompt; bo.n_prompt = n_prompt;
    return wk_transcribe_windows_ex(m, s, pcm_host, n_windows, stride, samples_per_window, st, &bo, results);
}

wk_status wk_session_stats(const wk_session* s, int64_t* out4) {
    if (!s || !out4) return WK_ERR_INVALID_ARGUMENT;
    memcpy(out4, s->stats, sizeof(s->stats));
    return WK_OK;
}

wk_status wk_session_set_language_tokens(wk_session* s, const int32_t* tokens, int32_t n) {
    if (!s || n < 0 || n > 4096 || (n > 0 && !tokens)) { set_error("wk_session_set_language_tokens: bad arguments (n %d, limit 4096)", n); return WK_ERR_INVALID_ARGUMENT; }
    for (int i = 0; i < n; ++i)
        if (tokens[i] < 0 || tokens[i] >= s->m->cfg.vocab) { set_error("wk_session_set_language_tokens: token %d outside the vocabulary", tokens[i]); return WK_ERR_INVALID_ARGUMENT; }
    s->lang_list.assign(tokens, tokens + n);
    return WK_OK;
}

wk_status wk_session_languages(const wk_session* s, int64_t n, int32_t* tokens, float* logprobs) {
    if (!s || n < 0 || (n > 0 && !tokens)) { set_error("wk_session_languages: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    if (n > (int64_t)s->win_lang_tok.size()) { set_error("wk_session_languages: %lld windows asked, the last call had %zu", (long long)n, s->win_lang_tok.size()); return WK_ERR_INVALID_ARGUMENT; }
    if (n > 0) memcpy(tokens, s->win_lang_tok.data(), (size_t)n * 4);
    if (n > 0 && logprobs) memcpy(logprobs, s->win_lang_lp.data(), (size_t)n * 4);
    return WK_OK;
}

wk_status wk_session_alignment_weights(wk_session* s, int32_t window, int32_t rows, float* out) {
    if (!s || !out || window < 0 || rows < 0 || rows > kKvMaxLen) { set_error("wk_session_alignment_weights: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    if (!s->align_on || !s->align_store || window >= s->align_store_n) { set_error("wk_session_alignment_weights: the last decode did not ask for word timestamps (or window %d is outside it)", window); return WK_ERR_INVALID_ARGUMENT; }
    WK_CUDA_CHECK(cudaSetDevice(s->m->device));
    const size_t T = s->m->cfg.n_audio_ctx;
    std::vector<__half> h((size_t)rows * T);
    WK_CUDA_CHECK(cudaMemcpyAsync(h.data(), (const __half*)s->align_store + (size_t)window * kKvMaxLen * T, h.size() * 2, cudaMemcpyDeviceToHost, s->stream));
    WK_CUDA_CHECK(cudaStreamSynchronize(s->stream));
    for (size_t i = 0; i < h.size(); ++i) out[i] = __half2float(h[i]);
    return WK_OK;
}

wk_status wk_session_alignment_weights_f16(wk_session* s, int32_t window, int32_t rows, uint16_t* out, int32_t sync) {
    if (!s || !out || window < 0 || rows < 0 || rows > kKvMaxLen) { set_error("wk_session_alignment_weights_f16: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    if (!s->align_on || !s->align_store || window >= s->align_store_n) { set_error("wk_session_alignment_weights_f16: the last decode did not ask for word timestamps (or window %d is outside it)", window); return WK_ERR_INVALID_ARGUMENT; }
    WK_CUDA_CHECK(cudaSetDevice(s->m->device));
    const size_t T = s->m->cfg.n_audio_ctx;
    if (rows > 0)
        WK_CUDA_CHECK(cudaMemcpyAsync(out, (const __half*)s->align_store + (size_t)window * kKvMaxLen * T, (size_t)rows * T * 2, cudaMemcpyDeviceToHost, s->stream));
    if (sync) WK_CUDA_CHECK(cudaStreamSynchronize(s->stream));
    return WK_OK;
}

// Average device time (ms) of one launch of a named hot kernel on the session's buffers (CUDA events on the stream the kernel runs on;
// decoder-side kernels are replayed `iters` times as one CUDA graph so that host launch cost stays out, as in the real step):
//   0 decoder cross-attention (one layer, `batch` live rows)      1 encoder FC1+GELU GEMM (M = batch*1500)   2 log-mel
//   3 encoder attention      4 decoder QKV swap-AB GEMM      5 encoder QKV GEMM      6/7 decoder d x d / FC2 GEMM (L2-warm weights)
//   8 split-K reduce + LN    9 decoder self-attention at position 100      10 sampler (V-long rows)
//   14-17 decoder GEMMs with the weights rotating over the layers (HBM-cold: d x d, FC1, FC2, QKV)
//   18 / 19 the fused phase chains B / C of one layer, weights rotating over the layers
// Also returns the algorithmic bytes (HBM-bound kernels) or FLOPs (tensor-bound) of one launch.
wk_status wk_bench_kernel(wk_model* m, wk_session* s, int32_t which, int32_t batch, int32_t iters, float* ms_out, double* work_out) {
    if (!m || !s || s->m != m || !ms_out || !work_out || iters < 1) return WK_ERR_INVALID_ARGUMENT;
    WK_CUDA_CHECK(cudaSetDevice(m->device));
    const wk_model_config& c = m->cfg;
    const int d = c.d_model, T = c.n_audio_ctx, H = c.n_heads, dt = c.dtype;
    const bool enc_side = which == 1 || which == 2 || which == 3 || which == 5;
    int B = batch;
    if (B < 1 || B > (enc_side ? c.max_batch : s->max_batch)) { set_error("wk_bench_kernel: bad batch"); return WK_ERR_INVALID_ARGUMENT; }
    if (enc_side) WK_CHECK(enc_ws_ensure(m, &s->ws, c.max_batch));
    const int64_t M = (int64_t)B * T;
    cudaStream_t st = enc_side ? s->enc_stream : s->stream;
    const int saved_batch = s->batch, saved_bp = s->bp;
    if (!enc_side) { s->batch = B; s->bp = round_up(B, 16); }
    const size_t cross_block = (size_t)s->max_batch * H * T * 64 * 2;
    static int32_t* pos100 = nullptr;
    if (which == 9 && !pos100) { std::vector<int32_t> h(256, 100); cudaMalloc(&pos100, 256 * 4); cudaMemcpy(pos100, h.data(), 256 * 4, cudaMemcpyHostToDevice); }
    int rot = 0;
    auto chain_desc = [&](int li, int which_chain, ChainDesc* cd) {
        memset(cd, 0, sizeof(*cd));
        const DecLayer& l = m->dec[li];
        cd->partial = s->partial; cd->x = s->x; cd->B = B; cd->Bp = s->bp; cd->d = d; cd->dtype = dt; cd->pdl = 0;
        const int set = rot & 1;   // alternate two word sets: each launch re-arms the other one
        cd->counters = s->chain_counters + set * 8; cd->reset_counters = s->chain_counters + (set ^ 1) * 8;
        auto gp = [&](const void* w, int N, int K, const void* act) { ChainPhaseDesc ph; memset(&ph, 0, sizeof(ph)); ph.kind = 0; ph.w = w; ph.n = N; ph.k = K; ph.act = act; ph.splits = choose_splits((N + 127) / 128, K / 64, m->num_sms); return ph; };
        auto lp = [&](const float* bias, const LayerNormW& ln) { ChainPhaseDesc ph; memset(&ph, 0, sizeof(ph)); ph.kind = 1; ph.bias = bias; ph.gamma = ln.g; ph.beta = ln.b; ph.out16 = s->xn; return ph; };
        if (which_chain == 0) {
            cd->ph[0] = gp(l.wo, d, d, s->attn); cd->ph[1] = lp(l.bo, l.lnx); cd->ph[2] = gp(l.wcq, d, d, s->xn); cd->n_phases = 3;
        } else {
            cd->ph[0] = gp(l.wco, d, d, s->attn); cd->ph[1] = lp(l.bco, l.ln3); cd->ph[2] = gp(l.w1, 4 * d, d, s->xn);
            cd->ph[3].kind = 2; cd->ph[3].bias = l.b1; cd->ph[3].out16 = s->ffn;
            cd->ph[4] = gp(l.w2, d, 4 * d, s->ffn); cd->ph[5] = lp(l.b2, l.ln1); cd->ph[6] = gp(l.wqkv, 3 * d, d, s->xn); cd->n_phases = 7;
        }
    };
    auto run = [&]() -> wk_status {
        int sp;
        switch (which) {
            case 0: return decoder_cross_attention(s->partial, 1, s->bp, m->dec[0].bcq, s->cross_kv, (char*)s->cross_kv + cross_block, s->attn, B, H, T, dt, st);
            case 1: return gemm_tcgen05(plain_gemm(s->ws.xn, M, d, m->enc[0].w1, 4 * d, dt, GEMM_OUT_T16, s->ws.ffn, 4 * d, m->enc[0].b1, 1), m->num_sms, st);
            case 2: return mel_forward(m->mel_tables, s->ws.pcm_dev, B, kWindowSamples, nullptr, s->ws.mel, s->ws.gmax, st);
            case 3: return encoder_attention(s->ws.qkv, s->ws.attn, B, T, H, dt, st);
            case 4: return dec_gemm(s, m->dec[0].wqkv, 3 * d, d, s->xn, &sp);
            case 5: return gemm_tcgen05(plain_gemm(s->ws.xn, M, d, m->enc[0].wqkv, 3 * d, dt, GEMM_OUT_T16, s->ws.qkv, 3 * d, m->enc[0].bqkv, 0), m->num_sms, st);
            case 6: return dec_gemm(s, m->dec[0].wo, d, d, s->attn, &sp);
            case 7: return dec_gemm(s, m->dec[0].w2, d, 4 * d, s->ffn, &sp);
            case 8: return decoder_reduce_resid_ln(s->partial, choose_splits((d + 127) / 128, d / 64, m->num_sms), s->bp, m->dec[0].bo, m->dec[0].lnx.g, m->dec[0].lnx.b, s->x, s->xn, B, d, dt, st);
            case 9: return decoder_self_attention(s->partial, 1, s->bp, m->dec[0].bq, m->dec[0].bv, s->self_k, s->self_v, pos100, nullptr, s->attn, B, H, kKvMaxLen, dt, st);
            case 14: case 15: case 16: case 17: {
                const int r = rot++;
                const DecLayer& l = m->dec[r % c.dec_layers];
                if (which == 14) { const void* w3[3] = {l.wo, l.wcq, l.wco}; return dec_gemm(s, w3[(r / c.dec_layers) % 3], d, d, s->attn, &sp); }
                if (which == 15) return dec_gemm(s, l.w1, 4 * d, d, s->xn, &sp);
                if (which == 16) return dec_gemm(s, l.w2, d, 4 * d, s->ffn, &sp);
                return dec_gemm(s, l.wqkv, 3 * d, d, s->xn, &sp);
            }
            case 18: case 19: {
                ChainDesc cd;
                chain_desc(rot % c.dec_layers, which - 18, &cd);
                ++rot;
                return decoder_chain(cd, m->num_sms, st);
            }
            default: set_error("wk_bench_kernel: unknown kernel %d", which); return WK_ERR_INVALID_ARGUMENT;
        }
    };
    switch (which) {
        case 0: *work_out = (double)B * H * T * 64 * 2 * 2; break;                         // K + V bytes
        case 1: *work_out = 2.0 * (double)M * d * 4 * d; break;                            // FLOPs
        case 2: *work_out = (double)B * (kWindowSamples * 4.0 + c.n_mels * 3000 * 2.0); break;  // bytes (SURVEY 8d)
        case 3: *work_out = 4.0 * (double)B * H * T * T * 64; break;                       // FLOPs
        case 4: case 17: *work_out = 3.0 * d * d * 2; break;                               // weight bytes
        case 5: *work_out = 2.0 * (double)M * d * 3 * d; break;
        case 6: case 14: *work_out = 1.0 * d * d * 2; break;
        case 7: case 15: case 16: *work_out = 4.0 * d * d * 2; break;
        case 9: *work_out = (double)B * H * 100 * 64 * 2 * 2; break;                       // K + V rows read at position 100
        case 18: *work_out = 2.0 * d * d * 2; break;                                       // out-proj + cross-Q weights
        case 19: *work_out = 12.0 * d * d * 2; break;                                      // cross-out + FC1 + FC2 + QKV weights
        default: *work_out = 0; break;
    }
    wk_status rs = WK_OK;
    for (int i = 0; i < 2 && rs == WK_OK; ++i) rs = run();
    float t = 0.f;
    if (rs == WK_OK && !enc_side) {
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        WK_CUDA_CHECK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        for (int i = 0; i < iters && rs == WK_OK; ++i) rs = run();
        WK_CUDA_CHECK(cudaStreamEndCapture(st, &graph));
        if (rs == WK_OK) {
            WK_CUDA_CHECK(cudaGraphInstantiate(&exec, graph, 0));
            WK_CUDA_CHECK(cudaGraphLaunch(exec, st));
            WK_CUDA_CHECK(cudaEventRecord(s->ev_t[8], st));
            WK_CUDA_CHECK(cudaGraphLaunch(exec, st));
            WK_CUDA_CHECK(cudaEventRecord(s->ev_t[9], st));
            WK_CUDA_CHECK(cudaEventSynchronize(s->ev_t[9]));
            cudaEventElapsedTime(&t, s->ev_t[8], s->ev_t[9]);
            cudaGraphExecDestroy(exec);
        }
        if (graph) cudaGraphDestroy(graph);
    } else if (rs == WK_OK) {
        WK_CUDA_CHECK(cudaEventRecord(s->ev_t[8], st));
        for (int i = 0; i < iters && rs == WK_OK; ++i) rs = run();
        WK_CUDA_CHECK(cudaEventRecord(s->ev_t[9], st));
        WK_CUDA_CHECK(cudaEventSynchronize(s->ev_t[9]));
        cudaEventElapsedTime(&t, s->ev_t[8], s->ev_t[9]);
    }
    s->batch = saved_batch; s->bp = saved_bp;
    *ms_out = t / iters;
    return rs;
}

// Debug readback of an internal buffer as f32 (tests/tools only).  which: session encoder workspace 0 mel[Bm,3002,128] 1 h1[Bm,3002,d]
// 2 x[M,d] 3 xn[M,d] 4 qkv[M,3d] 5 attn[M,d] 6 ffn[M,4d] 7 enc_out[M,d]; decode 10 x[Bp,d] 11 xn[Bp,d] 12 attn[Bp,d]
// 13 ffn[Bp,4d] 14 logits[S,V] 15 cross_kv (all) 16 self_k (all) 17 self_v (all) 18 partial; 20.. weights
wk_status wk_debug_read(wk_model* m, wk_session* s, int32_t which, int64_t offset_elems, float* dst, int64_t n) {
    if (!m || !dst) return WK_ERR_INVALID_ARGUMENT;
    WK_CUDA_CHECK(cudaSetDevice(m->device));
    const EncWorkspace* ws = s ? &s->ws : &m->ws;
    const void* src = nullptr;
    int dt = m->cfg.dtype;
    switch (which) {
        case 0: src = ws->mel; dt = WK_DTYPE_F16; break;
        case 1: src = ws->h1; dt = WK_DTYPE_F16; break;
        case 2: src = ws->x; dt = WK_DTYPE_F32; break;
        case 3: src = ws->xn; break;
        case 4: src = ws->qkv; break;
        case 5: src = ws->attn; break;
        case 6: src = ws->ffn; break;
        case 7: src = ws->enc_out; break;
        case 10: src = s ? s->x : nullptr; dt = WK_DTYPE_F32; break;
        case 11: src = s ? s->xn : nullptr; break;
        case 12: src = s ? s->attn : nullptr; break;
        case 13: src = s ? s->ffn : nullptr; break;
        case 14: src = s ? s->logits : nullptr; dt = WK_DTYPE_F32; break;
        case 15: src = s ? s->cross_kv : nullptr; break;
        case 16: src = s ? s->self_k : nullptr; break;
        case 17: src = s ? s->self_v : nullptr; break;
        case 18: src = s ? s->partial : nullptr; dt = WK_DTYPE_F32; break;
        case 20: src = m->enc[0].wqkv; break;
        case 21: src = m->emb; break;
        case 22: src = m->enc[0].w1; break;
        case 23: src = m->wckv; break;
        case 24: src = m->enc[0].b1; dt = WK_DTYPE_F32; break;
        case 25: src = m->enc[0].bqkv; dt = WK_DTYPE_F32; break;
        default: break;
    }
    if (!src) { set_error("wk_debug_read: unknown or unallocated buffer %d", which); return WK_ERR_INVALID_ARGUMENT; }
    std::lock_guard<std::mutex> lock(m->api_mu);
    float* tmp = nullptr;
    WK_CUDA_CHECK(cudaMalloc(&tmp, n * 4));
    WK_CUDA_CHECK(cudaDeviceSynchronize());
    wk_status r = convert_to_16((const char*)src + offset_elems * esize(dt), dt, tmp, WK_DTYPE_F32, n, m->stream);
    if (r == WK_OK) {
        cudaError_t e = cudaMemcpyAsync(dst, tmp, n * 4, cudaMemcpyDeviceToHost, m->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(m->stream);
        if (e != cudaSuccess) { set_error("wk_debug_read: %s", cudaGetErrorString(e)); r = WK_ERR_CUDA; }
    }
    cudaFree(tmp);
    return r;
}

}  // extern "C"
