// Internal launcher declarations shared by the .cu files of libwkb200.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/wkb200.h"

namespace wk {

void set_error(const char* fmt, ...);
const char* last_error_cstr();
void count_launch(int n = 1);

// ---------------------------------------------------------------- GEMM (gemm_tcgen05.cu)
enum GemmMode {
    GEMM_OUT_T16 = 0,        // out16[row, col] = act(acc + bias[col])
    GEMM_OUT_F32_ADD = 1,    // out32[row, col] += acc + bias[col]           (residual update in place)
    GEMM_OUT_F32_GELU_POS = 2,  // out32[row, col] = gelu(acc + bias[col]) + pos[row_in_batch, col]
    GEMM_OUT_PARTIAL_T = 3,  // out32[split][col][row] = acc                  (swap-AB split-K partials)
    GEMM_OUT_T16_HEADS = 4,  // out16[which][b][h][t][64] head-major scatter  (cross-attention K/V cache)
    GEMM_OUT_F32 = 5,        // out32[row, col] = acc + bias[col]
};

struct GemmDesc {
    // A operand: [a_rows, K] 16-bit, K contiguous.  If a_batches > 1 it is a 3-D tensor
    // [a_batches][a_rows_per_batch][a_cols] addressed per batch (conv-as-GEMM with taps).
    const void* a;
    int64_t a_rows;          // rows (per batch if a_batches > 1)
    int64_t a_cols;          // row length in elements (>= K for tap addressing)
    int64_t a_ld;            // row stride in elements
    int64_t a_batch_stride;  // elements between batches (3-D only)
    int a_batches;           // 1 = plain 2-D
    int a_3d;                // address A through a 3-D tensor map [a_batches][a_rows][a_cols]
    // B operand: [b_rows, K_total] 16-bit, K contiguous (weights [N,K] or, swap-AB, activations)
    const void* b;
    int64_t b_rows;
    int64_t b_ld;
    int in_dtype;            // WK_DTYPE_BF16 / WK_DTYPE_F16
    // problem
    int m_rows_per_batch;    // output rows per batch (== valid A rows per batch for this op)
    int n;                   // valid output columns (<= b_rows)
    int k;                   // K per tap (multiple of 64)
    int taps;                // 1, or 3 for the conv stem
    int tap_row_shift[3];    // A row offset per tap
    int tap_col_off[3];      // A column offset per tap (elements)
    int bn;                  // tile N (multiple of 16, <= 256)
    int splits;              // split-K (GEMM_OUT_PARTIAL_T only), divides taps*k/64
    // epilogue
    int mode;
    int gelu;
    void* out;
    int64_t ld_out;          // row stride of out (elements); PARTIAL_T: elements per [col] row = total M
    int64_t out_rows_per_batch;  // global out row = batch*out_rows_per_batch + row_in_batch
    int64_t partial_cols;    // PARTIAL_T: number of col rows per split (padded batch)
    const float* bias;       // indexed by col (row for PARTIAL_T is not biased)
    const float* pos;        // GELU_POS: [m_rows_per_batch, ld_pos]
    int64_t ld_pos;
    // HEADS scatter
    int heads_T, heads_B, heads_H, heads_dmodel;
    int pdl;                 // launch with programmatic dependent launch (decode-step chain)
    int max_stages;          // 0 = as many smem stages as fit; >0 caps the ring (lets other kernels co-reside on the SM)
    int a_static;            // A operand (weights) does not depend on the upstream kernel: with PDL its first tiles are fetched before griddepcontrol.wait
    int pair;                // run as 2-CTA clusters sharing the B (weight) tile by TMA multicast (plain 2-D, single-split GEMMs)
};

wk_status gemm_tcgen05(const GemmDesc& d, int num_sms, cudaStream_t stream);

// ---------------------------------------------------------------- mel (mel.cu)
struct MelTables;  // device tables (window, twiddles, sparse filterbank)
wk_status mel_tables_create(int n_mels, MelTables** out);
void mel_tables_free(MelTables* t);
// pcm [n_windows, stride] f32 device; out [n_windows, 3002, 128] f16 (rows 0 and 3001 are the conv zero pad, mel
// channels >= n_mels zero); gmax scratch [n_windows] int32
wk_status mel_forward(const MelTables* t, const float* pcm, int64_t n_windows, int64_t stride, const int32_t* n_valid,
                      void* out_f16, int32_t* gmax_scratch, cudaStream_t stream);
constexpr int kMelRows = 3002;
constexpr int kMelCols = 128;

// ---------------------------------------------------------------- encoder ops (encoder_ops.cu)
wk_status layernorm_f32_to_16(const float* x, const float* gamma, const float* beta, void* out, int64_t rows, int d, int dtype,
                              cudaStream_t stream);
wk_status layernorm_f32_to_f32(const float* x, const float* gamma, const float* beta, float* out, int64_t rows, int d,
                               cudaStream_t stream);
wk_status encoder_attention(const void* qkv, void* out, int B, int T, int n_heads, int dtype, cudaStream_t stream);
// tcgen05/TMA implementation (attention_tcgen05.cu) behind encoder_attention()
wk_status encoder_attention_tcgen05(const void* qkv, void* out, int B, int T, int n_heads, int dtype, cudaStream_t stream);
wk_status transpose_to_host_layout(const void* src, float* dst, int64_t B, int64_t rows, int64_t cols, int64_t src_rows_alloc,
                                   int64_t src_row_off, int64_t src_ld, int dtype, cudaStream_t stream);
wk_status fill_random_16(void* dst, int64_t n, uint64_t seed, float std, float mean, int dtype, cudaStream_t stream);
wk_status fill_random_f32(float* dst, int64_t n, uint64_t seed, float std, float mean, cudaStream_t stream);
wk_status convert_to_16(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, cudaStream_t stream);

// ---------------------------------------------------------------- decoder ops (decoder_ops.cu)
// Per-row decode options, device-resident: what differs between the items of transcribeWithOptions' decodeOptionsArray
// (WhisperKit.swift:716-735) and between the rungs of the temperature ladder (TranscribeTask.swift:316-411).
struct RowParams {
    int32_t prompt_len;          // initialPrompt.count
    int32_t sample_begin_ts;     // TimestampRulesFilter.sampleBegin, <0 = filter absent
    int32_t sample_begin_blank;  // SuppressBlankFilter.sampleBegin, <0 = absent
    int32_t max_steps;           // min(sampleLength, 223): loop bound (TextDecoder.swift:566)
    float temperature; int32_t top_k;
    int32_t has_first_thr; float first_thr;
    uint64_t seed;
    int32_t suppress_off, n_suppress;   // slice of the session's suppress-token pool
    // DecodingOptions.detectLanguage (TranscribeTask.swift:339-365): the row samples its language from the logits of SOT at position 0
    // (LanguageLogitsFilter over SamplerParams.language_tokens, then the rung's sampler) before its decode goes on
    int32_t lang_slot;           // prompt position the detected language is written to (the token after the first SOT), -1 = none
    int32_t lang_flags;          // kLangDetect | kLangPreStep
};
// kLangDetect: the row detects at step 0 (its prompt starts with SOT, so step 0 already runs SOT at position 0).
// kLangPreStep: the prompt starts elsewhere (<|startofprev|>): one extra pass feeds SOT at position 0, detects, and leaves steps at 0.
constexpr int32_t kLangDetect = 1, kLangPreStep = 2;

struct DecodeState {
    // all device pointers; one entry per decode row (slot).  A slot with done != 0 is skipped by every kernel of the step.
    int32_t* tokens;      // [Bmax, 224] currentTokens
    int32_t* n_tokens;    // [Bmax]
    float* logprobs;      // [Bmax, 224]
    int32_t* next_token;  // [Bmax]
    int32_t* done;        // [Bmax]
    int32_t* first_low;   // [Bmax]
    int32_t* steps;       // [Bmax] forward passes consumed = tokenIndex of the step about to run = KV-cache position
    int32_t* input_ids;   // [Bmax] token fed at this step (written by embed)
    int32_t* error;       // [Bmax] 1 = the sampler saw no finite logit (WhisperError.decodingLogitsFailed)
    const RowParams* rp;  // [Bmax]
    int32_t* lang_tok;    // [Bmax] detected language token, -1 = not detected (yet)
    float* lang_lp;       // [Bmax] its log-probability under the language filter
};

// Beam search (SURVEY 8f row 2; semantics restated from openai/whisper BeamSearchDecoder in oracle/beam_ref.py - the reference's
// BeamSearchTokenSampler is a fatalError stub, TokenSampler.swift:254-290).  Decode rows come in groups of `beam` consecutive rows per window.
constexpr int kMaxBeam = 8;
constexpr int kMaxCand = 8;        // maxCandidates = Int(Float(beamSize) * patience) (TokenSampler.swift:266)
struct BeamState {
    int beam;                      // rows per window; <= 1 = greedy / sampling, every field below unused
    int max_candidates;
    float* sum_lp;                 // [rows] cumulative log-prob of the sampled tokens of the beam
    int32_t* cand_tok; float* cand_lp;   // [rows][kMaxBeam + 1] best tokens of the step's filtered log-softmax, best first (-1 = none)
    int32_t* anc;                  // [rows][224] physical cache row that holds position t of this beam's self K/V
    int32_t* fin_tokens; float* fin_lps;   // [groups][kMaxCand][224] finished sequences (EOT included), per-token log-probs (EOT -> 0)
    int32_t* fin_len; float* fin_score;    // [groups][kMaxCand]
    int32_t* n_fin;                // [groups]
};

struct SamplerParams {
    wk_special_tokens st;
    int vocab;
    int is_multilingual;
    int loop_mode;           // 1: decode loop (per-row options from DecodeState.rp); 0: stateless (wk_filter_sample / detectLanguage)
    const int32_t* suppress; // loop mode: the pool RowParams.suppress_off indexes; stateless: the list itself
    // stateless: LanguageLogitsFilter(sampleBegin = language_sample_begin); loop mode: the session's allLanguageTokens, read only at the
    // detection step of rows with RowParams.lang_flags set
    const int32_t* language_tokens; int n_language_tokens; int language_sample_begin;
    int max_ctx;             // 224
    BeamState beam;          // loop mode with beam.beam > 1: the kernel only ranks candidates; beam_update() does the bookkeeping
    // stateless mode only
    int sample_begin_ts, sample_begin_blank, n_suppress;
    float temperature; int top_k; uint64_t seed;
};

// pos: explicit per-row positions (wk_decode_step) or nullptr = DecodeState.steps.  sot: the token a language-detection pre-step feeds
wk_status decoder_embed_ln(const void* emb16, const float* pos, const float* gamma, const float* beta, DecodeState st, int vocab,
                           int ts_begin, int sot, float* x, void* xn, int B, int d, int dtype, const int32_t* explicit_pos, cudaStream_t stream);
// x[b,:] += bias + sum_s partial[s][b][:]; xn = LN(x) (16-bit).  partial layout [S][Bp][d]
wk_status decoder_reduce_resid_ln(const float* partial, int splits, int Bp, const float* bias, const float* gamma,
                                  const float* beta, float* x, void* xn, int B, int d, int dtype, cudaStream_t stream);
// h = gelu(bias + sum partial) 16-bit [B, n]
wk_status decoder_reduce_bias_gelu(const float* partial, int splits, int Bp, const float* bias, void* out, int B, int n,
                                   int dtype, cudaStream_t stream);
// self attention for one new token per sequence; reduces qkv partials [S][Bp][3d], appends K/V at pos[b].  done != nullptr: rows with
// done[b] != 0 are skipped (their window has ended: no cache traffic)
// anc != nullptr (beam search): position t of row b is read from cache row anc[b][t]; the new row is written to row b itself
wk_status decoder_self_attention(const float* partial, int splits, int Bp, const float* bq, const float* bv, void* kcache,
                                 void* vcache, const int32_t* pos, const int32_t* done, void* out, int B, int H,
                                 int max_len, int dtype, cudaStream_t stream, const int32_t* anc = nullptr);
// cross attention over T encoder positions; reduces q partials [S][Bp][d]; K/V [B][H][T][64]
// align_scratch != nullptr: heads h with bit h of align_mask set also write their softmax row (f32, [slot][B][T], slot = rank of h in
// the mask) - the alignment heads behind the reference decoder's `alignment_heads_weights` output (TextDecoder.swift:310,414)
wk_status decoder_cross_attention(const float* partial, int splits, int Bp, const float* bq, const void* kcross,
                                  const void* vcross, void* out, int B, int H, int T, int dtype, cudaStream_t stream,
                                  const int32_t* done = nullptr, float* align_scratch = nullptr, uint32_t align_mask = 0, int kv_div = 1);
// kv_div > 1 (beam search): row b reads the K/V block of window b / kv_div; the CTAs of one (window, head) are adjacent in the grid so that
// their K/V stream is shared through L2
// tensor-core variant for nq = 2..8 rows per K/V block (cross_attention_mq.cu): one K/V stream per (window, head) serves all nq beams
wk_status decoder_cross_attention_mq(const float* partial, int splits, int Bp, const float* bq, const void* kcross, const void* vcross, void* out, int B, int H,
                                     int Tlen, int dtype, cudaStream_t stream, const int32_t* done, int nq);
// alignment row of the step just sampled (run AFTER the sampler advanced steps[b] to tokenIndex + 1): out[b][steps[b]][t] =
// Float16(mean over n_slots of scratch[slot][b][t]) unless done[b] (TextDecoder.updateAlignmentWeights, TextDecoder.swift:272-296:
// the slice of step tokenIndex lands in row tokenIndex + 1; a completed segment breaks out before the update, :668-674)
wk_status decoder_align_mean(const float* scratch, int n_slots, const int32_t* steps, const int32_t* done, void* out_f16, int B, int T,
                             int max_rows, cudaStream_t stream);
wk_status sampler_filter_sample(const float* logits, int64_t ld_logits, SamplerParams p, DecodeState st, const int32_t* tokens,
                                int ld_tokens, const int32_t* n_tokens, int32_t* token_out, float* logprob_out,
                                float* filtered_out, int B, cudaStream_t stream);
// (re)starts the decode of n slots: slot_ids[i] gets prompt row i of prompts [n][224] (length rp[i].prompt_len) and RowParams rp[i]
wk_status decode_slots_init(DecodeState st, RowParams* rp_dev, const int32_t* slot_ids, const int32_t* prompts, const RowParams* rp_new,
                            int n, cudaStream_t stream, BeamState beam = BeamState());
// the beam-search step after the sampler ranked every row's candidates: per window, merge the beams' candidates, move finished sequences
// to the finished list, permute token / log-prob histories and cache ancestry to the surviving beams, advance the loop state
wk_status beam_update(DecodeState st, BeamState beam, wk_special_tokens sp, int max_ctx, int groups, cudaStream_t stream);

// ---- a chain of decoder GEMM / split-K reduce phases in ONE persistent kernel with grid-wide barriers between the phases instead of
// kernel boundaries (fused_chain.cu)
wk_status make_tmap_2d(void* tm, const void* base, int dtype, uint64_t cols, uint64_t rows, uint64_t ld_elems, uint32_t box_cols, uint32_t box_rows);
constexpr int kChainMaxPhases = 7;
constexpr int kChainMaxGemms = 4;
struct ChainPhaseDesc {
    int kind;                  // 0 swap-AB split-K GEMM -> partials; 1 reduce + bias + residual + LayerNorm; 2 reduce + bias + GELU
    // kind 0
    const void* w; int n, k;   // weights [n][k]
    const void* act;           // activations [Bp][k], 16-bit
    int splits;
    // kind 1 / 2 (reduce the partials of the GEMM phase before it)
    const float* bias; const float* gamma; const float* beta;
    void* out16;               // LN output / GELU output, 16-bit [B][row length]
};
struct ChainDesc {
    int n_phases;
    ChainPhaseDesc ph[kChainMaxPhases];
    float* partial; float* x;  // split-K workspace, f32 residual stream [Bp][d]
    int B, Bp, d, dtype;
    unsigned int* counters;    // 8 words, zero before the launch: one per phase boundary
    unsigned int* reset_counters;  // 8 words of the sibling chain (already completed): zeroed by this launch; may be nullptr
    int pdl;
};
wk_status decoder_chain(const ChainDesc& c, int num_sms, cudaStream_t stream);

}  // namespace wk
