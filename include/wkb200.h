/*
 * wkb200.h - C ABI of libwkb200.so: the Blackwell (sm_100a) implementation of WhisperKit's hot path
 *            PCM -> log-mel -> audio encoder -> KV-cached text decoder -> logits filters -> sampler.
 *
 * Every entry point is what a Swift (or Python ctypes) host binds to replace one member of the
 * reference's protocol surface (paths relative to the WhisperKit repo):
 *
 *   wk_mel                  FeatureExtracting.logMelSpectrogram   Sources/WhisperKit/Core/FeatureExtractor.swift:13-17,40-56
 *   wk_encode               AudioEncoding.encodeFeatures          Sources/WhisperKit/Core/AudioEncoder.swift:10-18,50-63
 *   wk_session_create/reset TextDecoding.prepareDecoderInputs     Sources/WhisperKit/Core/TextDecoder.swift:109-161
 *   wk_build_prompt         TextDecoding.prefillDecoderInputs     Sources/WhisperKit/Core/TextDecoder.swift:163-216
 *   wk_decode_step          TextDecoding.predictLogits            Sources/WhisperKit/Core/TextDecoder.swift:361-418
 *   wk_detect_language      TextDecoding.detectLanguage           Sources/WhisperKit/Core/TextDecoder.swift:420-539
 *   wk_filter_sample        LogitsFiltering.filterLogits (x4) +   Sources/WhisperKit/Core/Text/LogitsFilter.swift:8-276
 *                           TokenSampling.update                  Sources/WhisperKit/Core/Text/TokenSampler.swift:8-11,215-240
 *   wk_decode_text          TextDecoding.decodeText (+ sampler    Sources/WhisperKit/Core/TextDecoder.swift:541-855
 *                           finalize, DecodingFallback)           Sources/WhisperKit/Core/Models.swift:357-381
 *   wk_transcribe_windows   the per-window body of                Sources/WhisperKit/Core/TranscribeTask.swift:116-278
 *                           TranscribeTask.run, batched like      Sources/WhisperKit/Core/WhisperKit.swift:716-812
 *                           WhisperKit.transcribeWithOptions
 *   wk_model_info           melCount/windowSamples/embedSize/     FeatureExtractor.swift:24-38, AudioEncoder.swift:24-38,
 *                           logitsSize/kvCache* properties        TextDecoder.swift:313-331
 *
 * Conventions: plain C types only; every function returns a wk_status (0 = ok, negative = error, mapped
 * 1:1 onto WhisperError cases, Sources/WhisperKit/Utilities/WhisperError.swift:6-19); the message of the
 * last error on the calling thread is wk_last_error().  Host pointers may be pageable or pinned; pointers
 * documented as "host or device" are resolved with cudaPointerGetAttributes.
 *
 * Threading (the reference calls the same protocol objects from up to concurrentWorkerCount tasks, WhisperKit.swift:735-791):
 * a finalized wk_model is immutable and may be used from any number of host threads - the model-level entry points
 * (wk_mel, wk_encode, wk_filter_sample, wk_tensor_*) serialise internally; a wk_session (the per-task DecodingInputs of
 * TranscribeTask.swift:83 plus its own mel/encoder workspace and CUDA streams) belongs to one thread at a time, and different
 * sessions of one model run concurrently.  wk_tensor results own their device buffer until wk_tensor_free.
 * There is NO CPU fallback: every compute entry point fails with WK_ERR_MODELS_UNAVAILABLE if no sm_100 device is present.
 */
#ifndef WKB200_H
#define WKB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int32_t wk_status;
enum {
    WK_OK = 0,
    WK_ERR_INVALID_ARGUMENT = -1,       /* (no Swift twin: argument validation)             */
    WK_ERR_MODELS_UNAVAILABLE = -2,     /* WhisperError.modelsUnavailable                    */
    WK_ERR_AUDIO_PROCESSING_FAILED = -3,/* WhisperError.audioProcessingFailed                */
    WK_ERR_PREPARE_DECODER_INPUTS = -4, /* WhisperError.prepareDecoderInputsFailed           */
    WK_ERR_DECODING_LOGITS_FAILED = -5, /* WhisperError.decodingLogitsFailed                 */
    WK_ERR_DECODING_FAILED = -6,        /* WhisperError.decodingFailed                       */
    WK_ERR_TRANSCRIPTION_FAILED = -7,   /* WhisperError.transcriptionFailed                  */
    WK_ERR_CUDA = -8                    /* CUDA runtime/driver failure (message has detail)  */
};

typedef struct wk_model wk_model;
typedef struct wk_session wk_session;
typedef struct wk_tensor wk_tensor;

enum { WK_DTYPE_F32 = 0, WK_DTYPE_F16 = 1, WK_DTYPE_BF16 = 2, WK_DTYPE_I32 = 3 };

/* Model dimensions.  The reference reads these off the CoreML model descriptions at run time
 * (TextDecoder.swift:313-331, AudioEncoder.swift:24-38, FeatureExtractor.swift:24-38). */
typedef struct wk_model_config {
    int32_t n_mels;      /* 80 or 128 */
    int32_t d_model;     /* embedSize */
    int32_t n_heads;     /* head dim must be 64 */
    int32_t enc_layers;
    int32_t dec_layers;
    int32_t vocab;       /* logitsSize */
    int32_t n_audio_ctx; /* 1500 */
    int32_t n_text_ctx;  /* 448 (positional table); kv_max_len is 224 = Constants.maxTokenContext */
    int32_t dtype;       /* WK_DTYPE_BF16 (default) or WK_DTYPE_F16: storage/MMA-input type; accumulation is f32 */
    int32_t max_batch;   /* windows processed per encoder/decoder pass (workspace sizing) */
} wk_model_config;

typedef struct wk_model_info {
    int32_t n_mels, n_audio_ctx, d_model, n_heads, enc_layers, dec_layers, vocab;
    int32_t kv_embed_dim;   /* kvCacheEmbedDim = dec_layers * d_model */
    int32_t kv_max_len;     /* kvCacheMaxSequenceLength = 224 */
    int32_t window_samples; /* 480000 */
    int32_t has_alignment_heads;
    int32_t is_multilingual; /* logitsSize != 51864 (ModelUtilities.swift:124-126) */
    int32_t dtype, max_batch;
} wk_model_info;

/* SpecialTokens (Models.swift:1111-1149) - supplied by the host tokenizer. */
typedef struct wk_special_tokens {
    int32_t end_token, english_token, no_speech_token, no_timestamps_token, special_token_begin,
        start_of_previous_token, start_of_transcript_token, time_token_begin, transcribe_token, translate_token,
        whitespace_token;
} wk_special_tokens;

/* DecodingOptions mirror (Configurations.swift:155-247), fields the hot path reads.
 * "has_*" = Swift optional is non-nil. */
typedef struct wk_decode_opts {
    int32_t task_translate;       /* task == .translate */
    int32_t language_token;       /* id of "<|xx|>" (tokenizer lookup done by the host); <0 -> english_token */
    float temperature;            /* 0 = greedy argmax; >0 = top-k multinomial (TokenSampler.swift:57-73) */
    int32_t sample_length;        /* default 224 */
    int32_t top_k;                /* default 5 */
    int32_t use_prefill_prompt;   /* default 1 */
    int32_t without_timestamps;   /* default 0 */
    int32_t suppress_blank;       /* default 0 */
    const int32_t* suppress_tokens; int32_t n_suppress_tokens;
    const int32_t* prompt_tokens;   int32_t n_prompt_tokens;   /* n < 0 -> nil */
    const int32_t* prefix_tokens;   int32_t n_prefix_tokens;   /* n < 0 -> nil */
    int32_t has_compression_ratio_threshold; float compression_ratio_threshold; /* 2.4 */
    int32_t has_logprob_threshold;           float logprob_threshold;           /* -1.0 */
    int32_t has_first_token_logprob_threshold; float first_token_logprob_threshold; /* -1.5 */
    int32_t has_no_speech_threshold;         float no_speech_threshold;         /* 0.6 */
    uint64_t seed;                /* Philox seed for temperature > 0 (the reference uses Float.random) */
    /* decodeWithFallback ladder (TranscribeTask.swift:316-411), applied by wk_transcribe_windows / wk_transcribe_streams only:
     * a window whose DecodingFallback.needsFallback is set is decoded again (same encoder output) at
     * Float16(temperature) + Float16(i) * Float16(increment), i = 1..count. */
    int32_t temperature_fallback_count;        /* default 5; 0 = no retries */
    float temperature_increment_on_fallback;   /* default 0.2 */
    int32_t word_timestamps;      /* wordTimestamps: the decode loop also fills the alignmentWeights tensor (wk_session_alignment_weights) */
    /* Beam search (SURVEY 8f row 2).  The reference's BeamSearchTokenSampler is an unimplemented stub (TokenSampler.swift:254-290) and its
     * DecodingOptions has no beam field, so these two are an extension: beam_size > 1 decodes every window with that many beams
     * (openai/whisper BeamSearchDecoder semantics inside the decodeText loop, specified by oracle/beam_ref.py; self-oracle parity only),
     * maxCandidates = Int(Float(beam_size) * beam_patience) as the stub fixes (:266).  One setting per call; the temperature ladder and
     * word timestamps do not combine with it. */
    int32_t beam_size;            /* <= 1: greedy / temperature sampling (default) */
    float beam_patience;          /* default 1 */
    /* DecodingOptions.detectLanguage (Configurations.swift:222, default !usePrefillPrompt; 0 here keeps every decode in the given language).
     * Honoured by decodeWithFallback's entry points (wk_transcribe_windows(_ex), wk_transcribe_windows_sharded, wk_transcribe_streams) for a
     * multilingual model and language_token < 0: every ladder rung first samples the window's language from the decoder's logits on
     * [SOT] (TranscribeTask.swift:339-365, TextDecoder.swift:420-539) with the session's language tokens (wk_session_set_language_tokens)
     * and the rung's temperature, then decodes with it in the prompt's language position (the token after the first SOT, if that token is
     * a language token; otherwise the detection is only reported).  A prompt that starts with SOT costs no extra decoder pass (the detection
     * rides on step 0); one that starts with <|startofprev|> costs one.  wk_decode_text(_ex) ignore it (decodeText never detects); with
     * beam_size > 1 the call fails with WK_ERR_INVALID_ARGUMENT.  Languages come back through wk_session_languages /
     * wk_transcription_language, wk_decode_result is unchanged. */
    int32_t detect_language;
} wk_decode_opts;

/* Per-window DecodingResult (Models.swift:383-439) in flat arrays; tokens = SOT..EOT slice. */
typedef struct wk_decode_result {
    int32_t n_tokens;                 /* filteredTokens.count */
    int32_t tokens[226];
    float token_logprobs[226];
    float avg_logprob;
    float compression_ratio;
    float temperature;
    int32_t needs_fallback;           /* DecodingFallback.needsFallback (0 if fallback == nil) */
    int32_t fallback_reason;          /* 0 nil, 1 firstTokenLogProbThreshold, 2 silence, 3 compressionRatio, 4 logProb */
    int32_t first_token_logprob_too_low;
    int32_t n_current_tokens;         /* currentTokens.count when the loop ended (before finalize) */
    int32_t steps;                    /* decoder forward passes run for this window */
} wk_decode_result;

const char* wk_last_error(void);
const char* wk_version(void);
/* 1 if a compute-capability 10.x device is visible. */
int32_t wk_device_available(void);

/* ---- model ---- */
void wk_default_config(const char* variant /* tiny[.en] base[.en] small[.en] medium[.en] large large-v2 large-v3 large-v3-turbo distil-large-v3 */,
                       wk_model_config* out);
/* ModelUtilities.detectVariant + tokenizerNameForVariant + isModelMultilingual (ModelUtilities.swift:124-205): static strings out. */
wk_status wk_detect_variant(int32_t logits_dim, int32_t encoder_dim, const char** variant, const char** tokenizer_repo, int32_t* is_multilingual);
wk_status wk_model_create(const wk_model_config* cfg, int32_t device, wk_model** out);
/* HuggingFace parameter names ("model.encoder.layers.0.self_attn.q_proj.weight", ...); data host or device. */
wk_status wk_model_set_tensor(wk_model* m, const char* name, const void* data, int32_t dtype, const int64_t* shape, int32_t ndim);
wk_status wk_model_finalize(wk_model* m);
/* HuggingFace checkpoint directory (config.json + *.safetensors, F32/F16/BF16); replaces loadModels (WhisperKit.swift:358-442). */
wk_status wk_model_load(const char* weights_dir, int32_t device, int32_t max_batch, int32_t dtype, wk_model** out);
/* Seeded synthetic weights generated on the device (benchmarks: no checkpoints are available offline). */
wk_status wk_model_init_random(wk_model* m, uint64_t seed, float std);
wk_status wk_model_info_get(const wk_model* m, wk_model_info* out);
void wk_model_free(wk_model* m);

/* ---- tensors (opaque device buffers passed mel -> encoder -> decoder without touching the host) ---- */
wk_status wk_tensor_shape(const wk_tensor* t, int64_t* shape4, int32_t* ndim, int32_t* dtype);
/* Copies to the host in the REFERENCE layout as f32: mel -> [B, nMels, 3000]; encoder output -> [B, d, 1500]. */
wk_status wk_tensor_to_host(const wk_tensor* t, float* dst, int64_t dst_elems);
/* Same, into a host MLMultiArray with explicit element strides (IOSurface-backed arrays pad their rows: every host access in the
 * reference goes through `strides`, TextDecoder.swift:222-227, MLMultiArrayExtensions.swift:75-82): dst[b*stride_b + c*stride_c + t*stride_t]. */
wk_status wk_tensor_to_host_strided(const wk_tensor* t, float* dst, int64_t stride_b, int64_t stride_c, int64_t stride_t, int64_t dst_elems);
/* Releases the tensor and (stream-ordered, after its last reader) its device buffer. */
void wk_tensor_free(wk_tensor* t);

/* ---- FeatureExtracting ---- */
/* pcm: n_windows rows of `stride` floats (host or device); samples_per_window[i] <= 480000 valid samples
 * (NULL = all 480000); the rest of the window is zero-padded (padOrTrimAudio, AudioProcessor.swift:151-174). */
wk_status wk_mel(wk_model* m, const float* pcm, int64_t n_windows, int64_t stride, const int32_t* samples_per_window, wk_tensor** mel_out);

/* ---- AudioEncoding ---- */
wk_status wk_encode(wk_model* m, const wk_tensor* mel, wk_tensor** enc_out);

/* ---- TextDecoding ---- */
wk_status wk_session_create(wk_model* m, int32_t max_batch, wk_session** out);
void wk_session_free(wk_session* s);
/* Bind encoder output for `batch` windows: computes the per-layer cross-attention K/V cache. */
wk_status wk_session_set_encoder_output(wk_session* s, const wk_tensor* enc);
/* Zero caches/masks (prepareDecoderInputs / DecodingInputs.reset). */
wk_status wk_session_reset(wk_session* s);
/* prefillDecoderInputs: builds initialPrompt into out (capacity cap); returns length in *n. */
wk_status wk_build_prompt(const wk_model* m, const wk_special_tokens* st, const wk_decode_opts* opts, int32_t use_options, int32_t* out, int32_t cap, int32_t* n);
/* predictLogits for every bound window: input_ids[B], cache_length[B] (host) -> logits [B, vocab] f32 (host, may be NULL). */
wk_status wk_decode_step(wk_session* s, const int32_t* input_ids, const int32_t* cache_length, float* logits_out);
/* TextDecoding.detectLanguage (TextDecoder.swift:420-539): one step on [SOT] + LanguageLogitsFilter + sampler, per bound window. */
wk_status wk_detect_language(wk_session* s, const wk_special_tokens* st, const int32_t* language_tokens, int32_t n_language_tokens,
                             float temperature, int32_t* token_out, float* logprob_out);
/* Filters + sampler alone (parity entry): logits [B, vocab] f32 host; tokens [B, ld_tokens], n_tokens[B] = currentTokens;
 * sample_begin_ts = TimestampRulesFilter.sampleBegin (<0: filter absent), sample_begin_blank = SuppressBlankFilter.sampleBegin
 * (<0: absent); language_tokens != NULL adds LanguageLogitsFilter(sampleBegin = language_sample_begin).
 * Writes token_out[B], logprob_out[B] and (optional) the masked logits back into filtered_out [B, vocab]. */
wk_status wk_filter_sample(wk_model* m, const wk_special_tokens* st, const wk_decode_opts* opts, int32_t is_multilingual,
                           const float* logits, int32_t batch, int32_t vocab, const int32_t* tokens, int32_t ld_tokens,
                           const int32_t* n_tokens, int32_t sample_begin_ts, int32_t sample_begin_blank,
                           const int32_t* language_tokens, int32_t n_language_tokens, int32_t language_sample_begin,
                           int32_t* token_out, float* logprob_out, float* filtered_out);
/* decodeText for every bound window with one shared prompt (device-resident loop: no per-token host round trip).
 * results: array of `batch` wk_decode_result. */
wk_status wk_decode_text(wk_session* s, const wk_special_tokens* st, const wk_decode_opts* opts,
                         const int32_t* prompt, int32_t n_prompt, wk_decode_result* results);
/* Scheduler counters of the session's last batched call: [0] decode steps launched, [1] sum over those steps of the windows that were
 * live when their burst started (an upper bound of the rows that actually streamed K/V), [2] windows admitted to a slot, [3] ladder
 * re-admissions. */
wk_status wk_session_stats(const wk_session* s, int64_t* out4);
/* allLanguageTokens of this session (WhisperTokenizerWrapper.allLanguageTokens, Models.swift:1219): the ids detectLanguage chooses from,
 * and the ids recognised as a language in a decoded window.  n <= 4096, every id inside the vocabulary; n = 0 restores the default: the
 * ids strictly between start_of_transcript_token and min(translate_token, transcribe_token) of the call's special tokens (the language
 * block of every Whisper vocabulary: 99 ids, 100 in large-v3).  Per session, so setting it races no other thread. */
wk_status wk_session_set_language_tokens(wk_session* s, const int32_t* tokens, int32_t n);
/* The language of the first n windows of the session's last wk_transcribe_windows(_ex) call, as the reference's
 * `detectedLanguage ?? defaultLanguageCode` (TranscribeTask.swift:341-376): the detected token of the ladder rung whose result was kept
 * (logprob = the detection step's log-probability, DecodingResult.languageProbs); else the explicit language_token (logprob 0); else the
 * first language token of the result's tokens (TextDecoder.swift:804-822; logprob = its token_logprobs entry); else english_token (0).
 * logprobs may be NULL.  After wk_transcribe_windows_sharded every rank holds the languages of its own shard: they are not gathered. */
wk_status wk_session_languages(const wk_session* s, int64_t n, int32_t* tokens, float* logprobs);
/* Device logits of the last step, copied to host (debug / parity). */
wk_status wk_session_last_logits(wk_session* s, float* logits_out);

/* TranscriptionCallback (Models.swift TranscriptionProgress; TextDecoder.swift:724-762): called from the thread that runs the decode
 * every `progress_every` decoder steps with each live window's current tokens.  Returning 0 is the reference's `callback -> false`:
 * that window stops early (EarlyStopActor) and its result is built from the tokens it has. */
typedef int32_t (*wk_progress_fn)(void* user, int32_t window, const int32_t* tokens, int32_t n_tokens, float avg_logprob);

/* Per-item arguments of the batched entry points (transcribeWithOptions' decodeOptionsArray, WhisperKit.swift:716-735). */
typedef struct wk_batch_opts {
    const wk_decode_opts* opts;         /* n_opts == 1: shared by every window; else one per window */
    int32_t n_opts;
    const int32_t* const* prompts;      /* per-window initial prompts (prefillDecoderInputs output); NULL = one shared `prompt` */
    const int32_t* prompt_lens;
    const int32_t* prompt; int32_t n_prompt;   /* shared prompt when prompts == NULL; NULL too = built per window with wk_build_prompt */
    wk_progress_fn progress; void* progress_user;
    int32_t progress_every;             /* decoder steps between callbacks / completion polls; <= 0 = 16 */
    wk_status* status;                  /* per-window Result<> (WhisperKit.swift:775-790): WK_OK or that window's error; may be NULL */
    int32_t encoder_chunk;              /* windows per mel+encoder pass; <= 0 = the model's max_batch */
} wk_batch_opts;

/* ---- whole hot path: host PCM in, token IDs out (TranscribeTask.run body, batched) ----
 * Windows are independent units.  The session's max_batch decode slots run as one device-resident loop; a window that ends (EOT,
 * sampleLength, first-token threshold, early stop) retires from every kernel of the step at once and its slot is handed to the next
 * encoded window, while the mel + encoder pass of the following chunk runs on a second stream (tensor-bound encoder under the
 * HBM-bound decode).  The temperature ladder re-admits a window that asks for a fallback into its own slot (cross K/V kept). */
wk_status wk_transcribe_windows(wk_model* m, wk_session* s, const float* pcm_host /* host (pageable/pinned) or device */, int64_t n_windows, int64_t stride,
                                const int32_t* samples_per_window, const wk_special_tokens* st, const wk_decode_opts* opts,
                                const int32_t* prompt, int32_t n_prompt, wk_decode_result* results);
/* decodeText on the bound windows with per-window options / prompts / status and the progress callback (no temperature ladder, like
 * TextDecoding.decodeText itself). */
wk_status wk_decode_text_ex(wk_session* s, const wk_special_tokens* st, const wk_batch_opts* bo, wk_decode_result* results);
/* Same with per-window options / prompts / status and a progress callback.  Returns WK_OK when the call itself ran; per-window
 * failures are reported through bo->status (and fail the call only when status is NULL). */
wk_status wk_transcribe_windows_ex(wk_model* m, wk_session* s, const float* pcm_host, int64_t n_windows, int64_t stride,
                                   const int32_t* samples_per_window, const wk_special_tokens* st, const wk_batch_opts* bo,
                                   wk_decode_result* results);

/* ---- multi-GPU edges (SURVEY section 8e): one process per GPU, windows sharded, weights replicated; NCCL only moves PCM out and
 * results back (grouped ncclSend / ncclRecv over NVLink).  NCCL is resolved at run time from the process; wk_comm_unique_id fails with
 * WK_ERR_MODELS_UNAVAILABLE if it is not there.  The 128-byte id from rank 0 reaches the other ranks by whatever the host uses for
 * rendezvous (torch.distributed in bench.py, MPI, a file). */
typedef struct wk_comm wk_comm;
void wk_comm_shard_bounds(int64_t n_windows, int32_t world, int32_t rank, int64_t* lo, int64_t* hi);   /* contiguous, order preserving */
wk_status wk_comm_unique_id(uint8_t* out128);
wk_status wk_comm_create(const uint8_t* id128, int32_t rank, int32_t world, int32_t device, wk_comm** out);
void wk_comm_free(wk_comm* c);
/* root holds all_pcm [n_windows][stride] (host or device); every rank receives its shard into shard_dev (device). */
wk_status wk_comm_scatter_windows(wk_comm* c, const float* all_pcm, int64_t n_windows, int64_t stride, int32_t root, float* shard_dev, int64_t* n_local);
/* every rank hands in the results of its shard; root receives all n_windows in window order. */
wk_status wk_comm_gather_results(wk_comm* c, const wk_decode_result* local, int64_t n_local, int64_t n_windows, int32_t root, wk_decode_result* all);
/* scatter -> wk_transcribe_windows_ex on the shard -> gather; bo must carry shared options (n_opts == 1, no per-window arrays). */
wk_status wk_transcribe_windows_sharded(wk_comm* c, wk_model* m, wk_session* s, const float* all_pcm, int64_t n_windows, int64_t stride, int32_t root,
                                        const wk_special_tokens* st, const wk_batch_opts* bo, wk_decode_result* results);
/* host wall-clock milliseconds of the last sharded call on this rank: [0] scatter [1] transcribe [2] gather [3] total */
wk_status wk_comm_last_stage_ms(const wk_comm* c, float* ms4);

/* ---- long-form windowing (SURVEY section 8f rows 1 and 3): host logic, callable without a GPU ---- */
typedef struct wk_tokenizer_hooks wk_tokenizer_hooks;   /* defined with the word-timestamp API below */
typedef struct wk_word wk_word;
typedef struct wk_segment {             /* TranscriptionSegment (Models.swift), token-level fields */
    int32_t stream, id;
    int64_t seek;                       /* window start sample inside the stream */
    float start, end;                   /* seconds from the start of the stream */
    int64_t token_offset; int32_t n_tokens; /* slice of the flat token / logprob arrays */
    float temperature, avg_logprob, compression_ratio, no_speech_prob;
} wk_segment;
/* SegmentSeeking.findSeekPointAndSegments (Sources/WhisperKit/Core/Text/SegmentSeeker.swift:41-189).
 * *n_segs = -1 means the Swift function returned nil segments (window skipped as silent). token_offset is relative to `tokens`. */
wk_status wk_find_seek_point_and_segments(const int32_t* tokens, const float* token_logprobs, int32_t n_tokens, float no_speech_prob,
                                          float avg_logprob, float compression_ratio, float temperature, const wk_decode_opts* opts,
                                          int32_t all_segments_count, int64_t current_seek, int64_t segment_size, int32_t sample_rate,
                                          int32_t time_token, int64_t* new_seek, wk_segment* segs, int32_t cap, int32_t* n_segs);
/* DecodingOptions.prepareSeekClips (Sources/WhisperKit/Utilities/Extensions+Internal.swift:111-130); clips = [start0,end0,start1,...] */
wk_status wk_prepare_seek_clips(const float* clip_timestamps, int32_t n, int64_t content_frames, int64_t* clips, int32_t cap, int32_t* n_clips);
/* EnergyVAD.voiceActivity (EnergyVAD.swift:41-56, AudioProcessor.swift:674-702): RMS per frame > threshold */
wk_status wk_vad_voice_activity(const float* wav, int64_t n, int32_t frame_len, int32_t frame_overlap, float threshold, uint8_t* out,
                                int64_t cap, int64_t* n_frames);
/* VoiceActivityDetector.findLongestSilence (VoiceActivityDetector.swift:95-125); start = end = -1 when there is none */
wk_status wk_vad_find_longest_silence(const uint8_t* vad, int64_t n, int64_t* start, int64_t* end);
/* VoiceActivityDetector.calculateActiveChunks (:52-80); chunks = [start0,end0,...] */
wk_status wk_vad_active_chunks(const float* wav, int64_t n, int32_t frame_len, int32_t frame_overlap, float threshold, int64_t* chunks,
                               int32_t cap, int32_t* n_chunks);
/* VADAudioChunker.chunkAll (Sources/WhisperKit/Core/Audio/AudioChunker.swift:53-107); chunks = [seekOffsetIndex0,end0,...] */
wk_status wk_vad_chunk_all(const float* wav, int64_t n, int64_t max_chunk_len, const float* clip_timestamps, int32_t n_clip_timestamps,
                           int64_t window_padding, int32_t frame_len, int32_t frame_overlap, float threshold, int64_t* chunks, int32_t cap,
                           int32_t* n_chunks);
/* TranscribeTask.run's seek loop (TranscribeTask.swift:98-279) for MANY audio streams at once: every round the next <= 30 s
 * window of each unfinished stream is batched through the GPU path, then each stream's seek advances by its own decoded
 * timestamps.  chunking_vad != 0 first splits every stream with VADAudioChunker (WhisperKit.swift:878-911) so chunks become
 * independent units.  With opts->word_timestamps (and `hooks`, the host tokenizer) every window also runs addWordTimestamps
 * (TranscribeTask.swift:197-239): segment bounds follow the word timings, zero-length segments are dropped and the last word end
 * can pull the seek forward.  hooks may be NULL otherwise. */
typedef struct wk_transcription wk_transcription;
wk_status wk_transcribe_streams(wk_model* m, wk_session* s, const float* const* audio, const int64_t* n_samples, int32_t n_streams,
                                const wk_special_tokens* st, const wk_decode_opts* opts, const int32_t* prompt, int32_t n_prompt,
                                const float* clip_timestamps, int32_t n_clip_timestamps, float window_clip_time, int64_t max_window_seek,
                                int32_t chunking_vad, const wk_tokenizer_hooks* hooks, wk_transcription** out);
int32_t wk_transcription_segment_count(const wk_transcription* t);
int32_t wk_transcription_window_count(const wk_transcription* t);
int64_t wk_transcription_token_count(const wk_transcription* t);
wk_status wk_transcription_segments(const wk_transcription* t, wk_segment* segs, int32_t cap);
wk_status wk_transcription_tokens(const wk_transcription* t, int32_t* tokens, float* logprobs, int64_t cap);
int32_t wk_transcription_word_count(const wk_transcription* t);
wk_status wk_transcription_word(const wk_transcription* t, int32_t i, wk_word* out);   /* .segment indexes wk_transcription_segments */
/* TranscriptionResult.language of one stream (token, and the log-probability wk_session_languages gives for that window): with detection
 * on, the last window's detection (detectedLanguage is reassigned every window, TranscribeTask.swift:352); with it off, the first window's
 * language (:376).  A VAD-chunked stream takes its first chunk's (TranscriptionUtilities.swift:103); a stream with no window, english_token. */
wk_status wk_transcription_language(const wk_transcription* t, int32_t stream, int32_t* token, float* logprob);
void wk_transcription_free(wk_transcription* t);

/* ---- word timestamps (SURVEY section 8f row 1) ----
 * Device side: with wk_decode_opts.word_timestamps set, every decode step also writes the mean cross-attention softmax row of the
 * model's alignment heads into row tokenIndex + 1 of a [224][1500] Float16 tensor per window - the decoder model's
 * `alignment_heads_weights` output spliced by TextDecoder.updateAlignmentWeights (TextDecoder.swift:272-296,310,414,709-717).
 * Host side (C++, callable without a GPU): SegmentSeeker's DTW / alignment / punctuation / duration logic
 * (SegmentSeeker.swift:195-659).  The tokenizer stays with the host and is reached through wk_tokenizer_hooks. */
/* (layer, head) pairs, e.g. openai-whisper's per-checkpoint alignment heads; n_pairs = 0 restores the default
 * (all heads of the last half of the decoder layers). */
wk_status wk_model_set_alignment_heads(wk_model* m, const int32_t* layer_head_pairs, int32_t n_pairs);
/* DecodingResult.cache.alignmentWeights of one window of the last wk_decode_text, first `rows` rows, as f32 [rows][n_audio_ctx]. */
wk_status wk_session_alignment_weights(wk_session* s, int32_t window, int32_t rows, float* out);
/* The same rows as stored, Float16 (FloatType): an asynchronous device-to-host copy on the session stream into out (pinned memory for it
 * to be truly asynchronous); sync != 0 waits for it and for every copy queued before it. */
wk_status wk_session_alignment_weights_f16(wk_session* s, int32_t window, int32_t rows, uint16_t* out, int32_t sync);

struct wk_word {                   /* WordTiming (Models.swift:617-633) */
    const char* word;              /* UTF-8, NUL-terminated */
    const int32_t* tokens; int32_t n_tokens;
    float start, end, probability;
    int32_t segment;               /* set by the segment update: index of the segment that owns the word, else -1 */
};
typedef struct wk_words wk_words;  /* owning word list returned by the functions below */
int32_t wk_words_count(const wk_words* w);
wk_status wk_words_get(const wk_words* w, int32_t i, wk_word* out);   /* pointers stay valid until wk_words_free */
void wk_words_free(wk_words* w);

struct wk_tokenizer_hooks {
    /* WhisperTokenizer.splitToWordTokens (Models.swift:1291-1306): write the words as consecutive NUL-terminated UTF-8 strings into
     * `text` and each word's token count into `counts`; return the number of words, or < 0 on error / overflow. */
    int32_t (*split_to_word_tokens)(void* user, const int32_t* tokens, int32_t n_tokens, char* text, int32_t text_cap, int32_t* counts, int32_t counts_cap);
    /* WhisperTokenizer.decode(tokens:): NUL-terminated UTF-8 into `text`; return bytes written (without NUL) or < 0. May be NULL. */
    int32_t (*decode)(void* user, const int32_t* tokens, int32_t n_tokens, char* text, int32_t text_cap);
    void* user;
};

/* SegmentSeeker.dynamicTimeWarping (SegmentSeeker.swift:195-276); matrix row-major [rows][ld], dtype WK_DTYPE_F32 or WK_DTYPE_F16.
 * The path has at most rows + cols entries. */
wk_status wk_dtw(const void* matrix, int32_t dtype, int32_t rows, int32_t cols, int64_t ld, int32_t* text_indices, int32_t* time_indices,
                 int32_t cap, int32_t* n_path);
/* findAlignment (:340-408); `words` carry word + tokens (the host's splitToWordTokens), timings are ignored. */
wk_status wk_find_alignment(const wk_word* words, int32_t n_words, const void* matrix, int32_t dtype, int32_t rows, int32_t cols, int64_t ld,
                            const float* token_logprobs, int32_t n_logprobs, wk_words** out);
/* mergePunctuations (:278-338); NULL prepended/appended = Constants.default{Prepend,Append}Punctuations (Models.swift:1459-1460). */
wk_status wk_merge_punctuations(const wk_word* alignment, int32_t n, const char* prepended, const char* appended, wk_words** out);
/* calculateWordDurationConstraints (:498-508) and truncateLongWordsAtSentenceBoundaries (:510-526). */
wk_status wk_word_duration_constraints(const wk_word* alignment, int32_t n, float* constrained_median, float* max_duration);
wk_status wk_truncate_long_words(const wk_word* alignment, int32_t n, float max_duration, wk_words** out);
/* updateSegmentsWithWordTimings (:528-659): segs[i].start/end are updated in place; segment tokens are
 * tokens[segs[i].token_offset .. + n_tokens); out = every word with .segment set. */
wk_status wk_update_segments_with_word_timings(wk_segment* segs, int32_t n_segs, const int32_t* tokens, const wk_word* merged, int32_t n_merged,
                                               int64_t seek, float last_speech_timestamp, float constrained_median, float max_duration,
                                               int32_t special_token_begin, const wk_tokenizer_hooks* hooks, wk_words** out);
/* addWordTimestamps (:410-496), the whole per-window word-timing pass; alignment = [rows][ld] with row i = window token i. */
wk_status wk_add_word_timestamps(wk_segment* segs, int32_t n_segs, const int32_t* tokens, const float* token_logprobs,
                                 const void* alignment, int32_t dtype, int32_t rows, int32_t cols, int64_t ld,
                                 const wk_tokenizer_hooks* hooks, int64_t seek, float last_speech_timestamp, int32_t special_token_begin,
                                 const char* prepended, const char* appended, wk_words** out);

/* ---- tokenizer, decode side (SURVEY section 8f row 4): ids -> text without a Swift host ----
 * Byte-level BPE decode as swift-transformers does it (Tokenizer.swift:510-530, Decoder.swift:126-170): added tokens verbatim, the rest
 * through the GPT-2 byte alphabet into lossy UTF-8, then cleanUp; WhisperTokenizerWrapper's special-token lookups and word splitting
 * (Models.swift:1201-1306).  wk_tokenizer_encode is text -> ids WITHOUT the post-processor (no <|startoftranscript|> ... template): the
 * reference filters special tokens out of encoded prompts anyway (TranscribeCLIUtils / promptTokens). */
typedef struct wk_tokenizer wk_tokenizer;
/* path: a checkpoint directory (tokenizer.json, else vocab.json + added_tokens.json), or one of those files. */
wk_status wk_tokenizer_load(const char* path, wk_tokenizer** out);
/* From memory: flags bit 0 = added token (emitted verbatim), bit 1 = special (dropped by skip_special_tokens). */
wk_status wk_tokenizer_create(const char* const* tokens, const int32_t* ids, const uint8_t* flags, int32_t n, int32_t clean_up_tokenization_spaces,
                              wk_tokenizer** out);
void wk_tokenizer_free(wk_tokenizer* t);
int32_t wk_tokenizer_vocab_size(const wk_tokenizer* t);
int32_t wk_tokenizer_token_to_id(const wk_tokenizer* t, const char* token);   /* convertTokenToId; -1 = nil */
/* decode(tokens:skipSpecialTokens:): NUL-terminated UTF-8 into text; returns bytes written (without NUL), or -(bytes needed) if cap is short. */
int32_t wk_tokenizer_decode(const wk_tokenizer* t, const int32_t* tokens, int32_t n, int32_t skip_special_tokens, char* text, int32_t cap);
/* encode(text:) minus the post-processor: added tokens verbatim, then the GPT-2 pre-tokenizer pattern, byte alphabet and BPE merges
 * (merges come from tokenizer.json / merges.txt, or wk_tokenizer_set_merges).  Returns the id count, or -(ids needed) if cap is short. */
int32_t wk_tokenizer_encode(const wk_tokenizer* t, const char* text_utf8, int32_t* ids, int32_t cap);
wk_status wk_tokenizer_set_merges(wk_tokenizer* t, const char* const* left, const char* const* right, int32_t n);
/* SpecialTokens as WhisperTokenizerWrapper.init derives them, with its defaults for absent tokens. */
wk_status wk_tokenizer_special_tokens(const wk_tokenizer* t, wk_special_tokens* out);
/* splitToWordTokens in the wk_tokenizer_hooks layout (words as consecutive NUL-terminated strings, one token count per word; a NUL
 * byte inside a decoded word is dropped). */
int32_t wk_tokenizer_split_to_word_tokens(const wk_tokenizer* t, const int32_t* tokens, int32_t n, char* text, int32_t text_cap, int32_t* counts,
                                          int32_t counts_cap);
/* WhisperTokenizerWrapper.allLanguageTokens (Models.swift:1219), from the vocabulary: the ids of the added tokens whose content is "<|" + 2
 * or 3 lowercase ASCII letters + "|>", ascending.  Returns the count, or -(count needed) if cap is short. */
int32_t wk_tokenizer_language_tokens(const wk_tokenizer* t, int32_t* out, int32_t cap);
/* Fills `hooks` with this tokenizer's split / decode so wk_transcribe_streams and wk_add_word_timestamps run without host callbacks. */
wk_status wk_tokenizer_hooks_init(wk_tokenizer* t, wk_tokenizer_hooks* hooks);

/* ---- result writers (SURVEY section 8f row 4; Sources/WhisperKit/Utilities/ResultWriter.swift) ----
 * Cues are flat: one per word where the segment has word timings, else one per segment (the order WriteSRT / WriteVTT iterate).
 * Each function writes NUL-terminated UTF-8 into out and returns the byte count (without NUL), or -(bytes needed) if cap is short. */
int32_t wk_format_time(float seconds, int32_t always_include_hours, const char* decimal_marker, char* out, int32_t cap);   /* ResultWriting.formatTime, :14-26 */
int32_t wk_write_srt(const float* starts, const float* ends, const char* const* texts, int32_t n, char* out, int32_t cap);   /* WriteSRT, :70-101 */
int32_t wk_write_vtt(const float* starts, const float* ends, const char* const* texts, int32_t n, char* out, int32_t cap);   /* WriteVTT, :103-134 */

/* ---- instrumentation ---- */
/* Number of kernels launched by this library on the calling process since the last reset. */
int64_t wk_kernel_launch_count(int32_t reset);
/* Last-run stage timings in ms, TranscriptionTimings buckets (Models.swift:730-776):
 * [0] logmels [1] encoding [2] crossKV [3] decodingLoop [4] h2d [5] d2h */
wk_status wk_last_timings(wk_model* m, float* ms6);
/* Stream all work is enqueued on (cudaStream_t as void*), for CUDA-event timing by the host harness. */
void* wk_model_stream(wk_model* m);

/* ---- kernel-level test/bench hooks (used by tests/ and bench.py; device pointers) ---- */
/* C[M,N] = A[M,K] * W[N,K]^T (+bias) with the tcgen05 GEMM; out_dtype WK_DTYPE_BF16/F16/F32. */
wk_status wk_test_gemm(wk_model* m, const void* a, const void* w, const float* bias, void* out, int32_t M, int32_t N, int32_t K,
                       int32_t in_dtype, int32_t out_dtype, int32_t gelu);
/* out[M,N] (f32, in place) += A[M,K] * W[N,K]^T + bias: the residual-update epilogue of the encoder's out-proj / FC2. */
wk_status wk_test_gemm_residual(wk_model* m, const void* a, const void* w, const float* bias, float* out, int32_t M, int32_t N, int32_t K, int32_t in_dtype);
/* Same product through the decoder's swap-AB split-K path: out f32 [rows_x, N]. */
wk_status wk_test_gemm_splitk(wk_model* m, const void* w, const void* x, float* out, int32_t N, int32_t rows_x, int32_t K, int32_t in_dtype, int32_t splits);
/* Encoder attention on packed qkv [B*T, 3*d] -> out [B*T, d]. */
wk_status wk_test_attention(wk_model* m, const void* qkv, void* out, int32_t B, int32_t T, int32_t n_heads, int32_t dtype);
/* Decoder cross-attention kernel alone: q [B][H*64] f32, K/V [B][H][T][64] 16-bit -> out [B][H*64] 16-bit; done (device, may be NULL)
 * marks rows to skip. */
wk_status wk_test_cross_attention(wk_model* m, const float* q, const void* kcross, const void* vcross, void* out, int32_t B, int32_t H,
                                  int32_t T, int32_t dtype, const int32_t* done);
/* The beam-search form of the same kernel: groups of kv_div adjacent rows share one K/V block, K/V [B / kv_div][H][T][64]. */
wk_status wk_test_cross_attention_shared(wk_model* m, const float* q, const void* kcross, const void* vcross, void* out, int32_t B, int32_t H,
                                         int32_t T, int32_t dtype, const int32_t* done, int32_t kv_div);
/* Decoder self-attention kernel alone: qkv [B][3*H*64] f32 of the new token, caches [B][H][224][64] 16-bit (positions < pos[b] valid;
 * row pos[b] is appended), pos [B] device -> out [B][H*64] 16-bit. */
wk_status wk_test_self_attention(wk_model* m, const float* qkv, void* kcache, void* vcache, const int32_t* pos, void* out, int32_t B,
                                 int32_t H, int32_t dtype, const int32_t* done);

/* Average device time (ms) of one launch of a named hot kernel on the live buffers, plus its algorithmic work
 * (bytes for HBM-bound kernels, FLOPs for tensor-bound ones): 0 decoder cross-attention, 1 encoder FC1 GEMM,
 * 2 log-mel, 3 encoder attention, 4 decoder QKV swap-AB GEMM, 5 encoder QKV GEMM.  Used by bench.py's roofline. */
wk_status wk_bench_kernel(wk_model* m, wk_session* s, int32_t which, int32_t batch, int32_t iters, float* ms_out, double* work_out);

/* Debug readback of an internal device buffer converted to f32 (stage-by-stage parity debugging; see engine.cu). */
wk_status wk_debug_read(wk_model* m, wk_session* s, int32_t which, int64_t offset_elems, float* dst, int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* WKB200_H */
