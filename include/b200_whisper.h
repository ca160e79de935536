/*
 * b200_whisper.h -- C ABI of the B200-native Whisper backend (libb200whisper.so).
 *
 * This is the drop-in boundary for the hot path of brightleeh/whisper-streaming-stt-server:
 * everything `ModelBackend.transcribe` (reference stt_server/model/backends/base.py:24-35)
 * delegates to third-party arithmetic -- upstream `whisper.transcribe` called from
 * stt_server/model/backends/torch_whisper.py:55 and `WhisperModel.transcribe` called from
 * stt_server/model/backends/faster_whisper.py:35 -- is reached through these entry points.
 * The Python host (`whisper-streaming-stt-server_b200/backend.py`) binds them with ctypes;
 * INTEGRATION.md shows the stub.  Plain pointers and sizes only; no torch types.
 *
 * Conventions: every function returns 0 on success or a negative bw_status; on failure
 * bw_last_error() returns a thread-local message.  All entry points are thread-safe; the
 * blocking calls (`bw_call_decode`, `bw_call_detect_language`) may be issued from many host
 * threads at once -- the engine coalesces them into batched launches (the reference calls
 * `transcribe` from `pool_size` threads concurrently, model_registry.py:564-606).
 */
#ifndef B200_WHISPER_H
#define B200_WHISPER_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bw_engine bw_engine;
typedef struct bw_call bw_call;

enum bw_status {
  BW_OK = 0,
  BW_ERR_INVALID = -1,   /* bad argument / unknown tensor name / shape mismatch */
  BW_ERR_CUDA = -2,      /* CUDA runtime or driver error (message has the call) */
  BW_ERR_STATE = -3,     /* call made in the wrong engine state */
  BW_ERR_NOMEM = -4,     /* device pool exhausted */
  BW_ERR_NO_DEVICE = -5  /* no usable sm_100 device */
};

enum bw_compute {
  BW_COMPUTE_BF16 = 0,  /* product mode: bf16 weights/activations, fp32 accumulate, tcgen05 GEMMs */
  BW_COMPUTE_FP32 = 1   /* validation mode: fp32 storage + fp32 accumulate (SIMT), for token-id parity */
};

enum bw_dtype { BW_F32 = 0, BW_F16 = 1, BW_BF16 = 2 };

/* Mirrors upstream ModelDimensions (what `whisper.load_model` yields; torch_whisper.py:21). */
typedef struct bw_model_dims {
  int32_t n_mels, n_audio_ctx, n_audio_state, n_audio_head, n_audio_layer;
  int32_t n_vocab, n_text_ctx, n_text_state, n_text_head, n_text_layer;
} bw_model_dims;

typedef struct bw_engine_config {
  int32_t cuda_device;       /* ordinal */
  int32_t compute;           /* bw_compute */
  int32_t max_segments;      /* concurrent decode windows resident on the GPU (cross-KV slots); 0 = auto */
  int32_t max_sequences;     /* concurrent hypotheses (beams) resident (state slots); 0 = auto */
  int32_t max_encoder_batch; /* windows per encoder launch; 0 = auto */
  int32_t flags;             /* BW_FLAG_* */
  /* self-attention KV pool, in pages of 16 positions of one hypothesis (all layers, k and v); 0 = auto
   * (16 pages per hypothesis slot).  Pages are handed out as hypotheses grow and shared by beams over their common
   * prefix, so the pool follows the tokens in use; a window is admitted once its worst case is reservable. */
  int32_t max_kv_pages;
} bw_engine_config;

#define BW_FLAG_FORCE_SIMT_GEMM 1  /* debugging: use the SIMT GEMM/attention even in bf16 mode */
#define BW_FLAG_NO_SCHEDULER 2     /* stage-level use only (bw_mel / bw_encode / kernel tests) */
/* bf16 compute only: keep the cached encoder K/V (cross-attention) in 8 bits -- one fp32 scale per (layer, k|v, position,
 * head) -- for 0.53x the bytes per window and per decoder step.  Not bit-compatible with the bf16 cache: logits move
 * by the quantisation error.  Refused (BW_ERR_INVALID) with BW_COMPUTE_FP32 or BW_FLAG_FORCE_SIMT_GEMM. */
#define BW_FLAG_CROSS_KV_INT8 4
#define BW_FLAG_SIMT_ATTENTION 8   /* debugging: SIMT encoder self-attention in bf16 mode */

/* One tensor of the openai-whisper state dict (name = state_dict key). Host pointer. */
typedef struct bw_tensor_desc {
  const char* name;
  const void* data;
  int32_t dtype;     /* bw_dtype */
  int32_t ndim;
  int64_t shape[4];
} bw_tensor_desc;

/* Token-id tables (upstream tokenizer.py layout; the host derives them per vocabulary). */
typedef struct bw_token_tables {
  int32_t eot, sot, sot_prev, sot_lm, no_speech, no_timestamps, timestamp_begin;
  int32_t translate, transcribe;
  int32_t first_language_token, num_languages;
  const int32_t* suppress;  int32_t n_suppress;   /* SuppressTokens list (already includes specials) */
  const int32_t* blank;     int32_t n_blank;      /* SuppressBlank list: encode(" ") + eot */
} bw_token_tables;

/* Per-window decoding options == upstream DecodingOptions as reachable through
 * torch_whisper.py:78-110.  beam_size 0 selects GreedyDecoder semantics. */
typedef struct bw_decode_opts {
  const int32_t* initial_tokens;  /* [sot_prev + prompt +] sot sequence, built by the host */
  int32_t n_initial;
  int32_t sot_index;              /* position of <|sot|> inside initial_tokens */
  int32_t beam_size;              /* 0 = greedy, else BeamSearchDecoder(beam_size) */
  float patience;                 /* <= 0 -> 1.0 */
  float length_penalty;           /* < 0 -> None (length normalisation) */
  int32_t sample_len;             /* 0 -> n_text_ctx / 2 */
  int32_t without_timestamps;     /* 1 disables ApplyTimestampRules */
  int32_t suppress_blank;         /* upstream default 1 */
  int32_t max_initial_timestamp_index; /* < 0 -> None; upstream default 50 */
  /* GreedyDecoder at temperature > 0 (one rung of transcribe.py's decode_with_fallback ladder): next token ~
   * Categorical(logits / temperature), drawn by Gumbel-max with a counter-based generator keyed by
   * (seed, hypothesis, position, token id) -- reproducible for a given seed whatever the batch it runs in.
   * Needs beam_size == 0.  best_of = hypotheses sampled per window (0 -> 1); the best by the length-penalised
   * sum of log-probabilities (MaximumLikelihoodRanker) is returned. */
  float temperature;              /* 0 -> arg-max (fields below ignored) */
  int32_t best_of;
  uint32_t seed_lo, seed_hi;
  /* BeamSearchDecoder.max_candidates = round(beam_size * patience) as the HOST rounds it (Python: half to even);
   * 0 -> computed here with nearbyint (same rule under the default rounding mode). */
  int32_t max_candidates;
} bw_decode_opts;

#define BW_MAX_TOKENS 448

typedef struct bw_result {
  int32_t n_tokens;
  int32_t tokens[BW_MAX_TOKENS];  /* sampled part of the selected hypothesis, cut at the first EOT */
  float sum_logprob;
  float avg_logprob;
  float no_speech_prob;
  int32_t n_steps;                /* decoder steps this window took */
  /* timing diagnostics, seconds */
  float t_queue, t_encode, t_decode;
} bw_result;

typedef struct bw_lang_result {
  int32_t language_token;
  int32_t n_languages;
  float probs[128];               /* softmax over the language tokens, index = language order */
} bw_lang_result;

/* ---- engine life cycle ---- */
const char* bw_last_error(void);
int bw_version(void);
int bw_device_count(void);
int bw_engine_create(const bw_model_dims* dims, const bw_engine_config* cfg, bw_engine** out);
int bw_engine_load_weights(bw_engine*, const bw_tensor_desc* tensors, int32_t n);
int bw_engine_set_tables(bw_engine*, const bw_token_tables* tables);
int bw_engine_set_mel_filters(bw_engine*, const float* filters /* [n_mels, 201] */);
int bw_engine_finalize(bw_engine*);  /* packs weights, sizes the KV pools, starts the scheduler */
int bw_engine_destroy(bw_engine*);   /* drops one reference; the engine goes away with the last one */
/* refcount: one weight copy per (GPU, model, dtype) shared by pool handles.  Every open bw_call holds a reference
 * too, so destroying the engine while calls are open only defers the teardown to the last bw_call_close. */
int bw_engine_retain(bw_engine*);
int bw_engine_stats(bw_engine*, int64_t* out, int32_t n); /* see BW_STAT_* */

enum {
  BW_STAT_KERNEL_LAUNCHES = 0, BW_STAT_DECODE_STEPS, BW_STAT_ROWS, BW_STAT_WINDOWS,
  BW_STAT_MAX_SEGMENTS, BW_STAT_MAX_SEQUENCES, BW_STAT_ENCODER_BATCHES, BW_STAT_H2D_BYTES,
  BW_STAT_D2H_BYTES, BW_STAT_KV_PAGES_TOTAL, BW_STAT_KV_PAGES_IN_USE, BW_STAT_KV_PAGES_PEAK, BW_STAT_KV_PAGE_BYTES,
  BW_STAT_COUNT
};

/* ---- the hot call, split so the host keeps upstream's seek loop (transcribe.py) ---- */
/* Copies the PCM (host f32, 16 kHz, what ModelWorker._decode hands to transcribe, worker.py:119-125)
 * and computes the whole-call log-mel (global-max normalisation, padding = 30 s) on the device. */
int bw_call_open(bw_engine*, const float* pcm, int64_t n_samples, bw_call** out);

/* Raw ingest (SURVEY 8(f).2): the bytes the server receives -- PCM16 mono at `sample_rate` -- go to the device as
 * they are (half the H2D bytes of the f32 path) and `pcm16_to_float32` + `ensure_16k` run there
 * (stt_server/utils/audio.py:6-8 int16 -> float32 / 32768; :11-30 torchaudio sinc_interp_hann resampling to 16 kHz,
 * lowpass_filter_width 6, rolloff 0.99), feeding the log-mel kernel directly.
 * bw_engine_set_resampler registers the polyphase filter bank for one source rate: taps[new_freq][2*width+orig_freq]
 * fp32 exactly as torchaudio's `_get_sinc_resample_kernel` builds it (orig/new reduced by their gcd); 16 kHz needs none. */
int bw_engine_set_resampler(bw_engine*, int32_t sample_rate, int32_t orig_freq, int32_t new_freq, int32_t width, const float* taps);
int bw_call_open_pcm16(bw_engine*, const int16_t* pcm, int64_t n_samples, int32_t sample_rate, bw_call** out);
/* stage-level: resampled float32 audio back to the host (out holds ceil(new * n / orig) samples; count in *n_out) */
int bw_resample_pcm16(bw_engine*, const int16_t* pcm, int64_t n_samples, int32_t sample_rate, float* out, int64_t* n_out);
int bw_call_content_frames(bw_call*, int32_t* out);
/* Encoder + batched decoder for the 30 s window starting at mel frame `seek`. Blocking. */
int bw_call_decode(bw_call*, int32_t seek, const bw_decode_opts* opts, bw_result* out);
/* Explicit cross-session batch (SURVEY 8(f).3; what the reference declares as decode_batch_window_ms /
 * max_decode_batch_size, config/server.yaml:48-49, and never implements): n windows -- calls[i] at seeks[i] with
 * opts[i] -- are handed to the scheduler together by ONE host thread and share encoder launches and every decoder
 * step.  Blocking until all are done; statuses[i] (may be NULL) gets each window's bw_status, the return value is the
 * first non-zero one.  The same call may appear more than once (different seeks). */
int bw_decode_many(bw_call* const* calls, const int32_t* seeks, const bw_decode_opts* opts, bw_result* results,
                   int32_t* statuses, int32_t n);
/* upstream decoding.detect_language on the window at `seek`. Blocking. */
int bw_call_detect_language(bw_call*, int32_t seek, bw_lang_result* out);
/* A decode that detects its own language: bw_call_decode and bw_call_detect_language of the same window in one
 * admission, one encoder pass and one cross-KV write.  opts->initial_tokens is the sot sequence with the language left
 * open: initial_tokens[0] = <|sot|> (sot_index 0, no prompt in front) and initial_tokens[1] = -1, the placeholder the
 * engine fills with the detected language token, e.g. {sot, -1, transcribe [, no_timestamps]}.  The language is the
 * arg-max over the language tokens of the <|sot|> row's logits -- the row, and the arithmetic, of
 * bw_call_detect_language(call, seek) -- chosen on the device; `out` and `lang` then hold what bw_call_detect_language
 * followed by bw_call_decode with that language's sot sequence return.  The detected token counts as an initial token
 * (sample_begin, timestamp rules and log-probabilities are those of the two-call path).
 * Detection window: the decode window at `seek`, with zeros past content_frames -- the window bw_call_detect_language
 * uses.  (Upstream transcribe detects on the first 30 s of log-mel of the padded audio; the two coincide when
 * content_frames - seek >= 3000.)
 * BW_ERR_INVALID when the model has no language tokens (an English-only vocabulary, n_vocab < 51865, as upstream's
 * is_multilingual), sot_index != 0, initial_tokens[1] != -1 or -1 appears anywhere else. */
int bw_call_decode_detect(bw_call*, int32_t seek, const bw_decode_opts* opts, bw_result* out, bw_lang_result* lang);
/* bw_decode_many with detect-mode windows mixed in: window i is in detect mode when its initial tokens hold the
 * placeholder -1 (checked as above); its language goes to langs[i].  langs has one entry per window (NULL: no window is
 * in detect mode); the entries of the other windows are zeroed. */
int bw_decode_many_detect(bw_call* const* calls, const int32_t* seeks, const bw_decode_opts* opts, bw_result* results,
                          bw_lang_result* langs, int32_t* statuses, int32_t n);
int bw_call_close(bw_call*);

/* ---- stage-level entry points (parity tests, ncu isolation) ---- */
/* log_mel_spectrogram(audio, n_mels, padding): out [n_mels, (n+padding)/160] f32, host pointers */
int bw_mel(bw_engine*, const float* pcm, int64_t n_samples, int32_t padding, float* out_mel, int32_t* out_frames);
/* AudioEncoder.forward: mel [B, n_mels, 3000] f32 host -> out [B, 1500, d] f32 host */
int bw_encode(bw_engine*, const float* mel, int32_t batch, float* out);
/* AudioEncoder + TextDecoder.forward (no cache) for one already-normalised mel window [n_mels, 3000]:
 * tokens [n] -> logits [n, V] f32.  Goes through the scheduler like any other request. */
int bw_decode_logits(bw_engine*, const float* mel_window, const int32_t* tokens, int32_t n, float* out_logits);

#ifdef __cplusplus
}
#endif
#endif /* B200_WHISPER_H */
