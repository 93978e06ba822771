/*
 * sw_whisper.h - C ABI of the B200-native Whisper inference hot path.
 *
 * This is the drop-in boundary for the path the reference reaches through the
 * whisper.cpp C API from exactly one file, src/stt_engine.cpp (SURVEY.md §8b).
 * Each entry point names the reference interface it replaces (file:line in
 * /root/reference). Plain pointers and sizes only; no C++ or torch types.
 *
 * Conventions: functions returning int return 0 on success and a negative
 * value on failure; sw_last_error() then holds a thread-local message. No
 * exceptions cross this boundary. Handles are opaque. A sw_ctx may be shared by
 * threads; results are owned by the caller until sw_result_free().
 *
 * There is NO CPU fallback behind this ABI: every compute entry point fails
 * loudly (negative return + message) when no sm_100 device is present.
 */
#ifndef SW_WHISPER_H
#define SW_WHISPER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SW_API __attribute__((visibility("default")))

typedef struct sw_ctx sw_ctx;
typedef struct sw_result sw_result;

/* ---- library ---------------------------------------------------------- */
SW_API const char* sw_last_error(void);
SW_API const char* sw_version(void);
/* number of CUDA devices with compute capability 10.x; 0 if none / no driver */
SW_API int sw_device_count(void);

/* replaces whisper_log_set (main.cpp:71); level: 2=info 3=warn 4=error, the
 * ggml_log_level values the reference's bridge switches on (main.cpp:37-55) */
typedef void (*sw_log_callback)(int level, const char* text, void* user);
SW_API void sw_log_set(sw_log_callback cb, void* user);

/* ---- context lifecycle ------------------------------------------------ */
/* replaces whisper_context_default_params (stt_engine.cpp:28) */
typedef struct sw_ctx_params {
  int device;          /* CUDA ordinal */
  int max_batch;       /* windows decoded together (default 64) */
  int max_beams;       /* sizes the row budget: max_batch * max_beams decoder rows per step (default 5). Any request
                          may still use up to 8 decoders per window (WHISPER_MAX_DECODERS); it then gets fewer
                          windows per device pass */
  int flash_attn;      /* accepted for API compatibility; always fused */
  int n_lanes;         /* independent batches in flight on the device (each lane has its own KV caches,
                        * activations and stream; the weights are shared). A decoder step is a chain of
                        * latency-bound kernels around one HBM-bound cross attention, so a second lane fills
                        * the first one's bubbles. 0 = auto (2 when the second lane's buffers fit), 1, 2. */
  int reserved[11];
} sw_ctx_params;
SW_API sw_ctx_params sw_ctx_default_params(void);

/* replaces whisper_init_from_file_with_params + whisper_init_state
 * (stt_engine.cpp:33,39): parses the legacy ggml .bin, uploads weights to HBM
 * as bf16, allocates KV caches / activations for max_batch windows.
 * Returns NULL on failure. */
SW_API sw_ctx* sw_ctx_create(const char* ggml_model_path, const sw_ctx_params* params);
/* replaces whisper_free_state + whisper_free (stt_engine.cpp:56-57) */
SW_API void sw_ctx_destroy(sw_ctx* ctx);

/* model facts (whisper_model_* / whisper_n_* accessors upstream) */
typedef struct sw_model_info {
  int n_vocab, n_audio_ctx, n_audio_state, n_audio_head, n_audio_layer;
  int n_text_ctx, n_text_state, n_text_head, n_text_layer, n_mels, ftype;
  int is_multilingual;
  int token_eot, token_sot, token_translate, token_transcribe, token_solm;
  int token_prev, token_nosp, token_not, token_beg;
} sw_model_info;
SW_API int sw_ctx_model_info(const sw_ctx* ctx, sw_model_info* out);
/* replaces whisper_token_to_str (stt_engine.cpp:291); borrowed pointer */
SW_API const char* sw_token_to_str(const sw_ctx* ctx, int token);
/* replaces whisper_token_eot (stt_engine.cpp:292) */
SW_API int sw_token_eot(const sw_ctx* ctx);
/* whisper_lang_id upstream: "en" -> 0 ...; -1 if unknown */
SW_API int sw_lang_id(const char* lang);

/* ---- decode parameters ------------------------------------------------ */
/* replaces whisper_full_params as filled at stt_engine.cpp:204-243 */
typedef int (*sw_abort_callback)(void* user); /* nonzero = abort (stt_engine.cpp:17-23) */
typedef struct sw_full_params {
  int strategy;            /* 0 greedy, 1 beam search (stt_engine.cpp:210-212) */
  int beam_size;           /* stt_engine.cpp:236 */
  int best_of;             /* stt_engine.cpp:238 */
  float temperature;       /* stt_engine.cpp:234 */
  float temperature_inc;   /* upstream default 0.2; 0 disables fallback */
  float entropy_thold;     /* stt_engine.cpp:241 */
  float logprob_thold;     /* stt_engine.cpp:242 */
  float no_speech_thold;   /* stt_engine.cpp:227 */
  int translate;           /* stt_engine.cpp:228 */
  int tdrz_enable;         /* stt_engine.cpp:229 */
  int suppress_nst;        /* stt_engine.cpp:226 */
  int suppress_blank;      /* upstream default 1 */
  int token_timestamps;    /* stt_engine.cpp:225 */
  int no_timestamps;       /* upstream default 0 */
  int single_segment;      /* upstream default 0 */
  int no_context;          /* upstream default 1 */
  float max_initial_ts;    /* upstream default 1.0 */
  float length_penalty;    /* upstream default -1 */
  const char* language;    /* stt_engine.cpp:232; "auto" or NULL = detect */
  const char* initial_prompt; /* stt_engine.cpp:233 */
  const int32_t* prompt_tokens; /* pre-tokenised prompt (upstream field of the same name) */
  int prompt_n_tokens;
  sw_abort_callback abort_callback;    /* stt_engine.cpp:217 */
  void* abort_callback_user_data;      /* stt_engine.cpp:218 */
  int n_threads;           /* stt_engine.cpp:243; host sequencer threads */
  int reserved[8];
} sw_full_params;
/* replaces whisper_full_default_params (stt_engine.cpp:214) */
SW_API sw_full_params sw_full_default_params(int strategy);

/* ---- the hot path ------------------------------------------------------ */
/* replaces whisper_full_with_state (stt_engine.cpp:245-246) for ONE utterance
 * of 16 kHz mono float PCM in host memory. *out receives the result. Returns 0
 * ok, non-zero on failure or abort (upstream convention). */
SW_API int sw_full(sw_ctx* ctx, const sw_full_params* params, const float* pcm, int n_samples,
                   sw_result** out);
/* int16 entry: folds the reference's host-side /32768 conversion loop
 * (transcribe_pcm16, stt_engine.cpp:117-125) into the device front end. */
SW_API int sw_full_pcm16(sw_ctx* ctx, const sw_full_params* params, const int16_t* pcm,
                         int n_samples, sw_result** out);
/* Batched entry the reference lacks (it runs one whisper_state per request,
 * stt_engine.cpp:36-42): n utterances decoded together. pcm16[i] points at
 * n_samples[i] int16 host samples. out[i] receives one result per utterance. */
SW_API int sw_full_batch_pcm16(sw_ctx* ctx, const sw_full_params* params,
                               const int16_t* const* pcm16, const int* n_samples, int n,
                               sw_result** out);
SW_API int sw_full_batch_f32(sw_ctx* ctx, const sw_full_params* params, const float* const* pcm,
                             const int* n_samples, int n, sw_result** out);
/* The same with a language per utterance: languages[i] is "en", "tr", ... or "auto" / NULL (detect); languages == NULL
 * means params->language for all. The language is the one per-request setting that only changes a prompt token
 * (stt_engine.cpp:230-232), so requests in different languages can share a device pass. */
SW_API int sw_full_batch_pcm16_lang(sw_ctx* ctx, const sw_full_params* params, const int16_t* const* pcm16,
                                    const int* n_samples, int n, const char* const* languages, sw_result** out);
SW_API int sw_full_batch_f32_lang(sw_ctx* ctx, const sw_full_params* params, const float* const* pcm,
                                  const int* n_samples, int n, const char* const* languages, sw_result** out);
/* page-locked host memory for PCM staging (optional; any host pointer is accepted) */
SW_API void* sw_host_alloc(size_t bytes);
SW_API void sw_host_free(void* p);

/* ---- result accessors (whisper_full_*_from_state, stt_engine.cpp:261-292) */
typedef struct sw_token_data { /* whisper_token_data */
  int32_t id, tid;
  float p, plog, pt, ptsum;
  int64_t t0, t1, t_dtw;
  float vlen;
} sw_token_data;
SW_API int sw_result_n_segments(const sw_result* r);                       /* :261 */
SW_API const char* sw_result_segment_text(const sw_result* r, int i);      /* :267 */
SW_API int64_t sw_result_segment_t0(const sw_result* r, int i);            /* :280 */
SW_API int64_t sw_result_segment_t1(const sw_result* r, int i);            /* :281 */
SW_API int sw_result_segment_speaker_turn_next(const sw_result* r, int i); /* :283 */
SW_API int sw_result_n_tokens(const sw_result* r, int i);                  /* :286 */
SW_API sw_token_data sw_result_token_data(const sw_result* r, int i, int j); /* :290 */
SW_API int sw_result_lang_id(const sw_result* r);
/* decode-loop statistics for the benchmark */
SW_API int sw_result_n_decode_steps(const sw_result* r);
SW_API int sw_result_n_windows(const sw_result* r);
SW_API void sw_result_free(sw_result* r);

/* ---- per-context device-time statistics (CUDA events on the engine's stream) ---- */
typedef struct sw_stats {
  double ms_mel, ms_encode, ms_decode; /* accumulated device time per stage */
  long n_windows, n_steps, n_launches; /* windows encoded, decoder steps, kernels launched */
  double decode_bytes;                 /* algorithmic bytes of the sampled decode steps */
  double decoder_weight_bytes;         /* bytes of decoder weights one step streams */
  double h2d_bytes, d2h_bytes;         /* PCM uploaded / picks + token-timestamp energy read back */
  double ms_xattn;                     /* device time inside cross-attention launches (kernel timing on) */
  long n_xattn;                        /* number of those launches */
  double xattn_bytes;                  /* their algorithmic bytes (cross-KV of the active windows, q, out) */
  long n_lanes;                        /* lanes of the context; the ms_* above are SUMS over lanes that overlap in time */
} sw_stats;
/* bracket every cross-attention launch with CUDA events on the engine's stream (bench roofline) */
SW_API void sw_ctx_set_kernel_timing(sw_ctx* ctx, int on);
SW_API int sw_ctx_get_stats(sw_ctx* ctx, sw_stats* out, int reset);

/* ---- per-segment prosody (SURVEY.md §8(f) rank 3) ----------------------- *
 * replaces the extract_prosody call the reference makes for every segment
 * (stt_engine.cpp:313-334 -> prosody_extractor.cpp:31-224): all segments of one
 * utterance in two kernel launches; the record has AffectiveTags' fields
 * (prosody_extractor.h:6-18). Segments shorter than 160 samples get the
 * reference's neutral record ('?', neutral, zeros). Results are bit-identical
 * to the reference's host code (tests/test_prosody.py). */
typedef struct sw_prosody_opts {   /* ProsodyOptions, prosody_extractor.h:20-26 */
  float lpf_alpha, gender_threshold, min_pitch, max_pitch;
} sw_prosody_opts;
enum { SW_EMOTION_NEUTRAL = 0, SW_EMOTION_EXCITED = 1, SW_EMOTION_SAD = 2, SW_EMOTION_ANGRY = 3 };
typedef struct sw_prosody {
  char gender;                     /* 'M', 'F' or '?' (gender_proxy) */
  int emotion;                     /* SW_EMOTION_* (emotion_proxy) */
  float arousal, valence, pitch_mean, pitch_std, energy_mean, energy_std, spectral_centroid,
      zero_crossing_rate;
  float speaker_vec[8];
} sw_prosody;
SW_API sw_prosody_opts sw_prosody_default_opts(void);
/* pcm: the utterance (host or device memory); segment i covers samples
 * [seg_begin[i], seg_end[i]) - the caller does the centisecond -> sample
 * conversion of stt_engine.cpp:313-320. out[n_segs]. */
SW_API int sw_prosody_segments_f32(sw_ctx* ctx, const float* pcm, int64_t n_samples, int sample_rate,
                                   const int64_t* seg_begin, const int64_t* seg_end, int n_segs,
                                   const sw_prosody_opts* opts, sw_prosody* out);
SW_API int sw_prosody_segments_pcm16(sw_ctx* ctx, const int16_t* pcm, int64_t n_samples, int sample_rate,
                                     const int64_t* seg_begin, const int64_t* seg_end, int n_segs,
                                     const sw_prosody_opts* opts, sw_prosody* out);

/* ---- sample-rate conversion (SURVEY.md §8(f) rank 4) -------------------- *
 * stands in for SttEngine::resample_audio (stt_engine.cpp:87-115, libsamplerate
 * src_simple(SRC_SINC_FASTEST), called at :138-145 for inputs that are not
 * 16 kHz). libsamplerate is not in the reference tree: the same published
 * method (windowed-sinc band-limited interpolation) with its own window;
 * parity with libsamplerate is not claimed (> 89 dB tone SNR instead). */
SW_API int64_t sw_resample_out_len(int64_t n_in, int sr_in, int sr_out); /* floor(n_in * sr_out / sr_in) */
/* in: n_in samples (host or device); out: sw_resample_out_len samples (host or device) */
SW_API int sw_resample_f32(sw_ctx* ctx, const float* in, int64_t n_in, int sr_in, int sr_out, float* out);

/* ---- stage-level hooks (parity tests and roofline measurement) --------- *
 * Host pointers in, host pointers out, synchronous. */
/* log-mel of one utterance (whisper.cpp log_mel_spectrogram): out is
 * [n_mel][n_len] f32 mel-major; returns n_len via *n_len. Pass out=NULL to
 * query n_len only. */
SW_API int sw_mel_pcm16(sw_ctx* ctx, const int16_t* pcm, int n_samples, float* out, int* n_len);
SW_API int sw_mel_f32(sw_ctx* ctx, const float* pcm, int n_samples, float* out, int* n_len);
/* encoder over n_windows windows of mel [n_windows][n_mel][3000] f32;
 * out [n_windows][1500][d] f32 (post ln_post). */
SW_API int sw_encode(sw_ctx* ctx, const float* mel, int n_windows, float* out);
/* teacher-forced decoder: tokens [n_windows][n_tok]; returns raw logits
 * [n_windows][n_tok][n_vocab] f32 for the windows last passed to sw_encode. */
SW_API int sw_decode_logits(sw_ctx* ctx, const int32_t* tokens, int n_windows, int n_tok,
                            float* logits);

/* ---- device-pointer kernel hooks (tests/bench; pointers are DEVICE) ---- */
/* C[M,N] = epi(A[M,K] . B[N,K]^T), bf16 in, flags: 1 gelu, 2 f32 out, 4 row bias */
SW_API int sw_dev_gemm_bf16(const void* dA, const void* dB, void* dC, const float* d_bias,
                            const float* d_residual, int M, int N, int K, int lda, int ldb, int ldc,
                            int flags, int block_n, void* stream);

/* decoder-step kernels in isolation (tools/dev_decode_kernels.py): skinny weight-streaming GEMM
 * (split <= 0: automatic) and the fused split-K-reduce + residual + LayerNorm */
SW_API int sw_dev_skinny_gemm(const void* dX, const void* dW, int R, int N, int K, const float* d_bias,
                              int gelu, void* d_out, float* d_partial, int split, void* stream);
SW_API int sw_dev_skinny_split(int N, int K);
/* the same with the kernel named: 0 = the engine's choice, 1 = mma.sync tiles (skinny_gemm.cu), 2 = tcgen05 with the
   weight rows in the M dimension (skinny_gemm_tc.cu) */
SW_API int sw_dev_skinny_gemm_k(int kernel, const void* dX, const void* dW, int R, int N, int K, const float* d_bias,
                                int gelu, void* d_out, float* d_partial, int split, void* stream);
SW_API int sw_dev_skinny_split_k(int kernel, int N, int K);
SW_API int sw_dev_layer_norm(float* d_x, int rows, int d, const float* g, const float* b,
                             void* d_out_bf16, const float* d_partial, int n_split, const float* d_bias,
                             void* stream);
/* encoder self attention: qkv [n_win*T][3d] bf16 (Q | K | V), out [n_win*T][d] bf16 */
SW_API int sw_dev_encoder_attention(const void* d_qkv, void* d_out, int n_win, int T, int d, int n_head, void* stream);
/* cross attention + combine; ws >= sw_dev_cross_attention_ws_floats(R, d, n_head) floats; max_ctas 0 = one CTA per SM */
SW_API size_t sw_dev_cross_attention_ws_floats(int R, int d, int n_head);
SW_API int sw_dev_cross_attention(const void* d_q, const void* d_kv, int64_t kv_rows, const int* d_grp_win,
                                  const int* d_grp_start, const int* d_grp_count, int n_groups, int max_count, int R,
                                  int T, int d, int n_head, float* d_ws, void* d_out, int max_ctas, void* stream);
/* paged causal self attention + append; rows: R DecRow records of 20 int32 each
   (slot, pos, win, pos0, pages[14], pad[2]); pool [page][n_layer][2][32][d] bf16 */
SW_API int sw_dev_self_attention(const void* d_qkv, const int* d_rows, int R, int d, int n_head, void* d_pool,
                                 int layer, int n_layer, void* d_out, void* stream);
/* development: hold n_ctas SMs (smem_bytes of shared memory and most of the register file each) for ms
   milliseconds on a private stream, optionally streaming stream_bytes of HBM meanwhile; n_ctas <= 0 waits
   for it to leave (tools/dev_chain_occupied.py: cost of a decoder layer's latency chain beside a resident
   cross attention) */
SW_API int sw_dev_occupy(int n_ctas, int smem_bytes, float ms, size_t stream_bytes);

#ifdef __cplusplus
}
#endif
#endif /* SW_WHISPER_H */
