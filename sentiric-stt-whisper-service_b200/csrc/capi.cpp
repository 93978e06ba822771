// C ABI (include/sw_whisper.h): the drop-in boundary for the whisper.cpp C API subset that
// /root/reference/src/stt_engine.cpp binds (SURVEY.md §8b). No exceptions cross it.
#include <stdlib.h>
#include <string.h>

#include <new>

#include "sequencer.h"

using sw::Engine;
using sw::set_last_error;

#define API_GUARD_BEGIN try {
#define API_GUARD_END(fail)                                   \
  }                                                           \
  catch (const std::bad_alloc&) {                             \
    set_last_error("out of host memory");                     \
    return fail;                                              \
  }                                                           \
  catch (const std::exception& ex) {                          \
    set_last_error("internal error: %s", ex.what());          \
    return fail;                                              \
  }

extern "C" {

sw_ctx_params sw_ctx_default_params(void) {
  sw_ctx_params p;
  memset(&p, 0, sizeof(p));
  p.device = 0;
  p.max_batch = 64;
  p.max_beams = 5;
  p.flash_attn = 1;
  return p;
}

sw_ctx* sw_ctx_create(const char* path, const sw_ctx_params* params) {
  API_GUARD_BEGIN
  if (!path) {
    set_last_error("null model path");
    return nullptr;
  }
  const sw_ctx_params pi = params ? *params : sw_ctx_default_params();
  Engine* e = sw::engine_create(path, &pi);
  if (!e) return nullptr;
  if (const char* v = getenv("SW_XA_CTAS")) e->xa_max_ctas = atoi(v);  // development: cap also without lanes
  sw_ctx* c = new sw_ctx();
  c->e = e;
  // further lanes (sw_ctx_params.n_lanes; SW_LANES overrides for experiments). Auto: a second lane when
  // its buffers fit twice over in what is left of the device memory.
  int want = pi.n_lanes;
  if (const char* v = getenv("SW_LANES")) want = atoi(v);
  if (want <= 0) {
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    want = (e->max_batch >= 2 && free_b > 2 * e->buffer_bytes + (size_t(2) << 30)) ? 2 : 1;
  }
  if (want > 4) want = 4;
  for (int k = 1; k < want; ++k) {
    Engine* l = sw::engine_create_lane(e);
    if (!l) {
      sw::log_msg(3, "lane %d not created (%s): running with %d lane(s)", k, sw_last_error(), k);
      cudaGetLastError();
      break;
    }
    c->lanes.push_back(l);
  }
  if (!c->lanes.empty()) {
    // several lanes: the persistent cross attention leaves a third of the SMs to the other lanes' small
    // kernels (large-v3, 2 lanes x 64 windows: 148 CTAs 3033x, 111 3144x, 96 3200x, 80 3140x, 64 2963x RTFx;
    // profiles/r1_bench_lanes.log). The cache stream stays HBM-bound on 96 SMs.
    int cap = 0;
    if (const char* v = getenv("SW_XA_CTAS")) cap = atoi(v);
    else {
      int sms = 148;
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device);
      cap = sms * 13 / 20;
    }
    e->xa_max_ctas = cap;
    for (Engine* l : c->lanes) l->xa_max_ctas = cap;
  }
  return c;
  API_GUARD_END(nullptr)
}

void sw_ctx_destroy(sw_ctx* ctx) {
  if (!ctx) return;
  if (ctx->e) {
    cudaSetDevice(ctx->e->device);
    cudaDeviceSynchronize();
    sw::prosody_state_free(ctx->prosody.load());
    sw::resample_state_free(ctx->resample.load());
    for (Engine* l : ctx->lanes) delete l;
    delete ctx->e;
  }
  delete ctx;
}

int sw_ctx_model_info(const sw_ctx* ctx, sw_model_info* out) {
  if (!ctx || !out) {
    set_last_error("null argument");
    return -1;
  }
  const sw::HParams& hp = ctx->e->model->hp;
  const sw::Vocab& v = ctx->e->model->vocab;
  out->n_vocab = hp.n_vocab; out->n_audio_ctx = hp.n_audio_ctx; out->n_audio_state = hp.n_audio_state;
  out->n_audio_head = hp.n_audio_head; out->n_audio_layer = hp.n_audio_layer; out->n_text_ctx = hp.n_text_ctx;
  out->n_text_state = hp.n_text_state; out->n_text_head = hp.n_text_head; out->n_text_layer = hp.n_text_layer;
  out->n_mels = hp.n_mels; out->ftype = hp.ftype;
  out->is_multilingual = v.multilingual;
  out->token_eot = v.eot; out->token_sot = v.sot; out->token_translate = v.translate;
  out->token_transcribe = v.transcribe; out->token_solm = v.solm; out->token_prev = v.prev;
  out->token_nosp = v.nosp; out->token_not = v.not_; out->token_beg = v.beg;
  return 0;
}

const char* sw_token_to_str(const sw_ctx* ctx, int token) {
  if (!ctx || token < 0 || token >= (int)ctx->e->model->vocab.id_to_token.size()) return "";
  return ctx->e->model->vocab.id_to_token[token].c_str();
}
int sw_token_eot(const sw_ctx* ctx) { return ctx ? ctx->e->model->vocab.eot : -1; }
int sw_lang_id(const char* lang) { return sw::lang_id(lang); }

sw_full_params sw_full_default_params(int strategy) {
  sw_full_params p;
  memset(&p, 0, sizeof(p));
  p.strategy = strategy;
  p.beam_size = strategy == 1 ? 5 : -1;
  p.best_of = strategy == 0 ? 5 : -1;
  p.temperature = 0.0f;
  p.temperature_inc = 0.2f;
  p.entropy_thold = 2.4f;
  p.logprob_thold = -1.0f;
  p.no_speech_thold = 0.6f;
  p.suppress_blank = 1;
  p.no_context = 1;
  p.max_initial_ts = 1.0f;
  p.length_penalty = -1.0f;
  p.language = "en";
  p.n_threads = 4;
  return p;
}

int sw_full_batch_pcm16(sw_ctx* ctx, const sw_full_params* params, const int16_t* const* pcm16,
                        const int* n_samples, int n, sw_result** out) {
  API_GUARD_BEGIN
  if (!ctx || !params || !pcm16 || !n_samples || !out) {
    set_last_error("null argument");
    return -1;
  }
  return sw::run_full_batch_lanes(ctx, params, reinterpret_cast<const void* const*>(pcm16), n_samples, n, false, out);
  API_GUARD_END(-1)
}

int sw_full_batch_pcm16_lang(sw_ctx* ctx, const sw_full_params* params, const int16_t* const* pcm16,
                             const int* n_samples, int n, const char* const* languages, sw_result** out) {
  API_GUARD_BEGIN
  if (!ctx || !params || !pcm16 || !n_samples || !out) {
    set_last_error("null argument");
    return -1;
  }
  return sw::run_full_batch_lanes(ctx, params, reinterpret_cast<const void* const*>(pcm16), n_samples, n, false, out,
                                  languages);
  API_GUARD_END(-1)
}

int sw_full_batch_f32_lang(sw_ctx* ctx, const sw_full_params* params, const float* const* pcm, const int* n_samples,
                           int n, const char* const* languages, sw_result** out) {
  API_GUARD_BEGIN
  if (!ctx || !params || !pcm || !n_samples || !out) {
    set_last_error("null argument");
    return -1;
  }
  return sw::run_full_batch_lanes(ctx, params, reinterpret_cast<const void* const*>(pcm), n_samples, n, true, out,
                                  languages);
  API_GUARD_END(-1)
}

int sw_full_batch_f32(sw_ctx* ctx, const sw_full_params* params, const float* const* pcm,
                      const int* n_samples, int n, sw_result** out) {
  API_GUARD_BEGIN
  if (!ctx || !params || !pcm || !n_samples || !out) {
    set_last_error("null argument");
    return -1;
  }
  return sw::run_full_batch_lanes(ctx, params, reinterpret_cast<const void* const*>(pcm), n_samples, n, true, out);
  API_GUARD_END(-1)
}

int sw_full(sw_ctx* ctx, const sw_full_params* params, const float* pcm, int n_samples, sw_result** out) {
  const float* arr[1] = {pcm};
  return sw_full_batch_f32(ctx, params, arr, &n_samples, 1, out);
}
int sw_full_pcm16(sw_ctx* ctx, const sw_full_params* params, const int16_t* pcm, int n_samples,
                  sw_result** out) {
  const int16_t* arr[1] = {pcm};
  return sw_full_batch_pcm16(ctx, params, arr, &n_samples, 1, out);
}

int sw_result_n_segments(const sw_result* r) { return r ? (int)r->segs.size() : 0; }
const char* sw_result_segment_text(const sw_result* r, int i) { return r->segs[i].text.c_str(); }
int64_t sw_result_segment_t0(const sw_result* r, int i) { return r->segs[i].t0; }
int64_t sw_result_segment_t1(const sw_result* r, int i) { return r->segs[i].t1; }
int sw_result_segment_speaker_turn_next(const sw_result* r, int i) { return r->segs[i].speaker_turn_next; }
int sw_result_n_tokens(const sw_result* r, int i) { return (int)r->segs[i].tokens.size(); }
sw_token_data sw_result_token_data(const sw_result* r, int i, int j) { return r->segs[i].tokens[j]; }
int sw_result_lang_id(const sw_result* r) { return r ? r->lang_id : -1; }
int sw_result_n_decode_steps(const sw_result* r) { return r ? r->n_decode_steps : 0; }
int sw_result_n_windows(const sw_result* r) { return r ? r->n_windows : 0; }
void sw_result_free(sw_result* r) { delete r; }

void sw_ctx_set_kernel_timing(sw_ctx* ctx, int on) {
  if (!ctx) return;
  ctx->e->kernel_timing = on != 0;
  for (Engine* l : ctx->lanes) l->kernel_timing = on != 0;
}

int sw_ctx_get_stats(sw_ctx* ctx, sw_stats* out, int reset) {
  if (!ctx || !out) {
    set_last_error("null argument");
    return -1;
  }
  sw::StageTimes t = ctx->e->times;
  for (Engine* l : ctx->lanes) {  // sums over lanes (their device times overlap)
    const sw::StageTimes& u = l->times;
    t.ms_mel += u.ms_mel; t.ms_encode += u.ms_encode; t.ms_decode += u.ms_decode;
    t.n_windows += u.n_windows; t.n_steps += u.n_steps; t.n_launches += u.n_launches;
    t.decode_bytes += u.decode_bytes; t.h2d_bytes += u.h2d_bytes; t.d2h_bytes += u.d2h_bytes;
    t.ms_xattn += u.ms_xattn; t.n_xattn += u.n_xattn; t.xattn_bytes += u.xattn_bytes;
  }
  out->ms_mel = t.ms_mel; out->ms_encode = t.ms_encode; out->ms_decode = t.ms_decode;
  out->n_windows = t.n_windows; out->n_steps = t.n_steps; out->n_launches = t.n_launches;
  out->decode_bytes = t.decode_bytes;
  out->h2d_bytes = t.h2d_bytes; out->d2h_bytes = t.d2h_bytes;
  out->ms_xattn = t.ms_xattn; out->n_xattn = t.n_xattn; out->xattn_bytes = t.xattn_bytes;
  out->decoder_weight_bytes = (double)ctx->e->model->weight_bytes_decoder;
  out->n_lanes = 1 + (long)ctx->lanes.size();
  if (reset) {
    ctx->e->times = sw::StageTimes();
    for (Engine* l : ctx->lanes) l->times = sw::StageTimes();
  }
  return 0;
}

}  // extern "C"
