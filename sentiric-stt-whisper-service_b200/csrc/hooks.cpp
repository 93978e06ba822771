// Stage-level hooks of the C ABI (parity tests and roofline measurement): host buffers in, host
// buffers out, synchronous. They run exactly the kernels the full path runs.
#include <string.h>

#include <algorithm>
#include <vector>

#include "sequencer.h"

namespace sw {
namespace {

int mel_hook(Engine* e, const void* pcm, int n_samples, bool is_f32, float* out, int* n_len_out) {
  SW_CHECK(n_samples >= 0, "negative sample count");
  std::lock_guard<std::mutex> lk(e->mu);
  SW_CUDA_CHECK(cudaSetDevice(e->device));
  const Model& m = *e->model;
  const int n_mel = m.hp.n_mels;
  MelUtt mu;
  mu.pcm_off = 0;
  mu.n_samples = n_samples;
  mu.n_len = (int)(((int64_t)n_samples + 30 * 16000 + 400 - 400) / 160);
  mu.n_active = std::min((n_samples + 200) / 160 + 1, mu.n_len);
  mu.log_off = 0;
  if (n_len_out) *n_len_out = mu.n_len;
  if (!out) return 0;
  SW_CHECK(n_samples == 0 || pcm, "null PCM");
  const size_t es = is_f32 ? 4 : 2;
  DevBuf<uint8_t> d_pcm;
  DevBuf<float> d_log, d_out;
  DevBuf<MelUtt> d_utt;
  DevBuf<unsigned> d_max;
  if (d_pcm.alloc((size_t)n_samples * es + 16) || d_log.alloc((size_t)n_mel * mu.n_active + 1) ||
      d_out.alloc((size_t)n_mel * mu.n_len) || d_utt.alloc(1) || d_max.alloc(1))
    return -1;
  cudaStream_t st = e->stream;
  if (n_samples) SW_CUDA_CHECK(cudaMemcpyAsync(d_pcm.p, pcm, (size_t)n_samples * es, cudaMemcpyHostToDevice, st));
  SW_CUDA_CHECK(cudaMemcpyAsync(d_utt.p, &mu, sizeof(mu), cudaMemcpyHostToDevice, st));
  const float neg10 = -10.0f;
  unsigned b;
  memcpy(&b, &neg10, 4);
  b = ~b;
  SW_CUDA_CHECK(cudaMemcpyAsync(d_max.p, &b, 4, cudaMemcpyHostToDevice, st));
  if (mel_log_power(d_pcm.p, is_f32, d_utt.p, 1, mu.n_active, m.filters, m.filter_span, n_mel, d_log.p, d_max.p, st)) return -1;
  if (mel_finalize_full(d_log.p, d_utt.p, d_max.p, 0, n_mel, mu.n_len, mu.n_active, d_out.p, st)) return -1;
  SW_CUDA_CHECK(cudaMemcpyAsync(out, d_out.p, (size_t)n_mel * mu.n_len * 4, cudaMemcpyDeviceToHost, st));
  SW_CUDA_CHECK(cudaStreamSynchronize(st));
  return 0;
}

}  // namespace
}  // namespace sw

using namespace sw;

extern "C" {

int sw_mel_pcm16(sw_ctx* ctx, const int16_t* pcm, int n_samples, float* out, int* n_len) {
  if (!ctx) {
    set_last_error("null context");
    return -1;
  }
  return mel_hook(ctx->e, pcm, n_samples, false, out, n_len);
}
int sw_mel_f32(sw_ctx* ctx, const float* pcm, int n_samples, float* out, int* n_len) {
  if (!ctx) {
    set_last_error("null context");
    return -1;
  }
  return mel_hook(ctx->e, pcm, n_samples, true, out, n_len);
}

int sw_encode(sw_ctx* ctx, const float* mel, int n_windows, float* out) {
  SW_CHECK(ctx && mel && n_windows > 0, "bad arguments");
  Engine* e = ctx->e;
  std::lock_guard<std::mutex> lk(e->mu);
  SW_CUDA_CHECK(cudaSetDevice(e->device));
  const HParams& hp = e->model->hp;
  const size_t win_in = (size_t)hp.n_mels * 3000, win_out = (size_t)1500 * hp.n_audio_state;
  DevBuf<float> d_mel, d_out;
  const int chunk = std::min(n_windows, e->max_batch);
  if (d_mel.alloc(win_in * chunk) || (out && d_out.alloc(win_out * chunk))) return -1;
  for (int w0 = 0; w0 < n_windows; w0 += chunk) {
    const int nb = std::min(chunk, n_windows - w0);
    SW_CUDA_CHECK(cudaMemcpyAsync(d_mel.p, mel + w0 * win_in, win_in * nb * 4, cudaMemcpyHostToDevice, e->stream));
    if (mel_f32_to_conv_input(d_mel.p, nb, hp.n_mels, e->conv_in.p, e->stream)) return -1;
    if (engine_encode(e, nb, out ? d_out.p : nullptr)) return -1;
    if (out)
      SW_CUDA_CHECK(cudaMemcpyAsync(out + w0 * win_out, d_out.p, win_out * nb * 4, cudaMemcpyDeviceToHost, e->stream));
    SW_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  }
  return 0;
}

int sw_decode_logits(sw_ctx* ctx, const int32_t* tokens, int n_windows, int n_tok, float* logits) {
  SW_CHECK(ctx && tokens && logits && n_windows > 0 && n_tok > 0, "bad arguments");
  Engine* e = ctx->e;
  std::lock_guard<std::mutex> lk(e->mu);
  SW_CUDA_CHECK(cudaSetDevice(e->device));
  const HParams& hp = e->model->hp;
  SW_CHECK(n_windows <= e->max_batch && n_windows <= e->max_rows, "n_windows %d exceeds max_batch", n_windows);
  SW_CHECK(n_tok <= hp.n_text_ctx, "n_tok %d exceeds the text context", n_tok);
  for (int i = 0; i < n_windows * n_tok; ++i)
    SW_CHECK(tokens[i] >= 0 && tokens[i] < hp.n_vocab, "token %d out of range", tokens[i]);
  e->pager.reset(e->n_pages, e->max_rows);
  LogitCfg cfg;
  memset(&cfg, 0, sizeof(cfg));
  for (int pos = 0; pos < n_tok; ++pos) {
    StepRows step(e);
    for (int w = 0; w < n_windows; ++w) {
      if (e->pager.ensure(w, pos)) return -1;
      step.open(w);
      step.add(w, pos, pos, tokens[(size_t)w * n_tok + pos]);
      step.close();
    }
    if (engine_decode_step(e, step, true, 0, cfg)) return -1;
    SW_CUDA_CHECK(cudaMemcpy2DAsync(logits + (size_t)pos * hp.n_vocab, (size_t)n_tok * hp.n_vocab * 4,
                                    e->logits.p, e->logits_ld * 4, (size_t)hp.n_vocab * 4, n_windows,
                                    cudaMemcpyDeviceToHost, e->stream));
    SW_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  }
  return 0;
}

void* sw_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) {
    cudaGetLastError();
    set_last_error("cudaMallocHost(%zu) failed", bytes);
    return nullptr;
  }
  return p;
}
void sw_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

}  // extern "C"
