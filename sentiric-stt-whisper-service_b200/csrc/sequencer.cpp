// Host sequencer: the control flow of whisper_full_with_state (SURVEY.md A.6; reference call site
// stt_engine.cpp:245-246) re-organised around BATCHES of 30 s windows. Per utterance it keeps the
// data-dependent `seek` loop, prompt construction, timestamp-rule state, greedy / beam-search /
// temperature-fallback bookkeeping, segment splitting and token-level timestamps; all arithmetic
// (mel, encoder, decoder, logit rules, argmax / draws) runs in the CUDA kernels driven from here.
#include "sequencer.h"

#include <math.h>
#include <string.h>

#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <deque>
#include <map>
#include <random>
#include <thread>

#include "host_common.h"

namespace sw {
namespace {

double wall_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

constexpr int SR = 16000;
constexpr int CHUNK_CS = 3000;  // 30 s in centiseconds
constexpr int DELTA_MIN = 10;

struct Sequence {
  std::vector<sw_token_data> tokens;
  int result_len = 0;
  double sum_logprobs_all = 0, sum_logprobs = 0, avg_logprobs = 0, entropy = 0, score = 0;
};
struct Decoder {
  Sequence seq;
  int seek_delta = CHUNK_CS;
  bool failed = false, completed = false, has_ts = false;
};
struct Utt {
  int n_samples = 0, n_len = 0, n_len_org = 0, n_active = 0;
  int lang = -1;
  int seek = 0, seek_end = 0;
  std::vector<int> prompt_past;
  std::mt19937 rng[8];
  int64_t en_off = 0;  // its smoothed |x| in the engine's device energy buffer (same offset as its PCM)
  int blk_off = 0;     // its 256-sample blocks in the block min / max arrays
  int n_energy = 0;
  int64_t t_beg = 0, t_last = 0;
  int tid_last = 0;
  sw_result* res = nullptr;
};
struct Job {
  int utt;
  int temp_idx;
};
struct Window {  // one job in flight
  int utt = 0, temp_idx = 0, seek = 0;
  float t_cur = 0.f;
  int n_cur = 1;
  std::vector<int> prompt;
  int n_init = 0;  // trailing prompt_init tokens
  Decoder dec[8];
  float no_speech_prob = 0.f;
  bool done = false;  // all decoders completed or failed
  std::vector<int> tt_segs;  // result segments this window emitted whose token times still need the energy pass
};

// whisper_sequence_score
void sequence_score(const sw_full_params& p, Sequence& s) {
  if (s.result_len == 0) return;
  double r = 0.0;
  for (int i = 0; i < s.result_len; ++i) r += s.tokens[i].plog;
  s.sum_logprobs = r;
  s.avg_logprobs = r / s.result_len;
  double penalty = s.result_len;
  if (p.length_penalty > 0.0f) penalty = pow((5.0 + penalty) / 6.0, p.length_penalty);
  s.score = r / penalty;
  std::map<int, int> cnt;
  int c = 0;
  for (int i = std::max(0, s.result_len - 32); i < s.result_len; ++i) {
    cnt[s.tokens[i].id]++;
    c++;
  }
  double e = 0.0;
  for (auto& kv : cnt) {
    const double q = kv.second / (double)c;
    e -= q * log(q);
  }
  s.entropy = e;
}

bool same_tokens(const Sequence& a, const Sequence& b) {
  if (a.tokens.size() != b.tokens.size()) return false;
  for (size_t k = 0; k < a.tokens.size(); ++k)
    if (a.tokens[k].id != b.tokens[k].id) return false;
  return true;
}

// ---- token-level timestamps (whisper_exp_compute_token_level_timestamps, SURVEY.md A.7) ----
float voice_length(const std::string& text) {
  float r = 0.f;
  for (char c : text) {
    if (c == ' ') r += 0.01f;
    else if (c == ',') r += 2.00f;
    else if (c == '.' || c == '!' || c == '?') r += 3.00f;
    else if (c >= '0' && c <= '9') r += 3.00f;
    else r += 1.00f;
  }
  return r;
}
inline int ts_to_sample(int64_t t, int n) { return std::max(0, std::min(n - 1, (int)((t * SR) / 100))); }
inline int64_t sample_to_ts(int i) { return (100ll * i) / SR; }

// first half of whisper_exp_compute_token_level_timestamps; returns true if the segment needs the energy pass
bool token_timestamps(const Model& m, Utt& u, sw_segment& seg) {
  const float thold_pt = 0.01f, thold_ptsum = 0.01f;
  auto& tk = seg.tokens;
  const int n_samples = u.n_energy;
  const int n = (int)tk.size();
  if (n_samples == 0 || n == 0) return false;
  const int64_t t0 = seg.t0, t1 = seg.t1;
  if (n == 1) {
    tk[0].t0 = t0;
    tk[0].t1 = t1;
    return false;
  }
  const int beg = m.vocab.beg;
  for (int j = 0; j < n; ++j) {
    sw_token_data& t = tk[j];
    if (j == 0) {
      if (t.id == beg) {
        tk[0].t0 = t0;
        tk[0].t1 = t0;
        tk[1].t0 = t0;
        u.t_beg = t0;
        u.t_last = t0;
        u.tid_last = beg;
      } else {
        tk[0].t0 = u.t_last;
      }
    }
    const int64_t tt = u.t_beg + 2 * (t.tid - beg);
    t.vlen = voice_length(m.vocab.id_to_token[t.id]);
    if (t.pt > thold_pt && t.ptsum > thold_ptsum && t.tid > u.tid_last && tt <= t1) {
      if (j > 0) tk[j - 1].t1 = tt;
      t.t0 = tt;
      u.tid_last = t.tid;
    }
  }
  tk[n - 2].t1 = t1;
  tk[n - 1].t0 = t1;
  tk[n - 1].t1 = t1;
  u.t_last = t1;
  // unknown stretches: split proportionally to the voice length
  for (int p0 = 0, p1 = 0;;) {
    while (p1 < n && tk[p1].t1 < 0) p1++;
    if (p1 >= n) p1--;
    if (p1 > p0) {
      double psum = 0.0;
      for (int j = p0; j <= p1; ++j) psum += tk[j].vlen;
      const double dt = (double)(tk[p1].t1 - tk[p0].t0);
      for (int j = p0 + 1; j <= p1; ++j) {
        const double ct = tk[j - 1].t0 + dt * tk[j - 1].vlen / psum;
        tk[j - 1].t1 = (int64_t)ct;
        tk[j].t0 = (int64_t)ct;
      }
    }
    p1++;
    p0 = p1;
    if (p1 >= n) break;
  }
  for (int j = 0; j < n - 1; ++j) {
    if (tk[j].t1 < 0) tk[j + 1].t0 = tk[j].t1;
    if (j > 0 && tk[j - 1].t1 > tk[j].t0) {
      tk[j].t0 = tk[j - 1].t1;
      tk[j].t1 = std::max(tk[j].t0, tk[j].t1);
    }
  }
  // the expand / contract of every text token on the smoothed signal energy follows on the device, for all
  // segments of the finished batch at once (Run::refine_token_times -> token_times.cu)
  return true;
}

// whisper_tokenize stand-in for initial_prompt: greedy longest match over the vocabulary
std::vector<int> tokenize(const Model& m, const char* text) {
  std::vector<int> out;
  const std::string s(text ? text : "");
  size_t i = 0;
  while (i < s.size()) {
    int found = -1;
    size_t flen = 0;
    for (size_t len = std::min<size_t>(s.size() - i, 32); len >= 1; --len) {
      auto it = m.vocab.token_to_id.find(s.substr(i, len));
      if (it != m.vocab.token_to_id.end() && it->second < m.vocab.eot) {
        found = it->second;
        flen = len;
        break;
      }
    }
    if (found < 0) {
      ++i;
      continue;
    }
    out.push_back(found);
    i += flen;
  }
  return out;
}

struct Run {
  Engine* e;
  const sw_full_params& p;
  const Model& m;
  std::vector<Utt> utts;
  std::vector<float> temps;
  std::vector<int> prompt_init_tail;  // [transcribe|translate] (+ [not])
  LogitCfg cfg;
  int beam = 1, best_of = 1;
  Run(Engine* e_, const sw_full_params& p_) : e(e_), p(p_), m(*e_->model) {}

  bool aborted() const { return p.abort_callback && p.abort_callback(p.abort_callback_user_data); }

  int setup_logit_cfg() {
    const Vocab& v = m.vocab;
    std::vector<uint8_t> sup(m.hp.n_vocab, 0);
    sup[v.not_] = 1;
    if (p.no_timestamps)
      for (int i = v.beg; i < m.hp.n_vocab; ++i) sup[i] = 1;
    sup[v.sot] = 1;
    sup[v.nosp] = 1;
    if (!p.tdrz_enable) sup[v.solm] = 1;
    sup[v.translate] = 1;
    sup[v.transcribe] = 1;
    sup[v.prev] = 1;
    for (int i = 0; i < v.n_langs; ++i) sup[v.sot + 1 + i] = 1;
    if (p.suppress_nst)
      for (int id : v.nst_ids) sup[id] = 1;
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_suppress.p, sup.data(), sup.size(), cudaMemcpyHostToDevice, e->stream));
    SW_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    cfg.n_vocab = m.hp.n_vocab;
    cfg.token_eot = v.eot;
    cfg.token_beg = v.beg;
    cfg.token_nosp = v.nosp;
    cfg.token_space = v.space;
    cfg.suppress_blank = p.suppress_blank;
    cfg.max_initial_ts_id = m.hp.n_vocab;
    if (p.max_initial_ts > 0.0f) {
      const float precision = 30.0f / m.hp.n_audio_ctx;
      cfg.max_initial_ts_id = v.beg + (int)roundf(p.max_initial_ts / precision) + 1;
    }
    cfg.d_suppress = e->d_suppress.p;
    return 0;
  }

  // ---- front end for the whole batch of utterances
  int front_end(const void* const* pcm, const int* n_samples, int n, bool is_f32) {
    const int n_mel = m.hp.n_mels;
    const size_t es = is_f32 ? 4 : 2;
    std::vector<MelUtt> mu(n);
    int64_t pcm_off = 0, log_off = 0;
    int max_active = 0, blk_off = 0;
    utts.resize(n);
    for (int i = 0; i < n; ++i) {
      Utt& u = utts[i];
      u.n_samples = n_samples[i];
      const int64_t n_padded = (int64_t)u.n_samples + 30 * SR + 400;
      u.n_len = (int)((n_padded - 400) / 160);
      u.n_len_org = 1 + (u.n_samples + 200 - 400) / 160;
      u.n_active = std::min((u.n_samples + 200) / 160 + 1, u.n_len);
      mu[i].pcm_off = pcm_off;
      mu[i].n_samples = u.n_samples;
      mu[i].n_active = u.n_active;
      mu[i].n_len = u.n_len;
      mu[i].log_off = log_off;
      mu[i].blk_off = blk_off;
      blk_off += (u.n_samples + 255) / 256;
      pcm_off += ((int64_t)u.n_samples + 7) / 8 * 8;
      log_off += (int64_t)n_mel * u.n_active;
      max_active = std::max(max_active, u.n_active);
      for (int j = 0; j < 8; ++j) u.rng[j] = std::mt19937(j);
    }
    if ((size_t)pcm_off * es > e->pcm_capacity) {
      e->d_pcm.release();
      e->pcm_capacity = (size_t)pcm_off * es * 5 / 4 + 1024;
      if (e->d_pcm.alloc(e->pcm_capacity)) return -1;
    }
    if ((size_t)log_off > e->log_capacity) {
      e->d_log.release();
      e->log_capacity = (size_t)log_off * 5 / 4 + 1024;
      if (e->d_log.alloc(e->log_capacity)) return -1;
    }
    if (n > e->utt_capacity) {
      e->d_utts.release();
      e->d_max_enc.release();
      e->utt_capacity = n * 2 + 64;
      if (e->d_utts.alloc(e->utt_capacity) || e->d_max_enc.alloc(e->utt_capacity)) return -1;
    }
    if (!e->d_win_utt.p) {
      if (e->d_win_utt.alloc(e->max_batch) || e->d_win_seek.alloc(e->max_batch)) return -1;
    }
    cudaStream_t st = e->stream;
    SW_CUDA_CHECK(cudaEventRecord(e->ev0, st));
    for (int i = 0; i < n; ++i)
      if (n_samples[i] > 0)
        SW_CUDA_CHECK(cudaMemcpyAsync(e->d_pcm.p + mu[i].pcm_off * es, pcm[i], (size_t)n_samples[i] * es,
                                      cudaMemcpyDefault, st));  // host (pageable/pinned) or device source
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_utts.p, mu.data(), n * sizeof(MelUtt), cudaMemcpyHostToDevice, st));
    // running max starts at log10(1e-10) = -10: every utterance has zero-pad frames
    std::vector<unsigned> init(n);
    {
      const float neg10 = -10.0f;
      unsigned b;
      memcpy(&b, &neg10, 4);
      std::fill(init.begin(), init.end(), ~b);  // ordered encoding of a negative float = complement
    }
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_max_enc.p, init.data(), n * sizeof(unsigned), cudaMemcpyHostToDevice, st));
    if (mel_log_power(e->d_pcm.p, is_f32, e->d_utts.p, n, max_active, m.filters, m.filter_span, n_mel, e->d_log.p,
                      e->d_max_enc.p, st))
      return -1;
    e->times.n_launches++;
    if (p.token_timestamps && pcm_off > 0) {
      int max_n = 0;
      for (int i = 0; i < n; ++i) max_n = std::max(max_n, n_samples[i]);
      if ((size_t)pcm_off > e->energy_capacity) {
        e->d_energy.release();
        e->energy_capacity = (size_t)pcm_off * 5 / 4 + 1024;
        if (e->d_energy.alloc(e->energy_capacity)) return -1;
      }
      if ((size_t)blk_off > e->eblk_capacity) {
        e->d_eblk.release();
        e->eblk_capacity = (size_t)blk_off * 5 / 4 + 64;
        if (e->d_eblk.alloc(2 * e->eblk_capacity)) return -1;
      }
      if (signal_energy(e->d_pcm.p, is_f32, e->d_utts.p, n, max_n, 32, e->d_energy.p, e->d_eblk.p,
                        e->d_eblk.p + e->eblk_capacity, st))
        return -1;
      e->times.n_launches++;
      // the energy stays in HBM: the token-time pass that reads it runs there too (refine_token_times)
      for (int i = 0; i < n; ++i) {
        utts[i].en_off = mu[i].pcm_off;
        utts[i].blk_off = mu[i].blk_off;
        utts[i].n_energy = n_samples[i];
      }
    }
    SW_CUDA_CHECK(cudaEventRecord(e->ev1, st));
    SW_CUDA_CHECK(cudaEventSynchronize(e->ev1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev0, e->ev1);
    e->times.ms_mel += ms;
    for (int i = 0; i < n; ++i) e->times.h2d_bytes += (double)n_samples[i] * es;
    return 0;
  }

  int finalize_windows(const std::vector<int>& wutt, const std::vector<int>& wseek) {
    const int n = (int)wutt.size();
    cudaStream_t st = e->stream;
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_win_utt.p, wutt.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_win_seek.p, wseek.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
    if (mel_finalize_windows(e->d_log.p, e->d_utts.p, e->d_max_enc.p, e->d_win_utt.p, e->d_win_seek.p, n,
                             m.hp.n_mels, e->conv_in.p, nullptr, st))
      return -1;
    e->times.n_launches++;
    SW_CUDA_CHECK(cudaStreamSynchronize(st));  // wutt/wseek are pageable
    return 0;
  }

  // ---- language auto-detect (whisper_lang_auto_detect_with_state): encode window 0, decode [sot]
  int detect_languages(const std::vector<int>& need) {
    const Vocab& v = m.vocab;
    for (size_t b0 = 0; b0 < need.size(); b0 += e->max_batch) {
      const int nb = (int)std::min<size_t>(e->max_batch, need.size() - b0);
      std::vector<int> wutt(need.begin() + b0, need.begin() + b0 + nb), wseek(nb, 0);
      if (finalize_windows(wutt, wseek)) return -1;
      if (engine_encode(e, nb, nullptr)) return -1;
      e->pager.reset(e->n_pages, e->max_rows);
      StepRows step(e);
      for (int w = 0; w < nb; ++w) {
        if (e->pager.ensure(w, 0)) return -1;
        step.open(w);
        step.add(w, 0, 0, v.sot);
        step.close();
      }
      if (engine_decode_step(e, step, true, 0, cfg)) return -1;
      std::vector<float> lg((size_t)nb * v.n_langs);
      SW_CUDA_CHECK(cudaMemcpy2DAsync(lg.data(), v.n_langs * sizeof(float), e->logits.p + v.sot + 1,
                                      e->logits_ld * sizeof(float), v.n_langs * sizeof(float), nb,
                                      cudaMemcpyDeviceToHost, e->stream));
      SW_CUDA_CHECK(cudaStreamSynchronize(e->stream));
      for (int w = 0; w < nb; ++w) {
        int best = 0;
        for (int i = 1; i < v.n_langs; ++i)
          if (lg[(size_t)w * v.n_langs + i] > lg[(size_t)w * v.n_langs + best]) best = i;
        utts[wutt[w]].lang = best;
      }
    }
    return 0;
  }

  void fill_lrow(LogitRow& lr, const Window& w, int j, int logits_row, bool initial) {
    const Decoder& d = w.dec[j];
    const int beg = m.vocab.beg;
    const auto& tk = d.seq.tokens;
    memset(&lr, 0, sizeof(lr));
    lr.is_initial = initial ? 1 : 0;
    lr.last_ts = (!initial && !tk.empty() && tk.back().id >= beg) ? 1 : 0;
    lr.penult_ts = (initial || tk.size() < 2 || tk[tk.size() - 2].id >= beg) ? 1 : 0;
    lr.ts_min = d.has_ts ? d.seek_delta / 2 : 0;
    lr.temperature = w.t_cur;
    lr.logits_row = logits_row;
    Utt& u = utts[w.utt];
    if (p.strategy == 1) {
      // beam strategy: whisper_sample_token_topk = beam_size draws from the decoder's own rng
      lr.n_draws = beam;
      for (int k = 0; k < beam; ++k) lr.u[k] = std::generate_canonical<double, 53>(u.rng[j]);
    } else if (w.t_cur >= 1e-6f) {
      lr.n_draws = 1;  // whisper_sample_token(best = false)
      lr.u[0] = std::generate_canonical<double, 53>(u.rng[j]);
    } else {
      lr.n_draws = 0;  // argmax
    }
  }

  static sw_token_data to_token(const PickOut& o) {
    sw_token_data t;
    t.id = o.id;
    t.tid = o.tid;
    t.p = o.p;
    t.plog = o.plog;
    t.pt = o.pt;
    t.ptsum = o.ptsum;
    t.t0 = -1;
    t.t1 = -1;
    t.t_dtw = -1;
    t.vlen = 0.f;
    return t;
  }

  // per-decoder state update after a token was appended at iteration i (upstream "update the decoder state")
  void update_decoder(Window& w, Decoder& d, int i, int n_max) {
    const Vocab& v = m.vocab;
    const Utt& u = utts[w.utt];
    const sw_token_data& tk = d.seq.tokens.back();
    if (tk.id > v.beg) {
      const int sd_new = 2 * (tk.id - v.beg);
      if (d.has_ts && d.seek_delta > sd_new && d.seq.result_len < i) {
        d.failed = true;
        return;
      }
      d.seek_delta = sd_new;
      d.seq.result_len = i + 1;
      d.has_ts = true;
    }
    if (tk.id == v.eot || (d.has_ts && w.seek + d.seek_delta + DELTA_MIN >= u.seek_end)) {
      if (d.seq.result_len == 0 && !p.no_timestamps) {
        if (w.seek + d.seek_delta + DELTA_MIN >= u.seek_end) d.seq.result_len = i + 1;
        else {
          d.failed = true;
          return;
        }
      }
      if (p.single_segment || p.no_timestamps) {
        d.seq.result_len = i + 1;
        d.seek_delta = CHUNK_CS;
      }
      d.completed = true;
      return;
    }
    if (i == n_max - 1 && (d.seq.result_len == 0 || d.seek_delta < CHUNK_CS / 2)) d.failed = true;
  }

  using Picks = std::vector<std::vector<std::vector<PickOut>>>;  // [window][decoder][draw] of the last step

  // ---- the prompt of every window into the self-KV of its first slot; the step in which a window's prompt ends
  // gives each of its decoders its first distribution. Common case ([sot, lang, task]): every position in ONE step -
  // the rows of a window share its cross-KV read (they sit in the M dimension of the cross-attention MMAs, which take
  // up to 8 rows per window) and self attention is causal over the positions appended in the same step. Longer
  // prompts go one position per step.
  int prefill(std::vector<Window>& wins, const std::vector<int>& slot0, Picks& picks) {
    int max_prompt = 0, total = 0;
    for (auto& w : wins) {
      max_prompt = std::max(max_prompt, (int)w.prompt.size());
      total += (int)w.prompt.size();
    }
    const int chunk = total <= e->max_rows && max_prompt <= 8 ? max_prompt : 1;
    for (int pos0 = 0; pos0 < max_prompt; pos0 += chunk) {
      StepRows step(e);
      std::vector<std::pair<int, int>> lmap;  // (window, decoder) of each logit row
      for (int wi = 0; wi < (int)wins.size(); ++wi) {
        Window& w = wins[wi];
        const int P = (int)w.prompt.size(), end = std::min(P, pos0 + chunk);
        if (pos0 >= P) continue;
        int row = 0;
        step.open(wi);
        for (int pos = pos0; pos < end; ++pos) {
          if (e->pager.ensure(slot0[wi], pos)) return -1;
          row = step.add(slot0[wi], pos, pos0, w.prompt[pos]);
        }
        step.close();
        if (end < P) continue;
        for (int j = 0; j < w.n_cur; ++j) {
          fill_lrow(e->h_lrows.p[lmap.size()], w, j, row, true);
          lmap.push_back({wi, j});
        }
        utts[w.utt].res->n_decode_steps++;
      }
      const int n_lr = (int)lmap.size();
      if (engine_decode_step(e, step, n_lr > 0, n_lr, cfg)) return -1;
      for (int k = 0; k < n_lr; ++k)
        std::copy_n(e->h_picks.p + k * 8, 8, picks[lmap[k].first][lmap[k].second].begin());
    }
    return 0;
  }

  // ---- beam search over one window at iteration i: the decoders continue the best distinct candidates among
  // beam draws of each, and positions [0, prompt + i) of the self-KV follow each candidate's source decoder
  int select_beams(Window& w, const std::vector<std::vector<PickOut>>& wp, int i, int slot0, std::vector<int>& copies,
                   std::vector<int>& release) {
    struct Cand {
      int decoder_idx, seek_delta;
      bool has_ts;
      Sequence seq;
    };
    std::vector<Cand> cands;
    for (int j = 0; j < w.n_cur; ++j) {
      Decoder& d = w.dec[j];
      if (d.completed || d.failed) continue;
      for (int k = 0; k < beam; ++k) {
        Cand c{j, d.seek_delta, d.has_ts, d.seq};
        const sw_token_data t = to_token(wp[j][k]);
        c.seq.tokens.push_back(t);
        c.seq.sum_logprobs_all += t.plog;
        cands.push_back(std::move(c));
      }
    }
    std::stable_sort(cands.begin(), cands.end(), [](const Cand& a, const Cand& b) {
      if (a.seq.sum_logprobs_all != b.seq.sum_logprobs_all) return a.seq.sum_logprobs_all > b.seq.sum_logprobs_all;
      return a.decoder_idx < b.decoder_idx;
    });
    size_t cc = 0;
    std::vector<int> src(w.n_cur, -1);
    for (int j = 0; j < w.n_cur; ++j) {
      Decoder& d = w.dec[j];
      if (d.completed || d.failed) continue;
      if (cc >= cands.size()) cc = 0;
      Cand& cur = cands[cc++];
      while (cands.size() > cc && same_tokens(cands[cc].seq, cur.seq) && i > 0) ++cc;
      d.seek_delta = cur.seek_delta;
      d.has_ts = cur.has_ts;
      d.seq = cur.seq;
      src[j] = cur.decoder_idx;
    }
    return e->pager.remap(slot0, src, (int)w.prompt.size() + i, copies, release);
  }

  // ---- the step at position prompt + i: one row per active decoder, grouped by window; its picks go to `picks`
  int next_step(std::vector<Window>& wins, const std::vector<int>& slot0, int i, Picks& picks) {
    StepRows step(e);
    std::vector<std::pair<int, int>> rmap;  // (window, decoder) of each row
    double kv_tokens = 0;                   // self-KV positions the rows read
    for (int wi = 0; wi < (int)wins.size(); ++wi) {
      Window& w = wins[wi];
      if (w.done) continue;
      const int pos = (int)w.prompt.size() + i;
      step.open(wi);
      for (int j = 0; j < w.n_cur; ++j) {
        Decoder& d = w.dec[j];
        if (d.completed || d.failed) continue;
        if (e->pager.ensure(slot0[wi] + j, pos)) return -1;
        const int row = step.add(slot0[wi] + j, pos, pos, d.seq.tokens.back().id);
        fill_lrow(e->h_lrows.p[row], w, j, row, false);
        rmap.push_back({wi, j});
        kv_tokens += pos + 1;
      }
      step.close();
      utts[w.utt].res->n_decode_steps++;
    }
    if (engine_decode_step(e, step, true, step.R, cfg)) return -1;
    for (int k = 0; k < step.R; ++k)
      std::copy_n(e->h_picks.p + k * 8, 8, picks[rmap[k].first][rmap[k].second].begin());
    // decode-step byte accounting (roofline): weights + per-window cross-KV + self-KV read
    const double L = m.hp.n_text_layer, dd = m.hp.n_text_state;
    e->times.decode_bytes +=
        (double)m.weight_bytes_decoder + step.G * L * 2.0 * 1500 * dd * 2.0 + L * 2.0 * dd * 2.0 * kv_tokens;
    return 0;
  }

  // ---- decode a batch of windows to completion; cross-KV for window index w is already in place
  int decode_windows(std::vector<Window>& wins) {
    const int nw = (int)wins.size();
    // self-KV slots: window w owns slots [slot0[w], slot0[w] + n_cur) - the batch was admitted with
    // sum(n_cur) <= max_rows rows, so every slot index stays below the pager's max_rows slots
    std::vector<int> slot0(nw, 0);
    for (int w = 1; w < nw; ++w) slot0[w] = slot0[w - 1] + wins[w - 1].n_cur;
    e->pager.reset(e->n_pages, e->max_rows);
    Picks picks(nw);
    for (int wi = 0; wi < nw; ++wi) picks[wi].assign(wins[wi].n_cur, std::vector<PickOut>(8));
    if (prefill(wins, slot0, picks)) return -1;
    for (int wi = 0; wi < nw; ++wi) wins[wi].no_speech_prob = picks[wi][0][0].no_speech_prob;
    // every decoder of a window starts from the prompt KV of its first
    std::vector<int> copies, release;
    for (int wi = 0; wi < nw; ++wi)
      if (e->pager.remap(slot0[wi], std::vector<int>(wins[wi].n_cur, 0), (int)wins[wi].prompt.size(), copies,
                         release))
        return -1;
    if (engine_copy_pages(e, copies)) return -1;
    e->pager.unref(release);
    const int n_max = m.hp.n_text_ctx / 2 - 4;
    for (int i = 0; i < n_max; ++i) {
      if (aborted()) {
        set_last_error("aborted by callback");
        return -6;
      }
      copies.clear();
      release.clear();
      bool any_active = false;
      for (int wi = 0; wi < nw; ++wi) {
        Window& w = wins[wi];
        if (w.done) continue;
        if (p.strategy == 1) {
          if (select_beams(w, picks[wi], i, slot0[wi], copies, release)) return -1;
        } else {
          for (int j = 0; j < w.n_cur; ++j) {
            Decoder& d = w.dec[j];
            if (d.completed || d.failed) continue;
            const sw_token_data t = to_token(picks[wi][j][0]);
            d.seq.tokens.push_back(t);
            d.seq.sum_logprobs_all += t.plog;
          }
        }
        bool all_done = true;
        for (int j = 0; j < w.n_cur; ++j) {
          Decoder& d = w.dec[j];
          if (d.completed || d.failed) continue;
          update_decoder(w, d, i, n_max);
          if (!d.completed && !d.failed) all_done = false;
        }
        w.done = all_done;
        if (!all_done) any_active = true;
      }
      if (engine_copy_pages(e, copies)) return -1;
      e->pager.unref(release);
      if (!any_active) break;
      if (next_step(wins, slot0, i, picks)) return -1;
    }
    return 0;
  }

  // ---- second half of the token-level timestamps for every segment the windows of a finished batch emitted:
  // token times up, one kernel over the energy that never left the device, token times back (token_times.cu).
  // Called from the post-processing thread of the batch, on the engine's post stream.
  int refine_token_times(std::vector<Window>& ws) {
    size_t n_seg = 0, n_tok = 0;
    for (auto& w : ws)
      for (int si : w.tt_segs) {
        ++n_seg;
        n_tok += utts[w.utt].res->segs[si].tokens.size();
      }
    if (n_seg == 0) return 0;
    SW_CUDA_CHECK(cudaSetDevice(e->device));
    if (n_seg > e->tt_seg_capacity) {
      e->d_tt_seg.release();
      e->h_tt_seg.release();
      e->tt_seg_capacity = n_seg * 2 + 64;
      if (e->d_tt_seg.alloc(e->tt_seg_capacity) || e->h_tt_seg.alloc(e->tt_seg_capacity)) return -1;
    }
    if (n_tok > e->tt_tok_capacity) {
      e->d_tt_t.release();
      e->h_tt_t.release();
      e->d_tt_flag.release();
      e->h_tt_flag.release();
      e->d_tt_thold.release();
      e->tt_tok_capacity = n_tok * 2 + 256;
      if (e->d_tt_t.alloc(2 * e->tt_tok_capacity) || e->h_tt_t.alloc(2 * e->tt_tok_capacity) ||
          e->d_tt_flag.alloc(e->tt_tok_capacity) || e->h_tt_flag.alloc(e->tt_tok_capacity) ||
          e->d_tt_thold.alloc(e->tt_tok_capacity))
        return -1;
    }
    const size_t cap = e->tt_tok_capacity;
    long long *h0 = e->h_tt_t.p, *h1 = e->h_tt_t.p + cap;
    size_t is = 0, it = 0;
    for (auto& w : ws) {
      const Utt& u = utts[w.utt];
      for (int si : w.tt_segs) {
        const sw_segment& sg = u.res->segs[si];
        TtSeg& d = e->h_tt_seg.p[is++];
        d.en_off = u.en_off;
        d.blk_off = u.blk_off;
        d.n_samples = u.n_energy;
        d.tok_off = (int)it;
        d.n_tok = (int)sg.tokens.size();
        for (const sw_token_data& t : sg.tokens) {
          h0[it] = t.t0;
          h1[it] = t.t1;
          e->h_tt_flag.p[it] = t.id < m.vocab.eot ? 1 : 0;
          ++it;
        }
      }
    }
    cudaStream_t ps = e->post_stream;
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_tt_seg.p, e->h_tt_seg.p, n_seg * sizeof(TtSeg), cudaMemcpyHostToDevice, ps));
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_tt_t.p, h0, n_tok * sizeof(long long), cudaMemcpyHostToDevice, ps));
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_tt_t.p + cap, h1, n_tok * sizeof(long long), cudaMemcpyHostToDevice, ps));
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_tt_flag.p, e->h_tt_flag.p, n_tok, cudaMemcpyHostToDevice, ps));
    if (token_time_refine(e->d_energy.p, e->d_eblk.p, e->d_eblk.p + e->eblk_capacity, e->d_tt_seg.p, (int)n_seg,
                          e->d_tt_t.p, e->d_tt_t.p + cap, e->d_tt_flag.p, e->d_tt_thold.p, ps))
      return -1;
    SW_CUDA_CHECK(cudaMemcpyAsync(h0, e->d_tt_t.p, n_tok * sizeof(long long), cudaMemcpyDeviceToHost, ps));
    SW_CUDA_CHECK(cudaMemcpyAsync(h1, e->d_tt_t.p + cap, n_tok * sizeof(long long), cudaMemcpyDeviceToHost, ps));
    SW_CUDA_CHECK(cudaStreamSynchronize(ps));
    it = 0;
    for (auto& w : ws) {
      Utt& u = utts[w.utt];
      for (int si : w.tt_segs)
        for (sw_token_data& t : u.res->segs[si].tokens) {
          t.t0 = h0[it];
          t.t1 = h1[it];
          ++it;
        }
      w.tt_segs.clear();
    }
    tt_launches += 1;
    tt_d2h_bytes += (double)n_tok * 2 * sizeof(long long);
    return 0;
  }
  long tt_launches = 0;      // folded into the engine's counters by the main thread (collect)
  double tt_d2h_bytes = 0;

  // ---- after the decode loop of one window: rank, fallback decision, segments, seek
  // returns true if the window must be re-run at the next temperature
  bool finish_window(Window& w) {
    const Vocab& v = m.vocab;
    Utt& u = utts[w.utt];
    double best_score = -INFINITY;
    int best_id = 0;
    for (int j = 0; j < w.n_cur; ++j) {
      Decoder& d = w.dec[j];
      if (d.failed) continue;
      d.seq.tokens.resize(d.seq.result_len);
      sequence_score(p, d.seq);
      if (d.seq.result_len > 32 && d.seq.entropy < p.entropy_thold) {
        d.failed = true;
        continue;
      }
      if (best_score < d.seq.score) {
        best_score = d.seq.score;
        best_id = j;
      }
    }
    Decoder& bd = w.dec[best_id];
    const bool success =
        !(bd.failed || (bd.seq.avg_logprobs < p.logprob_thold && w.no_speech_prob < p.no_speech_thold));
    if (!success && w.temp_idx + 1 < (int)temps.size()) return true;

    int seek_delta = bd.seek_delta;
    const int result_len = bd.seq.result_len;
    auto& tc = bd.seq.tokens;
    if ((int)tc.size() > result_len) tc.resize(result_len);
    const bool is_no_speech = w.no_speech_prob > p.no_speech_thold && bd.seq.avg_logprobs < p.logprob_thold;
    u.prompt_past.clear();
    if (!w.prompt.empty() && w.prompt.front() == v.prev)
      u.prompt_past.insert(u.prompt_past.end(), w.prompt.begin() + 1, w.prompt.end() - w.n_init);
    for (int i = 0; i < result_len && !is_no_speech; ++i) u.prompt_past.push_back(tc[i].id);

    if (!tc.empty() && !is_no_speech) {
      int i0 = 0;
      int64_t t0 = w.seek + 2 * (tc.front().tid - v.beg);
      std::string text;
      bool turn = false;
      auto emit = [&](int64_t a, int64_t b, int j0, int j1) {
        sw_segment sg;
        sg.t0 = a;
        sg.t1 = b;
        sg.text = text;
        sg.speaker_turn_next = turn;
        sg.tokens.assign(tc.begin() + j0, tc.begin() + j1 + 1);
        if (p.token_timestamps && token_timestamps(m, u, sg)) w.tt_segs.push_back((int)u.res->segs.size());
        u.res->segs.push_back(std::move(sg));
      };
      for (int i = 0; i < (int)tc.size(); ++i) {
        if (tc[i].id < v.eot) text += m.vocab.id_to_token[tc[i].id];
        if (p.tdrz_enable && tc[i].id == v.solm) turn = true;
        if (tc[i].id > v.beg && !p.single_segment) {
          const int64_t t1 = w.seek + 2 * (tc[i].tid - v.beg);
          if (!text.empty()) emit(t0, t1, i0, i);
          text.clear();
          while (i < (int)tc.size() && tc[i].id > v.beg) i++;
          i--;
          t0 = t1;
          i0 = i + 1;
          turn = false;
        }
      }
      if (!text.empty()) emit(t0, w.seek + seek_delta, i0, (int)tc.size() - 1);
    }
    const bool single_ts_end =
        tc.size() > 1 && tc[tc.size() - 2].id < v.beg && tc[tc.size() - 1].id > v.beg;
    if (single_ts_end) seek_delta = std::min(u.seek_end - w.seek, CHUNK_CS);
    u.seek = w.seek + seek_delta;
    return false;
  }

  void make_window(Window& w, const Job& job) {
    const Vocab& v = m.vocab;
    Utt& u = utts[job.utt];
    w.utt = job.utt;
    w.temp_idx = job.temp_idx;
    w.seek = u.seek;
    w.t_cur = temps[job.temp_idx];
    w.n_cur = 1;
    if (p.strategy == 0) {
      if (w.t_cur > 0.0f) w.n_cur = best_of;
    } else {
      w.n_cur = w.t_cur > 0.0f ? best_of : beam;
    }
    w.n_cur = std::max(1, w.n_cur);
    w.prompt.clear();
    if (!u.prompt_past.empty() && w.t_cur < 0.5f) {
      const int n_take = std::min(m.hp.n_text_ctx / 2, (int)u.prompt_past.size());
      w.prompt.push_back(v.prev);
      w.prompt.insert(w.prompt.end(), u.prompt_past.end() - n_take, u.prompt_past.end());
    }
    w.prompt.push_back(v.sot);
    w.n_init = 1;
    if (v.multilingual) {
      w.prompt.push_back(v.sot + 1 + u.lang);
      w.prompt.push_back(p.translate ? v.translate : v.transcribe);
      w.n_init += 2;
    }
    if (p.no_timestamps) {
      w.prompt.push_back(v.not_);
      w.n_init++;
    }
    for (int j = 0; j < 8; ++j) w.dec[j] = Decoder();
    w.done = false;
  }

  // ---- decoders per window and the temperature ladder
  int setup_decoding() {
    beam = p.strategy == 1 ? std::max(1, p.beam_size) : 1;
    best_of = std::max(1, p.best_of);
    if (p.strategy == 1) best_of = std::max(1, p.best_of);  // upstream: used when falling back to t > 0
    // whisper.cpp allows WHISPER_MAX_DECODERS = 8 decoders per window whatever the context was created with;
    // sw_ctx_params.max_beams only sizes the row budget (max_batch * max_beams rows per step): a request with more
    // decoders per window than that runs with fewer windows per device pass
    SW_CHECK(beam <= 8, "beam_size %d exceeds the 8 decoders per window whisper.cpp allows", beam);
    if (p.temperature_inc > 0.0f || p.temperature > 0.0f)
      SW_CHECK(best_of <= 8, "best_of %d exceeds the 8 decoders per window whisper.cpp allows", best_of);
    if (p.temperature_inc > 0.0f)
      for (float t = p.temperature; t < 1.0f + 1e-6f; t += p.temperature_inc) temps.push_back(t);
    else
      temps.push_back(p.temperature);
    return 0;
  }

  // ---- per utterance: its language (given, or detected on its first window), the initial prompt and its first job
  int plan_utterances(int n, const char* const* langs, std::deque<Job>& queue) {
    const Vocab& v = m.vocab;
    // language
    std::vector<int> need;
    for (int i = 0; i < n; ++i) {
      Utt& u = utts[i];
      if (!v.multilingual) {
        u.lang = -1;
        continue;
      }
      const char* lg = langs ? langs[i] : p.language;  // per utterance (sw_full_batch_*_lang) or the call's
      if (!lg || !lg[0] || strcmp(lg, "auto") == 0) {
        need.push_back(i);
      } else {
        u.lang = lang_id(lg);
        SW_CHECK(u.lang >= 0 && u.lang < v.n_langs, "unknown language '%s'", lg);
      }
    }
    if (!need.empty() && detect_languages(need)) return -1;
    // initial prompt
    std::vector<int> init_prompt;
    if (p.prompt_tokens && p.prompt_n_tokens > 0)
      init_prompt.assign(p.prompt_tokens, p.prompt_tokens + p.prompt_n_tokens);
    else if (p.initial_prompt && p.initial_prompt[0])
      init_prompt = tokenize(m, p.initial_prompt);
    for (int t : init_prompt) SW_CHECK(t >= 0 && t < m.hp.n_vocab, "prompt token %d out of range", t);

    for (int i = 0; i < n; ++i) {
      Utt& u = utts[i];
      u.res->lang_id = u.lang;
      u.seek = 0;
      u.seek_end = u.n_len_org;
      u.prompt_past = init_prompt;
      if (u.seek_end < u.seek + 10) continue;  // "input is too short"
      if (u.seek + 100 >= u.seek_end) continue;
      queue.push_back(Job{i, 0});
    }
    return 0;
  }

  int run(const void* const* pcm, const int* n_samples, int n, bool is_f32, sw_result** out,
          const char* const* langs) {
    if (setup_decoding()) return -1;
    for (int i = 0; i < n; ++i) SW_CHECK(n_samples[i] >= 0 && (n_samples[i] == 0 || pcm[i]), "utterance %d: null PCM", i);
    const bool trace = getenv("SW_TRACE") != nullptr;
    const double tf0 = wall_ms();
    if (setup_logit_cfg()) return -1;
    if (front_end(pcm, n_samples, n, is_f32)) return -1;
    if (trace) fprintf(stderr, "[sw trace] front end of %d utterances: %.1f ms (wall)\n", n, wall_ms() - tf0);
    for (int i = 0; i < n; ++i) {
      out[i] = new sw_result();
      utts[i].res = out[i];
    }
    std::deque<Job> queue;
    if (plan_utterances(n, langs, queue)) return -1;
    // Host post-processing of a finished batch (ranking, segments, token-level timestamps) runs on
    // worker threads while the GPU already encodes / decodes the next batch of other utterances.
    struct Pending {
      std::vector<Window> wins;
      std::vector<char> rerun;
      std::thread th;
      std::string error;
      bool active = false, failed = false;
      ~Pending() {
        if (th.joinable()) th.join();
      }
    } pend;
    const int n_workers = std::max(1, std::min(p.n_threads > 0 ? p.n_threads : 4, 64));
    auto start_finish = [&](std::vector<Window>&& ws) {
      pend.wins = std::move(ws);
      pend.rerun.assign(pend.wins.size(), 0);
      pend.active = true;
      pend.th = std::thread([this, &pend, n_workers] {
        std::atomic<int> next{0};
        auto work = [&] {
          try {
            for (;;) {
              const int i = next.fetch_add(1);
              if (i >= (int)pend.wins.size()) break;
              pend.rerun[i] = finish_window(pend.wins[i]) ? 1 : 0;
            }
          } catch (...) {
            pend.failed = true;
          }
        };
        std::vector<std::thread> pool;
        const int nt = std::min<int>(n_workers, (int)pend.wins.size());
        for (int t = 1; t < nt; ++t) pool.emplace_back(work);
        work();
        for (auto& t : pool) t.join();
        if (!pend.failed && refine_token_times(pend.wins)) {
          pend.failed = true;
          pend.error = last_error_string();  // thread-local: hand it to the thread that reports
        }
      });
    };
    auto collect = [&]() -> int {
      if (!pend.active) return 0;
      const double tc0 = wall_ms();
      pend.th.join();
      if (trace) fprintf(stderr, "[sw trace] waited %.1f ms for the host post-processing of %d windows\n", wall_ms() - tc0, (int)pend.wins.size());
      pend.active = false;
      SW_CHECK(!pend.failed, "%s", pend.error.empty() ? "out of host memory while building results" : pend.error.c_str());
      e->times.n_launches += tt_launches;
      e->times.d2h_bytes += tt_d2h_bytes;
      tt_launches = 0;
      tt_d2h_bytes = 0;
      for (size_t i = 0; i < pend.wins.size(); ++i) {
        const Window& w = pend.wins[i];
        const Utt& u = utts[w.utt];
        if (pend.rerun[i]) queue.push_back(Job{w.utt, w.temp_idx + 1});
        else if (u.seek + 100 < u.seek_end) queue.push_back(Job{w.utt, 0});
      }
      return 0;
    };
    std::vector<Window> wins;
    while (true) {
      if (queue.empty()) {
        if (collect()) return -1;
        if (queue.empty()) break;
      }
      if (aborted()) {
        set_last_error("aborted by callback");
        return -6;
      }
      // take jobs while both the window and the decoder-row budgets hold
      wins.clear();
      int rows = 0;
      while (!queue.empty() && (int)wins.size() < e->max_batch) {
        Window w;
        make_window(w, queue.front());
        if (rows + w.n_cur > e->max_rows) break;
        rows += w.n_cur;
        wins.push_back(std::move(w));
        queue.pop_front();
      }
      std::vector<int> wutt, wseek;
      for (auto& w : wins) {
        wutt.push_back(w.utt);
        wseek.push_back(w.seek);
        utts[w.utt].res->n_windows++;
      }
      const double tw0 = wall_ms();
      if (finalize_windows(wutt, wseek)) return -1;
      if (engine_encode(e, (int)wins.size(), nullptr)) return -1;
      const double tw1 = wall_ms();
      const int rc = decode_windows(wins);
      if (rc) return rc;
      const double tw2 = wall_ms();
      if (collect()) return -1;  // at most one batch of host post-processing in flight
      if (trace)
        fprintf(stderr, "[sw trace] batch of %d windows: encode %.1f ms, decode %.1f ms, wait for previous finish %.1f ms (wall)\n",
                (int)wins.size(), tw1 - tw0, tw2 - tw1, wall_ms() - tw2);
      start_finish(std::move(wins));
    }
    if (trace) fprintf(stderr, "[sw trace] run of %d utterances: %.1f ms (wall)\n", n, wall_ms() - tf0);
    return 0;
  }
};

}  // namespace

int run_full_batch(Engine* e, const sw_full_params* params, const void* const* pcm, const int* n_samples,
                   int n, bool is_f32, sw_result** out, const char* const* langs) {
  SW_CHECK(e && params && out && n > 0, "bad arguments");
  std::lock_guard<std::mutex> lk(e->mu);
  SW_CUDA_CHECK(cudaSetDevice(e->device));
  for (int i = 0; i < n; ++i) out[i] = nullptr;
  Run r(e, *params);
  const int rc = r.run(pcm, n_samples, n, is_f32, out, langs);
  if (rc) {
    for (int i = 0; i < n; ++i) {
      delete out[i];
      out[i] = nullptr;
    }
  }
  return rc;
}

int run_full_batch_lanes(sw_ctx* ctx, const sw_full_params* params, const void* const* pcm, const int* n_samples,
                         int n, bool is_f32, sw_result** out, const char* const* langs) {
  SW_CHECK(ctx && ctx->e && params && out && n > 0, "bad arguments");
  const int n_lanes = 1 + (int)ctx->lanes.size();
  if (n_lanes == 1 || n < 2) return run_full_batch(ctx->e, params, pcm, n_samples, n, is_f32, out, langs);
  // deal the utterances: lane k takes every n_lanes-th one, so ragged lengths spread evenly
  struct LaneJob {
    std::vector<const void*> pcm;
    std::vector<const char*> langs;
    std::vector<int> n_samples, index;
    std::vector<sw_result*> out;
    int rc = 0;
    std::string err;
  };
  std::vector<LaneJob> jobs(n_lanes);
  for (int i = 0; i < n; ++i) {
    LaneJob& j = jobs[i % n_lanes];
    j.pcm.push_back(pcm[i]);
    if (langs) j.langs.push_back(langs[i]);
    j.n_samples.push_back(n_samples[i]);
    j.index.push_back(i);
  }
  auto work = [&](int k) {
    LaneJob& j = jobs[k];
    if (j.index.empty()) return;
    j.out.assign(j.index.size(), nullptr);
    Engine* e = k == 0 ? ctx->e : ctx->lanes[k - 1];
    try {
      j.rc = run_full_batch(e, params, j.pcm.data(), j.n_samples.data(), (int)j.index.size(), is_f32, j.out.data(),
                            langs ? j.langs.data() : nullptr);
    } catch (const std::exception& ex) {
      set_last_error("internal error: %s", ex.what());
      j.rc = -1;
    }
    if (j.rc) j.err = last_error_string();  // the error string is thread-local: hand it to the caller
  };
  std::vector<std::thread> th;
  for (int k = 1; k < n_lanes; ++k) th.emplace_back(work, k);
  work(0);
  for (auto& t : th) t.join();
  int rc = 0;
  for (auto& j : jobs)
    if (j.rc && !rc) {
      rc = j.rc;
      set_last_error("%s", j.err.c_str());
    }
  for (int i = 0; i < n; ++i) out[i] = nullptr;
  for (auto& j : jobs)
    for (size_t q = 0; q < j.out.size(); ++q) {
      if (rc) delete j.out[q];
      else out[j.index[q]] = j.out[q];
    }
  return rc;
}

}  // namespace sw
