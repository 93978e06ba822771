// Device pipelines of the engine (see engine.h): buffer setup, conv stem + encoder + cross-KV,
// and one batched decoder step. Host control flow only; every arithmetic op is one of the
// hand-written kernels in this directory (no cuBLAS/cuDNN/torch).
#include "engine.h"

#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <tuple>

#include "common.cuh"
#include "gemm.cuh"

namespace sw {

static void engine_free_step_graphs(Engine* e);

// Programmatic dependent launch of the step kernels: ON unless SW_PDL=0. Round 1 measured it at -7 % inside the
// step graph (154.7 vs 144.1 us per layer, profiles/r1_step_kernel_costs_pdl_*.log): the cross attention released
// its dependents at its START, so the merge, the cross-out GEMM, ... became resident while it streamed for ~85 us
// and held shared memory on the SMs the other lane's chain needs. Since round 2 the cross attention releases them
// only when it ends, and the tcgen05 decoder GEMMs (skinny_gemm_tc.cu) occupy ~50 SMs each, so a dependent's
// prologue and first weight tiles run on free SMs under its predecessor: chain of a layer on the 52 SMs a resident
// cross attention leaves 72 -> 65 us, bench 3 761 -> 3 911 audio-s/s on the same box (profiles/r2_chain_occupied.txt).
bool pdl_enabled() {
  static const bool on = [] {
    const char* p = getenv("SW_PDL");
    return !(p && strcmp(p, "0") == 0);
  }();
  return on;
}

Engine::~Engine() {
  if (ev0) cudaEventDestroy(ev0);
  if (ev1) cudaEventDestroy(ev1);
  for (auto ev : xa_ev)
    if (ev) cudaEventDestroy(ev);
  engine_free_step_graphs(this);
  if (stream) cudaStreamDestroy(stream);
  if (post_stream) cudaStreamDestroy(post_stream);
  if (owns_model) delete model;
}

static int engine_init(Engine* e, const char* path, const sw_ctx_params* p, const Engine* primary) {
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
    cudaGetLastError();
    set_last_error("no CUDA device: this library has no CPU fallback");
    return -1;
  }
  e->device = p ? p->device : 0;
  SW_CHECK(e->device >= 0 && e->device < n_dev, "device %d out of range (%d present)", e->device, n_dev);
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, e->device);
  SW_CHECK(major == 10, "device %d has compute capability %d.x; this build is sm_100a only", e->device, major);
  SW_CUDA_CHECK(cudaSetDevice(e->device));
  e->max_batch = (p && p->max_batch > 0) ? p->max_batch : 64;
  e->max_beams = (p && p->max_beams > 0) ? p->max_beams : 5;
  SW_CHECK(e->max_beams <= 8, "max_beams %d > 8", e->max_beams);
  e->max_rows = std::max(8, e->max_batch * e->max_beams);  // any single window may run 8 decoders
  {
    const char* g = getenv("SW_GRAPHS");  // development switch: SW_GRAPHS=0 launches the step kernel by kernel
    e->use_graphs = !(g && strcmp(g, "0") == 0);
  }
  size_t free0 = 0, total0 = 0;
  if (primary) {
    e->model = primary->model;
    e->owns_model = false;
  } else {
    e->model = load_model(path);
    if (!e->model) return -1;
  }
  cudaMemGetInfo(&free0, &total0);
  SW_CUDA_CHECK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  SW_CUDA_CHECK(cudaStreamCreateWithFlags(&e->post_stream, cudaStreamNonBlocking));
  SW_CUDA_CHECK(cudaEventCreate(&e->ev0));
  SW_CUDA_CHECK(cudaEventCreate(&e->ev1));
  e->xa_ev.assign(2 * (size_t)64, nullptr);
  for (auto& ev : e->xa_ev) SW_CUDA_CHECK(cudaEventCreate(&ev));

  const HParams& hp = e->model->hp;
  const size_t d = hp.n_audio_state, nm = hp.n_mels, B = e->max_batch, R = e->max_rows;
  const size_t M = B * 1500;
  if (e->conv_in.alloc(B * 3002 * nm)) return -1;
  if (e->h1.alloc(B * 3002 * d)) return -1;
  SW_CUDA_CHECK(cudaMemset(e->h1.p, 0, B * 3002 * d * sizeof(bf16)));
  if (e->x.alloc(M * d)) return -1;
  if (e->hb.alloc(M * d)) return -1;
  if (e->qkv.alloc(M * 3 * d)) return -1;
  if (e->ff.alloc(M * 4 * d)) return -1;
  if (e->cross_kv.alloc((size_t)hp.n_text_layer * M * 2 * d)) return -1;
  // decoder
  e->logits_ld = (hp.n_vocab + 3) / 4 * 4;
  if (e->dx.alloc(R * d) || e->dh.alloc(R * d) || e->dqkv.alloc(R * 3 * d) || e->datt.alloc(R * d) ||
      e->dq.alloc(R * d) || e->dff.alloc(R * 4 * d) || e->logits.alloc(R * e->logits_ld) ||
      e->xa_ws.alloc(cross_attention_ws_floats((int)R, (int)d, hp.n_text_head)) || e->dpart.alloc(32 * R * d))
    return -1;
  e->n_pages = (int)(R * KV_MAX_PAGES + R);
  const size_t page_elems = (size_t)hp.n_text_layer * 2 * KV_PAGE * d;
  if (e->kv_pool.alloc((size_t)e->n_pages * page_elems)) return -1;
  if (e->d_tok.alloc(R) || e->d_pos.alloc(R) ||
      e->d_grp_win.alloc(R) || e->d_grp_start.alloc(R) || e->d_grp_count.alloc(R) || e->d_rows.alloc(R) ||
      e->d_lrows.alloc(R) || e->d_picks.alloc(R * 8) || e->d_suppress.alloc(hp.n_vocab) ||
      e->d_copy_pairs.alloc(2 * R))
    return -1;
  if (e->h_tok.alloc(R) || e->h_pos.alloc(R) || e->h_grp.alloc(3 * R) || e->h_rows.alloc(R) ||
      e->h_lrows.alloc(R) || e->h_picks.alloc(R * 8))
    return -1;
  SW_CUDA_CHECK(cudaDeviceSynchronize());
  {
    size_t free1 = 0, total1 = 0;
    cudaMemGetInfo(&free1, &total1);
    e->buffer_bytes = free0 > free1 ? free0 - free1 : 0;
  }
  if (!primary)
    log_msg(2, "model loaded: d=%d layers=%d/%d n_mels=%d n_vocab=%d; max_batch=%d max_beams=%d",
          hp.n_audio_state, hp.n_audio_layer, hp.n_text_layer, hp.n_mels, hp.n_vocab, e->max_batch,
          e->max_beams);
  return 0;
}

Engine* engine_create(const char* model_path, const sw_ctx_params* params) {
  Engine* e = new Engine();
  if (engine_init(e, model_path, params, nullptr)) {
    delete e;
    return nullptr;
  }
  return e;
}

Engine* engine_create_lane(const Engine* primary) {
  sw_ctx_params p;
  memset(&p, 0, sizeof(p));
  p.device = primary->device;
  p.max_batch = primary->max_batch;
  p.max_beams = primary->max_beams;
  Engine* e = new Engine();
  if (engine_init(e, nullptr, &p, primary)) {
    delete e;
    return nullptr;
  }
  return e;
}

// kernel timing (bench roofline) brackets the cross attention of every 8th layer only: an event node between two
// kernels turns their programmatic edge into a full dependency
static constexpr int XA_TIMED_EVERY = 8;

#define GEMM(args)                                   \
  do {                                               \
    if (gemm_bf16_tn(args, e->stream)) return -1;    \
    e->times.n_launches++;                           \
  } while (0)

int engine_encode(Engine* e, int n_win, float* enc_out_f32) {
  const Model& m = *e->model;
  const HParams& hp = m.hp;
  const int d = hp.n_audio_state, nm = hp.n_mels;
  const int64_t M = (int64_t)n_win * 1500;
  SW_CHECK(n_win > 0 && n_win <= e->max_batch, "encode: %d windows exceed max_batch %d", n_win, e->max_batch);
  cudaStream_t st = e->stream;
  SW_CUDA_CHECK(cudaEventRecord(e->ev0, st));
  {  // conv1 (k=3, s=1, p=1) as an implicit GEMM over overlapping rows of the padded input, + GELU
    GemmArgs a;
    a.A = e->conv_in.p; a.lda = nm; a.a_batch_stride = (int64_t)3002 * nm;
    a.B = m.conv1_w; a.ldb = 3 * nm;
    a.C = e->h1.p + d; a.ldc = d; a.c_batch_stride = (int64_t)3002 * d;
    a.bias = m.conv1_b;
    a.M = 3000; a.N = d; a.K = 3 * nm; a.batch = n_win;
    a.flags = GEMM_GELU;
    GEMM(a);
  }
  {  // conv2 (k=3, s=2, p=1) + GELU + positional embedding -> residual stream x (f32)
    GemmArgs a;
    a.A = e->h1.p; a.lda = 2 * d; a.a_batch_stride = (int64_t)3002 * d;
    a.B = m.conv2_w; a.ldb = 3 * d;
    a.C = e->x.p; a.ldc = d; a.c_batch_stride = (int64_t)1500 * d;
    a.bias = m.conv2_b;
    a.residual = m.enc_pos; a.ldr = d; a.r_batch_stride = 0; a.res_mod = 1500;
    a.M = 1500; a.N = d; a.K = 3 * d; a.batch = n_win;
    a.flags = GEMM_GELU | GEMM_OUT_F32;
    GEMM(a);
  }
  for (int l = 0; l < hp.n_audio_layer; ++l) {
    const EncLayerW& w = m.enc[l];
    if (layer_norm(e->x.p, (int)M, d, w.ln1.g, w.ln1.b, e->hb.p, nullptr, nullptr, 0, 0, nullptr, st)) return -1;
    {
      GemmArgs a;
      a.A = e->hb.p; a.lda = d; a.B = w.wqkv; a.ldb = d; a.C = e->qkv.p; a.ldc = 3 * d;
      a.bias = w.bqkv; a.M = (int)M; a.N = 3 * d; a.K = d;
      GEMM(a);
    }
    if (encoder_attention_tc(e->qkv.p, e->hb.p, n_win, 1500, d, hp.n_audio_head, st)) return -1;
    {
      GemmArgs a;
      a.A = e->hb.p; a.lda = d; a.B = w.wo; a.ldb = d; a.C = e->x.p; a.ldc = d;
      a.bias = w.bo; a.residual = e->x.p; a.ldr = d; a.M = (int)M; a.N = d; a.K = d;
      a.flags = GEMM_OUT_F32;
      GEMM(a);
    }
    if (layer_norm(e->x.p, (int)M, d, w.ln2.g, w.ln2.b, e->hb.p, nullptr, nullptr, 0, 0, nullptr, st)) return -1;
    {
      GemmArgs a;
      a.A = e->hb.p; a.lda = d; a.B = w.w1; a.ldb = d; a.C = e->ff.p; a.ldc = 4 * d;
      a.bias = w.b1; a.M = (int)M; a.N = 4 * d; a.K = d; a.flags = GEMM_GELU;
      GEMM(a);
    }
    {
      GemmArgs a;
      a.A = e->ff.p; a.lda = 4 * d; a.B = w.w2; a.ldb = 4 * d; a.C = e->x.p; a.ldc = d;
      a.bias = w.b2; a.residual = e->x.p; a.ldr = d; a.M = (int)M; a.N = d; a.K = 4 * d;
      a.flags = GEMM_OUT_F32;
      GEMM(a);
    }
    e->times.n_launches += 3;
  }
  if (layer_norm(e->x.p, (int)M, d, m.ln_post.g, m.ln_post.b, e->hb.p, enc_out_f32, nullptr, 0, 0, nullptr, st))
    return -1;
  e->times.n_launches++;
  const int64_t layer_stride = (int64_t)e->max_batch * 1500 * 2 * d;
  for (int l = 0; l < hp.n_text_layer; ++l) {
    const DecLayerW& w = m.dec[l];
    GemmArgs a;
    a.A = e->hb.p; a.lda = d; a.B = w.wxkv; a.ldb = d; a.C = e->cross_kv.p + l * layer_stride; a.ldc = 2 * d;
    a.bias = w.bxkv; a.M = (int)M; a.N = 2 * d; a.K = d;
    GEMM(a);
  }
  SW_CUDA_CHECK(cudaEventRecord(e->ev1, st));
  SW_CUDA_CHECK(cudaEventSynchronize(e->ev1));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->times.ms_encode += ms;
  e->times.n_windows += n_win;
  return 0;
}

int engine_copy_pages(Engine* e, const std::vector<int>& pairs) {
  const HParams& hp = e->model->hp;
  const int64_t page_elems = (int64_t)hp.n_text_layer * 2 * KV_PAGE * hp.n_text_state;
  // in chunks of what d_copy_pairs holds; each chunk completes before the next overwrites the buffer
  for (size_t c0 = 0; c0 < pairs.size(); c0 += e->d_copy_pairs.n) {
    const size_t n = std::min(e->d_copy_pairs.n, pairs.size() - c0);
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_copy_pairs.p, pairs.data() + c0, n * sizeof(int), cudaMemcpyHostToDevice,
                                  e->stream));
    if (kv_copy_pages(e->kv_pool.p, e->d_copy_pairs.p, (int)n / 2, page_elems, e->stream)) return -1;
    e->times.n_launches++;
    SW_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  }
  return 0;
}

// Everything one decoder step puts on the stream (uploads, kernels, pick read-back). `launches`
// counts kernels; `capturing` selects graph-safe event records for the kernel-timing probes.
static int enqueue_decode_step(Engine* e, const StepRows& step, bool want_logits, int n_lrows, const LogitCfg& cfg,
                               bool capturing, long* launches) {
  const int R = step.R, n_groups = step.G, max_count = step.max_count;
  const Model& m = *e->model;
  const HParams& hp = m.hp;
  const int d = hp.n_text_state, L = hp.n_text_layer;
  cudaStream_t st = e->stream;
  const unsigned ev_flags = capturing ? cudaEventRecordExternal : cudaEventRecordDefault;
  SW_CUDA_CHECK(cudaMemcpyAsync(e->d_rows.p, e->h_rows.p, R * sizeof(DecRow), cudaMemcpyHostToDevice, st));
  SW_CUDA_CHECK(cudaMemcpyAsync(e->d_tok.p, e->h_tok.p, R * sizeof(int), cudaMemcpyHostToDevice, st));
  SW_CUDA_CHECK(cudaMemcpyAsync(e->d_pos.p, e->h_pos.p, R * sizeof(int), cudaMemcpyHostToDevice, st));
  SW_CUDA_CHECK(cudaMemcpyAsync(e->d_grp_win.p, e->h_grp.p, n_groups * sizeof(int), cudaMemcpyHostToDevice, st));
  SW_CUDA_CHECK(cudaMemcpyAsync(e->d_grp_start.p, e->h_grp.p + e->max_rows, n_groups * sizeof(int), cudaMemcpyHostToDevice, st));
  SW_CUDA_CHECK(cudaMemcpyAsync(e->d_grp_count.p, e->h_grp.p + 2 * e->max_rows, n_groups * sizeof(int), cudaMemcpyHostToDevice, st));
  if (n_lrows > 0)  // up front, so that nothing but kernels sits between the step's kernels (PDL chain)
    SW_CUDA_CHECK(cudaMemcpyAsync(e->d_lrows.p, e->h_lrows.p, n_lrows * sizeof(LogitRow), cudaMemcpyHostToDevice, st));
  if (embed_tokens(m.tok_emb, m.dec_pos, e->d_tok.p, e->d_pos.p, R, d, e->dx.p, st)) return -1;
  const int64_t layer_stride = (int64_t)e->max_batch * 1500 * 2 * d;
  // Weight-streaming GEMMs (skinny_gemm.cu). Projections that feed the residual stream or the
  // cross-attention query are split along K; their f32 partial sums are folded in by the consumer
  // (the fused LayerNorm adds bias + partials into x; cross_attention reduces its query on load).
  const int sp_d = skinny_split_for(d, d), sp_ff = skinny_split_for(d, 4 * d);
  const int64_t ps = (int64_t)R * d;  // stride between the K slices of the partial sums
  float* part = e->dpart.p;
  const float* pend_bias = nullptr;  // bias of the FC2 partials still to be folded into x
  int pend_split = 0;
  // development switch: SW_SKIP=<bitmask> leaves kernels out of the step (results are garbage) so that
  // the in-graph cost of each one can be read off as a time difference (tools/dev_step_time.py)
  static const int skip = getenv("SW_SKIP") ? atoi(getenv("SW_SKIP")) : 0;
#define STEP_K(bit, call)                    \
  do {                                       \
    if (!(skip & (bit))) {                   \
      if (call) return -1;                   \
      ++*launches;                           \
    }                                        \
  } while (0)
  for (int l = 0; l < L; ++l) {
    const DecLayerW& w = m.dec[l];
    STEP_K(1, layer_norm(e->dx.p, R, d, w.ln1.g, w.ln1.b, e->dh.p, nullptr, pend_split ? part : nullptr, pend_split, ps,
                         pend_bias, st));
    STEP_K(2, skinny_gemm(e->dh.p, d, w.wqkv, R, 3 * d, d, w.bqkv, 0, e->dqkv.p, 3 * d, nullptr, 1, st));
    STEP_K(4, self_attention(e->dqkv.p, e->d_rows.p, R, d, hp.n_text_head, e->kv_pool.p, l, L, e->datt.p, st));
    STEP_K(8, skinny_gemm(e->datt.p, d, w.wo, R, d, d, nullptr, 0, nullptr, 0, part, sp_d, st));
    STEP_K(1, layer_norm(e->dx.p, R, d, w.lnx.g, w.lnx.b, e->dh.p, nullptr, part, sp_d, ps, w.bo, st));
    STEP_K(16, skinny_gemm(e->dh.p, d, w.wxq, R, d, d, nullptr, 0, nullptr, 0, part, sp_d, st));
    STEP_K(32, reduce_partials(part, sp_d, ps, R, d, w.bxq, e->dq.p, st));
    const bool timed = e->kernel_timing && l % XA_TIMED_EVERY == 0;
    if (timed) SW_CUDA_CHECK(cudaEventRecordWithFlags(e->xa_ev[2 * l], st, ev_flags));
    if (!(skip & 64)) {
      if (cross_attention(e->dq.p, e->cross_kv.p + l * layer_stride, (int64_t)e->max_batch * 1500, e->d_grp_win.p,
                          e->d_grp_start.p, e->d_grp_count.p, n_groups, max_count, R, 1500, d, hp.n_text_head,
                          e->xa_ws.p, e->datt.p, st, timed ? e->xa_ev[2 * l + 1] : nullptr, ev_flags, e->xa_max_ctas))
        return -1;
      *launches += 2;
    } else if (timed) {
      SW_CUDA_CHECK(cudaEventRecordWithFlags(e->xa_ev[2 * l + 1], st, ev_flags));
    }
    STEP_K(256, skinny_gemm(e->datt.p, d, w.wxo, R, d, d, nullptr, 0, nullptr, 0, part, sp_d, st));
    STEP_K(1, layer_norm(e->dx.p, R, d, w.ln2.g, w.ln2.b, e->dh.p, nullptr, part, sp_d, ps, w.bxo, st));
    STEP_K(512, skinny_gemm(e->dh.p, d, w.w1, R, 4 * d, d, w.b1, 1, e->dff.p, 4 * d, nullptr, 1, st));
    STEP_K(1024, skinny_gemm(e->dff.p, 4 * d, w.w2, R, d, 4 * d, nullptr, 0, nullptr, 0, part, sp_ff, st));
    pend_bias = w.b2;
    pend_split = sp_ff;
  }
#undef STEP_K
  (*launches) += 1;
  if (want_logits || n_lrows > 0) {  // the final LayerNorm folds the last FC2 partials in
    if (layer_norm(e->dx.p, R, d, m.dec_ln.g, m.dec_ln.b, e->dh.p, nullptr, pend_split ? part : nullptr, pend_split,
                   ps, pend_bias, st))
      return -1;
    (*launches) += 1;
    GemmArgs a;
    a.A = e->dh.p; a.lda = d; a.B = m.tok_emb; a.ldb = d; a.C = e->logits.p; a.ldc = e->logits_ld;
    a.M = R; a.N = hp.n_vocab; a.K = d; a.flags = GEMM_OUT_F32;
    if (gemm_bf16_tn(a, st)) return -1;
    (*launches) += 1;
  }
  if (n_lrows > 0) {
    if (process_logits_pick(e->logits.p, e->logits_ld, e->d_lrows.p, n_lrows, cfg, e->d_picks.p, st)) return -1;
    SW_CUDA_CHECK(cudaMemcpyAsync(e->h_picks.p, e->d_picks.p, (size_t)n_lrows * 8 * sizeof(PickOut),
                                  cudaMemcpyDeviceToHost, st));
    (*launches) += 1;
  }
  return 0;
}

// Everything that shapes the captured launch sequence OR is passed to a kernel BY VALUE: a graph replays
// the arguments it was captured with, so the by-value members of LogitCfg (sw_full_params.suppress_blank,
// .max_initial_ts) are part of the key. Pointers (d_suppress, the row descriptors) are fixed per lane and
// their contents are refreshed per run / per step.
struct StepKey {
  int R, G, max_count, want_logits, n_lrows, timing, suppress_blank, max_initial_ts_id;
  bool operator<(const StepKey& o) const {
    return std::tie(R, G, max_count, want_logits, n_lrows, timing, suppress_blank, max_initial_ts_id) <
           std::tie(o.R, o.G, o.max_count, o.want_logits, o.n_lrows, o.timing, o.suppress_blank, o.max_initial_ts_id);
  }
};
struct StepGraph {
  cudaGraphExec_t exec = nullptr;
  long launches = 0;
};
struct StepGraphCache {
  std::map<StepKey, StepGraph> graphs;
  ~StepGraphCache() {
    for (auto& kv : graphs)
      if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  }
};

static void engine_free_step_graphs(Engine* e) {
  delete static_cast<StepGraphCache*>(e->step_graphs);
  e->step_graphs = nullptr;
}

int engine_decode_step(Engine* e, const StepRows& step, bool want_logits, int n_lrows, const LogitCfg& cfg) {
  const HParams& hp = e->model->hp;
  const int d = hp.n_text_state, L = hp.n_text_layer, R = step.R;
  SW_CHECK(R > 0 && R <= e->max_rows, "decode step with %d rows (max %d)", R, e->max_rows);
  cudaStream_t st = e->stream;
  for (int r = 0; r < R; ++r) e->pager.fill(e->h_rows.p[r].slot, e->h_rows.p[r].pages);
  if (!e->use_graphs) {
    SW_CUDA_CHECK(cudaEventRecord(e->ev0, st));
    long launches = 0;
    if (enqueue_decode_step(e, step, want_logits, n_lrows, cfg, false, &launches)) return -1;
    e->times.n_launches += launches;
  } else {
    // The step is a fixed launch sequence for a given shape: capture it once per shape and replay
    // it (one host call per step instead of ~460, and no inter-kernel launch gaps).
    if (!e->step_graphs) e->step_graphs = new StepGraphCache();
    StepGraphCache& cache = *static_cast<StepGraphCache*>(e->step_graphs);
    const StepKey key{R, step.G, step.max_count, want_logits ? 1 : 0, n_lrows, e->kernel_timing ? 1 : 0,
                      cfg.suppress_blank, cfg.max_initial_ts_id};
    auto it = cache.graphs.find(key);
    if (it == cache.graphs.end()) {
      if (cache.graphs.size() > 512) {  // bounded: drop everything and start over
        for (auto& kv : cache.graphs) cudaGraphExecDestroy(kv.second.exec);
        cache.graphs.clear();
      }
      StepGraph g;
      SW_CUDA_CHECK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      const int rc = enqueue_decode_step(e, step, want_logits, n_lrows, cfg, true, &g.launches);
      cudaGraph_t graph = nullptr;
      const cudaError_t ce = cudaStreamEndCapture(st, &graph);
      if (rc || ce != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        if (!rc) set_last_error("decode step graph capture failed: %s", cudaGetErrorString(ce));
        cudaGetLastError();
        return -1;
      }
      const cudaError_t ie = cudaGraphInstantiate(&g.exec, graph, 0);
      cudaGraphDestroy(graph);
      SW_CHECK(ie == cudaSuccess, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ie));
      it = cache.graphs.emplace(key, g).first;
    }
    SW_CUDA_CHECK(cudaEventRecord(e->ev0, st));
    SW_CUDA_CHECK(cudaGraphLaunch(it->second.exec, st));
    e->times.n_launches += it->second.launches;
  }
  SW_CUDA_CHECK(cudaEventRecord(e->ev1, st));
  SW_CUDA_CHECK(cudaEventSynchronize(e->ev1));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->times.ms_decode += ms;
  e->times.n_steps++;
  if (n_lrows > 0) e->times.d2h_bytes += (double)n_lrows * 8 * sizeof(PickOut);
  if (e->kernel_timing) {
    int n_timed = 0;
    for (int l = 0; l < L; l += XA_TIMED_EVERY, ++n_timed) {
      float t = 0;
      cudaEventElapsedTime(&t, e->xa_ev[2 * l], e->xa_ev[2 * l + 1]);
      e->times.ms_xattn += t;
    }
    e->times.n_xattn += n_timed;
    // per launch: the cross-KV of every active window once + q in + attention out
    e->times.xattn_bytes += (double)n_timed * ((double)step.G * 1500 * 2 * d * 2 + (double)R * d * 4);
  }
  return 0;
}

}  // namespace sw
