// Engine context behind the C ABI: model in HBM, activation/KV buffers sized for max_batch
// windows, and the device pipelines (front end, encoder, one batched decoder step).
// The host sequencer (sequencer.cpp) drives them; capi.cpp exposes them.
#pragma once
#include <stdint.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/sw_whisper.h"
#include "host_common.h"
#include "kernels.cuh"
#include "kv_pager.h"
#include "model.h"

namespace sw {

struct StageTimes {  // accumulated device time per stage (CUDA events), for the benchmark
  double ms_mel = 0, ms_encode = 0, ms_decode = 0;
  long n_windows = 0, n_steps = 0, n_launches = 0;
  double h2d_bytes = 0, d2h_bytes = 0;  // PCM in, picks / energy out
  double ms_xattn = 0;        // device time inside cross_attention launches (kernel timing on)
  long n_xattn = 0;
  double xattn_bytes = 0;     // algorithmic bytes of those launches (cross-KV of the active windows)
  double decode_bytes = 0;  // algorithmic bytes streamed by the decode steps (weights + cross-KV + self-KV)
};

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  int alloc(size_t count) {
    n = count;
    SW_CUDA_CHECK(cudaMalloc(&p, count * sizeof(T)));
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  ~DevBuf() { release(); }
};
template <typename T>
struct PinBuf {
  T* p = nullptr;
  size_t n = 0;
  int alloc(size_t count) {
    n = count;
    SW_CUDA_CHECK(cudaMallocHost(&p, count * sizeof(T)));
    return 0;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    n = 0;
  }
  ~PinBuf() { release(); }
};

struct Engine {
  int device = 0;
  int max_batch = 64, max_beams = 5, max_rows = 320;
  Model* model = nullptr;
  bool owns_model = true;   // false for the further lanes of a context (they share lane 0's weights)
  int xa_max_ctas = 0;      // cap on the persistent cross-attention grid (0 = every SM); contexts with
                            // several lanes leave SMs to the other lane's latency-bound kernels
  size_t buffer_bytes = 0;  // device memory of this lane's buffers (without the weights)
  cudaStream_t stream = nullptr;
  std::mutex mu;  // one batch in flight per context

  // ---- front end
  DevBuf<uint8_t> d_pcm;        // batch PCM (int16 or f32)
  size_t pcm_capacity = 0;
  DevBuf<float> d_log;          // log-mel before normalisation, all utterances of the batch
  size_t log_capacity = 0;
  DevBuf<MelUtt> d_utts;
  DevBuf<unsigned> d_max_enc;
  DevBuf<int> d_win_utt, d_win_seek;
  DevBuf<float> d_energy;       // token-timestamp signal energy, same offsets as the PCM; never leaves HBM
  DevBuf<float> d_eblk;         // per 256-sample block min | max of the energy (two halves)
  size_t eblk_capacity = 0;
  size_t energy_capacity = 0;
  // token-time refinement of a finished batch (token_times.cu), on its own stream: it runs from the host
  // thread that post-processes batch i while the main stream already decodes batch i + 1
  cudaStream_t post_stream = nullptr;
  DevBuf<TtSeg> d_tt_seg;
  PinBuf<TtSeg> h_tt_seg;
  DevBuf<long long> d_tt_t;     // t0 | t1 (two halves of tt_tok_capacity)
  PinBuf<long long> h_tt_t;
  DevBuf<uint8_t> d_tt_flag;
  PinBuf<uint8_t> h_tt_flag;
  DevBuf<float> d_tt_thold;
  size_t tt_seg_capacity = 0, tt_tok_capacity = 0;
  int utt_capacity = 0;
  // ---- encoder activations (max_batch windows)
  DevBuf<bf16> conv_in, h1, hb, qkv, ff;
  DevBuf<float> x;
  DevBuf<bf16> cross_kv;        // [n_text_layer][max_batch*1500][2d]
  // ---- decoder
  DevBuf<float> dx, logits, xa_ws, dpart;  // dpart: split-K partial sums [split][R][d]
  DevBuf<bf16> dh, dqkv, datt, dq, dff;
  DevBuf<bf16> kv_pool;
  int n_pages = 0;
  KvPager pager;                // which kv_pool pages each self-KV slot holds
  DevBuf<int> d_tok, d_pos, d_grp_win, d_grp_start, d_grp_count;
  DevBuf<DecRow> d_rows;
  DevBuf<LogitRow> d_lrows;
  DevBuf<PickOut> d_picks;
  DevBuf<uint8_t> d_suppress;
  DevBuf<int> d_copy_pairs;
  PinBuf<int> h_tok, h_pos, h_grp;  // step rows: written through StepRows only
  PinBuf<DecRow> h_rows;
  PinBuf<LogitRow> h_lrows;
  PinBuf<PickOut> h_picks;
  int64_t logits_ld = 0;

  StageTimes times;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool use_graphs = true;       // replay each decoder step from a CUDA graph captured per step shape
  void* step_graphs = nullptr;  // StepGraphCache (engine.cu)
  bool kernel_timing = false;   // bracket each cross_attention launch with events (bench roofline)
  std::vector<cudaEvent_t> xa_ev;

  ~Engine();
};

Engine* engine_create(const char* model_path, const sw_ctx_params* params);
// a further lane next to `primary`: same model (shared, not owned), same limits, own buffers and stream
Engine* engine_create_lane(const Engine* primary);

// conv stem + encoder stack + ln_post + cross-KV for n_win windows whose conv input is in conv_in.
// enc_out_f32 (device, [n_win*1500][d]) may be null.
int engine_encode(Engine* e, int n_win, float* enc_out_f32);

// The rows of one decoder step, grouped by window, in the engine's pinned step buffers: per row h_rows, h_tok and
// h_pos; per group h_grp = window | first row | row count, at stride max_rows. The rows of a group are added
// between open(win) and close(); engine_decode_step fills their page lists from e->pager.
struct StepRows {
  Engine* e;
  int R = 0, G = 0, max_count = 0;  // rows, groups, most rows in one group
  explicit StepRows(Engine* eng) : e(eng) {}
  void open(int win) {
    e->h_grp.p[G] = win;
    e->h_grp.p[e->max_rows + G] = R;
  }
  // the row of `slot` at position pos; positions pos0..pos of the slot are rows of this step. Returns its index.
  int add(int slot, int pos, int pos0, int token) {
    e->h_rows.p[R] = DecRow{slot, pos, e->h_grp.p[G], pos0};
    e->h_tok.p[R] = token;
    e->h_pos.p[R] = pos;
    return R++;
  }
  void close() {
    const int n = R - e->h_grp.p[e->max_rows + G];
    e->h_grp.p[2 * e->max_rows + G++] = n;
    max_count = std::max(max_count, n);
  }
};

// one decoder step over the rows of `step`.
// want_logits: final LN + logits GEMM for all rows (e->logits). If n_lrows > 0, h_lrows[0..n_lrows) are
// processed into h_picks. Synchronises the stream before returning so the host can read them.
int engine_decode_step(Engine* e, const StepRows& step, bool want_logits, int n_lrows, const LogitCfg& cfg);
// device-side copies of whole KV pages: pairs [src0, dst0, src1, dst1, ...], any number of them
int engine_copy_pages(Engine* e, const std::vector<int>& pairs);

}  // namespace sw
