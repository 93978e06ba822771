// Host-side launchers of the hand-written sm_100a kernels of the Whisper hot path
// (everything whisper_full_with_state does on the device; reference call site
// /root/reference/src/stt_engine.cpp:245-246). All launchers enqueue on `stream`
// and return 0 or -1 (sw_last_error()).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sw {

typedef __nv_bfloat16 bf16;

// ------------------------------------------------------------------ front end (mel.cu)
constexpr int MEL_N_FFT = 400;
constexpr int MEL_HOP = 160;
constexpr int MEL_N_BINS = 201;
constexpr int MEL_WIN_FRAMES = 3000;

struct MelUtt {            // one utterance, device-side descriptor
  int64_t pcm_off;         // element offset of its PCM in the batch PCM buffer
  int n_samples;           //
  int n_active;            // frames that see audio: min(n_eff/160 + 1, n_len)
  int n_len;               // frames incl. the 30 s zero pad
  int blk_off;             // offset of its 256-sample blocks in the energy block-min / block-max arrays
  int64_t log_off;         // element offset of its [n_mel][n_active] log-mel in the log buffer
};
// log10 mel power of every active frame (before clamp/normalise) + per-utterance max.
// pcm is int16 (is_f32 = 0, scaled by 1/32768 in-register) or f32.
// d_filter_span[m] = {first bin rounded down to a multiple of 4, one past the last bin} with a non-zero weight
int mel_log_power(const void* pcm, int is_f32, const MelUtt* d_utts, int n_utts, int max_active,
                  const float* d_filters, const int2* d_filter_span, int n_mel, float* d_log,
                  unsigned* d_max_enc, cudaStream_t stream);
// clamp to max-8, (x+4)/4; window w reads utterance win_utt[w] at frame win_seek[w].
//   out_bf16: [n_win][3002][n_mel] time-major, rows 0 and 3001 zero (conv1's implicit-GEMM input)
//   out_f32 : [n_win][n_mel][3000] mel-major (may be null)
int mel_finalize_windows(const float* d_log, const MelUtt* d_utts, const unsigned* d_max_enc,
                         const int* d_win_utt, const int* d_win_seek, int n_win, int n_mel,
                         bf16* out_bf16, float* out_f32, cudaStream_t stream);
// whole-utterance normalised mel [n_mel][n_len] f32 (the sw_mel_* hooks)
int mel_finalize_full(const float* d_log, const MelUtt* d_utts, const unsigned* d_max_enc, int utt,
                      int n_mel, int n_len, int n_active, float* out, cudaStream_t stream);
// host mel [n_win][n_mel][3000] f32 -> conv1 input layout (the sw_encode hook)
int mel_f32_to_conv_input(const float* d_mel, int n_win, int n_mel, bf16* out, cudaStream_t stream);
// get_signal_energy (token-level timestamps) for every utterance of the batch:
// out[pcm_off + i] = sum_{|j|<=hw} |x[i+j]| / (2hw+1), summed in upstream's order (bit-exact)
// blk_min / blk_max [blk_off + b]: min / max of out over samples [256 b, 256 b + 256) of the utterance, so
// that the host's threshold scans (whisper_exp_compute_token_level_timestamps) can step over whole blocks
int signal_energy(const void* pcm, int is_f32, const MelUtt* d_utts, int n_utts, int max_n, int hw,
                  float* out, float* blk_min, float* blk_max, cudaStream_t stream);

// ------------------------------------------------------------------ token-level timestamps (token_times.cu)
struct TtSeg {            // one result segment whose tokens' [t0, t1] are refined on the signal energy
  long long en_off;       // element offset of its utterance in the energy buffer (= MelUtt::pcm_off)
  int blk_off;            // offset of the utterance's 256-sample blocks in the block min / max arrays
  int n_samples;          // samples of the utterance
  int tok_off;            // first token of the segment in the token arrays
  int n_tok;              // its tokens (text and others; only text tokens are refined)
};
static_assert(sizeof(TtSeg) == 24, "TtSeg is uploaded as is");
// t0 / t1: centiseconds, in and out; is_text: token id < eot; thold: scratch, one float per token
int token_time_refine(const float* d_energy, const float* d_blk_min, const float* d_blk_max, const TtSeg* d_segs,
                      int n_segs, long long* d_t0, long long* d_t1, const uint8_t* d_is_text, float* d_thold,
                      cudaStream_t stream);

// ------------------------------------------------------------------ elementwise (elementwise.cu)
// y = LN(x) * g + b over rows of d (eps 1e-5, f32 statistics). out_bf16/out_f32 may be null.
// If partial != null: x += bias + sum_{s<n_split} partial[s][row][:] first (split-K reduce + residual).
int layer_norm(float* x, int rows, int d, const float* g, const float* b, bf16* out_bf16,
               float* out_f32, const float* partial, int n_split, int64_t split_stride,
               const float* add_bias, cudaStream_t stream);
// out[r][:] = bf16(bias + sum_s partial[s][r][:])
int reduce_partials(const float* partial, int n_split, int64_t split_stride, int rows, int d,
                    const float* bias, bf16* out, cudaStream_t stream);
// zero the pad rows (0 and 3001) of a [n_win][3002][d] bf16 buffer
int zero_conv_pad_rows(bf16* buf, int n_win, int d, cudaStream_t stream);
// x[r][:] = tok_emb[tok[r]][:] + pos_emb[pos[r]][:]
int embed_tokens(const bf16* tok_emb, const float* pos_emb, const int* d_tok, const int* d_pos,
                 int rows, int d, float* x, cudaStream_t stream);
int convert_f16_to_bf16(const uint16_t* src, bf16* dst, int64_t n, cudaStream_t stream);
int convert_f32_to_bf16(const float* src, bf16* dst, int64_t n, cudaStream_t stream);

// ------------------------------------------------------------------ encoder attention (attn_enc_tc.cu)
// non-causal MHA over T keys per (window, head); qkv [n_win*T][3d] bf16 (Q | K | V), out [n_win*T][d].
// tcgen05 / TMEM / TMA flash attention
int encoder_attention_tc(const bf16* qkv, bf16* out, int n_win, int T, int d, int n_head,
                         cudaStream_t stream);

// ------------------------------------------------------------------ decoder (decode.cu)
constexpr int KV_PAGE = 32;       // tokens per self-KV page
constexpr int KV_MAX_PAGES = 14;  // 448 / 32

struct DecRow {    // one decoder row of a step
  int slot;        // self-KV slot (whose page list the pager keeps)
  int pos;         // position of this token
  int win;         // window index into the cross-KV batch
  int pos0;        // first position of this slot whose K/V is produced in this very step: positions
                   // pos0..pos come from rows r-(pos-pos0)..r of the step (contiguous), older ones from the cache
  int pages[KV_MAX_PAGES];  // the slot's page list (filled by engine_decode_step from the host pager):
                            // the attention kernel needs no second dependent lookup
  int pad[2];
};
static_assert(sizeof(MelUtt) == 32, "MelUtt is uploaded as is");
static_assert(sizeof(DecRow) == 80, "DecRow is uploaded as 20 ints");
// pool layout: [page][layer][2][KV_PAGE][d]
// pool[dst page] = pool[src page] for n pairs (src, dst); page_elems bf16 elements per page
int kv_copy_pages(bf16* pool, const int* d_pairs, int n, int64_t page_elems, cudaStream_t stream);
// causal self attention of each row over cache[slot][0..pos0) + the K/V this step produces for
// positions pos0..pos (read from qkv [R][3d] bf16); also appends the row's own K,V to the paged
// cache of layer `layer` (what kv_append did as a separate launch). out [R][d] bf16
int self_attention(const bf16* qkv, const DecRow* d_rows, int R, int d, int n_head, bf16* pool,
                   int layer, int n_layer, bf16* out, cudaStream_t stream);
// cross attention: q [R][d] bf16; kv = cross-KV of this layer [n_win][T][2d] bf16 (K | V per key).
// rows must be grouped by window: window g covers rows [grp_start[g], grp_start[g]+grp_count[g]).
// workspace: f32, >= n_groups*n_chunks*max_cnt*(d + 2*n_head) ... see cross_attention_ws_floats().
size_t cross_attention_ws_floats(int R, int d, int n_head);
// kv_rows: keys the cross-KV buffer of this layer holds (max_batch * T), for the TMA tensor map
int cross_attention(const bf16* q, const bf16* kv, int64_t kv_rows, const int* d_grp_win,
                    const int* d_grp_start, const int* d_grp_count, int n_groups, int max_count, int R,
                    int T, int d, int n_head, float* ws, bf16* out, cudaStream_t stream,
                    cudaEvent_t ev_main_done = nullptr, unsigned ev_flags = 0,  // event after the main kernel
                    int max_ctas = 0);  // cap on the persistent grid (0 = one CTA per SM)

// weight-streaming GEMM for <= 64-row blocks (skinny_gemm.cu): out = X . W^T
//   split == 1: out bf16 [R][ldo] = act(acc + bias);   split > 1: partial f32 [split][R][N] (raw sums)
int skinny_split_for(int N, int K);
int skinny_gemm(const bf16* X, int ldx, const bf16* W, int R, int N, int K, const float* bias, int gelu,
                bf16* out, int ldo, float* partial, int split, cudaStream_t stream);
// the mma.sync kernel whatever skinny_use_tc says (skinny_gemm() routes the shapes skinny_use_tc rejects here)
int skinny_gemm_mma(const bf16* X, int ldx, const bf16* W, int R, int N, int K, const float* bias, int gelu,
                    bf16* out, int ldo, float* partial, int split, cudaStream_t stream);
// generation 3 (skinny_gemm_tc.cu): 128 weight rows per CTA in the M dimension of tcgen05.mma; skinny_gemm() and
// skinny_split_for() route the wide models' matrices to it (skinny_use_tc)
bool skinny_use_tc(int N, int K);
int skinny_mma_split_for(int N, int K);  // the plan of the mma.sync kernel whatever skinny_use_tc says
int skinny_tc_split_for(int N, int K);
int skinny_gemm_tc(const bf16* X, int ldx, const bf16* W, int R, int N, int K, const float* bias, int gelu, bf16* out,
                   int ldo, float* partial, int split, cudaStream_t stream);

// ------------------------------------------------------------------ prosody (prosody.cu)
// per-segment DSP of prosody_extractor.cpp:31-224 for all segments of an utterance (SURVEY.md §8(f) rank 3)
struct ProsodySeg {     // one segment: samples [begin, begin + n_frames * shift) are analysed
  int64_t begin;        // first sample in the PCM buffer
  int n_frames;         // complete 10 ms frames
  int frame_off;        // offset of its frames in the frame buffer
};
struct ProsodyFrame {   // per 10 ms frame
  float rms;            // sqrt(mean x^2)
  int zc;               // sign changes of the low-passed frame
  int cycles;           // hysteresis cycle count of the low-passed frame
  float sc;             // sum(|dx| k) / sum(|dx|)
};
struct ProsodyRaw {     // per segment, before the heuristics (which stay on the host: capi.cpp)
  float energy_mean, energy_std, zcr_mean, sc_mean, pitch_median, pitch_std;
  int peaks, n_frames, n_f0, pad;
};
int prosody_frames(const void* d_pcm, int is_f32, const ProsodySeg* d_segs, int n_segs, int max_frames, int shift,
                   int warm, float alpha, ProsodyFrame* d_frames, cudaStream_t stream);
int prosody_reduce(const ProsodySeg* d_segs, const ProsodyFrame* d_frames, int n_segs, int shift, int sample_rate,
                   float min_pitch, float max_pitch, ProsodyRaw* d_out, cudaStream_t stream);

// ------------------------------------------------------------------ sample-rate conversion (resample.cu)
constexpr int RS_ZEROS = 16, RS_GRID = 256;  // zero crossings per side of the windowed sinc, table points per crossing
int resample_f32(const float* d_in, int64_t n_in, int sr_in, int sr_out, const float* d_table, float scale,
                 float gscale, int half, int64_t n_out, float* d_out, cudaStream_t stream);

// logit rules + log-softmax + pick (whisper_process_logits + whisper_sample_token)
struct LogitRow {        // per-row rule state, built by the host sequencer
  int is_initial;        // no token sampled yet in this window
  int last_ts;           // last sampled token was a timestamp
  int penult_ts;         // the one before was (or fewer than 2 tokens)
  int ts_min;            // has_ts ? seek_delta/2 : 0  -> timestamps below beg+ts_min suppressed
  float temperature;     // > 0: logits /= temperature
  int n_draws;           // 0: argmax; k>0: k inverse-CDF draws with the uniforms below
  int logits_row;        // row of the logits matrix
  int pad;
  double u[8];           // uniforms for the draws (host mt19937, libstdc++ generate_canonical)
};
struct PickOut {         // per draw (n_draws or 1 entries per row, stride 8)
  int id, tid;
  float p, plog, pt, ptsum;
  float no_speech_prob;  // softmax(raw logits)[nosp] (only meaningful on prompt rows)
  int pad;
};
struct LogitCfg {
  int n_vocab, token_eot, token_beg, token_nosp, token_space;
  int suppress_blank, max_initial_ts_id;  // beg + tid0 + 1 (first suppressed), or n_vocab
  const uint8_t* d_suppress;              // [n_vocab] 1 = always suppressed under these params
};
int process_logits_pick(const float* logits, int64_t ld, const LogitRow* d_rows, int R,
                        const LogitCfg& cfg, PickOut* d_out, cudaStream_t stream);

}  // namespace sw
