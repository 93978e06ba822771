// Per-token decoder kernels: paged self-KV append + causal self attention, the cross attention
// that streams each window's cross-KV exactly once per step, and the logit rules / log-softmax /
// argmax-or-draw kernel. Together they replace, for one batched step, the device part of
// whisper_decode_internal and the CPU whisper_process_logits / whisper_sample_token* of
// whisper.cpp (SURVEY.md A.5-A.6; reference call site stt_engine.cpp:245).
#include <type_traits>

#include "common.cuh"
#include "kernels.cuh"

namespace sw {
namespace {

__device__ __forceinline__ void bf16x8_to_f32(const uint4& u, float (&f)[8]) {
  f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xffff0000u);
  f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xffff0000u);
  f[4] = __uint_as_float(u.z << 16); f[5] = __uint_as_float(u.z & 0xffff0000u);
  f[6] = __uint_as_float(u.w << 16); f[7] = __uint_as_float(u.w & 0xffff0000u);
}

// ------------------------------------------------------------------------------------------
__global__ void kv_copy_pages_kernel(bf16* __restrict__ pool, const int* __restrict__ pairs, int64_t page_elems) {
  const int src = pairs[2 * blockIdx.y], dst = pairs[2 * blockIdx.y + 1];
  const uint4* s = reinterpret_cast<const uint4*>(pool + (int64_t)src * page_elems);
  uint4* d = reinterpret_cast<uint4*>(pool + (int64_t)dst * page_elems);
  const int64_t nv = page_elems / 8;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x)
    d[i] = s[i];
}

// one CTA (128 threads) per (row, head); n_kv = pos + 1 <= 448. The CTA also appends the row's own
// K/V head slice to the paged cache (no separate append launch); keys of positions >= pos0 are
// produced by rows of this same step and are read from the qkv buffer, not from the cache.
// Built for latency, not throughput (the whole launch moves a few MB): the row descriptor carries
// its page list, so the dependent chain is descriptor -> K and V loads (issued together, V kept in
// registers while the softmax statistics are reduced) -> store. Generation 1 walked the keys of the
// P.V product one dependent load at a time and cost 13 us per layer inside the step graph.
__device__ __forceinline__ const bf16* sa_kv_ptr(const bf16* pool, const DecRow& row, const bf16* own, int k, int kv,
                                                 int layer, int n_layer, int d, int h) {
  if (k >= row.pos0) return own - (int64_t)(row.pos - k) * 3 * d + (1 + kv) * d;  // produced in this step
  const int page = row.pages[k / KV_PAGE];
  return pool + ((((int64_t)page * n_layer + layer) * 2 + kv) * KV_PAGE + (k % KV_PAGE)) * d + h * 64;
}

__global__ void __launch_bounds__(128)
self_attention_kernel(const bf16* __restrict__ qkv, const DecRow* __restrict__ rows, int d,
                      bf16* __restrict__ pool, int layer, int n_layer, bf16* __restrict__ out) {
  __shared__ DecRow row;
  __shared__ float qs[64];
  __shared__ float sc[448];
  __shared__ float red[4];
  __shared__ float part[16][65];
  const int r = blockIdx.x, h = blockIdx.y, tid = threadIdx.x;
  pdl_launch_dependents();
  pdl_wait();
  const bf16* own = qkv + (int64_t)r * 3 * d + h * 64;  // q | k (+d) | v (+2d) of this row and head
  constexpr int ROW_INTS = sizeof(DecRow) / 4;
  if (tid < ROW_INTS) reinterpret_cast<int*>(&row)[tid] = reinterpret_cast<const int*>(rows + r)[tid];
  uint4 mine = make_uint4(0, 0, 0, 0);
  if (tid >= 32 && tid < 48) mine = reinterpret_cast<const uint4*>(own + (1 + ((tid - 32) >> 3)) * d)[tid & 7];
  if (tid >= 64) qs[tid - 64] = __bfloat162float(own[tid - 64]) * 0.125f;
  __syncthreads();
  const int n_kv = row.pos + 1;
  if (tid >= 32 && tid < 48) {  // append: 2 x 128 bytes
    const int kv = (tid - 32) >> 3;
    const int page = row.pages[row.pos / KV_PAGE];
    bf16* dst = pool + ((((int64_t)page * n_layer + layer) * 2 + kv) * KV_PAGE + (row.pos % KV_PAGE)) * d + h * 64;
    reinterpret_cast<uint4*>(dst)[tid & 7] = mine;
  }
  // ---- issue the K loads (thread = key) and the first V loads (thread = (key group, 8-dim chunk)) together
  const int kg = tid >> 3, vc = tid & 7;
  uint4 kreg[8], vreg[4];
  if (tid < n_kv) {
    const uint4* kp = reinterpret_cast<const uint4*>(sa_kv_ptr(pool, row, own, tid, 0, layer, n_layer, d, h));
#pragma unroll
    for (int c = 0; c < 8; ++c) kreg[c] = kp[c];
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int k = kg + 16 * j;
    vreg[j] = make_uint4(0, 0, 0, 0);
    if (k < n_kv) vreg[j] = reinterpret_cast<const uint4*>(sa_kv_ptr(pool, row, own, k, 1, layer, n_layer, d, h))[vc];
  }
  float lmax = -INFINITY;
  if (tid < n_kv) {
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float f[8];
      bf16x8_to_f32(kreg[c], f);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc += qs[c * 8 + e] * f[e];
    }
    sc[tid] = acc;
    lmax = acc;
  }
  for (int k = tid + 128; k < n_kv; k += 128) {  // long contexts
    const uint4* kp = reinterpret_cast<const uint4*>(sa_kv_ptr(pool, row, own, k, 0, layer, n_layer, d, h));
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float f[8];
      bf16x8_to_f32(kp[c], f);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc += qs[c * 8 + e] * f[e];
    }
    sc[k] = acc;
    lmax = fmaxf(lmax, acc);
  }
  lmax = warp_max(lmax);
  if ((tid & 31) == 0) red[tid >> 5] = lmax;
  __syncthreads();
  const float mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  __syncthreads();
  float lsum = 0.f;
  for (int k = tid; k < n_kv; k += 128) {
    const float p = __expf(sc[k] - mx);
    sc[k] = p;
    lsum += p;
  }
  lsum = warp_sum(lsum);
  if ((tid & 31) == 0) red[tid >> 5] = lsum;
  __syncthreads();
  const float inv = 1.0f / (red[0] + red[1] + red[2] + red[3]);
  // ---- P.V: thread (kg, vc) accumulates keys kg, kg+16, ... for dims vc*8..vc*8+7
  float a[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) a[e] = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int k = kg + 16 * j;
    if (k < n_kv) {
      const float p = sc[k];
      float f[8];
      bf16x8_to_f32(vreg[j], f);
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] += p * f[e];
    }
  }
  for (int k0 = 64; k0 < n_kv; k0 += 64) {
    uint4 v4[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + kg + 16 * j;
      v4[j] = make_uint4(0, 0, 0, 0);
      if (k < n_kv) v4[j] = reinterpret_cast<const uint4*>(sa_kv_ptr(pool, row, own, k, 1, layer, n_layer, d, h))[vc];
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + kg + 16 * j;
      if (k < n_kv) {
        const float p = sc[k];
        float f[8];
        bf16x8_to_f32(v4[j], f);
#pragma unroll
        for (int e = 0; e < 8; ++e) a[e] += p * f[e];
      }
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) part[kg][vc * 8 + e] = a[e];
  __syncthreads();
  if (tid < 64) {
    float v = 0.f;
#pragma unroll
    for (int g = 0; g < 16; ++g) v += part[g][tid];
    out[(int64_t)r * d + h * 64 + tid] = __float2bfloat16_rn(v * inv);
  }
}

// ------------------------------------------------------------------------------------------
// logits: rules -> log-softmax -> timestamp-vs-text -> argmax or inverse-CDF draws
// ------------------------------------------------------------------------------------------
constexpr int LP_THREADS = 1024;

// exp for the vocabulary-wide passes (arguments <= 0): ex2.approx of x log2(e), relative error ~1e-6 at |x| = 20 -
// four orders of magnitude below what the bf16 logits GEMM leaves in the probabilities; libm's expf costs ~20
// instructions and a slow-path branch per element (the kernel was issue-bound: ncu 56 % issue-active on 64 SMs)
__device__ __forceinline__ float fast_expf(float x) { return __expf(x); }

struct ArgMax {
  float v;
  int i;
};
__device__ __forceinline__ ArgMax am_better(ArgMax a, ArgMax b) {  // larger v, then smaller index
  if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
  return a;
}
__device__ float block_max(float v, float* red) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0];
  for (int i = 1; i < LP_THREADS / 32; ++i) r = fmaxf(r, red[i]);
  return r;
}
__device__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
  for (int i = 0; i < LP_THREADS / 32; ++i) r += red[i];
  return r;
}
__device__ double block_sum_d(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = 0.0;
  for (int i = 0; i < LP_THREADS / 32; ++i) r += red[i];
  return r;
}
__device__ ArgMax block_argmax(ArgMax a, float* redv, int* redi) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMax b;
    b.v = __shfl_xor_sync(0xffffffffu, a.v, o);
    b.i = __shfl_xor_sync(0xffffffffu, a.i, o);
    a = am_better(a, b);
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) {
    redv[threadIdx.x >> 5] = a.v;
    redi[threadIdx.x >> 5] = a.i;
  }
  __syncthreads();
  ArgMax r = {redv[0], redi[0]};
  for (int i = 1; i < LP_THREADS / 32; ++i) r = am_better(r, ArgMax{redv[i], redi[i]});
  return r;
}

// ---- a row of logits is shared by a thread-block CLUSTER of CL CTAs (CL = 1, 2 or 4): CTA `rank` owns the
// vocabulary slice [rank * per_cta, ...), keeps it in its own shared memory, and every vocabulary-wide reduction is
// a block reduction followed by one exchange through distributed shared memory (each CTA publishes its partial in a
// slot of its own, barrier.cluster, everybody combines the CL partials in rank order - so all CTAs hold bit-identical
// results). With one CTA per row 64 rows kept 64 of the 148 SMs busy for 62 us (ncu: profiles/r2_ncu_process_logits_v1.txt).
__device__ __forceinline__ uint32_t cl_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cl_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
template <typename T>
__device__ __forceinline__ T cl_read(const T* local, uint32_t rank) {  // the same variable in CTA `rank` of the cluster
  uint32_t a;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(smem_u32(local)), "r"(rank));
  T v;
  if constexpr (sizeof(T) == 8) {
    unsigned long long u;
    asm volatile("ld.shared::cluster.b64 %0, [%1];" : "=l"(u) : "r"(a) : "memory");
    v = *reinterpret_cast<T*>(&u);
  } else {
    uint32_t u;
    asm volatile("ld.shared::cluster.b32 %0, [%1];" : "=r"(u) : "r"(a) : "memory");
    v = *reinterpret_cast<T*>(&u);
  }
  return v;
}

struct LpXchg {  // what a CTA publishes to its cluster, one slot per value so that no slot is ever rewritten
  float rmax, ts_raw, tx_raw, rsum, se, ts_se, best_v, best_ts_v;
  int best_i, best_ts_i;
  double sum_ts, sum_all, mass;
  int draw[8];
};

template <int CL>
__global__ void __launch_bounds__(LP_THREADS, 1)
process_logits_kernel(const float* __restrict__ logits, int64_t ld, const LogitRow* __restrict__ rows,
                      LogitCfg cfg, PickOut* __restrict__ out) {
  extern __shared__ __align__(16) float lg[];  // this CTA's slice: masked logits, then probs
  __shared__ float red[LP_THREADS / 32];
  __shared__ int redi[LP_THREADS / 32];
  __shared__ double redd[LP_THREADS / 32];
  __shared__ double seg_prefix[LP_THREADS];
  __shared__ LpXchg xc;
  pdl_launch_dependents();
  pdl_wait();
  const int rank = CL > 1 ? (int)cl_rank() : 0;
  const int row_idx = blockIdx.x / CL;
  const LogitRow row = rows[row_idx];
  const float* src = logits + (int64_t)row.logits_row * ld;
  const int n = cfg.n_vocab, beg = cfg.token_beg, tid = threadIdx.x;
  const int per_cta = ((n + CL - 1) / CL + 3) & ~3;
  const int lo = min(n, rank * per_cta), hi = min(n, lo + per_cta);  // my slice of the vocabulary
  const float NEG = -INFINITY;

  // pass A: raw maximum (no_speech_prob), masked copy into smem, maxima of the masked text and timestamp logits
  // (max_i fl(x_i - lse) == fl(max_i x_i - lse): the log-probability maxima of the timestamp-vs-text rule need no pass
  // of their own)
  float rmax = NEG, ts_raw = NEG, tx_raw = NEG;
  // (two instantiations: the IEEE division by the temperature - upstream's `logits[i] /= temperature` - costs an
  // FCHK + slow-path branch per element and greedy rows, temperature 0, do not divide at all)
  auto pass_a = [&](auto has_t) {
    for (int i = lo + tid; i < hi; i += LP_THREADS) {
      const float raw = src[i];
      rmax = fmaxf(rmax, raw);
      float v = raw;
      if (decltype(has_t)::value) v = raw / row.temperature;
      bool sup = cfg.d_suppress[i] != 0;
      if (row.is_initial) {
        if (cfg.suppress_blank && (i == cfg.token_eot || i == cfg.token_space)) sup = true;
        if (i >= cfg.max_initial_ts_id) sup = true;
      }
      if (row.last_ts) {
        if (row.penult_ts) {
          if (i >= beg) sup = true;
        } else {
          if (i < cfg.token_eot) sup = true;
        }
      }
      if (i >= beg && i < beg + row.ts_min) sup = true;
      v = sup ? NEG : v;
      lg[i - lo] = v;
      if (i >= beg) ts_raw = fmaxf(ts_raw, v);
      else tx_raw = fmaxf(tx_raw, v);
    }
  };
  if (row.temperature > 0.f) pass_a(std::true_type{});
  else pass_a(std::false_type{});
  rmax = block_max(rmax, red);
  ts_raw = block_max(ts_raw, red);
  tx_raw = block_max(tx_raw, red);
  if (CL > 1) {
    if (tid == 0) { xc.rmax = rmax; xc.ts_raw = ts_raw; xc.tx_raw = tx_raw; }
    cl_sync();
    rmax = ts_raw = tx_raw = NEG;
    for (int c = 0; c < CL; ++c) {
      rmax = fmaxf(rmax, cl_read(&xc.rmax, c));
      ts_raw = fmaxf(ts_raw, cl_read(&xc.ts_raw, c));
      tx_raw = fmaxf(tx_raw, cl_read(&xc.tx_raw, c));
    }
  }
  const float mx = fmaxf(ts_raw, tx_raw);
  // pass B: both softmax denominators (raw: no_speech_prob; masked: log-softmax)
  float rsum = 0.f, se = 0.f;
  for (int i = lo + tid; i < hi; i += LP_THREADS) {
    rsum += fast_expf(src[i] - rmax);
    const float v = lg[i - lo];
    if (v > NEG) se += fast_expf(v - mx);
  }
  rsum = block_sum(rsum, red);
  se = block_sum(se, red);
  if (CL > 1) {
    if (tid == 0) { xc.rsum = rsum; xc.se = se; }
    cl_sync();
    rsum = se = 0.f;
    for (int c = 0; c < CL; ++c) {
      rsum += cl_read(&xc.rsum, c);
      se += cl_read(&xc.se, c);
    }
  }
  const float nosp = expf(src[cfg.token_nosp] - (logf(rsum) + rmax));
  const float lse = logf(se) + mx;

  // timestamp mass vs best text token
  const float ts_mx = ts_raw > NEG ? ts_raw - lse : NEG, tx_mx = tx_raw > NEG ? tx_raw - lse : NEG;
  float ts_se = 0.f;
  for (int i = max(beg, lo) + tid; i < hi; i += LP_THREADS) {
    const float v = lg[i - lo];
    if (v > NEG) ts_se += fast_expf((v - lse) - ts_mx);
  }
  ts_se = block_sum(ts_se, red);
  if (CL > 1) {
    if (tid == 0) xc.ts_se = ts_se;
    cl_sync();
    ts_se = 0.f;
    for (int c = 0; c < CL; ++c) ts_se += cl_read(&xc.ts_se, c);
  }
  const float ts_lp = ts_se > 0.f ? logf(ts_se) + ts_mx : NEG;
  const bool force_ts = ts_lp > tx_mx;

  // probs (in place), argmax, timestamp statistics
  ArgMax best = {0.f, 0x7fffffff}, best_ts = {0.f, 0x7fffffff};
  double sum_ts = 0.0, sum_all = 0.0;
  const bool draws = row.n_draws > 0;  // the total mass is only needed by the inverse-CDF draws
  for (int i = lo + tid; i < hi; i += LP_THREADS) {
    float v = lg[i - lo];
    if (force_ts && i < beg) v = NEG;
    const float p = v > NEG ? fast_expf(v - lse) : 0.f;
    lg[i - lo] = p;
    if (draws) sum_all += (double)p;
    if (p > best.v) best = ArgMax{p, i};
    if (i >= beg) {
      sum_ts += (double)p;
      if (p > best_ts.v) best_ts = ArgMax{p, i};
    }
  }
  best = block_argmax(best, red, redi);
  best_ts = block_argmax(best_ts, red, redi);
  sum_ts = block_sum_d(sum_ts, redd);
  if (draws) sum_all = block_sum_d(sum_all, redd);
  if (CL > 1) {
    if (tid == 0) {
      xc.best_v = best.v; xc.best_i = best.i; xc.best_ts_v = best_ts.v; xc.best_ts_i = best_ts.i;
      xc.sum_ts = sum_ts; xc.sum_all = sum_all;
    }
    cl_sync();
    best = ArgMax{0.f, 0x7fffffff};
    best_ts = best;
    sum_ts = sum_all = 0.0;
    for (int c = 0; c < CL; ++c) {
      best = am_better(best, ArgMax{cl_read(&xc.best_v, c), cl_read(&xc.best_i, c)});
      best_ts = am_better(best_ts, ArgMax{cl_read(&xc.best_ts_v, c), cl_read(&xc.best_ts_i, c)});
      sum_ts += cl_read(&xc.sum_ts, c);
      sum_all += cl_read(&xc.sum_all, c);
    }
  }
  const int tid_ts = best_ts.i == 0x7fffffff ? 0 : best_ts.i;  // upstream starts from tid = 0
  const float pt = (float)((double)best_ts.v / (sum_ts + 1e-10));
  const float ptsum = (float)sum_ts;

  PickOut* o = out + (int64_t)row_idx * 8;
  if (!draws) {
    if (tid == 0 && rank == 0) {
      PickOut r;
      r.id = best.i == 0x7fffffff ? 0 : best.i;
      r.p = best.i == 0x7fffffff ? 0.f : best.v;
      // plog = logprobs[id] = masked logit - lse, recomputed from the unnormalised value
      const float raw = src[r.id];
      const float v = row.temperature > 0.f ? raw / row.temperature : raw;
      r.plog = best.i == 0x7fffffff ? 0.f : v - lse;
      r.tid = tid_ts;
      r.pt = pt;
      r.ptsum = ptsum;
      if (r.id >= beg) {
        r.tid = r.id;
        r.pt = r.p;
      }
      r.no_speech_prob = nosp;
      r.pad = 0;
      o[0] = r;
    }
    if (CL > 1) cl_sync();  // nobody leaves while a neighbour may still read its slots
    return;
  }
  // ---- inverse-CDF draws (std::discrete_distribution: p_i / sum, partial sums, lower_bound(u)): per-thread
  // segments of the slice, exclusive prefixes inside the CTA, the CTAs' masses in rank order in front
  const int per = (hi - lo + LP_THREADS - 1) / LP_THREADS;
  const int i0 = min(hi, lo + tid * per), i1 = min(hi, i0 + per);
  double loc = 0.0;
  for (int i = i0; i < i1; ++i) loc += (double)lg[i - lo] / sum_all;
  seg_prefix[tid] = loc;
  __syncthreads();
  if (tid == 0) {
    double run = 0.0;
    for (int i = 0; i < LP_THREADS; ++i) {
      const double t = seg_prefix[i];
      seg_prefix[i] = run;  // exclusive
      run += t;
    }
    xc.mass = run;
  }
  __syncthreads();
  double base = 0.0, next_base = 2.0;  // cumulative mass in front of my slice / of the next CTA's slice
  if (CL > 1) {
    cl_sync();
    double cum = 0.0;
    for (int c = 0; c < CL; ++c) {
      if (c == rank) base = cum;
      cum += cl_read(&xc.mass, c);
      if (c == rank && c + 1 < CL) next_base = cum;
    }
  }
  __shared__ int draw_id[8];
  if (tid < 8) draw_id[tid] = n - 1;  // cp.back() is forced to 1.0 upstream
  __syncthreads();
  for (int k = 0; k < row.n_draws && k < 8; ++k) {
    const double u = row.u[k];
    const double plo = base + seg_prefix[tid];
    const double phi = (tid + 1 < LP_THREADS) ? base + seg_prefix[tid + 1] : next_base;
    if (i0 < i1 && plo < u && u <= phi) {  // first index whose inclusive prefix >= u lies in my segment
      double run = plo;
      int pick = i1 - 1;
      for (int i = i0; i < i1; ++i) {
        run += (double)lg[i - lo] / sum_all;
        if (run >= u) {
          pick = i;
          break;
        }
      }
      atomicMin(&draw_id[k], pick);
    }
    if (tid == 0 && rank == 0 && u <= 0.0) atomicMin(&draw_id[k], 0);
  }
  __syncthreads();
  if (CL > 1) {
    if (tid < 8) xc.draw[tid] = draw_id[tid];
    cl_sync();
  }
  if (rank == 0 && tid < row.n_draws && tid < 8) {
    PickOut r;
    int id = draw_id[tid];
    if (CL > 1)
      for (int c = 1; c < CL; ++c) id = min(id, cl_read(&xc.draw[tid], c));
    r.id = id;
    const int owner = min(CL - 1, id / per_cta);
    r.p = CL > 1 ? cl_read(&lg[id - owner * per_cta], owner) : lg[id];
    const float raw = src[r.id];
    const float v = row.temperature > 0.f ? raw / row.temperature : raw;
    r.plog = r.p > 0.f ? v - lse : -INFINITY;
    r.tid = tid_ts;
    r.pt = pt;
    r.ptsum = ptsum;
    if (r.id >= beg) {
      r.tid = r.id;
      r.pt = r.p;
    }
    r.no_speech_prob = nosp;
    r.pad = 0;
    o[tid] = r;
  }
  if (CL > 1) cl_sync();  // the slices stay alive until rank 0 has read the drawn probabilities
}

}  // namespace

int kv_copy_pages(bf16* pool, const int* d_pairs, int n, int64_t page_elems, cudaStream_t stream) {
  if (n <= 0) return 0;
  kv_copy_pages_kernel<<<dim3(32, n), 256, 0, stream>>>(pool, d_pairs, page_elems);
  SW_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int self_attention(const bf16* qkv, const DecRow* d_rows, int R, int d, int n_head, bf16* pool,
                   int layer, int n_layer, bf16* out, cudaStream_t stream) {
  if (R <= 0) return 0;
  SW_CHECK(d == n_head * 64, "self_attention: head dim must be 64");
  SW_CUDA_CHECK(launch_pdl(self_attention_kernel, dim3(R, n_head), dim3(128), 0, stream, qkv, d_rows, d, pool,
                           layer, n_layer, out));
  return 0;
}

template <int CL>
static int launch_process_logits(const float* logits, int64_t ld, const LogitRow* d_rows, int R, const LogitCfg& cfg,
                                 PickOut* d_out, cudaStream_t stream) {
  const int per_cta = ((cfg.n_vocab + CL - 1) / CL + 3) & ~3;
  const size_t smem = (size_t)per_cta * sizeof(float);
  SW_CHECK(smem <= 210 * 1024, "process_logits: vocabulary of %d does not fit shared memory", cfg.n_vocab);
  static SmemOptIn opt_in;  // per device (host_common.h)
  SW_CUDA_CHECK(opt_in.ensure(process_logits_kernel<CL>, (int)smem));
  cudaLaunchConfig_t lc = {};
  lc.gridDim = dim3(R * CL);
  lc.blockDim = dim3(LP_THREADS);
  lc.dynamicSmemBytes = smem;
  lc.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (CL > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = CL;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  lc.attrs = attr;
  lc.numAttrs = na;
  SW_CUDA_CHECK(cudaLaunchKernelEx(&lc, process_logits_kernel<CL>, logits, ld, d_rows, cfg, d_out));
  return 0;
}

int process_logits_pick(const float* logits, int64_t ld, const LogitRow* d_rows, int R,
                        const LogitCfg& cfg, PickOut* d_out, cudaStream_t stream) {
  if (R <= 0) return 0;
  // CTAs per row: as many as keep the launch inside one wave (a CTA is 1024 threads x 64 registers = one SM)
  const int sms = device_sm_count();
  const int cl = R * 4 <= sms ? 4 : R * 2 <= sms ? 2 : 1;
  if (cl == 4) return launch_process_logits<4>(logits, ld, d_rows, R, cfg, d_out, stream);
  if (cl == 2) return launch_process_logits<2>(logits, ld, d_rows, R, cfg, d_out, stream);
  return launch_process_logits<1>(logits, ld, d_rows, R, cfg, d_out, stream);
}

}  // namespace sw
