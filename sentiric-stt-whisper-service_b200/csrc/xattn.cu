// Decoder cross attention over the 1500 encoder positions of each active window: the kernel that
// streams the cross-KV cache (245.8 MB per window for large-v3) once per decoder step and therefore
// dominates the step (DESIGN.md §4). Replaces ggml's flash_attn_ext in whisper_decode_internal
// (SURVEY.md A.5, §2.3).
//
// Persistent: one CTA per SM walks work items (group g = one window and its <= 8 decoder rows,
// chunk of `spc` 16-key stages) blockIdx.x, +gridDim.x, ... so the grid is a whole number of waves
// whatever the batch size. One producer thread issues ONE 3-D TMA load per stage: box
// {64 dims, 16 keys, 2*n_head segments} of the [key][K row | V row] cache lands in shared memory as
// [segment][key][64] tiles with the 128-byte swizzle, i.e. exactly the operand tiles ldmatrix wants.
// Consumer warps own whole heads (head h -> warp h % n_consumers) and run flash-decoding on the
// tensor pipe: S[16 x 16 keys] = Q K^T and O[16 x 64] += P V with mma.sync m16n8k16, where the M
// dimension holds the <= 8 decoders (beams) that share the window - so the cache is read from HBM
// once however many beams there are, and no cross-warp merge is needed. Generation 1 did the dot
// products on CUDA cores and was instruction-issue bound at ~68 % of HBM (profiles/r1_ncu_xattn_v1.txt).
//
// The flash-decoding merge of the per-chunk partials is a second, tiny kernel chained by programmatic
// dependent launch. (Fusing it into this kernel - last-arriving warp merges - was measured at 155 us
// per launch instead of 79 + combine: the merging warp stalls the two-stage TMA pipeline of its CTA.)
// The cache does not depend on the previous kernel of the step, so under programmatic dependent
// launch the producer starts streaming it before griddepcontrol.wait; only the query load and the
// stores wait. The kernel itself never calls launch_dependents: its successors (the merge, the cross-out
// GEMM, ...) must not become resident while it streams (see the comment in the kernel).
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

namespace sw {
namespace {

constexpr int XA_KEYS = 16;
constexpr int XA_MAX_CONSUMERS = 10;
constexpr int XA_MAX_CHUNKS = 32;
constexpr int XA_MAX_HPW = 3;  // heads per warp

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int HPW>
__global__ void __launch_bounds__((XA_MAX_CONSUMERS + 1) * 32, 1)
cross_attention_kernel(const __grid_constant__ CUtensorMap map_kv, const bf16* __restrict__ q,
                       const int* __restrict__ grp_win, const int* __restrict__ grp_start,
                       const int* __restrict__ grp_count, int T, int d, int n_head, int n_cons, int spc,
                       int n_stages, int n_chunks, int n_items, float* __restrict__ ws, uint32_t zero, int n_hsplit) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const uint32_t sbase = smem_u32(smem);
  // a work item is (window, chunk of keys, group of heads): with n_hsplit = 2 a CTA streams the K and V rows of half
  // the heads only, so a stage is half as large and the ring twice as deep (large-v3: 5 x 40 KB instead of 2 x 80 KB)
  const int nh_cta = n_head / n_hsplit;  // heads of one item
  const int half_bytes = XA_KEYS * nh_cta * 64 * 2;  // the K tiles (or the V tiles) of a stage
  const int stage_bytes = 2 * half_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)n_stages * stage_bytes);
  uint64_t* empty = full + n_stages;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp: provably uniform
  const int row_f = d + 2 * n_head;  // floats per (row, chunk) partial

  // No early launch_dependents here: the dependents (the merge, then the cross-out GEMM, ...) would become resident
  // while this kernel streams for ~85 us and hold shared memory on exactly the SMs the OTHER lane's chain runs on.
  // They are released when this CTA has nothing left to do (end of the kernel).
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_kv);
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], n_cons);
    }
    fence_mbar_init();
  }
  __syncthreads();

  if (warp == n_cons) {
    // no pdl_wait here: the cross-KV cache and the group tables were complete before the step's
    // first kernel started; the loads only fill this CTA's own shared memory
    if (elect_one_sync()) {  // not a lane test: one UTMALDG per load instead of a loop over the active lanes
      // the cache is read once per step: evict-first keeps it from pushing the lanes' shared weights out of L2
      // (+1.2 % on the two-lane bench against the default policy, measured ABAB on one box: 3 796 / 3 851 / 3 809 /
      // 3 844 audio-s/s)
      const uint64_t pol = l2_policy_evict_first();
      int it = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int gc = item / n_hsplit, hh = item - gc * n_hsplit;
        const int g = gc / n_chunks, chunk = gc - g * n_chunks;
        const int win = grp_win[g];
        const int key_begin = chunk * spc * XA_KEYS;
        const int key_end = min(T, key_begin + spc * XA_KEYS);
        const int n_st = (key_end - key_begin + XA_KEYS - 1) / XA_KEYS;
        for (int i = 0; i < n_st; ++i, ++it) {
          const int s = it % n_stages;
          const uint32_t ph = (it / n_stages) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          mbar_arrive_expect_tx(&full[s], stage_bytes);
          uint8_t* dst = smem + (size_t)s * stage_bytes;
          const int key = win * T + key_begin + i * XA_KEYS;
          // segments of the [K row | V row] cache line: K heads 0 .. n_head-1, then V heads. Not unrolled: with the
          // two loads written out, ptxas spills more in the consumers of the 2- and 3-heads-per-warp instantiations
#pragma unroll 1
          for (int kv = 0; kv < 2; ++kv)
            tma_load_3d_hint(dst + kv * half_bytes, &map_kv, &full[s], 0, key, kv * n_head + hh * nh_cta, pol);
        }
      }
    }
    return;
  }
  if (warp > n_cons) return;

  // ---- consumers
  pdl_wait();  // q comes from the previous kernel; ws / out may still be read by earlier ones
  const int g8 = lane >> 2, t4 = lane & 3;
  const float qs = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e), applied to the f32 scores
  // raw query fragments of the next item: [head slot][k-step][a0, a2]
  uint32_t qn[HPW][4][2];
  auto prefetch_q = [&](int item) {
    const int gc = item / n_hsplit, hh = item - gc * n_hsplit;
    const int g = gc / n_chunks;
    const int cnt = grp_count[g], r0 = grp_start[g];
#pragma unroll
    for (int hs = 0; hs < HPW; ++hs) {
      const int hl = warp + hs * n_cons;          // head within the item
      const int h = hh * nh_cta + hl;
      const bool ok = hl < nh_cta && g8 < cnt;
      const bf16* qp = q + (int64_t)(r0 + g8) * d + h * 64 + 2 * t4;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        qn[hs][ks][0] = ok ? *reinterpret_cast<const uint32_t*>(qp + ks * 16) : 0u;
        qn[hs][ks][1] = ok ? *reinterpret_cast<const uint32_t*>(qp + ks * 16 + 8) : 0u;
      }
    }
  };
  if ((int)blockIdx.x < n_items) prefetch_q(blockIdx.x);
  int it = 0;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int gc = item / n_hsplit, hh = item - gc * n_hsplit;
    const int g = gc / n_chunks, chunk = gc - g * n_chunks;
    const int r0 = grp_start[g], cnt = grp_count[g];
    const int key_begin = chunk * spc * XA_KEYS;
    const int key_end = min(T, key_begin + spc * XA_KEYS);
    const int n_st = (key_end - key_begin + XA_KEYS - 1) / XA_KEYS;
    uint32_t qa[HPW][4][4];
    float o[HPW][8][2], m[HPW], l[HPW];
#pragma unroll
    for (int hs = 0; hs < HPW; ++hs) {
      m[hs] = -INFINITY;
      l[hs] = 0.f;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        qa[hs][ks][0] = qn[hs][ks][0];
        qa[hs][ks][1] = 0u;  // rows 8..15 of the m16 tile are unused (<= 8 decoders per window)
        qa[hs][ks][2] = qn[hs][ks][1];
        qa[hs][ks][3] = 0u;
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) o[hs][nt][0] = o[hs][nt][1] = 0.f;
    }
    if (item + (int)gridDim.x < n_items) prefetch_q(item + gridDim.x);

    for (int i = 0; i < n_st; ++i, ++it) {
      const int s = it % n_stages;
      const uint32_t ph = (it / n_stages) & 1;
      mbar_wait(&full[s], ph);
      const uint32_t st = sbase + s * stage_bytes;
      const int nk = min(XA_KEYS, key_end - key_begin - i * XA_KEYS);
      uint32_t dep = 0;  // one result register of every ldmatrix of this stage (mbar_arrive_after_reads)
#pragma unroll
      for (int hs = 0; hs < HPW; ++hs) {
        const int hl = warp + hs * n_cons;
        if (hl >= nh_cta) continue;
        const uint32_t kt = st + hl * 2048, vt = st + half_bytes + hl * 2048;  // [16 keys][128 B] swizzled tiles
        float sc[2][4];
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          uint32_t b[4];
          const int key = (lane & 7) + (lane >> 4) * 8;
          const int ch = ks * 2 + ((lane >> 3) & 1);
          ldmatrix_x4(b, kt + key * 128 + ((ch ^ (key & 7)) << 4));
          dep ^= b[0];
          const uint32_t b01[2] = {b[0], b[1]}, b23[2] = {b[2], b[3]};
          mma_m16n8k16_bf16(sc[0], qa[hs][ks], b01);
          mma_m16n8k16_bf16(sc[1], qa[hs][ks], b23);
        }
        // row g8 (decoder), keys nt*8 + 2*t4 + {0,1}
        float v00 = sc[0][0] * qs, v01 = sc[0][1] * qs, v10 = sc[1][0] * qs, v11 = sc[1][1] * qs;
        if (nk < XA_KEYS) {
          if (2 * t4 >= nk) v00 = -INFINITY;
          if (2 * t4 + 1 >= nk) v01 = -INFINITY;
          if (8 + 2 * t4 >= nk) v10 = -INFINITY;
          if (8 + 2 * t4 + 1 >= nk) v11 = -INFINITY;
        }
        float rmax = fmaxf(fmaxf(v00, v01), fmaxf(v10, v11));
        rmax = fmaxf(rmax, __shfl_xor_sync(0xffffffffu, rmax, 1));
        rmax = fmaxf(rmax, __shfl_xor_sync(0xffffffffu, rmax, 2));
        const float mn = fmaxf(m[hs], rmax);
        const float alpha = fast_exp2(m[hs] - mn);
        const float p00 = fast_exp2(v00 - mn), p01 = fast_exp2(v01 - mn);
        const float p10 = fast_exp2(v10 - mn), p11 = fast_exp2(v11 - mn);
        m[hs] = mn;
        l[hs] = l[hs] * alpha + (p00 + p01) + (p10 + p11);  // per-thread partial; quad-reduced at the end
        uint32_t pa[4];
        pa[0] = pack_bf16x2(p00, p01);
        pa[1] = 0u;
        pa[2] = pack_bf16x2(p10, p11);
        pa[3] = 0u;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          o[hs][nt][0] *= alpha;
          o[hs][nt][1] *= alpha;
        }
#pragma unroll
        for (int dp = 0; dp < 4; ++dp) {
          uint32_t b[4];
          const int key = (lane & 7) + ((lane >> 3) & 1) * 8;
          const int ch = dp * 2 + (lane >> 4);
          ldmatrix_x4_trans(b, vt + key * 128 + ((ch ^ (key & 7)) << 4));
          dep ^= b[0];
          const uint32_t b01[2] = {b[0], b[1]}, b23[2] = {b[2], b[3]};
          float acc0[4] = {o[hs][2 * dp][0], o[hs][2 * dp][1], 0.f, 0.f};
          float acc1[4] = {o[hs][2 * dp + 1][0], o[hs][2 * dp + 1][1], 0.f, 0.f};
          mma_m16n8k16_bf16(acc0, pa, b01);
          mma_m16n8k16_bf16(acc1, pa, b23);
          o[hs][2 * dp][0] = acc0[0];
          o[hs][2 * dp][1] = acc0[1];
          o[hs][2 * dp + 1][0] = acc1[0];
          o[hs][2 * dp + 1][1] = acc1[1];
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive_after_reads(&empty[s], dep, zero);
    }
    // ---- partial result of this (window, chunk): unnormalised O, running max m and sum l per head
#pragma unroll
    for (int hs = 0; hs < HPW; ++hs) {
      const int hl = warp + hs * n_cons;
      if (hl >= nh_cta) continue;
      const int h = hh * nh_cta + hl;
      float ls = l[hs];
      ls += __shfl_xor_sync(0xffffffffu, ls, 1);
      ls += __shfl_xor_sync(0xffffffffu, ls, 2);
      if (g8 < cnt) {
        float* op = ws + ((int64_t)(r0 + g8) * n_chunks + chunk) * row_f;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
          *reinterpret_cast<float2*>(op + h * 64 + nt * 8 + 2 * t4) = make_float2(o[hs][nt][0], o[hs][nt][1]);
        if (t4 == 0) {
          op[d + h] = m[hs];
          op[d + n_head + h] = ls;
        }
      }
    }
  }
}

// Merge the per-chunk partials of a row: one warp per (row, group of 4 heads); lane = (head, 8-dim chunk).
__global__ void __launch_bounds__(32)
cross_combine_kernel(const float* __restrict__ ws, int n_chunks, int d, int n_head, bf16* __restrict__ out) {
  pdl_launch_dependents();
  const int r = blockIdx.x;
  const int h = blockIdx.y * 4 + (threadIdx.x >> 3);
  pdl_wait();
  if (h >= n_head) return;
  const int c = h * 8 + (threadIdx.x & 7);  // 8-float chunk of the row
  const int row_f = d + 2 * n_head;
  const float* base = ws + (int64_t)r * n_chunks * row_f;
  float M = -INFINITY;
#pragma unroll 8
  for (int k = 0; k < n_chunks; ++k) M = fmaxf(M, base[(int64_t)k * row_f + d + h]);
  float L = 0.f, a[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) a[e] = 0.f;
#pragma unroll 4
  for (int k = 0; k < n_chunks; ++k) {
    const float* p = base + (int64_t)k * row_f;
    const float m1 = p[d + h];
    const float wgt = (m1 == -INFINITY) ? 0.f : fast_exp2(m1 - M);
    L += p[d + n_head + h] * wgt;
    const float4 x0 = reinterpret_cast<const float4*>(p + c * 8)[0];
    const float4 x1 = reinterpret_cast<const float4*>(p + c * 8)[1];
    a[0] += x0.x * wgt; a[1] += x0.y * wgt; a[2] += x0.z * wgt; a[3] += x0.w * wgt;
    a[4] += x1.x * wgt; a[5] += x1.y * wgt; a[6] += x1.z * wgt; a[7] += x1.w * wgt;
  }
  const float inv = 1.0f / L;
  uint4 o;
  o.x = pack_bf16x2(a[0] * inv, a[1] * inv);
  o.y = pack_bf16x2(a[2] * inv, a[3] * inv);
  o.z = pack_bf16x2(a[4] * inv, a[5] * inv);
  o.w = pack_bf16x2(a[6] * inv, a[7] * inv);
  reinterpret_cast<uint4*>(out + (int64_t)r * d)[c] = o;
}

int xa_num_sms() { return device_sm_count(); }  // of the current device, cached per ordinal (host_common.h)

// stages per work item: the value that leaves the fewest idle SM-slots in the last wave
void xa_plan(int n_groups, int T, int d, int max_ctas, int n_hsplit, int* spc_out, int* n_chunks, int* n_stages,
             int* grid) {
  const int total_stages = (T + XA_KEYS - 1) / XA_KEYS;
  int sms = xa_num_sms();
  if (max_ctas > 0 && max_ctas < sms) sms = max_ctas;
  int best_spc = 3;
  double best_eff = -1.0;
  for (int spc = 3; spc <= 16; ++spc) {
    const int nch = (total_stages + spc - 1) / spc;
    if (nch > XA_MAX_CHUNKS) continue;
    const int items = n_groups * nch * n_hsplit;
    const int g = items < sms ? items : sms;
    const int rounds = (items + g - 1) / g;
    const double eff = (double)n_groups * n_hsplit * total_stages / ((double)g * rounds * spc) * (g / (double)sms);
    if (eff >= best_eff) {
      best_eff = eff;
      best_spc = spc;
    }
  }
  *spc_out = best_spc;
  *n_chunks = (total_stages + best_spc - 1) / best_spc;
  const int items = n_groups * *n_chunks * n_hsplit;
  *grid = items < sms ? items : sms;
  const int stage_bytes = XA_KEYS * 2 * (d / n_hsplit) * 2;
  int ns = (220 * 1024) / stage_bytes;
  if (ns > 8) ns = 8;
  if (ns < 2) ns = 2;
  *n_stages = ns;
}

}  // namespace

size_t cross_attention_ws_floats(int R, int d, int n_head) {
  return (size_t)R * XA_MAX_CHUNKS * (d + 2 * n_head);
}

int cross_attention(const bf16* q, const bf16* kv, int64_t kv_rows, const int* d_grp_win,
                    const int* d_grp_start, const int* d_grp_count, int n_groups, int max_count, int R,
                    int T, int d, int n_head, float* ws, bf16* out, cudaStream_t stream,
                    cudaEvent_t ev_main_done, unsigned ev_flags, int max_ctas) {
  if (n_groups <= 0 || R <= 0) return 0;
  SW_CHECK(d == n_head * 64, "cross_attention: head dim must be 64");
  SW_CHECK(max_count >= 1 && max_count <= 8, "cross_attention: group of %d rows", max_count);
  // wide models: a CTA takes half the heads of a (window, chunk), so a stage is 40 KB instead of 80 KB (large-v3) and
  // the ring 5 deep instead of 2 - with two stages an SM streamed 55 GB/s whatever the grid (64, 96 CTAs measured),
  // i.e. the ring, not HBM, bounded every capped launch. Narrow models, whose ring of whole-window stages is 3 or
  // more deep, keep whole windows per CTA.
  const int n_hsplit = (XA_KEYS * 2 * d * 2 * 3 > 220 * 1024 && n_head % 2 == 0) ? 2 : 1;
  const int nh_cta = n_head / n_hsplit;
  // consumer warps: the largest divisor of the item's heads that is <= 10, so every warp owns the same number of heads
  int n_cons = 1;
  for (int c = 1; c <= XA_MAX_CONSUMERS; ++c)
    if (nh_cta % c == 0) n_cons = c;
  const int hpw = nh_cta / n_cons;
  SW_CHECK(hpw <= XA_MAX_HPW, "cross_attention: %d heads per warp", hpw);
  int spc, n_chunks, n_stages, grid;
  xa_plan(n_groups, T, d, max_ctas, n_hsplit, &spc, &n_chunks, &n_stages, &grid);
  const int stage_bytes = XA_KEYS * 2 * (d / n_hsplit) * 2;
  const size_t smem = (size_t)n_stages * stage_bytes + 1024 + 2 * n_stages * sizeof(uint64_t);
  SW_CHECK(smem <= 227 * 1024, "cross_attention: %zu bytes of shared memory", smem);
  const int n_items = n_groups * n_chunks * n_hsplit;
  // the cache as a 3-D tensor {64 dims, keys, 2*n_head segments of the [K | V] row}; one box = the K (or V) tiles
  // of an item's heads
  CUtensorMap map;
  const int64_t dims[3] = {64, kv_rows, 2 * n_head};
  const int64_t strides[2] = {(int64_t)2 * d * 2, 128};
  const int box[3] = {64, XA_KEYS, nh_cta};
  if (make_tma_map_3d_bf16(&map, kv, dims, strides, box)) return -1;
  const int threads = (n_cons + 1) * 32;
#define XA_LAUNCH(H)                                                                                  \
  do {                                                                                                \
    static SmemOptIn opt_in; /* per device (host_common.h) */                                         \
    SW_CUDA_CHECK(opt_in.ensure(cross_attention_kernel<H>, (int)smem));                               \
    SW_CUDA_CHECK(launch_pdl(cross_attention_kernel<H>, dim3(grid), dim3(threads), smem, stream, map, \
                             q, d_grp_win, d_grp_start, d_grp_count, T, d, n_head, n_cons, spc,        \
                             n_stages, n_chunks, n_items, ws, 0u, n_hsplit));                         \
  } while (0)
  switch (hpw) {
    case 1: XA_LAUNCH(1); break;
    case 2: XA_LAUNCH(2); break;
    case 3: XA_LAUNCH(3); break;
    default: set_last_error("cross_attention: unsupported head split"); return -1;
  }
#undef XA_LAUNCH
  if (ev_main_done) SW_CUDA_CHECK(cudaEventRecordWithFlags(ev_main_done, stream, ev_flags));
  SW_CUDA_CHECK(launch_pdl(cross_combine_kernel, dim3(R, (n_head + 3) / 4), dim3(32), 0, stream, ws, n_chunks, d, n_head,
                           out));
  return 0;
}

}  // namespace sw
