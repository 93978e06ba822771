// Weight-streaming GEMM for the decoder step: out[R][N] = X[R][K] . W[N][K]^T with R = the few
// decoder rows of a step (<= 64 per row block) and W a bf16 weight matrix that is read from HBM
// exactly once. This is what ggml's mul_mat_vec / small-batch mul_mat does per token in
// whisper_decode_internal (SURVEY.md §2.3); the 128-row tcgen05 tiles of gemm_tcgen05.cu leave
// most SMs idle at these shapes (N/64 CTAs), so the step is bound by how many SMs pull weights.
//
// CTA tile 64 (rows) x BN (32 or 40 weight rows) x 64 (k) per stage, 8-stage smem ring, two CTAs per SM.
// One producer thread issues two TMA tile loads per stage (128B-swizzled, rows past R / N are
// zero-filled by the TMA unit) that complete on an mbarrier, so the 8 consumer warps execute
// nothing but ldmatrix + mma.sync m16n8k16 (the math is ~1 % of the tensor peak: HBM/L2-bound by
// construction). Generation 1 issued per-thread cp.async and was instruction-latency bound at
// ~1 TB/s (profiles/r1_ncu_skinny_v1.txt); per-row 128-byte bulk copies were slower still.
// N-small matrices are split along K so that >= 148 CTAs stream weights; split partials are f32
// and are reduced by the consumer (fused LayerNorm / reduce_partials).
//
// What bounds a launch (tools/dev_decode_kernels.py, profiles/r1_skinny_shapes.log): a fixed ~3.8 us
// chain (launch -> first tile -> store) plus the bytes the MOST LOADED SM has to take in through TMA at
// ~46 B/clk (~88 GB/s): every CTA re-reads its 8 KB activation tile per k-block next to 4-5 KB of
// weights. 160 CTAs on 148 SMs (FC1 / FC2 with 32-column tiles) put two CTAs on 12 SMs and cost
// 9.8 us; the same matrix cut into 148 CTAs costs 6.6 us. skinny_plan() therefore picks the tile
// width (32 or 40 columns) and the K split that minimise the bytes of the most loaded SM:
// 40 columns x split 4 (128 CTAs) for the d x d and FC2 matrices, 40 x 1 (128 CTAs) for FC1,
// 32 x 1 (120 CTAs) for QKV. L2-resident weights change nothing (r1_skinny_l2.log): it is SM
// ingest, not HBM.
// Tried and rejected, measured with tools/dev_decode_kernels.py (profiles/r1_skinny_ab.log): (a) one
// persistent CTA per SM with a 16-stage ring: ~2x slower (half the consumer warps per SM); (b) a
// software-pipelined consumer (fragments of k-block i+1 loaded before the MMAs of k-block i, four
// accumulator chains): 8.1 vs 6.4 us on QKV, 13.0 vs 9.5 us on FC1. The launch is bound by ring bytes
// in flight x latency (96 KB per CTA, two thirds of it re-read activations), not by the consumers;
// (c) tcgen05.mma with M = 64, N = 32 and a TMEM accumulator (tools/dev/skinny_gemm_tcgen05_m64.cu.txt,
// profiles/r1_skinny_tcgen05_m64.log): correct, but 10.8 vs 6.4 us on QKV - tiny SS-mode MMAs are
// dispatch-latency bound and 16 of 32 lanes per epilogue warp idle.
// The weight tiles of the first ring fill do not depend on the previous kernel, so the producer
// issues them before griddepcontrol.wait (only matters when SW_PDL=1).
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

namespace sw {
namespace {

constexpr int SK_BM = 64, SK_BK = 64, SK_STAGES = 8;
constexpr int SK_X_BYTES = SK_BM * SK_BK * 2;
constexpr int SK_CONSUMERS = 8;
constexpr int SK_THREADS = (SK_CONSUMERS + 1) * 32;
template <int BN>
struct SkCfg {
  static constexpr int W_BYTES = BN * SK_BK * 2;
  static constexpr int STAGE_BYTES = SK_X_BYTES + W_BYTES;  // 12 / 13 KB: stage bases stay 1024-byte aligned
  static constexpr int smem(int n_stages) { return n_stages * STAGE_BYTES + 1024 + 2 * n_stages * 8; }
  static constexpr int NT = BN / 8;        // 8-column MMA tiles of the CTA
  static constexpr int NT0 = (NT + 1) / 2;  // tiles of column-warp 0 (column-warp 1 takes the rest)
};

template <int BN>
__global__ void __launch_bounds__(SK_THREADS, 2)
skinny_gemm_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, int R,
                   int N, int k_slice, const float* __restrict__ bias, int gelu, bf16* __restrict__ out, int ldo,
                   float* __restrict__ partial, uint32_t zero, int n_stages) {
  using C = SkCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const uint32_t sbase = smem_u32(smem);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + n_stages * C::STAGE_BYTES);
  uint64_t* empty = full + n_stages;
  const int n0 = blockIdx.x * BN;
  const int k_begin = blockIdx.y * k_slice;
  const int r0 = blockIdx.z * SK_BM;
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;  // warp: provably uniform
  const int n_kb = k_slice / SK_BK;

  pdl_launch_dependents();
  if (tid == 0) {
    tma_prefetch_desc(&map_x);
    tma_prefetch_desc(&map_w);
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], SK_CONSUMERS);
    }
    fence_mbar_init();
  }
  __syncthreads();

  if (warp == SK_CONSUMERS) {
    // elect.sync rather than a lane test: ptxas then emits each TMA instruction once instead of inside a loop over
    // the active lanes (R2UR + ELECT + BRA.U.ANY around every UTMALDG)
    if (elect_one_sync()) {
      // weights first (independent of the predecessor), activations once it has finished
      const int pre = n_kb < n_stages ? n_kb : n_stages;
      for (int kb = 0; kb < pre; ++kb) {
        mbar_arrive_expect_tx(&full[kb], C::STAGE_BYTES);
        tma_load_2d(smem + kb * C::STAGE_BYTES + SK_X_BYTES, &map_w, &full[kb], k_begin + kb * SK_BK, n0);
      }
      pdl_wait();
      for (int kb = 0; kb < pre; ++kb)
        tma_load_2d(smem + kb * C::STAGE_BYTES, &map_x, &full[kb], k_begin + kb * SK_BK, r0);
      for (int kb = pre; kb < n_kb; ++kb) {
        const int s = kb % n_stages;
        const uint32_t ph = (kb / n_stages) & 1;
        mbar_wait(&empty[s], ph ^ 1);
        mbar_arrive_expect_tx(&full[s], C::STAGE_BYTES);
        uint8_t* xs = smem + s * C::STAGE_BYTES;
        tma_load_2d(xs, &map_x, &full[s], k_begin + kb * SK_BK, r0);
        tma_load_2d(xs + SK_X_BYTES, &map_w, &full[s], k_begin + kb * SK_BK, n0);
      }
    }
    return;
  }

  // ---- consumers: warp (rw, nh) owns rows 16*rw.. of the row block and the 8-column tiles
  // [t0, t0 + nt) of the CTA (column-warp 0: the first NT0 tiles, column-warp 1: the rest)
  const int rw = warp & 3, nh = warp >> 2;
  const int t0 = nh ? C::NT0 : 0;
  const int nt_mine = nh ? C::NT - C::NT0 : C::NT0;
  float acc[C::NT0][4];
#pragma unroll
  for (int i = 0; i < C::NT0; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
  // 128B-swizzled tiles: 16-byte chunk c of row r lives at r*128 + ((c ^ (r & 7)) << 4)
  const int a_row = rw * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, a_ch = lane >> 4;
  // weight fragments: x4 = two tiles (rows +0..7 | +8..15, k lo | k hi), x2 = one tile (lanes 0-15 address it)
  const int b_row4 = t0 * 8 + (lane & 7) + (lane >> 4) * 8;
  const int b_ch = (lane >> 3) & 1;
  for (int kb = 0; kb < n_kb; ++kb) {
    const int s = kb % n_stages;
    const uint32_t ph = (kb / n_stages) & 1;
    mbar_wait(&full[s], ph);
    const uint32_t xs = sbase + s * C::STAGE_BYTES, ws = xs + SK_X_BYTES;
    uint32_t a[SK_BK / 16][4], b[SK_BK / 16][C::NT0][2];
    uint32_t dep = 0;  // one result register of every ldmatrix of this stage (mbar_arrive_after_reads)
#pragma unroll
    for (int ks = 0; ks < SK_BK / 16; ++ks) {
      ldmatrix_x4(a[ks], xs + a_row * 128 + (((ks * 2 + a_ch) ^ (a_row & 7)) << 4));
      dep ^= a[ks][0];
#pragma unroll
      for (int tp = 0; tp + 1 < C::NT0 + 1; tp += 2) {
        if (tp + 1 < nt_mine) {  // a pair of tiles
          uint32_t t[4];
          const int row = b_row4 + tp * 8;
          ldmatrix_x4(t, ws + row * 128 + (((ks * 2 + b_ch) ^ (row & 7)) << 4));
          b[ks][tp][0] = t[0]; b[ks][tp][1] = t[1];
          if (tp + 1 < C::NT0) { b[ks][tp + 1][0] = t[2]; b[ks][tp + 1][1] = t[3]; }
          dep ^= t[0];
        } else if (tp < nt_mine) {  // a last single tile
          uint32_t t[2];
          const int row = (t0 + tp) * 8 + (lane & 7);
          ldmatrix_x2(t, ws + row * 128 + (((ks * 2 + b_ch) ^ (row & 7)) << 4));
          b[ks][tp][0] = t[0]; b[ks][tp][1] = t[1];
          dep ^= t[0];
        }
      }
    }
#pragma unroll
    for (int ks = 0; ks < SK_BK / 16; ++ks)
#pragma unroll
      for (int t = 0; t < C::NT0; ++t)
        if (t < nt_mine) mma_m16n8k16_bf16(acc[t], a[ks], b[ks][t]);
    __syncwarp();
    if (lane == 0) mbar_arrive_after_reads(&empty[s], dep, zero);  // every fragment is in registers: the slot can be refilled
  }

  pdl_wait();  // (already satisfied: the activations we consumed were loaded after the producer's wait)
  const int g = lane >> 2, t4 = lane & 3;
  const int row0 = r0 + rw * 16 + g, row1 = row0 + 8;
#pragma unroll
  for (int t = 0; t < C::NT0; ++t) {
    const int col = n0 + (t0 + t) * 8 + 2 * t4;
    if (t >= nt_mine || col >= N) continue;
    if (partial) {
      float* p = partial + ((int64_t)blockIdx.y * R) * N;
      if (row0 < R) *reinterpret_cast<float2*>(p + (int64_t)row0 * N + col) = make_float2(acc[t][0], acc[t][1]);
      if (row1 < R) *reinterpret_cast<float2*>(p + (int64_t)row1 * N + col) = make_float2(acc[t][2], acc[t][3]);
    } else {
      float v0 = acc[t][0], v1 = acc[t][1], v2 = acc[t][2], v3 = acc[t][3];
      if (bias) {
        const float b0 = __ldg(bias + col), b1 = __ldg(bias + col + 1);
        v0 += b0; v1 += b1; v2 += b0; v3 += b1;
      }
      if (gelu) {
        v0 = gelu_tanh(v0); v1 = gelu_tanh(v1); v2 = gelu_tanh(v2); v3 = gelu_tanh(v3);
      }
      if (row0 < R) *reinterpret_cast<uint32_t*>(out + (int64_t)row0 * ldo + col) = pack_bf16x2(v0, v1);
      if (row1 < R) *reinterpret_cast<uint32_t*>(out + (int64_t)row1 * ldo + col) = pack_bf16x2(v2, v3);
    }
  }
}

// bytes the most loaded SM takes in for tile width bn and `split` K slices (CTAs dealt round-robin
// over the SMs, two resident per SM); a third CTA on an SM would be a second wave: excluded
double sk_cost(int N, int K, int row_blocks, int bn, int split) {
  const int n_cta = ((N + bn - 1) / bn) * split * row_blocks;
  if (n_cta > 2 * 148 && split > 1) return 1e30;
  const double per_cta = (double)(K / split / SK_BK) * (SK_X_BYTES + bn * SK_BK * 2) + 4096.0 * split;
  return per_cta * ((n_cta + 147) / 148);
}
int sk_pick_bn(int N, int K, int row_blocks, int split) {
  return sk_cost(N, K, row_blocks, 40, split) < sk_cost(N, K, row_blocks, 32, split) ? 40 : 32;
}

}  // namespace

int skinny_split_for(int N, int K) { return skinny_use_tc(N, K) ? skinny_tc_split_for(N, K) : skinny_mma_split_for(N, K); }

int skinny_mma_split_for(int N, int K) {
  // the K split (a divisor of the k-block count, slices of >= 2 k-blocks) that, with the better of the
  // two tile widths, leaves the fewest bytes on the most loaded SM; ties go to fewer splits
  const int n_kb = K / SK_BK;
  int best = 1;
  double best_cost = 1e31;
  for (int s = 1; s <= 32 && (s == 1 || s <= n_kb / 2); ++s) {
    if (n_kb % s) continue;
    const double c = fmin(sk_cost(N, K, 1, 32, s), sk_cost(N, K, 1, 40, s));
    if (c < best_cost * 0.999) {
      best_cost = c;
      best = s;
    }
  }
  return best;
}

int skinny_gemm(const bf16* X, int ldx, const bf16* W, int R, int N, int K, const float* bias, int gelu,
                bf16* out, int ldo, float* partial, int split, cudaStream_t stream) {
  if (skinny_use_tc(N, K)) return skinny_gemm_tc(X, ldx, W, R, N, K, bias, gelu, out, ldo, partial, split, stream);
  return skinny_gemm_mma(X, ldx, W, R, N, K, bias, gelu, out, ldo, partial, split, stream);
}

int skinny_gemm_mma(const bf16* X, int ldx, const bf16* W, int R, int N, int K, const float* bias, int gelu,
                    bf16* out, int ldo, float* partial, int split, cudaStream_t stream) {
  if (R <= 0) return 0;
  SW_CHECK(K % SK_BK == 0 && ldx % 8 == 0 && N % 2 == 0, "skinny_gemm: unsupported shape N=%d K=%d ldx=%d", N, K, ldx);
  SW_CHECK(split >= 1 && split <= 32 && (split == 1 || partial), "skinny_gemm: split-K needs a partial buffer");
  SW_CHECK(K % (split * SK_BK) == 0, "skinny_gemm: K=%d not divisible into %d slices of 64-element blocks", K, split);
  SW_CHECK(partial || out, "skinny_gemm: null output");
  SW_CHECK((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0,
           "skinny_gemm: operands must be 16-byte aligned");
  static SmemOptIn opt_in32, opt_in40;  // per device (host_common.h)
  SW_CUDA_CHECK(opt_in32.ensure(skinny_gemm_kernel<32>, SkCfg<32>::smem(SK_STAGES)));
  SW_CUDA_CHECK(opt_in40.ensure(skinny_gemm_kernel<40>, SkCfg<40>::smem(SK_STAGES)));
  const int k_slice = K / split;
  const int row_blocks = (R + SK_BM - 1) / SK_BM;
  const int bn = sk_pick_bn(N, K, row_blocks, split);
  CUtensorMap map_x, map_w;
  if (make_tma_map_2d_bf16(&map_x, X, K, R, ldx, SK_BK, SK_BM)) return -1;
  if (make_tma_map_2d_bf16(&map_w, W, K, N, K, SK_BK, bn)) return -1;
  dim3 grid((N + bn - 1) / bn, split, row_blocks);
  if (bn == 40)
    SW_CUDA_CHECK(launch_pdl(skinny_gemm_kernel<40>, grid, dim3(SK_THREADS), SkCfg<40>::smem(SK_STAGES), stream, map_x,
                             map_w, R, N, k_slice, bias, gelu, out, ldo, partial, 0u, SK_STAGES));
  else
    SW_CUDA_CHECK(launch_pdl(skinny_gemm_kernel<32>, grid, dim3(SK_THREADS), SkCfg<32>::smem(SK_STAGES), stream, map_x,
                             map_w, R, N, k_slice, bias, gelu, out, ldo, partial, 0u, SK_STAGES));
  return 0;
}

}  // namespace sw
