// Weight-streaming GEMM of the decoder step, generation 3: out[R][N] = X[R][K] . W[N][K]^T with the WEIGHT rows
// in the M dimension of tcgen05.mma. Same contract as skinny_gemm.cu (what ggml's small-batch mul_mat does per
// token in whisper_decode_internal, SURVEY.md §2.3), used for the wide models.
//
// Why: under lanes a decoder layer's latency chain runs on the ~52 SMs the other lane's cross attention leaves
// free, and there the mma.sync kernel of skinny_gemm.cu is bound by what an SM can take in through TMA
// (~46 B/clk): its 64 x 40 tile re-reads 8 KB of activations next to every 5 KB of weights, 120 MB of ingest per
// layer for 50 MB of weights (tools/dev_chain_occupied.py, profiles/r2_chain_occupied.txt: the seven GEMMs of a
// layer cost 48 us with the GPU to themselves and 80 us on 52 SMs). Here a CTA owns 128 weight rows x a K slice:
// per 64-element k-block it takes in 16 KB of weights and RB x 128 B of activations (RB = the row block, 64 for a
// greedy batch of 64 windows), i.e. 1.5 bytes per weight byte instead of 2.6 - 3, and the tensor core reads both
// operands straight from shared memory, so no warp spends issue slots on ldmatrix.
//   warp 0     : TMA producer (one elected thread): two tile loads per stage
//   warp 1     : TMEM allocator + MMA issuer: 4 x tcgen05.mma (M = 128 weight rows, N = RB rows, K = 16) per stage
//   warps 2..5 : epilogue: thread = weight row (TMEM lane), columns = decoder rows; a warp store of one decoder row
//                covers 32 consecutive outputs (128 B of f32 partials, 64 B of bf16)
// The accumulator is the TRANSPOSE of the output tile; bias is per lane. Split-K partials are f32 [split][R][N]
// exactly as in skinny_gemm.cu, so the consumers (fused LayerNorm, reduce_partials) do not change.
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

namespace sw {
namespace {

constexpr int ST_BM = 128, ST_BK = 64;
constexpr int ST_W_BYTES = ST_BM * ST_BK * 2;
constexpr int ST_THREADS = 6 * 32;
constexpr int ST_MAX_STAGES = 8;

__global__ void __launch_bounds__(ST_THREADS, 1)
skinny_gemm_tc_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_x, int R, int N,
                      int k_slice, const float* __restrict__ bias, int gelu, bf16* __restrict__ out, int ldo,
                      float* __restrict__ partial, int RB, int n_stages, int tmem_cols) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const int stage_bytes = ST_W_BYTES + RB * ST_BK * 2;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + n_stages * stage_bytes);
  uint64_t* empty = full + n_stages;
  uint64_t* acc_full = empty + n_stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
  const int n0 = blockIdx.x * ST_BM;
  const int k_begin = blockIdx.y * k_slice;
  const int r0 = blockIdx.z * RB;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp: provably uniform
  const int n_kb = k_slice / ST_BK;

  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_w);
    tma_prefetch_desc(&map_x);
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_slot;

  if (warp == 0) {
    if (elect_one_sync()) {
      // weights first (they do not depend on the predecessor), activations once it has finished
      const int pre = n_kb < n_stages ? n_kb : n_stages;
      for (int kb = 0; kb < pre; ++kb) {
        mbar_arrive_expect_tx(&full[kb], stage_bytes);
        tma_load_2d(smem + kb * stage_bytes, &map_w, &full[kb], k_begin + kb * ST_BK, n0);
      }
      pdl_wait();
      for (int kb = 0; kb < pre; ++kb)
        tma_load_2d(smem + kb * stage_bytes + ST_W_BYTES, &map_x, &full[kb], k_begin + kb * ST_BK, r0);
      for (int kb = pre; kb < n_kb; ++kb) {
        const int s = kb % n_stages;
        mbar_wait(&empty[s], ((kb / n_stages) & 1) ^ 1);
        mbar_arrive_expect_tx(&full[s], stage_bytes);
        uint8_t* ws = smem + s * stage_bytes;
        tma_load_2d(ws, &map_w, &full[s], k_begin + kb * ST_BK, n0);
        tma_load_2d(ws + ST_W_BYTES, &map_x, &full[s], k_begin + kb * ST_BK, r0);
      }
    }
  } else if (warp == 1) {
    if (elect_one_sync()) {
      const uint32_t idesc = make_idesc_bf16(ST_BM, RB);
      for (int kb = 0; kb < n_kb; ++kb) {
        const int s = kb % n_stages;
        mbar_wait(&full[s], (kb / n_stages) & 1);
        tc_fence_after();
        const uint32_t ws = smem_u32(smem + s * stage_bytes);
        const uint64_t adesc = make_umma_desc_sw128(ws), bdesc = make_umma_desc_sw128(ws + ST_W_BYTES);
#pragma unroll
        for (int k = 0; k < ST_BK / 16; ++k) umma_bf16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
        umma_commit(&empty[s]);  // the slot is free once these MMAs have read it
      }
      umma_commit(acc_full);
    }
  } else {
    // ---- epilogue: this thread owns weight row n (TMEM lane 32 q + lane); column j of the accumulator is decoder row r0 + j
    const int q = warp & 3;
    const int n = n0 + q * 32 + lane;
    const bool n_ok = n < N;
    const float bv = (bias && n_ok && !partial) ? __ldg(bias + n) : 0.f;
    pdl_wait();  // the output buffers may still be read by the predecessor's consumers
    mbar_wait(acc_full, 0);
    tc_fence_after();
    const uint32_t taddr = tmem_d + (static_cast<uint32_t>(q * 32) << 16);
    float* pp = partial ? partial + (int64_t)blockIdx.y * R * N + n : nullptr;
    for (int c = 0; c < RB / 32; ++c) {
      const int row0 = r0 + c * 32;
      if (row0 >= R) break;  // warp-uniform
      uint32_t v[32];
      tmem_ld_32x32b_x32(taddr + c * 32, v);
      tmem_ld_wait(v);
      if (!n_ok) continue;
      if (pp) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (row0 + j < R) pp[(int64_t)(row0 + j) * N] = __uint_as_float(v[j]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float f = __uint_as_float(v[j]) + bv;
          if (gelu) f = gelu_tanh(f);
          if (row0 + j < R) out[(int64_t)(row0 + j) * ldo + n] = __float2bfloat16_rn(f);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_d, tmem_cols);
  }
}

}  // namespace

bool skinny_use_tc(int N, int K) {
  if (K % ST_BK) return false;
  // small (d = 768) and wider: measured on BASELINE config 3 (small, beam 5) 9 654 -> 9 980 audio-s/s, config 2
  // (base, d = 512) unchanged - below that a matrix has too few 128-row tiles to stream from
  return N >= 768 && K >= 768;
}

// K split of the tcgen05 kernel: about 50 CTAs (weight tiles x slices) of >= 4 k-blocks each - as many as the SMs
// a resident cross attention of the other lane leaves, and every one streams >= 64 KB of weights
int skinny_tc_split_for(int N, int K) {
  const int tiles = (N + ST_BM - 1) / ST_BM, n_kb = K / ST_BK;
  int best = 1;
  for (int s = 1; s <= 32; ++s)
    if (n_kb % s == 0 && n_kb / s >= 4 && tiles * s <= 56) best = s;
  return best;
}

int skinny_gemm_tc(const bf16* X, int ldx, const bf16* W, int R, int N, int K, const float* bias, int gelu, bf16* out,
                   int ldo, float* partial, int split, cudaStream_t stream) {
  if (R <= 0) return 0;
  SW_CHECK(K % ST_BK == 0 && ldx % 8 == 0, "skinny_gemm_tc: unsupported shape N=%d K=%d ldx=%d", N, K, ldx);
  SW_CHECK(split >= 1 && split <= 32 && (split == 1 || partial), "skinny_gemm_tc: split-K needs a partial buffer");
  SW_CHECK(K % (split * ST_BK) == 0, "skinny_gemm_tc: K=%d not divisible into %d slices of 64-element blocks", K, split);
  SW_CHECK(partial || out, "skinny_gemm_tc: null output");
  SW_CHECK((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0,
           "skinny_gemm_tc: operands must be 16-byte aligned");
  // row blocks of <= 256 decoder rows (the N dimension of the MMA), multiples of 32 (one tcgen05.ld chunk)
  const int row_blocks = (R + 255) / 256;
  const int RB = (((R + row_blocks - 1) / row_blocks) + 31) / 32 * 32;
  int tmem_cols = 32;
  while (tmem_cols < RB) tmem_cols *= 2;
  const int k_slice = K / split, n_kb = k_slice / ST_BK;
  const int stage_bytes = ST_W_BYTES + RB * ST_BK * 2;
  int n_stages = (200 * 1024) / stage_bytes;
  if (n_stages > ST_MAX_STAGES) n_stages = ST_MAX_STAGES;
  if (n_stages > n_kb) n_stages = n_kb;
  const int smem = n_stages * stage_bytes + 1024 + (2 * n_stages + 1) * 8 + 16;
  static SmemOptIn opt_in;  // per device (host_common.h)
  SW_CUDA_CHECK(opt_in.ensure(skinny_gemm_tc_kernel, 227 * 1024));
  CUtensorMap map_w, map_x;
  if (make_tma_map_2d_bf16(&map_w, W, K, N, K, ST_BK, ST_BM)) return -1;
  if (make_tma_map_2d_bf16(&map_x, X, K, R, ldx, ST_BK, RB)) return -1;
  dim3 grid((N + ST_BM - 1) / ST_BM, split, row_blocks);
  SW_CUDA_CHECK(launch_pdl(skinny_gemm_tc_kernel, grid, dim3(ST_THREADS), smem, stream, map_w, map_x, R, N, k_slice, bias,
                           gelu, out, ldo, partial, RB, n_stages, tmem_cols));
  return 0;
}

}  // namespace sw
