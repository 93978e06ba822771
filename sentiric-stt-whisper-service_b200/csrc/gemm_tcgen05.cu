// bf16 x bf16 -> f32 GEMM for sm_100a: TMA -> 128B-swizzled smem ring ->
// tcgen05.mma (accumulators in TMEM, double buffered) -> tcgen05.ld epilogue.
//
// Two kernels share the epilogue: gemm_tcgen05_kernel<64/128/256> (one CTA per 128 x N tile) and
// gemm_tcgen05_pair_kernel (a CTA pair, cta_group::2, per 256 x 256 tile; used for M >= 2048 with N tiles of 256,
// see the comment above it). Both are persistent and warp specialised, one CTA per SM:
//   warp 0      : TMA producer (one thread, chosen by elect.sync)
//   warp 1      : TMEM allocator + MMA issuer (one thread, chosen by elect.sync)
//   warps 2..9  : epilogue; warp w drains TMEM lanes [32*(w%4), 32*(w%4)+32) of one column half of the
//                 accumulator (warps 2-5 the first half, 6-9 the second): eight warps keep twice the loads
//                 and stores in flight and give every scheduler two warps to alternate between; the residual
//                 row segment of the next 32 columns is requested before the current one is consumed.
//                 Measured on the encoder of a 2-layer large-v3-width model, 64 windows, same box, alternating:
//                 12.82 ms with four warps and no prefetch, 12.22 ms with this (-4.7 %).
//                 Tried and rejected: staging every 32 x 32 chunk through an XOR-swizzled shared-memory tile so
//                 that global loads and stores leave coalesced (one instruction = 4 rows x 128 B instead of 32
//                 rows x 16 B). Bit-identical, but SLOWER (12.86 ms; 48 000 x 512 x 512: 375 instead of 544
//                 TFLOP/s): the main loop is bound by shared-memory traffic (TMA writes + operand reads of a
//                 128 x 256 tile per SM), and the staging adds to exactly that. The same on the CTA-pair kernel
//                 (where ncu shows l1tex__data_pipe_lsu_wavefronts at 52-67 % of peak in the K = 1280 GEMMs and the
//                 tensor pipe waiting for a free accumulator 25-65 % of the time): encoder of the 2-layer model
//                 0.180 ms per window direct, 0.198 staged; FC1 + GELU 1.17 -> 1.78 ms. Variants kept as
//                 tools/dev/gemm_epilogue_staged.cu.txt and gemm_epilogue_staged_pair.cu.txt. What is left to try
//                 is a TMA store out of the tile (no LDS / STG in the warps at all).
//
// This is the kernel behind every dense contraction of the Whisper path the
// reference runs through ggml's mul_mat (SURVEY.md §2.3): conv stem (implicit
// GEMM through strided TMA maps), encoder QKV/out/MLP projections, cross-KV
// projection and the decoder's prompt/logit projections
// (call site in the reference: whisper_full_with_state, stt_engine.cpp:245).
#include "common.cuh"
#include "gemm.cuh"

#include <stdlib.h>

#include <mutex>

namespace sw {

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;
constexpr int NUM_THREADS = 320;
constexpr int EPI_WARPS = 8;
constexpr int EPI_WARP0 = 2;
constexpr int SMEM_BUDGET = 227 * 1024;

template <int BLOCK_N>
struct Cfg {
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_BYTES = BLOCK_N * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES_RAW = (SMEM_BUDGET - 2048) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static constexpr int TMEM_COLS = 2 * BLOCK_N;  // double-buffered accumulator
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

struct EpiParams {
  void* C;
  int64_t ldc, c_batch_stride;
  const float* bias;
  const float* residual;
  int64_t ldr, r_batch_stride;
  int res_mod;
  int flags;
  int wide;  // C and residual rows are 32-byte aligned: 256-bit accesses allowed
};

// 256-bit global accesses (sm_100): a thread of the epilogue owns a row and touches 32 different cache lines per
// warp instruction, so the LSU cost is per instruction, not per byte - 32 bytes per access halve it.
__device__ __forceinline__ void ldg256(const float* p, float4& a, float4& b) {
  asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(p));
}
__device__ __forceinline__ void stg256(float* p, float a0, float a1, float a2, float a3, float a4, float a5, float a6,
                                       float a7) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(a0), "f"(a1), "f"(a2), "f"(a3),
               "f"(a4), "f"(a5), "f"(a6), "f"(a7)
               : "memory");
}
__device__ __forceinline__ void stg256(void* p, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t a4,
                                       uint32_t a5, uint32_t a6, uint32_t a7) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(a0), "r"(a1), "r"(a2), "r"(a3),
               "r"(a4), "r"(a5), "r"(a6), "r"(a7)
               : "memory");
}

// Epilogue of one accumulator tile for one warp: `row` is the output row this thread owns (its TMEM lane),
// `tmem_acc` the accumulator's address with the warp's lane quarter in the upper half, `n0` the tile's first
// column, `chalf` which half of its BLOCK_N columns this warp drains. Waits for the accumulator itself (after
// requesting the first residual segment).
template <int BLOCK_N>
__device__ __forceinline__ void epilogue_tile(const EpiParams& epi, int M, int N, int row, int n0, int b,
                                              uint32_t tmem_acc, int chalf, uint64_t* full_bar, uint32_t full_phase) {
  const bool out_f32 = (epi.flags & GEMM_OUT_F32) != 0;
  const bool do_gelu = (epi.flags & GEMM_GELU) != 0;
  const bool bias_row = (epi.flags & GEMM_BIAS_ROW) != 0;
  const bool row_ok = row < M;
  const int64_t rrow = epi.res_mod > 0 ? (row % epi.res_mod) : row;
  const float* rptr =
      (epi.residual && row_ok) ? epi.residual + b * epi.r_batch_stride + rrow * epi.ldr : nullptr;
  const float row_bias = (bias_row && epi.bias && row_ok) ? epi.bias[row] : 0.0f;
  constexpr int CHUNKS = BLOCK_N / 32 / 2;  // 32-column chunks per warp (its half of the accumulator)
  const int c_begin = chalf * CHUNKS;
  // residual of a full chunk, requested one chunk ahead (the first one before the accumulator is waited for)
  float4 rv[8];
  auto load_res = [&](int c, float4 (&dst)[8]) {
    const int col0 = n0 + c * 32;
    if (rptr && col0 + 32 <= N) {
      if (epi.wide) {
#pragma unroll
        for (int j = 0; j < 4; ++j) ldg256(rptr + col0 + 8 * j, dst[2 * j], dst[2 * j + 1]);
      } else {
        const float4* rp = reinterpret_cast<const float4*>(rptr + col0);
#pragma unroll
        for (int j = 0; j < 8; ++j) dst[j] = rp[j];
      }
    }
  };
  load_res(c_begin, rv);

  mbar_wait(full_bar, full_phase);
  tc_fence_after();

#pragma unroll 1
  for (int c = c_begin; c < c_begin + CHUNKS; ++c) {
    const int col0 = n0 + c * 32;
    if (col0 >= N) break;  // warp-uniform
    uint32_t r[32];
    tmem_ld_32x32b_x32(tmem_acc + c * 32,
                       r);
    float4 rn[8];
    if (c + 1 < c_begin + CHUNKS) load_res(c + 1, rn);
    tmem_ld_wait(r);
    if (!row_ok) continue;
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
    const bool full = (col0 + 32 <= N);
    if (epi.bias) {
      if (bias_row) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += row_bias;
      } else if (full) {
        const float4* bp = reinterpret_cast<const float4*>(epi.bias + col0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float4 t = __ldg(bp + j);
          v[4 * j + 0] += t.x;
          v[4 * j + 1] += t.y;
          v[4 * j + 2] += t.z;
          v[4 * j + 3] += t.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (col0 + j < N) v[j] += epi.bias[col0 + j];
      }
    }
    if (do_gelu) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = gelu_tanh(v[j]);
    }
    if (rptr) {
      if (full) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          v[4 * j + 0] += rv[j].x;
          v[4 * j + 1] += rv[j].y;
          v[4 * j + 2] += rv[j].z;
          v[4 * j + 3] += rv[j].w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (col0 + j < N) v[j] += rptr[col0 + j];
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) rv[j] = rn[j];
    if (out_f32) {
      float* cp = static_cast<float*>(epi.C) + b * epi.c_batch_stride + (int64_t)row * epi.ldc + col0;
      if (full && epi.wide) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          stg256(cp + 8 * j, v[8 * j], v[8 * j + 1], v[8 * j + 2], v[8 * j + 3], v[8 * j + 4], v[8 * j + 5],
                 v[8 * j + 6], v[8 * j + 7]);
      } else if (full) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          reinterpret_cast<float4*>(cp)[j] =
              make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (col0 + j < N) cp[j] = v[j];
      }
    } else {
      __nv_bfloat16* cp = static_cast<__nv_bfloat16*>(epi.C) + b * epi.c_batch_stride +
                          (int64_t)row * epi.ldc + col0;
      if (full && epi.wide) {
#pragma unroll
        for (int j = 0; j < 2; ++j)
          stg256(static_cast<void*>(cp + 16 * j), pack_bf16x2(v[16 * j + 0], v[16 * j + 1]),
                 pack_bf16x2(v[16 * j + 2], v[16 * j + 3]), pack_bf16x2(v[16 * j + 4], v[16 * j + 5]),
                 pack_bf16x2(v[16 * j + 6], v[16 * j + 7]), pack_bf16x2(v[16 * j + 8], v[16 * j + 9]),
                 pack_bf16x2(v[16 * j + 10], v[16 * j + 11]), pack_bf16x2(v[16 * j + 12], v[16 * j + 13]),
                 pack_bf16x2(v[16 * j + 14], v[16 * j + 15]));
      } else if (full) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 o;
          o.x = pack_bf16x2(v[8 * j + 0], v[8 * j + 1]);
          o.y = pack_bf16x2(v[8 * j + 2], v[8 * j + 3]);
          o.z = pack_bf16x2(v[8 * j + 4], v[8 * j + 5]);
          o.w = pack_bf16x2(v[8 * j + 6], v[8 * j + 7]);
          reinterpret_cast<uint4*>(cp)[j] = o;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (col0 + j < N) cp[j] = __float2bfloat16_rn(v[j]);
      }
    }
  }
}

template <int BLOCK_N>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap map_a,
                    const __grid_constant__ CUtensorMap map_b, EpiParams epi, int M, int N, int K,
                    int batch, int b_batched) {
  using C = Cfg<BLOCK_N>;
  extern __shared__ uint8_t smem_raw[];
  // 128B swizzle atoms need 1024-byte aligned tiles.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tmem_full_bar = empty_bar + C::STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp_idx = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // provably warp-uniform
  const int lane = threadIdx.x & 31;

  const int m_tiles = (M + BLOCK_M - 1) / BLOCK_M;
  const int n_tiles = (N + BLOCK_N - 1) / BLOCK_N;
  const int k_blocks = (K + BLOCK_K - 1) / BLOCK_K;
  const int total_tiles = m_tiles * n_tiles * batch;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full_bar[a], 1);
      mbar_init(&tmem_empty_bar[a], EPI_WARPS);  // one arrive per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp_idx == 1) {
    tmem_alloc(tmem_base_slot, C::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;

  if (warp_idx == 0) {
    // ===================== TMA producer =====================
    // (elect.sync, not a lane test: ptxas then emits each UTMALDG / UTCHMMA once; under `lane == 0` it wraps every
    // one in a loop over the active lanes - R2UR, ELECT, BRA.U.ANY - about 100 cycles per instruction)
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int n_blk = tile % n_tiles;
        const int m_blk = (tile / n_tiles) % m_tiles;
        const int b = tile / (n_tiles * m_tiles);
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * C::STAGE_BYTES;
          uint8_t* sb = sa + C::A_BYTES;
          mbar_arrive_expect_tx(&full_bar[stage], C::STAGE_BYTES);
          tma_load_3d(sa, &map_a, &full_bar[stage], kb * BLOCK_K, m_blk * BLOCK_M, b);
          tma_load_3d(sb, &map_b, &full_bar[stage], kb * BLOCK_K, n_blk * BLOCK_N,
                      b_batched ? b : 0);
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================== MMA issuer =====================
    if (elect_one_sync()) {
      constexpr uint32_t idesc = make_idesc_bf16(BLOCK_M, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::STAGE_BYTES);
          const uint32_t sb = sa + C::A_BYTES;
          const uint64_t adesc = make_umma_desc_sw128(sa);
          const uint64_t bdesc = make_umma_desc_sw128(sb);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            // advance 32 B (16 bf16) inside the 128B swizzle row: +2 in the
            // (addr >> 4) start-address field
            umma_bf16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
          }
          umma_commit(&empty_bar[stage]);  // frees the smem slot when the MMAs retire
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&tmem_full_bar[acc]);  // accumulator complete -> epilogue
      }
    }
  } else {
    // ===================== epilogue warps =====================
    const int q = warp_idx & 3;  // TMEM lane quarter this warp may touch
    const int chalf = (warp_idx - EPI_WARP0) >> 2;  // which half of the accumulator's columns
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int n_blk = tile % n_tiles;
      const int m_blk = (tile / n_tiles) % m_tiles;
      const int b = tile / (n_tiles * m_tiles);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;

      epilogue_tile<BLOCK_N>(epi, M, N, m_blk * BLOCK_M + q * 32 + lane, n_blk * BLOCK_N, b,
                             tmem_base + acc * BLOCK_N + (static_cast<uint32_t>(q * 32) << 16), chalf,
                             &tmem_full_bar[acc], acc_phase);
      // hand the accumulator back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------
// CTA-pair variant (cta_group::2): one 256 x 256 tile per pair of SMs
// ---------------------------------------------------------------------------
// The single-CTA kernel above moves (128 + 256) x 64 operand elements into shared memory per k-block and SM, and
// its main loop is bound by exactly that traffic (TMA writes + operand reads). A CTA pair computes a 256 x 256
// tile with each CTA holding 128 rows of A and 128 rows of B per k-block - two thirds of the bytes per SM for the
// same MMA time. CTA 0 of the pair issues the MMAs (tcgen05.mma.cta_group::2 reads both CTAs' shared memory and
// writes 128 accumulator rows into each CTA's tensor memory); both CTAs load with TMA (completing on CTA 0's
// barrier), both drain their own half of the accumulator.
namespace pair {
constexpr int BN = 256;                      // tile columns (128 rows of B per CTA)
constexpr int A_BYTES = 128 * BLOCK_K * 2;   // per CTA
constexpr int B_BYTES = 128 * BLOCK_K * 2;   // per CTA
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int STAGES = 7;  // 7 x 32 KB + barriers = 225.3 KB of the 227 KB
constexpr int TMEM_COLS = 2 * BN;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load of a CTA pair: the bytes land in this CTA's shared memory, the transaction completes on `bar_cluster`
__device__ __forceinline__ void tma_load_3d_pair(void* smem_dst, const void* map, uint32_t bar_cluster, int c0, int c1,
                                                 int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs once all earlier MMAs of this thread have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(static_cast<uint16_t>(3))
      : "memory");
}
}  // namespace pair

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
gemm_tcgen05_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                         EpiParams epi, int M, int N, int K, int batch, int b_batched) {
  using namespace pair;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);  // used in CTA 0 only
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;  // used in CTA 0 only
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp_idx = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair_idx = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

  const int m_tiles = (M + 255) / 256;
  const int n_tiles = (N + BN - 1) / BN;
  const int k_blocks = (K + BLOCK_K - 1) / BLOCK_K;
  const int total_tiles = m_tiles * n_tiles * batch;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full_bar[a], 1);
      mbar_init(&tmem_empty_bar[a], 2 * EPI_WARPS);  // the epilogue warps of both CTAs
    }
    fence_mbar_init();
  }
  if (warp_idx == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();  // barriers of both CTAs initialised, tensor memory allocated in both
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;

  if (warp_idx == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair_idx; tile < total_tiles; tile += n_pairs) {
        const int n_blk = tile % n_tiles;
        const int m_blk = (tile / n_tiles) % m_tiles;
        const int b = tile / (n_tiles * m_tiles);
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * STAGE_BYTES;
          uint8_t* sb = sa + A_BYTES;
          const uint32_t full0 = map_to_cta(smem_u32(&full_bar[stage]), 0);
          if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * STAGE_BYTES);  // both CTAs' bytes
          tma_load_3d_pair(sa, &map_a, full0, kb * BLOCK_K, m_blk * 256 + (int)rank * 128, b);
          tma_load_3d_pair(sb, &map_b, full0, kb * BLOCK_K, n_blk * BN + (int)rank * 128, b_batched ? b : 0);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================== MMA issuer (CTA 0 only) =====================
    if (rank == 0 && elect_one_sync()) {
      constexpr uint32_t idesc = make_idesc_bf16(256, BN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = pair_idx; tile < total_tiles; tile += n_pairs, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint64_t adesc = make_umma_desc_sw128(sa);
          const uint64_t bdesc = make_umma_desc_sw128(sa + A_BYTES);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
            umma_bf16_pair(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
          umma_commit_pair(&empty_bar[stage]);  // frees the slot in both CTAs
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit_pair(&tmem_full_bar[acc]);  // accumulator complete -> both CTAs' epilogues
      }
    }
  } else {
    // ===================== epilogue warps (both CTAs, own 128 rows each) =====================
    const int q = warp_idx & 3;
    const int chalf = (warp_idx - EPI_WARP0) >> 2;
    int it = 0;
    for (int tile = pair_idx; tile < total_tiles; tile += n_pairs, ++it) {
      const int n_blk = tile % n_tiles;
      const int m_blk = (tile / n_tiles) % m_tiles;
      const int b = tile / (n_tiles * m_tiles);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      epilogue_tile<BN>(epi, M, N, m_blk * 256 + (int)rank * 128 + q * 32 + lane, n_blk * BN, b,
                        tmem_base + acc * BN + (static_cast<uint32_t>(q * 32) << 16), chalf, &tmem_full_bar[acc],
                        acc_phase);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(map_to_cta(smem_u32(&tmem_empty_bar[acc]), 0));
    }
  }

  tc_fence_before();
  cluster_sync_all();  // nobody touches the peer's shared or tensor memory after this
  if (warp_idx == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) ==
            cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// 3-D bf16 K-major operand map: dims {K, rows, batch}, box {64, box_rows, 1}, 128B swizzle.
int make_operand_map(CUtensorMap* map, const void* base, int64_t K, int64_t rows, int64_t batch,
                     int64_t ld_elems, int64_t batch_stride_elems, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  SW_CHECK(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
  SW_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "GEMM operand base not 16B aligned");
  SW_CHECK((ld_elems * 2) % 16 == 0, "GEMM operand row stride %lld not a multiple of 8 elements",
           (long long)ld_elems);
  if (batch <= 1 || batch_stride_elems == 0) {
    batch = 1;
    batch_stride_elems = rows * ld_elems;
  }
  SW_CHECK((batch_stride_elems * 2) % 16 == 0, "GEMM batch stride not 16B aligned");
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)ld_elems * 2, (cuuint64_t)batch_stride_elems * 2};
  cuuint32_t box[3] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SW_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed: %d (K=%lld rows=%lld ld=%lld)", (int)r,
           (long long)K, (long long)rows, (long long)ld_elems);
  return 0;
}

// 256-bit epilogue accesses need 32-byte aligned rows of C (and of the residual, when there is one);
// otherwise the epilogue keeps 128-bit accesses
bool epilogue_wide_ok(const GemmArgs& a) {
  const int64_t esz = (a.flags & GEMM_OUT_F32) ? 4 : 2;
  bool ok = (reinterpret_cast<uintptr_t>(a.C) & 31) == 0 && (a.ldc * esz) % 32 == 0 && (a.c_batch_stride * esz) % 32 == 0;
  if (a.residual)
    ok = ok && (reinterpret_cast<uintptr_t>(a.residual) & 31) == 0 && (a.ldr * 4) % 32 == 0 && (a.r_batch_stride * 4) % 32 == 0;
  return ok;
}

int num_sms() { return device_sm_count(); }  // of the current device (host_common.h)

template <int BLOCK_N>
int launch(const GemmArgs& a, cudaStream_t stream) {
  using C = Cfg<BLOCK_N>;
  static SmemOptIn opt_in;  // per device (host_common.h)
  SW_CUDA_CHECK(opt_in.ensure(gemm_tcgen05_kernel<BLOCK_N>, C::SMEM_BYTES));
  CUtensorMap map_a, map_b;
  if (make_operand_map(&map_a, a.A, a.K, a.M, a.batch, a.lda, a.a_batch_stride, BLOCK_M)) return -1;
  const bool b_batched = a.b_batch_stride != 0 && a.batch > 1;
  if (make_operand_map(&map_b, a.B, a.K, a.N, b_batched ? a.batch : 1, a.ldb, a.b_batch_stride,
                       BLOCK_N))
    return -1;
  EpiParams epi;
  epi.C = a.C;
  epi.ldc = a.ldc;
  epi.c_batch_stride = a.c_batch_stride;
  epi.bias = a.bias;
  epi.residual = a.residual;
  epi.ldr = a.ldr;
  epi.r_batch_stride = a.r_batch_stride;
  epi.res_mod = a.res_mod;
  epi.flags = a.flags;
  epi.wide = epilogue_wide_ok(a);
  const int m_tiles = (a.M + BLOCK_M - 1) / BLOCK_M;
  const int n_tiles = (a.N + BLOCK_N - 1) / BLOCK_N;
  const int64_t tiles = (int64_t)m_tiles * n_tiles * a.batch;
  const int grid = (int)(tiles < num_sms() ? tiles : num_sms());
  gemm_tcgen05_kernel<BLOCK_N><<<grid, NUM_THREADS, C::SMEM_BYTES, stream>>>(
      map_a, map_b, epi, a.M, a.N, a.K, a.batch, b_batched ? 1 : 0);
  SW_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_pair(const GemmArgs& a, cudaStream_t stream) {
  static SmemOptIn opt_in;
  SW_CUDA_CHECK(opt_in.ensure(gemm_tcgen05_pair_kernel, pair::SMEM_BYTES));
  CUtensorMap map_a, map_b;
  if (make_operand_map(&map_a, a.A, a.K, a.M, a.batch, a.lda, a.a_batch_stride, 128)) return -1;
  const bool b_batched = a.b_batch_stride != 0 && a.batch > 1;
  if (make_operand_map(&map_b, a.B, a.K, a.N, b_batched ? a.batch : 1, a.ldb, a.b_batch_stride, 128)) return -1;
  EpiParams epi;
  epi.C = a.C;
  epi.ldc = a.ldc;
  epi.c_batch_stride = a.c_batch_stride;
  epi.bias = a.bias;
  epi.residual = a.residual;
  epi.ldr = a.ldr;
  epi.r_batch_stride = a.r_batch_stride;
  epi.res_mod = a.res_mod;
  epi.flags = a.flags;
  epi.wide = epilogue_wide_ok(a);
  const int64_t tiles = (int64_t)((a.M + 255) / 256) * ((a.N + pair::BN - 1) / pair::BN) * a.batch;
  const int pairs_max = num_sms() / 2;
  const int grid = 2 * (int)(tiles < pairs_max ? tiles : pairs_max);
  gemm_tcgen05_pair_kernel<<<grid, NUM_THREADS, pair::SMEM_BYTES, stream>>>(map_a, map_b, epi, a.M, a.N, a.K, a.batch,
                                                                           b_batched ? 1 : 0);
  SW_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

int make_tma_map_2d_bf16(void* map_out, const void* base, int64_t inner, int64_t rows, int64_t ld_elems,
                         int box_inner, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  SW_CHECK(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
  SW_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (ld_elems * 2) % 16 == 0, "TMA operand not 16B aligned");
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld_elems * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(static_cast<CUtensorMap*>(map_out), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base),
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SW_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(2d) failed: %d", (int)r);
  return 0;
}

int make_tma_map_3d_bf16(void* map_out, const void* base, const int64_t dims_in[3], const int64_t strides_bytes[2],
                         const int box_in[3]) {
  EncodeTiledFn enc = get_encode_fn();
  SW_CHECK(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
  SW_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "TMA operand not 16B aligned");
  cuuint64_t dims[3] = {(cuuint64_t)dims_in[0], (cuuint64_t)dims_in[1], (cuuint64_t)dims_in[2]};
  cuuint64_t strides[2] = {(cuuint64_t)strides_bytes[0], (cuuint64_t)strides_bytes[1]};
  cuuint32_t box[3] = {(cuuint32_t)box_in[0], (cuuint32_t)box_in[1], (cuuint32_t)box_in[2]};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(static_cast<CUtensorMap*>(map_out), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base),
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SW_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(3d) failed: %d", (int)r);
  return 0;
}

int gemm_bf16_tn(const GemmArgs& a, cudaStream_t stream) {
  SW_CHECK(a.M > 0 && a.N > 0 && a.K > 0 && a.batch > 0, "gemm: empty problem");
  SW_CHECK(a.A && a.B && a.C, "gemm: null operand");
  const bool out_f32 = (a.flags & GEMM_OUT_F32) != 0;
  SW_CHECK(a.ldc % (out_f32 ? 4 : 8) == 0, "gemm: ldc %lld breaks 16B store alignment",
           (long long)a.ldc);
  SW_CHECK((reinterpret_cast<uintptr_t>(a.C) & 15) == 0, "gemm: C not 16B aligned");
  if (a.residual) SW_CHECK(a.ldr % 4 == 0, "gemm: ldr must be a multiple of 4");
  int bn = a.block_n;
  if (bn == 0) {
    // Largest tile that still gives every SM work; small problems prefer more tiles.
    const int64_t m_tiles = (a.M + BLOCK_M - 1) / BLOCK_M;
    bn = 256;
    while (bn > 64 && (m_tiles * ((a.N + bn - 1) / bn) * a.batch < num_sms() || a.N <= bn / 2))
      bn >>= 1;
    if (bn == 256 && a.M >= 2048) bn = 512;  // CTA pairs for the large encoder shapes
  }
  if (bn == 512) return launch_pair(a, stream);
  switch (bn) {
    case 64: return launch<64>(a, stream);
    case 128: return launch<128>(a, stream);
    case 256: return launch<256>(a, stream);
    default: set_last_error("gemm: unsupported block_n %d", bn); return -1;
  }
}

}  // namespace sw
