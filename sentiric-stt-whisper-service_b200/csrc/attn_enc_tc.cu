// Encoder self-attention: flash attention on the 5th-generation tensor cores.
// One CTA = (window, head, 128-query tile); keys/values stream in 128-key tiles:
//   warp 0 : TMA producer (Q once, then K/V tiles into a 2-stage ring; 128B-swizzled boxes of the
//            packed [Q | K | V] activation, no separate transposes)
//   warp 1 : tcgen05.mma issuer (one thread chosen by elect.sync) - S = Q K^T (128x128x64, both operands
//            K-major) into TMEM, and O_j = P V_j (128x64x128): P read from tensor memory (TS form), V consumed
//            MN-major straight from its [key][dim] tile
//   warps 2..9 : softmax, two threads per query row (= TMEM lane): read S with tcgen05.ld, keep the running
//            max / sum, write P as bf16 into P's TMEM columns with tcgen05.st, then fold O_j into an f32
//            register accumulator (acc = acc * alpha + O_j), so TMEM is never read-modify-written.
// Order of a key tile: the moment the softmax threads have read S(j) (= P(j) written) the issuer queues
// S(j+1) and only then P V(j); the serial chain is softmax -> S(j+1), while P V(j) and the fold of O(j-1) run in
// its shadow and meet it again at pass 2 of tile j+1, which needs P's columns back.
// Two CTAs share an SM (112 KB smem, 256 TMEM columns each): one CTA's softmax overlaps the other's
// MMAs. Replaces ggml's flash_attn_ext in whisper_encode_internal (SURVEY.md A.4); generation 1
// (mma.sync) reached 298 TFLOP/s and was 35 % of the encoder time.
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

namespace sw {
namespace {

constexpr int TQ = 128, TK = 128, DH = 64;
constexpr int TILE_BYTES = 128 * 64 * 2;  // 16 KB: one [128 rows][64 bf16] swizzled tile
constexpr int SM_Q = 0, SM_K = TILE_BYTES, SM_V = 3 * TILE_BYTES;
constexpr int SM_BARS = 5 * TILE_BYTES;
constexpr int SM_XCH = SM_BARS + 128;  // [2 halves][128 rows] bf16: the row maxima the two threads of a row exchange
constexpr int ATT_SMEM = SM_XCH + 512;  // two CTAs per SM: 2 x (ATT_SMEM + 1 KB reserved) <= 228 KB
constexpr int ATT_THREADS = 320;       // warp 0: TMA, warp 1: TMEM + MMA issue, warps 2-9: softmax
// Tensor memory: S (f32 scores, 128 keys) | P (bf16, two keys per 32-bit column: 64 columns) | O (f32, 64 dims).
// P has its own columns so that S(j+1) can be computed while P V(j) still reads P(j). (An earlier layout kept P
// over the scores it came from and double-buffered O instead: P V(j) then had to be issued BEFORE S(j+1) and sat
// on the serial chain; 1.44 vs 1.37 ms per layer for 64 windows.)
constexpr int TMEM_COLS = 256, TM_P = 128, TM_O = 192;
// Measured and rejected (round 2, DESIGN.md §4 "Where the time is now"): a third of the exponentials on the FMA pipe
// (slower: pass 2 is bound by issue slots, not by the MUFU unit alone) and a one-pass softmax shifted by the maximum
// of the previous tiles (encoder time unchanged: the two CTAs of an SM are bound by the exponentials they share).

// MN-major 128B-swizzled operand (the V tile: rows = keys (K), 64 dims (MN) contiguous per row):
// canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units -> SBO = 1024 B between 8-key groups
__device__ __forceinline__ uint64_t make_umma_desc_mn_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>(1) << 16;   // LBO: unused for a single 64-element MN block
  d |= static_cast<uint64_t>(64) << 32;  // SBO = 1024 B
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(ATT_THREADS, 2)
encoder_attention_tc_kernel(const __grid_constant__ CUtensorMap map_qkv, bf16* __restrict__ out, int T, int d) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_BARS);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;    // [2]
  uint64_t* v_full = bars + 3;    // [2]
  uint64_t* kv_empty = bars + 5;  // [2]
  uint64_t* s_full = bars + 7;
  uint64_t* p_ready = bars + 8;
  uint64_t* o_full = bars + 9;   // P V(j) has completed: O(j) can be folded, P's columns can be rewritten
  uint64_t* o_free = bars + 10;  // the softmax threads have folded O(j-1): P V(j) may overwrite O
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 11);

  const int qt = blockIdx.x, h = blockIdx.y, w = blockIdx.z;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp: provably uniform
  const int q0 = qt * TQ;
  const int n_tiles = (T + TK - 1) / TK;
  const int row_base = w * T;

  if (threadIdx.x == 0) {
    if (smem_u32(smem) & 1023) {
      printf("encoder_attention_tc: shared memory base not 1024-byte aligned\n");
      __trap();
    }
    tma_prefetch_desc(&map_qkv);
    mbar_init(q_full, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&v_full[s], 1);
      mbar_init(&kv_empty[s], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_ready, 8);  // one arrive per softmax warp
    mbar_init(o_full, 1);
    mbar_init(o_free, 8);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (elect_one_sync()) {
      mbar_arrive_expect_tx(q_full, TILE_BYTES);
      tma_load_2d(smem + SM_Q, &map_qkv, q_full, h * DH, row_base + q0);
      for (int j = 0; j < n_tiles; ++j) {
        const int s = j & 1;
        const uint32_t ph = (j >> 1) & 1;
        mbar_wait(&kv_empty[s], ph ^ 1);
        mbar_arrive_expect_tx(&k_full[s], TILE_BYTES);
        tma_load_2d(smem + SM_K + s * TILE_BYTES, &map_qkv, &k_full[s], d + h * DH, row_base + j * TK);
        mbar_arrive_expect_tx(&v_full[s], TILE_BYTES);
        tma_load_2d(smem + SM_V + s * TILE_BYTES, &map_qkv, &v_full[s], 2 * d + h * DH, row_base + j * TK);
      }
    }
  } else if (warp == 1) {
    // elect.sync, not `lane == 0`: ptxas then knows a single thread runs the branch and emits each tcgen05.mma
    // once; under a lane test it wraps every one in a loop over the active lanes (R2UR, ELECT, BRA.U.ANY:
    // ~110 cycles per MMA, which was the whole "MMA dispatch" share of a key tile)
    if (elect_one_sync()) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, 128);              // S = Q K^T, both K-major
      constexpr uint32_t idesc_o = make_idesc_bf16(128, 64) | (1u << 16);  // O = P V, B (V) MN-major
      const uint32_t sq = smem_u32(smem + SM_Q);
      mbar_wait(q_full, 0);
      auto issue_s = [&](int j) {  // S_j = Q K_j^T
        const int s = j & 1;
        mbar_wait(&k_full[s], (j >> 1) & 1);
        tc_fence_after();
        const uint64_t adesc = make_umma_desc_sw128(sq);
        const uint64_t bdesc = make_umma_desc_sw128(smem_u32(smem + SM_K + s * TILE_BYTES));
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) umma_bf16(tmem, adesc + 2 * k, bdesc + 2 * k, idesc_s, k != 0);
        umma_commit(s_full);
      };
      issue_s(0);
      for (int j = 0; j < n_tiles; ++j) {
        const int s = j & 1;
        const uint32_t ph = (j >> 1) & 1;
        const uint32_t sv = smem_u32(smem + SM_V + s * TILE_BYTES);
        mbar_wait(p_ready, j & 1);
        tc_fence_after();
        // every softmax thread is past its last read of S(j): the next scores go first, so that the serial chain
        // of a key tile is softmax -> S(j+1) and P V(j) runs in its shadow
        if (j + 1 < n_tiles) issue_s(j + 1);
        mbar_wait(o_free, j & 1);
        tc_fence_after();
        mbar_wait(&v_full[s], ph);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < TK / 16; ++k) {
          // A = P in tensor memory (16 keys = 8 packed columns per k-step); B = V: 16 keys = 2 KB per k-step
          const uint64_t bdesc = make_umma_desc_mn_sw128(sv + k * 2048);
          umma_bf16_ts(tmem + TM_O, tmem + TM_P + k * 8, bdesc, idesc_o, k != 0);
        }
        umma_commit(o_full);
        umma_commit(&kv_empty[s]);
      }
    }
  } else {
    // ---------------- softmax warps: TWO threads per query row (= TMEM lane): warps 2-5 take keys 0..63 of
    // every 128-key tile and output dims 0..31, warps 6-9 keys 64..127 and dims 32..63. Generation 2 had one
    // thread per row: two softmax warps per scheduler (two CTAs per SM) left every pipe under 42 % busy
    // (MUFU 42 %, ALU 40 %, FMA 21 %, issue 54 %; profiles/r1_ncu_attn_tc_v2.txt) - latency-bound.
    const int qd = warp & 3;              // TMEM lane quarter this warp may touch
    const int half = (warp - 2) >> 2;     // which 64 keys / 32 output dims
    const int row = qd * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(qd * 32) << 16;
    const float sc = 0.125f * 1.4426950408889634f;
    float m = -INFINITY, l = 0.f;
    float acc[DH / 2];
#pragma unroll
    for (int i = 0; i < DH / 2; ++i) acc[i] = 0.f;
    uint16_t* xch = reinterpret_cast<uint16_t*>(smem + SM_XCH);
    float alpha_prev = 1.f;
    auto fold_o = [&](int j, float a) {  // acc = acc * a + O_j (this thread's 32 dims)
      mbar_wait(o_full, j & 1);
      tc_fence_after();
      uint32_t r[32];
      tmem_ld_32x32b_x32(tmem + lane_addr + TM_O + half * 32, r);
      tmem_ld_wait(r);
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = acc[i] * a + __uint_as_float(r[i]);
      tc_fence_before();
    };
    const uint32_t s_addr = tmem + lane_addr + half * 64;
    const uint32_t p_addr = tmem + lane_addr + TM_P + half * 32;  // this thread's 64 probabilities: 32 packed columns
    for (int j = 0; j < n_tiles; ++j) {
      const int valid = min(TK, T - j * TK);
      mbar_wait(s_full, j & 1);
      tc_fence_after();
      // ---- pass 1: the maximum of this thread's 64 scores
      float mx = -INFINITY;
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int c = half * 2 + cc;
        uint32_t r[32];
        tmem_ld_32x32b_x32(s_addr + cc * 32, r);
        tmem_ld_wait(r);
        if (c * 32 + 32 <= valid) {
#pragma unroll
          for (int i = 0; i < 32; ++i) mx = fmaxf(mx, __uint_as_float(r[i]));
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (c * 32 + i < valid) mx = fmaxf(mx, __uint_as_float(r[i]));
        }
      }
      // the row maximum of this thread's 64 scores meets its partner's in shared memory. The partner's previous read
      // of this slot happened before it arrived on p_ready for tile j-1, and S_j (whose completion we just waited
      // for) was issued after all eight warps had arrived: no race. Exchanged as bf16 ROUNDED UP (both threads of
      // the row must use the same value; 512 bytes instead of 1 KB keep two CTAs on an SM).
      {
        const uint32_t u = __float_as_uint(mx);
        uint32_t t = u & 0xffff0000u;
        if (t != u && !(u >> 31)) t += 0x10000u;
        mx = __uint_as_float(t);
        xch[half * 128 + row] = static_cast<uint16_t>(t >> 16);
        asm volatile("bar.sync 1, 256;" ::: "memory");
        mx = fmaxf(mx, __uint_as_float(static_cast<uint32_t>(xch[(half ^ 1) * 128 + row]) << 16));
      }
      const float m_prev = m;
      m = fmaxf(m, mx * sc);
      // ---- pass 2: P = exp2(S * sc - m) -> bf16 -> tensor memory (the A operand of P V, TS form), and this
      // thread's share of the row sum
      float lsum = 0.f;
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int c = half * 2 + cc;
        uint32_t r[32];
        tmem_ld_32x32b_x32(s_addr + cc * 32, r);
        tmem_ld_wait(r);
        uint32_t pk[16];
        if (c * 32 + 32 <= valid) {  // no masking
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float p0 = fast_exp2(__uint_as_float(r[2 * i]) * sc - m);
            const float p1 = fast_exp2(__uint_as_float(r[2 * i + 1]) * sc - m);
            lsum += p0 + p1;
            pk[i] = pack_bf16x2(p0, p1);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float p0 = fast_exp2(__uint_as_float(r[2 * i]) * sc - m);
            float p1 = fast_exp2(__uint_as_float(r[2 * i + 1]) * sc - m);
            if (c * 32 + 2 * i >= valid) p0 = 0.f;
            if (c * 32 + 2 * i + 1 >= valid) p1 = 0.f;
            lsum += p0 + p1;
            pk[i] = pack_bf16x2(p0, p1);
          }
        }
        // P's columns are free once P V(j-1) has completed. It was queued behind S(j), whose completion started
        // this pass; by the time the first 32 probabilities exist it is long done, so the wait sits here and not in
        // front of the pass
        if (cc == 0 && j > 0) {
          mbar_wait(o_full, (j - 1) & 1);
          tc_fence_after();
        }
        // 32 keys = 16 packed columns of this row, over scores this thread has already consumed
        tmem_st_32x32b_x16(p_addr + cc * 16, pk);
      }
      const float alpha = j == 0 ? 1.f : fast_exp2(m_prev - m);
      l = l * alpha + lsum;  // this thread's half of the row sum (same alpha in both halves)
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_ready);
      // fold the PREVIOUS tile's O while the tensor core works on this tile's P V and the next Q K^T
      if (j > 0) fold_o(j - 1, alpha_prev);
      __syncwarp();  // O is free: P V(j), queued behind S(j+1), may overwrite it
      if (lane == 0) mbar_arrive(o_free);
      alpha_prev = alpha;
    }
    fold_o(n_tiles - 1, alpha_prev);
    // the two halves of the row sum meet in the first K buffer, which is free once the last P V has completed
    float* lx = reinterpret_cast<float*>(smem + SM_K);
    asm volatile("bar.sync 1, 256;" ::: "memory");  // every thread is past its wait for the last O
    lx[half * 128 + row] = l;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    l += lx[(half ^ 1) * 128 + row];
    if (q0 + row < T) {
      const float inv = 1.0f / l;
      bf16* op = out + (int64_t)(row_base + q0 + row) * d + h * DH + half * 32;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        uint4 o;
        o.x = pack_bf16x2(acc[8 * i] * inv, acc[8 * i + 1] * inv);
        o.y = pack_bf16x2(acc[8 * i + 2] * inv, acc[8 * i + 3] * inv);
        o.z = pack_bf16x2(acc[8 * i + 4] * inv, acc[8 * i + 5] * inv);
        o.w = pack_bf16x2(acc[8 * i + 6] * inv, acc[8 * i + 7] * inv);
        reinterpret_cast<uint4*>(op)[i] = o;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}

}  // namespace

int encoder_attention_tc(const bf16* qkv, bf16* out, int n_win, int T, int d, int n_head, cudaStream_t stream) {
  if (n_win <= 0) return 0;
  SW_CHECK(d == n_head * DH, "encoder_attention: head dim must be 64 (d=%d heads=%d)", d, n_head);
  static SmemOptIn opt_in;  // per device (host_common.h)
  SW_CUDA_CHECK(opt_in.ensure(encoder_attention_tc_kernel, ATT_SMEM));
  CUtensorMap map;
  if (make_tma_map_2d_bf16(&map, qkv, 3 * (int64_t)d, (int64_t)n_win * T, 3 * (int64_t)d, 64, 128)) return -1;
  dim3 grid((T + TQ - 1) / TQ, n_head, n_win);
  encoder_attention_tc_kernel<<<grid, ATT_THREADS, ATT_SMEM, stream>>>(map, out, T, d);
  SW_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace sw
