// Host-side interface of the tcgen05 GEMM family (implementation: gemm_tcgen05.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sw {

enum GemmFlags : int {
  GEMM_GELU = 1,      // v = gelu_tanh(v) after bias
  GEMM_OUT_F32 = 2,   // C is float (default: bf16)
  GEMM_BIAS_ROW = 4,  // bias indexed by output row (swap-AB use) instead of column
};

// C[b][m][n] = epi( sum_k A[b][m][k] * B[b?][n][k] )   (both operands K-major bf16)
//   epi(v) = [gelu](v + bias) + residual[b][m % res_mod or m][n]
// Row strides (lda/ldb) may describe overlapping rows (the conv stem reads its
// im2col matrix straight out of the activation buffer through the TMA strides).
struct GemmArgs {
  const __nv_bfloat16* A = nullptr;
  int64_t lda = 0;             // elements
  int64_t a_batch_stride = 0;  // elements
  const __nv_bfloat16* B = nullptr;
  int64_t ldb = 0;
  int64_t b_batch_stride = 0;  // 0: B shared by all batches
  void* C = nullptr;
  int64_t ldc = 0;
  int64_t c_batch_stride = 0;
  const float* bias = nullptr;
  const float* residual = nullptr;  // f32
  int64_t ldr = 0;
  int64_t r_batch_stride = 0;
  int res_mod = 0;  // >0: residual row = m % res_mod
  int M = 0, N = 0, K = 0, batch = 1;
  int flags = 0;
  int block_n = 0;  // 0 = auto (64/128/256, or CTA pairs for M >= 2048 at 256); 64/128/256: that single-CTA tile;
                    // 512: CTA pairs (2 x 256)
};

// Enqueue on `stream`. Returns 0 or -1 (see sw_last_error()).
int gemm_bf16_tn(const GemmArgs& args, cudaStream_t stream);

// 2-D bf16 tensor map {inner, rows} with a {box_inner (=64), box_rows} box and 128B swizzle; map_out is a CUtensorMap*
int make_tma_map_2d_bf16(void* map_out, const void* base, int64_t inner, int64_t rows, int64_t ld_elems,
                         int box_inner, int box_rows);

// general 3-D bf16 tensor map (128B swizzle): dims innermost first, strides of dims 1 and 2 in bytes
int make_tma_map_3d_bf16(void* map_out, const void* base, const int64_t dims[3], const int64_t strides_bytes[2],
                         const int box[3]);

// FLOPs actually requested (2*M*N*K*batch) - for roofline accounting.
inline double gemm_flops(const GemmArgs& a) {
  return 2.0 * a.M * (double)a.N * a.K * a.batch;
}

}  // namespace sw
