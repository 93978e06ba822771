// Device-pointer kernel hooks of the C ABI (tests / bench only).
#include "../../include/sw_whisper.h"
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

namespace {
// Development occupier (tools/dev_chain_occupied.py): holds `gridDim.x` SMs (dynamic shared memory + a register
// footprint that keeps other CTAs out, like a resident cross-attention CTA) for `ns` nanoseconds; `buf` != null:
// additionally streams it (HBM contention). Measures what a decoder layer's latency chain costs on the SMs and the
// HBM share a concurrent cross attention leaves it.
__global__ void __launch_bounds__(512, 1) occupy_kernel(unsigned long long ns, const uint4* __restrict__ buf, size_t n_vec,
                                                       float* sink) {
  extern __shared__ uint8_t occ_smem[];
  float r[96];
#pragma unroll
  for (int i = 0; i < 96; ++i) r[i] = (float)(threadIdx.x + i);
  unsigned long long t0, t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  uint4 acc = make_uint4(0, 0, 0, 0);
  do {
    if (buf) {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const uint4 v = __ldcs(buf + (idx + u * stride) % n_vec);
        acc.x ^= v.x; acc.y ^= v.y; acc.z ^= v.z; acc.w ^= v.w;
      }
      idx += 8 * stride;
    }
#pragma unroll
    for (int i = 0; i < 96; ++i) r[i] = fmaf(r[i], 1.0000001f, 1e-9f);
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  } while (t - t0 < ns);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 96; ++i) s += r[i];
  if (s == 12345.678f || (acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x12345u) sink[0] = s + occ_smem[threadIdx.x];
}
}  // namespace

extern "C" {

int sw_dev_occupy(int n_ctas, int smem_bytes, float ms, size_t stream_bytes) {
  static cudaStream_t st = nullptr;
  static uint4* buf = nullptr;
  static size_t buf_bytes = 0;
  static float* sink = nullptr;
  if (!st) {
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) return -1;
    if (cudaMalloc(&sink, 16) != cudaSuccess) return -1;
  }
  if (n_ctas <= 0) return cudaStreamSynchronize(st) == cudaSuccess ? 0 : -1;  // wait for the occupier to leave
  if (stream_bytes > buf_bytes) {
    if (buf) cudaFree(buf);
    if (cudaMalloc(&buf, stream_bytes) != cudaSuccess) return -1;
    cudaMemsetAsync(buf, 1, stream_bytes, st);
    buf_bytes = stream_bytes;
  }
  if (cudaFuncSetAttribute(occupy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes) != cudaSuccess) return -1;
  occupy_kernel<<<n_ctas, 512, smem_bytes, st>>>((unsigned long long)(ms * 1e6), stream_bytes ? buf : nullptr,
                                                  stream_bytes / 16, sink);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int sw_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    int major = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i);
    if (major == 10) ++ok;
  }
  return ok;
}

int sw_dev_gemm_bf16(const void* dA, const void* dB, void* dC, const float* d_bias,
                     const float* d_residual, int M, int N, int K, int lda, int ldb, int ldc,
                     int flags, int block_n, void* stream) {
  sw::GemmArgs a;
  a.A = static_cast<const __nv_bfloat16*>(dA);
  a.B = static_cast<const __nv_bfloat16*>(dB);
  a.C = dC;
  a.lda = lda;
  a.ldb = ldb;
  a.ldc = ldc;
  a.bias = d_bias;
  a.residual = d_residual;
  a.ldr = ldc;
  a.M = M;
  a.N = N;
  a.K = K;
  a.flags = flags;
  a.block_n = block_n;
  return sw::gemm_bf16_tn(a, static_cast<cudaStream_t>(stream));
}

int sw_dev_skinny_gemm(const void* dX, const void* dW, int R, int N, int K, const float* d_bias, int gelu,
                       void* d_out, float* d_partial, int split, void* stream) {
  if (split <= 0) split = sw::skinny_split_for(N, K);
  return sw::skinny_gemm(static_cast<const sw::bf16*>(dX), K, static_cast<const sw::bf16*>(dW), R, N, K, d_bias,
                         gelu, static_cast<sw::bf16*>(d_out), N, d_partial, split, static_cast<cudaStream_t>(stream));
}
int sw_dev_skinny_split(int N, int K) { return sw::skinny_split_for(N, K); }
// kernel: 0 = what the engine would pick, 1 = mma.sync (skinny_gemm.cu), 2 = tcgen05 (skinny_gemm_tc.cu)
int sw_dev_skinny_gemm_k(int kernel, const void* dX, const void* dW, int R, int N, int K, const float* d_bias, int gelu,
                         void* d_out, float* d_partial, int split, void* stream) {
  const sw::bf16* X = static_cast<const sw::bf16*>(dX);
  const sw::bf16* W = static_cast<const sw::bf16*>(dW);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (kernel == 2) {
    if (split <= 0) split = sw::skinny_tc_split_for(N, K);
    return sw::skinny_gemm_tc(X, K, W, R, N, K, d_bias, gelu, static_cast<sw::bf16*>(d_out), N, d_partial, split, st);
  }
  if (kernel == 1) {
    if (split <= 0) split = sw::skinny_mma_split_for(N, K);
    return sw::skinny_gemm_mma(X, K, W, R, N, K, d_bias, gelu, static_cast<sw::bf16*>(d_out), N, d_partial, split, st);
  }
  if (split <= 0) split = sw::skinny_split_for(N, K);
  return sw::skinny_gemm(X, K, W, R, N, K, d_bias, gelu, static_cast<sw::bf16*>(d_out), N, d_partial, split, st);
}
int sw_dev_skinny_split_k(int kernel, int N, int K) {
  return kernel == 2 ? sw::skinny_tc_split_for(N, K) : kernel == 1 ? sw::skinny_mma_split_for(N, K) : sw::skinny_split_for(N, K);
}
int sw_dev_layer_norm(float* d_x, int rows, int d, const float* g, const float* b, void* d_out_bf16,
                      const float* d_partial, int n_split, const float* d_bias, void* stream) {
  return sw::layer_norm(d_x, rows, d, g, b, static_cast<sw::bf16*>(d_out_bf16), nullptr, d_partial, n_split,
                        (int64_t)rows * d, d_bias, static_cast<cudaStream_t>(stream));
}
int sw_dev_encoder_attention(const void* d_qkv, void* d_out, int n_win, int T, int d, int n_head, void* stream) {
  return sw::encoder_attention_tc(static_cast<const sw::bf16*>(d_qkv), static_cast<sw::bf16*>(d_out), n_win, T, d,
                                  n_head, static_cast<cudaStream_t>(stream));
}
size_t sw_dev_cross_attention_ws_floats(int R, int d, int n_head) { return sw::cross_attention_ws_floats(R, d, n_head); }
int sw_dev_cross_attention(const void* d_q, const void* d_kv, int64_t kv_rows, const int* d_grp_win,
                           const int* d_grp_start, const int* d_grp_count, int n_groups, int max_count, int R,
                           int T, int d, int n_head, float* d_ws, void* d_out, int max_ctas, void* stream) {
  return sw::cross_attention(static_cast<const sw::bf16*>(d_q), static_cast<const sw::bf16*>(d_kv), kv_rows, d_grp_win,
                             d_grp_start, d_grp_count, n_groups, max_count, R, T, d, n_head, d_ws,
                             static_cast<sw::bf16*>(d_out), static_cast<cudaStream_t>(stream), nullptr, 0, max_ctas);
}
int sw_dev_self_attention(const void* d_qkv, const int* d_rows, int R, int d, int n_head, void* d_pool,
                          int layer, int n_layer, void* d_out, void* stream) {
  return sw::self_attention(static_cast<const sw::bf16*>(d_qkv), reinterpret_cast<const sw::DecRow*>(d_rows), R, d,
                            n_head, static_cast<sw::bf16*>(d_pool), layer, n_layer, static_cast<sw::bf16*>(d_out),
                            static_cast<cudaStream_t>(stream));
}
}
