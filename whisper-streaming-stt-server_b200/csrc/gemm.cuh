// GEMM interface shared by the tcgen05 kernel (gemm_tc.cu) and the SIMT kernel (gemm_simt.cu).
//
//   D[z][i][j] = act( sum_k A[z][i][k] * B[z][j][k] + bias ) (+ residual)       i < M, j < N
//
// A and B are K-major ("row-major [rows, K]", leading dimension lda/ldb elements); the weight
// matrices of torch Linear layers ([out, in]) are K-major B operands as they are.  `transposed`
// stores D^T (out[j*ldc + i], bias[i], residual[j*ldres + i]): the decoder's skinny GEMMs run
// "swap-AB" -- the weight is the 128-row M operand, the few live sequences are the N operand.
#pragma once
#include <atomic>

#include "common.cuh"

namespace bw {

struct GemmArgs {
  const void* A = nullptr;  // [Z?][M, K]
  const void* B = nullptr;  // [Z?][N, K]
  void* C = nullptr;
  const float* bias = nullptr;      // fp32
  const float* residual = nullptr;  // fp32
  int M = 0, N = 0, K = 0;
  int lda = 0, ldb = 0, ldc = 0, ldres = 0;
  int Z = 1;
  int a_rows = 0, b_rows = 0;  // allocated rows behind A / B (>= M / N) used for the TMA maps; 0 = M / N
  long long a_zstride = 0, b_zstride = 0, c_zstride = 0, bias_zstride = 0, res_zstride = 0;  // elements
  bool gelu = false;
  bool out_fp32 = false;    // else same storage type as the inputs
  bool transposed = false;
  // C (fp32) += A.B^T (+ bias): split-K CTAs reduce with red.global.add.f32 straight into the fp32 residual
  // stream (or a zeroed buffer); `residual` must be null.  tcgen05 path only.
  bool accumulate = false;
  int ksplit = 0;  // 0 = choose
  // ---- decoder LayerNorm fusion (gemm_tc_rows only; see gemm_tc.cu) ----
  // producer: besides C (fp32 residual stream) also store bf16(C) into xb_out (leading dimension ldc) and, per row
  // and 64-column tile, the LayerNorm partials (mean, M2) of the bf16-rounded values: ln_stats_out[row * N/64 + tile]
  void* xb_out = nullptr;
  float2* ln_stats_out = nullptr;
  // consumer: A = bf16(x) un-normalised, B = W * gamma (folded), bias = beta.W + b, ln_c1[n] = sum_k B[n][k]:
  //   out = rstd_r * (acc - mean_r * ln_c1[n]) + bias[n], mean / rstd from ln_stats_in[row * K/64 + tile]
  const float2* ln_stats_in = nullptr;
  const float* ln_c1 = nullptr;
  float ln_eps = 1e-5f;
};

// The kernel a GEMM runs on and its parameter: K split of the cluster split-K and row kernels (1 = the unsplit row
// kernel), tile width BN of the plain tile kernel, 0 for the pair and SIMT kernels.
enum class GemmKernel : int { none = 0, pair = 1, splitk = 2, rows = 3, tile = 4, simt = 5 };
struct GemmRoute {
  GemmKernel kernel = GemmKernel::none;
  int param = 0;
};

// bf16 inputs, fp32 accumulate, tcgen05.mma + TMEM + TMA. Throws on CUDA errors.  Same as
// gemm_tc_launch(g, gemm_tc_choose(g), stream).
void gemm_tc_bf16(const GemmArgs& g, cudaStream_t stream);
// The tcgen05 kernel gemm_tc_bf16 runs for `g`: host only (shape, operand strides and the B200W_* switches).
GemmRoute gemm_tc_choose(const GemmArgs& g);
// Why `r` cannot run `g` (nullptr: it can).  The dispatcher only ever picks routes that can.
const char* gemm_tc_route_error(const GemmArgs& g, GemmRoute r);
// Runs `g` on route `r`; throws std::invalid_argument if gemm_tc_route_error(g, r) says it cannot.
void gemm_tc_launch(const GemmArgs& g, GemmRoute r, cudaStream_t stream);
// Row GEMM of the decoder step (M = live hypotheses): always the push-reduced split-K kernel, any M (more waves for
// many rows).  The only kernel that understands the LayerNorm-fusion fields of GemmArgs.  N % 64 == 0 required.
void gemm_tc_rows(const GemmArgs& g, cudaStream_t stream);
// SIMT tiled GEMM: T = float (validation mode) or bf16 (fallback / cross-check).
template <typename T> void gemm_simt(const GemmArgs& g, cudaStream_t stream);

extern std::atomic<long long> g_kernel_launches;  // counted by every launcher in this library

}  // namespace bw
