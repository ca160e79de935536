// tcgen05 GEMM for sm_100a: TMA (cp.async.bulk.tensor, SWIZZLE_128B) -> shared -> tcgen05.mma
// (cta_group::1, kind::f16, M=128, N=BN) with the fp32 accumulator in TMEM -> tcgen05.ld ->
// fused bias / GELU / residual epilogue.  Warp roles: warp 0 = TMA producer, warp 1 = TMEM
// allocator + single-thread MMA issuer, warps 2..5 = epilogue (one TMEM lane quarter each).
//
// Replaces the cuBLAS GEMMs that upstream `whisper.model.Linear` / `Conv1d` dispatch to from
// `TorchWhisperBackend.transcribe` (reference stt_server/model/backends/torch_whisper.py:55);
// see SURVEY.md section 2.2 rows K2/K4.
#include <cuda.h>

#include <stdlib.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <unordered_map>

#include "gemm.cuh"

namespace bw {

std::atomic<long long> g_kernel_launches{0};
thread_local bool tl_pdl = false;
unsigned long long* g_trace_dev = nullptr;

namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 B = one SWIZZLE_128B row

struct GemmDev {
  void* C;
  const float* bias;
  const float* residual;
  int M, N, K;
  int ldc, ldres;
  long long c_zstride, bias_zstride, res_zstride;
  int a_z_bcast, b_z_bcast;
  int gelu, out_fp32, transposed;
  int accumulate, ksplit;
  unsigned long long* trace;  // debug timeline (null = off)
  // LayerNorm fusion of the decoder row GEMMs (rows kernel only)
  bf16* xb;               // producer: bf16 copy of C
  float2* st_out;         // producer: [row][N / 64] (mean, M2) of the bf16-rounded outputs of each 64-column tile
  const float2* st_in;    // consumer: [row][K / 64]
  const float* c1;        // consumer: row sums of the folded weight
  int st_in_tiles;
  float ln_eps;
  int vec8 = 0;           // pair kernel: C / residual rows are 32-byte aligned -> 256-bit epilogue loads and stores
  int res_prefetch = 0;   // pair kernel: L2-prefetch the residual rows of a tile before waiting for its accumulator
};

template <int BN, int STAGES>
struct SmemLayout {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kBarOffset = STAGES * kStageBytes;
  static constexpr int kTotal = kBarOffset + 256 + 1024;  // + barriers + alignment slack
};

template <int BN, int STAGES, int MINB>
__global__ void __launch_bounds__(192, MINB)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmDev p) {
  using L = SmemLayout<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BN;
  const int m0 = blockIdx.y * BM;
  const int z = blockIdx.z / p.ksplit;
  const int ks = blockIdx.z - z * p.ksplit;
  const int total_kb = (p.K + BK - 1) / BK;
  const int kb0 = (int)((long long)ks * total_kb / p.ksplit);           // balanced split: every CTA gets >= 1 block
  const int num_kb = (int)((long long)(ks + 1) * total_kb / p.ksplit) - kb0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, BN);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  unsigned long long* const trace = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 ? p.trace : nullptr;
  if (threadIdx.x == 0) trace_mark(trace, (6u << 24) | 1);
  pdl_trigger();
  pdl_wait();
  if (threadIdx.x == 0) trace_mark(trace, (6u << 24) | 2);

  if (warp == 0) {
    if (lane == 0) {
      const int za = p.a_z_bcast ? 0 : z;
      const int zb = p.b_z_bcast ? 0 : z;
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % STAGES;
        const uint32_t phase = (kb / STAGES) & 1;
        mbar_wait(&empty_bar[s], phase ^ 1);
        uint8_t* sa = smem + s * L::kStageBytes;
        uint8_t* sb = sa + L::kABytes;
        mbar_arrive_expect_tx(&full_bar[s], L::kStageBytes);
        tma_load_3d(sa, &tmA, &full_bar[s], (kb0 + kb) * BK, m0, za);
        tma_load_3d(sb, &tmB, &full_bar[s], (kb0 + kb) * BK, n0, zb);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, 0, 0);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % STAGES;
        const uint32_t phase = (kb / STAGES) & 1;
        mbar_wait(&full_bar[s], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + s * L::kStageBytes);
        const uint32_t sb = sa + L::kABytes;
        const uint64_t adesc = umma_smem_desc_sw128(sa, 16, 1024);
        const uint64_t bdesc = umma_smem_desc_sw128(sb, 16, 1024);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          // +32 B per UMMA_K=16 step inside the 128 B swizzle row (descriptor address units of 16 B)
          umma_f16(tmem_base, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
        }
        umma_commit(&empty_bar[s]);  // frees the smem stage once these MMAs have read it
      }
      umma_commit(tmem_full_bar);    // accumulator complete
    }
    __syncwarp();
  } else {
    // ---- epilogue: 4 warps, warp (w & 3) owns TMEM lanes [32*(w&3), +32) ----
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    const int i = m0 + row;
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const float* bias = (p.bias && ks == 0) ? p.bias + (long long)z * p.bias_zstride : nullptr;
    const float* res = p.residual ? p.residual + (long long)z * p.res_zstride : nullptr;
    const bool row_ok = i < p.M;
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      const int j0 = n0 + c * 32;
      if (j0 >= p.N) break;  // warp-uniform
      uint32_t r[32];
      tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(c * 32), r);
      tmem_ld_wait();
      float v[32];
      if (!p.transposed) {
        const bool full = (j0 + 32 <= p.N);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float x = __uint_as_float(r[j]);
          if (bias && (full || j0 + j < p.N)) x += __ldg(bias + j0 + j);
          if (p.gelu) x = gelu_erf_fast(x);
          v[j] = x;
        }
        if (row_ok) {
          if (res) {
            const float* rr = res + (long long)i * p.ldres + j0;
            if (full && ((p.ldres & 3) == 0)) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const float4 t = *reinterpret_cast<const float4*>(rr + j);
                v[j] += t.x; v[j + 1] += t.y; v[j + 2] += t.z; v[j + 3] += t.w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j0 + j < p.N) v[j] += rr[j];
            }
          }
          if (p.accumulate) {
            float* o = reinterpret_cast<float*>(p.C) + (long long)z * p.c_zstride + (long long)i * p.ldc + j0;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j0 + j < p.N) atomicAdd(o + j, v[j]);
          } else if (p.out_fp32) {
            float* o = reinterpret_cast<float*>(p.C) + (long long)z * p.c_zstride + (long long)i * p.ldc + j0;
            if (full && ((p.ldc & 3) == 0)) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j0 + j < p.N) o[j] = v[j];
            }
          } else {
            bf16* o = reinterpret_cast<bf16*>(p.C) + (long long)z * p.c_zstride + (long long)i * p.ldc + j0;
            if (full && ((p.ldc & 7) == 0)) {
#pragma unroll
              for (int j = 0; j < 32; j += 8) {
                uint4 t;
                t.x = pack_bf16x2(v[j], v[j + 1]);
                t.y = pack_bf16x2(v[j + 2], v[j + 3]);
                t.z = pack_bf16x2(v[j + 4], v[j + 5]);
                t.w = pack_bf16x2(v[j + 6], v[j + 7]);
                *reinterpret_cast<uint4*>(o + j) = t;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j0 + j < p.N) o[j] = __float2bfloat16(v[j]);
            }
          }
        }
      } else {
        // D^T: out[j*ldc + i]; consecutive lanes = consecutive i -> coalesced per j
        const float b = (bias && row_ok) ? __ldg(bias + i) : 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float x = __uint_as_float(r[j]) + b;
          if (p.gelu) x = gelu_erf_fast(x);
          if (row_ok && j0 + j < p.N) {
            if (res) x += res[(long long)(j0 + j) * p.ldres + i];
            if (p.accumulate)
              atomicAdd((reinterpret_cast<float*>(p.C) + (long long)z * p.c_zstride) + (long long)(j0 + j) * p.ldc + i, x);
            else if (p.out_fp32)
              (reinterpret_cast<float*>(p.C) + (long long)z * p.c_zstride)[(long long)(j0 + j) * p.ldc + i] = x;
            else
              (reinterpret_cast<bf16*>(p.C) + (long long)z * p.c_zstride)[(long long)(j0 + j) * p.ldc + i] = __float2bfloat16(x);
          }
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (threadIdx.x == 0) trace_mark(trace, (6u << 24) | 8);
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, BN);
  }
}


// ------------------------------------------------------------------------------------------------
// Split-K over a thread-block cluster (KS CTAs along K per 128x128 output tile), for GEMMs whose M x N
// tile count cannot fill the 148 SMs -- the decoder step's skinny GEMMs (M = live sequences) above all.
// Each CTA accumulates its K range in TMEM, parks the fp32 tile in its own shared memory (re-using the
// pipeline stages), the cluster synchronises, and CTA rank r reduces tile rows [r*128/KS, (r+1)*128/KS)
// across all peers through distributed shared memory and runs the normal bias / GELU / residual epilogue.
// No atomics, deterministic summation order, every weight byte still streamed from HBM exactly once.
__device__ __forceinline__ float4 ld_dsmem_f4(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local_smem_addr), "r"(rank));
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(remote) : "memory");
  return v;
}

template <int KS>
__global__ void __launch_bounds__(192, 2)
gemm_tc_splitk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmDev p) {
  constexpr int BN = 128, STAGES = 3;
  using L = SmemLayout<BN, STAGES>;
  static_assert(STAGES * L::kStageBytes >= BM * BN * 4, "reduction tile must fit in the pipeline stages");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BN;
  const int m0 = blockIdx.y * BM;
  const int z = blockIdx.z / KS;
  const int ks = (int)cluster_ctarank();  // == blockIdx.z % KS for cluster dims (1, 1, KS)
  const int total_kb = (p.K + BK - 1) / BK;
  const int kb0 = (int)((long long)ks * total_kb / KS);
  const int num_kb = (int)((long long)(ks + 1) * total_kb / KS) - kb0;  // >= 1: host guarantees KS <= total_kb
  unsigned long long* const trace = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 ? p.trace : nullptr;
  const unsigned ttag = (1u << 24) | (gridDim.x << 8);
  if (threadIdx.x == 0) trace_mark(trace, ttag | 0);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, BN);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  // PDL: let the next kernel start its prologue, pull this CTA's slice of the WEIGHT operand (B, never written
  // during a step) towards L2 while the preceding kernel is still draining, then wait for it.
  pdl_trigger();
  if (warp == 0 && lane == 0) {
    const int zb = p.b_z_bcast ? 0 : z;
    for (int kb = 0; kb < num_kb; ++kb) tma_prefetch_l2_3d(&tmB, (kb0 + kb) * BK, n0, zb);
  }
  if (threadIdx.x == 0) trace_mark(trace, ttag | 1);
  pdl_wait();
  if (threadIdx.x == 0) trace_mark(trace, ttag | 2);

  if (warp == 0) {
    if (lane == 0) {
      const int za = p.a_z_bcast ? 0 : z;
      const int zb = p.b_z_bcast ? 0 : z;
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % STAGES;
        const uint32_t phase = (kb / STAGES) & 1;
        mbar_wait(&empty_bar[s], phase ^ 1);
        uint8_t* sa = smem + s * L::kStageBytes;
        uint8_t* sb = sa + L::kABytes;
        mbar_arrive_expect_tx(&full_bar[s], L::kStageBytes);
        tma_load_3d(sa, &tmA, &full_bar[s], (kb0 + kb) * BK, m0, za);
        tma_load_3d(sb, &tmB, &full_bar[s], (kb0 + kb) * BK, n0, zb);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, 0, 0);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % STAGES;
        const uint32_t phase = (kb / STAGES) & 1;
        mbar_wait(&full_bar[s], phase);
        if (kb == 0) trace_mark(trace, ttag | 3);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + s * L::kStageBytes);
        const uint32_t sb = sa + L::kABytes;
        const uint64_t adesc = umma_smem_desc_sw128(sa, 16, 1024);
        const uint64_t bdesc = umma_smem_desc_sw128(sb, 16, 1024);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k)
          umma_f16(tmem_base, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
        umma_commit(&empty_bar[s]);
      }
      umma_commit(tmem_full_bar);
    }
    __syncwarp();
  } else {
    // park the partial tile: red[row][f4 ^ (row & 31)] (float4 granules; conflict-free for a warp of rows)
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    mbar_wait(tmem_full_bar, 0);  // all MMAs retired -> the stage buffers are free to be overwritten
    if (threadIdx.x == 64) trace_mark(trace, ttag | 4);
    tc_fence_after();
    float4* red = reinterpret_cast<float4*>(smem);
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      uint32_t r[32];
      tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(c * 32), r);
      tmem_ld_wait();
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const int f4 = c * 8 + g;
        red[row * 32 + (f4 ^ (row & 31))] = make_float4(__uint_as_float(r[g * 4]), __uint_as_float(r[g * 4 + 1]),
                                                        __uint_as_float(r[g * 4 + 2]), __uint_as_float(r[g * 4 + 3]));
      }
    }
    tc_fence_before();
    if (threadIdx.x == 64) trace_mark(trace, ttag | 5);
  }
  cluster_sync_all();  // every thread of every CTA in the cluster
  if (threadIdx.x == 64) trace_mark(trace, ttag | 6);
  if (warp >= 2) {
    constexpr int RPC = BM / KS;  // tile rows reduced by this CTA
    const int t = threadIdx.x - 64;
    const float* bias = p.bias ? p.bias + (long long)z * p.bias_zstride : nullptr;
    const float* res = p.residual ? p.residual + (long long)z * p.res_zstride : nullptr;
    const uint32_t red_base = smem_u32(smem);
    for (int e = t; e < RPC * 32; e += 128) {
      const int row = ks * RPC + (e >> 5);
      const int f4 = e & 31;
      const uint32_t off = red_base + (uint32_t)((row * 32 + (f4 ^ (row & 31))) * 16);
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int pr = 0; pr < KS; ++pr) {
        const float4 v = ld_dsmem_f4(off, (uint32_t)pr);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
      const int i = m0 + row;
      const int j0 = n0 + f4 * 4;
      if (i >= p.M || j0 >= p.N) continue;
      float v[4] = {acc.x, acc.y, acc.z, acc.w};
      const bool full = (j0 + 4 <= p.N);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (!full && j0 + q >= p.N) continue;
        float x = v[q];
        if (bias) x += __ldg(bias + (p.transposed ? i : j0 + q));
        if (p.gelu) x = gelu_erf_fast(x);
        if (res) x += p.transposed ? res[(long long)(j0 + q) * p.ldres + i] : res[(long long)i * p.ldres + j0 + q];
        v[q] = x;
      }
      if (p.transposed) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (j0 + q >= p.N) continue;
          const long long oi = (long long)z * p.c_zstride + (long long)(j0 + q) * p.ldc + i;
          if (p.out_fp32) reinterpret_cast<float*>(p.C)[oi] = v[q];
          else reinterpret_cast<bf16*>(p.C)[oi] = __float2bfloat16(v[q]);
        }
      } else {
        const long long oi = (long long)z * p.c_zstride + (long long)i * p.ldc + j0;
        if (p.out_fp32) {
          float* o = reinterpret_cast<float*>(p.C) + oi;
          if (full && ((p.ldc & 3) == 0)) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
          else
            for (int q = 0; q < 4; ++q) if (j0 + q < p.N) o[q] = v[q];
        } else {
          bf16* o = reinterpret_cast<bf16*>(p.C) + oi;
          if (full && ((p.ldc & 3) == 0)) {
            uint2 w;
            w.x = pack_bf16x2(v[0], v[1]);
            w.y = pack_bf16x2(v[2], v[3]);
            *reinterpret_cast<uint2*>(o) = w;
          } else
            for (int q = 0; q < 4; ++q) if (j0 + q < p.N) o[q] = __float2bfloat16(v[q]);
        }
      }
    }
  }
  if (threadIdx.x == 64) trace_mark(trace, ttag | 7);
  cluster_sync_all();  // peers may still be reading this CTA's shared memory
  if (threadIdx.x == 64) trace_mark(trace, ttag | 8);
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, BN);
  }
}


// ------------------------------------------------------------------------------------------------
// Split-K v2 for the decoder step's row GEMMs (M = live hypotheses <= a few hundred, N a multiple of 64).
// The in-situ timeline (tools/trace_step.py, profiles/r1_trace_notes.md) showed the v1 kernel spending 4-6 of its
// ~10 us in the reduction: DSMEM *loads* plus the bias / residual loads sit on a serial latency chain.  Here
//   * partial tiles are PUSHED: each epilogue thread reads its accumulator row from TMEM and stores it straight
//     into the shared memory of the CTA that owns the row (st.shared::cluster, fire and forget);
//   * one cluster barrier later every CTA sums its rows from LOCAL shared memory in fixed order (deterministic);
//   * bias / residual for the elements a thread will finalise are loaded right after the dependency wait, i.e.
//     underneath the TMA + MMA phase;
//   * the first weight tiles are requested before griddepcontrol.wait (weights never change inside a step);
//   * 128x64 tiles with a private 32 KB reduction area: 105 KB per CTA, two CTAs per SM, so N = 5120 at KS = 2
//     (160 CTAs) or N = 1280 at KS = 8 (160 CTAs) are a single wave.
constexpr int R_BN = 64, R_STAGES = 3;
constexpr int R_A_BYTES = BM * BK * 2, R_B_BYTES = R_BN * BK * 2, R_STAGE_BYTES = R_A_BYTES + R_B_BYTES;
constexpr int R_SLOT_OFF = R_STAGES * R_STAGE_BYTES;
constexpr int R_SLOT_BYTES = BM * R_BN * 4;
constexpr int R_BAR_OFF = R_SLOT_OFF + R_SLOT_BYTES;
constexpr int R_SMEM_TOTAL = R_BAR_OFF + 128 + 1024;

__device__ __forceinline__ void st_dsmem_f4(uint32_t remote_addr, float a, float b, float c, float d) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(remote_addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

template <int KS>
__global__ void __launch_bounds__(192, 2)
gemm_tc_rows_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmDev p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + R_BAR_OFF);
  uint64_t* empty_bar = full_bar + R_STAGES;
  uint64_t* tmem_full_bar = empty_bar + R_STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * R_BN, m0 = blockIdx.y * BM;
  const int z = blockIdx.z / KS;
  const int ks = KS == 1 ? 0 : (int)cluster_ctarank();  // == blockIdx.z % KS for cluster dims (1, 1, KS)
  const int total_kb = (p.K + BK - 1) / BK;
  const int kb0 = (int)((long long)ks * total_kb / KS);
  const int num_kb = (int)((long long)(ks + 1) * total_kb / KS) - kb0;  // >= 1: host guarantees KS <= total_kb
  const int za = p.a_z_bcast ? 0 : z, zb = p.b_z_bcast ? 0 : z;
  unsigned long long* const trace = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 ? p.trace : nullptr;
  const unsigned ttag = (1u << 24) | (gridDim.x << 8);
  if (threadIdx.x == 0) trace_mark(trace, ttag | 0);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < R_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, R_BN);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_trigger();
  const int n_pre = min(num_kb, R_STAGES);
  if (warp == 0 && lane == 0) {
    for (int kb = 0; kb < n_pre; ++kb) {  // weight tiles of the first stages: in flight before the dependency resolves
      mbar_arrive_expect_tx(&full_bar[kb], R_STAGE_BYTES);
      tma_load_3d(smem + kb * R_STAGE_BYTES + R_A_BYTES, &tmB, &full_bar[kb], (kb0 + kb) * BK, n0, zb);
    }
    for (int kb = n_pre; kb < num_kb; ++kb) tma_prefetch_l2_3d(&tmB, (kb0 + kb) * BK, n0, zb);
  }
  if (threadIdx.x == 0) trace_mark(trace, ttag | 1);
  pdl_wait();
  if (threadIdx.x == 0) trace_mark(trace, ttag | 2);

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % R_STAGES;
        uint8_t* sa = smem + s * R_STAGE_BYTES;
        if (kb >= n_pre) {
          mbar_wait(&empty_bar[s], ((kb / R_STAGES) & 1) ^ 1);
          mbar_arrive_expect_tx(&full_bar[s], R_STAGE_BYTES);
          tma_load_3d(sa + R_A_BYTES, &tmB, &full_bar[s], (kb0 + kb) * BK, n0, zb);
        }
        tma_load_3d(sa, &tmA, &full_bar[s], (kb0 + kb) * BK, m0, za);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(BM, R_BN, 0, 0);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % R_STAGES;
        mbar_wait(&full_bar[s], (kb / R_STAGES) & 1);
        if (kb == 0) trace_mark(trace, ttag | 3);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + s * R_STAGE_BYTES);
        const uint64_t adesc = umma_smem_desc_sw128(sa, 16, 1024);
        const uint64_t bdesc = umma_smem_desc_sw128(sa + R_A_BYTES, 16, 1024);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k)
          umma_f16(tmem_base, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
        umma_commit(&empty_bar[s]);
      }
      umma_commit(tmem_full_bar);
    }
    __syncwarp();
  }

  if constexpr (KS == 1) {
    // No split: the accumulator in TMEM is final.  Used for the step's WIDE consumer GEMMs (qkv, mlp.0) once the rows fill
    // more than one M tile (beam batches): tiles x 2 CTAs would not be co-resident, one wave of full-K CTAs is.
    // One epilogue thread per accumulator row: LayerNorm statistics of the row, then 64 columns straight to global memory.
    if (warp >= 2) {
      const int wq = warp & 3;
      const int gi = m0 + wq * 32 + lane;
      const bool row_ok = gi < p.M;
      float mean = 0.f, rstd = 1.f;
      if (p.st_in && row_ok) {
        const float2* sp = p.st_in + (long long)gi * p.st_in_tiles;
        float ms = 0.f;
        for (int i = 0; i < p.st_in_tiles; ++i) ms += sp[i].x;
        mean = ms / (float)p.st_in_tiles;
        float m2 = 0.f;
        for (int i = 0; i < p.st_in_tiles; ++i) { const float2 q = sp[i]; m2 += q.y + 64.f * (q.x - mean) * (q.x - mean); }
        rstd = rsqrtf(m2 / (64.f * (float)p.st_in_tiles) + p.ln_eps);
      }
      mbar_wait(tmem_full_bar, 0);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < R_BN / 32; ++c) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(c * 32), r);
        tmem_ld_wait();
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const int j0 = n0 + c * 32 + g * 4;
          if (!row_ok || j0 >= p.N) continue;
          float v[4] = {__uint_as_float(r[g * 4]), __uint_as_float(r[g * 4 + 1]), __uint_as_float(r[g * 4 + 2]), __uint_as_float(r[g * 4 + 3])};
          if (p.st_in) {
            const float4 c1 = __ldg(reinterpret_cast<const float4*>(p.c1 + j0));
            v[0] = rstd * (v[0] - mean * c1.x); v[1] = rstd * (v[1] - mean * c1.y);
            v[2] = rstd * (v[2] - mean * c1.z); v[3] = rstd * (v[3] - mean * c1.w);
          }
          if (p.bias) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + (long long)z * p.bias_zstride + j0));
            v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
          }
          if (p.gelu) {
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = gelu_erf_fast(v[q]);
          }
          if (p.residual) {
            const float4 rr = *reinterpret_cast<const float4*>(p.residual + (long long)z * p.res_zstride + (long long)gi * p.ldres + j0);
            v[0] += rr.x; v[1] += rr.y; v[2] += rr.z; v[3] += rr.w;
          }
          const long long oi = (long long)z * p.c_zstride + (long long)gi * p.ldc + j0;
          if (p.out_fp32) *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.C) + oi) = make_float4(v[0], v[1], v[2], v[3]);
          else *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(p.C) + oi) = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
        }
      }
      tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
      tc_fence_after();
      tmem_dealloc(tmem_base, R_BN);
    }
    return;
  }
  // ---- epilogue threads: what this thread will finalise after the reduction ----
  constexpr int RPC = BM / KS;      // tile rows owned (reduced + stored) by each CTA of the cluster
  constexpr int NI = RPC / 8;       // float4 granules per epilogue thread (RPC rows x 16 granules / 128 threads)
  const int t = threadIdx.x - 64;
  float4 resv[NI], biasv[NI], c1v[NI];
  float ln_mean[NI], ln_rstd[NI];
  if (warp >= 2) {
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int e = t + i * 128;
      const int gi = m0 + ks * RPC + (e >> 4), c4 = e & 15, j0 = n0 + c4 * 4;
      const bool ok = gi < p.M && j0 < p.N;
      biasv[i] = (p.bias && ok) ? __ldg(reinterpret_cast<const float4*>(p.bias + (long long)z * p.bias_zstride + j0)) : make_float4(0.f, 0.f, 0.f, 0.f);
      resv[i] = (p.residual && ok) ? *reinterpret_cast<const float4*>(p.residual + (long long)z * p.res_zstride + (long long)gi * p.ldres + j0)
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
      c1v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      ln_mean[i] = 0.f; ln_rstd[i] = 1.f;
      if (p.st_in) {
        // LayerNorm statistics of row gi from the producer's per-tile partials.  The 16 lanes that share a row each
        // fetch up to two tiles (K <= 2048) and combine them with Chan's formula through shuffles (all lanes take part).
        c1v[i] = ok ? __ldg(reinterpret_cast<const float4*>(p.c1 + j0)) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float2* sp = p.st_in + (long long)gi * p.st_in_tiles;
        const bool row_ok = gi < p.M;
        const float2 p0 = (row_ok && c4 < p.st_in_tiles) ? sp[c4] : make_float2(0.f, 0.f);
        const float2 p1 = (row_ok && c4 + 16 < p.st_in_tiles) ? sp[c4 + 16] : make_float2(0.f, 0.f);
        float ms = p0.x + p1.x;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) ms += __shfl_xor_sync(0xffffffffu, ms, o);
        const float mean = ms / (float)p.st_in_tiles;
        float m2 = 0.f;
        if (c4 < p.st_in_tiles) m2 += p0.y + 64.f * (p0.x - mean) * (p0.x - mean);
        if (c4 + 16 < p.st_in_tiles) m2 += p1.y + 64.f * (p1.x - mean) * (p1.x - mean);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) m2 += __shfl_xor_sync(0xffffffffu, m2, o);
        ln_mean[i] = mean;
        ln_rstd[i] = rsqrtf(m2 / (64.f * (float)p.st_in_tiles) + p.ln_eps);
      }
    }
    // ---- push my accumulator row into the owner CTA's reduction area: slots[ks][row % RPC][granule ^ (row & 15)] ----
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    const int owner = row / RPC, lr = row % RPC;
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(smem + R_SLOT_OFF) + (uint32_t)((ks * RPC + lr) * 256)), "r"((uint32_t)owner));
    mbar_wait(tmem_full_bar, 0);
    if (threadIdx.x == 64) trace_mark(trace, ttag | 4);
    tc_fence_after();
#pragma unroll
    for (int c = 0; c < R_BN / 32; ++c) {
      uint32_t r[32];
      tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(c * 32), r);
      tmem_ld_wait();
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const int f4 = c * 8 + g;
        st_dsmem_f4(remote + (uint32_t)((f4 ^ (lr & 15)) << 4), __uint_as_float(r[g * 4]), __uint_as_float(r[g * 4 + 1]),
                    __uint_as_float(r[g * 4 + 2]), __uint_as_float(r[g * 4 + 3]));
      }
    }
    tc_fence_before();
    if (threadIdx.x == 64) trace_mark(trace, ttag | 5);
  }
  cluster_sync_all();  // release/acquire: every partial row has landed in its owner's shared memory
  if (threadIdx.x == 64) trace_mark(trace, ttag | 6);
  if (warp >= 2) {
    const float4* slots = reinterpret_cast<const float4*>(smem + R_SLOT_OFF);
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int e = t + i * 128;
      const int lr = e >> 4, c4 = e & 15;
      const int gi = m0 + ks * RPC + lr, j0 = n0 + c4 * 4;
      float4 acc = slots[(0 * RPC + lr) * 16 + (c4 ^ (lr & 15))];
#pragma unroll
      for (int pr = 1; pr < KS; ++pr) {
        const float4 v = slots[(pr * RPC + lr) * 16 + (c4 ^ (lr & 15))];
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
      const bool ok = gi < p.M && j0 < p.N;  // no early exit: the statistics below use warp shuffles
      float v[4] = {acc.x, acc.y, acc.z, acc.w};
      if (p.st_in) {  // out = rstd * (x.W' - mean * sum_k W') + (beta.W + b)
        const float mu = ln_mean[i], rs = ln_rstd[i];
        v[0] = rs * (v[0] - mu * c1v[i].x); v[1] = rs * (v[1] - mu * c1v[i].y);
        v[2] = rs * (v[2] - mu * c1v[i].z); v[3] = rs * (v[3] - mu * c1v[i].w);
      }
      v[0] += biasv[i].x; v[1] += biasv[i].y; v[2] += biasv[i].z; v[3] += biasv[i].w;
      if (p.gelu) {
#pragma unroll
        for (int q = 0; q < 4; ++q) v[q] = gelu_erf_fast(v[q]);
      }
      v[0] += resv[i].x; v[1] += resv[i].y; v[2] += resv[i].z; v[3] += resv[i].w;
      const long long oi = (long long)z * p.c_zstride + (long long)gi * p.ldc + j0;
      const uint32_t b01 = pack_bf16x2(v[0], v[1]), b23 = pack_bf16x2(v[2], v[3]);
      if (ok) {
        if (p.out_fp32) *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.C) + oi) = make_float4(v[0], v[1], v[2], v[3]);
        else *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(p.C) + oi) = make_uint2(b01, b23);
        if (p.xb) *reinterpret_cast<uint2*>(p.xb + oi) = make_uint2(b01, b23);
      }
      if (p.st_out) {
        // LayerNorm partials of this row's 64-column tile, over the bf16-ROUNDED values (what the consumer GEMM will
        // actually multiply): tile mean, then centred second moment; the 16 lanes of the row reduce by shuffles
        const float r0 = __uint_as_float(b01 << 16), r1 = __uint_as_float(b01 & 0xffff0000u);
        const float r2 = __uint_as_float(b23 << 16), r3 = __uint_as_float(b23 & 0xffff0000u);
        float sm = (r0 + r1) + (r2 + r3);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
        const float tm = sm * (1.f / 64.f);
        float dv = (r0 - tm) * (r0 - tm) + (r1 - tm) * (r1 - tm) + (r2 - tm) * (r2 - tm) + (r3 - tm) * (r3 - tm);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) dv += __shfl_xor_sync(0xffffffffu, dv, o);
        if (ok && c4 == 0) p.st_out[(long long)gi * gridDim.x + blockIdx.x] = make_float2(tm, dv);
      }
    }
    if (threadIdx.x == 64) trace_mark(trace, ttag | 7);
  }
  if (warp == 1) {  // every epilogue thread read its TMEM row before the cluster barrier
    tc_fence_after();
    tmem_dealloc(tmem_base, R_BN);
  }
}


// ------------------------------------------------------------------------------------------------
// Persistent CTA-pair GEMM (the encoder / cross-KV workhorse): cluster (2,1,1), tcgen05.mma.cta_group::2 with
// M=256 N=256 per pair, so each SM stages 128 rows of A and 128 rows of B per k-block (32 KB for 128x256x64
// MACs = 64 B/clk/SM, half of what 128x128 single-CTA tiles pull through L2 and shared memory).
// 6-stage TMA ring, two 256-column TMEM accumulators per SM: the epilogue of tile i overlaps the main
// loop of tile i+1.  warp 0 = TMA producer (both CTAs; bytes are credited to the leader's barrier),
// warp 1 = MMA issuer (leader CTA only), warp 2 = TMEM allocator, warps 4..11 = epilogue.
// 256-bit global accesses (LDG / STG .256 on sm_100): an epilogue thread owns one accumulator ROW, so every access of a warp
// touches 32 different lines; with 32 bytes per thread each instruction moves whole sectors (a float4 is half a sector, which
// doubles the LSU transactions and makes every store a partial-sector write for L2 to merge).
__device__ __forceinline__ void ldg256(const float* ptr, float* v) {
  asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(ptr));
}
__device__ __forceinline__ void stg256(float* ptr, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "l"(ptr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void stg256_bf16x16(bf16* ptr, const float* v) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "l"(ptr), "r"(pack_bf16x2(v[0], v[1])), "r"(pack_bf16x2(v[2], v[3])), "r"(pack_bf16x2(v[4], v[5])),
                  "r"(pack_bf16x2(v[6], v[7])), "r"(pack_bf16x2(v[8], v[9])), "r"(pack_bf16x2(v[10], v[11])),
                  "r"(pack_bf16x2(v[12], v[13])), "r"(pack_bf16x2(v[14], v[15])) : "memory");
}

constexpr int P_STAGES = 6;
constexpr int P_STAGE_BYTES = 2 * BM * BK * 2;  // A half + B half
constexpr int P_BAR_OFF = P_STAGES * P_STAGE_BYTES;
constexpr int P_SMEM_TOTAL = P_BAR_OFF + 256 + 1024;

__global__ void __launch_bounds__(384, 1)
gemm_tc_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmDev p,
                    int m_pairs, int n_tiles, int n_pair_tiles_total) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + P_BAR_OFF);
  uint64_t* empty_bar = full_bar + P_STAGES;
  uint64_t* tmem_full_bar = empty_bar + P_STAGES;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;     // [2] (used on the leader)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int num_kb = (p.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < P_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], 2); }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc_2sm(tmem_ptr_smem, 512);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  auto tile_coords = [&](int t, int& m0, int& n0, int& z) {
    const int per_z = m_pairs * n_tiles;
    z = t / per_z;
    const int r = t - z * per_z;
    n0 = (r / m_pairs) * 256;  // m fastest: pairs running together share the weight tile in L2
    m0 = (r % m_pairs) * 256;
  };

  if (warp == 0) {
    if (lane == 0) {
      int it = 0;
      for (int t = pair; t < n_pair_tiles_total; t += n_pairs) {
        int m0, n0, z;
        tile_coords(t, m0, n0, z);
        const int za = p.a_z_bcast ? 0 : z, zb = p.b_z_bcast ? 0 : z;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % P_STAGES;
          mbar_wait(&empty_bar[s], ((it / P_STAGES) & 1) ^ 1);
          uint8_t* sa = smem + s * P_STAGE_BYTES;
          uint8_t* sb = sa + BM * BK * 2;
          if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * P_STAGE_BYTES);  // both CTAs' bytes land here
          tma_load_3d_2sm(sa, &tmA, &full_bar[s], kb * BK, m0 + (int)rank * BM, za);
          tma_load_3d_2sm(sb, &tmB, &full_bar[s], kb * BK, n0 + (int)rank * BM, zb);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (leader && lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(256, 256, 0, 0);
      int it = 0, ti = 0;
      for (int t = pair; t < n_pair_tiles_total; t += n_pairs, ++ti) {
        const int a = ti & 1;
        mbar_wait(&tmem_empty_bar[a], ((ti >> 1) & 1) ^ 1);  // both CTAs' epilogues drained this accumulator
        tc_fence_after();
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % P_STAGES;
          mbar_wait(&full_bar[s], (it / P_STAGES) & 1);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + s * P_STAGE_BYTES);
          const uint32_t sb = sa + BM * BK * 2;
          const uint64_t adesc = umma_smem_desc_sw128(sa, 16, 1024);
          const uint64_t bdesc = umma_smem_desc_sw128(sb, 16, 1024);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            umma_f16_2sm(tmem_base + a * 256, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
          umma_commit_2sm(&empty_bar[s]);
        }
        umma_commit_2sm(&tmem_full_bar[a]);
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // 8 epilogue warps: two per TMEM lane quarter, each draining 128 of the accumulator's 256 columns
    const int wq = warp & 3;
    const int chalf = (warp - 4) >> 2;
    const int row = wq * 32 + lane;
    int ti = 0;
    for (int t = pair; t < n_pair_tiles_total; t += n_pairs, ++ti) {
      int m0, n0, z;
      tile_coords(t, m0, n0, z);
      const int a = ti & 1;
      const int i = m0 + (int)rank * BM + row;
      const bool row_ok = i < p.M;
      const float* bias = p.bias ? p.bias + (long long)z * p.bias_zstride : nullptr;
      const float* res = p.residual ? p.residual + (long long)z * p.res_zstride : nullptr;
      if (res && row_ok && p.res_prefetch) {
        // the residual rows this thread will add come from HBM: ask for them while the main loop of the tile still runs
        const float* rr = res + (long long)i * p.ldres + n0 + chalf * 128;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (n0 + chalf * 128 + k * 32 < p.N) asm volatile("prefetch.global.L2 [%0];" :: "l"(rr + k * 32));
      }
      mbar_wait(&tmem_full_bar[a], (ti >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int c = chalf * 4; c < chalf * 4 + 4; ++c) {
        const int j0 = n0 + c * 32;
        if (j0 >= p.N) break;  // warp-uniform
        uint32_t r[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(a * 256 + c * 32), r);
        tmem_ld_wait();
        const bool full = (j0 + 32 <= p.N);
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (bias) {
          if (full) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {  // same address in every lane: one broadcast transaction per float4
              const float4 q = __ldg(reinterpret_cast<const float4*>(bias + j0 + j));
              v[j] += q.x; v[j + 1] += q.y; v[j + 2] += q.z; v[j + 3] += q.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j0 + j < p.N) v[j] += __ldg(bias + j0 + j);
          }
        }
        if (p.gelu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = gelu_erf_fast(v[j]);
        }
        if (row_ok) {
        if (res) {
          const float* rr = res + (long long)i * p.ldres + j0;
          if (full && p.vec8) {
            float q[32];
#pragma unroll
            for (int j = 0; j < 32; j += 8) ldg256(rr + j, q + j);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += q[j];
          } else if (full && ((p.ldres & 3) == 0)) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 q = *reinterpret_cast<const float4*>(rr + j);
              v[j] += q.x; v[j + 1] += q.y; v[j + 2] += q.z; v[j + 3] += q.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j0 + j < p.N) v[j] += rr[j];
          }
        }
        if (p.out_fp32) {
          float* o = reinterpret_cast<float*>(p.C) + (long long)z * p.c_zstride + (long long)i * p.ldc + j0;
          if (full && p.vec8) {
#pragma unroll
            for (int j = 0; j < 32; j += 8) stg256(o + j, v + j);
          } else if (full && ((p.ldc & 3) == 0)) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j0 + j < p.N) o[j] = v[j];
          }
        } else {
          bf16* o = reinterpret_cast<bf16*>(p.C) + (long long)z * p.c_zstride + (long long)i * p.ldc + j0;
          if (full && p.vec8) {
            stg256_bf16x16(o, v);
            stg256_bf16x16(o + 16, v + 16);
          } else if (full && ((p.ldc & 7) == 0)) {
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              uint4 q;
              q.x = pack_bf16x2(v[j], v[j + 1]); q.y = pack_bf16x2(v[j + 2], v[j + 3]);
              q.z = pack_bf16x2(v[j + 4], v[j + 5]); q.w = pack_bf16x2(v[j + 6], v[j + 7]);
              *reinterpret_cast<uint4*>(o + j) = q;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j0 + j < p.N) o[j] = __float2bfloat16(v[j]);
          }
        }
        }
      }
      // this CTA's 256 epilogue threads are done with accumulator `a` -> one arrival on the leader's barrier
      tc_fence_before();
      asm volatile("bar.sync 2, 256;" ::: "memory");
      if (threadIdx.x == 128) mbar_arrive_cluster(&tmem_empty_bar[a], 0);
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// ---- host side: tensor maps (driver entry point fetched through the runtime; no -lcuda) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !p)
      throw CudaError("cudaGetDriverEntryPoint(cuTensorMapEncodeTiled) failed");
    fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

struct MapKey {
  const void* ptr; int rows, K, ld, Z; long long zstride; int box_rows;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && rows == o.rows && K == o.K && ld == o.ld && Z == o.Z && zstride == o.zstride && box_rows == o.box_rows;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    auto mix = [&](long long v) { h ^= (size_t)v + 0x9e3779b97f4a7c15ULL + (h << 6) + (h >> 2); };
    mix(k.rows); mix(k.K); mix(k.ld); mix(k.Z); mix(k.zstride); mix(k.box_rows);
    return h;
  }
};

}  // namespace

// bf16 [Z][rows, K] K-major operand -> 3D tiled map {K, rows, Z}, box {64, box_rows, 1}, SWIZZLE_128B.
CUtensorMap make_operand_map(const void* ptr, int rows, int K, int ld, int Z, long long zstride, int box_rows) {
  static std::mutex mu;
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  MapKey key{ptr, rows, K, ld, Z, zstride, box_rows};
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
  }
  BW_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA operand must be 16-byte aligned");
  BW_CHECK((ld % 8) == 0, "TMA operand leading dimension must be a multiple of 8 bf16");
  CUtensorMap m;
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)(Z > 0 ? Z : 1)};
  long long zs = (Z > 1 && zstride > 0) ? zstride : (long long)rows * ld;
  BW_CHECK((zs % 8) == 0, "TMA operand batch stride must be a multiple of 8 bf16");
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)zs * 2};
  cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw CudaError("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
  std::lock_guard<std::mutex> g(mu);
  if (cache.size() > 65536) cache.clear();
  cache.emplace(key, m);
  return m;
}

// Generic bf16 3D tiled map {inner, rows, outer} with a {box_inner, box_rows, 1} SWIZZLE_128B box (box_inner * 2 B = 128 B).
CUtensorMap make_box_map(const void* ptr, int inner, int rows, int outer, long long row_stride, long long outer_stride,
                         int box_inner, int box_rows) {
  BW_CHECK(box_inner == 64, "SWIZZLE_128B box must be 64 bf16 wide");
  BW_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && (row_stride % 8) == 0 && (outer_stride % 8) == 0, "TMA alignment");
  CUtensorMap m;
  cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)rows, (cuuint64_t)outer};
  cuuint64_t strides[2] = {(cuuint64_t)row_stride * 2, (cuuint64_t)outer_stride * 2};
  cuuint32_t box[3] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw CudaError("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
  return m;
}

namespace {
template <int BN, int STAGES, int MINB>
void launch(const GemmArgs& g, cudaStream_t stream) {
  using L = SmemLayout<BN, STAGES>;
  static std::atomic<unsigned long long> attr_set{0};  // per-device bit
  auto kern = gemm_tc_kernel<BN, STAGES, MINB>;
  int dev = 0;
  BW_CUDA(cudaGetDevice(&dev));
  if (!(attr_set.load() >> dev & 1ull)) {
    BW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    attr_set.fetch_or(1ull << dev);
  }
  const bool a_bcast = (g.Z > 1 && g.a_zstride == 0), b_bcast = (g.Z > 1 && g.b_zstride == 0);
  CUtensorMap tmA = make_operand_map(g.A, g.a_rows > g.M ? g.a_rows : g.M, g.K, g.lda, a_bcast ? 1 : g.Z, g.a_zstride, BM);
  CUtensorMap tmB = make_operand_map(g.B, g.b_rows > g.N ? g.b_rows : g.N, g.K, g.ldb, b_bcast ? 1 : g.Z, g.b_zstride, BN);
  GemmDev p;
  p.C = g.C; p.bias = g.bias; p.residual = g.residual;
  p.M = g.M; p.N = g.N; p.K = g.K; p.ldc = g.ldc; p.ldres = g.ldres;
  p.c_zstride = g.c_zstride; p.bias_zstride = g.bias_zstride; p.res_zstride = g.res_zstride;
  p.a_z_bcast = a_bcast; p.b_z_bcast = b_bcast;
  p.gelu = g.gelu; p.out_fp32 = g.out_fp32; p.transposed = g.transposed;
  p.accumulate = g.accumulate;
  p.trace = g_trace_dev;
  p.xb = nullptr; p.st_out = nullptr; p.st_in = nullptr; p.c1 = nullptr; p.st_in_tiles = 0; p.ln_eps = 0.f;
  const int total_kb = (g.K + BK - 1) / BK;
  int ksplit = 1;
  if (g.accumulate) {
    BW_CHECK(!g.residual && !g.gelu, "accumulate GEMM takes no residual / activation");
    const long long tiles = (long long)((g.N + BN - 1) / BN) * ((g.M + BM - 1) / BM) * g.Z;
    ksplit = g.ksplit > 0 ? g.ksplit : (int)std::max<long long>(1, std::min<long long>(total_kb / 2, (2 * 148 + tiles - 1) / tiles));
    ksplit = std::max(1, std::min(ksplit, total_kb));
  }
  p.ksplit = ksplit;
  dim3 grid((g.N + BN - 1) / BN, (g.M + BM - 1) / BM, g.Z * ksplit);
  launch_kernel(kern, grid, dim3(192), L::kTotal, stream, tmA, tmB, p);
  ++g_kernel_launches;
}

template <int KS>
void launch_splitk(const GemmArgs& g, cudaStream_t stream) {
  constexpr int BN = 128, STAGES = 3;
  using L = SmemLayout<BN, STAGES>;
  static std::atomic<unsigned long long> attr_set{0};
  auto kern = gemm_tc_splitk_kernel<KS>;
  int dev = 0;
  BW_CUDA(cudaGetDevice(&dev));
  if (!(attr_set.load() >> dev & 1ull)) {
    BW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    attr_set.fetch_or(1ull << dev);
  }
  const bool a_bcast = (g.Z > 1 && g.a_zstride == 0), b_bcast = (g.Z > 1 && g.b_zstride == 0);
  CUtensorMap tmA = make_operand_map(g.A, g.a_rows > g.M ? g.a_rows : g.M, g.K, g.lda, a_bcast ? 1 : g.Z, g.a_zstride, BM);
  CUtensorMap tmB = make_operand_map(g.B, g.b_rows > g.N ? g.b_rows : g.N, g.K, g.ldb, b_bcast ? 1 : g.Z, g.b_zstride, BN);
  GemmDev p;
  p.C = g.C; p.bias = g.bias; p.residual = g.residual;
  p.M = g.M; p.N = g.N; p.K = g.K; p.ldc = g.ldc; p.ldres = g.ldres;
  p.c_zstride = g.c_zstride; p.bias_zstride = g.bias_zstride; p.res_zstride = g.res_zstride;
  p.a_z_bcast = a_bcast; p.b_z_bcast = b_bcast;
  p.gelu = g.gelu; p.out_fp32 = g.out_fp32; p.transposed = g.transposed;
  p.accumulate = 0; p.ksplit = KS;
  p.trace = g_trace_dev;
  p.xb = nullptr; p.st_out = nullptr; p.st_in = nullptr; p.c1 = nullptr; p.st_in_tiles = 0; p.ln_eps = 0.f;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((g.N + BN - 1) / BN, (g.M + BM - 1) / BM, g.Z * KS);
  cfg.blockDim = dim3(192);
  cfg.dynamicSmemBytes = L::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = KS;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = tl_pdl ? 2 : 1;
  BW_CUDA(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, p));
  ++g_kernel_launches;
}

template <int KS>
void launch_rows(const GemmArgs& g, cudaStream_t stream) {
  static std::atomic<unsigned long long> attr_set{0};
  auto kern = gemm_tc_rows_kernel<KS>;
  int dev = 0;
  BW_CUDA(cudaGetDevice(&dev));
  if (!(attr_set.load() >> dev & 1ull)) {
    BW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, R_SMEM_TOTAL));
    attr_set.fetch_or(1ull << dev);
  }
  const bool a_bcast = (g.Z > 1 && g.a_zstride == 0), b_bcast = (g.Z > 1 && g.b_zstride == 0);
  CUtensorMap tmA = make_operand_map(g.A, g.a_rows > g.M ? g.a_rows : g.M, g.K, g.lda, a_bcast ? 1 : g.Z, g.a_zstride, BM);
  CUtensorMap tmB = make_operand_map(g.B, g.b_rows > g.N ? g.b_rows : g.N, g.K, g.ldb, b_bcast ? 1 : g.Z, g.b_zstride, R_BN);
  GemmDev p;
  p.C = g.C; p.bias = g.bias; p.residual = g.residual;
  p.M = g.M; p.N = g.N; p.K = g.K; p.ldc = g.ldc; p.ldres = g.ldres;
  p.c_zstride = g.c_zstride; p.bias_zstride = g.bias_zstride; p.res_zstride = g.res_zstride;
  p.a_z_bcast = a_bcast; p.b_z_bcast = b_bcast;
  p.gelu = g.gelu; p.out_fp32 = g.out_fp32; p.transposed = 0;
  p.accumulate = 0; p.ksplit = KS;
  p.trace = g_trace_dev;
  p.xb = reinterpret_cast<bf16*>(g.xb_out); p.st_out = g.ln_stats_out; p.st_in = g.ln_stats_in; p.c1 = g.ln_c1;
  p.st_in_tiles = g.K / 64; p.ln_eps = g.ln_eps;
  if (g.ln_stats_in) BW_CHECK(g.ln_c1 && g.K % 64 == 0 && g.K / 64 <= 32 && g.Z == 1, "LayerNorm-fused GEMM needs K % 64 == 0, K <= 2048");
  if (g.ln_stats_out || g.xb_out) BW_CHECK(g.N % 64 == 0 && g.Z == 1 && g.out_fp32, "LayerNorm producer GEMM needs N % 64 == 0 and an fp32 C");
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((g.N + R_BN - 1) / R_BN, (g.M + BM - 1) / BM, g.Z * KS);
  cfg.blockDim = dim3(192);
  cfg.dynamicSmemBytes = R_SMEM_TOTAL;
  cfg.stream = stream;
  if (KS == 1) BW_CHECK(!g.xb_out && !g.ln_stats_out, "the unsplit row GEMM has no LayerNorm-producer epilogue");
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = KS;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = tl_pdl ? 2 : 1;
  BW_CUDA(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, p));
  ++g_kernel_launches;
}

void launch_pair(const GemmArgs& g, cudaStream_t stream) {
  static std::atomic<unsigned long long> attr_set{0};
  int dev = 0;
  BW_CUDA(cudaGetDevice(&dev));
  if (!(attr_set.load() >> dev & 1ull)) {
    BW_CUDA(cudaFuncSetAttribute(gemm_tc_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM_TOTAL));
    attr_set.fetch_or(1ull << dev);
  }
  const bool a_bcast = (g.Z > 1 && g.a_zstride == 0), b_bcast = (g.Z > 1 && g.b_zstride == 0);
  CUtensorMap tmA = make_operand_map(g.A, g.a_rows > g.M ? g.a_rows : g.M, g.K, g.lda, a_bcast ? 1 : g.Z, g.a_zstride, BM);
  CUtensorMap tmB = make_operand_map(g.B, g.b_rows > g.N ? g.b_rows : g.N, g.K, g.ldb, b_bcast ? 1 : g.Z, g.b_zstride, BM);
  GemmDev p;
  p.C = g.C; p.bias = g.bias; p.residual = g.residual;
  p.M = g.M; p.N = g.N; p.K = g.K; p.ldc = g.ldc; p.ldres = g.ldres;
  p.c_zstride = g.c_zstride; p.bias_zstride = g.bias_zstride; p.res_zstride = g.res_zstride;
  p.a_z_bcast = a_bcast; p.b_z_bcast = b_bcast;
  p.gelu = g.gelu; p.out_fp32 = g.out_fp32; p.transposed = 0; p.accumulate = 0; p.ksplit = 1;
  p.trace = nullptr;
  p.xb = nullptr; p.st_out = nullptr; p.st_in = nullptr; p.c1 = nullptr; p.st_in_tiles = 0; p.ln_eps = 0.f;
  {
    static const bool no_vec8 = getenv("B200W_NO_VEC8") != nullptr;
    const long long c_elems = g.out_fp32 ? 8 : 16;  // elements per 32 bytes of C
    auto aligned32 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 31) == 0; };
    p.vec8 = !no_vec8 && aligned32(g.C) && g.ldc % c_elems == 0 && g.c_zstride % c_elems == 0 &&
             (!g.residual || (aligned32(g.residual) && g.ldres % 8 == 0 && g.res_zstride % 8 == 0));
    static const bool no_prefetch = getenv("B200W_NO_RES_PREFETCH") != nullptr;
    p.res_prefetch = !no_prefetch && g.residual != nullptr;
  }
  const int m_pairs = (g.M + 255) / 256, n_tiles = (g.N + 255) / 256;
  const int total = m_pairs * n_tiles * g.Z;
  static int sm_count = 0;
  if (!sm_count) BW_CUDA(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev));
  const int n_pairs = std::min(total, sm_count / 2);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * n_pairs);
  cfg.blockDim = dim3(384);
  cfg.dynamicSmemBytes = P_SMEM_TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  BW_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_pair_kernel, tmA, tmB, p, m_pairs, n_tiles, total));
  ++g_kernel_launches;
}
}  // namespace

void gemm_tc_rows(const GemmArgs& g, cudaStream_t stream) {
  BW_CHECK(g.M > 0 && g.N > 0 && g.K > 0 && g.Z > 0, "empty GEMM");
  BW_CHECK(!g.transposed && !g.accumulate && (g.N % 4) == 0 && (g.ldc % 4) == 0 && (!g.residual || (g.ldres % 4) == 0),
           "row GEMM needs N, ldc, ldres % 4 == 0");
  const long long tiles64 = (long long)((g.M + BM - 1) / BM) * ((g.N + R_BN - 1) / R_BN) * g.Z;
  const int total_kb = (g.K + BK - 1) / BK;
  int ks = 8;  // keep the grid within one co-resident wave when possible (see gemm_tc_bf16)
  while (ks > 2 && (tiles64 * ks > (ks == 8 ? 256 : 288) || total_kb < 2 * ks)) ks >>= 1;
  // (capping KS at 4 / 2 so that every SM hosts one CTA was measured slower: 7.20 -> 7.26 / 7.75 ms per step)
  BW_CHECK(total_kb >= ks, "K too small for the row GEMM");
  // More than one M tile (beam batches: 320 rows = 3 tiles) and a wide N: even KS = 2 is two waves.  One wave of unsplit
  // CTAs instead (consumer / plain epilogues only; K <= 2048 keeps the serial main loop short).
  static const bool no_unsplit = getenv("B200W_ROWS_NO_UNSPLIT") != nullptr;
  if (!no_unsplit && ks == 2 && tiles64 * 2 > 288 && tiles64 <= 296 && total_kb <= 32 && !g.xb_out && !g.ln_stats_out)
    return launch_rows<1>(g, stream);
  if (ks == 8) return launch_rows<8>(g, stream);
  if (ks == 4) return launch_rows<4>(g, stream);
  return launch_rows<2>(g, stream);
}

GemmRoute gemm_tc_choose(const GemmArgs& g) {
  // Tile choice: 128x256 (fewer smem bytes per MMA) when it still fills the 148 SMs, else
  // 128x128 with two CTAs per SM; tiny N (swap-AB decode) uses the narrowest tile that covers it.
  const long long mt = (g.M + BM - 1) / BM;
  {
    // enough 256x256 pair tiles to fill the 74 SM pairs -> persistent cta_group::2 kernel
    static const bool no_pair = getenv("B200W_NO_PAIR") != nullptr;
    const long long pair_tiles = (long long)((g.M + 255) / 256) * ((g.N + 255) / 256) * g.Z;
    if (!no_pair && !g.transposed && !g.accumulate && pair_tiles >= 60 && g.N >= 256) return {GemmKernel::pair, 0};
  }
  if (!g.accumulate && g.N > 64 && g.ksplit >= 0) {
    // too few 128x128 tiles for 148 SMs -> split K over a cluster (DSMEM reduction, full epilogue)
    const long long tiles = mt * ((g.N + 127) / 128) * g.Z;
    const int total_kb = (g.K + BK - 1) / BK;
    static const bool no_splitk = getenv("B200W_NO_SPLITK") != nullptr;
    static const bool no_rows = getenv("B200W_SPLITK_V1") != nullptr;
    if (tiles < 120 && total_kb >= 4 && !no_splitk && !no_rows && !g.transposed && (g.N % 4) == 0 && (g.ldc % 4) == 0 &&
        (!g.residual || (g.ldres % 4) == 0) && (!g.bias || (g.bias_zstride % 4) == 0)) {
      // decoder-step row GEMMs: 128x64 tiles, push-reduced split-K; keep the whole grid co-resident (2 CTAs / SM,
      // clusters packed per GPC: ~256 CTAs at KS = 8, ~288 at KS <= 4)
      const long long tiles64 = mt * ((g.N + R_BN - 1) / R_BN) * g.Z;
      int ks = 8;
      while (ks > 2 && (tiles64 * ks > (ks == 8 ? 256 : 288) || total_kb < 2 * ks)) ks >>= 1;
      if (tiles64 * ks <= 288 && total_kb >= ks) return {GemmKernel::rows, ks};
    }
    if (tiles < 120 && total_kb >= 4 && !no_splitk) {
      int ks = 8;
      while (ks > 2 && (tiles * ks > 640 || total_kb < 2 * ks)) ks >>= 1;
      return {GemmKernel::splitk, ks};
    }
  }
  if (g.N <= 32) return {GemmKernel::tile, 32};
  if (g.N <= 64) return {GemmKernel::tile, 64};
  // 128x128 with two CTAs per SM: one CTA's epilogue overlaps the other's main loop.  (A 128x256 / 1 CTA
  // variant measured slower here -- profiles/r1a_summary.txt; large GEMMs take the persistent pair kernel above.)
  return {GemmKernel::tile, 128};
}

const char* gemm_tc_route_error(const GemmArgs& g, GemmRoute r) {
  const int total_kb = (g.K + BK - 1) / BK;
  switch (r.kernel) {
    case GemmKernel::pair:
      if (r.param != 0) return "the pair kernel takes no parameter";
      if (g.transposed || g.accumulate) return "the pair kernel has no transposed or accumulating epilogue";
      if (g.N < 256) return "the pair kernel needs N >= 256";
      return nullptr;
    case GemmKernel::splitk:
      if (r.param != 2 && r.param != 4 && r.param != 8) return "cluster split-K runs KS = 2, 4 or 8";
      if (g.accumulate) return "cluster split-K has no accumulating epilogue";
      if (total_kb < r.param) return "cluster split-K needs at least KS blocks of 64 along K";
      return nullptr;
    case GemmKernel::rows:
      if (r.param != 1 && r.param != 2 && r.param != 4 && r.param != 8) return "the row kernel runs KS = 1, 2, 4 or 8";
      if (g.transposed || g.accumulate) return "the row kernel has no transposed or accumulating epilogue";
      if ((g.N % 4) != 0 || (g.ldc % 4) != 0 || (g.residual && (g.ldres % 4) != 0) || (g.bias && (g.bias_zstride % 4) != 0))
        return "the row kernel needs N, ldc, ldres and bias_zstride % 4 == 0";
      if (total_kb < r.param) return "the row kernel needs at least KS blocks of 64 along K";
      return nullptr;
    case GemmKernel::tile:
      if (r.param != 32 && r.param != 64 && r.param != 128) return "the tile kernel runs BN = 32, 64 or 128";
      return nullptr;
    default:
      return "not a tcgen05 route";
  }
}

void gemm_tc_launch(const GemmArgs& g, GemmRoute r, cudaStream_t stream) {
  if (const char* why = gemm_tc_route_error(g, r)) throw std::invalid_argument(why);
  switch (r.kernel) {
    case GemmKernel::pair: return launch_pair(g, stream);
    case GemmKernel::splitk:
      if (r.param == 8) return launch_splitk<8>(g, stream);
      if (r.param == 4) return launch_splitk<4>(g, stream);
      return launch_splitk<2>(g, stream);
    case GemmKernel::rows:
      if (r.param == 8) return launch_rows<8>(g, stream);
      if (r.param == 4) return launch_rows<4>(g, stream);
      if (r.param == 2) return launch_rows<2>(g, stream);
      return launch_rows<1>(g, stream);
    default:
      if (r.param == 32) return launch<32, 5, 2>(g, stream);
      if (r.param == 64) return launch<64, 4, 2>(g, stream);
      return launch<128, 3, 2>(g, stream);
  }
}

void gemm_tc_bf16(const GemmArgs& g, cudaStream_t stream) {
  BW_CHECK(g.M > 0 && g.N > 0 && g.K > 0 && g.Z > 0, "empty GEMM");
  BW_CHECK(!g.xb_out && !g.ln_stats_out && !g.ln_stats_in, "LayerNorm-fusion fields are only understood by gemm_tc_rows");
  gemm_tc_launch(g, gemm_tc_choose(g), stream);
}

}  // namespace bw
