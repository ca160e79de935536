// Decoder cross-attention, bf16 product path: the HBM-bound kernel of the batched decoder step.
//
// The cached encoder K/V of a segment ([T_enc, 2d] per layer) is streamed ONCE per step for all hypotheses
// (beams) of that segment.  The SM's only job is to keep loads in flight, so the data path is
//   TMA (cp.async.bulk.tensor, SWIZZLE_128B, 6-stage mbarrier ring of 64-key K|V tiles = 96 KB per CTA)
//   -> ldmatrix -> mma.sync.m16n8k16 (q.K^T and P.V; rows 0..7 of the M=16 fragment are the <= 8 hypotheses)
// which needs ~7x fewer instructions per byte than the SIMT version (profiles/r1_xattn_simt_ncu_full.txt).
// One CTA = (head, segment group, T split); 4 consumer warps each own 16 of the 64 keys of a tile and keep
// their own running (max, sum, O); a 5th warp is the TMA producer.  Partials over warps are merged through
// shared memory, partials over T splits through the workspace + dec_cross_combine kernel (attention.cu).
// The 8-bit cross cache (BW_FLAG_CROSS_KV_INT8) has its own kernel below with the same structure, and the kernel that
// writes that cache: its layout (kernels.cuh, CrossKV) is known to these two only.
// Upstream: whisper/model.py MultiHeadAttention.forward with cached cross K/V (kv_cache hooks).
#include <cuda.h>

#include "kernels.cuh"

namespace bw {

CUtensorMap make_box_map(const void* ptr, int inner, int rows, int outer, long long row_stride, long long outer_stride,
                         int box_inner, int box_rows);

namespace {

constexpr int XT = 64;          // keys per tile
constexpr int XSTAGES = 6;
constexpr int XTILE_BYTES = XT * 128;  // one 64x64 bf16 tile
constexpr int XSM_BAR = XSTAGES * 2 * XTILE_BYTES;
constexpr int XSM_RED = XSM_BAR + 128;
constexpr int XSM_TOTAL = XSM_RED + 4 * 8 * 66 * 4 + 1024;
constexpr int kMaxSplitX = 8;

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float* c, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// After the consumer warps parked their (max, sum, O) partials in `red`: merge the 4 warps (thread -> (row, 4 dims)) and
// store the normalised row (one split) or the split's partial for dec_cross_combine_kernel.
__device__ __forceinline__ void merge_warps_and_store(const float* red, int nq, int row0, int h, int n_head, int sp, int n_split, int d,
                                                      bf16* __restrict__ out, float* __restrict__ ws) {
  if (threadIdx.x < 128) {
    const int r = threadIdx.x >> 4, c4 = (threadIdx.x & 15) * 4;
    if (r < nq) {
      float M = -INFINITY;
#pragma unroll
      for (int w = 0; w < 4; ++w) M = fmaxf(M, red[(w * 8 + r) * 66]);
      float num[4] = {0.f, 0.f, 0.f, 0.f}, den = 0.f;
      if (M != -INFINITY) {
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const float* pr = red + (w * 8 + r) * 66;
          const float e = fast_exp2(pr[0] - M);
          den = fmaf(e, pr[1], den);
#pragma unroll
          for (int i = 0; i < 4; ++i) num[i] = fmaf(e, pr[2 + c4 + i], num[i]);
        }
      }
      const int row = row0 + r;
      if (n_split == 1) {
        const float inv = 1.f / den;
        uint2 t;
        t.x = pack_bf16x2(num[0] * inv, num[1] * inv);
        t.y = pack_bf16x2(num[2] * inv, num[3] * inv);
        *reinterpret_cast<uint2*>(out + (long long)row * d + h * 64 + c4) = t;
      } else {
        float* w = ws + (((long long)row * n_head + h) * kMaxSplitX + sp) * 66;
        if (c4 == 0) { w[0] = (M == -INFINITY) ? -INFINITY : M * 0.6931471805599453f; w[1] = den; }  // natural-log max
#pragma unroll
        for (int i = 0; i < 4; ++i) w[2 + c4 + i] = num[i];
      }
    }
  }
}

__global__ void __launch_bounds__(160, 2)
dec_cross_attention_mma_kernel(const __grid_constant__ CUtensorMap tm, const int* __restrict__ group_first_row,
                               const int* __restrict__ group_n_rows, const int* __restrict__ group_xslot,
                               const float* __restrict__ q, int T_enc, int n_layer, int layer, int d, int n_split,
                               bf16* __restrict__ out, float* __restrict__ ws, unsigned long long* trace_buf) {
  extern __shared__ uint8_t smem_raw[];
  unsigned long long* trace = nullptr;
  unsigned ttag = 4u << 24;
  if (threadIdx.x == 0) {
    if ((blockIdx.x | blockIdx.y | blockIdx.z) == 0) trace = trace_buf;
    else if (blockIdx.x == gridDim.x - 1 && blockIdx.y == gridDim.y - 1 && blockIdx.z == gridDim.z - 1) { trace = trace_buf; ttag = 5u << 24; }
  }
  trace_mark(trace, ttag | 1);
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + XSM_BAR);
  uint64_t* empty_bar = full_bar + XSTAGES;
  float* red = reinterpret_cast<float*>(smem + XSM_RED);  // [4 warps][8 rows][66]: m, l, o[64]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x, g = blockIdx.y, sp = blockIdx.z, n_head = gridDim.x;
  const int row0 = group_first_row[g], nq = group_n_rows[g];
  const int chunk = ((T_enc + n_split - 1) / n_split + XT - 1) / XT * XT;
  const int t0 = sp * chunk, t1 = min(T_enc, t0 + chunk);
  const int n_tiles = (t1 - t0 + XT - 1) / XT;  // may be 0 for a trailing split

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm);
    for (int s = 0; s < XSTAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 4); }
    fence_barrier_init();
  }
  __syncthreads();
  // PDL: the cached encoder K/V is never written during a decoder step, so the producer starts streaming it
  // right away; only the consumers (which read q and write out / ws) wait for the preceding kernels.
  pdl_trigger();

  if (warp == 4) {
    if (lane == 0) {
      const int zc = group_xslot[g] * n_layer + layer;
      for (int it = 0; it < n_tiles; ++it) {
        const int s = it % XSTAGES;
        mbar_wait(&empty_bar[s], ((it / XSTAGES) & 1) ^ 1);
        mbar_arrive_expect_tx(&full_bar[s], 2 * XTILE_BYTES);
        uint8_t* ks = smem + s * 2 * XTILE_BYTES;
        tma_load_3d(ks, &tm, &full_bar[s], h * 64, t0 + it * XT, zc);
        tma_load_3d(ks + XTILE_BYTES, &tm, &full_bar[s], d + h * 64, t0 + it * XT, zc);
      }
    }
    __syncwarp();
  } else {
    pdl_wait();
    trace_mark(trace, ttag | 2);
    const int gid = lane >> 2, tig = lane & 3;  // query row (hypothesis) and column pair inside an n-tile
    // A fragments of q (rows 8..15 are zero): 4 k-steps of 16 dims; 1/sqrt(64) folded in (exact in bf16)
    uint32_t qa[4][2];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
      if (gid < nq) {
        const float* qr = q + (long long)(row0 + gid) * d + h * 64 + ks * 16 + tig * 2;
        v0 = qr[0] * 0.125f; v1 = qr[1] * 0.125f; v2 = qr[8] * 0.125f; v3 = qr[9] * 0.125f;
      }
      qa[ks][0] = pack_bf16x2(v0, v1);
      qa[ks][1] = pack_bf16x2(v2, v3);
    }
    const float LOG2E = 1.4426950408889634f;
    float m = -INFINITY, l = 0.f;  // running max (log2 domain) and this thread's partial row sum
    float o[8][4];
#pragma unroll
    for (int nd = 0; nd < 8; ++nd) { o[nd][0] = o[nd][1] = o[nd][2] = o[nd][3] = 0.f; }
    // ldmatrix lane roles
    const int lrow = lane & 7, lmat = lane >> 3;
    for (int it = 0; it < n_tiles; ++it) {
      const int s = it % XSTAGES;
      mbar_wait(&full_bar[s], (it / XSTAGES) & 1);
      const uint32_t kbase = smem_u32(smem + s * 2 * XTILE_BYTES);
      const uint32_t vbase = kbase + XTILE_BYTES;
      // ---- S[16 x 16 keys] = Q . K^T for this warp's keys [warp*16, +16) ----
      float sc[2][4];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
        const int krow = warp * 16 + nt * 8 + lrow;
#pragma unroll
        for (int half = 0; half < 2; ++half) {  // dims [32*half, +32): matrices = 16-byte chunks 4*half + lmat
          uint32_t b0, b1, b2, b3;
          ldsm_x4(kbase + krow * 128 + (((half * 4 + lmat) ^ (krow & 7)) << 4), b0, b1, b2, b3);
          mma_bf16(sc[nt], qa[half * 2][0], 0u, qa[half * 2][1], 0u, b0, b1);
          mma_bf16(sc[nt], qa[half * 2 + 1][0], 0u, qa[half * 2 + 1][1], 0u, b2, b3);
        }
      }
      // ---- online softmax for query row gid over these 16 keys (4 of them in this thread) ----
      const int key0 = t0 + it * XT + warp * 16 + tig * 2;
      float sv[4];
      sv[0] = (key0 < t1) ? sc[0][0] * LOG2E : -INFINITY;
      sv[1] = (key0 + 1 < t1) ? sc[0][1] * LOG2E : -INFINITY;
      sv[2] = (key0 + 8 < t1) ? sc[1][0] * LOG2E : -INFINITY;
      sv[3] = (key0 + 9 < t1) ? sc[1][1] * LOG2E : -INFINITY;
      float mx = fmaxf(fmaxf(sv[0], sv[1]), fmaxf(sv[2], sv[3]));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      const float m_new = fmaxf(m, mx);
      float p[4] = {0.f, 0.f, 0.f, 0.f};
      if (m_new != -INFINITY) {
        const float alpha = fast_exp2(m - m_new);
#pragma unroll
        for (int i = 0; i < 4; ++i) p[i] = fast_exp2(sv[i] - m_new);
        l = l * alpha + (p[0] + p[1]) + (p[2] + p[3]);
        if (alpha != 1.f) {
#pragma unroll
          for (int nd = 0; nd < 8; ++nd) { o[nd][0] *= alpha; o[nd][1] *= alpha; }
        }
        m = m_new;
      }
      const uint32_t pa0 = pack_bf16x2(p[0], p[1]), pa2 = pack_bf16x2(p[2], p[3]);
      // ---- O[16 x 64] += P[16 x 16 keys] . V[16 keys x 64 dims] ----
#pragma unroll
      for (int np = 0; np < 4; ++np) {  // pairs of 8-dim n-tiles
        const int vrow = warp * 16 + (lmat & 1) * 8 + lrow;
        uint32_t b0, b1, b2, b3;
        ldsm_x4_t(vbase + vrow * 128 + (((np * 2 + (lmat >> 1)) ^ (vrow & 7)) << 4), b0, b1, b2, b3);
        mma_bf16(o[np * 2], pa0, 0u, pa2, 0u, b0, b1);
        mma_bf16(o[np * 2 + 1], pa0, 0u, pa2, 0u, b2, b3);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);
    }
    // row sum over the 4 threads of a quad, then park this warp's partial
    l += __shfl_xor_sync(0xffffffffu, l, 1);
    l += __shfl_xor_sync(0xffffffffu, l, 2);
    float* mine = red + (warp * 8 + gid) * 66;
    if (tig == 0) { mine[0] = m; mine[1] = l; }
#pragma unroll
    for (int nd = 0; nd < 8; ++nd) { mine[2 + nd * 8 + tig * 2] = o[nd][0]; mine[2 + nd * 8 + tig * 2 + 1] = o[nd][1]; }
  }
  __syncthreads();
  merge_warps_and_store(red, nq, row0, h, n_head, sp, n_split, d, out, ws);
  trace_mark(trace, ttag | 8);
}

// ------------------------------------------------------------------------------------------------
// 8-bit cross cache (layout: kernels.cuh, next to CrossKV).  Same structure as the kernel above -- a producer warp
// streaming one chunk per 64-key tile (one bulk copy of codes + scales) through an mbarrier ring, four consumer warps
// with their own online softmax, the same T-split workspace -- but the fragments come from int8 codes:
//   * q.K^T on mma.sync f16 (int8 -> f16 is exact): thread (gid, tig) loads the 16 code bytes of dims [tig*16, +16) of
//     one key and uses word ks for k-step ks, so q's A fragment takes dims tig*16 + ks*4 + {0,1 | 2,3} in that order;
//     the S column n of n-tile nt is key (n >> 1)*4 + nt*2 + (n & 1) of the warp's 16, so each thread ends up with the
//     4 consecutive keys tig*4 + j, j = nt*2 + c;
//   * each S column times k_scale[key] (with 1/8 and log2 e folded in), v_scale[key] folded into P;
//   * P.V on mma.sync f16 from the transposed V codes: one 32-bit word = keys tig*4 + 0..3 of one dim, exactly the
//     B fragment for those keys.
constexpr int X8STAGES = 6;
constexpr int X8CH = kCrossInt8ChunkBytes;
constexpr int X8SM_BAR = X8STAGES * X8CH;
constexpr int X8SM_RED = X8SM_BAR + 128;
constexpr int X8SM_TOTAL = X8SM_RED + 4 * 8 * 66 * 4 + 128;
static_assert(X8CH % 128 == 0, "stages stay 128-byte aligned");

__device__ __forceinline__ void bulk_load(void* smem_dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// 4 int8 codes -> f16x2 {b0, b1} and {b2, b3}, exactly: 0x64XX is the f16 1024 + XX, XX = code + 128
__device__ __forceinline__ void i8x4_to_f16x2(uint32_t w, uint32_t& lo, uint32_t& hi) {
  const uint32_t u = w ^ 0x80808080u;
  const uint32_t bias = 0x64806480u;  // 1152, 1152
  asm("sub.rn.f16x2 %0, %1, %2;" : "=r"(lo) : "r"(__byte_perm(u, 0x64646464u, 0x4140)), "r"(bias));
  asm("sub.rn.f16x2 %0, %1, %2;" : "=r"(hi) : "r"(__byte_perm(u, 0x64646464u, 0x4342)), "r"(bias));
}
__device__ __forceinline__ void mma_f16(float* c, uint32_t a0, uint32_t a2, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(0u), "r"(a2), "r"(0u), "r"(b0), "r"(b1));
}

__global__ void __launch_bounds__(160, 3)
dec_cross_attention_int8_kernel(const uint8_t* __restrict__ cache, long long slot_bytes, const int* __restrict__ group_first_row,
                                const int* __restrict__ group_n_rows, const int* __restrict__ group_xslot,
                                const float* __restrict__ q, int T_enc, int layer, int d, int n_split, bf16* __restrict__ out,
                                float* __restrict__ ws, unsigned long long* trace_buf) {
  extern __shared__ uint8_t smem_raw[];
  unsigned long long* trace = nullptr;
  unsigned ttag = 6u << 24;
  if (threadIdx.x == 0) {
    if ((blockIdx.x | blockIdx.y | blockIdx.z) == 0) trace = trace_buf;
    else if (blockIdx.x == gridDim.x - 1 && blockIdx.y == gridDim.y - 1 && blockIdx.z == gridDim.z - 1) { trace = trace_buf; ttag = 7u << 24; }
  }
  trace_mark(trace, ttag | 1);
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~uintptr_t(127));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + X8SM_BAR);
  uint64_t* empty_bar = full_bar + X8STAGES;
  float* red = reinterpret_cast<float*>(smem + X8SM_RED);  // [4 warps][8 rows][66]: m, l, o[64]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x, g = blockIdx.y, sp = blockIdx.z, n_head = gridDim.x;
  const int row0 = group_first_row[g], nq = group_n_rows[g];
  const int chunk = ((T_enc + n_split - 1) / n_split + XT - 1) / XT * XT;
  const int t0 = sp * chunk, t1 = min(T_enc, t0 + chunk);
  const int n_tiles = (t1 - t0 + XT - 1) / XT;  // may be 0 for a trailing split

  if (threadIdx.x == 0) {
    for (int s = 0; s < X8STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 4); }
    fence_barrier_init();
  }
  __syncthreads();
  pdl_trigger();  // the cache is never written during a decoder step: stream it before the preceding kernels finish

  if (warp == 4) {
    if (lane == 0) {
      const int tiles_per_head = (T_enc + XT - 1) / XT;
      const uint8_t* src = cache + group_xslot[g] * slot_bytes +
                           ((long long)(layer * n_head + h) * tiles_per_head + t0 / XT) * X8CH;
      for (int it = 0; it < n_tiles; ++it) {
        const int s = it % X8STAGES;
        mbar_wait(&empty_bar[s], ((it / X8STAGES) & 1) ^ 1);
        mbar_arrive_expect_tx(&full_bar[s], X8CH);
        bulk_load(smem + s * X8CH, src + (long long)it * X8CH, X8CH, &full_bar[s]);
      }
    }
    __syncwarp();
  } else {
    pdl_wait();
    trace_mark(trace, ttag | 2);
    const int gid = lane >> 2, tig = lane & 3;
    // A fragments of q in f16 (rows 8..15 are zero): k-step ks = dims tig*16 + ks*4 + {0, 1} | {2, 3}
    uint32_t qa[4][2];
    {
      float4 v[4] = {};
      if (gid < nq) {
        const float4* qr = reinterpret_cast<const float4*>(q + (long long)(row0 + gid) * d + h * 64 + tig * 16);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) v[ks] = qr[ks];
      }
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) { qa[ks][0] = pack_f16x2(v[ks].x, v[ks].y); qa[ks][1] = pack_f16x2(v[ks].z, v[ks].w); }
    }
    const float SCL = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) and log2 e, applied with k_scale
    float m = -INFINITY, l = 0.f;
    float o[8][4];
#pragma unroll
    for (int nd = 0; nd < 8; ++nd) { o[nd][0] = o[nd][1] = o[nd][2] = o[nd][3] = 0.f; }
    const int kq = warp * 16 + tig * 4;  // this thread's 4 keys of the tile: kq + j
    for (int it = 0; it < n_tiles; ++it) {
      const int s = it % X8STAGES;
      mbar_wait(&full_bar[s], (it / X8STAGES) & 1);
      const uint32_t base = smem_u32(smem + s * X8CH);
      // ---- S[16 x 16 keys] = Q . K^T for this warp's keys ----
      float sc[2][4];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
        const int key = warp * 16 + (gid >> 1) * 4 + nt * 2 + (gid & 1);
        const uint4 kw = lds_v4(base + key * 64 + tig * 16);
        const uint32_t w4[4] = {kw.x, kw.y, kw.z, kw.w};
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          uint32_t b0, b1;
          i8x4_to_f16x2(w4[ks], b0, b1);
          mma_f16(sc[nt], qa[ks][0], qa[ks][1], b0, b1);
        }
      }
      const float4 kscale = lds_f4(base + 8192 + kq * 4);
      const float4 vscale = lds_f4(base + 8448 + kq * 4);
      // ---- online softmax for query row gid over these 16 keys (keys kq + 0..3 in this thread) ----
      const int key0 = t0 + it * XT + kq;
      float sv[4];
      sv[0] = (key0 < t1) ? sc[0][0] * (kscale.x * SCL) : -INFINITY;
      sv[1] = (key0 + 1 < t1) ? sc[0][1] * (kscale.y * SCL) : -INFINITY;
      sv[2] = (key0 + 2 < t1) ? sc[1][0] * (kscale.z * SCL) : -INFINITY;
      sv[3] = (key0 + 3 < t1) ? sc[1][1] * (kscale.w * SCL) : -INFINITY;
      float mx = fmaxf(fmaxf(sv[0], sv[1]), fmaxf(sv[2], sv[3]));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      const float m_new = fmaxf(m, mx);
      float p[4] = {0.f, 0.f, 0.f, 0.f};
      if (m_new != -INFINITY) {
        const float alpha = fast_exp2(m - m_new);
#pragma unroll
        for (int i = 0; i < 4; ++i) p[i] = fast_exp2(sv[i] - m_new);
        l = l * alpha + (p[0] + p[1]) + (p[2] + p[3]);
        if (alpha != 1.f) {
#pragma unroll
          for (int nd = 0; nd < 8; ++nd) { o[nd][0] *= alpha; o[nd][1] *= alpha; }
        }
        m = m_new;
      }
      const uint32_t pa0 = pack_f16x2(p[0] * vscale.x, p[1] * vscale.y), pa2 = pack_f16x2(p[2] * vscale.z, p[3] * vscale.w);
      // ---- O[16 x 64] += (P * v_scale)[16 x 16 keys] . V_codes[16 keys x 64 dims] ----
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        const uint4 vw = lds_v4(base + 4096 + warp * 1024 + hf * 512 + lane * 16);
        const uint32_t w4[4] = {vw.x, vw.y, vw.z, vw.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint32_t b0, b1;
          i8x4_to_f16x2(w4[i], b0, b1);
          mma_f16(o[hf * 4 + i], pa0, pa2, b0, b1);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);
    }
    l += __shfl_xor_sync(0xffffffffu, l, 1);
    l += __shfl_xor_sync(0xffffffffu, l, 2);
    float* mine = red + (warp * 8 + gid) * 66;
    if (tig == 0) { mine[0] = m; mine[1] = l; }
#pragma unroll
    for (int nd = 0; nd < 8; ++nd) { mine[2 + nd * 8 + tig * 2] = o[nd][0]; mine[2 + nd * 8 + tig * 2 + 1] = o[nd][1]; }
  }
  __syncthreads();
  merge_warps_and_store(red, nq, row0, h, n_head, sp, n_split, d, out, ws);
  trace_mark(trace, ttag | 8);
}

// One 64-dim slice: scale = amax / 127, code = nearest integer to x / scale (the residual test makes it exact where the
// rounded quotient sits on the wrong side of a half), clamped to +-127; an all-zero slice is scale 0, codes 0.
__device__ __forceinline__ float int8_scale(float amax) { return amax / 127.f; }
__device__ __forceinline__ int int8_code(float x, float scale) {
  if (scale == 0.f) return 0;
  float r = rintf(x / scale);
  const float e2 = 2.f * fmaf(-r, scale, x);  // x - r * scale exactly (doubled: no rounding of scale / 2 for denormals)
  if (e2 > scale) r += 1.f;
  else if (e2 < -scale) r -= 1.f;
  return (int)fminf(fmaxf(r, -127.f), 127.f);
}
// 64 bf16 (8 x uint4) -> 16 words of 4 codes in dim order; returns the scale
__device__ __forceinline__ float quantize_slice(const uint4* src, uint32_t* words) {
  float x[64];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint4 v = src[i];
    const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) { x[i * 8 + k * 2] = __uint_as_float(u[k] << 16); x[i * 8 + k * 2 + 1] = __uint_as_float(u[k] & 0xffff0000u); }
  }
  float amax = 0.f;
#pragma unroll
  for (int i = 0; i < 64; ++i) amax = fmaxf(amax, fabsf(x[i]));
  const float scale = int8_scale(amax);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    uint32_t w = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) w |= (uint32_t)(int8_code(x[i * 4 + j], scale) & 0xff) << (8 * j);
    words[i] = w;
  }
  return scale;
}

// One CTA per (tile, head, slot * L + layer): thread = (k | v, key of the tile).  The chunk is assembled in shared memory
// and written with coalesced 16-byte stores.
__global__ void __launch_bounds__(128)
cross_kv_int8_write_kernel(const bf16* __restrict__ rows, const int8_t* __restrict__ codes, const float* __restrict__ scales,
                           int T_enc, int d, uint8_t* __restrict__ cache) {
  __shared__ __align__(16) uint8_t ch[X8CH];
  const int tile = blockIdx.x, h = blockIdx.y, z = blockIdx.z, n_head = gridDim.y, n_tiles = gridDim.x;
  const int kv = threadIdx.x >> 6, key = threadIdx.x & 63, pos = tile * XT + key;
  uint32_t words[16];
  float scale = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) words[i] = 0u;
  if (pos < T_enc) {
    const long long r = (long long)z * T_enc + pos;
    if (rows) {
      scale = quantize_slice(reinterpret_cast<const uint4*>(rows + r * 2 * d + kv * d + h * 64), words);
    } else {
      const uint4* src = reinterpret_cast<const uint4*>(codes + r * 2 * d + kv * d + h * 64);
#pragma unroll
      for (int i = 0; i < 4; ++i) { const uint4 v = src[i]; words[i * 4] = v.x; words[i * 4 + 1] = v.y; words[i * 4 + 2] = v.z; words[i * 4 + 3] = v.w; }
      scale = scales[r * 2 * n_head + kv * n_head + h];
    }
  }
  reinterpret_cast<float*>(ch + 8192 + kv * 256)[key] = scale;
  if (kv == 0) {
    uint4* dst = reinterpret_cast<uint4*>(ch + key * 64);
#pragma unroll
    for (int i = 0; i < 4; ++i) dst[i] = make_uint4(words[i * 4], words[i * 4 + 1], words[i * 4 + 2], words[i * 4 + 3]);
  } else {
    uint8_t* vt = ch + 4096 + (key >> 4) * 1024 + ((key >> 2) & 3) * 16 + (key & 3);
#pragma unroll
    for (int dim = 0; dim < 64; ++dim) {
      const int nd = dim >> 3;
      vt[(nd >> 2) * 512 + (dim & 7) * 64 + (nd & 3) * 4] = (uint8_t)(words[dim >> 2] >> (8 * (dim & 3)));
    }
  }
  __syncthreads();
  uint4* out = reinterpret_cast<uint4*>(cache + (((long long)z * n_head + h) * n_tiles + tile) * X8CH);
  for (int i = threadIdx.x; i < X8CH / 16; i += blockDim.x) out[i] = reinterpret_cast<const uint4*>(ch)[i];
}

__global__ void quantize_int8_slices_kernel(const bf16* __restrict__ x, long long n, int8_t* __restrict__ codes, float* __restrict__ scales) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t words[16];
  scales[i] = quantize_slice(reinterpret_cast<const uint4*>(x + i * 64), words);
  uint4* dst = reinterpret_cast<uint4*>(codes + i * 64);
#pragma unroll
  for (int k = 0; k < 4; ++k) dst[k] = make_uint4(words[k * 4], words[k * 4 + 1], words[k * 4 + 2], words[k * 4 + 3]);
}

}  // namespace

void dec_cross_attention_mma(const int* group_first_row, const int* group_n_rows, const int* group_xslot, int n_groups,
                             const float* q, const CrossKV& kv, int n_layer, int layer, int d, int n_head, int n_split,
                             bf16* out, float* ws, cudaStream_t stream) {
  static std::atomic<unsigned long long> attr_set{0};
  int dev = 0;
  BW_CUDA(cudaGetDevice(&dev));
  if (!(attr_set.load() >> dev & 1ull)) {
    BW_CUDA(cudaFuncSetAttribute(dec_cross_attention_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, XSM_TOTAL));
    attr_set.fetch_or(1ull << dev);
  }
  // one map per (cache pointer, geometry); cheap enough to rebuild, but the decoder calls this 32x per step
  static thread_local const void* cached_ptr = nullptr;
  static thread_local int cached_geo[4] = {0, 0, 0, 0};
  static thread_local CUtensorMap cached_tm;
  if (cached_ptr != kv.cache || cached_geo[0] != d || cached_geo[1] != kv.T_enc || cached_geo[2] != kv.n_slots || cached_geo[3] != n_layer) {
    cached_tm = make_box_map(kv.cache, 2 * d, kv.T_enc, kv.n_slots * n_layer, 2LL * d, (long long)kv.T_enc * 2 * d, 64, XT);
    cached_ptr = kv.cache; cached_geo[0] = d; cached_geo[1] = kv.T_enc; cached_geo[2] = kv.n_slots; cached_geo[3] = n_layer;
  }
  const CUtensorMap tm = cached_tm;
  dim3 grid(n_head, n_groups, n_split);
  launch_kernel(dec_cross_attention_mma_kernel, grid, dim3(160), XSM_TOTAL, stream, tm, group_first_row, group_n_rows, group_xslot, q,
                kv.T_enc, n_layer, layer, d, n_split, out, ws, g_trace_dev);
  ++g_kernel_launches;
}

void dec_cross_attention_int8(const int* group_first_row, const int* group_n_rows, const int* group_xslot, int n_groups,
                              const float* q, const CrossKV& kv, int layer, int d, int n_head, int n_split, bf16* out, float* ws,
                              cudaStream_t stream) {
  BW_CHECK(kv.slot_stride == cross_int8_slot_bytes(kv.n_layer, kv.T_enc, n_head), "8-bit cross cache geometry");
  static std::atomic<unsigned long long> attr_set{0};
  int dev = 0;
  BW_CUDA(cudaGetDevice(&dev));
  if (!(attr_set.load() >> dev & 1ull)) {
    BW_CUDA(cudaFuncSetAttribute(dec_cross_attention_int8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, X8SM_TOTAL));
    attr_set.fetch_or(1ull << dev);
  }
  dim3 grid(n_head, n_groups, n_split);
  launch_kernel(dec_cross_attention_int8_kernel, grid, dim3(160), X8SM_TOTAL, stream, reinterpret_cast<const uint8_t*>(kv.cache),
                kv.slot_stride, group_first_row, group_n_rows, group_xslot, q, kv.T_enc, layer, d, n_split, out, ws, g_trace_dev);
  ++g_kernel_launches;
}

void cross_kv_int8_write(const bf16* rows, const int8_t* codes, const float* scales, int n_slots, int n_layer, int T_enc, int d,
                         void* cache, cudaStream_t stream) {
  BW_CHECK(d % 64 == 0 && (rows || (codes && scales)), "cross_kv_int8_write: bad argument");
  dim3 grid((T_enc + XT - 1) / XT, d / 64, n_slots * n_layer);
  cross_kv_int8_write_kernel<<<grid, 128, 0, stream>>>(rows, codes, scales, T_enc, d, reinterpret_cast<uint8_t*>(cache));
  BW_CUDA(cudaGetLastError());
  ++g_kernel_launches;
}

void quantize_int8_slices(const bf16* x, long long n_slices, int8_t* codes, float* scales, cudaStream_t stream) {
  if (n_slices <= 0) return;
  quantize_int8_slices_kernel<<<(unsigned)((n_slices + 127) / 128), 128, 0, stream>>>(x, n_slices, codes, scales);
  BW_CUDA(cudaGetLastError());
  ++g_kernel_launches;
}

}  // namespace bw
