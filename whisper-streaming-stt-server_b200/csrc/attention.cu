// Attention kernels (head dim 64 for every Whisper size).
//  * attn_encoder_simt : non-causal encoder self-attention, SIMT online softmax (fp32 validation mode
//    and cross-check for the tcgen05 kernel in attention_tc.cu).
//  * dec_self_attention : one query per live hypothesis over its paged self-KV (pages of 16 positions per
//    hypothesis slot behind a page table; the beam ancestry table `anc` redirects each position to the beam
//    slot that wrote it).
//  * dec_cross_attention: the decoder step's HBM-bound kernel -- streams the cached encoder K/V of a
//    segment ONCE for all beams of that segment (NQ queries share each 16-byte load), split along T.
// Upstream: whisper/model.py MultiHeadAttention.qkv_attention (SDPA, scale 1/sqrt(64)).
#include <stdlib.h>

#include <type_traits>

#include "kernels.cuh"

namespace bw {

void dec_cross_attention_mma(const int* group_first_row, const int* group_n_rows, const int* group_xslot, int n_groups,
                             const float* q, const CrossKV& kv, int n_layer, int layer, int d, int n_head, int n_split,
                             bf16* out, float* ws, cudaStream_t stream);
void dec_cross_attention_int8(const int* group_first_row, const int* group_n_rows, const int* group_xslot, int n_groups,
                              const float* q, const CrossKV& kv, int layer, int d, int n_head, int n_split, bf16* out, float* ws,
                              cudaStream_t stream);

namespace {

// fp32 validation mode uses the accurate expf; bf16 mode the fast intrinsic
template <typename T> __device__ __forceinline__ float exp_t(float x) { return __expf(x); }
template <> __device__ __forceinline__ float exp_t<float>(float x) { return expf(x); }

// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128)
attn_encoder_simt_kernel(const T* __restrict__ qkv, T* __restrict__ out, int T_len, int n_head) {
  constexpr int QT = 32, KT = 32;
  __shared__ float Qs[QT][65];
  __shared__ float Ks[KT][65];
  __shared__ float Vs[KT][64];
  __shared__ float Ps[QT][KT + 1];
  const int d = n_head * 64;
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * QT;
  const int tid = threadIdx.x;
  const int qi = tid >> 2, part = tid & 3;
  const T* base = qkv + (long long)b * T_len * 3 * d;
  for (int i = tid; i < QT * 64; i += 128) {
    const int r = i >> 6, c = i & 63;
    Qs[r][c] = (q0 + r < T_len) ? to_f(base[(long long)(q0 + r) * 3 * d + h * 64 + c]) * 0.125f : 0.f;
  }
  float m = -INFINITY, l = 0.f;
  float o[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) o[i] = 0.f;
  for (int k0 = 0; k0 < T_len; k0 += KT) {
    __syncthreads();
    for (int i = tid; i < KT * 64; i += 128) {
      const int r = i >> 6, c = i & 63;
      const bool ok = k0 + r < T_len;
      const T* row = base + (long long)(k0 + r) * 3 * d + h * 64 + c;
      Ks[r][c] = ok ? to_f(row[d]) : 0.f;
      Vs[r][c] = ok ? to_f(row[2 * d]) : 0.f;
    }
    __syncthreads();
    float s[8];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int key = part * 8 + j;
      float acc = 0.f;
#pragma unroll 16
      for (int c = 0; c < 64; ++c) acc = fmaf(Qs[qi][c], Ks[key][c], acc);
      s[j] = (k0 + key < T_len) ? acc : -INFINITY;
      mx = fmaxf(mx, s[j]);
    }
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    const float m_new = fmaxf(m, mx);
    const float alpha = (m == -INFINITY) ? 0.f : exp_t<T>(m - m_new);
    float ps = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float p = (s[j] == -INFINITY) ? 0.f : exp_t<T>(s[j] - m_new);
      Ps[qi][part * 8 + j] = p;
      ps += p;
    }
    ps += __shfl_xor_sync(0xffffffffu, ps, 1);
    ps += __shfl_xor_sync(0xffffffffu, ps, 2);
    l = l * alpha + ps;
    m = m_new;
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 16; ++i) o[i] *= alpha;
    for (int key = 0; key < KT; ++key) {
      const float p = Ps[qi][key];
#pragma unroll
      for (int i = 0; i < 16; ++i) o[i] = fmaf(p, Vs[key][part * 16 + i], o[i]);
    }
  }
  if (q0 + qi < T_len) {
    const float inv = 1.f / l;
    T* orow = out + ((long long)b * T_len + q0 + qi) * d + h * 64 + part * 16;
#pragma unroll
    for (int i = 0; i < 16; ++i) orow[i] = from_f<T>(o[i] * inv);
  }
}

// ------------------------------------------------------------------------------------------------
template <typename T> struct Vec16;
template <> struct Vec16<bf16> {
  static constexpr int N = 8;
  __device__ static void load(const bf16* p, float* f) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) { const float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
  }
  // streaming load: cached K/V are touched once per step -> do not pollute L1
  __device__ static void load_stream(const bf16* p, float* f) {
    uint4 u;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "l"(p));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) { const float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
  }
};
template <> struct Vec16<float> {
  static constexpr int N = 4;
  __device__ static void load(const float* p, float* f) {
    const float4 u = __ldg(reinterpret_cast<const float4*>(p));
    f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w;
  }
  __device__ static void load_stream(const float* p, float* f) { load(p, f); }
};

constexpr int kSingleBeamFlag = 0x40000000;  // set in seq_first[s] when the request has one hypothesis (anc == 0)

// One CTA per (head, row).  Fuses the KV append: this row's k/v head slice (fp32 qkv buffer -> T) is written to
// the pool, and keys/values of positions fed in THIS step (the row itself; earlier prefill rows of the same
// sequence) are taken from the qkv buffer instead of the pool, so no ordering between CTAs is needed.
// The cached K/V head slices are staged into shared memory with cp.async (every 16-byte request of a 128-position
// chunk in flight at once: the kernel is a pure HBM stream, 2*t*128 B per CTA), then consumed by 8-lane groups
// with an online softmax; one shared-memory merge at the end.  (The first version walked the keys with dependent
// global loads: 9 us per CTA and 2 waves at context 100 -- tools/trace_step.py.)
// positions staged per pass: 32 / 64 / 128, the smallest that covers the step's longest context (fewer bytes of shared
// memory per CTA = more CTAs per SM: 6 at 128, 9 (register-limited) at 64 and below)
__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
template <typename T> __device__ __forceinline__ void load_smem_vec(const T* p, float* f);
template <> __device__ __forceinline__ void load_smem_vec<bf16>(const bf16* p, float* f) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}
template <> __device__ __forceinline__ void load_smem_vec<float>(const float* p, float* f) {
  const float4 u = *reinterpret_cast<const float4*>(p);
  f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w;
}

template <typename T, int kSelfChunk>
__global__ void __launch_bounds__(128)
dec_self_attention_kernel(const int* __restrict__ row_seq, const int* __restrict__ row_pos, const int* __restrict__ row_bpos,
                          const int* __restrict__ row_page, const float* __restrict__ qkv, T* __restrict__ pool,
                          long long page_stride, int n_ctx, int n_blocks, int n_units, const int* __restrict__ page_table,
                          const int* __restrict__ seq_first, const unsigned char* __restrict__ anc, int layer, int d,
                          T* __restrict__ out, unsigned long long* trace_buf) {
  constexpr int VEC = Vec16<T>::N, LPR = 64 / VEC, RPW = 32 / LPR;
  extern __shared__ __align__(16) unsigned char self_smem[];
  T* Ks = reinterpret_cast<T*>(self_smem);  // [kSelfChunk][64]
  T* Vs = Ks + kSelfChunk * 64;
  __shared__ float part[4][66];
  __shared__ int s_pt[kMaxBeam * kMaxBlocks];  // page table rows of the request's beam slots
  unsigned long long* const trace = ((blockIdx.x | blockIdx.y) == 0 && threadIdx.x == 0) ? trace_buf : nullptr;
  trace_mark(trace, (3u << 24) | 1);
  pdl_trigger();
  // Everything read before the dependency wait was written by earlier STEPS (control block, ancestry, cached K/V),
  // never by the kernels of this step: the first chunk of the cache is already streaming in while the QKV
  // projection that precedes this kernel drains.  Only q and this step's own k/v rows need the wait.
  const int h = blockIdx.x, r = blockIdx.y;
  const int s = row_seq[r], pos = row_pos[r], bpos = row_bpos[r];
  const int sf = seq_first[s];
  const bool single = (sf & kSingleBeamFlag) != 0;
  const int first = sf & ~kSingleBeamFlag;
  const unsigned char* my_anc = anc + (long long)s * n_ctx;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sub = lane % LPR, rg = lane / LPR;
  const int n = pos + 1;
  // Page-table rows of the slots this hypothesis can descend from.  Entries that matter here (blocks holding positions
  // < bpos) were published by EARLIER steps; this step's embed kernel rewrites at most the current block's entry with
  // the value it already has, so reading them before the dependency wait is safe.
  if (bpos > 0) {
    const int nu = single ? 1 : min(kMaxBeam, n_units - first);
    for (int i = threadIdx.x; i < nu * n_blocks; i += 128) s_pt[i] = page_table[(long long)first * n_blocks + i];
    __syncthreads();
  }
  auto stage_cached = [&](int c0, int cn) {
    for (int idx = threadIdx.x; idx < cn * 2 * LPR; idx += 128) {
      const int ch = idx % LPR, kv = (idx / LPR) & 1, tl = idx / (2 * LPR);
      const int t = c0 + tl;
      if (t < bpos) {
        const int page = s_pt[(single ? 0 : my_anc[t]) * n_blocks + t / kPageTokens];
        cp_async_16((kv ? Vs : Ks) + tl * 64 + ch * VEC, pool + (long long)page * page_stride +
                                                               ((long long)(layer * 2 + kv) * kPageTokens + (t % kPageTokens)) * d + h * 64 + ch * VEC);
      }
    }
  };
  stage_cached(0, min(kSelfChunk, n));
  pdl_wait();
  trace_mark(trace, (3u << 24) | 2);
  const float* qrow = qkv + (long long)r * 3 * d + h * 64;
  // fused append: k/v of this row -> its page [layer][k|v][pos % kPageTokens]
  {
    const int c = threadIdx.x & 63, kvsel = threadIdx.x >> 6;  // 0: k, 1: v
    pool[(long long)row_page[r] * page_stride + ((long long)(layer * 2 + kvsel) * kPageTokens + (pos % kPageTokens)) * d + h * 64 + c] =
        from_f<T>(qrow[(1 + kvsel) * d + c]);
  }
  float qf[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) qf[i] = qrow[sub * VEC + i] * 0.125f;
  float m = -INFINITY, l = 0.f, acc[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
  for (int c0 = 0; c0 < n; c0 += kSelfChunk) {
    const int cn = min(kSelfChunk, n - c0);
    if (c0 > 0) {
      __syncthreads();  // the previous chunk has been consumed by every warp
      stage_cached(c0, cn);
    }
    // positions fed in this step: fp32 rows of the qkv buffer, rounded like the pool copy
    for (int idx = threadIdx.x; idx < cn * 2 * LPR; idx += 128) {
      const int ch = idx % LPR, kv = (idx / LPR) & 1, tl = idx / (2 * LPR);
      const int t = c0 + tl;
      if (t >= bpos) {
        T* dst = (kv ? Vs : Ks) + tl * 64 + ch * VEC;
        const float* src = qkv + (long long)(r - (pos - t)) * 3 * d + (1 + kv) * d + h * 64 + ch * VEC;
#pragma unroll
        for (int i = 0; i < VEC; ++i) dst[i] = from_f<T>(src[i]);
      }
    }
    cp_async_wait_all();
    __syncthreads();
    for (int tg = warp * RPW; tg < cn; tg += 4 * RPW) {
      const int tl = tg + rg;
      float kf[VEC], vf[VEC];
      float sc = 0.f;
      if (tl < cn) {
        load_smem_vec<T>(Ks + tl * 64 + sub * VEC, kf);
        load_smem_vec<T>(Vs + tl * 64 + sub * VEC, vf);
#pragma unroll
        for (int i = 0; i < VEC; ++i) sc = fmaf(qf[i], kf[i], sc);
      }
#pragma unroll
      for (int o = LPR / 2; o > 0; o >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, o);
      if (tl < cn) {
        const float m_new = fmaxf(m, sc);
        const float a = exp_t<T>(m - m_new), pr = exp_t<T>(sc - m_new);
        l = l * a + pr;
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] = fmaf(pr, vf[i], acc[i] * a);
        m = m_new;
      }
    }
  }
  // merge the row groups of this warp, then the 4 warps
#pragma unroll
  for (int o = LPR; o < 32; o <<= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), l2 = __shfl_xor_sync(0xffffffffu, l, o);
    const float M = fmaxf(m, m2);
    const float e1 = (m == -INFINITY) ? 0.f : exp_t<T>(m - M), e2 = (m2 == -INFINITY) ? 0.f : exp_t<T>(m2 - M);
    l = l * e1 + l2 * e2;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float a2 = __shfl_xor_sync(0xffffffffu, acc[i], o);
      acc[i] = acc[i] * e1 + a2 * e2;
    }
    m = M;
  }
  if (rg == 0) {
    if (sub == 0) { part[warp][0] = m; part[warp][1] = l; }
#pragma unroll
    for (int i = 0; i < VEC; ++i) part[warp][2 + sub * VEC + i] = acc[i];
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int c = threadIdx.x;
    float M = fmaxf(fmaxf(part[0][0], part[1][0]), fmaxf(part[2][0], part[3][0]));
    float num = 0.f, den = 0.f;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const float e = (part[w][0] == -INFINITY) ? 0.f : exp_t<T>(part[w][0] - M);
      num = fmaf(e, part[w][2 + c], num);
      den = fmaf(e, part[w][1], den);
    }
    out[(long long)r * d + h * 64 + c] = from_f<T>(num / den);
  }
  trace_mark(trace, (3u << 24) | 8);
}

// ------------------------------------------------------------------------------------------------
// v2: one WARP per (row, head), no shared-memory staging and no block-level synchronisation.  The staged kernel above
// keeps 6 (row, head) units resident per SM (32 KB of shared memory each) and pays ~5 dependent latencies per unit
// (profiles/r2_launches_dec64x5.csv: 67 us per layer at 320 rows, 2.7x its HBM bound); here every warp streams its own
// unit with 16 independent 16-byte loads in flight per lane, so ~20 units per SM overlap their latencies.
//   lanes: LPR = 64 / VEC lanes share one position (VEC dims each), PPI = 32 / LPR positions per pass, U passes unrolled.
template <typename T> struct Raw16 { uint4 v; };
template <typename T> __device__ __forceinline__ uint4 ld_raw16(const T* p) {
  uint4 u;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "l"(p));
  return u;
}
template <typename T> __device__ __forceinline__ void unpack16(const uint4& u, float* f);
template <> __device__ __forceinline__ void unpack16<bf16>(const uint4& u, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}
template <> __device__ __forceinline__ void unpack16<float>(const uint4& u, float* f) {
  f[0] = __uint_as_float(u.x); f[1] = __uint_as_float(u.y); f[2] = __uint_as_float(u.z); f[3] = __uint_as_float(u.w);
}

template <typename T>
__global__ void __launch_bounds__(128)
dec_self_attention_warp_kernel(const int* __restrict__ row_seq, const int* __restrict__ row_pos, const int* __restrict__ row_bpos,
                               const int* __restrict__ row_page, const float* __restrict__ qkv, T* __restrict__ pool,
                               long long page_stride, int n_ctx, int n_blocks, int n_units, const int* __restrict__ page_table,
                               const int* __restrict__ seq_first, const unsigned char* __restrict__ anc, int layer, int d,
                               int n_rows, int n_head, T* __restrict__ out, unsigned long long* trace_buf) {
  constexpr int VEC = Vec16<T>::N, LPR = 64 / VEC, PPI = 32 / LPR, U = 8;
  __shared__ int s_pt[4][kMaxBeam * kMaxBlocks];  // page-table rows of each warp's request (its beam slots)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x * 4 + warp;
  unsigned long long* const trace = (unit == 0 && lane == 0) ? trace_buf : nullptr;
  trace_mark(trace, (3u << 24) | 1);
  pdl_trigger();
  if (unit >= n_rows * n_head) return;  // warps are independent: no block-wide barrier below
  const int r = unit / n_head, h = unit - r * n_head;
  // Everything read before the dependency wait was written by earlier STEPS (control block, ancestry, page table
  // entries of blocks that hold positions < bpos, cached K/V); only q and this step's own k/v rows need the wait.
  const int s = row_seq[r], pos = row_pos[r], bpos = row_bpos[r];
  const int sf = seq_first[s];
  const bool single = (sf & kSingleBeamFlag) != 0;
  const int first = sf & ~kSingleBeamFlag;
  const unsigned char* my_anc = anc + (long long)s * n_ctx;
  const int sub = lane % LPR, pg = lane / LPR;
  int* pt = s_pt[warp];
  if (bpos > 0) {
    const int nu = single ? 1 : min(kMaxBeam, n_units - first);
    for (int i = lane; i < nu * n_blocks; i += 32) pt[i] = page_table[(long long)first * n_blocks + i];
    __syncwarp();
  }
  const long long plane = (long long)kPageTokens * d;                       // k plane -> v plane of a page's layer
  const long long lane_off = (long long)layer * 2 * plane + h * 64 + sub * VEC;
  auto load_batch = [&](int t0, uint4* kr, uint4* vr) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = t0 + u * PPI + pg;
      if (t < bpos) {
        const int page = pt[(single ? 0 : (int)my_anc[t]) * n_blocks + t / kPageTokens];
        const T* kp = pool + (long long)page * page_stride + lane_off + (long long)(t % kPageTokens) * d;
        kr[u] = ld_raw16<T>(kp);
        vr[u] = ld_raw16<T>(kp + plane);
      }
    }
  };
  uint4 kr[U], vr[U];
  load_batch(0, kr, vr);
  pdl_wait();
  trace_mark(trace, (3u << 24) | 2);
  const float* qrow = qkv + (long long)r * 3 * d + h * 64;
  // fused append: k / v of this row -> its page [layer][k | v][pos % kPageTokens]; 2 dims of each per lane
  {
    T* dst = pool + (long long)row_page[r] * page_stride + (long long)layer * 2 * plane + (long long)(pos % kPageTokens) * d + h * 64 + lane * 2;
    dst[0] = from_f<T>(qrow[d + lane * 2]); dst[1] = from_f<T>(qrow[d + lane * 2 + 1]);
    dst[plane] = from_f<T>(qrow[2 * d + lane * 2]); dst[plane + 1] = from_f<T>(qrow[2 * d + lane * 2 + 1]);
  }
  // bf16 mode works in the log2 domain (log2(e) folded into q: one MUFU.EX2 per exponential, no extra multiply);
  // the fp32 validation mode keeps expf
  constexpr bool kExp2 = !std::is_same<T, float>::value;
  const float qscale = kExp2 ? 0.125f * 1.4426950408889634f : 0.125f;
  float qf[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) qf[i] = qrow[sub * VEC + i] * qscale;
  float m = -INFINITY, l = 0.f, acc[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
  auto ex = [&](float x) { return kExp2 ? fast_exp2(x) : expf(x); };
  auto fold = [&](const float* kf, const float* vf, bool valid) {
    float sc = 0.f;
#pragma unroll
    for (int i = 0; i < VEC; ++i) sc = fmaf(qf[i], kf[i], sc);
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, o);
    if (valid) {
      if (sc > m) {  // the running maximum moves (rare after the first positions): rescale
        const float a = ex(m - sc);
        l *= a;
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] *= a;
        m = sc;
      }
      const float pr = ex(sc - m);
      l += pr;
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[i] = fmaf(pr, vf[i], acc[i]);
    }
  };
  // cached positions [0, bpos): U passes of PPI positions per batch
  for (int t0 = 0; t0 < bpos; t0 += PPI * U) {
    if (t0 > 0) load_batch(t0, kr, vr);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (t0 + u * PPI >= bpos) break;  // warp-uniform
      const bool valid = t0 + u * PPI + pg < bpos;
      float kf[VEC], vf[VEC];
      if (valid) { unpack16<T>(kr[u], kf); unpack16<T>(vr[u], vf); }
      else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) { kf[i] = 0.f; vf[i] = 0.f; }
      }
      fold(kf, vf, valid);
    }
  }
  // positions fed in THIS step [bpos, pos]: fp32 rows of the qkv buffer, rounded like the pool copy
  for (int t0 = bpos; t0 <= pos; t0 += PPI) {
    const int t = t0 + pg;
    const bool valid = t <= pos;
    float kf[VEC], vf[VEC];
    if (valid) {
      const float* src = qkv + (long long)(r - (pos - t)) * 3 * d + d + h * 64 + sub * VEC;
#pragma unroll
      for (int i = 0; i < VEC; ++i) { kf[i] = to_f(from_f<T>(src[i])); vf[i] = to_f(from_f<T>(src[d + i])); }
    } else {
#pragma unroll
      for (int i = 0; i < VEC; ++i) { kf[i] = 0.f; vf[i] = 0.f; }
    }
    fold(kf, vf, valid);
  }
  // merge the PPI position groups of the warp
#pragma unroll
  for (int o = LPR; o < 32; o <<= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), l2 = __shfl_xor_sync(0xffffffffu, l, o);
    const float M = fmaxf(m, m2);
    const float e1 = (m == -INFINITY) ? 0.f : ex(m - M), e2 = (m2 == -INFINITY) ? 0.f : ex(m2 - M);
    l = l * e1 + l2 * e2;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float a2 = __shfl_xor_sync(0xffffffffu, acc[i], o);
      acc[i] = acc[i] * e1 + a2 * e2;
    }
    m = M;
  }
  if (pg == 0) {
    const float inv = 1.f / l;
    T* o = out + (long long)r * d + h * 64 + sub * VEC;
#pragma unroll
    for (int i = 0; i < VEC; ++i) o[i] = from_f<T>(acc[i] * inv);
  }
  trace_mark(trace, (3u << 24) | 8);
}

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma16816(float* c, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}
// x0, x1 -> (bf16 high parts packed, bf16 low parts packed): x = high + low to ~16 mantissa bits
__device__ __forceinline__ void split_bf16x2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
  const __nv_bfloat162 hv(h0, h1);
  hi = *reinterpret_cast<const uint32_t*>(&hv);
  lo = pack_bf16x2(x0 - __bfloat162float(h0), x1 - __bfloat162float(h1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// pospage[r][t] = pool page that holds position t of row r's hypothesis, t < bpos (later positions are fed in this step).
// Deliberately WITHOUT an early launch_dependents: the self-attention of layer 0 reads the table before its own
// dependency wait, which is only safe if no later kernel of the step can start before this one has finished.
__global__ void __launch_bounds__(128)
dec_self_pospage_kernel(const int* __restrict__ row_seq, const int* __restrict__ row_bpos, int n_ctx, int n_blocks, int n_units,
                        const int* __restrict__ page_table, const int* __restrict__ seq_first, const unsigned char* __restrict__ anc,
                        int* __restrict__ pospage) {
  pdl_wait();
  const int r = blockIdx.x;
  const int s = row_seq[r], bpos = row_bpos[r];
  const int sf = seq_first[s];
  const bool single = (sf & kSingleBeamFlag) != 0;
  const int first = sf & ~kSingleBeamFlag;
  const unsigned char* my_anc = anc + (long long)s * n_ctx;
  for (int t = threadIdx.x; t < bpos; t += 128) {
    const int slot = first + (single ? 0 : (int)my_anc[t]);
    pospage[(long long)r * n_ctx + t] = slot < n_units ? page_table[(long long)slot * n_blocks + t / kPageTokens] : 0;
  }
}

// ------------------------------------------------------------------------------------------------
// v3 (bf16 product mode, the default): PERSISTENT WARPS on mma.sync.  A CTA is one warp; it owns units w, w + G, ... and
// a ring of kPwNB buffers of kPwCB positions (K and V head slices, 16-byte chunks XOR-swizzled by the row) that is fed with
// cp.async in consumption order ACROSS unit boundaries: while one item is folded the next is in flight, and the next unit's
// q / k / v rows and the next item's page lookups are already in registers.  Nothing in the loop is a block-wide barrier.
//   q.K^T : A = q (matrix row 0: bf16 high part, row 8: low part -> fp32-accurate q for free, M = 16 is otherwise wasted),
//           B = K via ldmatrix;  P.V : the score fragment of lanes 0..3 IS the A fragment of P (high / low parts again),
//           B = V via ldmatrix.trans.  ~65 warp instructions per 16 positions instead of ~600 in the SIMT kernels.
// How it got here (profiles/r2_notes.md, code of the discarded variants in commit e4f8ffe): v1 and v2 run in lockstep WAVES --
// every resident unit walks "control words -> page table -> K/V burst -> q -> fold" at the same time, so HBM idles while the
// SMs fold and the SMs idle while HBM streams (ncu: 2.9 waves of ~8 us for 65 MB that HBM delivers in 9 us), and their fp32
// FMAs on unpacked bf16 make the fold itself issue-bound (7000 warp instructions per unit).  A register-fed mma kernel,
// a CTA-wide persistent ring and a staged mma kernel each fixed one of the two and were no faster; this one fixes both.
// positions per ring buffer, buffers, resident warps per SM asked of the compiler (165 registers), most units per warp, and the
// unit count from which the kernel is taken.  A-B of the ring geometry: profiles/r2_selfattn_pw_configs.txt
constexpr int kPwCfgCB = 32, kPwCfgNB = 2, kPwCfgWarps = 12, kPwUnits = 32, kPwMinUnits = 512;  // A-B of 9 configurations: profiles/r2_selfattn_pw_configs.txt

template <int kPwCB, int kPwNB, int kPwMinWarps>
__global__ void __launch_bounds__(32, kPwMinWarps)
dec_self_attention_pw_kernel(const int* __restrict__ row_pos, const int* __restrict__ row_bpos, const int* __restrict__ row_page,
                             const float* __restrict__ qkv, bf16* __restrict__ pool, long long page_stride, int n_ctx,
                             const int* __restrict__ pospage, int layer, int d, int n_rows, int n_head, bf16* __restrict__ out,
                             unsigned long long* trace_buf) {
  extern __shared__ __align__(128) unsigned char smp[];  // kPwNB x { K [32][128 B], V [32][128 B] }
  constexpr uint32_t kBuf = kPwCB * 256u, kVOff = kPwCB * 128u;
  const int lane = threadIdx.x;
  const int G = gridDim.x, n_units = n_rows * n_head;
  const int K = (n_units - (int)blockIdx.x + G - 1) / G;  // units of this warp: blockIdx.x + k G
  unsigned long long* const trace = (blockIdx.x == 0 && lane == 0) ? trace_buf : nullptr;
  trace_mark(trace, (3u << 24) | 1);
  pdl_trigger();
  // Read before the dependency wait: the control block, pospage (dec_self_pospage_kernel) and cached K/V of earlier steps.
  int my_pos = 0, my_bpos = 0, my_page = 0;  // lane k: control words of unit k
  if (lane < K) {
    const int r = ((int)blockIdx.x + lane * G) / n_head;
    my_pos = row_pos[r]; my_bpos = row_bpos[r]; my_page = row_page[r];
  }
  const int grp = lane >> 3, ch8 = lane & 7;
  const int g = lane >> 2, tig = lane & 3;
  const long long plane = (long long)kPageTokens * d;
  const uint32_t sbase = smem_u32(smp);
  // ---- producer side: items (unit, chunk of kPwCB positions) in consumption order ----
  int pu = 0, pc = 0, p_r = (int)blockIdx.x / n_head, p_h = (int)blockIdx.x - p_r * n_head, p_bpos = 0, p_n = 1;
  int pg[kPwCB / 4];
  auto p_lookup = [&]() {  // pages of item (pu, pc); speculative (no dependence on the control words)
    const int* pp = pospage + (long long)p_r * n_ctx + pc * kPwCB;
#pragma unroll
    for (int i = 0; i < kPwCB / 4; ++i) pg[i] = (pc * kPwCB + grp + 4 * i < n_ctx) ? __ldg(pp + grp + 4 * i) : 0;
  };
  p_lookup();
  p_bpos = __shfl_sync(0xffffffffu, my_bpos, 0);
  p_n = __shfl_sync(0xffffffffu, my_pos, 0) + 1;
  auto p_request = [&](int slot) {  // item (pu, pc) -> buffer `slot`; then move on and look the next item's pages up
    if (pu < K) {
      const bf16* src0 = pool + (long long)layer * 2 * plane + p_h * 64 + ch8 * 8;
      const uint32_t dst0 = sbase + (uint32_t)slot * kBuf;
#pragma unroll
      for (int i = 0; i < kPwCB / 4; ++i) {
        const int tl = grp + 4 * i, t = pc * kPwCB + tl;
        if (t < p_bpos) {
          const bf16* src = src0 + (long long)pg[i] * page_stride + (long long)(t & (kPageTokens - 1)) * d;
          const uint32_t dst = dst0 + (uint32_t)tl * 128u + (uint32_t)((ch8 ^ (tl & 7)) << 4);
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + kVOff), "l"(src + plane) : "memory");
        }
      }
      if (++pc * kPwCB >= p_n) {
        pc = 0;
        if (++pu < K) {
          const int u = (int)blockIdx.x + pu * G;
          p_r = u / n_head; p_h = u - p_r * n_head;
          p_bpos = __shfl_sync(0xffffffffu, my_bpos, pu);
          p_n = __shfl_sync(0xffffffffu, my_pos, pu) + 1;
        }
      }
      if (pu < K) p_lookup();
    }
    cp_async_commit();  // an empty group when nothing is left: the consumer's wait counts groups
  };
#pragma unroll
  for (int i = 0; i < kPwNB - 1; ++i) p_request(i);  // the ring runs kPwNB - 1 items ahead of the fold
  pdl_wait();
  trace_mark(trace, (3u << 24) | 2);
  // ---- consumer side ----
  float2 qx[4], qy[4], kx, vx;  // raw q (lanes 0..3 only) and this row's k / v (2 dims per lane) of the NEXT unit to start
  auto q_prefetch = [&](int k) {
    const int u = (int)blockIdx.x + k * G;
    const int r = u / n_head, h = u - r * n_head;
    const float* qrow = qkv + (long long)r * 3 * d + h * 64;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      qx[j] = make_float2(0.f, 0.f); qy[j] = make_float2(0.f, 0.f);
      if (g == 0) { qx[j] = *reinterpret_cast<const float2*>(qrow + 16 * j + 2 * tig); qy[j] = *reinterpret_cast<const float2*>(qrow + 16 * j + 8 + 2 * tig); }
    }
    kx = *reinterpret_cast<const float2*>(qrow + d + lane * 2);
    vx = *reinterpret_cast<const float2*>(qrow + 2 * d + lane * 2);
  };
  q_prefetch(0);
  const int k_row = lane & 7, k_chunk = lane >> 3;
  const int v_row = (lane & 7) + ((lane >> 3) & 1) * 8, v_chunk = lane >> 4;
  int it = 0;
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const int u = (int)blockIdx.x + k * G;
    const int r = u / n_head, h = u - r * n_head;
    const int pos = __shfl_sync(0xffffffffu, my_pos, k), bpos = __shfl_sync(0xffffffffu, my_bpos, k);
    const int page = __shfl_sync(0xffffffffu, my_page, k);
    const int n = pos + 1;
    // q fragments in the log2 domain; matrix row 0 = bf16 high part, row 8 = low part, other rows zero
    uint32_t qa[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float qscale = 0.125f * 1.4426950408889634f;
      split_bf16x2(qx[j].x * qscale, qx[j].y * qscale, qa[j][0], qa[j][1]);
      split_bf16x2(qy[j].x * qscale, qy[j].y * qscale, qa[j][2], qa[j][3]);
    }
    const uint32_t own_k = pack_bf16x2(kx.x, kx.y), own_v = pack_bf16x2(vx.x, vx.y);
    {  // fused append: k / v of this row -> its page [layer][k | v][pos % 16]
      bf16* dst = pool + (long long)page * page_stride + (long long)layer * 2 * plane + (long long)(pos & (kPageTokens - 1)) * d + h * 64 + lane * 2;
      *reinterpret_cast<uint32_t*>(dst) = own_k;
      *reinterpret_cast<uint32_t*>(dst + plane) = own_v;
    }
    if (k + 1 < K) q_prefetch(k + 1);  // in flight while this unit is folded
    float m = -INFINITY, l = 0.f, o[8][4];
#pragma unroll
    for (int e = 0; e < 8; ++e) { o[e][0] = o[e][1] = o[e][2] = o[e][3] = 0.f; }
    const int n_items = (n + kPwCB - 1) / kPwCB;
#pragma unroll 1
    for (int c = 0; c < n_items; ++c, ++it) {
      const int c0 = c * kPwCB;
      const uint32_t kb = sbase + (uint32_t)(it % kPwNB) * kBuf, vb = kb + kVOff;
      const int cn = min(kPwCB, n - c0);  // positions of this item, cached or fed in this step
      if (c0 + cn > bpos) {
        // positions fed in THIS step [bpos, pos] and zero rows behind the last position (P = 0 there, but 0 x garbage
        // must not become NaN)
        const int t_hi = (cn + 15) & ~15;
        if (bpos == pos) {  // decode row: its own k / v are already in registers
          const int tl = pos - c0;
          const uint32_t a = (uint32_t)tl * 128u + (uint32_t)(((lane >> 2) ^ (tl & 7)) << 4) + (uint32_t)(lane & 3) * 4u;
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(kb + a), "r"(own_k) : "memory");
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(vb + a), "r"(own_v) : "memory");
          for (int z = cn; z < t_hi; ++z) {
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(kb + (uint32_t)z * 128u + (uint32_t)lane * 4u), "r"(0u) : "memory");
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(vb + (uint32_t)z * 128u + (uint32_t)lane * 4u), "r"(0u) : "memory");
          }
        } else {  // prefill rows: fp32 rows of the qkv buffer, rounded like the pool copy
          const int t_lo = max(bpos, c0) - c0;
          for (int idx = t_lo * 16 + lane; idx < t_hi * 16; idx += 32) {
            const int tl = idx >> 4, cc = idx & 15, sel = cc >> 3, ch = cc & 7;
            uint4 w = make_uint4(0u, 0u, 0u, 0u);
            if (tl < cn) {
              const float* src = qkv + (long long)(r - (pos - (c0 + tl))) * 3 * d + (1 + sel) * d + h * 64 + ch * 8;
              const float4 x0 = *reinterpret_cast<const float4*>(src), x1 = *reinterpret_cast<const float4*>(src + 4);
              w.x = pack_bf16x2(x0.x, x0.y); w.y = pack_bf16x2(x0.z, x0.w); w.z = pack_bf16x2(x1.x, x1.y); w.w = pack_bf16x2(x1.z, x1.w);
            }
            const uint32_t dst = (sel ? vb : kb) + (uint32_t)tl * 128u + (uint32_t)((ch ^ (tl & 7)) << 4);
            asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(dst), "r"(w.x), "r"(w.y), "r"(w.z), "r"(w.w) : "memory");
          }
        }
      }
      cp_async_wait_group<kPwNB - 2>();  // item `it` has landed (groups are committed in item order, kPwNB - 1 ahead)
      __syncwarp();                      // ... and the buffer refilled next (item it - 1's) is no longer being read
      p_request((it + kPwNB - 1) % kPwNB);
      for (int b0 = 0; b0 < cn; b0 += 16) {
        float c0f[4] = {0.f, 0.f, 0.f, 0.f}, c1f[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          uint32_t r0, r1, r2, r3;
          const int row0 = b0 + k_row, row1 = row0 + 8;
          ldsm_x4(kb + (uint32_t)row0 * 128u + (uint32_t)(((k_chunk + 4 * half) ^ (row0 & 7)) << 4), r0, r1, r2, r3);
          mma16816(c0f, qa[2 * half][0], qa[2 * half][1], qa[2 * half][2], qa[2 * half][3], r0, r1);
          mma16816(c0f, qa[2 * half + 1][0], qa[2 * half + 1][1], qa[2 * half + 1][2], qa[2 * half + 1][3], r2, r3);
          ldsm_x4(kb + (uint32_t)row1 * 128u + (uint32_t)(((k_chunk + 4 * half) ^ (row1 & 7)) << 4), r0, r1, r2, r3);
          mma16816(c1f, qa[2 * half][0], qa[2 * half][1], qa[2 * half][2], qa[2 * half][3], r0, r1);
          mma16816(c1f, qa[2 * half + 1][0], qa[2 * half + 1][1], qa[2 * half + 1][2], qa[2 * half + 1][3], r2, r3);
        }
        float sc[4] = {c0f[0] + c0f[2], c0f[1] + c0f[3], c1f[0] + c1f[2], c1f[1] + c1f[3]};
        if (b0 + 16 > cn) {
          const int t = b0 + 2 * tig;
          if (t >= cn) sc[0] = -INFINITY;
          if (t + 1 >= cn) sc[1] = -INFINITY;
          if (t + 8 >= cn) sc[2] = -INFINITY;
          if (t + 9 >= cn) sc[3] = -INFINITY;
        }
        float bm = fmaxf(fmaxf(sc[0], sc[1]), fmaxf(sc[2], sc[3]));
        bm = fmaxf(bm, __shfl_xor_sync(0xffffffffu, bm, 1));
        bm = fmaxf(bm, __shfl_xor_sync(0xffffffffu, bm, 2));
        if (bm > m) {
          const float a = fast_exp2(m - bm);
          l *= a;
#pragma unroll
          for (int e = 0; e < 8; ++e) { o[e][0] *= a; o[e][1] *= a; o[e][2] *= a; o[e][3] *= a; }
          m = bm;
        }
        const float p0 = fast_exp2(sc[0] - m), p1 = fast_exp2(sc[1] - m), p2 = fast_exp2(sc[2] - m), p3 = fast_exp2(sc[3] - m);
        l += (p0 + p1) + (p2 + p3);
        uint32_t a0, a1, a2, a3;
        split_bf16x2(p0, p1, a0, a1);
        split_bf16x2(p2, p3, a2, a3);
        if (g != 0) { a0 = a1 = a2 = a3 = 0u; }
#pragma unroll
        for (int e2 = 0; e2 < 4; ++e2) {
          uint32_t r0, r1, r2, r3;
          const int row = b0 + v_row;
          ldsm_x4_t(vb + (uint32_t)row * 128u + (uint32_t)(((2 * e2 + v_chunk) ^ (row & 7)) << 4), r0, r1, r2, r3);
          mma16816(o[2 * e2], a0, a1, a2, a3, r0, r1);
          mma16816(o[2 * e2 + 1], a0, a1, a2, a3, r2, r3);
        }
      }
    }
    l += __shfl_xor_sync(0xffffffffu, l, 1);
    l += __shfl_xor_sync(0xffffffffu, l, 2);
    if (g == 0) {  // lane tig: dims 8 e + 2 tig, + 1
      const float inv = 1.f / l;
      bf16* dst = out + (long long)r * d + h * 64 + 2 * tig;
#pragma unroll
      for (int e = 0; e < 8; ++e)
        *reinterpret_cast<uint32_t*>(dst + 8 * e) = pack_bf16x2((o[e][0] + o[e][2]) * inv, (o[e][1] + o[e][3]) * inv);
    }
  }
  cp_async_wait_group<0>();
  trace_mark(trace, (3u << 24) | 8);
}

// ------------------------------------------------------------------------------------------------
constexpr int XW = 8;  // warps per cross-attention CTA
constexpr int kMaxSplit = 8;

template <typename T, int NQ>
__global__ void __launch_bounds__(XW * 32)
dec_cross_attention_kernel(const int* __restrict__ group_first_row, const int* __restrict__ group_n_rows,
                           const int* __restrict__ group_xslot, const float* __restrict__ q, const T* __restrict__ cache,
                           long long slot_stride, int T_enc, int layer, int d, int n_split, T* __restrict__ out,
                           float* __restrict__ ws) {
  constexpr int VEC = Vec16<T>::N, LPR = 64 / VEC, RPW = 32 / LPR;
  constexpr int ROWS_IT = XW * RPW;  // rows per CTA iteration
  extern __shared__ float smx[];
  const int h = blockIdx.x, g = blockIdx.y, sp = blockIdx.z;
  const int n_head = gridDim.x;
  const int row0 = group_first_row[g], nq = group_n_rows[g];
  const int chunk = (T_enc + n_split - 1) / n_split;
  const int t0 = sp * chunk, t1 = min(T_enc, t0 + chunk);
  const int len = t1 - t0;
  float* sc = smx;                        // [NQ][chunk]
  float* osm = smx + NQ * chunk;          // [XW][NQ][64]
  __shared__ float red[NQ][XW];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sub = lane % LPR, rg = lane / LPR;
  const T* kbase = cache + (long long)group_xslot[g] * slot_stride + (long long)layer * T_enc * 2 * d + h * 64 + sub * VEC;
  const T* vbase = kbase + d;
  const long long rstride = 2LL * d;

  float qf[NQ][VEC];
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi) {
    if (qi < nq) {
#pragma unroll
      for (int i = 0; i < VEC; ++i) qf[qi][i] = q[(long long)(row0 + qi) * d + h * 64 + sub * VEC + i] * 0.125f;
    } else {
#pragma unroll
      for (int i = 0; i < VEC; ++i) qf[qi][i] = 0.f;
    }
  }
  // ---- scores: 4 independent 16-byte loads in flight per lane ----
  constexpr int U = 4;
  for (int tb = warp * RPW; tb < len; tb += ROWS_IT * U) {
    float kf[U][VEC];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = tb + u * ROWS_IT + rg;
      if (t < len) Vec16<T>::load_stream(kbase + (long long)(t0 + t) * rstride, kf[u]);
      else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) kf[u][i] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = tb + u * ROWS_IT + rg;
      if (tb + u * ROWS_IT >= len) break;  // warp-uniform
#pragma unroll
      for (int qi = 0; qi < NQ; ++qi) {
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc = fmaf(qf[qi][i], kf[u][i], acc);
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (sub == 0 && t < len) sc[qi * chunk + t] = acc;
      }
    }
  }
  __syncthreads();
  // ---- softmax statistics per query over this chunk ----
  float mloc[NQ], lloc[NQ];
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi) {
    float mx = -INFINITY;
    for (int t = threadIdx.x; t < len; t += XW * 32) mx = fmaxf(mx, sc[qi * chunk + t]);
    mx = warp_max(mx);
    if (lane == 0) red[qi][warp] = mx;
  }
  __syncthreads();
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi) {
    float mx = red[qi][0];
#pragma unroll
    for (int w = 1; w < XW; ++w) mx = fmaxf(mx, red[qi][w]);
    mloc[qi] = mx;
  }
  __syncthreads();
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi) {
    float sum = 0.f;
    for (int t = threadIdx.x; t < len; t += XW * 32) {
      const float p = exp_t<T>(sc[qi * chunk + t] - mloc[qi]);
      sc[qi * chunk + t] = p;
      sum += p;
    }
    sum = warp_sum(sum);
    if (lane == 0) red[qi][warp] = sum;
  }
  __syncthreads();
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi) {
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < XW; ++w) sum += red[qi][w];
    lloc[qi] = sum;
  }
  // ---- P.V ----
  float acc[NQ][VEC];
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi)
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[qi][i] = 0.f;
  for (int tb = warp * RPW; tb < len; tb += ROWS_IT * U) {
    float vf[U][VEC];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = tb + u * ROWS_IT + rg;
      if (t < len) Vec16<T>::load_stream(vbase + (long long)(t0 + t) * rstride, vf[u]);
      else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) vf[u][i] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = tb + u * ROWS_IT + rg;
      if (t < len) {
#pragma unroll
        for (int qi = 0; qi < NQ; ++qi) {
          const float p = sc[qi * chunk + t];
#pragma unroll
          for (int i = 0; i < VEC; ++i) acc[qi][i] = fmaf(p, vf[u][i], acc[qi][i]);
        }
      }
    }
  }
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi)
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      float v = acc[qi][i];
#pragma unroll
      for (int o = LPR; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (rg == 0) osm[(warp * NQ + qi) * 64 + sub * VEC + i] = v;
    }
  __syncthreads();
  for (int i = threadIdx.x; i < NQ * 64; i += XW * 32) {
    const int qi = i >> 6, c = i & 63;
    if (qi >= nq) continue;
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < XW; ++w) v += osm[(w * NQ + qi) * 64 + c];
    const int row = row0 + qi;
    if (n_split == 1) {
      out[(long long)row * d + h * 64 + c] = from_f<T>(v / lloc[qi]);
    } else {
      float* w = ws + (((long long)row * n_head + h) * kMaxSplit + sp) * 66;
      w[2 + c] = v;
      if (c == 0) { w[0] = mloc[qi]; w[1] = lloc[qi]; }
    }
  }
}

template <typename T>
__global__ void dec_cross_combine_kernel(const float* __restrict__ ws, int n_split, int d, T* __restrict__ out) {
  pdl_trigger();
  pdl_wait();
  const int h = blockIdx.x, row = blockIdx.y, n_head = gridDim.x, c = threadIdx.x;
  const float* w = ws + ((long long)row * n_head + h) * kMaxSplit * 66;
  float M = -INFINITY;
  for (int s = 0; s < n_split; ++s) M = fmaxf(M, w[s * 66]);
  float num = 0.f, den = 0.f;
  for (int s = 0; s < n_split; ++s) {
    const float e = exp_t<T>(w[s * 66] - M);
    num = fmaf(e, w[s * 66 + 2 + c], num);
    den = fmaf(e, w[s * 66 + 1], den);
  }
  out[(long long)row * d + h * 64 + c] = from_f<T>(num / den);
}

}  // namespace

int dec_self_chunk(int max_ctx) { return (max_ctx > 0 && max_ctx <= 32) ? 32 : (max_ctx > 0 && max_ctx <= 64) ? 64 : 128; }

template <typename T>
void attn_encoder_simt(const T* qkv, T* out, int batch, int T_len, int n_head, cudaStream_t stream) {
  dim3 grid((T_len + 31) / 32, n_head, batch);
  attn_encoder_simt_kernel<T><<<grid, 128, 0, stream>>>(qkv, out, T_len, n_head);
  BW_CUDA(cudaGetLastError());
  ++g_kernel_launches;
}
template void attn_encoder_simt<float>(const float*, float*, int, int, int, cudaStream_t);
template void attn_encoder_simt<bf16>(const bf16*, bf16*, int, int, int, cudaStream_t);

namespace { std::atomic<int> g_self_attn_mode{0}; }
void dec_self_attention_mode(int mode) { g_self_attn_mode.store(mode); }

namespace {
int self_attn_mode() {
  static const int forced = getenv("B200W_SELF_ATTN") ? atoi(getenv("B200W_SELF_ATTN")) : 0;  // 1 = staged, 2 = warp, 3 = persistent warps
  const int m = g_self_attn_mode.load();
  return m ? m : forced;
}
// bf16 product mode: persistent warps from 512 (row, head) units upwards (640 units: 0.4 - 1.7 % faster steps, 160 units: a tie);
// below that a unit per warp leaves most SMs with one warp and the staged kernel's 4 warps per unit are as fast
// (A-B: profiles/r2_selfattn_pw_ab.txt)
bool use_persistent_warps(const SelfKV& kv, int units) {
  const int mode = self_attn_mode();
  return kv.pospage && (mode == 3 || (mode == 0 && units >= kPwMinUnits));
}
}  // namespace

void dec_self_pospage(const DecRows& rows, const SelfKV& kv, int n_head, cudaStream_t stream) {
  if (rows.n_rows <= 0 || !use_persistent_warps(kv, rows.n_rows * n_head)) return;  // only the persistent kernel reads the table
  launch_kernel(dec_self_pospage_kernel, dim3(rows.n_rows), dim3(128), 0, stream, rows.row_seq, rows.row_bpos, kv.n_ctx, kv.n_blocks,
                kv.n_units, kv.page_table, kv.seq_first, kv.anc, kv.pospage);
  ++g_kernel_launches;
}

template <typename T>
void dec_self_attention(const DecRows& rows, const float* qkv, const SelfKV& kv, int layer, int d, int n_head, T* out,
                        cudaStream_t stream) {
  if (rows.n_rows <= 0) return;
  BW_CHECK(kv.n_ctx <= 448 && kv.n_blocks <= kMaxBlocks && kv.n_blocks * kPageTokens >= kv.n_ctx, "n_text_ctx > 448 unsupported");
  BW_CHECK(rows.row_page && kv.page_table, "paged self-attention needs row_page and a page table");
  const int units = n_head * rows.n_rows;
  const int mode = self_attn_mode();
  if constexpr (std::is_same<T, bf16>::value) {
    if (use_persistent_warps(kv, units)) {
      int dev = 0;
      BW_CUDA(cudaGetDevice(&dev));
      BW_CHECK(dev >= 0 && dev < 64, "device index");
      constexpr size_t smem = (size_t)kPwCfgNB * kPwCfgCB * 256;
      static std::atomic<int> pw_slots[64];  // resident warps of the kernel per device (occupancy x SMs)
      int slots = pw_slots[dev].load();
      if (slots == 0) {
        int occ = 0, sms = 0;
        BW_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dec_self_attention_pw_kernel<kPwCfgCB, kPwCfgNB, kPwCfgWarps>, 32, smem));
        BW_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        slots = std::max(occ, 1) * std::max(sms, 1);
        pw_slots[dev].store(slots);
      }
      BW_CHECK((units + slots - 1) / slots <= kPwUnits, "too many self-attention units for one launch");
      launch_kernel(dec_self_attention_pw_kernel<kPwCfgCB, kPwCfgNB, kPwCfgWarps>, dim3(std::min(units, slots)), dim3(32), smem, stream,
                    rows.row_pos, rows.row_bpos, rows.row_page, qkv, reinterpret_cast<bf16*>(kv.pool), kv.page_stride, kv.n_ctx,
                    (const int*)kv.pospage, layer, d, rows.n_rows, n_head, out, g_trace_dev);
      ++g_kernel_launches;
      return;
    }
  }
  if (mode == 2 || (mode != 1 && units >= 4000)) {
    launch_kernel(dec_self_attention_warp_kernel<T>, dim3((units + 3) / 4), dim3(128), 0, stream, rows.row_seq, rows.row_pos, rows.row_bpos,
                  rows.row_page, qkv, reinterpret_cast<T*>(kv.pool), kv.page_stride, kv.n_ctx, kv.n_blocks, kv.n_units, kv.page_table,
                  kv.seq_first, kv.anc, layer, d, rows.n_rows, n_head, out, g_trace_dev);
    ++g_kernel_launches;
    return;
  }
  dim3 grid(n_head, rows.n_rows);
  const int chunk = dec_self_chunk(rows.max_ctx);
  auto launch = [&](auto kern, int smem) {
    launch_kernel(kern, grid, dim3(128), (size_t)smem, stream, rows.row_seq, rows.row_pos, rows.row_bpos, rows.row_page, qkv,
                  reinterpret_cast<T*>(kv.pool), kv.page_stride, kv.n_ctx, kv.n_blocks, kv.n_units, kv.page_table, kv.seq_first, kv.anc,
                  layer, d, out, g_trace_dev);
  };
  static std::atomic<unsigned long long> attr_set{0};
  int dev = 0;
  BW_CUDA(cudaGetDevice(&dev));
  if (!(attr_set.load() >> dev & 1ull)) {
    BW_CUDA(cudaFuncSetAttribute(dec_self_attention_kernel<T, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 128 * 64 * (int)sizeof(T)));
    attr_set.fetch_or(1ull << dev);
  }
  if (chunk == 32) launch(dec_self_attention_kernel<T, 32>, 2 * 32 * 64 * (int)sizeof(T));
  else if (chunk == 64) launch(dec_self_attention_kernel<T, 64>, 2 * 64 * 64 * (int)sizeof(T));
  else launch(dec_self_attention_kernel<T, 128>, 2 * 128 * 64 * (int)sizeof(T));
  ++g_kernel_launches;
}
template void dec_self_attention<float>(const DecRows&, const float*, const SelfKV&, int, int, int, float*, cudaStream_t);
template void dec_self_attention<bf16>(const DecRows&, const float*, const SelfKV&, int, int, int, bf16*, cudaStream_t);

size_t dec_cross_workspace_floats(int n_rows, int n_head) { return (size_t)n_rows * n_head * kMaxSplit * 66; }

namespace {
template <typename T, int NQ>
void launch_cross(const int* gfr, const int* gnr, const int* gx, int n_groups, const float* q, const CrossKV& kv, int layer, int d,
                  int n_head, int n_split, T* out, float* ws, cudaStream_t stream) {
  const int chunk = (kv.T_enc + n_split - 1) / n_split;
  const size_t smem = sizeof(float) * ((size_t)NQ * chunk + (size_t)XW * NQ * 64);
  auto kern = dec_cross_attention_kernel<T, NQ>;
  static std::atomic<unsigned long long> attr_set{0};
  int dev = 0;
  BW_CUDA(cudaGetDevice(&dev));
  if (!(attr_set.load() >> dev & 1ull)) {
    BW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(sizeof(float) * ((size_t)NQ * 1504 + (size_t)XW * NQ * 64))));
    attr_set.fetch_or(1ull << dev);
  }
  dim3 grid(n_head, n_groups, n_split);
  kern<<<grid, XW * 32, smem, stream>>>(gfr, gnr, gx, q, reinterpret_cast<const T*>(kv.cache), kv.slot_stride, kv.T_enc, layer,
                                        d, n_split, out, ws);
  BW_CUDA(cudaGetLastError());
  ++g_kernel_launches;
}
}  // namespace

template <typename T>
void dec_cross_attention(const int* group_first_row, const int* group_n_rows, const int* group_xslot, int n_groups,
                         int max_group_rows, int n_rows, const float* q, const CrossKV& kv, int layer, int d, int n_head, T* out,
                         float* workspace, cudaStream_t stream, int force_split) {
  if (n_groups <= 0) return;
  BW_CHECK(max_group_rows <= 8, "at most 8 hypotheses per segment");
  BW_CHECK(kv.T_enc <= 1504, "n_audio_ctx > 1504 unsupported");
  // split T so that the grid covers the 148 SMs a few times over; each split re-reads nothing.
  int n_split = 1;
  const long long base = (long long)n_head * n_groups;
  while (n_split < kMaxSplit && base * n_split < 4 * 148) n_split *= 2;
  if (force_split > 0) n_split = std::min(force_split, (int)kMaxSplit);  // tests: any split count, not just powers of two
  if constexpr (std::is_same<T, bf16>::value) {
    // product mode: TMA + ldmatrix + mma.sync streaming kernel (attention_xdec.cu), on bf16 or 8-bit K/V
    BW_CHECK(kv.n_slots > 0 && kv.n_layer > 0, "cross-attention needs the cache geometry (TMA map)");
    if (kv.int8)
      dec_cross_attention_int8(group_first_row, group_n_rows, group_xslot, n_groups, q, kv, layer, d, n_head, n_split, out,
                               workspace, stream);
    else
      dec_cross_attention_mma(group_first_row, group_n_rows, group_xslot, n_groups, q, kv, kv.n_layer, layer, d, n_head, n_split,
                              out, workspace, stream);
  } else {
    BW_CHECK(!kv.int8, "the 8-bit cross cache needs bf16 compute");
    // fp32 validation mode: SIMT kernel with deterministic reduction order
    if (max_group_rows <= 1) launch_cross<T, 1>(group_first_row, group_n_rows, group_xslot, n_groups, q, kv, layer, d, n_head, n_split, out, workspace, stream);
    else if (max_group_rows <= 2) launch_cross<T, 2>(group_first_row, group_n_rows, group_xslot, n_groups, q, kv, layer, d, n_head, n_split, out, workspace, stream);
    else if (max_group_rows <= 4) launch_cross<T, 4>(group_first_row, group_n_rows, group_xslot, n_groups, q, kv, layer, d, n_head, n_split, out, workspace, stream);
    else launch_cross<T, 8>(group_first_row, group_n_rows, group_xslot, n_groups, q, kv, layer, d, n_head, n_split, out, workspace, stream);
  }
  if (n_split > 1) {
    dim3 grid(n_head, n_rows);
    launch_kernel(dec_cross_combine_kernel<T>, grid, dim3(64), 0, stream, (const float*)workspace, n_split, d, out);
    ++g_kernel_launches;
  }
}
template void dec_cross_attention<float>(const int*, const int*, const int*, int, int, int, const float*, const CrossKV&, int, int, int, float*, float*, cudaStream_t, int);
template void dec_cross_attention<bf16>(const int*, const int*, const int*, int, int, int, const float*, const CrossKV&, int, int, int, bf16*, float*, cudaStream_t, int);

}  // namespace bw
