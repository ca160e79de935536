// Bench and test hooks (include/b200_whisper_hooks.h): kernel-level entry points on device pointers, CUDA-event
// timers over resident synthetic data, the in-kernel debug timeline.  Not part of the drop-in boundary.
#include "../../include/b200_whisper_hooks.h"
#include "sched.cuh"

using namespace bw;

// every function below is declared extern "C" in include/b200_whisper_hooks.h and keeps that linkage

// ---- kernel-level entry points (device pointers / resident synthetic data; used by tests and bench.py) ----
int bw_gemm_bf16(int impl, const void* A, const void* B, void* C, const float* bias, const float* residual, int32_t M, int32_t N,
                 int32_t K, int32_t gelu, int32_t out_fp32, void* stream) {
  BW_API_BEGIN
  GemmArgs g;
  g.A = A; g.B = B; g.C = C; g.bias = bias; g.residual = residual;
  g.M = M; g.N = N; g.K = K; g.lda = K; g.ldb = K; g.ldc = N; g.ldres = N; g.gelu = gelu != 0; g.out_fp32 = out_fp32 != 0;
  if (impl == 0) gemm_tc_bf16(g, reinterpret_cast<cudaStream_t>(stream));
  else if (impl == 2) {  // swap-AB path of the decoder: C[M, N] computed as (B . A^T)^T
    GemmArgs s = g;
    s.A = B; s.B = A; s.M = N; s.N = M; s.transposed = true;
    gemm_tc_bf16(s, reinterpret_cast<cudaStream_t>(stream));
  } else gemm_simt<bf16>(g, reinterpret_cast<cudaStream_t>(stream));
  BW_API_END
}

namespace {
GemmArgs gemm_args_of(const bw_gemm_desc* d) {
  BW_CHECK(d, "null descriptor");
  BW_CHECK(d->M > 0 && d->N > 0 && d->K > 0 && d->Z > 0, "empty GEMM");
  BW_CHECK(d->lda >= d->K && d->ldb >= d->K && d->ldc >= (d->transposed ? d->M : d->N), "leading dimension too small");
  BW_CHECK(!d->residual || d->ldres >= (d->transposed ? d->M : d->N), "residual leading dimension too small");
  BW_CHECK((d->a_rows == 0 || d->a_rows >= d->M) && (d->b_rows == 0 || d->b_rows >= d->N), "a_rows / b_rows below M / N");
  BW_CHECK(d->a_zstride >= 0 && d->b_zstride >= 0 && d->c_zstride >= 0 && d->bias_zstride >= 0 && d->res_zstride >= 0,
           "negative batch stride");
  GemmArgs g;
  g.A = d->A; g.B = d->B; g.C = d->C; g.bias = d->bias; g.residual = d->residual;
  g.M = d->M; g.N = d->N; g.K = d->K;
  g.lda = d->lda; g.ldb = d->ldb; g.ldc = d->ldc; g.ldres = d->ldres;
  g.Z = d->Z; g.a_rows = d->a_rows; g.b_rows = d->b_rows;
  g.a_zstride = d->a_zstride; g.b_zstride = d->b_zstride; g.c_zstride = d->c_zstride;
  g.bias_zstride = d->bias_zstride; g.res_zstride = d->res_zstride;
  g.gelu = d->gelu != 0; g.out_fp32 = d->out_fp32 != 0; g.transposed = d->transposed != 0;
  return g;
}
int route_code(GemmRoute r) { return BW_GEMM_ROUTE((int)r.kernel, r.param); }
}  // namespace

int bw_test_gemm(const bw_gemm_desc* desc, int32_t dtype, int32_t route, int32_t* route_taken, void* stream) {
  BW_API_BEGIN
  BW_CHECK(route_taken, "null argument");
  const GemmArgs g = gemm_args_of(desc);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const GemmRoute simt{GemmKernel::simt, 0};
  if (dtype == 1) {
    BW_CHECK(route == 0 || route == route_code(simt), "the fp32 GEMM runs on the SIMT kernel only");
    BW_CHECK(g.out_fp32, "the fp32 GEMM writes fp32");
    gemm_simt<float>(g, st);
    *route_taken = route_code(simt);
  } else {
    BW_CHECK(dtype == 0, "dtype: 0 bf16, 1 fp32");
    if (route == route_code(simt)) {
      gemm_simt<bf16>(g, st);
      *route_taken = route;
    } else {
      const GemmRoute r = route == 0 ? gemm_tc_choose(g) : GemmRoute{(GemmKernel)(route / 1000), route % 1000};
      gemm_tc_launch(g, r, st);
      *route_taken = route_code(r);
    }
  }
  BW_API_END
}

int bw_test_gemm_route(const bw_gemm_desc* desc, int32_t* route) {
  BW_API_BEGIN
  BW_CHECK(route, "null argument");
  *route = route_code(gemm_tc_choose(gemm_args_of(desc)));
  BW_API_END
}

// Test hook for the decoder LayerNorm fusion: a producer row GEMM (x = res + A.Wp^T + bp, which also leaves bf16(x)
// and the LayerNorm partials) followed by a consumer row GEMM (out = [gelu](LayerNorm(x).Wc^T + bc) with the
// LayerNorm folded into Wc).  If A is null the producer is skipped and x = res goes through rows_ln_partials (the
// embedding path).  All pointers are device pointers; x_out fp32 [M, d], out fp32 [M, N].
int bw_test_ln_chain(const void* A, const void* Wp, const float* bp, const float* res, const float* gamma, const float* beta,
                     const float* Wc, const float* bc, int32_t M, int32_t d, int32_t Kp, int32_t N, int32_t gelu, float* x_out,
                     float* out, void* stream) {
  BW_API_BEGIN
  BW_CHECK(res && gamma && beta && Wc && x_out && out && M > 0 && d > 0 && N > 0 && d % 64 == 0 && N % 64 == 0, "bad argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  DevBuf Wf, c1, c2, xb, lst;
  Wf.alloc((size_t)N * d * 2); c1.alloc((size_t)N * 4); c2.alloc((size_t)N * 4);
  xb.alloc((size_t)M * d * 2); lst.alloc((size_t)M * (d / 64) * sizeof(float2));
  fold_layernorm(Wc, gamma, beta, bc, N, d, Wf.as<bf16>(), c1.as<float>(), c2.as<float>(), st);
  BW_CUDA(cudaMemcpyAsync(x_out, res, (size_t)M * d * 4, cudaMemcpyDeviceToDevice, st));
  if (A) {
    GemmArgs g;
    g.A = A; g.B = Wp; g.M = M; g.N = d; g.K = Kp; g.lda = Kp; g.ldb = Kp; g.ldc = d; g.ldres = d;
    g.bias = bp; g.residual = x_out; g.C = x_out; g.out_fp32 = true; g.xb_out = xb.p; g.ln_stats_out = lst.as<float2>();
    gemm_tc_rows(g, st);
  } else {
    rows_ln_partials(x_out, M, d, xb.as<bf16>(), lst.as<float2>(), st);
  }
  GemmArgs c;
  c.A = xb.p; c.B = Wf.p; c.M = M; c.N = N; c.K = d; c.lda = d; c.ldb = d; c.ldc = N;
  c.bias = c2.as<float>(); c.C = out; c.out_fp32 = true; c.gelu = gelu != 0;
  c.ln_stats_in = lst.as<float2>(); c.ln_c1 = c1.as<float>();
  gemm_tc_rows(c, st);
  BW_CUDA(cudaStreamSynchronize(st));
  BW_API_END
}

int bw_attention_bf16(int impl, const void* qkv, void* out, int32_t batch, int32_t T_len, int32_t n_head, void* stream) {
  BW_API_BEGIN
  if (impl == 0) attn_encoder_tc(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(out), batch, T_len, n_head, reinterpret_cast<cudaStream_t>(stream));
  else attn_encoder_simt<bf16>(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(out), batch, T_len, n_head, reinterpret_cast<cudaStream_t>(stream));
  BW_API_END
}

namespace {
// Deterministic pseudo-random fill (unit-variance-ish values in [-1.7, 1.7)): the timed kernels must not run on zeros
// (bandwidth is data independent, power and therefore clocks under a power cap are not).
template <typename T>
__global__ void fill_random_kernel(T* p, long long n, unsigned long long seed, float scale) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(i + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    const float u = (float)(unsigned int)(z >> 40) * (1.f / 16777216.f);  // [0, 1)
    p[i] = from_f<T>((u - 0.5f) * 3.4f * scale);
  }
}
template <typename T>
void fill_random(T* p, long long n, unsigned long long seed, float scale, cudaStream_t st) {
  if (n <= 0) return;
  fill_random_kernel<T><<<148 * 8, 256, 0, st>>>(p, n, seed, scale);
  BW_CUDA(cudaGetLastError());
}
void fill_cross_cache(bw_engine* e, int n_segments) {
  if (e->cross_int8) {  // valid codes and scales: random bf16 K/V of each window through the cache's own quantizer
    const auto& d = e->dims;
    const CrossKV x = engine_cross_kv_desc(e);
    for (int i = 0; i < n_segments; ++i) {
      fill_random<bf16>(e->cross_stage.as<bf16>(), (long long)(e->cross_stage.bytes / 2), 0x5eedull + i, 1.f, e->stream);
      cross_kv_int8_write(e->cross_stage.as<bf16>(), nullptr, nullptr, 1, d.n_text_layer, d.n_audio_ctx, d.n_text_state,
                          e->cross_cache.as<unsigned char>() + (long long)i * x.slot_stride, e->stream);
    }
    return;
  }
  const long long n = (long long)n_segments * (long long)(e->cross_cache.bytes / e->Q) / (e->fp32 ? 4 : 2);
  if (e->fp32) fill_random<float>(e->cross_cache.as<float>(), n, 0x5eedull, 1.f, e->stream);
  else fill_random<bf16>(e->cross_cache.as<bf16>(), n, 0x5eedull, 1.f, e->stream);
}
// algorithmic bytes of one layer's cached K/V of one window: codes + scales in the 8-bit mode
double cross_layer_bytes(const bw_engine* e) {
  const double d = e->dims.n_text_state, T = e->dims.n_audio_ctx;
  return e->cross_int8 ? 2 * T * d + 2 * T * e->dims.n_text_head * 4.0 : 2 * T * d * (e->fp32 ? 4 : 2);
}
struct EvTimer {
  cudaEvent_t a = nullptr, b = nullptr;
  cudaStream_t st;
  explicit EvTimer(cudaStream_t s) : st(s) { BW_CUDA(cudaEventCreate(&a)); BW_CUDA(cudaEventCreate(&b)); }
  ~EvTimer() { cudaEventDestroy(a); cudaEventDestroy(b); }
  void start() { BW_CUDA(cudaEventRecord(a, st)); }
  float stop_ms() { BW_CUDA(cudaEventRecord(b, st)); BW_CUDA(cudaEventSynchronize(b)); float ms = 0; BW_CUDA(cudaEventElapsedTime(&ms, a, b)); return ms; }
};
}  // namespace

int bw_bench_mel(bw_engine* e, int64_t n, int32_t iters, float* ms_out, double* bytes_out) {
  BW_API_BEGIN
  BW_CHECK(e && ms_out && bytes_out && iters > 0 && n > 400, "bad argument");
  DeviceGuard dg(e->device);
  const int nm = e->dims.n_mels;
  const int total = (int)((n + 480000) / 160);
  const int n_real = (int)std::min<long long>(total, (n + 200 + 159) / 160);
  const int ld = (n_real + 15) / 16 * 16;
  DevBuf pcm, logmel, gmax, a1;
  pcm.alloc((size_t)(n + 4) * 4); logmel.alloc((size_t)nm * ld * 4); gmax.alloc(4);
  fill_random<float>(pcm.as<float>(), (long long)n, 0x3e1ull, 0.25f, e->stream);
  BW_CUDA(cudaStreamSynchronize(e->stream));
  std::lock_guard<std::mutex> g(e->gpu_mu);
  EvTimer t(e->stream);
  auto once = [&] {
    mel_power(pcm.as<float>(), n, 480000, e->mel_tables.as<float>(), e->mel_filters.as<float>(), e->mel_ranges.as<int2>(), nm,
              logmel.as<float>(), ld, n_real, total, gmax.as<int>(), e->stream);
    engine_window_to_A1(e, logmel.as<float>(), ld, n_real, gmax.as<int>(), 0, std::min(3000, total - 3000), 0);
  };
  once();
  t.start();
  for (int i = 0; i < iters; ++i) once();
  *ms_out = t.stop_ms() / iters;
  // SURVEY 8(d): 4*(n+padding) read + 4*n_mels*(n+padding)/160 written
  *bytes_out = 4.0 * (double)(n + 480000) + 4.0 * nm * (double)total;
  BW_API_END
}

int bw_bench_encoder(bw_engine* e, int32_t batch, int32_t iters, float* ms_out, double* flops_out) {
  BW_API_BEGIN
  BW_CHECK(e && ms_out && flops_out && iters > 0, "bad argument");
  BW_CHECK(e->state == 1 && batch >= 1 && batch <= e->Be, "batch exceeds max_encoder_batch");
  DeviceGuard dg(e->device);
  std::lock_guard<std::mutex> g(e->gpu_mu);
  if (e->fp32) fill_random<float>(e->A1.as<float>(), (long long)(e->A1.bytes / 4), 0xa1ull, 0.5f, e->stream);
  else fill_random<bf16>(e->A1.as<bf16>(), (long long)(e->A1.bytes / 2), 0xa1ull, 0.5f, e->stream);
  engine_encoder_forward(e, batch);
  EvTimer t(e->stream);
  t.start();
  for (int i = 0; i < iters; ++i) engine_encoder_forward(e, batch);
  *ms_out = t.stop_ms() / iters;
  const double d = e->dims.n_audio_state, L = e->dims.n_audio_layer, nm = e->dims.n_mels;
  *flops_out = batch * (2.0 * 3000 * 3 * nm * d + 2.0 * 1500 * 3 * d * d + L * (8.0 * 1500 * d * d + 4.0 * 1500 * 1500 * d + 16.0 * 1500 * d * d));
  BW_API_END
}

namespace {
// Synthetic resident decode: `n_segments` windows x `n_group` hypotheses, positions [start_len, start_len + n_steps).
// pages of the synthetic decode: hypothesis slot u, block b -> page u * nb + b (the engine is idle: every page is free)
int synthetic_pages(bw_engine* e, int n_segments, int n_group, int max_len) {
  const int nb = kv_blocks_for(max_len);
  BW_CHECK((long long)n_segments * n_group * nb <= e->n_pages, "synthetic decode exceeds the self-KV page pool");
  std::vector<int> pt((size_t)e->S * e->n_blocks, 0);
  for (int u = 0; u < n_segments * n_group; ++u)
    for (int b = 0; b < nb; ++b) pt[(size_t)u * e->n_blocks + b] = u * nb + b;
  BW_CUDA(cudaMemcpy(e->d_page_table.p, pt.data(), pt.size() * 4, cudaMemcpyHostToDevice));
  return nb;
}
void synthetic_init(bw_engine* e, int n_segments, int n_group, int start_len) {
  for (int i = 0; i < n_segments; ++i) {
    int* rec = e->h_init + i * kInitRecInts;
    rec[0] = i; rec[1] = n_group; rec[2] = 0; rec[3] = 3; rec[4] = start_len; rec[5] = i * n_group; rec[6] = 0; rec[7] = 1;
    rec[8] = 50; rec[9] = kMaxFinished; rec[10] = e->tt.timestamp_begin - 1000;
    rec[11] = rec[12] = rec[13] = rec[14] = rec[15] = 0;
  }
  BW_CUDA(cudaMemcpyAsync(e->d_init.p, e->h_init, (size_t)n_segments * kInitRecInts * 4, cudaMemcpyHostToDevice, e->stream));
  engine_init_requests(e, e->d_init.as<int>(), n_segments);
  BW_CUDA(cudaStreamSynchronize(e->stream));
}
// One step: the control block filled as decode_step() fills it for decodes past their prompt, then the control
// upload, launches and completion read-back of decode_step() itself (enqueue_step, finish_step).
void synthetic_step(bw_engine* e, int n_segments, int n_group, int cur, int nb) {
  Ctl& c = e->dec.ctl;
  c.reset();
  for (int i = 0; i < n_segments; ++i) {
    c.grp_first[c.NG] = c.R; c.grp_n[c.NG] = n_group; c.grp_x[c.NG] = i; ++c.NG;
    c.max_grp = std::max(c.max_grp, n_group);
    c.max_ctx = std::max(c.max_ctx, cur);
    c.act_req[c.NA] = i; c.act_first[c.NA] = c.SR; c.act_force[c.NA] = -1; ++c.NA;
    for (int j = 0; j < n_group; ++j) {
      c.row_seq[c.R] = i * n_group + j; c.row_pos[c.R] = cur - 1; c.row_tok[c.R] = -1; c.row_bpos[c.R] = cur - 1;
      c.row_page[c.R] = (i * n_group + j) * nb + (cur - 1) / kPageTokens;
      c.lrow_src[c.LR] = c.R; c.srow_lrow[c.SR] = c.LR; c.srow_req[c.SR] = i; c.srow_seq[c.SR] = i * n_group + j;
      ++c.R; ++c.LR; ++c.SR;
    }
  }
  enqueue_step(e);
  finish_step(e);
}
}  // namespace

// One full decoder step (all layers + logits + sampling + beam update) over `n_segments` resident
// windows with `n_group` hypotheses each at context length `context_len`, timed with CUDA events.
int bw_bench_decoder_step(bw_engine* e, int32_t n_segments, int32_t n_group, int32_t context_len, int32_t iters, float* ms_out,
                          double* bytes_out) {
  BW_API_BEGIN
  BW_CHECK(e && ms_out && bytes_out && iters > 0, "bad argument");
  BW_CHECK(e->state == 1, "engine not finalized");
  BW_CHECK(n_segments >= 1 && n_segments <= e->Q && n_group >= 1 && n_group <= kMaxBeam && n_segments * n_group <= e->S, "exceeds pools");
  BW_CHECK(context_len >= 4 && context_len + iters + 2 < e->dims.n_text_ctx, "context_len out of range");
  DeviceGuard dg(e->device);
  std::lock_guard<std::mutex> g(e->gpu_mu);
  BW_CHECK(e->live.empty(), "engine busy");
  fill_cross_cache(e, n_segments);
  BW_CHECK(e->stat_pages_in_use == 0, "engine busy");
  const int nb = synthetic_pages(e, n_segments, n_group, context_len + iters + 2);
  {
    const long long n = (long long)n_segments * n_group * nb * (long long)(e->page_bytes / (e->fp32 ? 4 : 2));
    if (e->fp32) fill_random<float>(e->self_pool.as<float>(), n, 0x5e1full, 1.f, e->stream);
    else fill_random<bf16>(e->self_pool.as<bf16>(), n, 0x5e1full, 1.f, e->stream);
  }
  synthetic_init(e, n_segments, n_group, context_len);
  int cur = context_len;
  synthetic_step(e, n_segments, n_group, cur++, nb);
  EvTimer t(e->stream);  // e->stream is idle here; every step ends in a host synchronisation with the decoder stream
  t.start();
  for (int i = 0; i < iters; ++i) synthetic_step(e, n_segments, n_group, cur++, nb);
  *ms_out = t.stop_ms() / iters;
  const double ts = e->fp32 ? 4 : 2, d = e->dims.n_text_state, L = e->dims.n_text_layer, V = e->dims.n_vocab;
  const double S = (double)n_segments * n_group;
  *bytes_out = ts * (L * 14 * d * d + V * d) + n_segments * L * cross_layer_bytes(e) + S * ts * L * 2 * (context_len + iters / 2.0) * d + 4 * S * V;
  BW_API_END
}

// The whole hot path on device-resident PCM: log-mel -> encoder (batches of max_encoder_batch) -> cross-KV ->
// `n_steps` batched decoder steps for `n_segments` windows of `n_samples` samples each.  One CUDA-event pair
// on the engine stream brackets everything (bench.py `value`: inputs resident in HBM when timing starts).
int bw_bench_pipeline(bw_engine* e, const float* pcm_host, const int64_t* offsets, const int64_t* lengths, int32_t n_segments,
                      int32_t n_group, int32_t n_steps, float* ms_out) {
  BW_API_BEGIN
  BW_CHECK(e && pcm_host && offsets && lengths && ms_out, "bad argument");
  BW_CHECK(e->state == 1, "engine not finalized");
  BW_CHECK(n_segments >= 1 && n_segments <= e->Q && n_group >= 1 && n_group <= kMaxBeam && n_segments * n_group <= e->S, "exceeds pools");
  BW_CHECK(n_steps >= 1 && 3 + n_steps < e->dims.n_text_ctx, "n_steps out of range");
  for (int i = 0; i < n_segments; ++i) BW_CHECK(lengths[i] > 400 && lengths[i] <= e->call_pcm_cap, "segment length out of range");
  DeviceGuard dg(e->device);
  std::lock_guard<std::mutex> g(e->gpu_mu);
  BW_CHECK(e->live.empty(), "engine busy");
  std::vector<CallBuf> bufs;
  {
    std::lock_guard<std::mutex> cg(e->call_mu);
    BW_CHECK((int)e->call_pool.size() >= n_segments, "not enough call buffers");
    for (int i = 0; i < n_segments; ++i) { bufs.push_back(e->call_pool.back()); e->call_pool.pop_back(); }
  }
  for (int i = 0; i < n_segments; ++i)
    BW_CUDA(cudaMemcpyAsync(bufs[i].pcm, pcm_host + offsets[i], (size_t)lengths[i] * 4, cudaMemcpyHostToDevice, e->stream));
  BW_CUDA(cudaStreamSynchronize(e->stream));
  BW_CHECK(e->stat_pages_in_use == 0, "engine busy");
  const int nb = synthetic_pages(e, n_segments, n_group, 3 + n_steps + 1);
  auto frames = [&](int i, int& total, int& n_real, int& seg) {
    total = (int)((lengths[i] + 480000) / 160);
    n_real = (int)std::min<long long>(total, (lengths[i] + 200 + 159) / 160);
    seg = std::min(3000, total - 3000);
  };
  EvTimer t(e->stream);
  t.start();
  for (int i = 0; i < n_segments; ++i) {
    int total, n_real, seg;
    frames(i, total, n_real, seg);
    mel_power(bufs[i].pcm, lengths[i], 480000, e->mel_tables.as<float>(), e->mel_filters.as<float>(), e->mel_ranges.as<int2>(),
              e->dims.n_mels, bufs[i].logmel, bufs[i].ld, n_real, total, bufs[i].gmax, e->stream);
  }
  for (int s0 = 0; s0 < n_segments; s0 += e->Be) {
    const int nb = std::min(e->Be, n_segments - s0);
    for (int i = 0; i < nb; ++i) {
      int total, n_real, seg;
      frames(s0 + i, total, n_real, seg);
      engine_window_to_A1(e, bufs[s0 + i].logmel, bufs[s0 + i].ld, n_real, bufs[s0 + i].gmax, 0, seg, i);
    }
    engine_encoder_forward(e, nb);
    for (int i = 0; i < nb; ++i) engine_cross_kv(e, i, s0 + i);
  }
  synthetic_init(e, n_segments, n_group, 3);
  for (int i = 0; i < n_steps; ++i) synthetic_step(e, n_segments, n_group, 3 + i, nb);
  *ms_out = t.stop_ms();
  {
    std::lock_guard<std::mutex> cg(e->call_mu);
    for (auto& b : bufs) e->call_pool.push_back(b);
  }
  BW_API_END
}

// What the last bw_bench_pipeline decoded (same n_segments / n_group / n_steps), finalised per window as a decode
// request's result: the pipeline leaves window i's decoder state in request slot i, sequences i * n_group onwards.
int bw_bench_pipeline_results(bw_engine* e, int32_t n_segments, int32_t n_group, int32_t n_steps, float length_penalty,
                              bw_result* out) {
  BW_API_BEGIN
  BW_CHECK(e && out, "bad argument");
  BW_CHECK(e->state == 1, "engine not finalized");
  BW_CHECK(n_segments >= 1 && n_segments <= e->Q && n_group >= 1 && n_group <= kMaxBeam && n_segments * n_group <= e->S, "exceeds pools");
  BW_CHECK(n_steps >= 1 && 3 + n_steps < e->dims.n_text_ctx, "n_steps out of range");
  DeviceGuard dg(e->device);
  std::lock_guard<std::mutex> g(e->gpu_mu);
  BW_CHECK(e->live.empty(), "engine busy");
  const size_t blob = fin_blob_bytes(e);
  for (int i = 0; i < n_segments; ++i) {
    int* rec = e->h_init + i * 3;
    rec[0] = i; rec[1] = i * n_group; rec[2] = n_group;
  }
  BW_CUDA(cudaMemcpyAsync(e->d_init.p, e->h_init, (size_t)n_segments * 12, cudaMemcpyHostToDevice, e->stream));
  engine_gather_final(e, e->d_init.as<int>(), n_segments, (int)blob, e->d_fin.as<unsigned char>());
  BW_CUDA(cudaMemcpyAsync(e->h_fin, e->d_fin.p, (size_t)n_segments * blob, cudaMemcpyDeviceToHost, e->stream));
  BW_CUDA(cudaStreamSynchronize(e->stream));
  for (int i = 0; i < n_segments; ++i) {
    Request r;  // as synthetic_init admitted it: 3 prompt tokens, beam-search bookkeeping, then n_steps steps
    r.initial.assign(3, 0);
    r.greedy = 0;
    r.G = n_group;
    r.cur_len = 3 + n_steps;
    r.steps = n_steps;
    r.length_penalty = length_penalty;
    r.out = out + i;
    finalize_decode(e, &r, e->h_fin + (size_t)i * blob);
  }
  BW_API_END
}

// The decoder step's dominant kernel alone: cross-attention of one layer over resident K/V.
int bw_bench_cross_attention(bw_engine* e, int32_t n_segments, int32_t n_group, int32_t iters, float* ms_out, double* bytes_out) {
  BW_API_BEGIN
  BW_CHECK(e && ms_out && bytes_out && iters > 0, "bad argument");
  BW_CHECK(e->state == 1 && n_segments >= 1 && n_segments <= e->Q && n_group >= 1 && n_group <= kMaxBeam, "exceeds pools");
  BW_CHECK(n_segments * n_group <= e->R_max, "too many rows");
  DeviceGuard dg(e->device);
  std::lock_guard<std::mutex> g(e->gpu_mu);
  DecWorkspace& W = e->dec;
  Ctl& ctl = W.ctl;
  for (int i = 0; i < n_segments; ++i) { ctl.grp_first[i] = i * n_group; ctl.grp_n[i] = n_group; ctl.grp_x[i] = i; }
  BW_CUDA(cudaMemcpyAsync(W.d_ctrl.p, ctl.base, ctl.total * 4, cudaMemcpyHostToDevice, e->stream));
  fill_cross_cache(e, n_segments);
  const auto& d = e->dims;
  const int dm = d.n_text_state, L = d.n_text_layer;
  const int R = n_segments * n_group;
  fill_random<float>(W.d_q.as<float>(), (long long)R * dm, 0x9ull, 1.f, e->stream);
  auto run = [&](int layer) {
    const CrossKV x = engine_cross_kv_desc(e);
    if (e->fp32)
      dec_cross_attention<float>(W.dev(ctl.grp_first), W.dev(ctl.grp_n), W.dev(ctl.grp_x), n_segments, n_group, R, W.d_q.as<float>(), x,
                                 layer, dm, d.n_text_head, W.d_att.as<float>(), W.d_ws.as<float>(), e->stream);
    else
      dec_cross_attention<bf16>(W.dev(ctl.grp_first), W.dev(ctl.grp_n), W.dev(ctl.grp_x), n_segments, n_group, R, W.d_q.as<float>(), x,
                                layer, dm, d.n_text_head, W.d_att.as<bf16>(), W.d_ws.as<float>(), e->stream);
  };
  run(0);
  EvTimer t(e->stream);
  t.start();
  // walk the layers so that consecutive launches touch different K/V (as in the real step): inputs > L2
  for (int i = 0; i < iters; ++i) run(i % L);
  *ms_out = t.stop_ms() / iters;
  const double ts = e->fp32 ? 4 : 2;
  *bytes_out = (double)n_segments * cross_layer_bytes(e) + (double)R * dm * ts * 2;
  BW_API_END
}

int bw_debug_trace(bw_engine* e, int32_t enable, uint64_t* out, int32_t cap, int32_t* n_out) {
  BW_API_BEGIN
  // e may be null (kernel-level tools): then the current device is used
  int cur_dev = 0;
  BW_CUDA(cudaGetDevice(&cur_dev));
  DeviceGuard dg(e ? e->device : cur_dev);
  static std::mutex no_engine_mu;
  std::lock_guard<std::mutex> g(e ? e->gpu_mu : no_engine_mu);
  BW_CUDA(cudaDeviceSynchronize());
  static DevBuf buf;
  const size_t bytes = (1 + 2 * (size_t)kTraceCap) * 8;
  if (enable == 1) {
    if (buf.bytes < bytes) buf.alloc(bytes);
    BW_CUDA(cudaMemset(buf.p, 0, bytes));
    g_trace_dev = buf.as<unsigned long long>();
  } else if (enable == 2) {  // raw dump of the first `cap` records' worth of the buffer (fixed-slot users), then disarm
    BW_CHECK(out && cap >= 0, "null argument");
    unsigned long long* dev = g_trace_dev;
    g_trace_dev = nullptr;
    if (dev) BW_CUDA(cudaMemcpy(out, dev, std::min(bytes, (size_t)cap * 16), cudaMemcpyDeviceToHost));
  } else {
    BW_CHECK(out && n_out && cap >= 0, "null argument");
    unsigned long long* dev = g_trace_dev;
    g_trace_dev = nullptr;
    *n_out = 0;
    if (dev) {
      unsigned long long cnt = 0;
      BW_CUDA(cudaMemcpy(&cnt, dev, 8, cudaMemcpyDeviceToHost));
      const int n = (int)std::min<unsigned long long>(std::min<unsigned long long>(cnt, kTraceCap), (unsigned long long)cap);
      if (n > 0) BW_CUDA(cudaMemcpy(out, dev + 1, (size_t)n * 16, cudaMemcpyDeviceToHost));
      *n_out = n;
    }
  }
  BW_API_END
}

// ---- parity hooks for the bf16 product decoder ----
int bw_call_decode_forced(bw_call* c, int32_t seek, const bw_decode_opts* o, const int32_t* forced, int32_t n_forced,
                          float* step_logits, bw_result* out) {
  BW_API_BEGIN
  BW_CHECK(forced && n_forced >= 1, "forced tokens required");
  Request r;
  fill_decode_request(r, c, seek, o, out);
  BW_CHECK(r.greedy && r.G == 1 && r.temperature == 0.f, "teacher forcing needs GreedyDecoder semantics (beam_size 0, temperature 0)");
  BW_CHECK((int)r.initial.size() + n_forced <= c->eng->dims.n_text_ctx, "forced stream exceeds n_text_ctx");
  for (int i = 0; i < n_forced; ++i) BW_CHECK(forced[i] >= 0 && forced[i] < c->eng->dims.n_vocab, "token id out of range");
  r.forced.assign(forced, forced + n_forced);
  r.sample_len = n_forced;
  r.step_logits_out = step_logits;
  const int st = submit_and_wait(c->eng, r);
  if (st != BW_OK) return st;
  BW_API_END
}

int bw_test_dec_cross_attention(const void* cache, int32_t n_slots, int32_t n_layer, int32_t layer, int32_t T_enc, int32_t d,
                                int32_t n_head, const float* q, const int32_t* grp_first, const int32_t* grp_n,
                                const int32_t* grp_x, int32_t n_groups, int32_t max_group_rows, int32_t n_rows,
                                int32_t force_split, void* out, void* stream) {
  BW_API_BEGIN
  BW_CHECK(cache && q && grp_first && grp_n && grp_x && out, "null argument");
  BW_CHECK(n_slots >= 1 && n_layer >= 1 && layer >= 0 && layer < n_layer && d == 64 * n_head && n_groups >= 1 && n_rows >= 1, "bad geometry");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  DevBuf ws;
  ws.alloc(dec_cross_workspace_floats(n_rows, n_head) * 4);
  CrossKV x;
  x.cache = cache; x.slot_stride = (long long)n_layer * T_enc * 2 * d; x.T_enc = T_enc; x.n_slots = n_slots; x.n_layer = n_layer;
  dec_cross_attention<bf16>(grp_first, grp_n, grp_x, n_groups, max_group_rows, n_rows, q, x, layer, d, n_head,
                            reinterpret_cast<bf16*>(out), ws.as<float>(), st, force_split);
  BW_CUDA(cudaStreamSynchronize(st));
  BW_API_END
}

int bw_test_quantize_cross_kv(const void* x, int64_t n_rows, int32_t d, int8_t* codes, float* scales, void* stream) {
  BW_API_BEGIN
  BW_CHECK(x && codes && scales && n_rows >= 1 && d >= 64 && d % 64 == 0, "bad argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  quantize_int8_slices(reinterpret_cast<const bf16*>(x), n_rows * (d / 64), codes, scales, st);
  BW_CUDA(cudaStreamSynchronize(st));
  BW_API_END
}

int bw_test_dec_cross_attention_int8(const int8_t* codes, const float* scales, int32_t n_slots, int32_t n_layer, int32_t layer,
                                     int32_t T_enc, int32_t d, int32_t n_head, const float* q, const int32_t* grp_first,
                                     const int32_t* grp_n, const int32_t* grp_x, int32_t n_groups, int32_t max_group_rows,
                                     int32_t n_rows, int32_t force_split, void* out, void* stream) {
  BW_API_BEGIN
  BW_CHECK(codes && scales && q && grp_first && grp_n && grp_x && out, "null argument");
  BW_CHECK(n_slots >= 1 && n_layer >= 1 && layer >= 0 && layer < n_layer && d == 64 * n_head && n_groups >= 1 && n_rows >= 1 &&
           T_enc >= 1 && T_enc <= 1504, "bad geometry");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  CrossKV x;
  x.slot_stride = cross_int8_slot_bytes(n_layer, T_enc, n_head); x.T_enc = T_enc; x.n_slots = n_slots; x.n_layer = n_layer;
  x.int8 = true;
  DevBuf cache, ws;
  cache.alloc((size_t)(n_slots * x.slot_stride));
  ws.alloc(dec_cross_workspace_floats(n_rows, n_head) * 4);
  cross_kv_int8_write(nullptr, codes, scales, n_slots, n_layer, T_enc, d, cache.p, st);
  x.cache = cache.p;
  dec_cross_attention<bf16>(grp_first, grp_n, grp_x, n_groups, max_group_rows, n_rows, q, x, layer, d, n_head,
                            reinterpret_cast<bf16*>(out), ws.as<float>(), st, force_split);
  BW_CUDA(cudaStreamSynchronize(st));
  BW_API_END
}

int bw_test_dec_self_attention(int32_t n_rows, const int32_t* row_seq, const int32_t* row_pos, const int32_t* row_bpos,
                               const int32_t* row_page, const float* qkv, void* pool, int32_t n_layer, int32_t n_ctx, int32_t n_units,
                               const int32_t* page_table, const int32_t* seq_first, const uint8_t* anc, int32_t layer, int32_t d,
                               int32_t n_head, int32_t max_ctx, void* out, void* stream) {
  BW_API_BEGIN
  BW_CHECK(row_seq && row_pos && row_bpos && row_page && qkv && pool && page_table && seq_first && anc && out, "null argument");
  BW_CHECK(n_rows >= 1 && d == 64 * n_head && n_ctx >= 1 && layer >= 0 && layer < n_layer && n_units >= 1, "bad geometry");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  DecRows rows;
  rows.n_rows = n_rows; rows.row_seq = row_seq; rows.row_pos = row_pos; rows.row_bpos = row_bpos; rows.row_tok = nullptr;
  rows.row_page = row_page; rows.max_ctx = max_ctx;
  SelfKV kv;
  kv.pool = pool; kv.page_stride = (long long)n_layer * 2 * kPageTokens * d; kv.n_ctx = n_ctx;
  kv.n_blocks = (n_ctx + kPageTokens - 1) / kPageTokens; kv.n_units = n_units; kv.page_table = page_table;
  kv.seq_first = seq_first; kv.anc = anc;
  DevBuf pospage;
  pospage.alloc((size_t)n_rows * n_ctx * 4);
  kv.pospage = pospage.as<int>();
  dec_self_pospage(rows, kv, n_head, st);
  dec_self_attention<bf16>(rows, qkv, kv, layer, d, n_head, reinterpret_cast<bf16*>(out), st);
  BW_CUDA(cudaStreamSynchronize(st));
  BW_API_END
}

int bw_test_self_attention_mode(int32_t mode) {
  BW_API_BEGIN
  BW_CHECK(mode >= 0 && mode <= 3, "mode: 0 automatic, 1 staged, 2 warp per unit, 3 persistent warps");
  dec_self_attention_mode(mode);
  BW_API_END
}

int bw_test_sample_topk(bw_engine* e, const float* logits, int32_t n, const int32_t* state, int32_t* cand_tok, float* cand_lp) {
  BW_API_BEGIN
  BW_CHECK(e && logits && state && cand_tok && cand_lp && n >= 1, "bad argument");
  BW_CHECK(e->tables_set, "token tables not set");
  DeviceGuard dg(e->device);
  const int V = e->dims.n_vocab;
  // one request + G hypotheses per row; every hypothesis of a row shares the row's history (what sample_topk reads)
  std::vector<int> h_int((size_t)n * 13, 0);
  auto col = [&](int c) { return h_int.data() + (size_t)c * n; };
  int *n_beam = col(0), *greedy = col(1), *cur_len = col(2), *sample_begin = col(3), *without_ts = col(4), *suppress_blank = col(5),
      *max_initial_ts = col(6), *first_seq = col(7), *next_tok = col(8), *prev_tok = col(9), *last_ts = col(10), *lrow = col(11),
      *zero = col(12);
  for (int i = 0; i < n; ++i) {
    const int32_t* s = state + (size_t)i * 10;
    BW_CHECK(s[0] >= 1 && s[0] <= kMaxBeam, "n_beam out of range");
    n_beam[i] = s[0]; greedy[i] = s[1]; cur_len[i] = s[2]; sample_begin[i] = s[3]; without_ts[i] = s[4]; suppress_blank[i] = s[5];
    max_initial_ts[i] = s[6]; first_seq[i] = i; next_tok[i] = s[7]; prev_tok[i] = s[8]; last_ts[i] = s[9]; lrow[i] = i; zero[i] = 0;
  }
  DevBuf d_int, d_f, d_logits, d_tok, d_lp;
  d_int.alloc(h_int.size() * 4); d_f.alloc((size_t)n * 4); d_logits.alloc((size_t)n * V * 4);
  d_tok.alloc((size_t)n * kMaxCand * 4); d_lp.alloc((size_t)n * kMaxCand * 4);
  cudaStream_t st = e->front[0];
  std::lock_guard<std::mutex> g(e->front_mu[0]);
  BW_CUDA(cudaMemcpyAsync(d_int.p, h_int.data(), h_int.size() * 4, cudaMemcpyHostToDevice, st));
  BW_CUDA(cudaMemsetAsync(d_f.p, 0, (size_t)n * 4, st));  // temperature 0
  BW_CUDA(cudaMemcpyAsync(d_logits.p, logits, (size_t)n * V * 4, cudaMemcpyHostToDevice, st));
  BW_CUDA(cudaMemcpyAsync(d_tok.p, cand_tok, (size_t)n * kMaxCand * 4, cudaMemcpyHostToDevice, st));
  BW_CUDA(cudaMemcpyAsync(d_lp.p, cand_lp, (size_t)n * kMaxCand * 4, cudaMemcpyHostToDevice, st));
  auto dcol = [&](int c) { return d_int.as<int>() + (size_t)c * n; };
  ReqState rs{};
  SeqState ss{};
  rs.n_beam = dcol(0); rs.greedy = dcol(1); rs.cur_len = dcol(2); rs.sample_begin = dcol(3); rs.without_ts = dcol(4);
  rs.suppress_blank = dcol(5); rs.max_initial_ts = dcol(6); rs.first_seq = dcol(7); rs.temperature = d_f.as<float>();
  rs.seed_lo = reinterpret_cast<unsigned int*>(dcol(12)); rs.seed_hi = reinterpret_cast<unsigned int*>(dcol(12));
  ss.next_tok = dcol(8); ss.prev_tok = dcol(9); ss.last_ts = dcol(10);
  sample_topk(d_logits.as<float>(), V, V, dcol(11), dcol(11), dcol(11), n, e->tt, rs, ss, 0, d_tok.as<int>(), d_lp.as<float>(), st);
  BW_CUDA(cudaMemcpyAsync(cand_tok, d_tok.p, (size_t)n * kMaxCand * 4, cudaMemcpyDeviceToHost, st));
  BW_CUDA(cudaMemcpyAsync(cand_lp, d_lp.p, (size_t)n * kMaxCand * 4, cudaMemcpyDeviceToHost, st));
  BW_CUDA(cudaStreamSynchronize(st));
  BW_API_END
}

int bw_test_page_collector(int32_t n_hypotheses, int32_t n_initial, int32_t n_steps, const uint8_t* parents, uint8_t* alloc_masks,
                           int32_t* pages_in_use) {
  BW_API_BEGIN
  BW_CHECK(parents && alloc_masks && pages_in_use && n_steps >= 1, "bad argument");
  const int st = page_collector_replay(n_hypotheses, n_initial, n_steps, parents, alloc_masks, pages_in_use);
  if (st != BW_OK) { last_error() = "page collector replay: bad geometry or pages leaked"; return st; }
  BW_API_END
}
