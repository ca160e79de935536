// C ABI (include/b200_whisper.h): engine life cycle, calls, stage-level entry points.
#include "sched.cuh"

using namespace bw;

namespace bw {
std::string& last_error() {
  static thread_local std::string err;
  return err;
}
}  // namespace bw

namespace {

void compute_call_mel(bw_engine* e, bw_call* c, const float* pcm, long long n) {
  const unsigned idx = e->front_rr.fetch_add(1) % bw_engine::kFrontStreams;
  std::lock_guard<std::mutex> g(e->front_mu[idx]);
  cudaStream_t st = e->front[idx];
  BW_CUDA(cudaMemcpyAsync(c->buf.pcm, pcm, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  mel_power(c->buf.pcm, n, 480000, e->mel_tables.as<float>(), e->mel_filters.as<float>(), e->mel_ranges.as<int2>(), e->dims.n_mels,
            c->buf.logmel, c->buf.ld, c->n_real, c->total_frames, c->buf.gmax, st);
  BW_CUDA(cudaEventRecord(c->mel_done, st));
  e->stat_h2d += n * 4;
}

// raw ingest: H2D of the int16 samples, conversion (+ resampling) into the call's f32 PCM buffer, then the log-mel
const Resampler* find_resampler(bw_engine* e, int sample_rate) {
  if (sample_rate == 16000) return nullptr;
  std::lock_guard<std::mutex> g(e->resampler_mu);
  auto it = e->resamplers.find(sample_rate);
  if (it == e->resamplers.end())
    throw std::invalid_argument("no resampler registered for " + std::to_string(sample_rate) + " Hz (bw_engine_set_resampler)");
  return it->second.get();
}
long long resampled_length(const Resampler* r, long long n) {
  return r ? ((long long)r->nw * n + r->orig - 1) / r->orig : n;
}
// enqueue on `st`: pcm16 (host) -> staging -> f32 PCM at 16 kHz in `dst`
void ingest_pcm16(bw_engine* e, int front_idx, cudaStream_t st, const int16_t* pcm, long long n, const Resampler* r, float* dst, long long n16) {
  DevBuf& stage = e->front_pcm16[front_idx];
  if (stage.bytes < (size_t)n * 2 + 16) {
    BW_CUDA(cudaStreamSynchronize(st));  // earlier users of the old staging buffer
    stage.alloc(std::max((size_t)n * 2 + 16, (size_t)4 << 20));
  }
  BW_CUDA(cudaMemcpyAsync(stage.p, pcm, (size_t)n * 2, cudaMemcpyHostToDevice, st));
  if (r) pcm16_resample(stage.as<int16_t>(), n, r->taps.as<float>(), r->ranges.as<int2>(), r->orig, r->nw, r->K, r->width, dst, n16, st);
  else pcm16_to_f32(stage.as<int16_t>(), n, dst, st);
  e->stat_h2d += n * 2;
}

}  // namespace

// ================================================================================================
extern "C" {

const char* bw_last_error(void) { return last_error().c_str(); }
int bw_version(void) { return 100; }
int bw_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int bw_engine_create(const bw_model_dims* dims, const bw_engine_config* cfg, bw_engine** out) {
  BW_API_BEGIN
  BW_CHECK(dims && cfg && out, "null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { last_error() = "no CUDA device visible"; return BW_ERR_NO_DEVICE; }
  BW_CHECK(cfg->cuda_device >= 0 && cfg->cuda_device < ndev, "cuda_device out of range");
  cudaDeviceProp prop;
  BW_CUDA(cudaGetDeviceProperties(&prop, cfg->cuda_device));
  if (prop.major != 10) { last_error() = std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) + ", this library is built for sm_100a only"; return BW_ERR_NO_DEVICE; }
  BW_CHECK(dims->n_audio_state == dims->n_audio_head * 64 && dims->n_text_state == dims->n_text_head * 64, "head dim must be 64");
  BW_CHECK(dims->n_audio_state == dims->n_text_state, "encoder/decoder width must match");
  BW_CHECK(dims->n_audio_ctx == 1500 && dims->n_text_ctx <= BW_MAX_TOKENS && dims->n_text_ctx >= 8, "unsupported context sizes");
  BW_CHECK(dims->n_audio_state <= 1280 && dims->n_audio_state % 64 == 0, "n_state must be <= 1280");
  BW_CHECK(dims->n_mels > 0 && dims->n_mels <= 128 && (dims->n_mels * 3) % 8 == 0, "unsupported n_mels");
  BW_CHECK(dims->n_vocab > 50000 && dims->n_vocab < 60000, "unsupported vocabulary size");
  DeviceGuard dg(cfg->cuda_device);
  auto e = std::make_unique<bw_engine>();
  e->dims = *dims;
  e->cfg = *cfg;
  e->device = cfg->cuda_device;
  e->fp32 = cfg->compute == BW_COMPUTE_FP32;
  e->force_simt = (cfg->flags & BW_FLAG_FORCE_SIMT_GEMM) != 0;
  e->cross_int8 = (cfg->flags & BW_FLAG_CROSS_KV_INT8) != 0;
  BW_CHECK(!e->cross_int8 || (!e->fp32 && !e->force_simt),
           "BW_FLAG_CROSS_KV_INT8 needs BW_COMPUTE_BF16 on the tensor-core path (not with BW_COMPUTE_FP32 or BW_FLAG_FORCE_SIMT_GEMM)");
  e->fuse_ln = !e->fp32 && !e->force_simt && (dims->n_text_state % 64) == 0 && getenv("B200W_NO_LN_FUSION") == nullptr;
  BW_CUDA(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  BW_CUDA(cudaEventCreateWithFlags(&e->enc_fork, cudaEventDisableTiming));
  for (int i = 0; i < bw_engine::kEncStreams; ++i) {
    BW_CUDA(cudaStreamCreateWithFlags(&e->enc_streams[i], cudaStreamNonBlocking));
    BW_CUDA(cudaEventCreateWithFlags(&e->enc_join[i], cudaEventDisableTiming));
  }
  for (auto& s : e->front) BW_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  e->staging.alloc((size_t)64 << 20);
  engine_build_weight_table(e.get());
  e->loaded.assign(e->expected_names.size() + 1, 0);
  // mel constant tables
  std::vector<float> tab(mel_tables_floats());
  mel_fill_tables(tab.data());
  e->mel_tables.alloc(tab.size() * 4);
  BW_CUDA(cudaMemcpy(e->mel_tables.p, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
  *out = e.release();
  BW_API_END
}

int bw_engine_load_weights(bw_engine* e, const bw_tensor_desc* tensors, int32_t n) {
  BW_API_BEGIN
  BW_CHECK(e && tensors, "null argument");
  BW_CHECK(e->state == 0, "weights must be loaded before bw_engine_finalize");
  DeviceGuard dg(e->device);
  for (int i = 0; i < n; ++i) engine_load_tensor(e, tensors[i]);
  BW_API_END
}

int bw_engine_set_tables(bw_engine* e, const bw_token_tables* t) {
  BW_API_BEGIN
  BW_CHECK(e && t, "null argument");
  DeviceGuard dg(e->device);
  const int V = e->dims.n_vocab;
  TokenTables& tt = e->tt;
  tt.eot = t->eot; tt.sot = t->sot; tt.sot_prev = t->sot_prev; tt.sot_lm = t->sot_lm; tt.no_speech = t->no_speech;
  tt.no_timestamps = t->no_timestamps; tt.timestamp_begin = t->timestamp_begin; tt.translate = t->translate;
  tt.transcribe = t->transcribe; tt.first_language_token = t->first_language_token; tt.num_languages = t->num_languages;
  BW_CHECK(t->n_blank >= 0 && t->n_blank <= 4, "at most 4 blank ids");
  BW_CHECK(t->timestamp_begin > 0 && t->timestamp_begin < V && t->eot < t->timestamp_begin, "bad token layout");
  BW_CHECK(t->num_languages <= 128, "too many languages");
  tt.n_blank = t->n_blank;
  for (int i = 0; i < 4; ++i) tt.blank[i] = (i < t->n_blank) ? t->blank[i] : -1;
  std::vector<unsigned int> bits((V + 31) / 32, 0u);
  for (int i = 0; i < t->n_suppress; ++i) {
    BW_CHECK(t->suppress[i] >= 0 && t->suppress[i] < V, "suppress id out of range");
    bits[t->suppress[i] >> 5] |= 1u << (t->suppress[i] & 31);
  }
  e->suppress_bits.alloc(bits.size() * 4);
  BW_CUDA(cudaMemcpy(e->suppress_bits.p, bits.data(), bits.size() * 4, cudaMemcpyHostToDevice));
  tt.suppress_bits = e->suppress_bits.as<unsigned int>();
  e->tables_set = true;
  BW_API_END
}

int bw_engine_set_mel_filters(bw_engine* e, const float* filters) {
  BW_API_BEGIN
  BW_CHECK(e && filters, "null argument");
  DeviceGuard dg(e->device);
  const int nm = e->dims.n_mels;
  std::vector<int2> ranges(nm);
  for (int m = 0; m < nm; ++m) {
    int lo = 201, hi = 0;
    for (int k = 0; k < 201; ++k)
      if (filters[m * 201 + k] != 0.f) { lo = std::min(lo, k); hi = std::max(hi, k + 1); }
    if (lo > hi) { lo = 0; hi = 0; }
    ranges[m] = make_int2(lo, hi);
  }
  e->mel_filters.alloc((size_t)nm * 201 * 4);
  e->mel_ranges.alloc((size_t)nm * sizeof(int2));
  BW_CUDA(cudaMemcpy(e->mel_filters.p, filters, (size_t)nm * 201 * 4, cudaMemcpyHostToDevice));
  BW_CUDA(cudaMemcpy(e->mel_ranges.p, ranges.data(), (size_t)nm * sizeof(int2), cudaMemcpyHostToDevice));
  e->filters_set = true;
  BW_API_END
}

int bw_engine_finalize(bw_engine* e) {
  BW_API_BEGIN
  BW_CHECK(e, "null argument");
  BW_CHECK(e->state == 0, "already finalized");
  BW_CHECK(e->tables_set && e->filters_set, "bw_engine_set_tables and bw_engine_set_mel_filters must be called first");
  DeviceGuard dg(e->device);
  const auto& d = e->dims;
  for (size_t i = 0; i < e->expected_names.size(); ++i)
    if (!e->loaded[i]) throw std::invalid_argument("missing weight tensor: " + e->expected_names[i]);
  if (!e->loaded.back()) {  // encoder.positional_embedding = sinusoids(n_audio_ctx, d)
    const int ch = d.n_audio_state, len = d.n_audio_ctx;
    std::vector<float> pe((size_t)len * ch);
    const float inc = (float)(log(10000.0) / (ch / 2 - 1));
    for (int t = 0; t < len; ++t)
      for (int i = 0; i < ch / 2; ++i) {
        const float inv = expf(-inc * (float)i);
        const float a = (float)t * inv;
        pe[(size_t)t * ch + i] = sinf(a);
        pe[(size_t)t * ch + ch / 2 + i] = cosf(a);
      }
    BW_CUDA(cudaMemcpy(e->w.enc_pos, pe.data(), pe.size() * 4, cudaMemcpyHostToDevice));
  }
  engine_fold_layernorms(e);
  const size_t ts = e->fp32 ? 4 : 2;
  const size_t dm = d.n_audio_state;
  const size_t cross_bf16 = (size_t)d.n_text_layer * d.n_audio_ctx * 2 * dm * ts;
  const size_t cross_slot = e->cross_int8 ? (size_t)cross_int8_slot_bytes(d.n_text_layer, d.n_audio_ctx, d.n_text_head) : cross_bf16;
  const size_t cross_stage = e->cross_int8 ? cross_bf16 : 0;
  // self-KV pool: pages of kPageTokens positions for one hypothesis slot, every layer ([L][2][kPageTokens][d]).
  // Default budget: 256 positions (16 pages) per hypothesis slot -- a decode holds at most n_initial + sample_len
  // (<= 3 + 224 without a prompt) positions per hypothesis, and beam hypotheses share the pages of their common
  // prefix -- but never less than one worst-case request (n_text_ctx positions x kMaxBeam hypotheses).
  e->n_blocks = (d.n_text_ctx + kPageTokens - 1) / kPageTokens;
  BW_CHECK(e->n_blocks <= kMaxBlocks, "n_text_ctx too large for the page table");
  e->page_bytes = (size_t)d.n_text_layer * 2 * kPageTokens * dm * ts;
  int Q = e->cfg.max_segments > 0 ? e->cfg.max_segments : 64;
  int S = e->cfg.max_sequences > 0 ? e->cfg.max_sequences : std::max(2 * Q, kMaxBeam);
  int Be = e->cfg.max_encoder_batch > 0 ? e->cfg.max_encoder_batch : 8;
  const int min_pages = e->n_blocks * kMaxBeam;
  auto pages_for = [&](int s) { return e->cfg.max_kv_pages > 0 ? std::max(e->cfg.max_kv_pages, min_pages) : std::max(s * 16, min_pages); };
  size_t free_b = 0, total_b = 0;
  BW_CUDA(cudaMemGetInfo(&free_b, &total_b));
  const size_t enc_per = (size_t)(3000 * 3 * d.n_mels + 3000 * dm + 1500 * 3 * dm + 1500 * dm * 2 + 1500 * 3 * dm + 1500 * dm +
                                  1500 * 4 * dm + 1500 * dm) * 4;  // upper bound (fp32 sizes)
  for (int guard = 0; guard < 64; ++guard) {
    const double need = (double)Q * cross_slot + (double)cross_stage + (double)pages_for(S) * e->page_bytes + (double)Be * enc_per;
    if (!(need > 0.80 * (double)free_b && (Q > 1 || S > kMaxBeam || Be > 1))) break;
    if (Q > 1) Q = std::max(1, Q * 3 / 4);
    S = std::max(kMaxBeam, std::min(S, std::max(2 * Q, kMaxBeam)));
    if (Be > 1) Be = std::max(1, Be / 2);
  }
  Be = std::min(Be, Q);
  e->Q = Q; e->S = S; e->Be = Be;
  e->R_max = S + 512;
  e->LR_max = S + Q + BW_MAX_TOKENS;
  e->cross_cache.alloc((size_t)Q * cross_slot);
  if (e->cross_int8) e->cross_stage.alloc(cross_stage);
  e->n_pages = pages_for(S);
  e->self_pool.alloc((size_t)e->n_pages * e->page_bytes);
  e->d_page_table.alloc((size_t)S * e->n_blocks * 4);
  BW_CUDA(cudaMemset(e->d_page_table.p, 0, e->d_page_table.bytes));
  e->free_pages.clear();
  for (int pg = e->n_pages - 1; pg >= 0; --pg) e->free_pages.push_back(pg);
  e->pages_reserved = 0;
  // encoder activations
  e->A1.alloc((size_t)Be * 3000 * 3 * d.n_mels * ts);
  e->y1.alloc((size_t)Be * 3000 * dm * ts);
  e->A2.alloc((size_t)Be * 1500 * 3 * dm * ts);
  e->enc_x.alloc((size_t)Be * 1500 * dm * 4);
  e->enc_xn.alloc((size_t)Be * 1500 * dm * ts);
  e->enc_qkv.alloc((size_t)Be * 1500 * 3 * dm * ts);
  e->enc_att.alloc((size_t)Be * 1500 * dm * ts);
  e->enc_h.alloc((size_t)Be * 1500 * 4 * dm * ts);
  e->enc_out.alloc((size_t)Be * 1500 * dm * ts);
  // decoder activations
  const size_t R = e->R_max, LR = e->LR_max;
  DecWorkspace& W = e->dec;
  BW_CUDA(cudaStreamCreateWithFlags(&W.stream, cudaStreamNonBlocking));
  W.d_x.alloc(R * dm * 4);
  W.d_xn.alloc(R * dm * ts); W.d_qkv.alloc(R * 3 * dm * 4); W.d_att.alloc(R * dm * ts); W.d_q.alloc(R * dm * 4);
  W.d_h.alloc(R * 4 * dm * ts); W.d_lnrows.alloc(LR * dm * ts);
  if (e->fuse_ln) {
    W.d_xb.alloc(R * dm * 2);
    W.d_lnst.alloc(R * (dm / 64) * sizeof(float2));
    BW_CUDA(cudaMemset(W.d_xb.p, 0, W.d_xb.bytes));
    BW_CUDA(cudaMemset(W.d_lnst.p, 0, W.d_lnst.bytes));
  }
  W.d_pospage.alloc(R * (size_t)d.n_text_ctx * 4);
  BW_CUDA(cudaMemset(W.d_pospage.p, 0, W.d_pospage.bytes));
  W.d_logits.alloc(LR * (size_t)d.n_vocab * 4);
  W.d_ws.alloc(dec_cross_workspace_floats((int)R, d.n_text_head) * 4);
  W.d_cand_tok.alloc(LR * kMaxCand * 4); W.d_cand_lp.alloc(LR * kMaxCand * 4);
  // rows past the live count are read (and discarded) by the GEMMs' TMA boxes: keep them finite
  for (DevBuf* b : {&W.d_xn, &W.d_qkv, &W.d_att, &W.d_q, &W.d_h, &W.d_lnrows}) BW_CUDA(cudaMemset(b->p, 0, b->bytes));
  e->d_lang_probs.alloc(128 * 4); e->d_lang_arg.alloc(4);
  e->d_det_probs.alloc((size_t)Q * kMaxLanguages * 4); e->d_det_tok.alloc((size_t)Q * 4);
  BW_CUDA(cudaMemset(e->d_det_probs.p, 0, e->d_det_probs.bytes));
  BW_CUDA(cudaMemset(e->d_det_tok.p, 0, e->d_det_tok.bytes));
  BW_CUDA(cudaMemset(e->self_pool.p, 0, e->self_pool.bytes));
  // decoder state
  const size_t n_ctx = d.n_text_ctx;
  e->st_int.alloc(((size_t)Q * 13 + (size_t)Q * kMaxFinished * 2 + (size_t)S * 4) * 4);
  e->st_float.alloc(((size_t)Q * kMaxFinished + 2 * (size_t)Q + S) * 4);
  e->st_anc0.alloc((size_t)S * n_ctx); e->st_anc1.alloc((size_t)S * n_ctx);
  e->st_tok.alloc((size_t)Q * n_ctx * kMaxBeam * 4); e->st_parent.alloc((size_t)Q * n_ctx * kMaxBeam);
  e->step_out_bytes = (size_t)Q * 4 + (size_t)Q * kMaxBeam;
  e->st_step.alloc(e->step_out_bytes);
  for (DevBuf* b : {&e->st_int, &e->st_float, &e->st_anc0, &e->st_anc1, &e->st_tok, &e->st_parent, &e->st_step}) BW_CUDA(cudaMemset(b->p, 0, b->bytes));
  {
    int* p = e->st_int.as<int>();
    auto take = [&](size_t n) { int* r = p; p += n; return r; };
    ReqState& rs = e->rs;
    rs.n_beam = take(Q); rs.greedy = take(Q); rs.sample_begin = take(Q); rs.cur_len = take(Q); rs.first_seq = take(Q);
    rs.without_ts = take(Q); rs.suppress_blank = take(Q); rs.max_initial_ts = take(Q); rs.max_candidates = take(Q);
    rs.n_finished = take(Q); (void)take(Q);
    rs.completed = e->st_step.as<int>();                                          // read back after every step ...
    rs.last_src = e->st_step.as<unsigned char>() + (size_t)Q * 4;                // ... together with the parent slots
    rs.seed_lo = reinterpret_cast<unsigned int*>(take(Q)); rs.seed_hi = reinterpret_cast<unsigned int*>(take(Q));
    rs.fin_pos = take((size_t)Q * kMaxFinished); rs.fin_slot = take((size_t)Q * kMaxFinished);
    SeqState& ss = e->ss;
    ss.next_tok = take(S); ss.prev_tok = take(S); ss.last_ts = take(S); ss.seq_first = take(S);
    float* f = e->st_float.as<float>();
    rs.fin_score = f; f += (size_t)Q * kMaxFinished;
    rs.no_speech_prob = f; f += Q;
    rs.temperature = f; f += Q;
    ss.sum_logprob = f;
    ss.anc[0] = e->st_anc0.as<unsigned char>(); ss.anc[1] = e->st_anc1.as<unsigned char>();
    rs.tok = e->st_tok.as<int>(); rs.parent = e->st_parent.as<unsigned char>();
  }
  // decoder-step control block + admission records
  {
    W.ctl.layout(nullptr, e->R_max, e->LR_max, Q);  // sizes only
    BW_CUDA(cudaMallocHost(reinterpret_cast<void**>(&W.h_ctrl), W.ctl.total * 4));
    W.ctl.layout(W.h_ctrl, e->R_max, e->LR_max, Q);
    W.d_ctrl.alloc(W.ctl.total * 4);
    BW_CUDA(cudaMallocHost(reinterpret_cast<void**>(&e->h_init), (size_t)Q * kInitRecInts * 4));
    e->d_init.alloc((size_t)Q * kInitRecInts * 4);
    BW_CUDA(cudaMallocHost(reinterpret_cast<void**>(&e->h_flags), e->step_out_bytes));
    e->h_fin_bytes = fin_blob_bytes(e) * (size_t)Q;
    BW_CUDA(cudaMallocHost(reinterpret_cast<void**>(&e->h_fin), e->h_fin_bytes));
    e->d_fin.alloc(e->h_fin_bytes);
  }
  // call buffers: sized for 30 s of audio; longer calls allocate on demand
  e->call_pcm_cap = 480000 + 1600;
  e->call_ld = 3008;
  const int n_calls = 2 * Q + 8;
  for (int i = 0; i < n_calls; ++i) {
    CallBuf b;
    BW_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.pcm), (size_t)e->call_pcm_cap * 4));
    BW_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.logmel), (size_t)d.n_mels * e->call_ld * 4));
    BW_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.gmax), 4));
    b.pcm_cap = e->call_pcm_cap; b.ld = e->call_ld; b.pooled = true;
    e->call_pool.push_back(b);
  }
  e->free_q.clear();
  for (int q = Q - 1; q >= 0; --q) e->free_q.push_back(q);
  e->seq_used.assign(S, 0);
  BW_CUDA(cudaDeviceSynchronize());
  e->state = 1;
  if (!(e->cfg.flags & BW_FLAG_NO_SCHEDULER)) e->sched = std::thread(scheduler_main, e);
  BW_API_END
}

int bw_engine_retain(bw_engine* e) {
  if (!e) return BW_ERR_INVALID;
  e->refs.fetch_add(1);
  return BW_OK;
}

int bw_engine_destroy(bw_engine* e) {
  BW_API_BEGIN
  if (!e) return BW_OK;
  if (e->refs.fetch_sub(1) > 1) return BW_OK;
  {
    std::lock_guard<std::mutex> g(e->q_mu);
    e->stop = true;
  }
  e->q_cv.notify_all();
  if (e->sched.joinable()) e->sched.join();
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  for (auto& b : e->call_pool) { cudaFree(b.pcm); cudaFree(b.logmel); cudaFree(b.gmax); }
  for (auto& kv : e->dec.graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  if (e->dec.h_ctrl) cudaFreeHost(e->dec.h_ctrl);
  if (e->dec.stream) cudaStreamDestroy(e->dec.stream);
  if (e->h_init) cudaFreeHost(e->h_init);
  if (e->h_flags) cudaFreeHost(e->h_flags);
  if (e->h_fin) cudaFreeHost(e->h_fin);
  for (auto& s : e->front) if (s) cudaStreamDestroy(s);
  if (e->enc_fork) cudaEventDestroy(e->enc_fork);
  for (int i = 0; i < bw_engine::kEncStreams; ++i) {
    if (e->enc_join[i]) cudaEventDestroy(e->enc_join[i]);
    if (e->enc_streams[i]) cudaStreamDestroy(e->enc_streams[i]);
  }
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
  BW_API_END
}

int bw_engine_stats(bw_engine* e, int64_t* out, int32_t n) {
  BW_API_BEGIN
  BW_CHECK(e && out, "null argument");
  int64_t v[BW_STAT_COUNT] = {0};
  v[BW_STAT_KERNEL_LAUNCHES] = g_kernel_launches.load();
  v[BW_STAT_DECODE_STEPS] = e->stat_steps; v[BW_STAT_ROWS] = e->stat_rows; v[BW_STAT_WINDOWS] = e->stat_windows;
  v[BW_STAT_MAX_SEGMENTS] = e->Q; v[BW_STAT_MAX_SEQUENCES] = e->S; v[BW_STAT_ENCODER_BATCHES] = e->stat_enc_batches;
  v[BW_STAT_H2D_BYTES] = e->stat_h2d; v[BW_STAT_D2H_BYTES] = e->stat_d2h;
  v[BW_STAT_KV_PAGES_TOTAL] = e->n_pages; v[BW_STAT_KV_PAGES_IN_USE] = e->stat_pages_in_use; v[BW_STAT_KV_PAGES_PEAK] = e->stat_pages_peak;
  v[BW_STAT_KV_PAGE_BYTES] = (int64_t)e->page_bytes;
  for (int i = 0; i < n && i < BW_STAT_COUNT; ++i) out[i] = v[i];
  BW_API_END
}

// ---- calls ----
int bw_call_open(bw_engine* e, const float* pcm, int64_t n_samples, bw_call** out) {
  BW_API_BEGIN
  BW_CHECK(e && pcm && out, "null argument");
  BW_CHECK(e->state == 1, "engine not finalized");
  BW_CHECK(n_samples >= 1, "empty audio");
  DeviceGuard dg(e->device);
  auto c = std::make_unique<bw_call>();
  c->eng = e;
  c->n_samples = n_samples;
  c->total_frames = (int)((n_samples + 480000) / 160);
  c->content_frames = c->total_frames - 3000;
  c->n_real = (int)std::min<long long>(c->total_frames, (n_samples + 200 + 159) / 160);
  {
    std::lock_guard<std::mutex> g(e->call_mu);
    if (n_samples <= e->call_pcm_cap && c->n_real <= e->call_ld && !e->call_pool.empty()) {
      c->buf = e->call_pool.back();
      e->call_pool.pop_back();
    }
  }
  if (!c->buf.pcm) {
    CallBuf b;
    b.ld = (c->n_real + 15) / 16 * 16;
    b.pcm_cap = n_samples;
    BW_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.pcm), (size_t)(n_samples + 4) * 4));
    BW_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.logmel), (size_t)e->dims.n_mels * b.ld * 4));
    BW_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.gmax), 4));
    c->buf = b;
  }
  BW_CUDA(cudaEventCreateWithFlags(&c->mel_done, cudaEventDisableTiming));
  compute_call_mel(e, c.get(), pcm, n_samples);
  e->refs.fetch_add(1);  // released by bw_call_close
  *out = c.release();
  BW_API_END
}

int bw_engine_set_resampler(bw_engine* e, int32_t sample_rate, int32_t orig_freq, int32_t new_freq, int32_t width, const float* taps) {
  BW_API_BEGIN
  BW_CHECK(e && taps, "null argument");
  BW_CHECK(sample_rate > 0 && sample_rate != 16000, "16 kHz needs no resampler");
  BW_CHECK(orig_freq > 0 && new_freq > 0 && width > 0 && orig_freq <= 4096 && new_freq <= 4096 && width <= 4096, "bad filter geometry");
  BW_CHECK((long long)sample_rate * new_freq == 16000LL * orig_freq, "orig_freq / new_freq must equal sample_rate / 16000");
  DeviceGuard dg(e->device);
  auto r = std::make_unique<Resampler>();
  r->orig = orig_freq; r->nw = new_freq; r->width = width; r->K = 2 * width + orig_freq;
  std::vector<int2> ranges(new_freq);
  for (int i = 0; i < new_freq; ++i) {
    int lo = r->K, hi = 0;
    for (int k = 0; k < r->K; ++k)
      if (fabsf(taps[(size_t)i * r->K + k]) >= 1e-20f) { lo = std::min(lo, k); hi = std::max(hi, k + 1); }
    if (lo > hi) { lo = 0; hi = 0; }
    ranges[i] = make_int2(lo, hi);
  }
  r->taps.alloc((size_t)new_freq * r->K * 4);
  r->ranges.alloc((size_t)new_freq * sizeof(int2));
  BW_CUDA(cudaMemcpy(r->taps.p, taps, (size_t)new_freq * r->K * 4, cudaMemcpyHostToDevice));
  BW_CUDA(cudaMemcpy(r->ranges.p, ranges.data(), (size_t)new_freq * sizeof(int2), cudaMemcpyHostToDevice));
  std::lock_guard<std::mutex> g(e->resampler_mu);
  BW_CHECK(e->resamplers.find(sample_rate) == e->resamplers.end(), "resampler already registered for this rate");
  e->resamplers[sample_rate] = std::move(r);
  BW_API_END
}

int bw_call_open_pcm16(bw_engine* e, const int16_t* pcm, int64_t n_in, int32_t sample_rate, bw_call** out) {
  BW_API_BEGIN
  BW_CHECK(e && pcm && out, "null argument");
  BW_CHECK(e->state == 1, "engine not finalized");
  BW_CHECK(n_in >= 1, "empty audio");
  DeviceGuard dg(e->device);
  const Resampler* r = find_resampler(e, sample_rate);
  const long long n_samples = resampled_length(r, n_in);
  BW_CHECK(n_samples >= 1, "empty audio after resampling");
  auto c = std::make_unique<bw_call>();
  c->eng = e;
  c->n_samples = n_samples;
  c->total_frames = (int)((n_samples + 480000) / 160);
  c->content_frames = c->total_frames - 3000;
  c->n_real = (int)std::min<long long>(c->total_frames, (n_samples + 200 + 159) / 160);
  {
    std::lock_guard<std::mutex> g(e->call_mu);
    if (n_samples <= e->call_pcm_cap && c->n_real <= e->call_ld && !e->call_pool.empty()) {
      c->buf = e->call_pool.back();
      e->call_pool.pop_back();
    }
  }
  if (!c->buf.pcm) {
    CallBuf b;
    b.ld = (c->n_real + 15) / 16 * 16;
    b.pcm_cap = n_samples;
    BW_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.pcm), (size_t)(n_samples + 4) * 4));
    BW_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.logmel), (size_t)e->dims.n_mels * b.ld * 4));
    BW_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.gmax), 4));
    c->buf = b;
  }
  BW_CUDA(cudaEventCreateWithFlags(&c->mel_done, cudaEventDisableTiming));
  {
    const unsigned idx = e->front_rr.fetch_add(1) % bw_engine::kFrontStreams;
    std::lock_guard<std::mutex> g(e->front_mu[idx]);
    cudaStream_t st = e->front[idx];
    ingest_pcm16(e, (int)idx, st, pcm, n_in, r, c->buf.pcm, n_samples);
    mel_power(c->buf.pcm, n_samples, 480000, e->mel_tables.as<float>(), e->mel_filters.as<float>(), e->mel_ranges.as<int2>(),
              e->dims.n_mels, c->buf.logmel, c->buf.ld, c->n_real, c->total_frames, c->buf.gmax, st);
    BW_CUDA(cudaEventRecord(c->mel_done, st));
  }
  e->refs.fetch_add(1);  // released by bw_call_close
  *out = c.release();
  BW_API_END
}

int bw_resample_pcm16(bw_engine* e, const int16_t* pcm, int64_t n_in, int32_t sample_rate, float* out, int64_t* n_out) {
  BW_API_BEGIN
  BW_CHECK(e && pcm && out && n_out, "null argument");
  BW_CHECK(n_in >= 1, "empty audio");
  DeviceGuard dg(e->device);
  const Resampler* r = find_resampler(e, sample_rate);
  const long long n16 = resampled_length(r, n_in);
  DevBuf dst;
  dst.alloc((size_t)(n16 + 4) * 4);
  std::lock_guard<std::mutex> g(e->front_mu[0]);
  ingest_pcm16(e, 0, e->front[0], pcm, n_in, r, dst.as<float>(), n16);
  BW_CUDA(cudaMemcpyAsync(out, dst.p, (size_t)n16 * 4, cudaMemcpyDeviceToHost, e->front[0]));
  BW_CUDA(cudaStreamSynchronize(e->front[0]));
  *n_out = n16;
  BW_API_END
}

int bw_call_content_frames(bw_call* c, int32_t* out) {
  if (!c || !out) return BW_ERR_INVALID;
  *out = c->content_frames;
  return BW_OK;
}

int bw_call_close(bw_call* c) {
  BW_API_BEGIN
  if (!c) return BW_OK;
  bw_engine* e = c->eng;
  DeviceGuard dg(e->device);
  cudaEventSynchronize(c->mel_done);
  cudaEventDestroy(c->mel_done);
  if (c->buf.pooled) {
    std::lock_guard<std::mutex> g(e->call_mu);
    e->call_pool.push_back(c->buf);
  } else {
    cudaFree(c->buf.pcm); cudaFree(c->buf.logmel); cudaFree(c->buf.gmax);
  }
  delete c;
  return bw_engine_destroy(e);  // the call's reference
  BW_API_END
}

int bw_call_decode(bw_call* c, int32_t seek, const bw_decode_opts* o, bw_result* out) {
  BW_API_BEGIN
  Request r;
  fill_decode_request(r, c, seek, o, out);
  const int st = submit_and_wait(c->eng, r);
  if (st != BW_OK) return st;
  BW_API_END
}

int bw_call_decode_detect(bw_call* c, int32_t seek, const bw_decode_opts* o, bw_result* out, bw_lang_result* lang) {
  BW_API_BEGIN
  BW_CHECK(lang, "null argument");
  Request r;
  fill_decode_request(r, c, seek, o, out, lang);
  const int st = submit_and_wait(c->eng, r);
  if (st != BW_OK) return st;
  BW_API_END
}

int bw_decode_many(bw_call* const* calls, const int32_t* seeks, const bw_decode_opts* opts, bw_result* results,
                   int32_t* statuses, int32_t n) {
  return bw_decode_many_detect(calls, seeks, opts, results, nullptr, statuses, n);
}

int bw_decode_many_detect(bw_call* const* calls, const int32_t* seeks, const bw_decode_opts* opts, bw_result* results,
                          bw_lang_result* langs, int32_t* statuses, int32_t n) {
  BW_API_BEGIN
  BW_CHECK(calls && seeks && opts && results && n >= 0, "null argument");
  std::vector<std::unique_ptr<Request>> reqs;
  std::vector<Request*> ptrs;
  bw_engine* e = n > 0 && calls[0] ? calls[0]->eng : nullptr;
  for (int i = 0; i < n; ++i) {
    BW_CHECK(calls[i] && calls[i]->eng == e, "all calls of a batch must belong to one engine");
    // detect mode: the window's initial tokens hold the language placeholder (fill_decode_request checks where)
    const bw_decode_opts& o = opts[i];
    const bool detect = langs && o.initial_tokens && o.n_initial > 0 &&
                        std::find(o.initial_tokens, o.initial_tokens + o.n_initial, kLanguagePlaceholder) != o.initial_tokens + o.n_initial;
    if (langs && !detect) memset(&langs[i], 0, sizeof(langs[i]));
    reqs.emplace_back(new Request());
    fill_decode_request(*reqs.back(), calls[i], seeks[i], &o, &results[i], detect ? &langs[i] : nullptr);
    ptrs.push_back(reqs.back().get());
  }
  if (n == 0) return BW_OK;
  const int st = submit_many_and_wait(e, ptrs);
  int first = BW_OK;
  for (int i = 0; i < n; ++i) {
    if (statuses) statuses[i] = reqs[i]->status;
    if (first == BW_OK && reqs[i]->status != BW_OK) { first = reqs[i]->status; last_error() = reqs[i]->error; }
  }
  if (st != BW_OK) return st;
  if (first != BW_OK) return first;
  BW_API_END
}

int bw_call_detect_language(bw_call* c, int32_t seek, bw_lang_result* out) {
  BW_API_BEGIN
  BW_CHECK(c && out, "null argument");
  bw_engine* e = c->eng;
  BW_CHECK(e->tt.num_languages > 0, "model has no language tokens");
  Request r;
  r.kind = REQ_LANG;
  r.call = c;
  r.seek = seek;
  r.initial = {e->tt.sot};
  r.G = 1;
  memset(out, 0, sizeof(*out));
  r.lang_out = out;
  const int st = submit_and_wait(e, r);
  if (st != BW_OK) return st;
  BW_API_END
}

// ---- stage level ----
int bw_mel(bw_engine* e, const float* pcm, int64_t n, int32_t padding, float* out_mel, int32_t* out_frames) {
  BW_API_BEGIN
  BW_CHECK(e && pcm && out_mel && out_frames, "null argument");
  BW_CHECK(e->filters_set, "mel filters not set");
  BW_CHECK(n + padding > 400, "audio (+padding) must be longer than 400 samples");
  DeviceGuard dg(e->device);
  const int nm = e->dims.n_mels;
  const int total = (int)((n + padding) / 160);
  const int n_real = padding >= 200 ? (int)std::min<long long>(total, (n + 200 + 159) / 160) : total;
  const int ld = (std::max(n_real, 1) + 15) / 16 * 16;
  DevBuf pcm_d, logmel, gmax, outd;
  pcm_d.alloc((size_t)(n + 4) * 4);
  logmel.alloc((size_t)nm * ld * 4);
  gmax.alloc(4);
  outd.alloc((size_t)nm * std::max(total, 1) * 4);
  std::lock_guard<std::mutex> g(e->gpu_mu);
  BW_CUDA(cudaMemcpyAsync(pcm_d.p, pcm, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  mel_power(pcm_d.as<float>(), n, padding, e->mel_tables.as<float>(), e->mel_filters.as<float>(), e->mel_ranges.as<int2>(), nm,
            logmel.as<float>(), ld, n_real, total, gmax.as<int>(), e->stream);
  mel_normalize_f32(logmel.as<float>(), ld, n_real, gmax.as<int>(), nm, total, outd.as<float>(), e->stream);
  BW_CUDA(cudaMemcpyAsync(out_mel, outd.p, (size_t)nm * total * 4, cudaMemcpyDeviceToHost, e->stream));
  BW_CUDA(cudaStreamSynchronize(e->stream));
  *out_frames = total;
  BW_API_END
}

int bw_encode(bw_engine* e, const float* mel, int32_t batch, float* out) {
  BW_API_BEGIN
  BW_CHECK(e && mel && out, "null argument");
  BW_CHECK(e->state == 1, "engine not finalized");
  BW_CHECK(batch >= 1 && batch <= e->Be, "batch exceeds max_encoder_batch");
  DeviceGuard dg(e->device);
  const auto& d = e->dims;
  const size_t per = (size_t)d.n_mels * 3000;
  DevBuf tmp, outf;
  tmp.alloc(per * batch * 4);
  const size_t n_out = (size_t)batch * 1500 * d.n_audio_state;
  outf.alloc(n_out * 4);
  std::lock_guard<std::mutex> g(e->gpu_mu);
  BW_CUDA(cudaMemcpyAsync(tmp.p, mel, per * batch * 4, cudaMemcpyHostToDevice, e->stream));
  for (int b = 0; b < batch; ++b) engine_window_to_A1(e, tmp.as<float>() + per * b, 3000, 3000, nullptr, 0, 3000, b);
  engine_encoder_forward(e, batch);
  if (e->fp32) BW_CUDA(cudaMemcpyAsync(out, e->enc_out.p, n_out * 4, cudaMemcpyDeviceToHost, e->stream));
  else {
    f32_from_bf16(e->enc_out.as<bf16>(), outf.as<float>(), (long long)n_out, e->stream);
    BW_CUDA(cudaMemcpyAsync(out, outf.p, n_out * 4, cudaMemcpyDeviceToHost, e->stream));
  }
  BW_CUDA(cudaStreamSynchronize(e->stream));
  BW_API_END
}

int bw_decode_logits(bw_engine* e, const float* mel_window, const int32_t* tokens, int32_t n, float* out_logits) {
  BW_API_BEGIN
  BW_CHECK(e && mel_window && tokens && out_logits, "null argument");
  BW_CHECK(n >= 1 && n <= e->dims.n_text_ctx, "token count out of range");
  Request r;
  r.kind = REQ_LOGITS;
  r.host_mel = mel_window;
  r.initial.assign(tokens, tokens + n);
  r.G = 1;
  r.logits_out = out_logits;
  const int st = submit_and_wait(e, r);
  if (st != BW_OK) return st;
  BW_API_END
}

}  // extern "C"
