// Engine: weight packing, device pools, encoder forward, batched decoder step, continuous-batching
// scheduler.  One engine per (GPU, model, compute mode); many host threads block in bw_call_decode and
// the scheduler thread coalesces them -- the cross-session batching the reference declares
// (config/server.yaml:48-49 decode_batch_window_ms / max_decode_batch_size) but never implements
// (SURVEY.md section 0.4) has to live here.
#include "sched.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

namespace bw {

namespace {

__global__ void init_requests_kernel(const int* __restrict__ init, int n, ReqState rs, SeqState ss, int n_ctx) {
  // init record: q, G, greedy, sample_begin, cur_len, first_seq, without_ts, suppress_blank, max_initial_ts,
  //              max_candidates, last_init_tok, temperature (float bits), seed_lo, seed_hi, pad, pad
  const int* r = init + blockIdx.x * kInitRecInts;
  const int q = r[0], G = r[1], first_seq = r[5];
  if (threadIdx.x == 0) {
    rs.n_beam[q] = G; rs.greedy[q] = r[2]; rs.sample_begin[q] = r[3]; rs.cur_len[q] = r[4]; rs.first_seq[q] = first_seq;
    rs.without_ts[q] = r[6]; rs.suppress_blank[q] = r[7]; rs.max_initial_ts[q] = r[8]; rs.max_candidates[q] = r[9];
    rs.n_finished[q] = 0; rs.completed[q] = 0; rs.no_speech_prob[q] = nanf("");
    for (int j = 0; j < kMaxBeam; ++j) rs.last_src[q * kMaxBeam + j] = (unsigned char)j;
    rs.temperature[q] = __int_as_float(r[11]); rs.seed_lo[q] = (unsigned int)r[12]; rs.seed_hi[q] = (unsigned int)r[13];
    for (int j = 0; j < G; ++j) {
      const int s = first_seq + j;
      ss.sum_logprob[s] = 0.f; ss.next_tok[s] = r[10]; ss.prev_tok[s] = -1; ss.last_ts[s] = -1;
      ss.seq_first[s] = first_seq | (G == 1 ? 0x40000000 : 0);  // kSingleBeamFlag: ancestry is identically 0
    }
  }
  // Both ancestry buffers: the one current at the request's first sampling step is anc_cur for a decode prefilled in its
  // admission step, the other one for a detect-mode decode (its sot step flips anc_cur before any beam update), and the
  // sequence slots still hold the previous occupant's ancestry.
  unsigned char* a0 = ss.anc[0] + (long long)first_seq * n_ctx;
  unsigned char* a1 = ss.anc[1] + (long long)first_seq * n_ctx;
  for (int i = threadIdx.x; i < G * n_ctx; i += blockDim.x) { a0[i] = 0; a1[i] = 0; }
}

// Finished requests -> one contiguous blob each (layout: finalize_decode in scheduler.cu), so that the host needs ONE
// device-to-host copy per step instead of eight per finished request.
__global__ void gather_final_kernel(const int* __restrict__ list, ReqState rs, SeqState ss, int n_ctx, int blob_bytes,
                                    const int* __restrict__ det_tok, const float* __restrict__ det_probs,
                                    unsigned char* __restrict__ out) {
  const int q = list[blockIdx.x * 3], first_seq = list[blockIdx.x * 3 + 1], G = list[blockIdx.x * 3 + 2];
  unsigned char* b = out + (size_t)blockIdx.x * blob_bytes;
  float* f = reinterpret_cast<float*>(b);
  int* i32 = reinterpret_cast<int*>(b);
  for (int i = threadIdx.x; i < kMaxFinished; i += blockDim.x) {
    f[i] = rs.fin_score[q * kMaxFinished + i];
    i32[kMaxFinished + i] = rs.fin_pos[q * kMaxFinished + i];
    i32[2 * kMaxFinished + i] = rs.fin_slot[q * kMaxFinished + i];
  }
  if (threadIdx.x == 0) {
    i32[3 * kMaxFinished] = rs.n_finished[q];
    f[3 * kMaxFinished + 1] = rs.no_speech_prob[q];
  }
  for (int i = threadIdx.x; i < kMaxBeam; i += blockDim.x) f[3 * kMaxFinished + 2 + i] = i < G ? ss.sum_logprob[first_seq + i] : 0.f;
  int* tok = i32 + 3 * kMaxFinished + 2 + kMaxBeam;
  const int* tsrc = rs.tok + (size_t)q * n_ctx * kMaxBeam;
  for (int i = threadIdx.x; i < n_ctx * kMaxBeam; i += blockDim.x) tok[i] = tsrc[i];
  unsigned char* par = reinterpret_cast<unsigned char*>(tok + (size_t)n_ctx * kMaxBeam);
  const unsigned char* psrc = rs.parent + (size_t)q * n_ctx * kMaxBeam;
  for (int i = threadIdx.x; i < n_ctx * kMaxBeam; i += blockDim.x) par[i] = psrc[i];
  // the language slot (meaningful for detect-mode decodes only): token, then kMaxLanguages probabilities
  int* lang = reinterpret_cast<int*>(par + (size_t)n_ctx * kMaxBeam);
  if (threadIdx.x == 0) lang[0] = det_tok[q];
  for (int i = threadIdx.x; i < kMaxLanguages; i += blockDim.x) reinterpret_cast<float*>(lang)[1 + i] = det_probs[q * kMaxLanguages + i];
}

inline float bf16_bits_to_float(uint16_t b) {
  uint32_t u = (uint32_t)b << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
inline float half_bits_to_float(uint16_t h) {
  const uint32_t sign = (h >> 15) & 1, exp = (h >> 10) & 0x1f, man = h & 0x3ff;
  uint32_t u;
  if (exp == 0) {
    if (man == 0) u = sign << 31;
    else {
      int e = -1;
      uint32_t m = man;
      do { ++e; m <<= 1; } while (!(m & 0x400));
      u = (sign << 31) | ((uint32_t)(127 - 15 - e) << 23) | ((m & 0x3ff) << 13);
    }
  } else if (exp == 31) u = (sign << 31) | 0x7f800000u | (man << 13);
  else u = (sign << 31) | ((exp + 112) << 23) | (man << 13);
  float f;
  memcpy(&f, &u, 4);
  return f;
}

}  // namespace

// ================================================================================================
// Typed implementation (T = bf16 product mode, float validation mode)
// ================================================================================================
template <typename T>
struct Impl {
  bw_engine* e;
  cudaStream_t stream;
  explicit Impl(bw_engine* eng, cudaStream_t st = nullptr) : e(eng), stream(st ? st : eng->stream) {}
  const bw_model_dims& D() const { return e->dims; }

  void gemm(const GemmArgs& g) const {
    if constexpr (std::is_same<T, float>::value) gemm_simt<float>(g, stream);
    else {
      if (e->force_simt) gemm_simt<bf16>(g, stream);
      else gemm_tc_bf16(g, stream);
    }
  }

  // out[R, N] = act(X[R, K] . W[N, K]^T + bias) (+ residual[R, N]); decoder-side skinny GEMM.
  // tcgen05 path: the live sequences are the (zero-padded) 128-row M operand and the weight streams through
  // as the N operand; gemm_tc_bf16 splits K over a thread-block cluster so that hundreds of CTAs, not N/128,
  // pull the weight from HBM (DSMEM reduction, no atomics).  The vocabulary projection (406 N tiles) runs
  // swap-AB instead: weight rows fill the MMA's M, the few logit rows are a narrow N tile.
  void linear_rows(const T* X, int R, int x_rows_alloc, const void* W, int N, int K, const float* bias, const float* residual,
                   void* out, bool gelu, bool out_fp32) const {
    GemmArgs g;
    g.K = K; g.lda = K; g.ldb = K; g.ldc = N; g.ldres = N; g.bias = bias; g.residual = residual; g.C = out;
    g.gelu = gelu; g.out_fp32 = out_fp32;
    const bool tc = !std::is_same<T, float>::value && !e->force_simt;
    if (tc && N > 8192) {
      g.A = W; g.B = X; g.M = N; g.N = R; g.transposed = true; g.b_rows = x_rows_alloc;
    } else {
      g.A = X; g.B = W; g.M = R; g.N = N; g.a_rows = x_rows_alloc;
    }
    gemm(g);
  }

  // ---- encoder forward on windows [w0, w0 + nb) whose conv1 operand already sits in A1, on this Impl's stream ----
  // Every activation buffer is window-major, so a sub-batch is a row range of the same buffers.
  void encoder_forward(int nb, int w0 = 0) const {
    const auto& d = D();
    const int dm = d.n_audio_state, T_enc = d.n_audio_ctx, K1 = 3 * d.n_mels;
    const int M = nb * T_enc;
    cudaStream_t st = stream;
    const long long r0 = (long long)w0 * T_enc;  // first row of this sub-batch in the [windows * 1500, .] buffers
    T* A1 = e->A1.as<T>() + (long long)w0 * 3000 * K1;
    T* y1 = e->y1.as<T>() + (long long)w0 * 3000 * dm;
    T* A2 = e->A2.as<T>() + r0 * 3 * dm;
    float* x = e->enc_x.as<float>() + r0 * dm;
    T* xn = e->enc_xn.as<T>() + r0 * dm;
    T* qkv = e->enc_qkv.as<T>() + r0 * 3 * dm;
    T* att = e->enc_att.as<T>() + r0 * dm;
    T* hbuf = e->enc_h.as<T>() + r0 * 4 * dm;
    T* out = e->enc_out.as<T>() + r0 * dm;
    {  // conv1 + GELU
      GemmArgs g;
      g.A = A1; g.B = e->w.conv1_w; g.C = y1; g.bias = e->w.conv1_b;
      g.M = nb * 3000; g.N = dm; g.K = K1; g.lda = K1; g.ldb = K1; g.ldc = dm; g.gelu = true;
      gemm(g);
    }
    im2col_conv2<T>(y1, A2, nb, dm, st);
    {  // conv2 + GELU + positional embedding -> fp32 residual stream
      GemmArgs g;
      g.A = A2; g.B = e->w.conv2_w; g.C = x; g.bias = e->w.conv2_b; g.residual = e->w.enc_pos;
      g.M = T_enc; g.N = dm; g.K = 3 * dm; g.lda = 3 * dm; g.ldb = 3 * dm; g.ldc = dm; g.ldres = dm;
      g.Z = nb; g.a_zstride = (long long)T_enc * 3 * dm; g.b_zstride = 0; g.c_zstride = (long long)T_enc * dm;
      g.res_zstride = 0; g.bias_zstride = 0; g.gelu = true; g.out_fp32 = true;
      gemm(g);
    }
    for (int l = 0; l < d.n_audio_layer; ++l) {
      const LayerW& w = e->w.enc[l];
      layernorm<T>(x, w.ln1_g, w.ln1_b, xn, M, dm, st);
      {
        GemmArgs g;
        g.A = xn; g.B = w.wqkv; g.C = qkv; g.bias = w.bqkv;
        g.M = M; g.N = 3 * dm; g.K = dm; g.lda = dm; g.ldb = dm; g.ldc = 3 * dm;
        gemm(g);
      }
      if constexpr (std::is_same<T, float>::value) {
        attn_encoder_simt<float>(reinterpret_cast<const float*>(qkv), reinterpret_cast<float*>(att), nb, T_enc, d.n_audio_head, st);
      } else {
        if (e->force_simt || (e->cfg.flags & BW_FLAG_SIMT_ATTENTION)) attn_encoder_simt<bf16>(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(att), nb, T_enc, d.n_audio_head, st);
        else attn_encoder_tc(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(att), nb, T_enc, d.n_audio_head, st);
      }
      {
        GemmArgs g;
        g.A = att; g.B = w.wo; g.C = x; g.bias = w.bo; g.residual = x;
        g.M = M; g.N = dm; g.K = dm; g.lda = dm; g.ldb = dm; g.ldc = dm; g.ldres = dm; g.out_fp32 = true;
        gemm(g);
      }
      layernorm<T>(x, w.ln2_g, w.ln2_b, xn, M, dm, st);
      {
        GemmArgs g;
        g.A = xn; g.B = w.w1; g.C = hbuf; g.bias = w.b1;
        g.M = M; g.N = 4 * dm; g.K = dm; g.lda = dm; g.ldb = dm; g.ldc = 4 * dm; g.gelu = true;
        gemm(g);
      }
      {
        GemmArgs g;
        g.A = hbuf; g.B = w.w2; g.C = x; g.bias = w.b2; g.residual = x;
        g.M = M; g.N = dm; g.K = 4 * dm; g.lda = 4 * dm; g.ldb = 4 * dm; g.ldc = dm; g.ldres = dm; g.out_fp32 = true;
        gemm(g);
      }
    }
    layernorm<T>(x, e->w.ln_post_g, e->w.ln_post_b, out, M, dm, st);
  }

  // cross K/V of every decoder layer for batch element `bi` -> cross-cache slot q (one launch, z = layer); the 8-bit cache
  // takes the GEMM's bf16 output through the one-window staging buffer and quantizes it into the slot
  void cross_kv(int bi, int q) const {
    const auto& d = D();
    const int dm = d.n_text_state, T_enc = d.n_audio_ctx, L = d.n_text_layer;
    GemmArgs g;
    g.A = e->enc_out.as<T>() + (long long)bi * T_enc * dm; g.B = e->w.wkv_x; g.bias = e->w.bkv_x;
    g.C = e->cross_int8 ? e->cross_stage.as<T>() : e->cross_cache.as<T>() + (long long)q * L * T_enc * 2 * dm;
    g.M = T_enc; g.N = 2 * dm; g.K = dm; g.lda = dm; g.ldb = dm; g.ldc = 2 * dm;
    g.Z = L; g.a_zstride = 0; g.b_zstride = (long long)2 * dm * dm; g.c_zstride = (long long)T_enc * 2 * dm; g.bias_zstride = 2 * dm;
    gemm(g);
    if (e->cross_int8) {
      const CrossKV x = engine_cross_kv_desc(e);
      cross_kv_int8_write(e->cross_stage.as<bf16>(), nullptr, nullptr, 1, L, T_enc, dm,
                          e->cross_cache.as<unsigned char>() + (long long)q * x.slot_stride, stream);
    }
  }

  // ---- one decoder step over the rows of e->dec.ctl; control block already on the device ----
  SelfKV self_kv() const {
    const auto& d = D();
    SelfKV skv;
    skv.pool = e->self_pool.p;
    skv.page_stride = (long long)d.n_text_layer * 2 * kPageTokens * d.n_text_state;
    skv.n_ctx = d.n_text_ctx; skv.n_blocks = e->n_blocks; skv.n_units = e->S;
    skv.page_table = e->d_page_table.as<int>();
    skv.seq_first = e->ss.seq_first; skv.anc = e->ss.anc[e->anc_cur];
    skv.pospage = e->dec.d_pospage.as<int>();
    return skv;
  }
  void decoder_layers() const {
    static const bool use_pdl = getenv("B200W_NO_PDL") == nullptr;
    PdlScope pdl(use_pdl && !std::is_same<T, float>::value);
    const auto& d = D();
    const int dm = d.n_text_state, L = d.n_text_layer, H = d.n_text_head;
    cudaStream_t st = stream;
    const DecWorkspace& G = e->dec;
    const Ctl& c = G.ctl;
    DecRows rows;
    rows.n_rows = c.R; rows.row_seq = G.dev(c.row_seq); rows.row_pos = G.dev(c.row_pos); rows.row_tok = G.dev(c.row_tok);
    rows.row_bpos = G.dev(c.row_bpos); rows.row_page = G.dev(c.row_page); rows.max_ctx = c.max_ctx;
    float* x = G.d_x.as<float>();
    if constexpr (std::is_same<T, bf16>::value) {
      if (e->fuse_ln) return decoder_layers_fused(rows);
    }
    dec_embed<T>(rows, e->ss.next_tok, reinterpret_cast<const T*>(e->w.tok_emb), reinterpret_cast<const T*>(e->w.dec_pos), x, dm,
                 e->d_page_table.as<int>(), e->n_blocks, st);
    const SelfKV skv = self_kv();
    dec_self_pospage(rows, skv, H, st);
    const CrossKV xkv = engine_cross_kv_desc(e);
    const int Ra = e->R_max;
    for (int l = 0; l < L; ++l) {
      const LayerW& w = e->w.dec[l];
      layernorm<T>(x, w.ln1_g, w.ln1_b, G.d_xn.as<T>(), c.R, dm, st);
      linear_rows(G.d_xn.as<T>(), c.R, Ra, w.wqkv, 3 * dm, dm, w.bqkv, nullptr, G.d_qkv.p, false, true);
      dec_self_attention<T>(rows, G.d_qkv.as<float>(), skv, l, dm, H, G.d_att.as<T>(), st);
      linear_rows(G.d_att.as<T>(), c.R, Ra, w.wo, dm, dm, w.bo, x, x, false, true);
      layernorm<T>(x, w.lnx_g, w.lnx_b, G.d_xn.as<T>(), c.R, dm, st);
      linear_rows(G.d_xn.as<T>(), c.R, Ra, w.wq_x, dm, dm, w.bq_x, nullptr, G.d_q.p, false, true);
      dec_cross_attention<T>(G.dev(c.grp_first), G.dev(c.grp_n), G.dev(c.grp_x), c.NG, c.max_grp, c.R, G.d_q.as<float>(), xkv, l, dm, H,
                             G.d_att.as<T>(), G.d_ws.as<float>(), st);
      linear_rows(G.d_att.as<T>(), c.R, Ra, w.wo_x, dm, dm, w.bo_x, x, x, false, true);
      layernorm<T>(x, w.ln2_g, w.ln2_b, G.d_xn.as<T>(), c.R, dm, st);
      linear_rows(G.d_xn.as<T>(), c.R, Ra, w.w1, 4 * dm, dm, w.b1, nullptr, G.d_h.p, true, false);
      linear_rows(G.d_h.as<T>(), c.R, Ra, w.w2, dm, 4 * dm, w.b2, x, x, false, true);
    }
    // final LayerNorm only on the rows whose logits are needed, then the tied-embedding projection
    layernorm_gather<T>(x, G.dev(c.lrow_src), e->w.ln_g, e->w.ln_b, G.d_lnrows.as<T>(), c.LR, dm, st);
    linear_rows(G.d_lnrows.as<T>(), c.LR, e->LR_max, e->w.tok_emb, d.n_vocab, dm, nullptr, nullptr, G.d_logits.p, false, true);
  }

  // bf16 tensor-core mode: the three LayerNorms of a block live inside the row GEMMs.  Each GEMM that writes the
  // residual stream (attention out-projections, mlp.2; the embedding for layer 0) also leaves a bf16 copy of it and
  // per-row LayerNorm partials; each GEMM that used to read a LayerNorm output multiplies the raw bf16 rows with
  // W * gamma and normalises in its epilogue.  8 kernels per block instead of 11 (tools/trace_step.py: a LayerNorm
  // launch costs ~2.4 us of work + ~1.4 us of dependency release on the step's critical path).
  void rows_gemm(const void* A, int R, int a_rows, const void* W, int N, int K, const float* bias, const float* residual, void* out,
                 bool gelu, bool out_fp32, void* xb_out, float2* st_out, const float2* st_in, const float* c1) const {
    GemmArgs g;
    g.A = A; g.B = W; g.M = R; g.N = N; g.K = K; g.lda = K; g.ldb = K; g.ldc = N; g.ldres = N; g.a_rows = a_rows;
    g.bias = bias; g.residual = residual; g.C = out; g.gelu = gelu; g.out_fp32 = out_fp32;
    g.xb_out = xb_out; g.ln_stats_out = st_out; g.ln_stats_in = st_in; g.ln_c1 = c1;
    gemm_tc_rows(g, stream);
  }
  void decoder_layers_fused(const DecRows& rows) const {
    const auto& d = D();
    const int dm = d.n_text_state, L = d.n_text_layer, H = d.n_text_head;
    cudaStream_t st = stream;
    const DecWorkspace& G = e->dec;
    const Ctl& c = G.ctl;
    float* x = G.d_x.as<float>();
    bf16* xb = G.d_xb.as<bf16>();
    float2* lst = G.d_lnst.as<float2>();
    dec_embed_ln<bf16>(rows, e->ss.next_tok, reinterpret_cast<const bf16*>(e->w.tok_emb), reinterpret_cast<const bf16*>(e->w.dec_pos), x, dm,
                       xb, lst, e->d_page_table.as<int>(), e->n_blocks, st);
    const SelfKV skv = self_kv();
    dec_self_pospage(rows, skv, H, st);
    const CrossKV xkv = engine_cross_kv_desc(e);
    const int Ra = e->R_max;
    for (int l = 0; l < L; ++l) {
      const LayerW& w = e->w.dec[l];
      rows_gemm(xb, c.R, Ra, w.wqkv, 3 * dm, dm, w.c2_qkv, nullptr, G.d_qkv.p, false, true, nullptr, nullptr, lst, w.c1_qkv);
      dec_self_attention<bf16>(rows, G.d_qkv.as<float>(), skv, l, dm, H, G.d_att.as<bf16>(), st);
      rows_gemm(G.d_att.p, c.R, Ra, w.wo, dm, dm, w.bo, x, x, false, true, xb, lst, nullptr, nullptr);
      rows_gemm(xb, c.R, Ra, w.wq_x, dm, dm, w.c2_qx, nullptr, G.d_q.p, false, true, nullptr, nullptr, lst, w.c1_qx);
      dec_cross_attention<bf16>(G.dev(c.grp_first), G.dev(c.grp_n), G.dev(c.grp_x), c.NG, c.max_grp, c.R, G.d_q.as<float>(), xkv, l, dm, H,
                                G.d_att.as<bf16>(), G.d_ws.as<float>(), st);
      rows_gemm(G.d_att.p, c.R, Ra, w.wo_x, dm, dm, w.bo_x, x, x, false, true, xb, lst, nullptr, nullptr);
      rows_gemm(xb, c.R, Ra, w.w1, 4 * dm, dm, w.c2_w1, nullptr, G.d_h.p, true, false, nullptr, nullptr, lst, w.c1_w1);
      rows_gemm(G.d_h.p, c.R, Ra, w.w2, dm, 4 * dm, w.b2, x, x, false, true, xb, lst, nullptr, nullptr);
    }
    layernorm_gather<bf16>(x, G.dev(c.lrow_src), e->w.ln_g, e->w.ln_b, G.d_lnrows.as<bf16>(), c.LR, dm, st);
    linear_rows(G.d_lnrows.as<bf16>(), c.LR, e->LR_max, e->w.tok_emb, d.n_vocab, dm, nullptr, nullptr, G.d_logits.p, false, true);
  }

  void window_to_A1(const float* logmel, int ld, int n_real, const int* gmax, int seek, int seg, int bi) const {
    T* dst = e->A1.as<T>() + (long long)bi * 3000 * 3 * D().n_mels;
    mel_window<T>(logmel, ld, n_real, gmax, D().n_mels, seek, seg, dst, e->stream);
  }
};

// ================================================================================================
// engine-level helpers used by api.cu
// ================================================================================================
static void* alloc_weight(bw_engine* e, size_t bytes, bool zero) {
  auto b = std::make_unique<DevBuf>();
  b->alloc(bytes);
  if (zero) BW_CUDA(cudaMemset(b->p, 0, bytes));
  void* p = b->p;
  e->weight_bufs.push_back(std::move(b));
  return p;
}

void engine_build_weight_table(bw_engine* e) {
  const auto& d = e->dims;
  const size_t ts = e->fp32 ? 4 : 2;
  auto wt = [&](size_t elems) { return alloc_weight(e, elems * ts, false); };
  auto wf = [&](size_t elems) { return reinterpret_cast<float*>(alloc_weight(e, elems * 4, true)); };
  auto reg = [&](const std::string& name, void* p, size_t n, bool required = true) {
    e->named[name] = {p, n};
    if (required) e->expected_names.push_back(name);
  };
  auto off = [&](void* p, size_t elems) { return reinterpret_cast<void*>(reinterpret_cast<char*>(p) + elems * ts); };
  const size_t dm = d.n_audio_state;
  ModelW& w = e->w;
  w.conv1_w = wt(dm * 3 * d.n_mels); w.conv1_b = wf(dm);
  w.conv2_w = wt(dm * 3 * dm); w.conv2_b = wf(dm);
  w.enc_pos = wf((size_t)d.n_audio_ctx * dm);
  reg("encoder.conv1.weight", w.conv1_w, dm * 3 * d.n_mels); reg("encoder.conv1.bias", w.conv1_b, dm);
  reg("encoder.conv2.weight", w.conv2_w, dm * 3 * dm); reg("encoder.conv2.bias", w.conv2_b, dm);
  reg("encoder.positional_embedding", w.enc_pos, (size_t)d.n_audio_ctx * dm, false);
  auto block = [&](const std::string& p, LayerW& lw, size_t dd, bool cross) {
    lw.ln1_g = wf(dd); lw.ln1_b = wf(dd);
    lw.wqkv = wt(3 * dd * dd); lw.bqkv = wf(3 * dd);
    lw.wo = wt(dd * dd); lw.bo = wf(dd);
    reg(p + ".attn_ln.weight", lw.ln1_g, dd); reg(p + ".attn_ln.bias", lw.ln1_b, dd);
    reg(p + ".attn.query.weight", lw.wqkv, dd * dd); reg(p + ".attn.query.bias", lw.bqkv, dd);
    reg(p + ".attn.key.weight", off(lw.wqkv, dd * dd), dd * dd);
    reg(p + ".attn.value.weight", off(lw.wqkv, 2 * dd * dd), dd * dd); reg(p + ".attn.value.bias", lw.bqkv + 2 * dd, dd);
    reg(p + ".attn.out.weight", lw.wo, dd * dd); reg(p + ".attn.out.bias", lw.bo, dd);
    if (cross) {
      lw.lnx_g = wf(dd); lw.lnx_b = wf(dd);
      lw.wq_x = wt(dd * dd); lw.bq_x = wf(dd);
      lw.wo_x = wt(dd * dd); lw.bo_x = wf(dd);
      reg(p + ".cross_attn_ln.weight", lw.lnx_g, dd); reg(p + ".cross_attn_ln.bias", lw.lnx_b, dd);
      reg(p + ".cross_attn.query.weight", lw.wq_x, dd * dd); reg(p + ".cross_attn.query.bias", lw.bq_x, dd);
      reg(p + ".cross_attn.out.weight", lw.wo_x, dd * dd); reg(p + ".cross_attn.out.bias", lw.bo_x, dd);
    }
    lw.ln2_g = wf(dd); lw.ln2_b = wf(dd);
    lw.w1 = wt(4 * dd * dd); lw.b1 = wf(4 * dd);
    lw.w2 = wt(4 * dd * dd); lw.b2 = wf(dd);
    reg(p + ".mlp_ln.weight", lw.ln2_g, dd); reg(p + ".mlp_ln.bias", lw.ln2_b, dd);
    reg(p + ".mlp.0.weight", lw.w1, 4 * dd * dd); reg(p + ".mlp.0.bias", lw.b1, 4 * dd);
    reg(p + ".mlp.2.weight", lw.w2, 4 * dd * dd); reg(p + ".mlp.2.bias", lw.b2, dd);
  };
  w.enc.resize(d.n_audio_layer);
  for (int i = 0; i < d.n_audio_layer; ++i) block("encoder.blocks." + std::to_string(i), w.enc[i], dm, false);
  w.ln_post_g = wf(dm); w.ln_post_b = wf(dm);
  reg("encoder.ln_post.weight", w.ln_post_g, dm); reg("encoder.ln_post.bias", w.ln_post_b, dm);
  const size_t dt = d.n_text_state;
  w.tok_emb = wt((size_t)d.n_vocab * dt);
  w.dec_pos = wt((size_t)d.n_text_ctx * dt);
  reg("decoder.token_embedding.weight", w.tok_emb, (size_t)d.n_vocab * dt);
  reg("decoder.positional_embedding", w.dec_pos, (size_t)d.n_text_ctx * dt);
  w.wkv_x = wt((size_t)d.n_text_layer * 2 * dt * dt);
  w.bkv_x = wf((size_t)d.n_text_layer * 2 * dt);
  w.dec.resize(d.n_text_layer);
  auto master = [&](size_t elems) {
    auto b = std::make_unique<DevBuf>();
    b->alloc(elems * 4);
    BW_CUDA(cudaMemset(b->p, 0, elems * 4));
    float* p = b->as<float>();
    e->fold_masters.push_back(std::move(b));
    return p;
  };
  for (int i = 0; i < d.n_text_layer; ++i) {
    const std::string p = "decoder.blocks." + std::to_string(i);
    block(p, w.dec[i], dt, true);
    if (e->fuse_ln) {
      LayerW& lw = w.dec[i];
      lw.c1_qkv = wf(3 * dt); lw.c2_qkv = wf(3 * dt); lw.c1_qx = wf(dt); lw.c2_qx = wf(dt); lw.c1_w1 = wf(4 * dt); lw.c2_w1 = wf(4 * dt);
      lw.m_wqkv = master(3 * dt * dt); lw.m_wqx = master(dt * dt); lw.m_w1 = master(4 * dt * dt);
      e->named_master[p + ".attn.query.weight"] = lw.m_wqkv;
      e->named_master[p + ".attn.key.weight"] = lw.m_wqkv + dt * dt;
      e->named_master[p + ".attn.value.weight"] = lw.m_wqkv + 2 * dt * dt;
      e->named_master[p + ".cross_attn.query.weight"] = lw.m_wqx;
      e->named_master[p + ".mlp.0.weight"] = lw.m_w1;
    }
    reg(p + ".cross_attn.key.weight", off(w.wkv_x, (size_t)i * 2 * dt * dt), dt * dt);
    reg(p + ".cross_attn.value.weight", off(w.wkv_x, (size_t)i * 2 * dt * dt + dt * dt), dt * dt);
    reg(p + ".cross_attn.value.bias", w.bkv_x + (size_t)i * 2 * dt + dt, dt);
  }
  w.ln_g = wf(dt); w.ln_b = wf(dt);
  reg("decoder.ln.weight", w.ln_g, dt); reg("decoder.ln.bias", w.ln_b, dt);
}

static bool is_f32_dest(const std::string& name) {
  auto ends = [&](const char* s) { const size_t n = strlen(s); return name.size() >= n && name.compare(name.size() - n, n, s) == 0; };
  if (name == "encoder.positional_embedding") return true;
  if (ends(".bias")) return true;
  if (ends("_ln.weight") || ends("ln_post.weight") || name == "decoder.ln.weight") return true;
  return false;
}

void engine_load_tensor(bw_engine* e, const bw_tensor_desc& t) {
  BW_CHECK(t.name && t.data, "tensor name/data null");
  const std::string name(t.name);
  auto it = e->named.find(name);
  if (it == e->named.end()) {
    if (name == "alignment_heads" || name.find("mask") != std::string::npos) return;  // non-parameter buffers of upstream
    throw std::invalid_argument("unknown tensor name: " + name);
  }
  size_t n = 1;
  for (int i = 0; i < t.ndim; ++i) n *= (size_t)t.shape[i];
  BW_CHECK(n == it->second.second, ("element count mismatch for " + name).c_str());
  // stage as fp32 on the device
  if (e->staging.bytes < n * 4) e->staging.alloc(std::max(n * 4, (size_t)64 << 20));
  std::vector<float> tmp;
  const float* src = nullptr;
  if (t.dtype == BW_F32) src = reinterpret_cast<const float*>(t.data);
  else {
    tmp.resize(n);
    const uint16_t* h = reinterpret_cast<const uint16_t*>(t.data);
    if (t.dtype == BW_F16) for (size_t i = 0; i < n; ++i) tmp[i] = half_bits_to_float(h[i]);
    else if (t.dtype == BW_BF16) for (size_t i = 0; i < n; ++i) tmp[i] = bf16_bits_to_float(h[i]);
    else throw std::invalid_argument("unsupported dtype for " + name);
    src = tmp.data();
  }
  BW_CUDA(cudaMemcpyAsync(e->staging.p, src, n * 4, cudaMemcpyHostToDevice, e->stream));
  void* dst = it->second.first;
  const bool conv = (name == "encoder.conv1.weight" || name == "encoder.conv2.weight");
  if (conv) {
    BW_CHECK(t.ndim == 3 && t.shape[2] == 3, "conv weight must be [co, ci, 3]");
    if (e->fp32) permute_conv_weight<float>(e->staging.as<float>(), reinterpret_cast<float*>(dst), (int)t.shape[0], (int)t.shape[1], e->stream);
    else permute_conv_weight<bf16>(e->staging.as<float>(), reinterpret_cast<bf16*>(dst), (int)t.shape[0], (int)t.shape[1], e->stream);
  } else if (is_f32_dest(name) || e->fp32) {
    BW_CUDA(cudaMemcpyAsync(dst, e->staging.p, n * 4, cudaMemcpyDeviceToDevice, e->stream));
  } else {
    convert_f32<bf16>(e->staging.as<float>(), reinterpret_cast<bf16*>(dst), (long long)n, e->stream);
    auto mi = e->named_master.find(name);  // LayerNorm fusion: keep the fp32 values until bw_engine_finalize folds them
    if (mi != e->named_master.end()) BW_CUDA(cudaMemcpyAsync(mi->second, e->staging.p, n * 4, cudaMemcpyDeviceToDevice, e->stream));
  }
  BW_CUDA(cudaStreamSynchronize(e->stream));  // `tmp` / caller memory may go away
  for (size_t i = 0; i < e->expected_names.size(); ++i)
    if (e->expected_names[i] == name) e->loaded[i] = 1;
  if (name == "encoder.positional_embedding") e->loaded.back() = 1;
}

// bw_engine_finalize: fold attn_ln / cross_attn_ln / mlp_ln of every decoder block into the Linear behind it
void engine_fold_layernorms(bw_engine* e) {
  if (!e->fuse_ln) return;
  const int dt = e->dims.n_text_state;
  for (LayerW& lw : e->w.dec) {
    fold_layernorm(lw.m_wqkv, lw.ln1_g, lw.ln1_b, lw.bqkv, 3 * dt, dt, reinterpret_cast<bf16*>(lw.wqkv), lw.c1_qkv, lw.c2_qkv, e->stream);
    fold_layernorm(lw.m_wqx, lw.lnx_g, lw.lnx_b, lw.bq_x, dt, dt, reinterpret_cast<bf16*>(lw.wq_x), lw.c1_qx, lw.c2_qx, e->stream);
    fold_layernorm(lw.m_w1, lw.ln2_g, lw.ln2_b, lw.b1, 4 * dt, dt, reinterpret_cast<bf16*>(lw.w1), lw.c1_w1, lw.c2_w1, e->stream);
    lw.m_wqkv = lw.m_wqx = lw.m_w1 = nullptr;
  }
  BW_CUDA(cudaStreamSynchronize(e->stream));
  e->fold_masters.clear();
  e->named_master.clear();
}

// Large batches run as two sub-batches on two streams: the persistent GEMM / attention kernels end in a partly
// filled last wave (e.g. 1410 tile pairs over 74 SM pairs) and every kernel boundary drains the machine; a second,
// independent kernel chain fills those gaps (profiles/r1_notes.md: ~10 % of the encoder at batch 16).
template <typename T> static void encoder_forward_t(bw_engine* e, int nb) {
  static const bool no_split = getenv("B200W_ENC_NO_SPLIT") != nullptr;
  static const int chunk_env = getenv("B200W_ENC_CHUNK") ? atoi(getenv("B200W_ENC_CHUNK")) : 8;
  if (no_split || nb < 4 || !e->enc_streams[0]) return Impl<T>(e).encoder_forward(nb);
  // sub-batches of <= `chunk` windows, dealt alternately to the engine stream and one extra stream
  const int chunk = std::max(2, std::min(chunk_env, (nb + 1) / 2));
  BW_CUDA(cudaEventRecord(e->enc_fork, e->stream));           // conv1 operands of all windows are in A1
  cudaStream_t s2 = e->enc_streams[0];
  BW_CUDA(cudaStreamWaitEvent(s2, e->enc_fork, 0));
  int k = 0;
  for (int w0 = 0; w0 < nb; w0 += chunk, ++k) {
    const int n = std::min(chunk, nb - w0);
    if ((k & 1) == 0) Impl<T>(e).encoder_forward(n, w0);
    else Impl<T>(e, s2).encoder_forward(n, w0);
  }
  BW_CUDA(cudaEventRecord(e->enc_join[0], s2));
  BW_CUDA(cudaStreamWaitEvent(e->stream, e->enc_join[0], 0));
}
void engine_encoder_forward(bw_engine* e, int nb) {
  if (e->fp32) encoder_forward_t<float>(e, nb); else encoder_forward_t<bf16>(e, nb);
}
CrossKV engine_cross_kv_desc(const bw_engine* e) {
  const auto& d = e->dims;
  CrossKV x;
  x.cache = e->cross_cache.p; x.T_enc = d.n_audio_ctx; x.n_slots = e->Q; x.n_layer = d.n_text_layer; x.int8 = e->cross_int8;
  x.slot_stride = x.int8 ? cross_int8_slot_bytes(d.n_text_layer, d.n_audio_ctx, d.n_text_head)
                         : (long long)d.n_text_layer * d.n_audio_ctx * 2 * d.n_text_state;
  return x;
}

void engine_cross_kv(bw_engine* e, int bi, int q) {
  if (e->fp32) Impl<float>(e).cross_kv(bi, q); else Impl<bf16>(e).cross_kv(bi, q);
}
void engine_window_to_A1(bw_engine* e, const float* logmel, int ld, int n_real, const int* gmax, int seek, int seg, int bi) {
  if (e->fp32) Impl<float>(e).window_to_A1(logmel, ld, n_real, gmax, seek, seg, bi);
  else Impl<bf16>(e).window_to_A1(logmel, ld, n_real, gmax, seek, seg, bi);
}
void engine_decoder_layers(bw_engine* e) {
  if (e->fp32) Impl<float>(e, e->dec.stream).decoder_layers(); else Impl<bf16>(e, e->dec.stream).decoder_layers();
}
void engine_gather_final(bw_engine* e, const int* list_dev, int n, int blob_bytes, unsigned char* out_dev) {
  if (n <= 0) return;
  gather_final_kernel<<<n, 256, 0, e->stream>>>(list_dev, e->rs, e->ss, e->dims.n_text_ctx, blob_bytes, e->d_det_tok.as<int>(),
                                                e->d_det_probs.as<float>(), out_dev);
  BW_CUDA(cudaGetLastError());
  ++g_kernel_launches;
}
void engine_init_requests(bw_engine* e, const int* init_dev, int n) {
  if (n <= 0) return;
  init_requests_kernel<<<n, 128, 0, e->stream>>>(init_dev, n, e->rs, e->ss, e->dims.n_text_ctx);
  BW_CUDA(cudaGetLastError());
  ++g_kernel_launches;
}

}  // namespace bw
