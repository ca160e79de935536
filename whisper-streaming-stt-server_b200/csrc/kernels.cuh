// Launchers for the non-GEMM kernels of the Whisper hot path.  T is the activation/weight storage
// type: bf16 (product mode) or float (fp32 validation mode).  The residual stream is always fp32.
#pragma once
#include <atomic>

#include "common.cuh"
#include "gemm.cuh"

namespace bw {

// ---- mel.cu ----
size_t mel_tables_floats();
void mel_fill_tables(float* host);
void mel_power(const float* pcm_dev, long long n, long long padding, const float* tables, const float* filters,
               const int2* ranges, int n_mels, float* logmel, int ld, int n_real, int total_frames, int* gmax_bits,
               cudaStream_t stream);
void mel_normalize_f32(const float* logmel, int ld, int n_real, const int* gmax_bits, int n_mels, int total_frames,
                       float* out, cudaStream_t stream);
template <typename T>
void mel_window(const float* logmel, int ld, int n_real, const int* gmax_bits, int n_mels, int seek, int segment_size,
                T* A1, cudaStream_t stream);

// ---- ingest.cu ----
// out[i] = pcm[i] / 32768  (stt_server/utils/audio.py:6-8)
void pcm16_to_f32(const int16_t* pcm, long long n, float* out, cudaStream_t stream);
// Polyphase Hann-windowed-sinc resampling of int16 PCM to float32 (utils/audio.py:11-30 -> torchaudio resample):
// out[f * nw + i] = sum_k taps[i][k] * pcm[f * orig - width + k] / 32768, n_out = ceil(nw * n / orig).
// ranges[i] = [lo, hi) taps of phase i that are not negligible (< 1e-20 in magnitude: the clamped window tails).
void pcm16_resample(const int16_t* pcm, long long n, const float* taps, const int2* ranges, int orig, int nw, int K, int width,
                    float* out, long long n_out, cudaStream_t stream);

// ---- elementwise.cu ----
// out[r][:] = LayerNorm(x[r][:]) * gamma + beta   (fp32 statistics, eps 1e-5)
template <typename T>
void layernorm(const float* x, const float* gamma, const float* beta, T* out, int rows, int d, cudaStream_t stream);
void layernorm_f32out(const float* x, const float* gamma, const float* beta, float* out, int rows, int d, cudaStream_t stream);
// gathered variant for the decoder's final LN: out[i] = LN(x[rows_idx[i]])
template <typename T>
void layernorm_gather(const float* x, const int* rows_idx, const float* gamma, const float* beta, T* out, int n, int d,
                      cudaStream_t stream);
// conv2 operand: A2[b*1500+t][k*d + c] = y1[b][2t+k-1][c] (zero outside [0,3000))
template <typename T>
void im2col_conv2(const T* y1, T* A2, int batch, int d, cudaStream_t stream);
// fp32 -> T conversion (weight packing), optional [co][ci][k] -> [co][k][ci] conv-weight permute
template <typename T>
void convert_f32(const float* src, T* dst, long long n, cudaStream_t stream);
template <typename T>
void permute_conv_weight(const float* src, T* dst, int co, int ci, cudaStream_t stream);
void f32_from_bf16(const bf16* src, float* dst, long long n, cudaStream_t stream);

// ---- attention.cu ----
// Encoder self-attention, non-causal, head dim 64: qkv [B*T, 3*d] (q | k | v), out [B*T, d].
template <typename T>
void attn_encoder_simt(const T* qkv, T* out, int batch, int T_len, int n_head, cudaStream_t stream);
void attn_encoder_tc(const bf16* qkv, bf16* out, int batch, int T_len, int n_head, cudaStream_t stream);

constexpr int kMaxBeam = 8;           // beams per request (n_group)
constexpr int kPageTokens = 16;       // positions per page of the self-attention KV pool
constexpr int kMaxBlocks = 28;        // pages per hypothesis at n_text_ctx = 448

// Decoder row descriptors (one row = one (sequence, position) token fed through the decoder step)
struct DecRows {
  int n_rows = 0;
  const int* row_seq = nullptr;   // [R] sequence slot (state arrays are indexed by it)
  const int* row_pos = nullptr;   // [R] position of the row's token in its sequence
  const int* row_tok = nullptr;   // [R] token id, or -1: take next_tok[row_seq]
  const int* row_bpos = nullptr;  // [R] position of the first row of this sequence fed in THIS step (<= row_pos)
  const int* row_page = nullptr;  // [R] page of the self-KV pool that receives this row's k / v (every layer)
  int max_ctx = 0;                // longest context (row_pos + 1) among the rows, 0 = unknown: sizes the self-attention staging
};
int dec_self_chunk(int max_ctx);  // positions the self-attention kernel stages per pass for that context (32 / 64 / 128)

// x[r] = E[tok] + pos_emb[pos]  (fp32 residual stream).  First kernel of a decoder step: it also publishes the step's
// page assignments, page_table[row_seq * n_blocks + row_pos / kPageTokens] = row_page (page_table may be null).
template <typename T>
void dec_embed(const DecRows& rows, const int* next_tok, const T* tok_emb, const T* pos_emb, float* x, int d, int* page_table,
               int n_blocks, cudaStream_t stream);

// ---- decoder LayerNorm fusion (bf16 tensor-core mode): see gemm.cuh / gemm_tc_rows ----
// embedding rows + their bf16 copy + per-64-column LayerNorm partials (the first layer's consumer GEMM reads them)
template <typename T>
void dec_embed_ln(const DecRows& rows, const int* next_tok, const T* tok_emb, const T* pos_emb, float* x, int d, bf16* xb,
                  float2* stats, int* page_table, int n_blocks, cudaStream_t stream);
void rows_ln_partials(const float* x, int rows, int d, bf16* xb, float2* stats, cudaStream_t stream);
// Wf = bf16(W * gamma), c1 = rowsum(Wf), c2 = W.beta + bias   (W fp32 [N, K])
void fold_layernorm(const float* W, const float* gamma, const float* beta, const float* bias, int N, int K, bf16* Wf, float* c1,
                    float* c2, cudaStream_t stream);

// Paged self-attention KV pool.  A page holds kPageTokens consecutive positions of ONE hypothesis slot for every layer:
// [L][2 (k | v)][kPageTokens][d].  page_table[u * n_blocks + t / kPageTokens] = page of slot u's block; pages are handed
// out by the scheduler (host free list; memory follows the tokens in use) and published by the step's embed kernel.
// Beams of one request occupy adjacent slots starting at seq_first[s]; the key / value of hypothesis s at position t
// lives in slot seq_first[s] + anc[s][t] (beam reordering never copies K/V, it rewrites the ancestry row; pages no
// surviving hypothesis references any more go back to the free list).
struct SelfKV {
  void* pool = nullptr;                // T*
  long long page_stride = 0;           // elements per page = L * 2 * kPageTokens * d
  int n_ctx = 448;
  int n_blocks = kMaxBlocks;           // ceil(n_ctx / kPageTokens)
  int n_units = 0;                     // hypothesis slots behind page_table
  const int* page_table = nullptr;     // [n_units][n_blocks]
  const int* seq_first = nullptr;      // [S] first sequence slot of the owning request
  const unsigned char* anc = nullptr;  // [S][n_ctx] beam slot holding position t (current ping-pong buffer)
  int* pospage = nullptr;              // [rows of the step][n_ctx] scratch: page of (row, position), see dec_self_pospage
};
// Once per step, after the embed kernel: resolves seq_first / ancestry / page table into pospage[r][t] for t < row_bpos[r],
// so that the 32 layers' self-attention kernels follow one indirection instead of three (no-op when the step's shape does not
// take the persistent-warp kernel, the only reader).
void dec_self_pospage(const DecRows& rows, const SelfKV& kv, int n_head, cudaStream_t stream);
// test / A-B hook: 0 = automatic, 1 = staged CTA per (row, head), 2 = warp per (row, head), 3 = persistent warps on mma.sync
// (bf16 only, needs pospage)
void dec_self_attention_mode(int mode);
// out[r] = softmax(q_r . K[0..pos_r]) V   (head dim 64); q = first d columns of the fp32 qkv rows.
// Also appends this step's k/v (columns d..3d of the row) to the row's page.
template <typename T>
void dec_self_attention(const DecRows& rows, const float* qkv, const SelfKV& kv, int layer, int d, int n_head, T* out,
                        cudaStream_t stream);
// Cross attention over the cached encoder K/V of each row's segment:
// cross cache slot layout [L][T_enc][2*d] (k | v). Group g = rows [first_row, first_row + n_rows) that share
// segment slot group_xslot[g] (the beams of one request); groups tile [0, n_rows) in order.
//
// 8-bit cross cache (BW_FLAG_CROSS_KV_INT8, bf16 mode only).  One scale per (layer, k | v, position, head):
// scale = amax / 127 over that 64-dim head slice, code = rint(x / scale) clamped to [-127, 127]; an all-zero slice has
// scale 0 and codes 0.  A slot is [L][n_head][ceil(T_enc / 64)] chunks of kCrossInt8ChunkBytes, one per (layer, head,
// 64-key tile), each fetched by one bulk copy into a stage of dec_cross_attention_int8_kernel (attention_xdec.cu):
//   [0, 4096)     K codes  [key][dim]
//   [4096, 8192)  V codes transposed for the P.V fragments: byte w*1024 + hf*512 + (g*4 + c)*16 + i*4 + j
//                 holds V[key w*16 + c*4 + j][dim (hf*4 + i)*8 + g]
//   [8192, 8448)  K scales fp32 [key];  [8448, 8704)  V scales fp32 [key]
// Keys past T_enc hold code 0, scale 0.  Only cross_kv_int8_write writes this layout and only the int8 attention
// kernel reads it.
constexpr int kCrossInt8ChunkBytes = 2 * 64 * 64 + 2 * 64 * 4;
inline long long cross_int8_slot_bytes(int n_layer, int T_enc, int n_head) {
  return (long long)n_layer * n_head * ((T_enc + 63) / 64) * kCrossInt8ChunkBytes;
}
struct CrossKV {
  const void* cache = nullptr;   // T*, or the 8-bit chunks above
  long long slot_stride = 0;     // elements per slot = L*T_enc*2*d; bytes per slot (cross_int8_slot_bytes) when int8
  int T_enc = 1500;
  int n_slots = 0;               // slots behind `cache` (TMA map extent)
  int n_layer = 0;
  bool int8 = false;             // cache format: T (false) or 8-bit codes + scales
};
template <typename T>
void dec_cross_attention(const int* group_first_row, const int* group_n_rows, const int* group_xslot, int n_groups,
                         int max_group_rows, int n_rows, const float* q, const CrossKV& kv, int layer, int d, int n_head, T* out,
                         float* workspace, cudaStream_t stream, int force_split = 0);
size_t dec_cross_workspace_floats(int n_rows, int n_head);
// Writes 8-bit slots in the layout above.  rows != nullptr: quantizes bf16 rows [n_slots][L][T_enc][2d] (k | v, the
// cross-KV GEMM's output); else packs codes int8 [n_slots][L][T_enc][2d] + scales fp32 [n_slots][L][T_enc][2 * n_head]
// (k heads, then v heads) that are already quantized.
void cross_kv_int8_write(const bf16* rows, const int8_t* codes, const float* scales, int n_slots, int n_layer, int T_enc, int d,
                         void* cache, cudaStream_t stream);
// The same quantization on plain rows: x bf16 [n_slices][64] -> codes [n_slices][64], scales [n_slices]
void quantize_int8_slices(const bf16* x, long long n_slices, int8_t* codes, float* scales, cudaStream_t stream);

// ---- sampling.cu ----
struct TokenTables {
  int eot, sot, sot_prev, sot_lm, no_speech, no_timestamps, timestamp_begin, translate, transcribe;
  int first_language_token, num_languages;
  int n_blank;
  int blank[4];                           // SuppressBlank ids: encode(" ") + eot
  const unsigned int* suppress_bits = nullptr;  // [ceil(V/32)] bit set = SuppressTokens id
};

constexpr int kMaxCand = kMaxBeam + 1;
constexpr int kMaxFinished = 16;
constexpr int kInitRecInts = 16;      // admission record (init_requests_kernel input), ints per request

// Per-request decoding state (device, struct of arrays indexed by request slot q)
struct ReqState {
  int* n_beam;          // G
  int* greedy;          // GreedyDecoder semantics (G = 1 at temperature 0, G = best_of samples above it)
  float* temperature;   // GreedyDecoder temperature; > 0 selects Categorical(logits / T) sampling
  unsigned int* seed_lo;  // counter-based RNG key of the request (sample_uniform in sampling.cu)
  unsigned int* seed_hi;
  int* sample_begin;    // index of the first sampled position
  int* cur_len;         // tokens so far (positions [0, cur_len))
  int* first_seq;       // sequence slot of beam 0 (beams are adjacent)
  int* without_ts;      // ApplyTimestampRules off
  int* suppress_blank;
  int* max_initial_ts;  // index or -1
  int* max_candidates;  // round(beam * patience)
  int* n_finished;      // finished pool fill
  float* fin_score;     // [Q][kMaxFinished]
  int* fin_pos;         // [Q][kMaxFinished] position of last token before EOT
  int* fin_slot;        // [Q][kMaxFinished] beam slot holding that token
  int* completed;       // out: all candidates collected
  unsigned char* last_src;  // out [Q][kMaxBeam]: beam slot each surviving hypothesis descended from in the last update
  float* no_speech_prob;
  int* tok;             // [Q][n_ctx][kMaxBeam] token written at (position, slot)
  unsigned char* parent;  // [Q][n_ctx][kMaxBeam] slot of the predecessor token
};
struct SeqState {
  float* sum_logprob;   // [S]
  int* next_tok;        // [S] most recent token of the hypothesis (fed at the next step)
  int* prev_tok;        // [S] the token before it
  int* last_ts;         // [S] most recent sampled timestamp token, or -1
  int* seq_first;       // [S] first sequence slot of the owning request
  unsigned char* anc[2];  // ping-pong [S][n_ctx]
};

// Fused logit filters + log-softmax statistics + top-(G+1) per logits row (warp-level reductions).
// Sample row i reads logits row srow_lrow[i]; cand_tok/cand_lp: [n_sample_rows][kMaxCand]
void sample_topk(const float* logits, int ld, int V, const int* srow_lrow, const int* lrow_req, const int* lrow_seq, int n_lrows,
                 const TokenTables& tt, const ReqState& rs, const SeqState& ss, int anc_cur, int* cand_tok, float* cand_lp,
                 cudaStream_t stream);
// Beam bookkeeping (BeamSearchDecoder.update / GreedyDecoder.update) for each active request.
// active_force[i] >= 0 (greedy requests only): the token to feed next instead of the sampled one (teacher forcing).
void beam_update(const int* active_req, const int* req_first_lrow, const int* active_force, int n_active, const TokenTables& tt,
                 const ReqState& rs, const SeqState& ss, int anc_cur, int n_ctx, const int* cand_tok, const float* cand_lp,
                 cudaStream_t stream);
// probs_at_sot.softmax()[no_speech] for requests in their first step
void no_speech_prob(const float* logits, int ld, int V, const int* lrows, const int* reqs, int n, int no_speech_id,
                    float* out_prob, cudaStream_t stream);
// detect_language: softmax over the language tokens of one logits row
void language_probs(const float* logits, int V, int first_lang, int n_lang, float* probs_out, int* argmax_out,
                    cudaStream_t stream);
// The same for the n detect-mode decodes of a step at once: request reqs[i] reads logits row lrows[i]; its language
// token goes to lang_tok[q] and next_tok[first_seq[q]], its probabilities to probs[q][0, num_languages)
constexpr int kMaxLanguages = 128;
void detect_language(const float* logits, int ld, const int* lrows, const int* reqs, int n, const TokenTables& tt, const ReqState& rs,
                     const SeqState& ss, float* probs, int* lang_tok, cudaStream_t stream);

}  // namespace bw
