/*
 * b200_whisper_hooks.h -- bench and test hooks of libb200whisper.so.
 *
 * NOT part of the drop-in boundary (include/b200_whisper.h): nothing the reference's backend interface needs is
 * declared here.  These entry points exist so that tests/ and bench.py can reach single kernels through the C ABI
 * (device pointers, e.g. from torch tensors) and time them with CUDA events on the launching stream.
 */
#ifndef B200_WHISPER_HOOKS_H
#define B200_WHISPER_HOOKS_H

#include "b200_whisper.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- kernel-level entry points (device pointers; used by tests/bench for roofline timing) ---- */
/* C[M,N] = act(A[M,K] . B[N,K]^T + bias) (+ residual); bf16 in, fp32 accumulate. impl 0 = tcgen05, 1 = SIMT,
 * 2 = tcgen05 swap-AB (the decoder's skinny-GEMM path) */
int bw_gemm_bf16(int impl, const void* A, const void* B, void* C, const float* bias, const float* residual,
                 int32_t M, int32_t N, int32_t K, int32_t gelu, int32_t out_fp32, void* stream);
/* A GEMM in the argument form the engine launches (bw::GemmArgs): for z < Z,
 *   D_z[i][j] = [gelu](sum_k A_z[i][k] * B_z[j][k] + bias_z[j]) (+ residual_z[i][j])      i < M, j < N
 * with X_z = X + z * x_zstride (elements; a zero stride with Z > 1 broadcasts one slice), leading dimensions lda / ldb
 * / ldc / ldres, and a_rows / b_rows (>= M / N; 0 = M / N) rows allocated behind A / B.  transposed stores D^T
 * (C[j * ldc + i], bias_z[i], residual_z[j * ldres + i]).  Device pointers; bias and residual are fp32 or NULL. */
typedef struct bw_gemm_desc {
  const void* A;
  const void* B;
  void* C;
  const float* bias;
  const float* residual;
  int32_t M, N, K;
  int32_t lda, ldb, ldc, ldres;
  int32_t Z;
  int32_t a_rows, b_rows;
  int64_t a_zstride, b_zstride, c_zstride, bias_zstride, res_zstride;
  int32_t gelu, out_fp32, transposed;
} bw_gemm_desc;
/* GEMM kernel routes: BW_GEMM_ROUTE(kernel, param) with the K split of the split-K / row kernels (row KS 1 = the
 * unsplit row kernel), the tile width of the plain tile kernel, 0 for the pair and SIMT kernels. */
#define BW_GEMM_PAIR 1   /* persistent CTA-pair kernel (cta_group::2, 256x256 tiles) */
#define BW_GEMM_SPLITK 2 /* cluster split-K kernel, DSMEM pull reduction; KS 2 / 4 / 8 */
#define BW_GEMM_ROWS 3   /* 128x64 row kernel, DSMEM push reduction; KS 1 / 2 / 4 / 8 */
#define BW_GEMM_TILE 4   /* plain 128xBN tile kernel; BN 32 / 64 / 128 */
#define BW_GEMM_SIMT 5   /* SIMT kernel (the fp32 validation mode, and bf16 with BW_FLAG_FORCE_SIMT_GEMM) */
#define BW_GEMM_ROUTE(kernel, param) ((kernel) * 1000 + (param))
/* Runs one GEMM.  dtype 0: bf16 A / B, C bf16 or fp32 (out_fp32); dtype 1: fp32 A / B / C on the SIMT kernel, as the
 * fp32 validation mode does.  route 0 = the dispatcher's choice, else BW_GEMM_ROUTE(...) forces that kernel and fails
 * (BW_ERR_INVALID) if its preconditions do not hold; *route_taken receives the route that ran.  Asynchronous on
 * `stream` like the engine's launches. */
int bw_test_gemm(const bw_gemm_desc* desc, int32_t dtype, int32_t route, int32_t* route_taken, void* stream);
/* Host only (no GPU needed): the route bw_test_gemm(desc, 0, 0, ...) takes, i.e. what the bf16 dispatcher picks for
 * this argument form.  Pointers are not dereferenced; only whether bias / residual are NULL matters. */
int bw_test_gemm_route(const bw_gemm_desc* desc, int32_t* route);
/* Encoder self-attention on qkv [batch*T, 3*64*n_head] bf16 -> out [batch*T, 64*n_head] bf16. impl 0 = tcgen05, 1 = SIMT */
int bw_attention_bf16(int impl, const void* qkv, void* out, int32_t batch, int32_t T_len, int32_t n_head, void* stream);
/* Times `iters` launches of the decoder cross-attention kernel on synthetic resident data and returns
 * avg ms per launch (CUDA events on the launch stream); bytes_out = algorithmic bytes per launch. */
int bw_bench_cross_attention(bw_engine*, int32_t n_segments, int32_t n_group, int32_t iters, float* ms_out, double* bytes_out);
int bw_bench_encoder(bw_engine*, int32_t batch, int32_t iters, float* ms_out, double* flops_out);
int bw_bench_mel(bw_engine*, int64_t n_samples, int32_t iters, float* ms_out, double* bytes_out);
int bw_bench_decoder_step(bw_engine*, int32_t n_segments, int32_t n_group, int32_t context_len, int32_t iters,
                          float* ms_out, double* bytes_out);

/* Whole hot path on device-resident PCM (mel -> encoder -> cross-KV -> n_steps batched decoder steps), one
 * CUDA-event pair on the engine stream; returns total ms. */
int bw_bench_pipeline(bw_engine*, const float* pcm_host, const int64_t* offsets, const int64_t* lengths,
                      int32_t n_segments, int32_t n_group, int32_t n_steps, float* ms_out);
/* What the last bw_bench_pipeline call (same n_segments, n_group, n_steps) decoded: one bw_result per window, finalised
 * as bw_call_decode finalises a beam-search request (length_penalty < 0: none, as in bw_decode_opts). Untimed. */
int bw_bench_pipeline_results(bw_engine*, int32_t n_segments, int32_t n_group, int32_t n_steps, float length_penalty,
                              bw_result* out);

/* Test hook for the decoder LayerNorm fusion (device pointers): producer row GEMM x = res + A.Wp^T + bp (also
 * emits bf16(x) and per-row LayerNorm partials) then consumer row GEMM out = [gelu](LayerNorm(x; gamma, beta).Wc^T + bc)
 * with gamma folded into Wc.  A == NULL skips the producer (x = res).  A bf16 [M, Kp], Wp bf16 [d, Kp], Wc fp32 [N, d];
 * x_out fp32 [M, d], out fp32 [M, N]; d % 64 == 0, N % 64 == 0. */
int bw_test_ln_chain(const void* A, const void* Wp, const float* bp, const float* res, const float* gamma, const float* beta,
                     const float* Wc, const float* bc, int32_t M, int32_t d, int32_t Kp, int32_t N, int32_t gelu, float* x_out,
                     float* out, void* stream);

/* Debug timeline of the decoder step: enable != 0 arms a device buffer that the step's kernels append
 * (tag, globaltimer ns) records to; enable == 0 disarms it and copies up to `cap` records (2 x uint64 each:
 * smid << 32 | kernel id << 24 | grid.x << 8 | phase, then the timestamp) to `out`, count in *n_out.
 * enable == 2 dumps the raw buffer instead (kernels that store into fixed slots).
 * Run with B200W_NO_GRAPH=1 (captured graphs keep the pointer they were captured with). */
int bw_debug_trace(bw_engine*, int32_t enable, uint64_t* out, int32_t cap, int32_t* n_out);

/* ---- parity hooks for the bf16 product decoder (tests/test_gpu_decoder_kernels.py, tests/test_gpu_bf16_decode.py) ---- */
/* Teacher-forced decode through the REAL scheduler path (admission, encoder batch, cross-KV, continuous batching, CUDA
 * graphs, cached self/cross attention): like bw_call_decode with GreedyDecoder semantics (opts->beam_size == 0,
 * temperature 0), but step k feeds forced[k] as the next token whatever the step sampled, and the raw logits row the
 * step sampled from -- TextDecoder.forward at position n_initial - 1 + k -- is copied to step_logits[k * V] (host).
 * Runs exactly n_forced steps unless forced[k] is EOT. */
int bw_call_decode_forced(bw_call*, int32_t seek, const bw_decode_opts* opts, const int32_t* forced, int32_t n_forced,
                          float* step_logits, bw_result* out);
/* dec_cross_attention<bf16> (TMA + mma.sync kernel + T-split combine) on device pointers: cache bf16
 * [n_slots][n_layer][T_enc][2d] (k | v), q fp32 [n_rows, d], groups as in the step's control block (device int32),
 * force_split 0 = the launcher's own choice, else that many T splits (<= 8).  out bf16 [n_rows, d]. */
int bw_test_dec_cross_attention(const void* cache, int32_t n_slots, int32_t n_layer, int32_t layer, int32_t T_enc, int32_t d,
                                int32_t n_head, const float* q, const int32_t* grp_first, const int32_t* grp_n,
                                const int32_t* grp_x, int32_t n_groups, int32_t max_group_rows, int32_t n_rows,
                                int32_t force_split, void* out, void* stream);
/* The 8-bit cross cache's quantization (BW_FLAG_CROSS_KV_INT8) on device pointers: x bf16 [n_rows][d] (d % 64 == 0) ->
 * codes int8 [n_rows][d], scales fp32 [n_rows][d / 64]; each 64-element slice gets scale = amax / 127 and
 * code = rint(x / scale) clamped to [-127, 127] (an all-zero slice: scale 0, codes 0). */
int bw_test_quantize_cross_kv(const void* x, int64_t n_rows, int32_t d, int8_t* codes, float* scales, void* stream);
/* dec_cross_attention<bf16> on the 8-bit cross cache, arguments as bw_test_dec_cross_attention: codes int8
 * [n_slots][n_layer][T_enc][2d] (k | v) and scales fp32 [n_slots][n_layer][T_enc][2 * n_head] (k heads, then v heads),
 * i.e. what bw_test_quantize_cross_kv makes of a bf16 cache; they are packed into the engine's slot layout first. */
int bw_test_dec_cross_attention_int8(const int8_t* codes, const float* scales, int32_t n_slots, int32_t n_layer, int32_t layer,
                                     int32_t T_enc, int32_t d, int32_t n_head, const float* q, const int32_t* grp_first,
                                     const int32_t* grp_n, const int32_t* grp_x, int32_t n_groups, int32_t max_group_rows,
                                     int32_t n_rows, int32_t force_split, void* out, void* stream);
/* dec_self_attention<bf16> (+ fused K/V append) on device pointers over a paged pool: pages of 16 positions,
 * [n_pages][n_layer][2][16][d] bf16; page_table int32 [n_units][ceil(n_ctx / 16)]; row_page[r] = page that receives row
 * r's k / v.  max_ctx = longest context (row_pos + 1) among the rows or 0: picks the staged kernel's staging size (32 / 64 /
 * 128 positions per pass).  Other arguments as bw::SelfKV / bw::DecRows.  Runs dec_self_pospage first, like the step. */
int bw_test_dec_self_attention(int32_t n_rows, const int32_t* row_seq, const int32_t* row_pos, const int32_t* row_bpos,
                               const int32_t* row_page, const float* qkv, void* pool, int32_t n_layer, int32_t n_ctx, int32_t n_units,
                               const int32_t* page_table, const int32_t* seq_first, const uint8_t* anc, int32_t layer, int32_t d,
                               int32_t n_head, int32_t max_ctx, void* out, void* stream);
/* Which decoder self-attention kernel the bf16 path launches (process-wide; A-B runs and kernel tests): 0 = automatic
 * (persistent warps from 512 (row, head) units upwards, else staged), 1 = staged CTA per (row, head), 2 = warp per
 * (row, head), 3 = persistent warps on mma.sync. */
int bw_test_self_attention_mode(int32_t mode);
/* sample_topk_kernel on n independent logits rows (host pointers).  state[i][10] = n_beam, greedy, cur_len,
 * sample_begin, without_ts, suppress_blank, max_initial_ts (-1 = none), last token, the token before it (-1 = none),
 * most recent sampled timestamp token (-1 = none).  Writes the top-(n_beam + 1) (1 if greedy) candidates of each row:
 * cand_tok / cand_lp [n][9], unused entries untouched. */
int bw_test_sample_topk(bw_engine*, const float* logits, int32_t n, const int32_t* state, int32_t* cand_tok, float* cand_lp);

/* Host-only (no GPU needed): replays the scheduler's self-KV page bookkeeping for ONE request of n_hypotheses beams --
 * n_initial prompt positions, then n_steps decoder steps whose beam reorder is parents[step * n_hypotheses + j] (the slot
 * hypothesis j descends from, what beam_update reports back).  alloc_masks[step * 28 + block]: bit j set if (slot j, block)
 * holds a page after that step's collection; pages_in_use[step].  Fails if a page leaks. */
int bw_test_page_collector(int32_t n_hypotheses, int32_t n_initial, int32_t n_steps, const uint8_t* parents, uint8_t* alloc_masks,
                           int32_t* pages_in_use);

#ifdef __cplusplus
}
#endif
#endif /* B200_WHISPER_HOOKS_H */
