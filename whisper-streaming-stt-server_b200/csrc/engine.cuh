// Engine internals: packed weights, device pools, request/scheduler state.
#pragma once
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/b200_whisper.h"
#include "kernels.cuh"

namespace bw {

using Clock = std::chrono::steady_clock;

// ---- device memory helpers ----
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  void alloc(size_t n) {
    release();
    if (n == 0) return;
    BW_CUDA(cudaMalloc(&p, n));
    bytes = n;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  template <typename U> U* as() const { return reinterpret_cast<U*>(p); }
  ~DevBuf() { release(); }
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
};

struct LayerW {
  // all matrices are [out, in] (K-major B operands); biases / LayerNorm affine are fp32
  float *ln1_g, *ln1_b;
  void* wqkv; float* bqkv;   // [3d, d], key bias = 0
  void* wo;   float* bo;     // [d, d]
  float *lnx_g, *lnx_b;      // decoder only: cross_attn_ln
  void* wq_x; float* bq_x;   // decoder only: cross query [d, d]
  void* wo_x; float* bo_x;   // decoder only: cross out [d, d]
  float *ln2_g, *ln2_b;      // mlp_ln
  void* w1;   float* b1;     // [4d, d]
  void* w2;   float* b2;     // [d, 4d]
  // decoder LayerNorm fusion (engine->fuse_ln): wqkv / wq_x / w1 then hold W * gamma of the LayerNorm in front of
  // them; c1 = row sums of the folded weight, c2 = W.beta + bias (what the row GEMM's consumer epilogue needs).
  float *c1_qkv = nullptr, *c2_qkv = nullptr, *c1_qx = nullptr, *c2_qx = nullptr, *c1_w1 = nullptr, *c2_w1 = nullptr;
  float *m_wqkv = nullptr, *m_wqx = nullptr, *m_w1 = nullptr;  // fp32 masters, only between load and finalize
};

struct ModelW {
  void* conv1_w; float* conv1_b;  // [d, 3*n_mels] (k-major taps)
  void* conv2_w; float* conv2_b;  // [d, 3*d]
  float* enc_pos;                 // [1500, d] fp32 (added in the conv2 epilogue)
  std::vector<LayerW> enc, dec;
  float *ln_post_g, *ln_post_b;
  void* tok_emb;                  // [V, d]
  void* dec_pos;                  // [n_text_ctx, d]
  void* wkv_x; float* bkv_x;      // [L, 2d, d], [L, 2d] : cross key|value of every decoder layer (key bias = 0)
  float *ln_g, *ln_b;
};

enum ReqKind { REQ_DECODE = 0, REQ_LANG = 1, REQ_LOGITS = 2 };

struct StepGraphKey {
  int R, NG, LR, SR, NA, NNS, ND, max_grp, anc, self_chunk;  // self_chunk: the self-attention launch geometry (dec_self_chunk)
  bool operator==(const StepGraphKey& o) const {
    return R == o.R && NG == o.NG && LR == o.LR && SR == o.SR && NA == o.NA && NNS == o.NNS && ND == o.ND && max_grp == o.max_grp &&
           anc == o.anc && self_chunk == o.self_chunk;
  }
};
struct StepGraphKeyHash {
  size_t operator()(const StepGraphKey& k) const {
    size_t h = 1469598103934665603ull;
    for (int v : {k.R, k.NG, k.LR, k.SR, k.NA, k.NNS, k.ND, k.max_grp, k.anc, k.self_chunk}) h = (h ^ (size_t)v) * 1099511628211ull;
    return h;
  }
};
struct StepGraph {
  int seen = 0;
  unsigned long long last_use = 0;
  cudaGraphExec_t exec = nullptr;
};
constexpr size_t kMaxStepGraphs = 128;  // per engine; least recently used half is dropped beyond this

// ---- decoder-step control block (ints), mirrored host (pinned) / device ----
struct Ctl {
  int *row_seq, *row_pos, *row_tok, *row_bpos, *row_page, *grp_first, *grp_n, *grp_x, *lrow_src, *srow_lrow, *srow_req, *srow_seq, *act_req,
      *act_first, *act_force, *ns_lrow, *ns_req;
  int *det_lrow, *det_req;  // detect-mode decodes whose <|sot|> row this step feeds (detect_language)
  int* base = nullptr;
  size_t total = 0;
  // fill counters of the step being built
  int R = 0, NG = 0, LR = 0, SR = 0, NA = 0, NNS = 0, ND = 0, max_grp = 1, max_ctx = 0;
  void layout(int* b, int Rm, int LRm, int Q) {
    base = b;
    int* p = b;
    auto take = [&](size_t n) { int* r = p; p += n; return r; };
    row_seq = take(Rm); row_pos = take(Rm); row_tok = take(Rm); row_bpos = take(Rm); row_page = take(Rm);
    grp_first = take(Rm); grp_n = take(Rm); grp_x = take(Rm);
    lrow_src = take(LRm); srow_lrow = take(LRm); srow_req = take(LRm); srow_seq = take(LRm);
    act_req = take(Q); act_first = take(Q); act_force = take(Q); ns_lrow = take(Q); ns_req = take(Q);
    det_lrow = take(Q); det_req = take(Q);
    total = (size_t)(p - b);
  }
  void reset() { R = NG = LR = SR = NA = NNS = ND = 0; max_grp = 1; max_ctx = 0; }
};

// Decoder-step working set: activations, logits, control block and step graphs, with the step's own stream.
struct DecWorkspace {
  cudaStream_t stream = nullptr;
  // CUDA graphs of the whole decoder step, keyed by its shape: while the set of live requests is unchanged only the
  // control block's CONTENTS change from step to step, so ~360 launches collapse into one cudaGraphLaunch.
  std::unordered_map<StepGraphKey, StepGraph, StepGraphKeyHash> graphs;
  unsigned long long graph_clock = 0;
  DevBuf d_x, d_xn, d_qkv, d_att, d_q, d_h, d_lnrows, d_logits, d_ws, d_cand_tok, d_cand_lp, d_ctrl;
  DevBuf d_xb, d_lnst;  // LayerNorm fusion: bf16 copy of the residual stream, per-row / per-64-column partials
  DevBuf d_pospage;     // [R_max][n_text_ctx] page of (row, position) for the step's self-attention (dec_self_pospage)
  int* h_ctrl = nullptr;  // pinned host copy of the control block
  Ctl ctl;                // laid out over h_ctrl
  int* dev(const int* h) const { return d_ctrl.as<int>() + (h - ctl.base); }  // device address of a control array
};

// polyphase filter bank of one source sample rate (bw_engine_set_resampler)
struct Resampler {
  int orig = 0, nw = 0, width = 0, K = 0;
  DevBuf taps, ranges;
};

struct CallBuf {
  float* pcm = nullptr;     // device
  float* logmel = nullptr;  // device [n_mels][ld]
  int* gmax = nullptr;      // device
  long long pcm_cap = 0;
  int ld = 0;
  bool pooled = false;
};

}  // namespace bw

struct bw_call {
  bw_engine* eng = nullptr;
  bw::CallBuf buf;
  long long n_samples = 0;
  int n_real = 0, total_frames = 0, content_frames = 0;
  cudaEvent_t mel_done = nullptr;
};

namespace bw {

struct Request {
  int kind = REQ_DECODE;
  bw_call* call = nullptr;
  const float* host_mel = nullptr;  // REQ_LOGITS: normalised mel window [n_mels, 3000]
  int seek = 0;
  std::vector<int> initial;
  int sot_index = 0, beam = 0, greedy = 1, sample_len = 224, without_ts = 0, suppress_blank = 1, max_initial_ts = 50;
  float patience = 1.f, length_penalty = -1.f;
  float temperature = 0.f;          // > 0: GreedyDecoder sampling with G = best_of hypotheses
  unsigned long long seed = 0;
  int max_candidates = 1;           // BeamSearchDecoder: round(beam_size * patience), computed by the caller's rounding rule
  // test hook (bw_call_decode_forced): teacher forcing -- step k feeds forced[k] whatever was sampled, and the
  // step's raw logits row goes to step_logits_out + k * V
  std::vector<int> forced;
  float* step_logits_out = nullptr;
  // outputs
  bw_result* out = nullptr;
  bw_lang_result* lang_out = nullptr;
  float* logits_out = nullptr;
  int status = 0;
  std::string error;
  std::mutex mu;
  std::condition_variable cv;
  bool done = false;
  // self-KV pages (scheduler thread only): page of (beam slot, block) or -1; per hypothesis and block, the set of beam
  // slots whose pages its ancestry references (bit j = slot j) -- what the page collector works from
  std::vector<int> pages;
  std::vector<unsigned char> ref_mask;
  int pages_reserved = 0, n_blocks_max = 0;
  // detect mode (bw_call_decode_detect): initial[1] is the language placeholder (-1); the decode is prefilled in two
  // steps, <|sot|> alone (its logits row picks the language on the device), then positions [1, n_initial) -- see
  // decode_step.  The language comes back through lang_out.
  bool detect = false;
  // runtime
  int q = -1, first_seq = -1, G = 1, cur_len = 0, steps = 0;
  int prefill_pos = 0;  // first initial position the next prefill step feeds (1 after a detect-mode decode's first step)
  bool prefilled = false;
  int batch_index = -1;  // position inside the current encoder batch
  Clock::time_point t_submit, t_admit, t_encoded;
};

}  // namespace bw

struct bw_engine {
  bw_model_dims dims{};
  bw_engine_config cfg{};
  int device = 0;
  bool fp32 = false;       // validation mode
  bool force_simt = false;
  bool fuse_ln = false;    // decoder LayerNorms folded into the row GEMMs (bf16 tensor-core mode)
  bool cross_int8 = false; // BW_FLAG_CROSS_KV_INT8: 8-bit cross cache (kernels.cuh CrossKV)
  std::vector<std::unique_ptr<bw::DevBuf>> fold_masters;                    // released by bw_engine_finalize
  std::unordered_map<std::string, float*> named_master;                     // tensor name -> fp32 master slice
  std::atomic<int> refs{1};
  int state = 0;           // 0 = created, 1 = finalized
  cudaStream_t stream = nullptr;
  static constexpr int kEncStreams = 3;                // extra streams for the sub-batches of a split encoder batch
  cudaStream_t enc_streams[kEncStreams]{};
  cudaEvent_t enc_fork = nullptr, enc_join[kEncStreams]{};
  static constexpr int kFrontStreams = 4;
  cudaStream_t front[kFrontStreams]{};
  std::mutex front_mu[kFrontStreams];
  bw::DevBuf front_pcm16[kFrontStreams];  // int16 staging of the raw-ingest path (serialised by front_mu / stream order)
  std::mutex resampler_mu;
  std::unordered_map<int, std::unique_ptr<bw::Resampler>> resamplers;  // by source sample rate
  std::atomic<unsigned> front_rr{0};
  std::mutex gpu_mu;       // serialises users of `stream` and the activation buffers

  // weights
  std::vector<std::unique_ptr<bw::DevBuf>> weight_bufs;
  std::unordered_map<std::string, std::pair<void*, size_t>> named;  // name -> (device ptr, element count) for loading
  bw::ModelW w{};
  std::vector<char> loaded;
  std::vector<std::string> expected_names;
  bw::TokenTables tt{};
  bool tables_set = false, filters_set = false;
  bw::DevBuf suppress_bits, mel_tables, mel_filters, mel_ranges, staging;

  // pools
  int Q = 0, S = 0, Be = 0, R_max = 0, LR_max = 0;
  bw::DevBuf cross_cache, self_pool;
  bw::DevBuf cross_stage;  // 8-bit mode: bf16 cross K/V of one window ([L][T_enc][2d]), quantized into its slot
  // paged self-KV: n_pages pages of kPageTokens positions ([L][2][kPageTokens][d] each), page table on the device,
  // free list + reservations on the host (scheduler thread)
  int n_pages = 0, n_blocks = 0;
  size_t page_bytes = 0;
  bw::DevBuf d_page_table;
  std::vector<int> free_pages;
  int pages_reserved = 0;
  std::atomic<long long> stat_pages_in_use{0}, stat_pages_peak{0};
  // encoder activations
  bw::DevBuf A1, y1, A2, enc_x, enc_xn, enc_qkv, enc_att, enc_h, enc_out;
  // decoder activations
  bw::DecWorkspace dec;
  bw::DevBuf d_lang_probs, d_lang_arg;
  bw::DevBuf d_det_probs, d_det_tok;  // detect-mode decodes: [Q][kMaxLanguages] probabilities, [Q] language token
  // decoder state
  bw::DevBuf st_int, st_float, st_anc0, st_anc1, st_tok, st_parent, st_step;  // st_step: [Q] completed | [Q][kMaxBeam] last_src
  bw::ReqState rs{};
  bw::SeqState ss{};
  int anc_cur = 0;
  // admission records (init_requests_kernel input)
  bw::DevBuf d_init;
  int* h_init = nullptr;      // pinned
  int* h_flags = nullptr;     // pinned copy of st_step: [Q] completed flags, then [Q][kMaxBeam] parent slots (bytes)
  size_t step_out_bytes = 0;
  unsigned char* h_fin = nullptr;  // pinned scratch for finalisation
  bw::DevBuf d_fin;                // device side of it (gather_final_kernel packs finished requests here)
  size_t h_fin_bytes = 0;

  // call buffers
  std::mutex call_mu;
  std::vector<bw::CallBuf> call_pool;
  long long call_pcm_cap = 0;
  int call_ld = 0;

  // scheduler
  std::thread sched;
  std::mutex q_mu;
  std::condition_variable q_cv;
  std::deque<bw::Request*> pending;
  std::vector<bw::Request*> live;
  std::vector<int> free_q;
  std::vector<char> seq_used;
  bool stop = false;

  // stats
  std::atomic<long long> stat_steps{0}, stat_rows{0}, stat_windows{0}, stat_enc_batches{0}, stat_h2d{0}, stat_d2h{0};
};
