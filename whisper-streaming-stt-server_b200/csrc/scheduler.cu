// The continuous-batching scheduler thread of one engine: admission (log-mel window -> encoder batch -> cross-KV),
// one batched decoder step over every live hypothesis of every live request, completion + host-side finalisation.
// This is the cross-session batching the reference declares (config/server.yaml:48-49 decode_batch_window_ms /
// max_decode_batch_size) but never implements (SURVEY.md section 0.4).
#include "sched.cuh"

namespace bw {

namespace {

double secs(Clock::time_point a, Clock::time_point b) { return std::chrono::duration<double>(b - a).count(); }

void finish_request(Request* r, int status, const std::string& err) {
  std::lock_guard<std::mutex> g(r->mu);
  r->status = status;
  r->error = err;
  r->done = true;
  r->cv.notify_all();
}

// H2D of the control block + the whole decoder step (all layers, logits, filters/top-k, beam update), enqueued on the
// decoder stream.  No host synchronisation here.
void enqueue_step_eager(bw_engine* e) {
  DecWorkspace& W = e->dec;
  const Ctl& c = W.ctl;
  BW_CUDA(cudaMemcpyAsync(W.d_ctrl.p, c.base, c.total * 4, cudaMemcpyHostToDevice, W.stream));
  engine_decoder_layers(e);
  const float* logits = W.d_logits.as<float>();
  const int V = e->dims.n_vocab;
  static const bool use_pdl = getenv("B200W_NO_PDL") == nullptr;
  PdlScope pdl(use_pdl && !e->fp32);
  no_speech_prob(logits, V, V, W.dev(c.ns_lrow), W.dev(c.ns_req), c.NNS, e->tt.no_speech, e->rs.no_speech_prob, W.stream);
  detect_language(logits, V, W.dev(c.det_lrow), W.dev(c.det_req), c.ND, e->tt, e->rs, e->ss, e->d_det_probs.as<float>(),
                  e->d_det_tok.as<int>(), W.stream);
  sample_topk(logits, V, V, W.dev(c.srow_lrow), W.dev(c.srow_req), W.dev(c.srow_seq), c.SR, e->tt, e->rs, e->ss, e->anc_cur,
              W.d_cand_tok.as<int>(), W.d_cand_lp.as<float>(), W.stream);
  beam_update(W.dev(c.act_req), W.dev(c.act_first), W.dev(c.act_force), c.NA, e->tt, e->rs, e->ss, e->anc_cur, e->dims.n_text_ctx,
              W.d_cand_tok.as<int>(), W.d_cand_lp.as<float>(), W.stream);
}


}  // namespace

void enqueue_step(bw_engine* e) {
  DecWorkspace& W = e->dec;
  const Ctl& c = W.ctl;
  if (c.R == 0) return;
  e->stat_h2d += (long long)c.total * 4;
  static const bool use_graphs = getenv("B200W_NO_GRAPH") == nullptr;
  if (!use_graphs) return enqueue_step_eager(e);
  const StepGraphKey key{c.R, c.NG, c.LR, c.SR, c.NA, c.NNS, c.ND, c.max_grp, e->anc_cur, dec_self_chunk(c.max_ctx)};
  StepGraph& sg = W.graphs[key];
  sg.last_use = ++W.graph_clock;
  if (sg.exec) {
    BW_CUDA(cudaGraphLaunch(sg.exec, W.stream));
    return;
  }
  if (++sg.seen < 3) return enqueue_step_eager(e);  // early sightings also warm every lazy initialisation
  // third sighting of this shape: it is stable enough to pay for a capture (the launch sequence depends only on the key)
  cudaGraph_t graph = nullptr;
  BW_CUDA(cudaStreamBeginCapture(W.stream, cudaStreamCaptureModeThreadLocal));
  try {
    enqueue_step_eager(e);
  } catch (...) {
    cudaStreamEndCapture(W.stream, &graph);
    if (graph) cudaGraphDestroy(graph);
    throw;
  }
  BW_CUDA(cudaStreamEndCapture(W.stream, &graph));
  cudaGraphExec_t exec = nullptr;
  const cudaError_t st = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (st != cudaSuccess) throw CudaError(std::string("cudaGraphInstantiate -> ") + cudaGetErrorString(st));
  sg.exec = exec;
  sg.last_use = ++W.graph_clock;
  BW_CUDA(cudaGraphLaunch(exec, W.stream));
  if (W.graphs.size() > kMaxStepGraphs) {
    // bound the cache (shapes churn while requests come and go): drop the least recently used half, entries included.
    // `sg` is not touched after this point (erase invalidates references to the erased nodes only, but be explicit).
    std::vector<std::pair<unsigned long long, StepGraphKey>> order;
    order.reserve(W.graphs.size());
    for (auto& kv : W.graphs) order.emplace_back(kv.second.last_use, kv.first);
    std::sort(order.begin(), order.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
    BW_CUDA(cudaStreamSynchronize(W.stream));  // no captured graph of the evicted half may still be running
    for (size_t i = 0; i < order.size() / 2; ++i) {
      auto it = W.graphs.find(order[i].second);
      if (it->second.exec) cudaGraphExecDestroy(it->second.exec);
      W.graphs.erase(it);
    }
  }
}

void finish_step(bw_engine* e) {
  BW_CUDA(cudaMemcpyAsync(e->h_flags, e->st_step.p, e->step_out_bytes, cudaMemcpyDeviceToHost, e->dec.stream));
  BW_CUDA(cudaStreamSynchronize(e->dec.stream));
  e->anc_cur ^= 1;
}

// ---- self-KV page pool -------------------------------------------------------------------------------------------
// Host free list, scheduler thread only.  A request reserves its worst case at admission (every hypothesis holding every
// block up to n_initial + sample_len positions), so an allocation during decoding can never fail and nothing is ever
// preempted; pages are TAKEN only when a hypothesis slot first writes into a block and RETURNED as soon as no surviving
// hypothesis' ancestry references them (collect_pages), so the pool in use follows the tokens in use.
int kv_blocks_for(int n_tokens) { return (std::max(n_tokens, 1) + kPageTokens - 1) / kPageTokens; }

int kv_page_of(bw_engine* e, Request* r, int slot, int block) {
  int& pg = r->pages[(size_t)slot * e->n_blocks + block];
  if (pg < 0) {
    if (e->free_pages.empty()) throw std::runtime_error("self-KV page pool exhausted despite reservations (scheduler bug)");
    pg = e->free_pages.back();
    e->free_pages.pop_back();
    const long long used = ++e->stat_pages_in_use;
    if (used > e->stat_pages_peak) e->stat_pages_peak = used;
  }
  return pg;
}

void kv_release(bw_engine* e, Request* r) {
  for (int& pg : r->pages)
    if (pg >= 0) { e->free_pages.push_back(pg); pg = -1; --e->stat_pages_in_use; }
  e->pages_reserved -= r->pages_reserved;
  r->pages_reserved = 0;
}

namespace {

// admission: pages the request may need at worst; sets up its (empty) page table and ancestry masks
int kv_reserve(bw_engine* e, Request* r) {
  const int n_init = (int)r->initial.size();
  const int max_tokens = (r->kind == REQ_DECODE) ? std::min(e->dims.n_text_ctx, n_init + r->sample_len) : n_init;
  r->n_blocks_max = kv_blocks_for(max_tokens);
  return r->n_blocks_max * r->G;
}
void kv_begin(bw_engine* e, Request* r, int need) {
  r->pages.assign((size_t)r->G * e->n_blocks, -1);
  r->ref_mask.assign((size_t)r->G * e->n_blocks, 0);
  r->pages_reserved = need;
  e->pages_reserved += need;
}

// After a step: hypothesis j of request r descends from old hypothesis src[j] (beam_update's reorder).  Its ancestry
// references, per block, the beam slots of its parent; slot j itself holds the position it is about to write.  Pages of
// COMPLETE blocks that no surviving hypothesis references go back to the free list.
void collect_pages(bw_engine* e, Request* r, const unsigned char* src, int next_pos) {
  const int G = r->G, NB = e->n_blocks;
  if (G > 1) {
    unsigned char old[kMaxBeam * kMaxBlocks];
    memcpy(old, r->ref_mask.data(), (size_t)G * NB);
    for (int j = 0; j < G; ++j) memcpy(&r->ref_mask[(size_t)j * NB], &old[(size_t)std::min<int>(src[j], G - 1) * NB], NB);
    const int cur_block = std::min(next_pos / kPageTokens, NB);
    for (int b = 0; b < cur_block; ++b) {
      unsigned live = 0;
      for (int j = 0; j < G; ++j) live |= r->ref_mask[(size_t)j * NB + b];
      for (int j = 0; j < G; ++j) {
        int& pg = r->pages[(size_t)j * NB + b];
        if (pg >= 0 && !(live >> j & 1u)) { e->free_pages.push_back(pg); pg = -1; --e->stat_pages_in_use; }
      }
    }
  }
}

}  // namespace

// Host-only replay of the page bookkeeping of ONE request (no CUDA call): the same sequence decode_step() runs --
// prefill pages of slot 0, then per step one page lookup per hypothesis slot, the ancestry masks, the collector.
// alloc_masks[step * n_blocks + b] = bit j set if (slot j, block b) holds a page after that step's collection.
int page_collector_replay(int G, int n_init, int n_steps, const unsigned char* parents, unsigned char* alloc_masks, int* pages_in_use) {
  bw_engine e;  // default-constructed: no device memory, no streams
  e.n_blocks = kMaxBlocks;
  e.n_pages = kMaxBlocks * kMaxBeam;
  for (int pg = e.n_pages - 1; pg >= 0; --pg) e.free_pages.push_back(pg);
  Request r;
  r.kind = REQ_DECODE;
  r.G = G;
  r.initial.assign((size_t)n_init, 0);
  r.sample_len = n_steps;
  e.dims.n_text_ctx = kMaxBlocks * kPageTokens;
  if (G < 1 || G > kMaxBeam || n_init < 1 || n_init + n_steps > e.dims.n_text_ctx) return BW_ERR_INVALID;
  kv_begin(&e, &r, kv_reserve(&e, &r));
  const int NB = e.n_blocks;
  for (int t = 0; t < n_init; ++t) kv_page_of(&e, &r, 0, t / kPageTokens);
  for (int j = 0; j < G; ++j)
    for (int b = 0; b <= (n_init - 1) / kPageTokens; ++b) r.ref_mask[(size_t)j * NB + b] |= 1u;
  int cur_len = n_init;
  for (int step = 0; step < n_steps; ++step) {
    if (step > 0)  // cached step: slot j writes position cur_len - 1
      for (int j = 0; j < G; ++j) {
        kv_page_of(&e, &r, j, (cur_len - 1) / kPageTokens);
        r.ref_mask[(size_t)j * NB + (cur_len - 1) / kPageTokens] |= (unsigned char)(1u << j);
      }
    cur_len += 1;
    collect_pages(&e, &r, parents + (size_t)step * G, cur_len - 1);
    for (int b = 0; b < NB; ++b) {
      unsigned m = 0;
      for (int j = 0; j < G; ++j) if (r.pages[(size_t)j * NB + b] >= 0) m |= 1u << j;
      alloc_masks[(size_t)step * NB + b] = (unsigned char)m;
    }
    pages_in_use[step] = (int)e.stat_pages_in_use;
  }
  kv_release(&e, &r);
  return (e.stat_pages_in_use == 0 && (int)e.free_pages.size() == e.n_pages && e.pages_reserved == 0) ? BW_OK : BW_ERR_STATE;
}

namespace {

void release_slots(bw_engine* e, Request* r) {
  kv_release(e, r);
  if (r->q >= 0) e->free_q.push_back(r->q);
  if (r->first_seq >= 0)
    for (int j = 0; j < r->G; ++j) e->seq_used[r->first_seq + j] = 0;
  r->q = -1;
  r->first_seq = -1;
}

int find_seq_block(bw_engine* e, int G) {
  int run = 0;
  for (int s = 0; s < e->S; ++s) {
    run = e->seq_used[s] ? 0 : run + 1;
    if (run == G) return s - G + 1;
  }
  return -1;
}

}  // namespace

// host-side finalisation: BeamSearchDecoder.finalize / GreedyDecoder.finalize + MaximumLikelihoodRanker
void finalize_decode(bw_engine* e, Request* r, const unsigned char* blob) {
  const int n_ctx = e->dims.n_text_ctx;
  const float* fin_score = reinterpret_cast<const float*>(blob);
  const int* fin_pos = reinterpret_cast<const int*>(blob + kMaxFinished * 4);
  const int* fin_slot = fin_pos + kMaxFinished;
  const int* misc = fin_slot + kMaxFinished;  // n_finished
  const float* fmisc = reinterpret_cast<const float*>(misc + 1);  // no_speech_prob, sum_logprob[kMaxBeam]
  const int* tok = reinterpret_cast<const int*>(fmisc + 1 + kMaxBeam);
  const unsigned char* parent = reinterpret_cast<const unsigned char*>(tok + (size_t)n_ctx * kMaxBeam);
  const int sb = (int)r->initial.size();
  const int eot = e->tt.eot;
  auto backtrack = [&](int pos, int slot) {
    std::vector<int> seq;
    for (int t = pos; t >= sb; --t) {
      seq.push_back(tok[(size_t)t * kMaxBeam + slot]);
      slot = parent[(size_t)t * kMaxBeam + slot];
    }
    std::reverse(seq.begin(), seq.end());
    return seq;
  };
  std::vector<std::vector<int>> cand;
  std::vector<float> cand_lp;
  const int last_pos = std::min(r->cur_len - 1, n_ctx - 1);
  if (r->greedy) {
    // GreedyDecoder.finalize: every hypothesis of the group (1, or best_of samples) padded with one EOT
    for (int j = 0; j < r->G; ++j) {
      cand.push_back(backtrack(last_pos, j));
      cand.back().push_back(eot);
      cand_lp.push_back(fmisc[1 + j]);
    }
  } else {
    const int n_fin = misc[0];
    for (int i = 0; i < n_fin; ++i) {
      cand.push_back(backtrack(fin_pos[i], fin_slot[i]));
      cand.back().push_back(eot);
      cand_lp.push_back(fin_score[i]);
    }
    if ((int)cand.size() < r->G) {
      std::vector<int> order(r->G);
      for (int j = 0; j < r->G; ++j) order[j] = j;
      std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return fmisc[1 + a] > fmisc[1 + b]; });
      for (int j : order) {
        std::vector<int> seq = backtrack(last_pos, j);
        seq.push_back(eot);
        bool dup = false;
        for (size_t c = 0; c < cand.size(); ++c)
          if (cand[c] == seq) { cand_lp[c] = fmisc[1 + j]; dup = true; break; }
        if (!dup) { cand.push_back(std::move(seq)); cand_lp.push_back(fmisc[1 + j]); }
        if ((int)cand.size() >= r->G) break;
      }
    }
  }
  int best = 0;
  double best_score = -INFINITY;
  for (size_t c = 0; c < cand.size(); ++c) {
    auto& s = cand[c];
    size_t cut = 0;
    while (cut < s.size() && s[cut] != eot) ++cut;
    s.resize(cut);
    const double len = (double)s.size();
    const double penalty = (r->length_penalty < 0) ? len : pow((5.0 + len) / 6.0, (double)r->length_penalty);
    const double score = (double)cand_lp[c] / penalty;
    if (c == 0 || score > best_score) { best = (int)c; best_score = score; }
  }
  bw_result* o = r->out;
  const auto& sel = cand[best];
  o->n_tokens = (int)std::min(sel.size(), (size_t)BW_MAX_TOKENS);
  for (int i = 0; i < o->n_tokens; ++i) o->tokens[i] = sel[i];
  o->sum_logprob = cand_lp[best];
  o->avg_logprob = (float)((double)cand_lp[best] / (double)(sel.size() + 1));
  o->no_speech_prob = fmisc[0];
  o->n_steps = r->steps;
  if (r->detect) {  // the language slot behind the parents: token, then the probabilities
    const int* lang = reinterpret_cast<const int*>(parent + (size_t)n_ctx * kMaxBeam);
    bw_lang_result* l = r->lang_out;
    l->language_token = lang[0];
    l->n_languages = e->tt.num_languages;
    memcpy(l->probs, lang + 1, (size_t)e->tt.num_languages * 4);
  }
}

size_t fin_blob_bytes(bw_engine* e) {
  return (size_t)kMaxFinished * 12 + 4 + 4 + kMaxBeam * 4 + (size_t)e->dims.n_text_ctx * kMaxBeam * 4 +
         (size_t)e->dims.n_text_ctx * kMaxBeam + 4 + kMaxLanguages * 4 + 64;
}

namespace {

void fail_all(bw_engine* e, std::vector<Request*>& fresh, const std::string& msg, int code) {
  for (Request* r : fresh) { release_slots(e, r); finish_request(r, code, msg); }
  fresh.clear();
  for (Request* r : e->live) { release_slots(e, r); finish_request(r, code, msg); }
  e->live.clear();
}

void admit_batch(bw_engine* e, std::vector<Request*>& fresh) {
  const auto& d = e->dims;
  const int nb = (int)fresh.size();
  for (int i = 0; i < nb; ++i) {
    Request* r = fresh[i];
    r->batch_index = i;
    r->t_admit = Clock::now();
    if (r->kind == REQ_LOGITS) {
      const size_t n = (size_t)d.n_mels * 3000;
      float* tmp = e->staging.as<float>();
      BW_CUDA(cudaMemcpyAsync(tmp, r->host_mel, n * 4, cudaMemcpyHostToDevice, e->stream));
      engine_window_to_A1(e, tmp, 3000, 3000, nullptr, 0, 3000, i);
      BW_CUDA(cudaStreamSynchronize(e->stream));  // staging is reused by the next request
    } else {
      bw_call* c = r->call;
      BW_CUDA(cudaStreamWaitEvent(e->stream, c->mel_done, 0));
      const int seg = std::max(0, std::min(3000, c->content_frames - r->seek));
      engine_window_to_A1(e, c->buf.logmel, c->buf.ld, c->n_real, c->buf.gmax, r->seek, seg, i);
    }
  }
  engine_encoder_forward(e, nb);
  for (int i = 0; i < nb; ++i) engine_cross_kv(e, i, fresh[i]->q);
  for (int i = 0; i < nb; ++i) {
    Request* r = fresh[i];
    int* rec = e->h_init + i * kInitRecInts;
    const int n_init = (int)r->initial.size();
    rec[0] = r->q; rec[1] = r->G; rec[2] = r->greedy; rec[3] = n_init; rec[4] = n_init; rec[5] = r->first_seq;
    rec[6] = r->without_ts; rec[7] = r->suppress_blank; rec[8] = r->max_initial_ts;
    rec[9] = r->max_candidates;
    rec[10] = r->initial.back();
    memcpy(&rec[11], &r->temperature, 4);
    rec[12] = (int)(unsigned int)(r->seed & 0xffffffffull); rec[13] = (int)(unsigned int)(r->seed >> 32);
    rec[14] = rec[15] = 0;
    r->cur_len = n_init;
    r->steps = 0;
    r->prefilled = false;
  }
  int* init_dev = e->d_init.as<int>();
  BW_CUDA(cudaMemcpyAsync(init_dev, e->h_init, (size_t)nb * kInitRecInts * 4, cudaMemcpyHostToDevice, e->stream));
  engine_init_requests(e, init_dev, nb);
  // the pinned control block is rewritten by the next step: make sure the copy has been consumed
  BW_CUDA(cudaStreamSynchronize(e->stream));
  e->stat_windows += nb;
  e->stat_enc_batches += 1;
  e->stat_h2d += (long long)nb * kInitRecInts * 4;
  for (Request* r : fresh) { r->t_encoded = Clock::now(); e->live.push_back(r); }
  fresh.clear();
}

// teacher forcing (bw_call_decode_forced): the token step `r->steps` must feed next, or -1
int forced_token(const Request* r) {
  return (r->steps < (int)r->forced.size()) ? r->forced[r->steps] : -1;
}

void decode_step(bw_engine* e) {
  const auto& d = e->dims;
  struct Special { Request* r; int lrow0; int n; };
  std::vector<Special> lang_reqs, logit_reqs, forced_reqs;
  DecWorkspace& W = e->dec;
  Ctl& ctl = W.ctl;
  ctl.reset();
  for (Request* r : e->live) {
    int &R = ctl.R, &NG = ctl.NG, &LR = ctl.LR, &SR = ctl.SR, &NA = ctl.NA, &NNS = ctl.NNS, &max_grp = ctl.max_grp;
    if (!r->prefilled) {
      const int n_init = (int)r->initial.size();
      // Initial positions [t0, t1) are fed in this step.  A detect-mode decode takes two steps: first <|sot|> alone,
      // whose logits row detect_language reads, then [1, n_init) -- its language row (row_tok -1) embeds the
      // next_tok that detect_language wrote, and its sot K/V come from the page like any cached position.
      const bool detect_sot = r->detect && r->prefill_pos == 0;
      const int t0 = r->prefill_pos, t1 = detect_sot ? 1 : n_init;
      const int row0 = R;
      ctl.max_ctx = std::max(ctl.max_ctx, t1);
      for (int t = t0; t < t1; ++t) {
        ctl.row_seq[R] = r->first_seq; ctl.row_pos[R] = t; ctl.row_tok[R] = r->initial[t]; ctl.row_bpos[R] = t0;
        ctl.row_page[R] = kv_page_of(e, r, 0, t / kPageTokens);
        ++R;
      }
      // every hypothesis starts as a copy of slot 0's prefix
      for (int j = 0; j < r->G; ++j)
        for (int b = 0; b <= (t1 - 1) / kPageTokens; ++b) r->ref_mask[(size_t)j * e->n_blocks + b] |= 1u;
      for (int t = t0; t < t1; t += 8) {
        ctl.grp_first[NG] = row0 + t - t0; ctl.grp_n[NG] = std::min(8, t1 - t); ctl.grp_x[NG] = r->q;
        max_grp = std::max(max_grp, ctl.grp_n[NG]);
        ++NG;
      }
      if (detect_sot) {  // the sot row: no_speech_prob and the language, nothing sampled yet
        ctl.lrow_src[LR] = row0;
        ctl.ns_lrow[NNS] = LR; ctl.ns_req[NNS] = r->q; ++NNS;
        ctl.det_lrow[ctl.ND] = LR; ctl.det_req[ctl.ND] = r->q; ++ctl.ND;
        ++LR;
      } else if (r->kind == REQ_LANG) {
        ctl.lrow_src[LR] = row0;
        lang_reqs.push_back({r, LR, 1});
        ++LR;
      } else if (r->kind == REQ_LOGITS) {
        logit_reqs.push_back({r, LR, n_init});
        for (int t = 0; t < n_init; ++t) ctl.lrow_src[LR++] = row0 + t;
      } else {
        const int last_row = R - 1;
        if (!r->detect) {  // (a detect-mode decode took no_speech_prob from its sot step)
          int sot_lrow;
          if (r->sot_index != n_init - 1) {
            ctl.lrow_src[LR] = row0 + r->sot_index;
            sot_lrow = LR++;
          } else sot_lrow = LR;
          ctl.ns_lrow[NNS] = sot_lrow; ctl.ns_req[NNS] = r->q; ++NNS;
        }
        ctl.lrow_src[LR] = last_row;
        ctl.act_req[NA] = r->q; ctl.act_first[NA] = SR; ctl.act_force[NA] = forced_token(r); ++NA;
        ctl.srow_lrow[SR] = LR; ctl.srow_req[SR] = r->q; ctl.srow_seq[SR] = r->first_seq; ++SR;
        if (r->step_logits_out) forced_reqs.push_back({r, LR, 1});
        ++LR;
      }
    } else {
      ctl.grp_first[NG] = R; ctl.grp_n[NG] = r->G; ctl.grp_x[NG] = r->q;
      max_grp = std::max(max_grp, r->G);
      ctl.max_ctx = std::max(ctl.max_ctx, r->cur_len);
      ++NG;
      ctl.act_req[NA] = r->q; ctl.act_first[NA] = SR; ctl.act_force[NA] = forced_token(r); ++NA;
      if (r->step_logits_out) forced_reqs.push_back({r, LR, 1});
      for (int j = 0; j < r->G; ++j) {
        ctl.row_seq[R] = r->first_seq + j; ctl.row_pos[R] = r->cur_len - 1; ctl.row_tok[R] = -1; ctl.row_bpos[R] = r->cur_len - 1;
        ctl.row_page[R] = kv_page_of(e, r, j, (r->cur_len - 1) / kPageTokens);  // slot j writes position cur_len - 1
        r->ref_mask[(size_t)j * e->n_blocks + (r->cur_len - 1) / kPageTokens] |= (unsigned char)(1u << j);
        ctl.lrow_src[LR] = R;
        ctl.srow_lrow[SR] = LR; ctl.srow_req[SR] = r->q; ctl.srow_seq[SR] = r->first_seq + j;
        ++R; ++LR; ++SR;
      }
    }
  }
  enqueue_step(e);
  const int V = d.n_vocab;
  for (auto& s : lang_reqs) {
    language_probs(W.d_logits.as<float>() + (size_t)s.lrow0 * V, V, e->tt.first_language_token, e->tt.num_languages,
                   e->d_lang_probs.as<float>(), e->d_lang_arg.as<int>(), W.stream);
    BW_CUDA(cudaMemcpyAsync(s.r->lang_out->probs, e->d_lang_probs.p, (size_t)e->tt.num_languages * 4, cudaMemcpyDeviceToHost, W.stream));
    BW_CUDA(cudaMemcpyAsync(&s.r->lang_out->language_token, e->d_lang_arg.p, 4, cudaMemcpyDeviceToHost, W.stream));
    BW_CUDA(cudaStreamSynchronize(W.stream));
    s.r->lang_out->n_languages = e->tt.num_languages;
  }
  for (auto& s : logit_reqs)
    BW_CUDA(cudaMemcpyAsync(s.r->logits_out, W.d_logits.as<float>() + (size_t)s.lrow0 * V, (size_t)s.n * V * 4,
                            cudaMemcpyDeviceToHost, W.stream));
  for (auto& s : forced_reqs)  // teacher-forced test requests: the raw logits row this step sampled from
    BW_CUDA(cudaMemcpyAsync(s.r->step_logits_out + (size_t)s.r->steps * V, W.d_logits.as<float>() + (size_t)s.lrow0 * V,
                            (size_t)V * 4, cudaMemcpyDeviceToHost, W.stream));
  // completion flags + the beam reorder (parent slot of every surviving hypothesis, what the page collector needs)
  finish_step(e);
  e->stat_d2h += (long long)e->step_out_bytes;
  const unsigned char* h_src = reinterpret_cast<const unsigned char*>(e->h_flags) + (size_t)e->Q * 4;
  e->stat_steps += 1;
  e->stat_rows += ctl.R;

  // bookkeeping + completion
  std::vector<Request*> still, done;
  for (Request* r : e->live) {
    if (r->kind != REQ_DECODE) { done.push_back(r); continue; }
    if (r->detect && r->prefill_pos == 0) {  // its sot step: the language is chosen, nothing was sampled
      r->prefill_pos = 1;
      still.push_back(r);
      continue;
    }
    r->prefilled = true;
    r->cur_len += 1;
    r->steps += 1;
    collect_pages(e, r, h_src + (size_t)r->q * kMaxBeam, r->cur_len - 1);
    if (e->h_flags[r->q] || r->steps >= r->sample_len || r->cur_len > d.n_text_ctx) done.push_back(r);
    else still.push_back(r);
  }
  // Finished requests leave `live` before anything below can throw: their callers own the Request objects and
  // free them as soon as finish_request() returns, so the scheduler's error path must never see them again.
  e->live.swap(still);
  size_t n_finished = 0;
  if (!done.empty()) try {
    const size_t blob = fin_blob_bytes(e);
    size_t nd = 0;
    for (Request* r : done) {  // (q, first sequence, hypotheses) of every finished decode; h_init is idle during a step
      if (r->kind != REQ_DECODE) continue;
      int* rec = e->h_init + nd * 3;
      rec[0] = r->q; rec[1] = r->first_seq; rec[2] = r->G;
      ++nd;
    }
    if (nd > 0) {
      BW_CUDA(cudaMemcpyAsync(e->d_init.p, e->h_init, nd * 12, cudaMemcpyHostToDevice, e->stream));
      engine_gather_final(e, e->d_init.as<int>(), (int)nd, (int)blob, e->d_fin.as<unsigned char>());
      BW_CUDA(cudaMemcpyAsync(e->h_fin, e->d_fin.p, nd * blob, cudaMemcpyDeviceToHost, e->stream));
      e->stat_d2h += (long long)(nd * blob);
    }
    BW_CUDA(cudaStreamSynchronize(e->stream));
    nd = 0;
    const auto now = Clock::now();
    for (Request* r : done) {
      if (r->kind == REQ_DECODE) {
        finalize_decode(e, r, e->h_fin + nd * blob);
        r->out->t_queue = (float)secs(r->t_submit, r->t_admit);
        r->out->t_encode = (float)secs(r->t_admit, r->t_encoded);
        r->out->t_decode = (float)secs(r->t_encoded, now);
        ++nd;
      }
      {
        std::lock_guard<std::mutex> g(e->q_mu);
        release_slots(e, r);
      }
      ++n_finished;
      finish_request(r, BW_OK, "");
    }
  } catch (const std::exception& ex) {
    for (size_t i = n_finished; i < done.size(); ++i) {
      {
        std::lock_guard<std::mutex> g(e->q_mu);
        release_slots(e, done[i]);
      }
      finish_request(done[i], BW_ERR_CUDA, ex.what());
    }
    throw;
  }
}

}  // namespace

void scheduler_main(bw_engine* e) {
  cudaSetDevice(e->device);
  const char* wenv = getenv("B200W_BATCH_WINDOW_US");
  const int window_us = wenv ? atoi(wenv) : 300;
  for (;;) {
    std::vector<Request*> fresh;
    {
      std::unique_lock<std::mutex> lk(e->q_mu);
      e->q_cv.wait(lk, [&] { return e->stop || !e->pending.empty() || !e->live.empty(); });
      if (e->stop) {
        std::vector<Request*> all(e->pending.begin(), e->pending.end());
        e->pending.clear();
        lk.unlock();
        fail_all(e, all, "engine destroyed", BW_ERR_STATE);
        return;
      }
      if (e->live.empty() && !e->pending.empty() && (int)e->pending.size() < e->Be && window_us > 0) {
        // short batching window so that simultaneous callers share one encoder launch
        e->q_cv.wait_for(lk, std::chrono::microseconds(window_us), [&] { return e->stop || (int)e->pending.size() >= e->Be; });
      }
      int rows = 0, lrows = 0;
      // rows / logits rows of the live requests in the next step (a detect-mode decode past its sot step still prefills)
      for (Request* r : e->live) {
        rows += r->prefilled ? r->G : (int)r->initial.size() - r->prefill_pos;
        lrows += r->prefilled ? r->G : 2;
      }
      while (!e->pending.empty() && (int)fresh.size() < e->Be) {
        Request* r = e->pending.front();
        const int n_init = (int)r->initial.size();
        const int need_l = (r->kind == REQ_LOGITS) ? n_init : 2;
        if (e->free_q.empty() || rows + n_init > e->R_max || lrows + need_l > e->LR_max) break;
        const int need_pages = kv_reserve(e, r);
        if (need_pages > e->n_pages) {  // can never be admitted: fail it instead of blocking the queue behind it
          e->pending.pop_front();
          finish_request(r, BW_ERR_NOMEM, "window needs more self-KV pages than the pool holds (raise max_kv_pages)");
          continue;
        }
        if (e->pages_reserved + need_pages > e->n_pages) break;
        const int fs = find_seq_block(e, r->G);
        if (fs < 0) break;
        kv_begin(e, r, need_pages);
        r->q = e->free_q.back();
        e->free_q.pop_back();
        r->first_seq = fs;
        for (int j = 0; j < r->G; ++j) e->seq_used[fs + j] = 1;
        rows += n_init;
        lrows += need_l;
        fresh.push_back(r);
        e->pending.pop_front();
      }
    }
    try {
      std::lock_guard<std::mutex> g(e->gpu_mu);
      if (!fresh.empty()) admit_batch(e, fresh);
      if (!e->live.empty()) decode_step(e);
    } catch (const std::exception& ex) {
      std::lock_guard<std::mutex> g(e->q_mu);
      fail_all(e, fresh, ex.what(), BW_ERR_CUDA);
    }
  }
}

int submit_many_and_wait(bw_engine* e, const std::vector<Request*>& rs) {
  if (e->state != 1 || !e->sched.joinable()) { last_error() = "engine not finalized or scheduler disabled"; return BW_ERR_STATE; }
  const auto now = Clock::now();
  {
    std::lock_guard<std::mutex> g(e->q_mu);
    if (e->stop) { last_error() = "engine stopping"; return BW_ERR_STATE; }
    for (Request* r : rs) { r->t_submit = now; e->pending.push_back(r); }
  }
  e->q_cv.notify_all();
  for (Request* r : rs) {
    std::unique_lock<std::mutex> lk(r->mu);
    r->cv.wait(lk, [&] { return r->done; });
  }
  return BW_OK;
}

void fill_decode_request(Request& r, bw_call* c, int seek, const bw_decode_opts* o, bw_result* out, bw_lang_result* lang) {
  BW_CHECK(c && o && out, "null argument");
  bw_engine* e = c->eng;
  BW_CHECK(o->n_initial >= 1 && o->initial_tokens, "initial tokens required");
  BW_CHECK(o->n_initial < e->dims.n_text_ctx, "too many initial tokens");
  BW_CHECK(o->n_initial <= 448, "too many initial tokens");
  BW_CHECK(o->sot_index >= 0 && o->sot_index < o->n_initial, "sot_index out of range");
  BW_CHECK(o->beam_size >= 0 && o->beam_size <= kMaxBeam, "beam_size must be in [0, 8]");
  BW_CHECK(seek >= 0, "negative seek");
  if (lang) {
    // upstream: is_multilingual = n_vocab >= 51865; an English-only model's sot sequence has no language token to detect
    BW_CHECK(e->tt.num_languages > 0 && e->dims.n_vocab >= 51865,
             "language detection: the model has no language tokens (English-only vocabulary)");
    // upstream detect_language conditions on [sot] at position 0 alone: only then is the decode's sot row that row
    BW_CHECK(o->sot_index == 0, "language detection: <|sot|> must be initial_tokens[0] (no prompt in front of it)");
    BW_CHECK(o->n_initial >= 2 && o->initial_tokens[1] == kLanguagePlaceholder,
             "language detection: initial_tokens[1] must be the language placeholder -1");
  }
  for (int i = 0; i < o->n_initial; ++i) {
    if (lang && i == 1) continue;
    BW_CHECK(!(lang && o->initial_tokens[i] == kLanguagePlaceholder),
             "language detection: the placeholder -1 may only appear at initial_tokens[sot_index + 1]");
    BW_CHECK(o->initial_tokens[i] >= 0 && o->initial_tokens[i] < e->dims.n_vocab, "token id out of range");
  }
  if (lang) {
    memset(lang, 0, sizeof(*lang));
    r.detect = true;
    r.lang_out = lang;
  }
  r.kind = REQ_DECODE;
  r.call = c;
  r.seek = seek;
  r.initial.assign(o->initial_tokens, o->initial_tokens + o->n_initial);
  r.sot_index = o->sot_index;
  r.greedy = o->beam_size == 0;
  r.beam = o->beam_size;
  r.G = r.greedy ? 1 : o->beam_size;
  if (o->temperature > 0.f) {
    // upstream DecodingTask: GreedyDecoder(temperature) with n_group = best_of or 1; beam search is a T = 0 decoder
    BW_CHECK(r.greedy, "temperature > 0 needs beam_size == 0 (decode_with_fallback drops beam_size / patience above T = 0)");
    BW_CHECK(o->best_of >= 0 && o->best_of <= kMaxBeam, "best_of must be in [0, 8]");
    BW_CHECK(std::isfinite(o->temperature), "temperature must be finite");
    r.temperature = o->temperature;
    r.G = std::max(1, (int)o->best_of);
    r.seed = ((unsigned long long)o->seed_hi << 32) | (unsigned long long)o->seed_lo;
  }
  r.patience = o->patience > 0 ? o->patience : 1.f;
  r.length_penalty = o->length_penalty;
  r.sample_len = o->sample_len > 0 ? o->sample_len : e->dims.n_text_ctx / 2;
  r.without_ts = o->without_timestamps != 0;
  r.suppress_blank = o->suppress_blank != 0;
  r.max_initial_ts = o->max_initial_timestamp_index;
  // BeamSearchDecoder.max_candidates = round(beam_size * patience) with Python's round-half-to-even; the host passes its
  // own result when it can (engine.py), else nearbyint under the default FE_TONEAREST mode gives the same rule.
  r.max_candidates = o->max_candidates > 0 ? o->max_candidates : std::max(1, (int)nearbyint((double)r.G * (double)r.patience));
  BW_CHECK(r.max_candidates <= kMaxFinished, "beam_size * patience too large");
  memset(out, 0, sizeof(*out));
  r.out = out;
}

int submit_and_wait(bw_engine* e, Request& r) {
  if (e->state != 1 || !e->sched.joinable()) { last_error() = "engine not finalized or scheduler disabled"; return BW_ERR_STATE; }
  r.t_submit = Clock::now();
  {
    std::lock_guard<std::mutex> g(e->q_mu);
    if (e->stop) { last_error() = "engine stopping"; return BW_ERR_STATE; }
    e->pending.push_back(&r);
  }
  e->q_cv.notify_all();
  std::unique_lock<std::mutex> lk(r.mu);
  r.cv.wait(lk, [&] { return r.done; });
  if (r.status != BW_OK) last_error() = r.error;
  return r.status;
}

}  // namespace bw
