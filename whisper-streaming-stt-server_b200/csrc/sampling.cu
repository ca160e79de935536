// K7: fused logit filters + log-softmax + top-k, and device-side beam-search bookkeeping.
//
// Upstream whisper/decoding.py (reached from reference torch_whisper.py:55; SURVEY.md Appendix A.4):
//   SuppressBlank, SuppressTokens, ApplyTimestampRules  -> allowed() predicate evaluated on the fly
//   F.log_softmax + topk(beam+1) / argmax               -> block-wide (max,sum) + per-thread top lists
//   BeamSearchDecoder.update / GreedyDecoder.update     -> beam_update_kernel (one warp per request)
// Logits are never modified in place; the host is not consulted between steps.
#include <limits.h>

#include "kernels.cuh"

namespace bw {
namespace {

constexpr int ST = 1024; // threads of the per-row kernels (one CTA per logits row: 32 warps per SM keep more loads in flight than 16)
constexpr int SU = 8;    // logits loaded per thread per batch (keeps 8 coalesced loads in flight)

struct RowRules {
  int tb, eot, no_ts_id;
  int mask_all_ts;      // logits[tb:] = -inf
  int mask_below_eot;   // logits[:eot] = -inf
  int ts_floor;         // timestamps < ts_floor masked (tb if none)
  int first_text_mask;  // logits[:tb] = -inf at the first sampled position
  int ts_ceiling;       // timestamps > ts_ceiling masked (INT_MAX if none)
  int n_blank;
  int blank[4];
  int use_ts_rules;
  const unsigned int* suppress_bits;
};

__device__ __forceinline__ bool allowed(const RowRules& r, int id) {
  if (r.suppress_bits[id >> 5] >> (id & 31) & 1u) return false;
  if (r.n_blank && (id == r.blank[0] || id == r.blank[1] || id == r.blank[2] || id == r.blank[3])) return false;
  if (!r.use_ts_rules) return true;
  if (id == r.no_ts_id) return false;
  if (id >= r.tb) {
    if (r.mask_all_ts) return false;
    if (id < r.ts_floor || id > r.ts_ceiling) return false;
  } else {
    if (r.first_text_mask) return false;
    if (r.mask_below_eot && id < r.eot) return false;
  }
  return true;
}

__device__ __forceinline__ void ms_merge(float& m, float& s, float m2, float s2) {
  const float mm = fmaxf(m, m2);
  if (mm == -INFINITY) { m = mm; s = 0.f; return; }
  s = s * expf(m - mm) + s2 * expf(m2 - mm);
  m = mm;
}

// block-wide (max, sum-exp) reduction; result valid in all threads
__device__ void block_ms(float& m, float& s, float* sh_m, float* sh_s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
    const float s2 = __shfl_xor_sync(0xffffffffu, s, o);
    ms_merge(m, s, m2, s2);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) { sh_m[warp] = m; sh_s[warp] = s; }
  __syncthreads();
  m = sh_m[0]; s = sh_s[0];
  for (int w = 1; w < ST / 32; ++w) ms_merge(m, s, sh_m[w], sh_s[w]);
}

__device__ __forceinline__ bool better(float v, int id, float v2, int id2) { return v > v2 || (v == v2 && id < id2); }

// Counter-based generator for temperature sampling: the uniform of (request seed, hypothesis, position, token id)
// is a pure function of its key (splitmix64 finaliser), so a decode is reproducible whatever batch it runs in and
// whatever the launch geometry.  23 mantissa bits, u in (0, 1) exactly representable; oracle/whisper_oracle.py
// `gumbel_noise` restates it bit for bit.
__device__ __forceinline__ float sample_uniform(unsigned long long seed, int stream, int pos, int id) {
  unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(stream + 1);
  z ^= ((unsigned long long)(unsigned int)pos << 32) | (unsigned long long)(unsigned int)id;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return ((float)(unsigned int)(z >> 41) + 0.5f) * (1.f / 8388608.f);
}

__global__ void __launch_bounds__(ST)
sample_topk_kernel(const float* __restrict__ logits, int ld, int V, const int* __restrict__ srow_lrow,
                   const int* __restrict__ lrow_req, const int* __restrict__ lrow_seq, const TokenTables tt, const ReqState rs, const SeqState ss,
                   int* __restrict__ cand_tok, float* __restrict__ cand_lp) {
  __shared__ float sh_m[ST / 32], sh_s[ST / 32];
  __shared__ float wv[ST / 32];
  __shared__ int wi[ST / 32];
  __shared__ int win_i;
  pdl_trigger();
  pdl_wait();
  const int lr = blockIdx.x;
  const int q = lrow_req[lr], s = lrow_seq[lr];
  const float* x = logits + (long long)srow_lrow[lr] * ld;
  const int tb = tt.timestamp_begin;

  RowRules r;
  r.tb = tb; r.eot = tt.eot; r.no_ts_id = tt.no_timestamps; r.suppress_bits = tt.suppress_bits;
  const int cur_len = rs.cur_len[q], sb = rs.sample_begin[q];
  const bool first = (cur_len == sb);
  const int n_sampled = cur_len - sb;
  r.use_ts_rules = !rs.without_ts[q];
  const int last = ss.next_tok[s], prev = ss.prev_tok[s], lts = ss.last_ts[s];
  const bool last_ts = n_sampled >= 1 && last >= tb;
  const bool pen_ts = n_sampled < 2 || prev >= tb;
  r.mask_all_ts = last_ts && pen_ts;
  r.mask_below_eot = last_ts && !pen_ts;
  r.ts_floor = tb;
  if (lts >= 0) r.ts_floor = (last_ts && !pen_ts) ? lts : lts + 1;
  r.first_text_mask = first;
  r.ts_ceiling = INT_MAX;
  if (first && rs.max_initial_ts[q] >= 0) r.ts_ceiling = tb + rs.max_initial_ts[q];
  r.n_blank = 0;
  if (first && rs.suppress_blank[q]) {
    r.n_blank = tt.n_blank;
    for (int i = 0; i < 4; ++i) r.blank[i] = tt.blank[i];
  }

  // pass A: (max, sumexp) of the allowed text ids and of the allowed timestamp ids.
  // Loads are issued SU at a time, unconditionally, so the L2 latency is paid once per batch, not per element.
  float tm = -INFINITY, tsum = 0.f, sm = -INFINITY, ssum = 0.f;
  for (int base = 0; base < V; base += ST * SU) {
    float xv[SU];
#pragma unroll
    for (int u = 0; u < SU; ++u) {
      const int id = base + u * ST + threadIdx.x;
      xv[u] = (id < V) ? x[id] : -INFINITY;
    }
#pragma unroll
    for (int u = 0; u < SU; ++u) {
      const int id = base + u * ST + threadIdx.x;
      if (id >= V || !allowed(r, id)) continue;
      const float v = xv[u];
      if (id < tb) {
        if (v > tm) { tsum = tsum * __expf(tm - v) + 1.f; tm = v; } else tsum += __expf(v - tm);
      } else {
        if (v > sm) { ssum = ssum * __expf(sm - v) + 1.f; sm = v; } else ssum += __expf(v - sm);
      }
    }
  }
  block_ms(tm, tsum, sh_m, sh_s);
  block_ms(sm, ssum, sh_m, sh_s);
  bool mask_text = false;
  if (r.use_ts_rules && ssum > 0.f) {
    const float lse_ts = sm + logf(ssum);
    mask_text = lse_ts > tm;  // logsumexp(timestamp logprobs) > max text logprob
  }
  float lse;
  if (mask_text || tsum == 0.f) lse = sm + logf(ssum);
  else if (ssum == 0.f) lse = tm + logf(tsum);
  else { float m = tm, t = tsum; ms_merge(m, t, sm, ssum); lse = m + logf(t); }

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float temperature = rs.temperature[q];
  if (rs.greedy[q] && temperature > 0.f) {
    // GreedyDecoder.update at temperature T: next ~ Categorical(logits / T) over the filtered logits, drawn as
    // argmax(logits / T + Gumbel noise); its log-probability is taken from the un-tempered log-softmax (lse above).
    // First sampled position: all best_of hypotheses still share this one logits row -> one draw per hypothesis.
    const unsigned long long seed = ((unsigned long long)rs.seed_hi[q] << 32) | rs.seed_lo[q];
    const int n_draw = first ? rs.n_beam[q] : 1;
    for (int k = 0; k < n_draw; ++k) {
      const int stream = first ? k : s - rs.first_seq[q];
      float bv = -INFINITY;
      int bi = INT_MAX;
      for (int id = threadIdx.x; id < V; id += ST) {
        if ((mask_text && id < tb) || !allowed(r, id)) continue;
        const float xv = x[id];
        if (xv == -INFINITY) continue;
        const float u = sample_uniform(seed, stream, cur_len, id);
        const float key = xv / temperature - logf(-logf(u));
        if (better(key, id, bv, bi)) { bv = key; bi = id; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
      }
      __syncthreads();
      if (lane == 0) { wv[warp] = bv; wi[warp] = bi; }
      __syncthreads();
      if (threadIdx.x == 0) {
        float fv = wv[0]; int fi = wi[0];
        for (int w = 1; w < ST / 32; ++w)
          if (better(wv[w], wi[w], fv, fi)) { fv = wv[w]; fi = wi[w]; }
        cand_tok[lr * kMaxCand + k] = (fi == INT_MAX) ? -1 : fi;
        cand_lp[lr * kMaxCand + k] = (fi == INT_MAX) ? -INFINITY : x[fi] - lse;
      }
    }
    return;
  }

  // pass B: per-thread sorted top lists, then kMaxCand rounds of block-wide argmax
  float v[kMaxCand];
  int ix[kMaxCand];
#pragma unroll
  for (int i = 0; i < kMaxCand; ++i) { v[i] = -INFINITY; ix[i] = INT_MAX; }
  const int K = rs.greedy[q] ? 1 : rs.n_beam[q] + 1;
  for (int base = 0; base < V; base += ST * SU) {
    float xv[SU];
#pragma unroll
    for (int u = 0; u < SU; ++u) {
      const int id = base + u * ST + threadIdx.x;
      xv[u] = (id < V) ? x[id] : -INFINITY;
    }
#pragma unroll
    for (int u = 0; u < SU; ++u) {
      const int id = base + u * ST + threadIdx.x;
      const float val = xv[u];
      if (id >= V || !(val > v[kMaxCand - 1])) continue;  // cheap reject first: almost every element
      if (mask_text && id < tb) continue;
      if (!allowed(r, id)) continue;
      v[kMaxCand - 1] = val; ix[kMaxCand - 1] = id;
#pragma unroll
      for (int i = kMaxCand - 1; i > 0; --i) {
        if (v[i] > v[i - 1]) {
          const float tv = v[i]; v[i] = v[i - 1]; v[i - 1] = tv;
          const int ti = ix[i]; ix[i] = ix[i - 1]; ix[i - 1] = ti;
        }
      }
    }
  }
  for (int k = 0; k < K; ++k) {
    float bv = v[0];
    int bi = ix[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { wv[warp] = bv; wi[warp] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
      float fv = wv[0]; int fi = wi[0];
      for (int w = 1; w < ST / 32; ++w)
        if (better(wv[w], wi[w], fv, fi)) { fv = wv[w]; fi = wi[w]; }
      win_i = fi;
      cand_tok[lr * kMaxCand + k] = (fi == INT_MAX) ? -1 : fi;
      cand_lp[lr * kMaxCand + k] = (fi == INT_MAX) ? -INFINITY : fv - lse;
    }
    __syncthreads();
    if (ix[0] == win_i && win_i != INT_MAX) {
#pragma unroll
      for (int i = 0; i < kMaxCand - 1; ++i) { v[i] = v[i + 1]; ix[i] = ix[i + 1]; }
      v[kMaxCand - 1] = -INFINITY; ix[kMaxCand - 1] = INT_MAX;
    }
  }
}

__global__ void __launch_bounds__(32)
beam_update_kernel(const int* __restrict__ active_req, const int* __restrict__ req_first_lrow,
                   const int* __restrict__ active_force, const TokenTables tt,
                   const ReqState rs, const SeqState ss, int anc_cur, int n_ctx, const int* __restrict__ cand_tok,
                   const float* __restrict__ cand_lp) {
  pdl_trigger();
  pdl_wait();
  const int q = active_req[blockIdx.x];
  const int lr0 = req_first_lrow[blockIdx.x];
  const int lane = threadIdx.x;
  const int G = rs.n_beam[q];
  const int first_seq = rs.first_seq[q];
  const int cur_len = rs.cur_len[q];
  const int pos = cur_len - 1;  // position of the tokens that were just fed
  const bool first = (cur_len == rs.sample_begin[q]);
  const unsigned char* anc_c = ss.anc[anc_cur];
  unsigned char* anc_n = ss.anc[anc_cur ^ 1];
  __shared__ int new_src[kMaxBeam];
  __shared__ int n_new;

  if (lane == 0) {
    int old_next[kMaxBeam], old_lts[kMaxBeam];
    float old_sum[kMaxBeam];
    for (int j = 0; j < G; ++j) {
      old_next[j] = ss.next_tok[first_seq + j];
      old_lts[j] = ss.last_ts[first_seq + j];
      old_sum[j] = ss.sum_logprob[first_seq + j];
    }
    int ntok[kMaxBeam], nsrc[kMaxBeam];
    float nsum[kMaxBeam];
    int saved = 0;
    if (rs.greedy[q]) {
      // GreedyDecoder.update: n_group == 1 at temperature 0, best_of independent samples above it.  A hypothesis
      // that has emitted EOT keeps emitting it and stops accumulating; completed once every hypothesis ended.
      // Before the first sampled token all hypotheses share logits row lr0 (draw j of it belongs to hypothesis j).
      bool all_eot = true;
      for (int j = 0; j < G; ++j) {
        const int c = first ? lr0 * kMaxCand + j : (lr0 + j) * kMaxCand;
        const int force = active_force ? active_force[blockIdx.x] : -1;
        const int tok = force >= 0 ? force : cand_tok[c];
        const float lp = cand_lp[c];
        const int last = old_next[j];
        nsum[j] = old_sum[j] + ((last != tt.eot) ? lp : 0.f);
        ntok[j] = (last == tt.eot) ? tt.eot : tok;
        nsrc[j] = first ? 0 : j;
        all_eot = all_eot && ntok[j] == tt.eot;
      }
      saved = G;
      if (all_eot) rs.completed[q] = 1;
    } else {
      // BeamSearchDecoder.update: candidates (beam j, rank k), stable sort by cumulative logprob
      const int nb = first ? 1 : G;  // all beams are identical before the first sampled token
      const int K = G + 1;
      float sc[kMaxBeam * kMaxCand];
      short order[kMaxBeam * kMaxCand];
      int n = 0;
      for (int j = 0; j < nb; ++j)
        for (int k = 0; k < K; ++k) {
          const int lr = first ? lr0 : lr0 + j;
          if (cand_tok[lr * kMaxCand + k] < 0) continue;
          const float val = old_sum[j] + cand_lp[lr * kMaxCand + k];
          int p = n++;
          while (p > 0 && sc[p - 1] < val) { sc[p] = sc[p - 1]; order[p] = order[p - 1]; --p; }
          sc[p] = val; order[p] = (short)(j * kMaxCand + k);
        }
      int n_fin = rs.n_finished[q];
      const int max_cand = rs.max_candidates[q];
      for (int c = 0; c < n && saved < G; ++c) {
        const int j = order[c] / kMaxCand, k = order[c] % kMaxCand;
        const int lr = first ? lr0 : lr0 + j;
        const int tok = cand_tok[lr * kMaxCand + k];
        if (tok == tt.eot) {
          if (n_fin < max_cand && n_fin < kMaxFinished) {
            rs.fin_score[q * kMaxFinished + n_fin] = sc[c];
            rs.fin_pos[q * kMaxFinished + n_fin] = pos;
            rs.fin_slot[q * kMaxFinished + n_fin] = anc_c[(long long)(first_seq + j) * n_ctx + pos];
            ++n_fin;
          }
        } else {
          nsum[saved] = sc[c]; ntok[saved] = tok; nsrc[saved] = j;
          ++saved;
        }
      }
      while (saved < G && saved > 0) {  // degenerate: fewer than G finite candidates
        nsum[saved] = nsum[saved - 1]; ntok[saved] = ntok[saved - 1]; nsrc[saved] = nsrc[saved - 1];
        ++saved;
      }
      rs.n_finished[q] = n_fin;
      if (n_fin >= max_cand) rs.completed[q] = 1;
    }
    const int npos = pos + 1;
    for (int j = 0; j < saved; ++j) {
      const int sj = first_seq + j, src = nsrc[j];
      ss.sum_logprob[sj] = nsum[j];
      ss.prev_tok[sj] = old_next[src];
      ss.next_tok[sj] = ntok[j];
      ss.last_ts[sj] = (ntok[j] >= tt.timestamp_begin) ? ntok[j] : old_lts[src];
      if (npos < n_ctx) {
        rs.tok[((long long)q * n_ctx + npos) * kMaxBeam + j] = ntok[j];
        rs.parent[((long long)q * n_ctx + npos) * kMaxBeam + j] = anc_c[(long long)(first_seq + src) * n_ctx + pos];
      }
      new_src[j] = src;
      rs.last_src[q * kMaxBeam + j] = (unsigned char)src;
    }
    n_new = saved;
    rs.cur_len[q] = cur_len + 1;
  }
  __syncwarp();
  // ancestry tables of the surviving beams (this is rearrange_kv_cache: no K/V bytes move)
  const int nn = n_new;
  for (int j = 0; j < nn; ++j) {
    const unsigned char* src = anc_c + (long long)(first_seq + new_src[j]) * n_ctx;
    unsigned char* dst = anc_n + (long long)(first_seq + j) * n_ctx;
    for (int t = lane; t <= pos; t += 32) dst[t] = src[t];
    if (lane == 0 && pos + 1 < n_ctx) dst[pos + 1] = (unsigned char)j;
  }
}

__global__ void __launch_bounds__(ST)
no_speech_kernel(const float* __restrict__ logits, int ld, int V, const int* __restrict__ lrows, const int* __restrict__ reqs,
                 int no_speech_id, float* __restrict__ out_prob) {
  __shared__ float sh_m[ST / 32], sh_s[ST / 32];
  pdl_trigger();
  pdl_wait();
  const float* x = logits + (long long)lrows[blockIdx.x] * ld;
  float m = -INFINITY, s = 0.f;
  for (int id = threadIdx.x; id < V; id += ST) ms_merge(m, s, x[id], 1.f);
  block_ms(m, s, sh_m, sh_s);
  if (threadIdx.x == 0) out_prob[reqs[blockIdx.x]] = expf(x[no_speech_id] - m) / s;
}

// upstream detect_language on one logits row, for a block of 128 threads: every logit but the language tokens'
// masked, arg-max (lowest id on ties) and softmax.  probs[i] = P(first_lang + i); returns the arg-max token id in every
// thread.  Both detection paths (language_probs_kernel, detect_language_kernel) run exactly this arithmetic.
__device__ __forceinline__ int language_softmax_argmax(const float* __restrict__ logits, int first_lang, int n_lang,
                                                       float* __restrict__ probs) {
  __shared__ float sv[128];
  __shared__ int si[128];
  const int t = threadIdx.x;
  float v = (t < n_lang) ? logits[first_lang + t] : -INFINITY;
  sv[t] = v; si[t] = t;
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (t < o && better(sv[t + o], si[t + o], sv[t], si[t])) { sv[t] = sv[t + o]; si[t] = si[t + o]; }
    __syncthreads();
  }
  const float mx = sv[0];
  const int am = si[0];
  __syncthreads();
  const float e = (t < n_lang) ? expf(v - mx) : 0.f;
  sv[t] = e;
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (t < o) sv[t] += sv[t + o];
    __syncthreads();
  }
  if (t < n_lang) probs[t] = e / sv[0];
  return first_lang + am;
}

__global__ void __launch_bounds__(128)
language_probs_kernel(const float* __restrict__ logits, int first_lang, int n_lang, float* __restrict__ probs,
                      int* __restrict__ argmax_out) {
  const int tok = language_softmax_argmax(logits, first_lang, n_lang, probs);
  if (threadIdx.x == 0) *argmax_out = tok;
}

// One block per detect-mode decode in the step that fed its <|sot|> row: the language token goes to the request's
// language slot and to next_tok of its first hypothesis, which the next step's language row embeds (row_tok = -1).
__global__ void __launch_bounds__(128)
detect_language_kernel(const float* __restrict__ logits, int ld, const int* __restrict__ lrows, const int* __restrict__ reqs,
                       int first_lang, int n_lang, const ReqState rs, const SeqState ss, float* __restrict__ probs,
                       int* __restrict__ lang_tok) {
  pdl_trigger();
  pdl_wait();
  const int q = reqs[blockIdx.x];
  const int tok = language_softmax_argmax(logits + (long long)lrows[blockIdx.x] * ld, first_lang, n_lang, probs + (long long)q * kMaxLanguages);
  if (threadIdx.x == 0) {
    lang_tok[q] = tok;
    ss.next_tok[rs.first_seq[q]] = tok;
  }
}

}  // namespace

void sample_topk(const float* logits, int ld, int V, const int* srow_lrow, const int* lrow_req, const int* lrow_seq, int n_lrows,
                 const TokenTables& tt, const ReqState& rs, const SeqState& ss, int anc_cur, int* cand_tok, float* cand_lp,
                 cudaStream_t stream) {
  (void)anc_cur;
  if (n_lrows <= 0) return;
  launch_kernel(sample_topk_kernel, dim3(n_lrows), dim3(ST), 0, stream, logits, ld, V, srow_lrow, lrow_req, lrow_seq, tt, rs, ss, cand_tok, cand_lp);
  ++g_kernel_launches;
}

void beam_update(const int* active_req, const int* req_first_lrow, const int* active_force, int n_active, const TokenTables& tt,
                 const ReqState& rs, const SeqState& ss, int anc_cur, int n_ctx, const int* cand_tok, const float* cand_lp,
                 cudaStream_t stream) {
  if (n_active <= 0) return;
  launch_kernel(beam_update_kernel, dim3(n_active), dim3(32), 0, stream, active_req, req_first_lrow, active_force, tt, rs, ss, anc_cur,
                n_ctx, cand_tok, cand_lp);
  ++g_kernel_launches;
}

void no_speech_prob(const float* logits, int ld, int V, const int* lrows, const int* reqs, int n, int no_speech_id,
                    float* out_prob, cudaStream_t stream) {
  if (n <= 0) return;
  launch_kernel(no_speech_kernel, dim3(n), dim3(ST), 0, stream, logits, ld, V, lrows, reqs, no_speech_id, out_prob);
  ++g_kernel_launches;
}

void language_probs(const float* logits, int V, int first_lang, int n_lang, float* probs_out, int* argmax_out,
                    cudaStream_t stream) {
  (void)V;
  BW_CHECK(n_lang <= 128, "too many languages");
  language_probs_kernel<<<1, 128, 0, stream>>>(logits, first_lang, n_lang, probs_out, argmax_out);
  BW_CUDA(cudaGetLastError());
  ++g_kernel_launches;
}

void detect_language(const float* logits, int ld, const int* lrows, const int* reqs, int n, const TokenTables& tt, const ReqState& rs,
                     const SeqState& ss, float* probs, int* lang_tok, cudaStream_t stream) {
  if (n <= 0) return;
  BW_CHECK(tt.num_languages > 0 && tt.num_languages <= kMaxLanguages, "language detection needs 1 to 128 language tokens");
  launch_kernel(detect_language_kernel, dim3(n), dim3(128), 0, stream, logits, ld, lrows, reqs, tt.first_language_token, tt.num_languages,
                rs, ss, probs, lang_tok);
  ++g_kernel_launches;
}

}  // namespace bw
