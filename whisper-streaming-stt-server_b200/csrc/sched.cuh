// Internals shared by api.cu (C ABI), scheduler.cu (continuous-batching scheduler) and hooks.cu (bench / test hooks).
#pragma once
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <stdexcept>
#include <string>

#include "engine.cuh"

namespace bw {
// engine.cu
void engine_build_weight_table(bw_engine* e);
void engine_load_tensor(bw_engine* e, const bw_tensor_desc& t);
void engine_encoder_forward(bw_engine* e, int nb);
void engine_cross_kv(bw_engine* e, int bi, int q);
void engine_window_to_A1(bw_engine* e, const float* logmel, int ld, int n_real, const int* gmax, int seek, int seg, int bi);
void engine_decoder_layers(bw_engine* e, DecGroup& G, int R, int n_groups, int max_group_rows, int n_lrows, int max_ctx, const int* row_seq,
                           const int* row_pos, const int* row_tok, const int* row_bpos, const int* row_page, const int* grp_first,
                           const int* grp_n, const int* grp_x, const int* lrow_src);
void engine_init_requests(bw_engine* e, const int* init_dev, int n);
void engine_fold_layernorms(bw_engine* e);
void engine_gather_final(bw_engine* e, const int* list_dev, int n, int blob_bytes, unsigned char* out_dev);

std::string& last_error();  // thread-local message behind bw_last_error()

struct DeviceGuard {
  int prev = 0;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) BW_CUDA(cudaSetDevice(dev));
  }
  ~DeviceGuard() { cudaSetDevice(prev); }
};

// ---- per-group control block (ints), mirrored host (pinned) / device ----
struct Ctl {
  int *row_seq, *row_pos, *row_tok, *row_bpos, *row_page, *grp_first, *grp_n, *grp_x, *lrow_src, *srow_lrow, *srow_req, *srow_seq, *act_req,
      *act_first, *act_force, *ns_lrow, *ns_req;
  int* base = nullptr;
  size_t total = 0;
  // fill counters of the step being built
  int R = 0, NG = 0, LR = 0, SR = 0, NA = 0, NNS = 0, max_grp = 1, max_ctx = 0;
  void layout(int* b, int Rm, int LRm, int Q) {
    base = b;
    int* p = b;
    auto take = [&](size_t n) { int* r = p; p += n; return r; };
    row_seq = take(Rm); row_pos = take(Rm); row_tok = take(Rm); row_bpos = take(Rm); row_page = take(Rm);
    grp_first = take(Rm); grp_n = take(Rm); grp_x = take(Rm);
    lrow_src = take(LRm); srow_lrow = take(LRm); srow_req = take(LRm); srow_seq = take(LRm);
    act_req = take(Q); act_first = take(Q); act_force = take(Q); ns_lrow = take(Q); ns_req = take(Q);
    total = (size_t)(p - b);
  }
  void reset() { R = NG = LR = SR = NA = NNS = 0; max_grp = 1; max_ctx = 0; }
};

// scheduler.cu
void enqueue_group_step(bw_engine* e, DecGroup& G, Ctl& c);
int choose_groups(int n_segments);
void scheduler_main(bw_engine* e);
// self-KV page pool (host free list; scheduler thread / synthetic benches only)
int kv_blocks_for(int n_tokens);                       // pages one hypothesis needs for n_tokens positions
int kv_page_of(bw_engine* e, Request* r, int slot, int block);  // the request's page for (beam slot, block), allocated on demand
void kv_release(bw_engine* e, Request* r);             // every page + the reservation of a finished request
int page_collector_replay(int G, int n_init, int n_steps, const unsigned char* parents, unsigned char* alloc_masks, int* pages_in_use);
int submit_and_wait(bw_engine* e, Request& r);
// one host thread hands a whole batch to the scheduler and waits for every request of it
int submit_many_and_wait(bw_engine* e, const std::vector<Request*>& rs);
// validates `opts` and fills the decode fields of `r` (shared by bw_call_decode, bw_decode_many and the test hooks)
void fill_decode_request(Request& r, bw_call* c, int seek, const bw_decode_opts* o, bw_result* out);
size_t fin_blob_bytes(bw_engine* e);
// one finished request's blob (engine_gather_final) -> r->out: the ranker's pick among the request's hypotheses
void finalize_decode(bw_engine* e, Request* r, const unsigned char* blob);

}  // namespace bw

#define BW_API_BEGIN try {
#define BW_API_END                                                     \
  }                                                                    \
  catch (const bw::CudaError& ex) { bw::last_error() = ex.what(); return BW_ERR_CUDA; }      \
  catch (const std::invalid_argument& ex) { bw::last_error() = ex.what(); return BW_ERR_INVALID; } \
  catch (const std::bad_alloc& ex) { bw::last_error() = ex.what(); return BW_ERR_NOMEM; }    \
  catch (const std::exception& ex) { bw::last_error() = ex.what(); return BW_ERR_STATE; }    \
  return BW_OK;
