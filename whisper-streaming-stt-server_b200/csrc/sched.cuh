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
CrossKV engine_cross_kv_desc(const bw_engine* e);  // the cross cache as the decoder step reads it
void engine_window_to_A1(bw_engine* e, const float* logmel, int ld, int n_real, const int* gmax, int seek, int seg, int bi);
void engine_decoder_layers(bw_engine* e);  // the step that e->dec.ctl describes, on e->dec.stream
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

// scheduler.cu
// the decoder step that e->dec.ctl describes (control upload included), a CUDA graph from the third step of its shape
void enqueue_step(bw_engine* e);
// completion of the step: the flags and beam parents (st_step) to h_flags, one host synchronisation, anc_cur flipped
void finish_step(bw_engine* e);
void scheduler_main(bw_engine* e);
// self-KV page pool (host free list; scheduler thread / synthetic benches only)
int kv_blocks_for(int n_tokens);                       // pages one hypothesis needs for n_tokens positions
int kv_page_of(bw_engine* e, Request* r, int slot, int block);  // the request's page for (beam slot, block), allocated on demand
void kv_release(bw_engine* e, Request* r);             // every page + the reservation of a finished request
int page_collector_replay(int G, int n_init, int n_steps, const unsigned char* parents, unsigned char* alloc_masks, int* pages_in_use);
int submit_and_wait(bw_engine* e, Request& r);
// one host thread hands a whole batch to the scheduler and waits for every request of it
int submit_many_and_wait(bw_engine* e, const std::vector<Request*>& rs);
// validates `opts` and fills the decode fields of `r` (shared by bw_call_decode, bw_decode_many and the test hooks).
// lang != nullptr: detect mode (bw_call_decode_detect), initial_tokens[1] holds kLanguagePlaceholder.
constexpr int kLanguagePlaceholder = -1;
void fill_decode_request(Request& r, bw_call* c, int seek, const bw_decode_opts* o, bw_result* out, bw_lang_result* lang = nullptr);
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
