"""ctypes binding of libb200whisper.so (the C ABI declared in include/b200_whisper.h).

There is no fallback: if the shared library is missing or no sm_100 GPU is usable, importing the
engine raises.  Build with `python __graft_entry__.py build` (or `make -C csrc`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200W_LIB", os.path.join(_HERE, "libb200whisper.so"))

BW_MAX_TOKENS = 448
BW_COMPUTE_BF16, BW_COMPUTE_FP32 = 0, 1
BW_F32, BW_F16, BW_BF16 = 0, 1, 2
BW_FLAG_FORCE_SIMT_GEMM, BW_FLAG_NO_SCHEDULER, BW_FLAG_CROSS_KV_INT8, BW_FLAG_SIMT_ATTENTION = 1, 2, 4, 8
LANGUAGE_PLACEHOLDER = -1  # initial_tokens[1] of a detect-mode decode (bw_call_decode_detect): the engine fills it
STAT_NAMES = ("kernel_launches", "decode_steps", "rows", "windows", "max_segments", "max_sequences",
              "encoder_batches", "h2d_bytes", "d2h_bytes", "kv_pages_total", "kv_pages_in_use", "kv_pages_peak", "kv_page_bytes")

c_i32_p = C.POINTER(C.c_int32)
c_f32_p = C.POINTER(C.c_float)


class ModelDimsC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_mels", "n_audio_ctx", "n_audio_state", "n_audio_head", "n_audio_layer",
        "n_vocab", "n_text_ctx", "n_text_state", "n_text_head", "n_text_layer")]


class EngineConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "cuda_device", "compute", "max_segments", "max_sequences", "max_encoder_batch", "flags", "max_kv_pages")]


class TensorDescC(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("dtype", C.c_int32), ("ndim", C.c_int32),
                ("shape", C.c_int64 * 4)]


class TokenTablesC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "eot", "sot", "sot_prev", "sot_lm", "no_speech", "no_timestamps", "timestamp_begin",
        "translate", "transcribe", "first_language_token", "num_languages")] + [
        ("suppress", c_i32_p), ("n_suppress", C.c_int32), ("blank", c_i32_p), ("n_blank", C.c_int32)]


class DecodeOptsC(C.Structure):
    _fields_ = [("initial_tokens", c_i32_p), ("n_initial", C.c_int32), ("sot_index", C.c_int32),
                ("beam_size", C.c_int32), ("patience", C.c_float), ("length_penalty", C.c_float),
                ("sample_len", C.c_int32), ("without_timestamps", C.c_int32), ("suppress_blank", C.c_int32),
                ("max_initial_timestamp_index", C.c_int32), ("temperature", C.c_float), ("best_of", C.c_int32),
                ("seed_lo", C.c_uint32), ("seed_hi", C.c_uint32), ("max_candidates", C.c_int32)]


class GemmDescC(C.Structure):
    _fields_ = [("A", C.c_void_p), ("B", C.c_void_p), ("C", C.c_void_p), ("bias", C.c_void_p), ("residual", C.c_void_p)] + [
        (n, C.c_int32) for n in ("M", "N", "K", "lda", "ldb", "ldc", "ldres", "Z", "a_rows", "b_rows")] + [
        (n, C.c_int64) for n in ("a_zstride", "b_zstride", "c_zstride", "bias_zstride", "res_zstride")] + [
        (n, C.c_int32) for n in ("gelu", "out_fp32", "transposed")]


# bw_test_gemm routes: BW_GEMM_ROUTE(kernel, param) of include/b200_whisper_hooks.h
BW_GEMM_PAIR, BW_GEMM_SPLITK, BW_GEMM_ROWS, BW_GEMM_TILE, BW_GEMM_SIMT = 1, 2, 3, 4, 5


def gemm_route(kernel: int, param: int = 0) -> int:
    return kernel * 1000 + param


class ResultC(C.Structure):
    _fields_ = [("n_tokens", C.c_int32), ("tokens", C.c_int32 * BW_MAX_TOKENS), ("sum_logprob", C.c_float),
                ("avg_logprob", C.c_float), ("no_speech_prob", C.c_float), ("n_steps", C.c_int32),
                ("t_queue", C.c_float), ("t_encode", C.c_float), ("t_decode", C.c_float)]


class LangResultC(C.Structure):
    _fields_ = [("language_token", C.c_int32), ("n_languages", C.c_int32), ("probs", C.c_float * 128)]


# name -> (restype, argtypes); every symbol include/b200_whisper.h (the drop-in boundary) and
# include/b200_whisper_hooks.h (bench / test hooks) declare
SIGNATURES = {
    "bw_last_error": (C.c_char_p, []),
    "bw_version": (C.c_int, []),
    "bw_device_count": (C.c_int, []),
    "bw_engine_create": (C.c_int, [C.POINTER(ModelDimsC), C.POINTER(EngineConfigC), C.POINTER(C.c_void_p)]),
    "bw_engine_load_weights": (C.c_int, [C.c_void_p, C.POINTER(TensorDescC), C.c_int32]),
    "bw_engine_set_tables": (C.c_int, [C.c_void_p, C.POINTER(TokenTablesC)]),
    "bw_engine_set_mel_filters": (C.c_int, [C.c_void_p, c_f32_p]),
    "bw_engine_finalize": (C.c_int, [C.c_void_p]),
    "bw_engine_destroy": (C.c_int, [C.c_void_p]),
    "bw_engine_retain": (C.c_int, [C.c_void_p]),
    "bw_engine_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.c_int32]),
    "bw_call_open": (C.c_int, [C.c_void_p, c_f32_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "bw_engine_set_resampler": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_f32_p]),
    "bw_call_open_pcm16": (C.c_int, [C.c_void_p, C.POINTER(C.c_int16), C.c_int64, C.c_int32, C.POINTER(C.c_void_p)]),
    "bw_resample_pcm16": (C.c_int, [C.c_void_p, C.POINTER(C.c_int16), C.c_int64, C.c_int32, c_f32_p, C.POINTER(C.c_int64)]),
    "bw_call_content_frames": (C.c_int, [C.c_void_p, c_i32_p]),
    "bw_call_decode": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(DecodeOptsC), C.POINTER(ResultC)]),
    "bw_decode_many": (C.c_int, [C.POINTER(C.c_void_p), c_i32_p, C.POINTER(DecodeOptsC), C.POINTER(ResultC), c_i32_p, C.c_int32]),
    "bw_call_detect_language": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(LangResultC)]),
    "bw_call_decode_detect": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(DecodeOptsC), C.POINTER(ResultC), C.POINTER(LangResultC)]),
    "bw_decode_many_detect": (C.c_int, [C.POINTER(C.c_void_p), c_i32_p, C.POINTER(DecodeOptsC), C.POINTER(ResultC),
                                        C.POINTER(LangResultC), c_i32_p, C.c_int32]),
    "bw_call_close": (C.c_int, [C.c_void_p]),
    "bw_mel": (C.c_int, [C.c_void_p, c_f32_p, C.c_int64, C.c_int32, c_f32_p, c_i32_p]),
    "bw_encode": (C.c_int, [C.c_void_p, c_f32_p, C.c_int32, c_f32_p]),
    "bw_decode_logits": (C.c_int, [C.c_void_p, c_f32_p, c_i32_p, C.c_int32, c_f32_p]),
    "bw_gemm_bf16": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                               C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "bw_test_gemm": (C.c_int, [C.POINTER(GemmDescC), C.c_int32, C.c_int32, c_i32_p, C.c_void_p]),
    "bw_test_gemm_route": (C.c_int, [C.POINTER(GemmDescC), c_i32_p]),
    "bw_attention_bf16": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "bw_bench_cross_attention": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, c_f32_p, C.POINTER(C.c_double)]),
    "bw_bench_encoder": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, c_f32_p, C.POINTER(C.c_double)]),
    "bw_bench_mel": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, c_f32_p, C.POINTER(C.c_double)]),
    "bw_bench_pipeline": (C.c_int, [C.c_void_p, c_f32_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int32, C.c_int32,
                                    C.c_int32, c_f32_p]),
    "bw_bench_pipeline_results": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.POINTER(ResultC)]),
    "bw_bench_decoder_step": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_f32_p,
                                        C.POINTER(C.c_double)]),
    "bw_test_ln_chain": (C.c_int, [C.c_void_p] * 8 + [C.c_int32] * 5 + [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bw_debug_trace": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_uint64), C.c_int32, c_i32_p]),
    "bw_call_decode_forced": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(DecodeOptsC), c_i32_p, C.c_int32, c_f32_p, C.POINTER(ResultC)]),
    "bw_test_dec_cross_attention": (C.c_int, [C.c_void_p] + [C.c_int32] * 6 + [C.c_void_p] * 4 + [C.c_int32] * 4 + [C.c_void_p, C.c_void_p]),
    "bw_test_quantize_cross_kv": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bw_test_dec_cross_attention_int8": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 6 + [C.c_void_p] * 4 + [C.c_int32] * 4 +
                                         [C.c_void_p, C.c_void_p]),
    "bw_test_dec_self_attention": (C.c_int, [C.c_int32] + [C.c_void_p] * 6 + [C.c_int32] * 3 + [C.c_void_p] * 3 +
                                   [C.c_int32] * 4 + [C.c_void_p, C.c_void_p]),
    "bw_test_self_attention_mode": (C.c_int, [C.c_int32]),
    "bw_test_sample_topk": (C.c_int, [C.c_void_p, c_f32_p, C.c_int32, c_i32_p, c_i32_p, c_f32_p]),
    "bw_test_page_collector": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8), c_i32_p]),
}

_lib = None


class B200WhisperError(RuntimeError):
    """Raised for every non-zero bw_status (surfaces as ERR2002 in the reference server,
    stt_server/backend/component/decode_scheduler.py:632-644)."""


def load():
    """Load the shared library (once). Raises OSError with build instructions if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OSError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().bw_last_error()
        raise B200WhisperError(f"{what} failed (bw_status {status}): {msg.decode('utf-8', 'replace') if msg else ''}")
