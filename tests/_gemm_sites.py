"""The engine's GEMM call sites as bw_gemm_desc argument forms (csrc/engine.cu), and the names of the GEMM routes.

Shared by tests/test_gemm_routes_cpu.py (which route the dispatcher picks for each site) and
tests/test_gpu_gemm_layouts.py (each form and route against an fp64 reference on the B200)."""
from __future__ import annotations

import ctypes as C

from b200_whisper import _lib as L
from b200_whisper.synth import MODEL_DIMS

# every dimension set of the model zoo that the call-site table is built for (three vocabulary sizes: ragged M of the
# swap-AB vocabulary projection)
MODELS = ("test-tiny", "test-v3", "tiny.en", "tiny", "base", "small", "medium", "large-v3")

# engine pools with the default configuration (csrc/api.cu bw_engine_finalize): Q = max_segments = 64,
# S = max_sequences = 2 Q, R_max = S + 512 decoder rows, LR_max = S + Q + BW_MAX_TOKENS logit rows
Q_DEFAULT = 64
S_DEFAULT = 2 * Q_DEFAULT
R_MAX = S_DEFAULT + 512
LR_MAX = S_DEFAULT + Q_DEFAULT + L.BW_MAX_TOKENS
DECODER_ROWS = (1, 5, 37, 128, 129, 320, 640)
T_ENC = 1500  # n_audio_ctx of every model
ENC_CHUNK = 8  # encoder_forward_t's default sub-batch size (B200W_ENC_CHUNK)

ENCODER_SITES = ("conv1", "conv2", "enc_qkv", "enc_wo", "enc_w1", "enc_w2")
DECODER_SITES = ("dec_qkv", "dec_wo", "dec_q_x", "dec_wo_x", "dec_w1", "dec_w2", "vocab")
SITES = ENCODER_SITES + ("cross_kv",) + DECODER_SITES


def encoder_sub_batches(nb: int) -> list:
    """Window counts of the sub-batches encoder_forward_t (csrc/engine.cu:482) runs for a batch of nb windows."""
    if nb < 4:
        return [nb]
    chunk = max(2, min(ENC_CHUNK, (nb + 1) // 2))
    return [min(chunk, nb - w0) for w0 in range(0, nb, chunk)]


ENCODER_Z = tuple(sorted({n for nb in range(1, 17) for n in encoder_sub_batches(nb)}))


def _form(M, N, K, *, lda=None, ldb=None, ldc=None, ldres=None, Z=1, a_rows=0, b_rows=0, a_zstride=0, b_zstride=0,
          c_zstride=0, bias_zstride=0, res_zstride=0, gelu=False, out_fp32=False, transposed=False, bias=False,
          residual=False, inplace=False):
    return dict(M=M, N=N, K=K, lda=lda or K, ldb=ldb or K, ldc=ldc or (M if transposed else N),
                ldres=(ldres or (M if transposed else N)) if residual else 0, Z=Z, a_rows=a_rows, b_rows=b_rows,
                a_zstride=a_zstride, b_zstride=b_zstride, c_zstride=c_zstride, bias_zstride=bias_zstride,
                res_zstride=res_zstride, gelu=int(gelu), out_fp32=int(out_fp32), transposed=int(transposed), bias=bias,
                residual=residual, inplace=inplace)


def site_form(model: str, site: str, batch: int) -> dict:
    """The GemmArgs csrc/engine.cu builds for `site` of `model` in bf16 tensor-core mode.  batch = windows of the encoder
    sub-batch (encoder sites), ignored for cross_kv (Z = n_text_layer), decoder rows R (decoder sites; the vocabulary
    projection runs on the R logit rows)."""
    d = MODEL_DIMS[model]
    dm, nm = d.n_audio_state, d.n_mels
    n = batch
    if site == "conv1":  # engine.cu:145 conv1 + GELU, [n * 3000, 3 n_mels] x [dm, 3 n_mels]
        return _form(n * 3000, dm, 3 * nm, gelu=True, bias=True)
    if site == "conv2":  # engine.cu:152 per window: im2col [1500, 3 dm] x conv2_w (broadcast) + bias, GELU, + pos. emb.
        return _form(T_ENC, dm, 3 * dm, Z=n, a_zstride=T_ENC * 3 * dm, b_zstride=0, c_zstride=T_ENC * dm, res_zstride=0,
                     bias_zstride=0, gelu=True, out_fp32=True, bias=True, residual=True)
    if site == "enc_qkv":  # engine.cu:163
        return _form(n * T_ENC, 3 * dm, dm, bias=True)
    if site == "enc_wo":  # engine.cu:175, in place on the fp32 residual stream
        return _form(n * T_ENC, dm, dm, out_fp32=True, bias=True, residual=True, inplace=True)
    if site == "enc_w1":  # engine.cu:182
        return _form(n * T_ENC, 4 * dm, dm, gelu=True, bias=True)
    if site == "enc_w2":  # engine.cu:188, in place on the fp32 residual stream
        return _form(n * T_ENC, dm, 4 * dm, out_fp32=True, bias=True, residual=True, inplace=True)
    if site == "cross_kv":  # engine.cu:199 one launch, z = decoder layer: encoder output broadcast, per-layer W and bias
        L_ = d.n_text_layer
        return _form(T_ENC, 2 * dm, dm, Z=L_, a_zstride=0, b_zstride=2 * dm * dm, c_zstride=T_ENC * 2 * dm,
                     bias_zstride=2 * dm, bias=True)
    R = batch
    # linear_rows, engine.cu:114 (the decoder step without the LayerNorm fusion, B200W_NO_LN_FUSION): A = activations
    # with R_max rows allocated behind them
    if site == "dec_qkv":  # engine.cu:250
        return _form(R, 3 * dm, dm, a_rows=R_MAX, out_fp32=True, bias=True)
    if site in ("dec_wo", "dec_wo_x"):  # engine.cu:252 / 257, in place on the residual stream
        return _form(R, dm, dm, a_rows=R_MAX, out_fp32=True, bias=True, residual=True, inplace=True)
    if site == "dec_q_x":  # engine.cu:254
        return _form(R, dm, dm, a_rows=R_MAX, out_fp32=True, bias=True)
    if site == "dec_w1":  # engine.cu:259
        return _form(R, 4 * dm, dm, a_rows=R_MAX, gelu=True, bias=True)
    if site == "dec_w2":  # engine.cu:260, in place on the residual stream
        return _form(R, dm, 4 * dm, a_rows=R_MAX, out_fp32=True, bias=True, residual=True, inplace=True)
    if site == "vocab":  # engine.cu:264 / 308: N = n_vocab > 8192 -> swap-AB, logits [R, n_vocab] = (W . X^T)^T
        return _form(d.n_vocab, R, dm, ldc=d.n_vocab, b_rows=LR_MAX, out_fp32=True, transposed=True)
    raise KeyError(site)


def site_batches(site: str) -> tuple:
    if site in ENCODER_SITES:
        return ENCODER_Z
    if site == "cross_kv":
        return (0,)
    return DECODER_ROWS


def desc_of(form: dict, A=0x1000, B=0x2000, C_=0x3000, bias=0x4000, residual=0x5000) -> L.GemmDescC:
    """bw_gemm_desc of a form; the default pointers are placeholders for the host-only route query."""
    d = L.GemmDescC()
    d.A, d.B, d.C = A, B, C_
    d.bias = bias if form["bias"] else None
    d.residual = residual if form["residual"] else None
    for k in ("M", "N", "K", "lda", "ldb", "ldc", "ldres", "Z", "a_rows", "b_rows", "a_zstride", "b_zstride", "c_zstride",
              "bias_zstride", "res_zstride", "gelu", "out_fp32", "transposed"):
        setattr(d, k, int(form[k]))
    return d


_KERNELS = {L.BW_GEMM_PAIR: "pair", L.BW_GEMM_SPLITK: "splitk", L.BW_GEMM_ROWS: "rows", L.BW_GEMM_TILE: "tile",
            L.BW_GEMM_SIMT: "simt"}


def route_name(code: int) -> str:
    """'pair', 'splitk8', 'rows2', 'rows1' (unsplit), 'tile128', 'simt'"""
    kernel, param = divmod(code, 1000)
    return _KERNELS[kernel] + (str(param) if param else "")


def route_code(name: str) -> int:
    for kernel, kname in _KERNELS.items():
        if name.startswith(kname):
            rest = name[len(kname):]
            return L.gemm_route(kernel, int(rest) if rest else 0)
    raise KeyError(name)


def dispatcher_route(form: dict) -> str:
    lib = L.load()
    out = C.c_int32(-1)
    L.check(lib.bw_test_gemm_route(C.byref(desc_of(form)), C.byref(out)), "bw_test_gemm_route")
    return route_name(out.value)


# (model, call site, batch, route) the GPU layout test runs through the dispatcher: the cheapest production row of every
# (call site, route) pair of the table (ragged row counts where the route allows), plus large-v3 rows with the longest K
# and the largest batch strides.  tests/test_gemm_routes_cpu.py checks that the dispatcher picks `route` for each and that
# the list covers every pair.
GPU_DISPATCH_CASES = (
    ("tiny.en", "conv1", 3, "pair"),
    ("test-tiny", "conv1", 1, "rows2"),
    ("test-tiny", "conv1", 4, "splitk2"),
    ("test-tiny", "conv1", 6, "tile128"),
    ("tiny.en", "conv2", 5, "pair"),
    ("large-v3", "conv2", 2, "pair"),
    ("test-tiny", "conv2", 1, "rows2"),
    ("tiny.en", "conv2", 1, "rows4"),
    ("test-tiny", "conv2", 7, "splitk2"),
    ("tiny.en", "conv2", 3, "splitk4"),
    ("tiny.en", "conv2", 4, "tile128"),
    ("test-tiny", "enc_qkv", 5, "pair"),
    ("tiny.en", "enc_qkv", 1, "splitk2"),
    ("test-tiny", "enc_qkv", 1, "tile128"),
    ("tiny.en", "enc_wo", 5, "pair"),
    ("tiny.en", "enc_wo", 1, "rows2"),
    ("tiny.en", "enc_wo", 3, "splitk2"),
    ("base", "enc_wo", 2, "splitk4"),
    ("test-tiny", "enc_wo", 1, "tile128"),
    ("test-tiny", "enc_w1", 5, "pair"),
    ("test-tiny", "enc_w1", 1, "tile128"),
    ("tiny.en", "enc_w2", 5, "pair"),
    ("test-tiny", "enc_w2", 4, "rows2"),
    ("test-tiny", "enc_w2", 1, "rows4"),
    ("test-tiny", "enc_w2", 7, "splitk4"),
    ("tiny.en", "enc_w2", 4, "tile128"),
    ("large-v3", "enc_w2", 1, "tile128"),
    ("tiny.en", "cross_kv", 0, "pair"),
    ("large-v3", "cross_kv", 0, "pair"),
    ("test-tiny", "cross_kv", 0, "tile128"),
    ("tiny.en", "dec_qkv", 320, "rows2"),
    ("base", "dec_qkv", 1, "rows4"),
    ("small", "dec_qkv", 640, "splitk4"),
    ("test-tiny", "dec_qkv", 37, "tile128"),
    ("tiny.en", "dec_wo", 129, "rows2"),
    ("base", "dec_wo", 5, "rows4"),
    ("medium", "dec_wo", 1, "rows8"),
    ("test-tiny", "dec_wo", 129, "tile128"),
    ("tiny.en", "dec_q_x", 1, "rows2"),
    ("base", "dec_q_x", 37, "rows4"),
    ("medium", "dec_q_x", 128, "rows8"),
    ("test-tiny", "dec_q_x", 1, "tile128"),
    ("tiny.en", "dec_wo_x", 5, "rows2"),
    ("base", "dec_wo_x", 1, "rows4"),
    ("medium", "dec_wo_x", 5, "rows8"),
    ("test-tiny", "dec_wo_x", 5, "tile128"),
    ("large-v3", "dec_w1", 640, "pair"),
    ("tiny.en", "dec_w1", 37, "rows2"),
    ("base", "dec_w1", 129, "rows4"),
    ("base", "dec_w1", 640, "splitk4"),
    ("large-v3", "dec_w1", 129, "splitk8"),
    ("test-tiny", "dec_w1", 1, "tile128"),
    ("medium", "dec_w2", 640, "rows2"),
    ("test-tiny", "dec_w2", 1, "rows4"),
    ("tiny.en", "dec_w2", 37, "rows8"),
    ("large-v3", "dec_w2", 128, "rows8"),
    ("tiny.en", "vocab", 1, "tile32"),
    ("test-tiny", "vocab", 37, "tile64"),
    ("large-v3", "vocab", 129, "tile128"),
)

# (model, call site, batch, route) run on a route the dispatcher does not pick for that row, where its preconditions hold
GPU_FORCED_CASES = (
    ("tiny.en", "conv2", 4, "pair"),
    ("tiny.en", "conv2", 4, "rows2"),
    ("tiny.en", "conv2", 4, "splitk8"),
    ("tiny", "cross_kv", 0, "tile128"),
    ("tiny", "cross_kv", 0, "splitk2"),
    ("tiny", "cross_kv", 0, "rows4"),
    ("base", "dec_w2", 5, "rows1"),
    ("medium", "dec_qkv", 129, "rows1"),
    ("tiny.en", "vocab", 37, "splitk4"),
    ("test-tiny", "conv2", 2, "simt"),
    ("tiny", "dec_w1", 37, "simt"),
)

# every route of the exact-epilogue test (one-hot B: the accumulator is exact, the epilogue alone is compared)
EXACT_EPILOGUE_ROUTES = ("pair", "splitk2", "splitk4", "splitk8", "rows1", "rows2", "rows4", "rows8", "tile32", "tile64",
                         "tile128", "simt")
