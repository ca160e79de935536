"""Which GEMM kernel the bf16 dispatcher (gemm_tc_bf16 -> gemm_tc_choose, csrc/gemm_tc.cu) picks for every GEMM call site
of the engine, without a GPU: the call sites' argument forms (tests/_gemm_sites.py, citing csrc/engine.cu) go through the
host-only bw_test_gemm_route.  A change to the dispatch heuristics shows up here as a table diff, and the GPU layout test
(tests/test_gpu_gemm_layouts.py) must keep checking every (call site, route) pair the table contains."""
import pytest

from tests import _gemm_sites as G

# call site -> route per batch: encoder sites per sub-batch of Z = 1 ... 8 windows, cross_kv one launch (Z = n_text_layer),
# decoder sites per R = 1, 5, 37, 128, 129, 320, 640 rows (the vocabulary projection on R logit rows).
# The dec_* rows are linear_rows of the unfused decoder step (B200W_NO_LN_FUSION); the default bf16 step runs those
# GEMMs through gemm_tc_rows instead.  The vocabulary projection goes through the dispatcher in both.
EXPECTED = {
    "test-tiny": {
        "conv1": "rows2 rows2 rows2 splitk2 splitk2 tile128 tile128 tile128",
        "conv2": "rows2 rows2 rows2 rows2 rows2 rows2 splitk2 splitk2",
        "enc_qkv": "tile128 tile128 tile128 tile128 pair pair pair pair",
        "enc_wo": "tile128 tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "enc_w1": "tile128 tile128 tile128 tile128 pair pair pair pair",
        "enc_w2": "rows4 rows4 rows4 rows2 rows2 rows2 splitk4 splitk4",
        "cross_kv": "tile128",
        "dec_qkv": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_wo": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_q_x": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_wo_x": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_w1": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_w2": "rows4 rows4 rows4 rows4 rows4 rows4 rows4",
        "vocab": "tile32 tile32 tile64 tile128 tile128 tile128 tile128",
    },
    "test-v3": {
        "conv1": "rows2 rows2 rows2 splitk2 splitk2 tile128 tile128 tile128",
        "conv2": "rows2 rows2 rows2 rows2 rows2 rows2 splitk2 splitk2",
        "enc_qkv": "tile128 tile128 tile128 tile128 pair pair pair pair",
        "enc_wo": "tile128 tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "enc_w1": "tile128 tile128 tile128 tile128 pair pair pair pair",
        "enc_w2": "rows4 rows4 rows4 rows2 rows2 rows2 splitk4 splitk4",
        "cross_kv": "tile128",
        "dec_qkv": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_wo": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_q_x": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_wo_x": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_w1": "tile128 tile128 tile128 tile128 tile128 tile128 tile128",
        "dec_w2": "rows4 rows4 rows4 rows4 rows4 rows4 rows4",
        "vocab": "tile32 tile32 tile64 tile128 tile128 tile128 tile128",
    },
    "tiny.en": {
        "conv1": "rows2 tile128 pair pair pair pair pair pair",
        "conv2": "rows4 rows2 splitk4 tile128 pair pair pair pair",
        "enc_qkv": "splitk2 pair pair pair pair pair pair pair",
        "enc_wo": "rows2 rows2 splitk2 tile128 pair pair pair pair",
        "enc_w1": "tile128 pair pair pair pair pair pair pair",
        "enc_w2": "rows4 rows2 splitk4 tile128 pair pair pair pair",
        "cross_kv": "pair",
        "dec_qkv": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_wo": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_q_x": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_wo_x": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_w1": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_w2": "rows8 rows8 rows8 rows8 rows8 rows8 rows8",
        "vocab": "tile32 tile32 tile64 tile128 tile128 tile128 tile128",
    },
    "tiny": {
        "conv1": "rows2 tile128 pair pair pair pair pair pair",
        "conv2": "rows4 rows2 splitk4 tile128 pair pair pair pair",
        "enc_qkv": "splitk2 pair pair pair pair pair pair pair",
        "enc_wo": "rows2 rows2 splitk2 tile128 pair pair pair pair",
        "enc_w1": "tile128 pair pair pair pair pair pair pair",
        "enc_w2": "rows4 rows2 splitk4 tile128 pair pair pair pair",
        "cross_kv": "pair",
        "dec_qkv": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_wo": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_q_x": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_wo_x": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_w1": "rows2 rows2 rows2 rows2 rows2 rows2 rows2",
        "dec_w2": "rows8 rows8 rows8 rows8 rows8 rows8 rows8",
        "vocab": "tile32 tile32 tile64 tile128 tile128 tile128 tile128",
    },
    "base": {
        "conv1": "splitk2 tile128 pair pair pair pair pair pair",
        "conv2": "rows2 splitk4 tile128 tile128 pair pair pair pair",
        "enc_qkv": "tile128 pair pair pair pair pair pair pair",
        "enc_wo": "rows2 splitk4 tile128 tile128 pair pair pair pair",
        "enc_w1": "tile128 pair pair pair pair pair pair pair",
        "enc_w2": "rows2 splitk4 tile128 tile128 pair pair pair pair",
        "cross_kv": "pair",
        "dec_qkv": "rows4 rows4 rows4 rows4 rows4 rows4 rows2",
        "dec_wo": "rows4 rows4 rows4 rows4 rows4 rows4 rows4",
        "dec_q_x": "rows4 rows4 rows4 rows4 rows4 rows4 rows4",
        "dec_wo_x": "rows4 rows4 rows4 rows4 rows4 rows4 rows4",
        "dec_w1": "rows4 rows4 rows4 rows4 rows4 rows2 splitk4",
        "dec_w2": "rows8 rows8 rows8 rows8 rows8 rows8 rows4",
        "vocab": "tile32 tile32 tile64 tile128 tile128 tile128 tile128",
    },
    "small": {
        "conv1": "tile128 pair pair pair pair pair pair pair",
        "conv2": "rows2 tile128 tile128 pair pair pair pair pair",
        "enc_qkv": "tile128 pair pair pair pair pair pair pair",
        "enc_wo": "rows2 tile128 tile128 pair pair pair pair pair",
        "enc_w1": "pair pair pair pair pair pair pair pair",
        "enc_w2": "rows2 tile128 tile128 pair pair pair pair pair",
        "cross_kv": "pair",
        "dec_qkv": "rows4 rows4 rows4 rows4 rows4 rows2 splitk4",
        "dec_wo": "rows4 rows4 rows4 rows4 rows4 rows4 rows4",
        "dec_q_x": "rows4 rows4 rows4 rows4 rows4 rows4 rows4",
        "dec_wo_x": "rows4 rows4 rows4 rows4 rows4 rows4 rows4",
        "dec_w1": "rows4 rows4 rows4 rows4 rows2 rows2 tile128",
        "dec_w2": "rows8 rows8 rows8 rows8 rows8 rows4 rows4",
        "vocab": "tile32 tile32 tile64 tile128 tile128 tile128 tile128",
    },
    "medium": {
        "conv1": "tile128 pair pair pair pair pair pair pair",
        "conv2": "splitk4 tile128 pair pair pair pair pair pair",
        "enc_qkv": "pair pair pair pair pair pair pair pair",
        "enc_wo": "splitk4 tile128 pair pair pair pair pair pair",
        "enc_w1": "pair pair pair pair pair pair pair pair",
        "enc_w2": "splitk4 tile128 pair pair pair pair pair pair",
        "cross_kv": "pair",
        "dec_qkv": "rows4 rows4 rows4 rows4 rows2 rows2 tile128",
        "dec_wo": "rows8 rows8 rows8 rows8 rows8 rows4 rows2",
        "dec_q_x": "rows8 rows8 rows8 rows8 rows8 rows4 rows2",
        "dec_wo_x": "rows8 rows8 rows8 rows8 rows8 rows4 rows2",
        "dec_w1": "rows4 rows4 rows4 rows4 rows2 splitk4 tile128",
        "dec_w2": "rows8 rows8 rows8 rows8 rows8 rows4 rows2",
        "vocab": "tile32 tile32 tile64 tile128 tile128 tile128 tile128",
    },
    "large-v3": {
        "conv1": "pair pair pair pair pair pair pair pair",
        "conv2": "tile128 pair pair pair pair pair pair pair",
        "enc_qkv": "pair pair pair pair pair pair pair pair",
        "enc_wo": "tile128 pair pair pair pair pair pair pair",
        "enc_w1": "pair pair pair pair pair pair pair pair",
        "enc_w2": "tile128 pair pair pair pair pair pair pair",
        "cross_kv": "pair",
        "dec_qkv": "rows4 rows4 rows4 rows4 rows2 splitk4 tile128",
        "dec_wo": "rows8 rows8 rows8 rows8 rows4 rows4 rows2",
        "dec_q_x": "rows8 rows8 rows8 rows8 rows4 rows4 rows2",
        "dec_wo_x": "rows8 rows8 rows8 rows8 rows4 rows4 rows2",
        "dec_w1": "rows2 rows2 rows2 rows2 splitk8 tile128 pair",
        "dec_w2": "rows8 rows8 rows8 rows8 rows4 rows4 rows2",
        "vocab": "tile32 tile32 tile64 tile128 tile128 tile128 tile128",
    },
}


def test_encoder_sub_batches_span_one_to_eight_windows():
    assert G.ENCODER_Z == tuple(range(1, 9))
    for nb in range(1, 17):
        assert sum(G.encoder_sub_batches(nb)) == nb


@pytest.mark.parametrize("model", G.MODELS)
def test_dispatcher_routes_of_engine_call_sites(model):
    got = {s: " ".join(G.dispatcher_route(G.site_form(model, s, b)) for b in G.site_batches(s)) for s in G.SITES}
    diff = {s: (got[s], EXPECTED[model][s]) for s in G.SITES if got[s] != EXPECTED[model][s]}
    assert not diff, f"{model}: dispatcher routes changed (got, expected): {diff}"


def production_pairs():
    """{(site, route)} over every row of the table"""
    return {(s, r) for m in G.MODELS for s in G.SITES for r in EXPECTED[m][s].split()}


def test_gpu_cases_claim_the_dispatcher_route():
    for model, site, batch, route in G.GPU_DISPATCH_CASES:
        assert G.dispatcher_route(G.site_form(model, site, batch)) == route, (model, site, batch, route)


def test_gpu_cases_cover_every_production_route():
    covered = {(site, route) for _, site, _, route in G.GPU_DISPATCH_CASES}
    assert covered == production_pairs(), (sorted(production_pairs() - covered), sorted(covered - production_pairs()))


def test_routes_production_never_reaches():
    """The forced routes of the GPU layout test that no production row takes: the unsplit row kernel (only gemm_tc_rows,
    the LayerNorm-fused decoder GEMMs, launches it) and the SIMT kernel (fp32 validation mode / BW_FLAG_FORCE_SIMT_GEMM)."""
    reached = {r for _, r in production_pairs()}
    claimed = {route for *_, route in G.GPU_FORCED_CASES} | set(G.EXACT_EPILOGUE_ROUTES)
    assert reached <= claimed
    assert claimed - reached == {"rows1", "simt"}, sorted(claimed - reached)


def test_forced_routes_check_preconditions():
    import ctypes as C

    from b200_whisper import _lib as L

    lib = L.load()
    # the vocabulary projection is swap-AB (transposed): neither the pair nor the row kernel has that epilogue
    form = G.site_form("tiny", "vocab", 5)
    assert G.dispatcher_route(form) == "tile32"
    for bad in ("pair", "rows2", "splitk16", "tile256"):
        taken = C.c_int32(-1)
        st = lib.bw_test_gemm(C.byref(G.desc_of(form)), 0, G.route_code(bad), C.byref(taken), None)
        assert st != 0 and taken.value == -1, bad
    # split-K needs KS blocks of 64 along K: K = 240 has 4
    form = G.site_form("test-tiny", "conv1", 1)
    taken = C.c_int32(-1)
    assert lib.bw_test_gemm(C.byref(G.desc_of(form)), 0, G.route_code("splitk8"), C.byref(taken), None) != 0
    assert lib.bw_test_gemm(C.byref(G.desc_of(form)), 1, G.route_code("pair"), C.byref(taken), None) != 0
    assert taken.value == -1
