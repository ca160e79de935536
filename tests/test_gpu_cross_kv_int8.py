"""The 8-bit cross-KV mode (BW_FLAG_CROSS_KV_INT8, compute_type bfloat16_int8kv) on the GPU:

* the quantizer (bw_test_quantize_cross_kv): |code| <= 127, scale = fp32 amax / 127, every element within half a scale of
  code * scale, no NaN -- on random rows and on all-zero slices, single non-zero elements, +-bf16 max and denormals;
* `dec_cross_attention_int8_kernel` (+ the unchanged T-split combine) against fp32 torch on the DEQUANTIZED cache, on every
  case of the bf16 kernel's tests (tests/test_gpu_decoder_kernels.py) with the same bounds; the error against the
  unquantized bf16 K/V is reported;
* teacher-forced cached decode through the real scheduler against the fp32 oracle, with the product mode's bars
  (tests/test_gpu_bf16_decode.py);
* determinism and batch invariance of the decoded tokens; the flag's refusals; the bench hooks in the mode.
"""
import numpy as np
import pytest

from tests._util import ACCURATE, REALTIME, model_spec, oracle_model
from tests.test_gpu_bf16_decode import _forced_batch, _logit_stats, _oracle_window, _report

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

torch = pytest.importorskip("torch")

from b200_whisper import _lib as L  # noqa: E402
from b200_whisper.backend import B200WhisperBackend, load_checkpoint  # noqa: E402
from b200_whisper.engine import Engine  # noqa: E402
from b200_whisper.synth import synth_audio  # noqa: E402

DEV = "cuda"
BF16_MAX = float(torch.finfo(torch.bfloat16).max)


def _rel(a, b):
    return ((a.float() - b.float()).norm() / (b.float().norm() + 1e-30)).item()


def _i32(x):
    return torch.tensor(x, dtype=torch.int32, device=DEV)


def _quantize(x):
    """bf16 [n, d] on the device -> (codes int8 [n, d], scales fp32 [n, d / 64]) through the engine's quantizer"""
    n, d = x.shape
    codes = torch.full((n, d), 99, dtype=torch.int8, device=DEV)
    scales = torch.full((n, d // 64), float("nan"), device=DEV)
    torch.cuda.synchronize()
    L.check(L.load().bw_test_quantize_cross_kv(x.data_ptr(), n, d, codes.data_ptr(), scales.data_ptr(), None), "bw_test_quantize_cross_kv")
    return codes, scales


# ------------------------------------------------------------------------------------------------------ quantizer
def test_quantizer_codes_scales_and_edge_cases():
    g = torch.Generator(device=DEV).manual_seed(3)
    n, d = 4096, 256
    mag = torch.pow(10.0, torch.empty((n, d // 64), device=DEV).uniform_(-6, 6, generator=g)).repeat_interleave(64, 1)
    x = torch.randn((n, d), device=DEV, generator=g) * mag
    edge = torch.zeros((8, d), device=DEV)
    edge[1, 5] = 0.75                                   # one non-zero element (slice 0); slices 1..3 of row 1 all zero
    edge[1, 64 + 63] = -3.0e-5
    edge[2, :64] = BF16_MAX                             # +-bf16 max
    edge[2, 64:128] = torch.linspace(-1.0, 1.0, 64, device=DEV) * BF16_MAX
    edge[3, :] = torch.randn(d, device=DEV, generator=g) * 1e-39   # bf16 denormals
    edge[4, :64] = 9.18355e-41                          # smallest bf16 denormal
    edge[4, 64:128] = torch.randn(64, device=DEV, generator=g) * 1e-39
    edge[4, 70] = 1.0                                   # denormals next to a normal element
    edge[5, :] = torch.arange(d, device=DEV, dtype=torch.float32) - 127.5   # ramps
    edge[6, :] = -edge[5]
    xb = torch.cat([x, edge]).bfloat16()
    codes, scales = _quantize(xb)
    torch.cuda.synchronize()
    xs = xb.float().reshape(-1, 64).double().cpu()
    c = codes.reshape(-1, 64).double().cpu()
    s = scales.reshape(-1).cpu()
    assert not torch.isnan(s).any() and torch.isfinite(s).all()
    assert (c.abs() <= 127).all()
    amax = xb.float().reshape(-1, 64).abs().amax(1).cpu()
    want = amax / 127.0                                  # fp32 division, correctly rounded
    lo, hi = torch.nextafter(want, torch.zeros_like(want)), torch.nextafter(want, torch.full_like(want, float("inf")))
    assert ((s >= lo) & (s <= hi)).all(), "scale is not fp32 amax / 127 to 1 ulp"
    err = (c * s.double()[:, None] - xs).abs()
    assert (err <= s.double()[:, None] / 2 * (1 + 1e-6)).all(), f"worst err / scale {(err / s.double()[:, None].clamp_min(1e-300)).max()}"
    zero = amax == 0
    assert zero.sum() >= 3 and (s[zero] == 0).all() and (c[zero] == 0).all()
    assert (c.abs().amax(1)[~zero] == 127).all(), "the largest element of a slice maps to +-127"


# ------------------------------------------------------------------------------------------------ cross attention
def _cross_case_int8(n_groups, nq, n_head, n_layer, layer, force_split, seed, ragged=False, T_enc=1500):
    """tests/test_gpu_decoder_kernels.py::_cross_case on the 8-bit cache: (out, reference on the dequantized cache,
    reference on the bf16 cache)"""
    lib = L.load()
    d = 64 * n_head
    g = torch.Generator(device=DEV).manual_seed(seed)
    n_slots = n_groups + 3
    cache = (torch.randn((n_slots, n_layer, T_enc, 2 * d), device=DEV, generator=g) * 1.5).bfloat16()
    codes, scales = _quantize(cache.reshape(-1, 2 * d))
    deq = (codes.float().reshape(-1, 2 * n_head, 64) * scales[:, :, None]).reshape(n_slots, n_layer, T_enc, 2 * d)
    sizes = [(1 + (i * 5 + 2) % nq) if ragged else nq for i in range(n_groups)]
    first = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int32)
    R = int(sum(sizes))
    perm = torch.randperm(n_slots, generator=torch.Generator().manual_seed(seed))[:n_groups].to(torch.int32)
    q = torch.randn((R, d), device=DEV, generator=g) * 2.0
    out = torch.full((R, d), float("nan"), device=DEV, dtype=torch.bfloat16)
    gf, gn, gx = _i32(first), _i32(sizes), perm.to(DEV)
    torch.cuda.synchronize()
    L.check(lib.bw_test_dec_cross_attention_int8(codes.data_ptr(), scales.data_ptr(), n_slots, n_layer, layer, T_enc, d, n_head,
                                                 q.data_ptr(), gf.data_ptr(), gn.data_ptr(), gx.data_ptr(), n_groups, max(sizes), R,
                                                 force_split, out.data_ptr(), None),
            "bw_test_dec_cross_attention_int8")
    torch.cuda.synchronize()

    def reference(kvc):
        ref = torch.empty((R, d), device=DEV)
        for gi in range(n_groups):
            kv = kvc[int(perm[gi]), layer].float()
            k = kv[:, :d].reshape(T_enc, n_head, 64).permute(1, 0, 2)
            v = kv[:, d:].reshape(T_enc, n_head, 64).permute(1, 0, 2)
            rows = slice(int(first[gi]), int(first[gi]) + sizes[gi])
            qq = q[rows].reshape(-1, n_head, 64).permute(1, 0, 2)
            w = torch.softmax(qq @ k.transpose(1, 2) / 8.0, dim=-1)
            ref[rows] = (w @ v).permute(1, 0, 2).reshape(-1, d)
        return ref

    assert torch.isfinite(out.float()).all(), "rows left unwritten"
    return out, reference(deq), reference(cache)


def _check(out, ref, ref_bf16, what):
    r = _rel(out, ref)
    per_row = ((out.float() - ref).norm(dim=1) / ref.norm(dim=1)).max().item()
    print(f"{what}: rel-L2 {r:.2e} (worst row {per_row:.2e}) vs dequantized, {_rel(out, ref_bf16):.2e} vs bf16 K/V")
    assert r < 1.5e-2, f"{what}: rel-L2 {r}"
    assert per_row < 4e-2, f"{what}: worst row {per_row}"


@pytest.mark.parametrize("nq", [1, 5, 8])
@pytest.mark.parametrize("n_groups", [1, 7, 128])
def test_int8_cross_attention_rows_and_segments(nq, n_groups):
    out, ref, ref16 = _cross_case_int8(n_groups, nq, n_head=6, n_layer=2, layer=1, force_split=0, seed=nq * 131 + n_groups)
    _check(out, ref, ref16, f"nq {nq} segments {n_groups}")


@pytest.mark.parametrize("ragged", [False, True])
def test_int8_cross_attention_ragged_groups(ragged):
    out, ref, ref16 = _cross_case_int8(9, 8, n_head=20, n_layer=2, layer=0, force_split=0, seed=77, ragged=ragged)
    _check(out, ref, ref16, f"ragged {ragged}")


@pytest.mark.parametrize("n_split", [1, 2, 3, 4, 5, 6, 7, 8])
def test_int8_cross_attention_every_split_count(n_split):
    out, ref, ref16 = _cross_case_int8(3, 5, n_head=20, n_layer=3, layer=2, force_split=n_split, seed=500 + n_split, ragged=True)
    _check(out, ref, ref16, f"{n_split} splits")
    base, _, _ = _cross_case_int8(3, 5, n_head=20, n_layer=3, layer=2, force_split=1, seed=500 + n_split, ragged=True)
    assert _rel(out, base) < 6e-3, "split partials do not recombine to the single-pass result"


def test_int8_cross_attention_short_encoder_context():
    for T_enc, split in ((100, 0), (65, 2), (1500 - 37, 8)):
        out, ref, ref16 = _cross_case_int8(4, 8, n_head=6, n_layer=1, layer=0, force_split=split, seed=T_enc, T_enc=T_enc)
        _check(out, ref, ref16, f"T_enc {T_enc}")


# -------------------------------------------------------------------------------------- decode through the engine
def _backend(name, **kw):
    return B200WhisperBackend(model_spec(name), "cuda:0", "bfloat16_int8kv", **kw)


def _teacher_forced_int8(name, n_sessions, sample_len=None, seed0=300, dur0=2.0, dstep=0.45, **engine_kw):
    model = oracle_model(name)
    b = _backend(name, **engine_kw)
    assert b.compute == "bf16_int8kv"
    audios = [synth_audio(seed0 + i, dur0 + dstep * i) for i in range(n_sessions)]
    initial, streams, refs = None, [], []
    for a in audios:
        kw = {} if sample_len is None else {"sample_len": sample_len}
        initial, stream, logits, _ = _oracle_window(model, a, beam_size=1, **kw)
        streams.append(stream)
        refs.append(logits)
    outs = _forced_batch(b, audios, initial, streams)
    worst, agree_all, in5_all = 0.0, [], []
    for i, (res, got) in enumerate(outs):
        assert res["n_steps"] == len(streams[i])
        rels, agree, in5 = _logit_stats(got, refs[i])
        assert np.isfinite(got).all()
        assert rels.max() <= 3e-2, f"{name} session {i}: step {int(rels.argmax())} logits rel-L2 {rels.max():.4f}"
        worst = max(worst, float(rels.max()))
        agree_all.append(agree)
        in5_all.append(in5)
    agree_all, in5_all = np.concatenate(agree_all), np.concatenate(in5_all)
    rep = {"model": name, "compute": "bf16_int8kv", "sessions": n_sessions, "steps_per_session": int(np.mean([len(s) for s in streams])),
           "worst_step_rel_l2": worst, "argmax_agreement": float(agree_all.mean()), "oracle_argmax_in_top5": float(in5_all.mean())}
    _report(f"r3_int8kv_teacher_forced_{name}.json", rep)
    assert in5_all.mean() >= 0.97 and agree_all.mean() >= 0.80, rep


@pytest.mark.parametrize("name,n_sessions", [("test-tiny", 20), ("test-v3", 16), ("tiny.en", 16)])
def test_int8kv_teacher_forced_cached_decode_matches_oracle_logits(name, n_sessions):
    _teacher_forced_int8(name, n_sessions, max_segments=24, max_sequences=48)


def test_int8kv_large_v3_teacher_forced_cached_decode():
    _teacher_forced_int8("large-v3", 3, sample_len=64, seed0=600, dur0=4.0, dstep=1.5, max_segments=8, max_sequences=16,
                         max_encoder_batch=4)


def test_int8kv_decode_is_deterministic_and_batch_invariant():
    import threading

    b = _backend("test-tiny", max_segments=24, max_sequences=48)
    opts = dict(REALTIME, language="en")
    audios = [synth_audio(400 + i, 2.5 + 0.6 * i) for i in range(16)]

    def options(i):
        return b._normalize_options(opts if i % 4 else dict(ACCURATE, language="en"))

    def run_batch():
        out = [None] * len(audios)

        def work(i):
            out[i] = b.transcribe_raw(audios[i], **options(i))

        th = [threading.Thread(target=work, args=(i,)) for i in range(len(audios))]
        [t.start() for t in th]
        [t.join() for t in th]
        return [[s["tokens"] for s in r["segments"]] for r in out]

    first, again = run_batch(), run_batch()
    alone = [[s["tokens"] for s in b.transcribe_raw(a, **options(i))["segments"]] for i, a in enumerate(audios)]
    assert all(len(t) > 0 for r in first for t in r)
    same, same_alone = sum(a == c for a, c in zip(first, again)), sum(a == c for a, c in zip(first, alone))
    _report("r3_int8kv_batch_invariance.json", {"sessions": len(audios), "identical_tokens_batch_vs_batch": same,
                                                "identical_tokens_batch_vs_alone": same_alone})
    # the same tolerance as the bf16 mode: a window may differ only where its top-1 / top-2 margin is at rounding level
    assert same >= len(audios) - 1 and same_alone >= len(audios) - 1, (same, same_alone)


# ----------------------------------------------------------------------------------------- flag handling, bench hooks
@pytest.mark.parametrize("compute,flags", [("fp32", 0), ("bf16", L.BW_FLAG_FORCE_SIMT_GEMM)])
def test_int8kv_flag_refused_without_bf16_tensor_core_path(compute, flags):
    dims, state, _ = load_checkpoint(model_spec("test-tiny"))
    with pytest.raises(L.B200WhisperError, match="BW_FLAG_CROSS_KV_INT8"):
        Engine(dims, state, compute=compute, flags=flags | L.BW_FLAG_CROSS_KV_INT8, max_segments=2)


def test_int8kv_bench_hooks_run_in_the_mode():
    b16 = B200WhisperBackend(model_spec("test-v3"), "cuda:0", "bfloat16", max_segments=8, max_sequences=16)
    b8 = _backend("test-v3", max_segments=8, max_sequences=16)
    assert b8.engine is not b16.engine
    e, d = b8.engine, b8.engine.dims
    ms, by = e.bench_cross_attention(8, 2, 4)
    _, by16 = b16.engine.bench_cross_attention(8, 2, 4)
    T, dm, H = d.n_audio_ctx, d.n_text_state, d.n_text_head
    assert ms > 0 and by == pytest.approx(8 * (2 * T * dm + 2 * T * H * 4) + 16 * dm * 4)
    assert by16 - by == pytest.approx(8 * (2 * T * dm * 2 - 2 * T * dm - 2 * T * H * 4))
    ms, by = e.bench_decoder_step(4, 2, 20, 4)
    assert ms > 0 and by > 0
    audios = [synth_audio(900 + i, 3.0 + i) for i in range(4)]
    assert e.bench_pipeline(audios, 1, 8) > 0
    res = e.bench_pipeline_results(4, 1, 8, None)
    assert len(res) == 4 and all(len(r["tokens"]) > 0 for r in res)
