"""Detect-mode decodes (bw_call_decode_detect / bw_decode_many_detect): the window's own <|sot|> row picks the language on
the device, so language detection and the decode share one admission, one encoder pass and one cross-KV write.  The
result must be the one the two-call path (detect_language(0), then decode with that language's sot sequence) gives."""
import itertools
import time

import numpy as np
import pytest

from tests._util import REALTIME, model_spec, oracle_model

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

torch = pytest.importorskip("torch")

from b200_whisper import _lib as L  # noqa: E402
from b200_whisper.backend import B200WhisperBackend  # noqa: E402
from b200_whisper.synth import synth_audio  # noqa: E402
from oracle import whisper_oracle as wo  # noqa: E402
from oracle.tables import LANGUAGES  # noqa: E402

P = L.LANGUAGE_PLACEHOLDER
SAMPLE_LEN = 48  # both paths are cut at the same length; long enough for beams to finish and reorder
MODES = {
    "greedy": dict(beam_size=None, patience=None),
    "beam5": dict(beam_size=5, patience=1.0),
    "best_of3_t0.5": dict(beam_size=None, patience=None, temperature=0.5, best_of=3, seed=0x1234ABCD5678),
}


def backend(name, compute="float32"):
    return B200WhisperBackend(model_spec(name), "cuda:0", compute, max_segments=16, max_sequences=48)


def kwargs(mode, no_ts):
    return dict(MODES[mode], length_penalty=None, sample_len=SAMPLE_LEN, without_timestamps=no_ts)


def sequences(v, lang_tok, no_ts):
    """(two-call initial tokens with the detected language, detect-mode initial tokens)"""
    tail = [v.transcribe] + ([v.no_timestamps] if no_ts else [])
    return [v.sot, lang_tok] + tail, [v.sot, P] + tail


def bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


CASES = [(name, seconds) for name in ("test-tiny", "test-v3", "base") for seconds in (3.0, 10.0, 30.0, 45.0)]


@pytest.mark.parametrize("name,seconds", CASES)
def test_fp32_detect_mode_equals_two_call_path(name, seconds):
    """fp32 validation mode: language token and probabilities bit for bit, and the decode's tokens / log-probabilities /
    no_speech_prob exactly, for greedy, beam 5 and best_of sampling, with and without <|notimestamps|>"""
    b = backend(name)
    v = b.vocab
    with b.engine.open_call(synth_audio(int(seconds * 7) + 1, seconds)) as call:
        tok, probs = call.detect_language(0)
        for mode in MODES:
            for no_ts in (False, True):
                two_call, detect = sequences(v, tok, no_ts)
                want = call.decode(0, two_call, 0, **kwargs(mode, no_ts))
                got = call.decode_detect(0, detect, 0, **kwargs(mode, no_ts))
                where = f"{name} {seconds}s {mode} no_ts={no_ts}"
                assert got["language_token"] == tok, where
                np.testing.assert_array_equal(bits(got["language_probs"]), bits(probs), err_msg=where)
                assert got["tokens"] == want["tokens"], where
                for k in ("sum_logprob", "avg_logprob", "no_speech_prob"):
                    assert bits(got[k]) == bits(want[k]), (where, k, got[k], want[k])


@pytest.mark.parametrize("name", ["test-tiny", "test-v3"])
@pytest.mark.parametrize("seconds", [30.0, 45.0])
def test_fp32_detect_mode_matches_oracle(name, seconds):
    """at >= 30 s the decode window is upstream's detection window: the detected language and the fp32 token stream equal
    the oracle's detect_language followed by its decode of that window"""
    b = backend(name)
    v = b.vocab
    model = oracle_model(name)
    audio = synth_audio(int(seconds * 3) + 5, seconds)
    mel = wo.log_mel_spectrogram(audio, model.dims.n_mels, padding=480000)
    window = wo.pad_or_trim(mel, 3000)
    want_tok, _ = wo.detect_language(model, window)
    want_lang = LANGUAGES[want_tok - model.layout.sot - 1]
    for mode, opts in (("greedy", {}), ("beam5", dict(beam_size=5, patience=1.0))):
        ref = wo.decode_window(model, window, wo.DecodingOptions(language=want_lang, sample_len=SAMPLE_LEN, **opts))
        assert ref.min_margin > 2e-4, f"oracle margin {ref.min_margin} too small for an exactness claim; pick another seed"
        with b.engine.open_call(audio) as call:
            got = call.decode_detect(0, [v.sot, P, v.transcribe], 0, **kwargs(mode, False))
        assert got["language_token"] == want_tok, (name, seconds, mode)
        assert got["tokens"] == ref.tokens, (name, seconds, mode)


@pytest.mark.parametrize("name,seconds", CASES)
def test_bf16_detect_mode_matches_two_call_path(name, seconds):
    """bf16: the same language token, the same token stream; avg_logprob within the batch-composition envelope of
    test_gpu_bf16_decode (the prefill's rows are split differently over two steps: fp32 summation order only)"""
    b = backend(name, "bfloat16")
    v = b.vocab
    with b.engine.open_call(synth_audio(int(seconds * 7) + 1, seconds)) as call:
        tok, _ = call.detect_language(0)
        for mode in MODES:
            for no_ts in (False, True):
                two_call, detect = sequences(v, tok, no_ts)
                want = call.decode(0, two_call, 0, **kwargs(mode, no_ts))
                got = call.decode_detect(0, detect, 0, **kwargs(mode, no_ts))
                where = f"{name} {seconds}s {mode} no_ts={no_ts}"
                assert got["language_token"] == tok, where
                assert got["tokens"] == want["tokens"], where
                assert abs(got["avg_logprob"] - want["avg_logprob"]) <= 8e-3, where


def _mixed_batch(b, calls):
    """16 windows over several calls and seeks, detect and normal requests alternating"""
    v = b.vocab
    items = []
    for i in range(16):
        call = calls[i % len(calls)]
        seek = [0, 1000, 3000][i % 3] if call.content_frames > 3000 else 0
        mode = list(MODES)[i % 3]
        no_ts = bool(i // 3 % 2)
        if i % 2 == 0:
            items.append((call, seek, dict(kwargs(mode, no_ts), initial=sequences(v, 0, no_ts)[1], sot_index=0, detect=True)))
        else:
            lang = v.language_token(["en", "de", "ko"][i % 3])
            items.append((call, seek, dict(kwargs(mode, no_ts), initial=sequences(v, lang, no_ts)[0], sot_index=0)))
    return items


def _alone(call, seek, kw):
    kw = dict(kw)
    return call.decode_detect(seek, **kw) if kw.pop("detect", False) else call.decode(seek, **kw)


def _same(got, want, where):
    assert got["tokens"] == want["tokens"], where
    # sharing a step may change the cross-attention T-split of a launch: fp32 summation order only
    assert abs(got["avg_logprob"] - want["avg_logprob"]) <= 1e-4, where
    if "language_token" in want:
        assert got["language_token"] == want["language_token"], where
        np.testing.assert_allclose(got["language_probs"], want["language_probs"], rtol=1e-4, atol=1e-6, err_msg=where)
    else:
        assert "language_token" not in got, where


def test_decode_many_detect_mixed_batch_equals_windows_alone():
    b = backend("test-tiny")
    calls = [b.engine.open_call(synth_audio(70 + i, s)) for i, s in enumerate((3.0, 12.0, 45.0, 61.0))]
    try:
        items = _mixed_batch(b, calls)
        s0 = b.engine.stats()
        outs = b.engine.decode_many(items)
        s1 = b.engine.stats()
        # one bw_decode_many of 16 alternating windows, max_encoder_batch 8: two encoder batches of 4 detect + 4 normal
        assert s1["windows"] - s0["windows"] == 16 and s1["encoder_batches"] - s0["encoder_batches"] == 2
        for i, (it, got) in enumerate(zip(items, outs)):
            assert not isinstance(got, BaseException), got
            _same(got, _alone(*it), f"window {i}")
    finally:
        for c in calls:
            c.close()


def test_detect_windows_admitted_while_others_decode():
    """detect windows admitted in later steps while other requests are mid-decode: their sot step and prefill step run
    next to the sampling rows of requests admitted earlier"""
    import threading

    b = backend("test-tiny")
    v = b.vocab
    calls = [b.engine.open_call(synth_audio(90 + i, 8.0 + i)) for i in range(6)]
    try:
        long_kw = dict(kwargs("greedy", False), sample_len=224)
        running = [(calls[i], 0, dict(long_kw, initial=[v.sot, v.language_token("en"), v.transcribe], sot_index=0))
                   for i in range(3)]
        joining = [(calls[3 + i], 0, dict(kwargs(list(MODES)[i], i == 1), sample_len=16, initial=sequences(v, 0, i == 1)[1],
                                          sot_index=0, detect=True)) for i in range(3)]
        alone = [_alone(*it) for it in running + joining]
        out = {}
        s0 = b.engine.stats()
        th = threading.Thread(target=lambda: out.update(running=b.engine.decode_many(running)))
        th.start()
        deadline = time.time() + 60
        while b.engine.stats()["decode_steps"] - s0["decode_steps"] < 4 and time.time() < deadline:
            time.sleep(0.001)
        assert th.is_alive(), "the long decodes ended before the detect windows could join; nothing was checked"
        s1 = b.engine.stats()
        out["joining"] = b.engine.decode_many(joining)
        joined_mid_decode = th.is_alive()  # the detect windows were admitted, decoded and finished next to them
        th.join()
        s2 = b.engine.stats()
        assert joined_mid_decode, (s1, s2)
        assert s1["encoder_batches"] - s0["encoder_batches"] == 1 and s2["encoder_batches"] - s1["encoder_batches"] == 1
        for i, (got, want) in enumerate(zip(out["running"] + out["joining"], alone)):
            _same(got, want, f"window {i}")
    finally:
        for c in calls:
            c.close()


def test_detect_mode_on_sequence_slots_of_earlier_decodes():
    """Detect-mode decodes on sequence slots whose previous occupants were beam / best_of decodes of another initial length,
    at first_seq 0 and behind a single-hypothesis request: every hypothesis descends from the fresh prefix, not from the
    ancestry those slots held (a detect-mode decode's first beam update reads the ancestry buffer its admission step did
    not make current)"""
    b = B200WhisperBackend(model_spec("test-tiny", seed=1), "cuda:0", "float32", max_segments=4, max_sequences=16)
    v = b.vocab
    en = v.language_token("en")
    calls = [b.engine.open_call(synth_audio(500 + i, 6.0 + 3 * i)) for i in range(3)]
    try:
        def earlier():  # beam 5, beam 5 and best_of 3 over slots 0..12, three initial tokens: ancestry set past position 2
            b.engine.decode_many([(calls[i], 0, dict(kwargs(m, False), initial=[v.sot, en, v.transcribe], sot_index=0))
                                  for i, m in enumerate(("beam5", "beam5", "best_of3_t0.5"))])

        def detect_item(call, mode):
            return (call, 0, dict(kwargs(mode, True), initial=sequences(v, 0, True)[1], sot_index=0, detect=True))

        def two_call(item):
            call, seek, kw = item
            tok, _ = call.detect_language(seek)
            kw = {k: x for k, x in kw.items() if k not in ("detect", "initial")}
            return call.decode(seek, sequences(v, tok, True)[0], **kw)

        for layout in ("first_seq 0", "behind a single hypothesis"):
            earlier()
            items = [detect_item(calls[0], "beam5"), detect_item(calls[1], "best_of3_t0.5")]
            if layout != "first_seq 0":
                items = [(calls[2], 0, dict(kwargs("greedy", False), initial=[v.sot, en, v.transcribe], sot_index=0))] + items
            outs = b.engine.decode_many(items)
            for it, got in zip(items, outs):
                want = two_call(it) if it[2].get("detect") else _alone(*it)
                where = f"{layout}: {it[2].get('beam_size')} {it[2].get('best_of')}"
                assert got["tokens"] == want["tokens"], where
                assert abs(got["avg_logprob"] - want["avg_logprob"]) <= 1e-4, where
    finally:
        for c in calls:
            c.close()


def test_backend_admits_one_window_per_decoded_window():
    """language=None through the backend: the first window detects its own language -- one admitted window per window
    decoded, not two; transcribe_many over 8 calls admits 8 windows for the first seek"""
    b = backend("test-tiny", "bfloat16")
    opts = dict(REALTIME)  # one temperature rung: one decode per window
    s0 = b.engine.stats()
    segs, info = b.transcribe(synth_audio(5, 3.0), opts)
    s1 = b.engine.stats()
    assert s1["windows"] - s0["windows"] == 1 and s1["encoder_batches"] - s0["encoder_batches"] == 1
    assert info.language and b.last_language_probability is not None
    b.transcribe_many([synth_audio(200 + i, 3.0) for i in range(8)], opts)
    s2 = b.engine.stats()
    assert s2["windows"] - s1["windows"] == 8


def test_detect_mode_refusals():
    b = backend("test-tiny")
    v = b.vocab
    with b.engine.open_call(synth_audio(1, 3.0)) as call:
        for initial, sot_index, msg in (
                ([v.sot_prev, 100, v.sot, P, v.transcribe], 2, "no prompt"),  # a prompt in front of <|sot|>
                ([v.sot, v.language_token("en"), P], 0, "placeholder"),        # placeholder misplaced
                ([v.sot, P, v.transcribe, P], 0, "placeholder"),               # a stray -1
                ([v.sot, v.language_token("en"), v.transcribe], 0, "placeholder")):  # no placeholder
            with pytest.raises(L.B200WhisperError, match=rf"bw_status -1\).*{msg}"):
                call.decode_detect(0, initial, sot_index, None, None, None)
        with pytest.raises(L.B200WhisperError, match=r"bw_status -1\).*placeholder"):  # the batched entry point checks alike
            b.engine.decode_many([(call, 0, dict(initial=[v.sot, P, v.transcribe, P], sot_index=0, beam_size=None, patience=None,
                                                 length_penalty=None, detect=True))])
        with pytest.raises(L.B200WhisperError, match=r"bw_status -1\).*token id out of range"):  # plain decode: -1 stays invalid
            call.decode(0, [v.sot, P, v.transcribe], 0, None, None, None)
    en = backend("test-tiny.en")
    with en.engine.open_call(synth_audio(1, 3.0)) as call:
        with pytest.raises(L.B200WhisperError, match=r"bw_status -1\).*no language tokens"):
            call.decode_detect(0, [en.vocab.sot, P], 0, None, None, None)


@pytest.mark.parametrize("compute", ["float32", "bfloat16"])
def test_backend_language_none_matches_two_call_path(compute, monkeypatch):
    """transcribe / transcribe_many with language None give the segments and BackendInfo of the two-call path"""
    b = backend("test-tiny", compute)
    audios = [synth_audio(300 + i, s) for i, s in enumerate((2.0, 7.5, 33.0))]
    opts = dict(REALTIME, temperature=(0.0, 0.4), beam_size=2)

    def run():  # the same per-call sampling seeds on both paths (a backend derives them from its call count)
        b._call_counter = itertools.count()
        single = [b.transcribe_raw(a, **b._normalize_options(opts)) for a in audios]
        return single, b.transcribe_many(audios, opts)

    got, got_many = run()
    monkeypatch.setattr(b, "detect_in_decode", False)  # the separate detect_language pass
    want, want_many = run()
    for g, w in zip(got, want):
        assert g["language"] == w["language"] and g["language_probability"] == pytest.approx(w["language_probability"], rel=1e-4)
        assert [s["tokens"] for s in g["segments"]] == [s["tokens"] for s in w["segments"]]
        assert [(s["start"], s["end"], s["text"]) for s in g["segments"]] == [(s["start"], s["end"], s["text"]) for s in w["segments"]]
    assert got_many == want_many


def test_reference_model_worker_language_none(monkeypatch):
    """the reference's own ModelWorker (where its source is found) with language None on a multilingual random model"""
    import sys

    from tests.test_reference_worker_integration import LAYOUT, PKG_ROOT, _pcm

    if LAYOUT is None:
        pytest.skip("needs the upstream server source (stt_server): set STT_SERVER_ROOT or run tools/install_reference.sh")
    monkeypatch.syspath_prepend(PKG_ROOT)
    for name in [n for n in sys.modules if n == "stt_server" or n.startswith("stt_server.")]:
        monkeypatch.delitem(sys.modules, name)
    from b200_whisper import register

    register.install()
    import stt_server.model.worker as worker

    w = worker.ModelWorker(model_spec("test-tiny"), "cuda:0", "float32", None, False, base_options={"task": "transcribe"},
                           backend="b200_whisper")
    pcm = _pcm(11, 6.0)
    r = w.decode_sync(pcm, 16000, dict(REALTIME), time.perf_counter())
    audio = np.frombuffer(pcm, np.int16).astype(np.float32) / 32768.0
    eng = w.backend.engine
    with eng.open_call(audio) as call:
        tok, _ = call.detect_language(0)
    lang = w.backend.vocab.language_of_token(tok)
    want = w.backend.transcribe(audio, dict(REALTIME, language=lang, task="transcribe"))
    assert r.language_code == lang == want[1].language
    assert [(s.start, s.end, s.text) for s in r.segments] == [(s.start, s.end, s.text) for s in want[0]]
    w.close()
    for name in [n for n in sys.modules if n == "stt_server" or n.startswith("stt_server.")]:
        sys.modules.pop(name, None)
