"""Host side of detect-mode decodes without a GPU: when the backend's seek loop lets the first window detect its own
language, and the C-ABI declarations / ctypes bindings of the new entry points."""
import os
import re

import numpy as np
import pytest

import b200_whisper.backend as bk
from b200_whisper import _lib as L
from b200_whisper.backend import B200WhisperBackend
from b200_whisper.synth import synth_audio
from b200_whisper.vocab import vocab_for
from tests.test_host_logic import FakeCall, FakeEngine, res

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = L.LANGUAGE_PLACEHOLDER


class DetectCall(FakeCall):
    """FakeCall with detect mode: the window's decode returns the language it detected (always `ko` here)"""

    def decode_detect(self, seek, initial, sot_index, beam_size, patience, length_penalty, **kw):
        out = self.decode(seek, initial, sot_index, beam_size, patience, length_penalty, detect=True, **kw)
        v = self.engine.vocab
        probs = np.full(v.num_languages, 0.001, np.float32)
        probs[v.language_token("ko") - v.first_language_token] = 0.7
        return dict(out, language_token=v.language_token("ko"), language_probs=probs)

    def detect_language(self, seek=0):
        self.engine.separate_detections += 1
        return super().detect_language(seek)


class DetectEngine(FakeEngine):
    detects_in_decode = True

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.separate_detections = 0

    def open_call(self, audio, sample_rate=None):
        self.last_sample_rate = sample_rate
        return DetectCall(self, audio)

    def decode_many(self, items):
        self.batches = getattr(self, "batches", []) + [len(items)]
        out = []
        for call, seek, kw in items:
            kw = dict(kw)
            out.append(call.decode_detect(seek, **kw) if kw.pop("detect", False) else call.decode(seek, **kw))
        return out


@pytest.fixture
def detect_backend(monkeypatch):
    def make(script, n_vocab=51865):
        eng = DetectEngine(n_vocab, script)
        monkeypatch.setattr(bk, "get_engine", lambda *a, **k: eng)
        return B200WhisperBackend("random:test-tiny", "cuda:0", "bfloat16"), eng

    return make


def test_first_window_detects_when_language_unset(detect_backend):
    v = vocab_for(51865)
    tb = v.timestamp_begin
    # window 1 ends on a timestamp pair mid-window (seek moves to 5 s), so a second window follows
    b, eng = detect_backend([res([tb, 100, tb + 250, tb + 250, 200]), res([tb, 200, tb + 100])])
    segs, info = b.transcribe(synth_audio(1, 25.0), {"beam_size": 1, "temperature": 0.0})
    first, second = eng.all_decodes[0], eng.all_decodes[1]
    assert first["detect"] is True and first["initial"] == [v.sot, P, v.transcribe] and first["sot_index"] == 0
    i = second["sot_index"]  # (the second window is prompted with the first one's text)
    assert "detect" not in second and second["initial"][i:i + 3] == [v.sot, v.language_token("ko"), v.transcribe]
    assert eng.separate_detections == 0
    assert info.language == "ko" and abs(b.last_language_probability - 0.7) < 1e-6


def test_later_rungs_use_the_detected_language(detect_backend):
    v = vocab_for(51865)
    # the first rung fails the log-probability check, the second passes
    b, eng = detect_backend([res([100], avg=-3.0), res([101], avg=-0.2)])
    raw = b.transcribe_raw(synth_audio(2, 3.0), temperature=(0.0, 0.4), _without_timestamps=True)
    assert [d.get("detect", False) for d in eng.all_decodes] == [True, False]
    assert eng.all_decodes[0]["initial"] == [v.sot, P, v.transcribe, v.no_timestamps]
    assert eng.all_decodes[1]["initial"] == [v.sot, v.language_token("ko"), v.transcribe, v.no_timestamps]
    assert eng.all_decodes[1]["temperature"] == 0.4
    assert raw["language"] == "ko" and raw["segments"][0]["tokens"] == [101]


def test_transcribe_many_detects_in_the_batch(detect_backend):
    b, eng = detect_backend([res([100])])
    out = b.transcribe_many([synth_audio(i, 3.0) for i in range(4)], {"beam_size": 1})
    assert eng.batches == [4] and eng.separate_detections == 0
    assert all(d["detect"] for d in eng.all_decodes) and [i.language for _, i in out] == ["ko"] * 4


@pytest.mark.parametrize("options,n_vocab", [
    ({"language": "de"}, 51865),                 # explicit language
    ({}, 51864),                                 # .en vocabulary
    ({"initial_prompt": "hello"}, 51865),        # a prompt goes in front of <|sot|>: separate detection pass
])
def test_no_detect_mode(detect_backend, options, n_vocab):
    b, eng = detect_backend([res([100])], n_vocab)
    b.transcribe(synth_audio(3, 3.0), dict(options, beam_size=1))
    assert not any(d.get("detect") for d in eng.all_decodes) and P not in eng.all_decodes[0]["initial"]
    assert eng.separate_detections == (1 if "initial_prompt" in options else 0)


def test_detect_in_decode_off_or_not_supported(detect_backend, monkeypatch):
    """backend.detect_in_decode = False, or an engine without the capability: the separate detection pass as before"""
    v = vocab_for(51865)
    b, eng = detect_backend([res([100])])
    assert b.detect_in_decode
    b.detect_in_decode = False
    b.transcribe(synth_audio(3, 3.0), {"beam_size": 1})
    assert eng.separate_detections == 1 and "detect" not in eng.all_decodes[0]
    assert eng.all_decodes[0]["initial"] == [v.sot, v.language_token("ko"), v.transcribe]
    plain = FakeEngine(51865, [res([100])])
    monkeypatch.setattr(bk, "get_engine", lambda *a, **k: plain)
    assert not B200WhisperBackend("random:test-tiny", "cuda:0", "bfloat16").detect_in_decode


def test_audio_without_a_window_still_reports_its_language(detect_backend):
    """fewer than 160 samples: no window is decoded, so the language comes from the separate detection pass as before"""
    b, eng = detect_backend([res([])])
    raw = b.transcribe_raw(synth_audio(4, 0.005))
    assert eng.all_decodes == [] and eng.separate_detections == 1 and raw["language"] == "ko"


def test_entry_points_declared_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b200_whisper.h")).read(), flags=re.S)
    assert re.search(r"int bw_call_decode_detect\(bw_call\*, int32_t seek, const bw_decode_opts\* opts, bw_result\* out, "
                     r"bw_lang_result\* lang\);", src)
    assert re.search(r"int bw_decode_many_detect\(bw_call\* const\* calls, const int32_t\* seeks, const bw_decode_opts\* opts, "
                     r"bw_result\* results,\s+bw_lang_result\* langs, int32_t\* statuses, int32_t n\);", src)
    lib = L.load()
    for name, n_args in (("bw_call_decode_detect", 5), ("bw_decode_many_detect", 7)):
        assert len(L.SIGNATURES[name][1]) == n_args
        assert getattr(lib, name).argtypes == L.SIGNATURES[name][1]
    assert L.LANGUAGE_PLACEHOLDER == -1
