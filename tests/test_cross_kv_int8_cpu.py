"""The 8-bit cross-KV mode's host side, without a GPU: the C flag and its Python constant agree, its test hooks stay out of
the drop-in boundary header, and the backend's compute_type names map to the right engine compute."""
import os
import re

import pytest

from b200_whisper import _lib as L
from b200_whisper import backend as B
from b200_whisper.vocab import vocab_for

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDARY = os.path.join(ROOT, "include", "b200_whisper.h")
HOOKS = os.path.join(ROOT, "include", "b200_whisper_hooks.h")


def _defines(path):
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+(BW_FLAG_\w+)\s+(\d+)", open(path).read())}


def test_flag_values_match_the_header():
    flags = _defines(BOUNDARY)
    assert flags["BW_FLAG_CROSS_KV_INT8"] == L.BW_FLAG_CROSS_KV_INT8 == 4
    for name, value in flags.items():
        assert getattr(L, name) == value, name
    assert len(set(flags.values())) == len(flags), "two flags share a bit"
    assert all(v & (v - 1) == 0 for v in flags.values()), "a flag is not a single bit"


def test_int8_hooks_are_declared_only_in_the_hooks_header():
    def declared(path):
        src = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
        return set(re.findall(r"\b(bw_[a-z0-9_]+)\s*\(", src))

    new = {"bw_test_quantize_cross_kv", "bw_test_dec_cross_attention_int8"}
    assert new <= declared(HOOKS)
    assert not new & declared(BOUNDARY)
    assert new <= set(L.SIGNATURES)


@pytest.mark.parametrize("compute_type,compute", [
    ("bfloat16_int8kv", "bf16_int8kv"), ("bf16_int8kv", "bf16_int8kv"), ("BF16_INT8KV", "bf16_int8kv"),
    ("int8", "bf16"), ("int8_float16", "bf16"), ("int8_bfloat16", "bf16"), ("bfloat16", "bf16"), ("default", "bf16"),
    ("float32", "fp32"),
])
def test_compute_type_mapping(monkeypatch, compute_type, compute):
    """bfloat16_int8kv / bf16_int8kv get their own engine compute (and so their own engine: get_engine keys on it); the
    reference's int8* names keep running as plain bfloat16"""
    seen = []

    class FakeEngine:
        vocab = vocab_for(51865)

    def fake_get_engine(model_size, device_index, c, **kw):
        seen.append(c)
        return FakeEngine()

    monkeypatch.setattr(B, "get_engine", fake_get_engine)
    b = B.B200WhisperBackend("random:test-tiny", "cuda:0", compute_type)
    assert b.compute == compute and seen == [compute]

