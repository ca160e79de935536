"""The drop-in claim on a GPU with the REAL engine: the reference's own callers -- `ModelWorker.decode_sync`
(stt_server/model/worker.py:83-146), `ModelRegistry.submit_decode` / `_dispatch_loop` / `_worker_loop`
(stt_server/backend/application/model_registry.py:385-680) and the whole unmodified server over gRPC (CreateSession +
StreamingRecognize) under its own load generator tools/bench/grpc_load_test.py -- drive `B200WhisperBackend` on cuda:0.

The upstream server and its load generator are not part of this repository: these tests run where a checkout is found
($STT_SERVER_ROOT, or the unmodified install tools/install_reference.sh makes under the git-ignored baseline/_ref) and
skip elsewhere."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest

from tests._util import ACCURATE, REALTIME

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1200)]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from wire_bench import reference_layout  # noqa: E402

LAYOUT = reference_layout()
if LAYOUT is None:
    pytest.skip("needs the upstream server source (stt_server, tools/bench/grpc_load_test.py), which is not part of this "
                "repository: set STT_SERVER_ROOT or run tools/install_reference.sh", allow_module_level=True)
PKG_ROOT, TREE = LAYOUT

from b200_whisper.backend import B200WhisperBackend  # noqa: E402
from b200_whisper.synth import synth_audio  # noqa: E402


def _pcm(seed, seconds):
    return (np.clip(synth_audio(seed, seconds), -1, 1) * 32767).astype(np.int16).tobytes()


@pytest.fixture(scope="module")
def reference_modules():
    sys.path.insert(0, PKG_ROOT)
    from b200_whisper import protostubs, register

    register.install()
    protostubs.install(os.path.join(TREE, "proto", "stt.proto"))
    import stt_server.model.worker as worker
    from stt_server.backend.application.model_registry import ModelRegistry

    yield worker, ModelRegistry
    sys.path.remove(PKG_ROOT)


def test_real_worker_and_registry_drive_the_real_engine(reference_modules):
    worker, ModelRegistry = reference_modules
    spec = "random:test-tiny:0:0.1:4.0"  # EOT-biased: hypotheses end, segments are short
    direct = B200WhisperBackend(spec, "cuda:0", "float32")
    w = worker.ModelWorker(spec, "cuda:0", "float32", "en", False, base_options={"task": "transcribe"}, backend="b200_whisper")
    assert isinstance(w.backend, B200WhisperBackend) and w.backend.engine is direct.engine
    pcm = _pcm(31, 5.0)
    audio = np.frombuffer(pcm, np.int16).astype(np.float32) / 32768.0
    for profile in (REALTIME, ACCURATE):
        r = w.decode_sync(pcm, 16000, dict(profile), time.perf_counter())
        segs, info = direct.transcribe(audio, dict(profile, language="en", task="transcribe"))
        assert [(s.start, s.end, s.text) for s in r.segments] == [(s.start, s.end, s.text) for s in segs] and r.segments
        assert r.language_code == "en" and r.language_probability == -1.0 and abs(r.audio_duration - 5.0) < 1e-6 and r.rtf > 0
    # 8 kHz stream: the worker's torchaudio resampling in front of the backend
    r8 = w.decode_sync((np.frombuffer(pcm, np.int16)[::2]).tobytes(), 8000, dict(REALTIME), time.perf_counter())
    assert abs(r8.audio_duration - 5.0) < 1e-3 and isinstance(r8.segments, list)
    w.close()
    # the registry's pool: pool_size handles, one engine, concurrent dispatch; finals evict queued partials
    reg = ModelRegistry()
    reg.load_model("m", {"model_size": spec, "device": "cuda:0", "compute_type": "float32", "pool_size": 6, "backend": "b200_whisper",
                         "language": "en", "language_fix": True, "task": "transcribe"})
    try:
        steps0 = direct.engine.stats()["decode_steps"]
        pcms = [_pcm(40 + i, 2.0 + 0.5 * i) for i in range(12)]
        futs = [reg.submit_decode("m", f"session-{i}", pcms[i], 16000, dict(REALTIME), is_final=True) for i in range(12)]
        done = [f.result(timeout=120) for f in futs]
        for i, r in enumerate(done):
            a = np.frombuffer(pcms[i], np.int16).astype(np.float32) / 32768.0
            segs, _ = direct.transcribe(a, dict(REALTIME, language="en", task="transcribe"))
            assert [(s.start, s.end, s.text) for s in r.segments] == [(s.start, s.end, s.text) for s in segs], f"session {i}"
        assert direct.engine.stats()["decode_steps"] > steps0
    finally:
        reg.close()


def _wire(channels, seconds, pool, model, extra=()):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "wire_bench.py"), "--channels", str(channels), "--seconds", str(seconds),
                          "--pool-size", str(pool), "--model", model, "--json", "--server-log", os.path.join(ROOT, "gpurun_out", "wire_server.log"),
                          *extra], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_unmodified_server_under_its_own_load_generator_real_engine():
    """grpc_load_test.py, unchanged, against the unmodified server started by b200_whisper.launcher with the real engine:
    every session succeeds and gets a final result; with the server's VAD gate on (energy stand-in for the absent Silero
    model) its partial-decode schedule runs too and the decode-latency metadata comes back."""
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    rep = _wire(16, 6.0, 8, "random:tiny:0:0.1")
    info = rep["summary"]["Info"]
    assert rep["load_test_exit"] in (0, None) and info["Sessions"] == 16 and info["Failures"] == 0 and info["Responses"] >= 16
    assert rep["summary"]["Decode Inference"]["p95"] > 0
    vad = _wire(16, 8.0, 8, "random:tiny:0:0.1", ("--energy-vad",))
    assert vad["summary"]["Info"]["Failures"] == 0 and vad["summary"]["Info"]["Responses"] >= 16
    with open(os.path.join(ROOT, "gpurun_out", "r2_wire_tiny.json"), "w") as fh:
        json.dump({"vad_off": rep, "energy_vad": vad}, fh, indent=1)
