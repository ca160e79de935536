"""The drop-in claim against the REAL caller: the reference's own `ModelWorker` (stt_server/model/worker.py) resolves
`backend="b200_whisper"` through its registry, constructs `B200WhisperBackend` the way it constructs its own backends and
drives it through `decode_sync` -- bytes in, `DecodeResult` out.  The upstream source is not part of this repository: the
tests that import it run where a checkout is found ($STT_SERVER_ROOT, or the install tools/install_reference.sh makes) and
skip elsewhere.  The engine below the backend is the host-logic fake (no CUDA needed).  The run-time proto stubs are
checked on a stored wire schema (tests/golden/stt_wire.proto) everywhere, and on the upstream proto where it is found."""
import os
import sys
import time

import numpy as np
import pytest

import b200_whisper.backend as bk
from b200_whisper.synth import synth_audio
from b200_whisper.vocab import vocab_for
from tests._util import ACCURATE, REALTIME
from tests.test_host_logic import FakeEngine, res

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from wire_bench import reference_layout  # noqa: E402

LAYOUT = reference_layout()
PKG_ROOT, TREE = LAYOUT or (None, None)  # upstream package root (for sys.path), directory holding its config/ and proto/
needs_upstream = pytest.mark.skipif(LAYOUT is None, reason="needs the upstream server source (stt_server), which is not part of "
                                                           "this repository: set STT_SERVER_ROOT or run tools/install_reference.sh")
STORED_PROTO = os.path.join(ROOT, "tests", "golden", "stt_wire.proto")


@pytest.fixture
def reference_worker(monkeypatch):
    monkeypatch.syspath_prepend(PKG_ROOT)
    for name in [n for n in sys.modules if n == "stt_server" or n.startswith("stt_server.")]:
        monkeypatch.delitem(sys.modules, name)
    from b200_whisper import register

    register.install()  # wraps the real get_backend in stt_server.model.backends AND stt_server.model.worker
    import stt_server.model.worker as worker

    v = vocab_for(51865)
    tb = v.timestamp_begin
    eng = FakeEngine(51865, [res([tb, 11, 12, tb + 150, tb + 150, 13, tb + 260])])
    audios = []
    real_open = eng.open_call

    def open_call(audio, sample_rate=None):
        audios.append(np.array(audio, dtype=np.float32, copy=True))
        return real_open(audio, sample_rate)

    eng.open_call = open_call
    monkeypatch.setattr(bk, "get_engine", lambda *a, **k: eng)
    yield worker, eng, audios
    for name in [n for n in sys.modules if n == "stt_server" or n.startswith("stt_server.")]:
        sys.modules.pop(name, None)


def _pcm(seed, seconds, rate=16000):
    a = synth_audio(seed, seconds)
    if rate != 16000:
        a = a[:: 16000 // rate] if 16000 % rate == 0 else a
    return (np.clip(a, -1, 1) * 32767).astype(np.int16).tobytes()


@needs_upstream
def test_real_model_worker_drives_the_backend(reference_worker):
    worker, eng, audios = reference_worker
    assert worker.get_backend("b200_whisper") is bk.B200WhisperBackend
    assert worker.get_backend("faster_whisper").__name__ == "FasterWhisperBackend"  # the reference's own entries survive
    with pytest.raises(RuntimeError, match="openai-whisper"):                       # ... including their own failures
        worker.get_backend("torch_whisper")
    with pytest.raises(ValueError):
        worker.get_backend("no_such_backend")
    w = worker.ModelWorker("random:test-tiny", "cuda:0", "bfloat16", "en", False, base_options={"task": "transcribe"},
                           backend="b200_whisper")
    assert isinstance(w.backend, bk.B200WhisperBackend) and w.backend_name == "b200_whisper"
    pcm = _pcm(3, 4.0)
    opts = dict(REALTIME)
    r = w.decode_sync(pcm, 16000, opts, time.perf_counter())
    assert isinstance(r, worker.DecodeResult) and opts == REALTIME
    assert [(s.start, s.end, s.text) for s in r.segments] == [(0.0, 3.0, "<11><12>"), (3.0, 5.2, "<13>")]
    assert r.language_code == "en" and r.language_probability == -1.0 and abs(r.audio_duration - 4.0) < 1e-6
    assert r.latency_sec > 0 and r.rtf > 0 and r.queue_wait_sec >= 0
    # what reached the backend is exactly pcm16_to_float32(bytes) (utils/audio.py:6-8); language / task came from the worker
    np.testing.assert_array_equal(audios[-1], np.frombuffer(pcm, np.int16).astype(np.float32) / 32768.0)
    d = eng.all_decodes[-1]
    v = vocab_for(51865)
    assert d["initial"] == v.sot_sequence("en", "transcribe") and d["beam"] == 1
    # accurate profile -> beam 5; a per-request language overrides the worker's
    r = w.decode_sync(pcm, 16000, dict(ACCURATE, language="ko"), time.perf_counter())
    assert eng.all_decodes[-1]["beam"] == 5 and eng.all_decodes[-1]["initial"][1] == v.language_token("ko") and r.language_code == "ko"
    # 8 kHz stream: the worker resamples with torchaudio and hands a float array of twice the length
    r = w.decode_sync(_pcm(3, 2.0, 8000), 8000, dict(REALTIME), time.perf_counter())
    assert abs(len(audios[-1]) - 32000) <= 2 and abs(r.audio_duration - 2.0) < 1e-3
    # empty PCM never reaches the backend (worker.py:108-117)
    n = len(eng.all_decodes)
    r = w.decode_sync(b"", 16000, dict(REALTIME), time.perf_counter())
    assert r.segments == [] and r.rtf == -1.0 and len(eng.all_decodes) == n
    # backend errors surface as the exception types the scheduler maps to ERR2002 (decode_scheduler.py:632-644)
    with pytest.raises((RuntimeError, ValueError, TypeError, OSError, TimeoutError)):
        w.decode_sync(pcm, 16000, dict(REALTIME, beam_size=99), time.perf_counter())
    w.close()


@needs_upstream
def test_real_worker_pool_shares_one_engine(reference_worker, monkeypatch):
    """model_registry.py:230-247 builds pool_size workers with identical arguments: every handle must share one engine."""
    worker, eng, _ = reference_worker
    made = []
    monkeypatch.setattr(bk, "get_engine", lambda *a, **k: (made.append(a), eng)[1])
    pool = [worker.ModelWorker("random:test-tiny", "cuda:0", "bfloat16", None, False, backend="b200_whisper") for _ in range(4)]
    assert len({id(p.backend.engine) for p in pool}) == 1 and len({a for a in made}) == 1
    with pytest.raises(ValueError):  # constructor failures are of a type load_model aborts on cleanly (model_registry.py:281-289)
        worker.ModelWorker("random:test-tiny", "cpu", "bfloat16", None, False, backend="b200_whisper")
    for p in pool:
        p.close()


def test_runtime_proto_stubs_roundtrip():
    """protostubs builds stt_pb2 / stt_pb2_grpc from a .proto without grpc_tools: the stored wire schema, and the upstream
    proto/stt.proto where a checkout is found."""
    for path in [STORED_PROTO] + ([os.path.join(TREE, "proto", "stt.proto")] if TREE else []):
        _check_proto_stubs(path)


def _check_proto_stubs(path):
    from b200_whisper import protostubs

    pb2 = protostubs.build_pb2_module(protostubs.parse_proto(open(path).read()), "x_pb2")
    grpc_mod = protostubs.build_grpc_module(pb2, "x_pb2_grpc")
    req = pb2.SessionRequest(session_id="s", vad_mode=pb2.VAD_AUTO_END, task=pb2.TASK_TRANSLATE, decode_profile=pb2.DECODE_PROFILE_ACCURATE)
    req.attributes["k"] = "v"
    assert not req.HasField("vad_threshold_override")
    req.vad_threshold_override = 0.0  # proto3 `optional`: explicit presence
    back = pb2.SessionRequest.FromString(req.SerializeToString())
    assert back.HasField("vad_threshold_override") and back.attributes["k"] == "v" and back.decode_profile == 2
    assert pb2.Task.Name(back.task) == "TASK_TRANSLATE" and pb2.DecodeProfile.Value("DECODE_PROFILE_REALTIME") == 1
    chunk = pb2.AudioChunk(pcm16=b"\x01\x02", sample_rate=16000, is_final=True, session_id="s")
    assert pb2.AudioChunk.FromString(chunk.SerializeToString()).pcm16 == b"\x01\x02"
    assert {f.name: f.number for f in pb2.STTResult.DESCRIPTOR.fields}["committed_text"] == 10
    svc = pb2.DESCRIPTOR.services_by_name["STTBackend"]
    assert [(m.name, m.client_streaming, m.server_streaming) for m in svc.methods] == \
           [("CreateSession", False, False), ("StreamingRecognize", True, True)]
    assert all(hasattr(grpc_mod, n) for n in ("STTBackendStub", "STTBackendServicer", "add_STTBackendServicer_to_server"))


@needs_upstream
def test_real_model_registry_dispatches_to_the_backend(reference_worker, monkeypatch):
    """SURVEY 8a row a1 with the REAL code: `ModelRegistry.load_model` builds a pool of `b200_whisper` workers, and
    `submit_decode` / `_dispatch_loop` / `_worker_loop` (model_registry.py:385-680) call `transcribe` from pool_size threads at
    once.  Needs the run-time proto stubs: everything under stt_server.backend imports the generated modules."""
    import threading

    from b200_whisper import protostubs

    worker, eng, _ = reference_worker
    protostubs.install(os.path.join(TREE, "proto", "stt.proto"))
    from stt_server.backend.application.model_registry import ModelRegistry

    lock = threading.Lock()
    state = {"now": 0, "peak": 0, "threads": set()}
    real_open = eng.open_call

    def open_call(audio, sample_rate=None):
        call = real_open(audio, sample_rate)
        real_decode = call.decode

        def decode(*a, **k):
            with lock:
                state["now"] += 1
                state["peak"] = max(state["peak"], state["now"])
                state["threads"].add(threading.get_ident())
            time.sleep(0.05)  # the GPU work; ctypes releases the GIL there
            try:
                return real_decode(*a, **k)
            finally:
                with lock:
                    state["now"] -= 1

        call.decode = decode
        return call

    eng.open_call = open_call
    reg = ModelRegistry()
    reg.load_model("m", {"model_size": "random:test-tiny", "device": "cuda:0", "compute_type": "bfloat16", "pool_size": 4,
                         "backend": "b200_whisper", "language": "en", "language_fix": True, "task": "transcribe"})
    try:
        assert reg.is_loaded("m")
        pool = [reg.get_worker("m") for _ in range(8)]
        assert all(isinstance(w.backend, bk.B200WhisperBackend) for w in pool) and len({id(w.backend.engine) for w in pool}) == 1
        pcm = _pcm(9, 2.0)
        futs = [reg.submit_decode("m", f"session-{i % 8}", pcm, 16000, dict(REALTIME), is_final=(i >= 8)) for i in range(16)]
        done = [f.result(timeout=30) for f in futs if not f.cancelled()]
        assert len(done) >= 8 and all(r.language_code == "en" and len(r.segments) == 2 for r in done)
        assert 2 <= state["peak"] <= 4 and len(state["threads"]) >= 2  # pool_size callers at once, never more
        with pytest.raises(ValueError):
            reg.load_model("bad", {"model_size": "random:test-tiny", "device": "cpu", "backend": "b200_whisper"})
        assert not reg.is_loaded("bad")
    finally:
        reg.close()


def _free_port():
    import socket

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@needs_upstream
def test_unmodified_server_end_to_end_over_grpc(tmp_path):
    """The wire-level drop-in (SURVEY 8(f) row 4): the UNMODIFIED reference server -- gRPC servicer, session manager, stream
    orchestrator, decode scheduler, model registry, ModelWorker -- started by `b200_whisper.launcher` with
    `--model-backend b200_whisper` (run-time proto stubs, wrapped registry), serving CreateSession + StreamingRecognize to a
    client built from the same proto.  The engine below the backend is the host-logic fake (tests/_ref_server_driver.py)."""
    import subprocess

    import grpc

    from b200_whisper import protostubs

    port, mport, wport = _free_port(), _free_port(), _free_port()
    cfg = tmp_path / "server.yaml"
    # the shipped server configuration (limits, partial-decode schedule, ...) + a loopback WebSocket port of our own
    cfg.write_text(open(os.path.join(TREE, "config", "server.yaml")).read() + f"\nws_host: 127.0.0.1\nws_port: {wport}\n")
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    proc = subprocess.Popen(
        [sys.executable, os.path.join(repo, "tests", "_ref_server_driver.py"), "--config", str(cfg), "--model-backend", "b200_whisper",
         "--model", "random:test-tiny", "--device", "cuda:0", "--port", str(port), "--metrics-port", str(mport),
         "--vad-threshold", "0", "--model-pool-size", "2", "--language", "en", "--log-level", "INFO"],
        cwd=repo, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=dict(os.environ, STT_SERVER_ROOT=PKG_ROOT))
    pb2 = protostubs.build_pb2_module(protostubs.parse_proto(open(os.path.join(TREE, "proto", "stt.proto")).read()), "client_pb2")
    pb2_grpc = protostubs.build_grpc_module(pb2, "client_pb2_grpc")
    results, log = [], ""
    try:
        channel = grpc.insecure_channel(f"127.0.0.1:{port}")
        grpc.channel_ready_future(channel).result(timeout=90)
        stub = pb2_grpc.STTBackendStub(channel)
        sessions = {}
        for sid, profile in (("s-rt", pb2.DECODE_PROFILE_REALTIME), ("s-acc", pb2.DECODE_PROFILE_ACCURATE)):
            rsp = stub.CreateSession(pb2.SessionRequest(session_id=sid, vad_mode=pb2.VAD_CONTINUE, task=pb2.TASK_TRANSCRIBE,
                                                        decode_profile=profile, language_code="en"), timeout=20)
            assert rsp.decode_profile == profile and rsp.language_code == "en"
            sessions[sid] = rsp
        pcm = _pcm(3, 3.0)

        def chunks(sid):
            step = 3200  # 100 ms slices with is_final on the last one, like the reference's batch client
            for i in range(0, len(pcm), step):
                yield pb2.AudioChunk(pcm16=pcm[i:i + step], sample_rate=16000, is_final=(i + step >= len(pcm)), session_id=sid,
                                     session_token=sessions[sid].token)
                time.sleep(0.01)

        for sid in sessions:
            results.append([(r.text, r.is_final, round(r.start_sec, 2), round(r.end_sec, 2), r.language_code)
                            for r in stub.StreamingRecognize(chunks(sid), timeout=60)])
        channel.close()
    finally:
        proc.terminate()
        try:
            log, _ = proc.communicate(timeout=40)
        except subprocess.TimeoutExpired:
            proc.kill()
            log, _ = proc.communicate()
    for got in results:
        finals = [r for r in got if r[1]]
        assert finals and finals[-1] == ("<11><12>", True, 0.0, 2.0, "en"), (got, log[-2000:])
    assert len(results) == 2
    assert "decode_profile=realtime" in log and "decode_profile=accurate" in log and "Scheduled decode" in log, log[-2000:]
