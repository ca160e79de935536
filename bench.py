#!/usr/bin/env python
"""bench.py -- RTFx (audio-seconds transcribed per wall-second) of the Whisper hot path on B200.

Default workload (BASELINE.json configs[4], the per-GPU shard of the config the metric is quoted on):
large-v3 (128 mel bins), realtime decode profile (beam_size=1), 128 concurrent streaming sessions
per GPU, each submitting one partial-decode window of its last 2-10 s of audio per step (seeded
lengths; every window is a full 30 s encoder pass, as in the reference).  Random-init weights of the
named architecture and synthetic audio (no network) -> hypotheses never reach EOT and every window
runs the full 224 decoder steps: the worst case.  One "step" = one such batch of 128 windows.
`--config N` selects another BASELINE.json configs[N] (table CONFIGS below): the same line, per config.

  value : whole-job RTFx with the PCM already resident in HBM, timed with CUDA events on the engine
          stream around mel -> encoder -> cross-KV -> 224 batched decoder steps (max over ranks)
  e2e   : the same metric through the public backend (`B200WhisperBackend.transcribe`, the call
          ModelWorker makes, reference worker.py:125) from 128 host threads with host numpy buffers;
          host->device PCM copies and device->host results are inside the timed region
  --impl reference : the reference's CPU path (fp32 torch restatement of torch_whisper, `oracle/`)
          on all host cores, one window per step (bounded sample), same metric/config

Weak scaling: sessions per GPU are fixed; ranks never exchange data (sessions shard), torch.distributed
is used only for the barrier and the max-over-ranks reduction.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ENC_BATCH = 16  # windows admitted per encoder pass (8 is 5 % more efficient per window, but the 128-session burst of the
                # e2e leg then needs 16 admission rounds interleaved with decoder steps: e2e 351 vs 373 audio-s/s)

# the server's two decode profiles (reference config/model.yaml:42-65, stt_server/config/default/model.py:17-27)
REALTIME = {"beam_size": 1, "best_of": 1, "patience": 1.0, "temperature": 0.0, "length_penalty": 1.0,
            "without_timestamps": True, "compression_ratio_threshold": 2.4, "no_speech_threshold": 0.6,
            "log_prob_threshold": -1.0, "language": "en", "task": "transcribe"}
ACCURATE = dict(REALTIME, beam_size=5, best_of=5)

# BASELINE.json `configs`, as this bench drives them at the ModelWorker.decode_sync boundary (SURVEY.md 8(d)).
# windows: "partial" = one 2-10 s partial window per session per step; "utterance" = one VAD-endpointed utterance of
# 1-8 s per session per step (finals only); "chunk30" = one 30 s chunk per session per step.
CONFIGS = {
    0: dict(model="tiny.en", sessions=1, profile="realtime", windows="chunk30", gpus=(1,),
            label="configs[0]: tiny.en, batch client, single 30 s synthetic chunk (the reference's CPU int8 case; this arm runs it on the GPU)"),
    1: dict(model="base", sessions=16, profile="realtime", windows="partial", gpus=(1,),
            label="configs[1]: base multilingual (language fixed to en), realtime profile, 16 concurrent streaming sessions, 1 B200"),
    2: dict(model="small", sessions=64, profile="realtime", windows="utterance", gpus=(1, 2, 4),
            label="configs[2]: small, 64 concurrent sessions per GPU, VAD-endpointed utterances (finals only), realtime profile"),
    3: dict(model="large-v3", sessions=64, profile="accurate", windows="chunk30", gpus=(1,),
            label="configs[3]: large-v3 (128 mel bins), accurate profile (beam 5), 64 back-to-back 30 s chunks per step, 1 B200"),
    4: dict(model="large-v3", sessions=128, profile="realtime", windows="partial", gpus=(1, 2, 4, 8),
            label="configs[4] per-GPU shard: large-v3 realtime profile (beam_size=1), 128 concurrent sessions per GPU, one 2-10 s "
                  "partial window per session per step"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=sorted(CONFIGS), help="BASELINE.json configs[N] (default 4)")
    ap.add_argument("--model", default=None, help="override the config's model")
    ap.add_argument("--sessions", type=int, default=0, help="override the config's concurrent sessions per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--streaming-seconds", type=float, default=10.0,
                    help="length of the real-time streaming-session run reported under `streaming` (0 = skip)")
    ap.add_argument("--streaming-sessions", type=int, default=0, help="sessions per GPU in that run (0 = 3 x --sessions)")
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--wire-channels", type=int, default=-1,
                    help="streams of the wire-level leg (unmodified server + its own grpc_load_test.py); 0 = skip, -1 = 64 at N = 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step decoded (rank 0's windows) to DIR/<name>.npy, for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return resolve_config(args)


def resolve_config(args):
    """fill model / sessions / decode profile / window kind from BASELINE.json configs[args.config]"""
    cfg = CONFIGS[args.config]
    args.model = args.model or cfg["model"]
    args.sessions = args.sessions or cfg["sessions"]
    args.profile = dict(ACCURATE if cfg["profile"] == "accurate" else REALTIME)
    args.n_group = 5 if cfg["profile"] == "accurate" else 1
    args.windows = cfg["windows"]
    args.cfg = cfg
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic(sessions: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the roofline kernel from the committed ncu --set full
    capture (profiles/r1_xattn_mma_ncu_full.txt); only valid for the captured configuration (128 sessions)."""
    path = os.path.join(ROOT, "profiles", "r1_xattn_mma_traffic.json")
    if sessions == 128 and os.path.exists(path):
        with open(path) as fh:
            return json.load(fh)["dram_bytes_per_launch"]
    return None


def window_lengths(rank: int, sessions: int, kind: str = "partial"):
    rng = np.random.default_rng(4242 + rank)
    if kind == "chunk30":
        return [30.0] * sessions
    lo, hi = (2.0, 10.0) if kind == "partial" else (1.0, 8.0)  # utterance: the burst lengths of tools/stream_bench.py
    return [float(np.round(rng.uniform(lo, hi), 2)) for _ in range(sessions)]


def dump_outputs(out_dir: str, results, lengths) -> None:
    """The decoded result of every window as a caller of the decode path receives it (tokens cut at the first EOT,
    padded with -1; sum / average log-probability), plus the window lengths it came from.  No no-speech probability:
    the timed pipeline starts decoding after the prompt and never computes one."""
    os.makedirs(out_dir, exist_ok=True)
    n = max([len(r["tokens"]) for r in results] + [1])
    tokens = np.full((len(results), n), -1.0, dtype=np.float64)
    for i, r in enumerate(results):
        tokens[i, :len(r["tokens"])] = r["tokens"]
    arrays = {"tokens": tokens, "n_tokens": np.array([len(r["tokens"]) for r in results], dtype=np.float64),
              "sum_logprob": np.array([r["sum_logprob"] for r in results], dtype=np.float32),
              "avg_logprob": np.array([r["avg_logprob"] for r in results], dtype=np.float32),
              "window_seconds": np.array(lengths, dtype=np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def faster_whisper_row():
    """the reference's other baseline (stt_server/model/backends/faster_whisper.py:14-39, CTranslate2 int8 on the CPU):
    probed at run time, never estimated"""
    try:
        import faster_whisper  # noqa: F401
    except Exception as exc:  # noqa: BLE001
        return f"not runnable: {type(exc).__name__}: {exc} (module absent from this image, no network to install it)"
    return "importable, but no pretrained CTranslate2 checkpoint is available offline: not run"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.proc = None
        self.lines = []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus: int):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod

        torch.cuda.set_device(local)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    return rank, world, local, dist


def _dist_tensor(dist, local, values):
    import torch

    dev = f"cuda:{local}" if dist.get_backend() == "nccl" else "cpu"
    return torch.tensor(values, device=dev, dtype=torch.float64)


def barrier_max(dist, local, value: float) -> float:
    """barrier + max over ranks (the timed region of a multi-GPU run is the slowest rank's)"""
    if dist is None:
        return value
    t = _dist_tensor(dist, local, [value])
    dist.barrier()
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(dist, local, value: float) -> float:
    if dist is None:
        return value
    t = _dist_tensor(dist, local, [value])
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def whole_job_rtfx(dist, local, audio_sec_local: float, seconds_local: float) -> float:
    """Sessions shard across ranks with no data-path collective: whole-job throughput = all ranks' audio / slowest rank."""
    return sum_over_ranks(dist, local, audio_sec_local) / barrier_max(dist, local, seconds_local)


def cpu_oracle_window(state, model_name: str, seconds: float, sample_len=None, threads: int = 0, profile=None):
    """One window through the CPU oracle (reference torch_whisper path restated); returns (elapsed s, cores)."""
    import torch

    from b200_whisper.synth import MODEL_DIMS, synth_audio
    from oracle import whisper_oracle as wo

    cores = threads or os.cpu_count() or 1
    torch.set_num_threads(cores)
    dims = MODEL_DIMS[model_name]
    model = wo.Whisper(wo.ModelDimensions(**dims.__dict__), state)
    audio = synth_audio(999, seconds)
    opts = wo.normalize_options(dict(profile or REALTIME))  # the wrapper's option handling (torch_whisper.py:78-110)
    if sample_len:
        opts["sample_len"] = sample_len
    t0 = time.perf_counter()
    wo.transcribe(model, audio, **opts)
    return time.perf_counter() - t0, cores


def workload_name(args) -> str:
    name = args.cfg["label"]
    if args.model != args.cfg["model"] or args.sessions != args.cfg["sessions"]:
        name += f" [overridden: model {args.model}, {args.sessions} sessions per GPU]"
    return name


def wire_leg(args, channels: int):
    """Secondary e2e (SURVEY 8(d)): the UNMODIFIED reference server, started by b200_whisper.launcher with this backend and
    the real engine, under the reference's own load generator tools/bench/grpc_load_test.py run unchanged (100 ms chunks in
    real time; the server's VAD gate on over an energy stand-in for the absent Silero model so that its partial-decode
    schedule runs).  The reference tree is not on the GPU box: tools/install_reference.sh puts it under baseline/_ref."""
    cmd = [sys.executable, os.path.join(ROOT, "tools", "wire_bench.py"), "--json", "--channels", str(channels), "--seconds", "10",
           "--pool-size", str(channels), "--model", f"random:{args.model}:0:0.1", "--energy-vad", "--ready-timeout", "240",
           "--decode-profile", args.cfg["profile"]]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=420, cwd=ROOT)
        rep = json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as exc:  # noqa: BLE001 - the wire leg must never take the bench line down with it
        return {"unavailable": f"{type(exc).__name__}: {exc}"[:300]}
    if "unavailable" in rep:
        return rep
    sm = rep.get("summary", {})
    pick = lambda sec: {k: sm.get(sec, {}).get(k) for k in ("p50", "p95", "p99")}  # noqa: E731
    return {"channels": channels, "audio_s_per_channel": rep["audio_s_per_channel"], "wall_s": rep["wall_s"],
            "audio_s_per_s": sm.get("Info", {}).get("Audio-sec/sec"), "sessions": sm.get("Info", {}).get("Sessions"),
            "failures": sm.get("Info", {}).get("Failures"), "responses": sm.get("Info", {}).get("Responses"),
            "decode_inference_s": pick("Decode Inference"), "decode_queue_wait_s": pick("Decode Queue Wait"),
            "decode_total_s": pick("Decode Total"), "decodes_per_session": pick("Decode Count"), "tail_latency_s": pick("Tail"),
            "note": "unmodified server + grpc_load_test.py (reference tools/bench/grpc_load_test.py:742,1028-1052), real-time pacing: "
                    "audio_s_per_s is bounded by channels x 1.0; latencies are the server's own stt-decode-* metadata; VAD gate on over "
                    "an energy stand-in (silero_vad absent); the server process builds its own engine next to the bench's"}


def cpu_sample_seconds(args) -> float:
    return 30.0 if args.windows == "chunk30" else 6.0


def run_reference(args):
    # the CPU arm needs no process group: under torchrun rank 0 alone runs and prints, the other ranks exit 0 without work
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from b200_whisper.synth import MODEL_DIMS, random_state_dict

    state = random_state_dict(MODEL_DIMS[args.model], 0, emb_std=0.1)
    seconds = cpu_sample_seconds(args)
    for _ in range(args.warmup):  # nothing to warm on the CPU but threads/allocator: short decodes
        cpu_oracle_window(state, args.model, seconds, sample_len=4, threads=args.cpu_threads, profile=args.profile)
    times = []
    cores = 1
    for _ in range(args.steps):
        dt, cores = cpu_oracle_window(state, args.model, seconds, threads=args.cpu_threads, profile=args.profile)
        times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = seconds / (ms / 1e3)
    sample = (f"1 session x 1 window ({seconds:.0f} s audio -> full 30 s encoder pass + 224 decoder steps, "
              f"beam {args.profile['beam_size']}) per step")
    emit(json.dumps({
        "impl": "reference", "metric": "RTFx (audio-seconds transcribed per second)", "value": value, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic audio, random-init weights",
        "config": {"workload": workload_name(args),
                   "sample": f"bounded sample of that workload: ONE of its windows per step ({seconds:.0f} s) on the host cores, fp32 torch",
                   "note": "warm-up steps decode 4 tokens only; timed steps are full windows (224 decoder steps)"},
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample},
        "faster_whisper_int8": faster_whisper_row(),
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_b200(args):
    rank, world, local, dist = dist_setup(args.gpus)
    import torch  # device plumbing only (set_device / barrier)

    torch.cuda.set_device(local)
    from b200_whisper.backend import B200WhisperBackend, _ENGINES
    from b200_whisper.synth import MODEL_DIMS, random_state_dict, synth_audio

    pk = peaks()
    S = args.sessions
    dims = MODEL_DIMS[args.model]
    spec = f"random:{args.model}:0:0.1"
    # the engine materialises the seeded random checkpoint one tensor at a time (backend.load_checkpoint); only the CPU
    # baseline at the end (rank 0, N = 1) needs the whole fp32 state dict on the host
    NG = args.n_group
    handles = [B200WhisperBackend(spec, f"cuda:{local}", "bfloat16", max_segments=S, max_sequences=max(2 * S, NG * S, 320 if args.config == 4 and S >= 64 else 8),
                                  max_encoder_batch=min(ENC_BATCH, S)) for _ in range(S)]
    eng = handles[0].engine
    lengths = window_lengths(rank, S, args.windows)
    audios = [synth_audio(rank * 100000 + i, lengths[i]) for i in range(S)]
    audio_sec = float(sum(a.size for a in audios)) / 16000.0
    n_steps = dims.n_text_ctx // 2  # 224: random weights never emit EOT (worst case)

    # ---- value: device-timed pipeline on resident PCM ----
    for _ in range(args.warmup):
        eng.bench_pipeline(audios, NG, n_steps)
    barrier_max(dist, local, 0.0)
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = eng.stats()["kernel_launches"]
    total_ms = 0.0
    for _ in range(args.steps):
        total_ms += eng.bench_pipeline(audios, NG, n_steps)
    torch.cuda.synchronize()
    launches = eng.stats()["kernel_launches"] - l0
    value = whole_job_rtfx(dist, local, audio_sec * args.steps, total_ms / 1e3)
    total_ms = barrier_max(dist, local, total_ms)
    clocks = sampler.stop() if sampler else None
    ms_per_step = total_ms / args.steps
    if args.dump_outputs and rank == 0:  # before the e2e leg reuses the engine's decoder state
        dump_outputs(args.dump_outputs, eng.bench_pipeline_results(S, NG, n_steps, args.profile["length_penalty"]), lengths)

    # ---- e2e: public backend call from S host threads, host buffers ----
    lat = []

    def e2e_step(record: bool):
        def work(i):
            t0 = time.perf_counter()
            handles[i].transcribe(audios[i], args.profile)
            if record:
                lat.append(time.perf_counter() - t0)

        th = [threading.Thread(target=work, args=(i,)) for i in range(S)]
        t0 = time.perf_counter()
        [t.start() for t in th]
        [t.join() for t in th]
        return time.perf_counter() - t0

    for _ in range(max(1, args.warmup - 1)):
        e2e_step(False)
    barrier_max(dist, local, 0.0)
    s0 = eng.stats()
    e2e_total = 0.0
    for _ in range(args.steps):
        e2e_total += e2e_step(True)
    s1 = eng.stats()
    e2e_value = whole_job_rtfx(dist, local, audio_sec * args.steps, e2e_total)
    e2e_total = barrier_max(dist, local, e2e_total)
    lat_sorted = sorted(lat)
    p95 = lat_sorted[max(0, int(np.ceil(0.95 * len(lat_sorted))) - 1)] if lat_sorted else None  # nearest rank

    # ---- streaming sessions in real time (tools/stream_bench.py): the orchestrator's partial / final schedule ----
    streaming = None
    if args.streaming_seconds > 0 and args.windows != "chunk30":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from stream_bench import run_stream_sim

        # configs[4]: 3 x the per-GPU shard (how many streams one GPU carries); configs[1] / [2]: the named session count
        n_stream = args.streaming_sessions or (3 * S if args.config == 4 else S)
        while len(handles) < n_stream:
            handles.append(B200WhisperBackend(spec, f"cuda:{local}", "bfloat16"))
        barrier_max(dist, local, 0.0)
        streaming = run_stream_sim(handles[:n_stream], args.streaming_seconds, seed=rank, opts=args.profile,
                                   finals_only=args.windows == "utterance")
        streaming["note"] = ("real-time pacing; decodes bounded by DecodingOptions.sample_len = 3.5 tokens per audio second + 4 "
                             "(random weights never emit EOT); per GPU, rank 0 shown")

    if rank != 0:
        return
    # ---- roofline of the dominant kernel (decoder cross-attention, HBM-bound), timed live ----
    xa_ms, xa_bytes = eng.bench_cross_attention(S, NG, 64)
    achieved = xa_bytes / (xa_ms * 1e-3) / 1e9
    stages = {}
    enc_b = min(ENC_BATCH, S)
    ems, eflops = eng.bench_encoder(enc_b, 3)
    stages["encoder"] = {"batch": enc_b, "ms": ems, "tflops": eflops / (ems * 1e-3) / 1e12,
                         "frac_of_bf16_sustained": eflops / (ems * 1e-3) / 1e12 / pk["bf16_tflops_sustained"]}
    eng.bench_decoder_step(S, NG, 100, 6)  # the step graph of this shape is captured at its third sighting: not in the timed run
    dms, dbytes = eng.bench_decoder_step(S, NG, 100, 20)
    stages["decoder_step"] = {"segments": S, "hypotheses_per_segment": NG, "context": 100, "ms": dms, "gbs": dbytes / (dms * 1e-3) / 1e9,
                              "frac_of_hbm": dbytes / (dms * 1e-3) / 1e9 / pk["hbm_gbs"]}
    if args.config == 4 and S >= 64:  # the other headline shape (configs[3]: 64 windows x beam 5) on the same engine
        eng.bench_decoder_step(64, 5, 100, 6)
        bms, bbytes = eng.bench_decoder_step(64, 5, 100, 20)
        stages["decoder_step_beam5"] = {"segments": 64, "hypotheses_per_segment": 5, "context": 100, "ms": bms,
                                        "gbs": bbytes / (bms * 1e-3) / 1e9, "frac_of_hbm": bbytes / (bms * 1e-3) / 1e9 / pk["hbm_gbs"]}
    mel_n = int(cpu_sample_seconds(args) * 16000)
    mms, mbytes = eng.bench_mel(mel_n, 20)
    stages["mel"] = {"audio_s": mel_n / 16000.0, "ms": mms, "gbs": mbytes / (mms * 1e-3) / 1e9, "frac_of_hbm": mbytes / (mms * 1e-3) / 1e9 / pk["hbm_gbs"]}

    out = {
        "metric": "RTFx (audio-seconds transcribed per second)", "value": value, "unit": "audio-s/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic audio, random-init weights (no EOT: 224 decoder steps per window)",
        "impl": "b200",
        "config": {"workload": workload_name(args), "baseline_config_index": args.config,
                   "sessions_per_gpu": S, "audio_s_per_step_per_gpu": audio_sec, "decoder_steps_per_window": n_steps,
                   "l2": "inputs larger than L2 (cross-KV cache %.1f GB per step)" % (S * dims.n_text_layer * 1500 * 2 * dims.n_text_state * 2 / 1e9),
                   "timing": "CUDA events on the engine stream inside libb200whisper.so, max over ranks", "peaks": pk["source"]},
        "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": (s1["h2d_bytes"] - s0["h2d_bytes"]) // args.steps,
                "d2h_bytes_per_step": (s1["d2h_bytes"] - s0["d2h_bytes"]) // args.steps,
                "ms_per_step": 1e3 * e2e_total / args.steps, "p95_partial_latency_s": p95, "host_threads": S},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"kernel": "dec_cross_attention_mma_kernel (decoder cross-attention over the cached encoder K/V)", "bound": "hbm",
                     "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
                     "traffic": ncu_traffic(S) if args.config == 4 else None, "ms_per_launch": xa_ms,
                     "algorithmic_bytes_per_launch": xa_bytes},
        "stages": stages,
    }
    if streaming is not None:
        out["streaming"] = streaming
    if world == 1 and not args.no_cpu_baseline:
        state = random_state_dict(dims, 0, emb_std=0.1)
        cs = cpu_sample_seconds(args)
        dt, cores = cpu_oracle_window(state, args.model, cs, threads=args.cpu_threads, profile=args.profile)
        out["cpu_baseline"] = {"value": cs / dt, "unit": "audio-s/s", "cores": cores, "kind": "port",
                               "sample": f"1 session x 1 window ({cs:.0f} s audio, full 30 s encoder pass + 224 decoder steps, beam "
                                         f"{args.profile['beam_size']}), fp32 torch on {cores} threads, {dt:.1f} s"}
    out["faster_whisper_int8"] = faster_whisper_row()
    wire_channels = args.wire_channels if args.wire_channels >= 0 else (64 if world == 1 and args.windows != "chunk30" else 0)
    if wire_channels > 0:
        out["wire"] = wire_leg(args, wire_channels)
    emit(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: str) -> None:
    """The ONE JSON line goes to the real stdout; everything else a library prints (NCCL banner, ...) went to stderr."""
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (line + "\n").encode())


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # fd 1 -> stderr for the duration of the run
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
