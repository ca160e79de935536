"""Language detection inside the first window's decode (detect mode) against the two-call path, with the language unset
as a multilingual deployment leaves it.  For large-v3 and base (random init), in one process, alternating the two paths
over the same seeded 2-10 s partial windows (bench.py's "partial" lengths), at 16 and 128 concurrent calls:

* threads: one host thread per call, each opening its call and decoding its window --
  two-call: call.detect_language(0), then call.decode with that language's sot sequence;
  detect:   call.decode_detect with the language left open;
* transcribe_many: the backend's batched seek loop over all calls (language None, one temperature rung) -- two-call:
  backend.detect_in_decode = False, so the backend runs its separate detect_language pass per call first (what it did
  before detect mode); detect: the backend's default.

Reported per configuration and path: wall time per batch (every repeat, and the median), and the BW_STAT_WINDOWS /
BW_STAT_ENCODER_BATCHES deltas per batch; plus the GPU's name and power limit, read in the same run.

Usage: python tools/auto_language_bench.py [--out profiles/r4_auto_language.json] [--repeats 3]"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], check=True,
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [v.strip() for v in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def run_threads(b, audios, detect):
    v, eng = b.vocab, b.engine

    def work(audio):
        with eng.open_call(audio) as call:
            if detect:
                call.decode_detect(0, [v.sot, -1, v.transcribe], 0, None, None, None)
            else:
                tok, _ = call.detect_language(0)
                call.decode(0, [v.sot, tok, v.transcribe], 0, None, None, None)

    th = [threading.Thread(target=work, args=(a,)) for a in audios]
    [t.start() for t in th]
    [t.join() for t in th]


def run_many(b, audios, detect, opts):
    b.detect_in_decode = detect  # off: the backend's separate detect_language pass per call (its path before detect mode)
    b.transcribe_many(audios, opts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_auto_language.json"))
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--models", default="large-v3,base")
    args = ap.parse_args()

    from b200_whisper.backend import B200WhisperBackend
    from b200_whisper.synth import synth_audio
    from bench import ENC_BATCH, window_lengths

    info = gpu_info()
    # one temperature rung and no thresholds: every call decodes its window(s) exactly once on both paths
    opts = {"beam_size": None, "temperature": 0.0, "compression_ratio_threshold": None, "log_prob_threshold": None,
            "no_speech_threshold": None}
    results = {}
    for model in args.models.split(","):
        b = B200WhisperBackend(f"random:{model}:0:0.1", "cuda:0", "bfloat16", max_segments=128, max_sequences=320,
                               max_encoder_batch=ENC_BATCH)
        lengths = window_lengths(0, 128, "partial")
        audios = [synth_audio(i, lengths[i]) for i in range(128)]
        res = {}
        for n in (16, 128):
            for driver in ("threads", "transcribe_many"):
                batch = audios[:n]

                def once(detect):
                    s0 = b.engine.stats()
                    t0 = time.perf_counter()
                    if driver == "threads":
                        run_threads(b, batch, detect)
                    else:
                        run_many(b, batch, detect, opts)
                    wall = time.perf_counter() - t0
                    s1 = b.engine.stats()
                    return wall, s1["windows"] - s0["windows"], s1["encoder_batches"] - s0["encoder_batches"]

                cfg = {p: {"wall_s": [], "windows": [], "encoder_batches": []} for p in ("two_call", "detect")}
                once(False), once(True)  # warm-up: modules, step graphs of these shapes
                for rep in range(args.repeats):
                    for p in ("two_call", "detect") if rep % 2 == 0 else ("detect", "two_call"):
                        wall, nw, ne = once(p == "detect")
                        cfg[p]["wall_s"].append(wall)
                        cfg[p]["windows"].append(nw)
                        cfg[p]["encoder_batches"].append(ne)
                for p in cfg:
                    cfg[p]["wall_s_median"] = float(np.median(cfg[p]["wall_s"]))
                cfg["wall_ratio_detect_over_two_call"] = cfg["detect"]["wall_s_median"] / cfg["two_call"]["wall_s_median"]
                key = f"{n}_calls_{driver}"
                res[key] = cfg
                print(model, key, json.dumps({p: {k: v for k, v in c.items()} if isinstance(c, dict) else c for p, c in cfg.items()}),
                      flush=True)
        results[model] = {"audio_s_of_the_128_windows": float(sum(lengths)), "configs": res}
        b.engine.close()
    out = {"gpu": info, "time": time.strftime("%Y-%m-%d %H:%M:%S"), "repeats": args.repeats, "compute": "bf16",
           "models": "random-init weights, seed 0", "window_lengths": "bench.py window_lengths(0, n, 'partial'): 2-10 s",
           "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({"gpu": info}, indent=1))


if __name__ == "__main__":
    main()
