"""The 8-bit cross-KV mode (compute_type bfloat16_int8kv) against the bf16 product mode, large-v3 on one GPU, both engines in
one process and the two modes alternated, three repeats each:

* decoder step time at 128 x 1 and 64 x 5 windows x hypotheses, context 100 (bw_bench_decoder_step, CUDA graphs warm);
* cross-attention kernel time per launch and GB/s of algorithmic bytes (bw_bench_cross_attention);
* cross-KV stage per window: the pair GEMM and, in the 8-bit mode, the quantize kernel (torch.profiler kernel times over
  one pipeline run);
* bw_bench_pipeline audio-s/s at bench.py's default shape (configs[4]: 128 windows of 2-10 s, beam 1, 224 steps);
* free device memory after each engine's creation at max_segments 128;
* token agreement of the two modes on that pipeline's decoded windows (bw_bench_pipeline_results);
* the GPU's name and power limit, read in the same run.

Usage: python tools/cross_kv_int8_bench.py [--out profiles/r3_cross_kv_int8.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], check=True,
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [v.strip() for v in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def cross_kv_stage_us(eng, audios, n_steps, int8):
    """kernel times per window of the cross-KV stage in one pipeline run: the GEMM launched right before each quantize
    kernel (8-bit mode), the quantize kernel itself; the bf16 mode launches the same GEMM into the slot directly"""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.bench_pipeline(audios, 1, n_steps)
    kernels = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
    if not int8:
        return None
    gemm, quant, names = [], [], set()
    for i, k in enumerate(kernels):
        if "cross_kv_int8_write_kernel" in k.name:
            quant.append(k.time_range.elapsed_us())
            prev = [p for p in kernels[:i] if getattr(p, "device_resource_id", None) == getattr(k, "device_resource_id", None)]
            gemm.append(prev[-1].time_range.elapsed_us())
            names.add(prev[-1].name[:120])
    assert len(quant) == len(audios), (len(quant), len(audios))
    return {"gemm_us": float(np.mean(gemm)), "quantize_us": float(np.mean(quant)), "total_us": float(np.mean(gemm) + np.mean(quant)),
            "gemm_kernel": sorted(names)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_cross_kv_int8.json"))
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()

    import torch

    from b200_whisper.backend import B200WhisperBackend
    from b200_whisper.synth import synth_audio
    from bench import ENC_BATCH, window_lengths

    info = gpu_info()
    spec = "random:large-v3:0:0.1"
    modes = {"bf16": "bfloat16", "bf16_int8kv": "bfloat16_int8kv"}
    engines, mem = {}, {}
    for mode, ct in modes.items():
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        b = B200WhisperBackend(spec, "cuda:0", ct, max_segments=128, max_sequences=320, max_encoder_batch=ENC_BATCH)
        torch.cuda.synchronize()
        free1 = torch.cuda.mem_get_info()[0]
        engines[mode] = b.engine
        st = b.engine.stats()
        mem[mode] = {"free_before_gb": free0 / 1e9, "free_after_gb": free1 / 1e9, "engine_gb": (free0 - free1) / 1e9,
                     "max_segments": st["max_segments"], "max_sequences": st["max_sequences"]}
    dims = engines["bf16"].dims
    lengths = window_lengths(0, 128, "partial")
    audios = [synth_audio(i, lengths[i]) for i in range(128)]
    audio_sec = float(sum(a.size for a in audios)) / 16000.0
    n_steps = dims.n_text_ctx // 2

    res = {m: {"step_128x1_ms": [], "step_64x5_ms": [], "xattn_128x1_us": [], "xattn_128x1_gbs": [], "xattn_64x5_us": [],
               "xattn_64x5_gbs": [], "step_128x1_gb": None, "pipeline_ms": [], "pipeline_audio_s_per_s": []} for m in modes}
    for m, eng in engines.items():  # warm-up: graphs captured, modules loaded
        for seg, grp in ((128, 1), (64, 5)):
            eng.bench_decoder_step(seg, grp, 100, 4)
            eng.bench_cross_attention(seg, grp, 16)
        eng.bench_pipeline(audios, 1, n_steps)
    for rep in range(args.repeats):
        for m, eng in engines.items():
            for seg, grp in ((128, 1), (64, 5)):
                ms, by = eng.bench_decoder_step(seg, grp, 100, 12)
                res[m][f"step_{seg}x{grp}_ms"].append(ms)
                if (seg, grp) == (128, 1):
                    res[m]["step_128x1_gb"] = by / 1e9
                ms, by = eng.bench_cross_attention(seg, grp, 64)
                res[m][f"xattn_{seg}x{grp}_us"].append(ms * 1e3)
                res[m][f"xattn_{seg}x{grp}_gbs"].append(by / ms / 1e6)
            ms = eng.bench_pipeline(audios, 1, n_steps)
            res[m]["pipeline_ms"].append(ms)
            res[m]["pipeline_audio_s_per_s"].append(audio_sec / (ms / 1e3))
            print(m, rep, {k: (v[-1] if isinstance(v, list) else v) for k, v in res[m].items()}, flush=True)
    toks = {m: [r["tokens"] for r in eng.bench_pipeline_results(128, 1, n_steps, None)] for m, eng in engines.items()}
    for m in modes:
        for k in list(res[m]):
            if isinstance(res[m][k], list):
                res[m][k + "_median"] = float(np.median(res[m][k]))
    stage = {}
    for m, eng in engines.items():
        try:
            stage[m] = cross_kv_stage_us(eng, audios[:ENC_BATCH], n_steps=1, int8=(m == "bf16_int8kv"))
        except Exception as exc:  # noqa: BLE001 -- the profiler's event fields differ across torch versions
            stage[m] = f"not measured: {exc!r}"
    a, b = toks["bf16"], toks["bf16_int8kv"]
    lead = [next((k for k in range(min(len(x), len(y))) if x[k] != y[k]), min(len(x), len(y))) for x, y in zip(a, b)]
    agreement = {"windows": len(a), "identical_windows": int(sum(x == y for x, y in zip(a, b))),
                 "leading_token_agreement": float(sum(lead) / max(1, sum(len(x) for x in a))),
                 "tokens_bf16": int(sum(len(x) for x in a)), "tokens_int8kv": int(sum(len(x) for x in b))}
    out = {"gpu": info, "model": "large-v3 (random-init, seed 0)", "time": time.strftime("%Y-%m-%d %H:%M:%S"),
           "audio_seconds_per_pipeline": audio_sec, "pipeline_steps": n_steps, "repeats": args.repeats,
           "engine_memory": mem, "modes": res, "cross_kv_stage_per_window": stage, "pipeline_token_agreement": agreement}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({"gpu": info, "engine_memory": mem, "stage": stage, "agreement": agreement,
                      "medians": {m: {k: v for k, v in res[m].items() if k.endswith("_median")} for m in modes}}, indent=1))


if __name__ == "__main__":
    main()
