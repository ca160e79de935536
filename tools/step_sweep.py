"""Decoder-step time over batch shapes (run once with and once without B200W_NO_GRAPH=1 for the graph/eager A-B).
Usage: python tools/step_sweep.py [model]      (SWEEP_SHAPES=128x1,64x5 SWEEP_CTX=100,200 narrow the sweep)"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from b200_whisper.backend import B200WhisperBackend  # noqa: E402

model = sys.argv[1] if len(sys.argv) > 1 else "large-v3"
b = B200WhisperBackend(f"random:{model}:0:0.1", "cuda:0", "bfloat16", max_segments=128, max_sequences=320, max_encoder_batch=1)
eng = b.engine
mode = "eager" if os.environ.get("B200W_NO_GRAPH") else "graph"
shapes = ((1, 1), (8, 1), (32, 1), (64, 1), (128, 1), (1, 5), (16, 5), (64, 5))
if os.environ.get("SWEEP_SHAPES"):
    shapes = tuple(tuple(int(v) for v in s.split("x")) for s in os.environ["SWEEP_SHAPES"].split(","))
ctxs = tuple(int(v) for v in os.environ.get("SWEEP_CTX", "20,100,200").split(","))
for seg, grp in shapes:
    for ctx in ctxs:
        eng.bench_decoder_step(seg, grp, ctx, 4)  # the shape's CUDA graph is captured at its third sighting: not in the timed run
        ms, by = eng.bench_decoder_step(seg, grp, ctx, 12)
        print(f"{mode} step {seg:3d} x {grp}  ctx {ctx:3d}: {ms:7.3f} ms  {by / ms / 1e6:7.1f} GB/s  ({by / ms / 1e6 / 6546.6 * 100:4.1f} % of HBM)", flush=True)
