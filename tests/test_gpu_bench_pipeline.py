"""The timed pipeline behind bench.py's `value` (bw_bench_pipeline) and what it decoded (bw_bench_pipeline_results,
what `bench.py --dump-outputs` writes): one result per window, each belonging to its own window, and the same on a
second run."""
import numpy as np
import pytest

from b200_whisper.backend import B200WhisperBackend
from b200_whisper.synth import synth_audio

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

N_STEPS = 24


def _decoded(rs):
    # no_speech_prob is left out: the pipeline starts decoding after the prompt and never computes one (NaN)
    return [(r["tokens"], r["sum_logprob"]) for r in rs]


@pytest.mark.parametrize("n_group", [1, 5])
def test_pipeline_results_belong_to_their_windows(n_group):
    be = B200WhisperBackend("random:test-tiny:0:0.1", "cuda:0", "bfloat16", max_segments=4, max_sequences=20)
    eng = be.engine
    audios = [synth_audio(70 + i, s) for i, s in enumerate((2.0, 6.0, 10.0))]

    def run(windows):
        assert eng.bench_pipeline(windows, n_group, N_STEPS) > 0
        return eng.bench_pipeline_results(len(windows), n_group, N_STEPS, 1.0)

    first, second = run(audios), run(audios)
    assert len(first) == len(audios) and _decoded(first) == _decoded(second)
    for r in first:
        assert len(r["tokens"]) <= N_STEPS and r["n_steps"] == N_STEPS
        assert all(0 <= t < eng.dims.n_vocab for t in r["tokens"])
        assert np.isfinite(r["sum_logprob"]) and r["sum_logprob"] <= 0
    # different audio decodes differently: a result read from the wrong slot could not pass the checks below
    lps = [r["sum_logprob"] for r in first]
    assert min(abs(a - b) for i, a in enumerate(lps) for b in lps[i + 1:]) > 1e-2, lps
    # the same windows in reverse order: the same shapes, so result i of the reversed batch is window n - 1 - i's
    rev = run(audios[::-1])[::-1]
    for i, (a, b) in enumerate(zip(first, rev)):
        assert a["tokens"] == b["tokens"] and abs(a["sum_logprob"] - b["sum_logprob"]) < 1e-3, (i, a, b)
    # each window alone: the token stream survives the batch, the log-probability moves in its last bits at most
    # (the tolerance of tests/test_gpu_bf16_decode.py's batch-invariance check, per token)
    for i, a in enumerate(audios):
        (b,) = run([a])
        r = first[i]
        assert r["tokens"] == b["tokens"], i
        assert abs(r["sum_logprob"] - b["sum_logprob"]) < 3e-2 * (len(r["tokens"]) + 1), (i, r["sum_logprob"], b["sum_logprob"])
