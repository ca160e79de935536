"""bench.py's command line and its --dump-outputs files, without a GPU."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_steps_must_be_positive(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse_args()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--warmup", "0", "--dump-outputs", "d"])
    args = bench.parse_args()
    assert args.steps == 7 and args.warmup == 0 and args.dump_outputs == "d"
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--dump-outputs", "d"])
    with pytest.raises(SystemExit):
        bench.parse_args()


def test_dump_outputs_files(tmp_path):
    results = [{"tokens": [5, 6, 7], "sum_logprob": -1.5, "avg_logprob": -0.375, "no_speech_prob": 0.25},
               {"tokens": [], "sum_logprob": -0.5, "avg_logprob": -0.5, "no_speech_prob": 0.5}]
    bench.dump_outputs(str(tmp_path / "out"), results, [2.5, 9.75])
    got = {f[:-4]: np.load(tmp_path / "out" / f) for f in sorted(os.listdir(tmp_path / "out"))}
    assert sorted(got) == ["avg_logprob", "n_tokens", "sum_logprob", "tokens", "window_seconds"]
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    np.testing.assert_array_equal(got["tokens"], [[5, 6, 7], [-1, -1, -1]])
    np.testing.assert_array_equal(got["n_tokens"], [3, 0])
    np.testing.assert_array_equal(got["sum_logprob"], np.float32([-1.5, -0.5]))
    np.testing.assert_array_equal(got["window_seconds"], [2.5, 9.75])
