"""Python face of one GPU engine (thin ctypes layer over the C ABI; no torch in the call path)."""
from __future__ import annotations

import ctypes as C
import threading
from typing import Dict, Optional, Sequence

import numpy as np

from . import _lib as L
from .melfilters import mel_filterbank
from .synth import ModelDims
from .vocab import Vocab, vocab_for


def _as_f32(a) -> np.ndarray:
    if hasattr(a, "detach"):  # torch tensor hand-off
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, dtype=np.float32)


def _as_i16(pcm) -> np.ndarray:
    """bytes / bytearray / memoryview (PCM16 LE, what the gRPC stream carries) or an int16 array"""
    if isinstance(pcm, (bytes, bytearray, memoryview)):
        if len(pcm) % 2:
            raise ValueError("PCM16 byte length must be even")
        return np.frombuffer(pcm, dtype="<i2")
    a = np.asarray(pcm)
    if a.dtype != np.int16:
        raise TypeError(f"PCM16 samples must be int16, got {a.dtype}")
    return np.ascontiguousarray(a.reshape(-1))


def decode_opts(initial: Sequence[int], sot_index: int, beam_size: Optional[int], patience: Optional[float],
                length_penalty: Optional[float], sample_len: int = 0, without_timestamps: bool = False,
                suppress_blank: bool = True, max_initial_timestamp_index: Optional[int] = 50, temperature: float = 0.0,
                best_of: Optional[int] = None, seed: int = 0):
    """bw_decode_opts for one window; returns (struct, objects that must outlive it)."""
    init = (C.c_int32 * len(initial))(*initial)
    beam = int(beam_size or 0)
    # BeamSearchDecoder.max_candidates = round(beam_size * patience) with Python's own round() (half to even), as upstream
    max_cand = max(1, round(beam * float(patience or 1.0))) if beam else 0
    o = L.DecodeOptsC(init, len(initial), sot_index, beam, float(patience or 0.0),
                      -1.0 if length_penalty is None else float(length_penalty), int(sample_len),
                      int(bool(without_timestamps)), int(bool(suppress_blank)),
                      -1 if max_initial_timestamp_index is None else int(max_initial_timestamp_index),
                      float(temperature), int(best_of or 0), int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF, max_cand)
    return o, init


def result_dict(r: "L.ResultC", lang: Optional["L.LangResultC"] = None) -> dict:
    d = {"tokens": list(r.tokens[: r.n_tokens]), "sum_logprob": r.sum_logprob, "avg_logprob": r.avg_logprob,
         "no_speech_prob": r.no_speech_prob, "n_steps": r.n_steps, "t_queue": r.t_queue, "t_encode": r.t_encode,
         "t_decode": r.t_decode}
    if lang is not None:  # a detect-mode decode: the language it chose, as detect_language returns it
        d["language_token"] = lang.language_token
        d["language_probs"] = np.array(lang.probs[: lang.n_languages], dtype=np.float32)
    return d


class Call:
    """One `transcribe()` call: PCM resident on the device + its whole-call log-mel."""

    def __init__(self, engine: "Engine", audio, sample_rate: Optional[int] = None):
        """`audio`: float32 at 16 kHz (sample_rate None), or PCM16 bytes / int16 samples at `sample_rate` Hz
        (converted and resampled on the device)."""
        self.engine = engine
        self._h = C.c_void_p()
        if sample_rate is None:
            audio = _as_f32(audio)
            L.check(engine.lib.bw_call_open(engine.handle, audio.ctypes.data_as(L.c_f32_p), audio.size, C.byref(self._h)),
                    "bw_call_open")
        else:
            pcm = _as_i16(audio)
            engine.ensure_resampler(int(sample_rate))
            L.check(engine.lib.bw_call_open_pcm16(engine.handle, pcm.ctypes.data_as(C.POINTER(C.c_int16)), pcm.size, int(sample_rate),
                                                  C.byref(self._h)), "bw_call_open_pcm16")
        n = C.c_int32()
        L.check(engine.lib.bw_call_content_frames(self._h, C.byref(n)), "bw_call_content_frames")
        self.content_frames = n.value

    def decode(self, seek: int, initial: Sequence[int], sot_index: int, beam_size: Optional[int], patience: Optional[float],
               length_penalty: Optional[float], sample_len: int = 0, without_timestamps: bool = False,
               suppress_blank: bool = True, max_initial_timestamp_index: Optional[int] = 50, temperature: float = 0.0,
               best_of: Optional[int] = None, seed: int = 0) -> dict:
        """One 30 s window.  temperature > 0: GreedyDecoder sampling with `best_of` hypotheses (beam_size must be
        None, as upstream's decode_with_fallback guarantees), reproducible for a given 64-bit `seed`."""
        o, _keep = decode_opts(initial, sot_index, beam_size, patience, length_penalty, sample_len, without_timestamps,
                               suppress_blank, max_initial_timestamp_index, temperature, best_of, seed)
        r = L.ResultC()
        L.check(self.engine.lib.bw_call_decode(self._h, int(seek), C.byref(o), C.byref(r)), "bw_call_decode")
        return result_dict(r)

    def decode_forced(self, seek: int, initial: Sequence[int], sot_index: int, forced: Sequence[int], want_logits: bool = True,
                      without_timestamps: bool = False):
        """Test hook (bw_call_decode_forced): teacher-forced greedy decode through the scheduler; returns
        (result dict, logits [len(forced), V] or None) -- logits[k] is the row step k sampled from."""
        o, _keep = decode_opts(initial, sot_index, None, None, None, 0, without_timestamps, True, 50, 0.0, None, 0)
        f = (C.c_int32 * len(forced))(*forced)
        logits = np.empty((len(forced), self.engine.dims.n_vocab), dtype=np.float32) if want_logits else None
        r = L.ResultC()
        L.check(self.engine.lib.bw_call_decode_forced(self._h, int(seek), C.byref(o), f, len(forced),
                                                      logits.ctypes.data_as(L.c_f32_p) if want_logits else None, C.byref(r)),
                "bw_call_decode_forced")
        return result_dict(r), logits

    def detect_language(self, seek: int = 0):
        r = L.LangResultC()
        L.check(self.engine.lib.bw_call_detect_language(self._h, int(seek), C.byref(r)), "bw_call_detect_language")
        return r.language_token, np.array(r.probs[: r.n_languages], dtype=np.float32)

    def decode_detect(self, seek: int, initial: Sequence[int], sot_index: int, beam_size: Optional[int], patience: Optional[float],
                      length_penalty: Optional[float], sample_len: int = 0, without_timestamps: bool = False,
                      suppress_blank: bool = True, max_initial_timestamp_index: Optional[int] = 50, temperature: float = 0.0,
                      best_of: Optional[int] = None, seed: int = 0) -> dict:
        """decode() of a window that detects its own language (bw_call_decode_detect): `initial` = [sot, LANGUAGE_PLACEHOLDER,
        task, ...] with sot_index 0.  Returns decode()'s dict plus `language_token` and `language_probs` -- what
        detect_language(seek) followed by decode() with that language's sot sequence return, for one encoder pass."""
        o, _keep = decode_opts(initial, sot_index, beam_size, patience, length_penalty, sample_len, without_timestamps,
                               suppress_blank, max_initial_timestamp_index, temperature, best_of, seed)
        r, lang = L.ResultC(), L.LangResultC()
        L.check(self.engine.lib.bw_call_decode_detect(self._h, int(seek), C.byref(o), C.byref(r), C.byref(lang)),
                "bw_call_decode_detect")
        return result_dict(r, lang)

    def close(self) -> None:
        if self._h:
            self.engine.lib.bw_call_close(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Engine:
    """One weight copy + KV pools + scheduler thread on one GPU.  compute: "bf16" (product mode), "bf16_int8kv" (bf16 with the
    cached encoder K/V in 8 bits, BW_FLAG_CROSS_KV_INT8) or "fp32" (validation mode)."""

    # Call.decode_detect / detect windows in decode_many: a window's decode can detect its own language
    detects_in_decode = True

    def __init__(self, dims: ModelDims, state: Dict[str, object], device_index: int = 0, compute: str = "bf16",
                 max_segments: int = 0, max_sequences: int = 0, max_encoder_batch: int = 0, flags: int = 0, max_kv_pages: int = 0):
        self.lib = L.load()
        if self.lib.bw_device_count() <= 0:
            raise L.B200WhisperError("no CUDA device visible: the b200_whisper backend has no CPU fallback")
        self.dims = dims
        self.vocab: Vocab = vocab_for(dims.n_vocab)
        self.compute = compute
        self.device_index = device_index
        self.handle = C.c_void_p()
        self._lock = threading.Lock()
        self._resampler_lock = threading.Lock()
        self._resamplers = set()
        cd = L.ModelDimsC(*[getattr(dims, f) for f, _ in L.ModelDimsC._fields_])
        if compute == "bf16_int8kv":
            flags |= L.BW_FLAG_CROSS_KV_INT8
        cfg = L.EngineConfigC(device_index, L.BW_COMPUTE_FP32 if compute == "fp32" else L.BW_COMPUTE_BF16, max_segments,
                              max_sequences, max_encoder_batch, flags, max_kv_pages)
        L.check(self.lib.bw_engine_create(C.byref(cd), C.byref(cfg), C.byref(self.handle)), "bw_engine_create")
        try:
            self._load(state)
            v = self.vocab
            sup = v.suppress_tokens()
            sup_c = (C.c_int32 * len(sup))(*sup)
            blank = list(v.blank) + [v.eot]
            blank_c = (C.c_int32 * len(blank))(*blank)
            tt = L.TokenTablesC(v.eot, v.sot, v.sot_prev, v.sot_lm, v.no_speech, v.no_timestamps, v.timestamp_begin, v.translate,
                                v.transcribe, v.first_language_token, v.num_languages, sup_c, len(sup), blank_c, len(blank))
            L.check(self.lib.bw_engine_set_tables(self.handle, C.byref(tt)), "bw_engine_set_tables")
            filt = np.ascontiguousarray(mel_filterbank(dims.n_mels), dtype=np.float32)
            L.check(self.lib.bw_engine_set_mel_filters(self.handle, filt.ctypes.data_as(L.c_f32_p)), "bw_engine_set_mel_filters")
            L.check(self.lib.bw_engine_finalize(self.handle), "bw_engine_finalize")
        except Exception:
            self.lib.bw_engine_destroy(self.handle)
            self.handle = C.c_void_p()
            raise

    def _load(self, state: Dict[str, object]) -> None:
        for name, t in state.items():
            if hasattr(t, "detach"):
                import torch

                t = t.detach()
                if t.dtype == torch.bfloat16:
                    arr = t.contiguous().cpu().view(torch.int16).numpy()
                    dtype = L.BW_BF16
                elif t.dtype == torch.float16:
                    arr = t.contiguous().cpu().view(torch.int16).numpy()
                    dtype = L.BW_F16
                else:
                    arr = t.to(torch.float32).contiguous().cpu().numpy()
                    dtype = L.BW_F32
            else:
                arr = np.ascontiguousarray(t, dtype=np.float32)
                dtype = L.BW_F32
            if arr.ndim > 4:
                raise ValueError(f"{name}: rank {arr.ndim} tensor")
            shape = (C.c_int64 * 4)(*(list(arr.shape) + [1] * (4 - arr.ndim)))
            desc = L.TensorDescC(name.encode(), arr.ctypes.data_as(C.c_void_p), dtype, arr.ndim, shape)
            L.check(self.lib.bw_engine_load_weights(self.handle, C.byref(desc), 1), f"bw_engine_load_weights({name})")

    # ---- stage-level ----
    def mel(self, audio, padding: int = 0) -> np.ndarray:
        audio = _as_f32(audio)
        frames = (audio.size + padding) // 160
        out = np.empty((self.dims.n_mels, frames), dtype=np.float32)
        n = C.c_int32()
        L.check(self.lib.bw_mel(self.handle, audio.ctypes.data_as(L.c_f32_p), audio.size, padding, out.ctypes.data_as(L.c_f32_p),
                                C.byref(n)), "bw_mel")
        assert n.value == frames
        return out

    def encode(self, mel) -> np.ndarray:
        mel = _as_f32(mel)
        if mel.ndim == 2:
            mel = mel[None]
        b = mel.shape[0]
        assert mel.shape[1:] == (self.dims.n_mels, 3000), mel.shape
        out = np.empty((b, 1500, self.dims.n_audio_state), dtype=np.float32)
        L.check(self.lib.bw_encode(self.handle, mel.ctypes.data_as(L.c_f32_p), b, out.ctypes.data_as(L.c_f32_p)), "bw_encode")
        return out

    def decode_logits(self, mel_window, tokens: Sequence[int]) -> np.ndarray:
        mel = _as_f32(mel_window)
        assert mel.shape == (self.dims.n_mels, 3000)
        toks = (C.c_int32 * len(tokens))(*tokens)
        out = np.empty((len(tokens), self.dims.n_vocab), dtype=np.float32)
        L.check(self.lib.bw_decode_logits(self.handle, mel.ctypes.data_as(L.c_f32_p), toks, len(tokens), out.ctypes.data_as(L.c_f32_p)),
                "bw_decode_logits")
        return out

    def open_call(self, audio, sample_rate: Optional[int] = None) -> Call:
        return Call(self, audio, sample_rate)

    def decode_many(self, items: Sequence[tuple]) -> list:
        """One blocking bw_decode_many for a batch of windows.  items[i] = (call, seek, kwargs of decode_opts); returns a
        list of result dicts, or the B200WhisperError of the window that failed, in input order.  A window whose kwargs
        carry detect=True is a Call.decode_detect window (bw_decode_many_detect): its dict has the language too."""
        n = len(items)
        if n == 0:
            return []
        calls = (C.c_void_p * n)(*[it[0]._h for it in items])
        seeks = (C.c_int32 * n)(*[int(it[1]) for it in items])
        opts = (L.DecodeOptsC * n)()
        keep = []
        detect = []
        for i, it in enumerate(items):
            kw = dict(it[2])
            detect.append(bool(kw.pop("detect", False)))
            o, k = decode_opts(**kw)
            opts[i] = o
            keep.append(k)
        results = (L.ResultC * n)()
        statuses = (C.c_int32 * n)()
        langs = (L.LangResultC * n)() if any(detect) else None
        if langs is None:
            st = self.lib.bw_decode_many(calls, seeks, opts, results, statuses, n)
        else:
            st = self.lib.bw_decode_many_detect(calls, seeks, opts, results, langs, statuses, n)
        if st != 0 and all(s == 0 for s in statuses):
            L.check(st, "bw_decode_many")
        out = []
        for i in range(n):
            if statuses[i] != 0:
                msg = self.lib.bw_last_error()
                out.append(L.B200WhisperError(f"bw_decode_many window {i} failed (bw_status {statuses[i]}): "
                                              f"{msg.decode('utf-8', 'replace') if msg else ''}"))
            else:
                out.append(result_dict(results[i], langs[i] if detect[i] else None))
        return out

    def stats(self) -> Dict[str, int]:
        buf = (C.c_int64 * len(L.STAT_NAMES))()
        L.check(self.lib.bw_engine_stats(self.handle, buf, len(L.STAT_NAMES)), "bw_engine_stats")
        return dict(zip(L.STAT_NAMES, list(buf)))

    # ---- timing helpers used by bench.py (CUDA events inside the library) ----
    def _bench(self, fn, *args):
        ms, q = C.c_float(), C.c_double()
        L.check(fn(self.handle, *args, C.byref(ms), C.byref(q)), fn.__name__)
        return ms.value, q.value

    def bench_mel(self, n_samples: int, iters: int):
        return self._bench(self.lib.bw_bench_mel, C.c_int64(n_samples), iters)

    def bench_encoder(self, batch: int, iters: int):
        return self._bench(self.lib.bw_bench_encoder, batch, iters)

    def bench_cross_attention(self, n_segments: int, n_group: int, iters: int):
        return self._bench(self.lib.bw_bench_cross_attention, n_segments, n_group, iters)

    def bench_decoder_step(self, n_segments: int, n_group: int, context_len: int, iters: int):
        return self._bench(self.lib.bw_bench_decoder_step, n_segments, n_group, context_len, iters)

    def ensure_resampler(self, sample_rate: int) -> None:
        """Register the ensure_16k filter bank of `sample_rate` with the engine (once per rate)."""
        if sample_rate == 16000:
            return
        with self._resampler_lock:
            if sample_rate in self._resamplers:
                return
            from .ingest import resample_taps

            orig, new, width, taps = resample_taps(sample_rate)
            L.check(self.lib.bw_engine_set_resampler(self.handle, sample_rate, orig, new, width, taps.ctypes.data_as(L.c_f32_p)),
                    "bw_engine_set_resampler")
            self._resamplers.add(sample_rate)

    def resample_pcm16(self, pcm, sample_rate: int) -> np.ndarray:
        """Stage-level: PCM16 at `sample_rate` -> float32 at 16 kHz, computed on the device."""
        from .ingest import resampled_length

        pcm = _as_i16(pcm)
        self.ensure_resampler(int(sample_rate))
        out = np.empty(resampled_length(pcm.size, sample_rate), dtype=np.float32)
        n = C.c_int64()
        L.check(self.lib.bw_resample_pcm16(self.handle, pcm.ctypes.data_as(C.POINTER(C.c_int16)), pcm.size, int(sample_rate),
                                           out.ctypes.data_as(L.c_f32_p), C.byref(n)), "bw_resample_pcm16")
        assert n.value == out.size, (n.value, out.size)
        return out

    def trace_begin(self) -> None:
        """Arm the debug timeline (run with B200W_NO_GRAPH=1)."""
        L.check(self.lib.bw_debug_trace(self.handle, 1, None, 0, None), "bw_debug_trace")

    def trace_end(self, cap: int = 1 << 16) -> np.ndarray:
        """Disarm the timeline; returns records [n, 2] uint64: (smid << 32 | kernel << 24 | grid.x << 8 | phase, ns)."""
        out = np.zeros((cap, 2), dtype=np.uint64)
        n = C.c_int32()
        L.check(self.lib.bw_debug_trace(self.handle, 0, out.ctypes.data_as(C.POINTER(C.c_uint64)), cap, C.byref(n)), "bw_debug_trace")
        return out[: n.value]

    def bench_pipeline(self, audios, n_group: int, n_steps: int) -> float:
        """Device-timed ms for mel -> encoder -> cross-KV -> n_steps decoder steps over `audios` (resident PCM)."""
        audios = [_as_f32(a) for a in audios]
        flat = np.ascontiguousarray(np.concatenate(audios))
        lengths = (C.c_int64 * len(audios))(*[a.size for a in audios])
        offs = np.cumsum([0] + [a.size for a in audios[:-1]])
        offsets = (C.c_int64 * len(audios))(*[int(o) for o in offs])
        ms = C.c_float()
        L.check(self.lib.bw_bench_pipeline(self.handle, flat.ctypes.data_as(L.c_f32_p), offsets, lengths, len(audios), n_group,
                                           n_steps, C.byref(ms)), "bw_bench_pipeline")
        return ms.value

    def bench_pipeline_results(self, n_segments: int, n_group: int, n_steps: int, length_penalty: Optional[float]) -> list:
        """Result dicts (as decode_many returns them) of every window of the last bench_pipeline call with these arguments."""
        results = (L.ResultC * n_segments)()
        L.check(self.lib.bw_bench_pipeline_results(self.handle, n_segments, n_group, n_steps,
                                                   -1.0 if length_penalty is None else float(length_penalty), results),
                "bw_bench_pipeline_results")
        return [result_dict(r) for r in results]

    def retain(self) -> None:
        self.lib.bw_engine_retain(self.handle)

    def close(self) -> None:
        with self._lock:
            if self.handle:
                self.lib.bw_engine_destroy(self.handle)
                self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
