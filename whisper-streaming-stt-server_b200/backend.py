"""`B200WhisperBackend` -- the drop-in `ModelBackend` for `--model-backend b200_whisper`.

Mirrors the reference's backend interface (stt_server/model/backends/base.py:24-35): same constructor
`(model_size, device, compute_type)`, same `transcribe(audio, options) -> (List[Segment], BackendInfo)`,
same option handling and result mapping as `TorchWhisperBackend`
(stt_server/model/backends/torch_whisper.py:49-110), whose semantics are this backend's parity target.
The host side keeps upstream `whisper.transcribe`'s seek loop and segment assembly in Python (the
reference's host language); mel, encoder and the batched decoder run in libb200whisper.so.

Temperature: a scalar or upstream's fallback ladder (tuple) -- `decode_with_fallback` of upstream transcribe.py:
rungs above 0 sample `best_of` hypotheses on the device (Categorical(logits / T) by Gumbel-max, counter-based
generator), beam search only runs at temperature 0.  Draws are reproducible for a given seed
(`B200_WHISPER_SEED`, else one random seed per backend instance), not equal to torch's global generator.

Deviations, all explicit:
* `word_timestamps` (DTW alignment) is accepted and ignored; `initial_prompt` needs the tokenizer rank
  file (`B200_WHISPER_VOCAB_DIR`) and is dropped with a warning without it;
* like torch_whisper, `without_timestamps` is converted to `word_timestamps` and so does NOT disable
  timestamp tokens, unless B200_WHISPER_HONOR_WITHOUT_TIMESTAMPS=1 (faster_whisper-like behaviour).
"""
from __future__ import annotations

import atexit
import itertools
import logging
import os
import threading
import zlib
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np

from ._lib import LANGUAGE_PLACEHOLDER
from .engine import Engine
from .synth import MODEL_DIMS, LazyRandomState, ModelDims, random_state_dict
from .vocab import Detokenizer, Vocab, normalize_language, vocab_for

LOGGER = logging.getLogger("stt_server.model_backend")

try:  # use the server's own dataclasses when running inside it
    from stt_server.model.backends.base import BackendInfo, Segment  # type: ignore
except Exception:  # pragma: no cover - exercised when the reference is not importable

    @dataclass(frozen=True)
    class Segment:  # stt_server/model/backends/base.py:7-13
        start: float
        end: float
        text: str

    @dataclass(frozen=True)
    class BackendInfo:  # stt_server/model/backends/base.py:16-21
        language: str
        language_probability: float


N_FRAMES = 3000
HOP_LENGTH = 160
SAMPLE_RATE = 16000
FP32_ALIASES = {"float32", "fp32"}
BF16_ALIASES = {"bfloat16", "bf16", "default", "auto"}
# compute types the reference's backends give another meaning to (torch_whisper.py:36-47: fp16 aliases -> .half(), int8* ->
# float32; faster_whisper: CTranslate2 quantisation).  This engine has no fp16 or int8-weight mode, so they run as bfloat16 -- loudly.
REMAPPED_TO_BF16 = {"float16", "fp16", "half", "int8", "int8_float16", "int8_bfloat16", "int8_float32"}
# bfloat16 with the cached encoder K/V (cross-attention) in 8 bits: half the decoder step's bytes, not bf16-exact
BF16_INT8KV_ALIASES = {"bfloat16_int8kv", "bf16_int8kv"}
_REMAP_WARNED: set = set()

SUPPORTED_OPTIONS = {  # torch_whisper.py:79-97
    "temperature", "compression_ratio_threshold", "logprob_threshold", "no_speech_threshold",
    "condition_on_previous_text", "initial_prompt", "word_timestamps", "prepend_punctuations",
    "append_punctuations", "language", "task", "beam_size", "best_of", "patience", "length_penalty", "fp16", "prompt",
}

_ENGINES: Dict[tuple, Engine] = {}
_ENGINES_LOCK = threading.Lock()
_INSTANCE_COUNTER = itertools.count()
_M64 = (1 << 64) - 1


def window_seed(base_seed: int, seek: int, attempt: int) -> int:
    """Seed of one decode attempt: window at mel frame `seek`, rung `attempt` of the temperature ladder."""
    return (base_seed + 0x632BE59BD9B4E019 * (seek + 1) + 0xD1342543DE82EF95 * (attempt + 1)) & _M64


def _close_engines() -> None:
    with _ENGINES_LOCK:
        for e in _ENGINES.values():
            try:
                e.close()
            except Exception:
                pass
        _ENGINES.clear()


atexit.register(_close_engines)


def parse_device(device: str, instance_index: int) -> int:
    """`cuda` / `cuda:N` -> ordinal; `cuda:auto` spreads pool handles round-robin over the visible GPUs
    (SURVEY.md section 8e option B).  Anything else is refused: there is no CPU path."""
    dev = (device or "cuda").lower()
    if not dev.startswith("cuda"):
        raise ValueError(f"b200_whisper backend needs a CUDA device, got device={device!r} (no CPU fallback)")
    if dev == "cuda":
        return 0
    suffix = dev.split(":", 1)[1]
    if suffix == "auto":
        from . import _lib

        n = max(1, _lib.load().bw_device_count())
        return instance_index % n
    return int(suffix)


def load_checkpoint(model_size: str) -> Tuple[ModelDims, Dict[str, Any], str]:
    """Resolve `model_size` to (dims, state_dict, canonical name).

    * `random:<name>[:seed[:emb_std[:eot_bias]]]` -- seeded random init (tests / bench; no network here);
    * a path to an openai-whisper `.pt` checkpoint (`{"dims": ..., "model_state_dict": ...}`);
    * a model name looked up as `<name>.pt` under $B200_WHISPER_MODEL_DIR and ~/.cache/whisper
      (where `whisper.load_model`, reference torch_whisper.py:21, caches its downloads).
    """
    if model_size.startswith("random:"):
        parts = model_size.split(":")
        name = parts[1]
        if name not in MODEL_DIMS:
            raise ValueError(f"unknown model name {name!r}")
        seed = int(parts[2]) if len(parts) > 2 else 0
        emb_std = float(parts[3]) if len(parts) > 3 else 0.1
        eot_bias = float(parts[4]) if len(parts) > 4 else 0.0
        # materialised one tensor at a time while the engine loads it (6 GB of host memory per process otherwise)
        return MODEL_DIMS[name], LazyRandomState(MODEL_DIMS[name], seed, emb_std=emb_std, eot_bias=eot_bias), model_size
    candidates = [model_size]
    for root in (os.environ.get("B200_WHISPER_MODEL_DIR"), os.path.expanduser("~/.cache/whisper")):
        if root:
            candidates.append(os.path.join(root, f"{model_size}.pt"))
    for path in candidates:
        if os.path.isfile(path):
            import torch

            # {"dims": dict, "model_state_dict": tensors}: nothing that needs unpickling arbitrary objects (upstream
            # whisper.load_model passes weights_only=True as well)
            ckpt = torch.load(path, map_location="cpu", weights_only=True)
            dims = ModelDims(**{k: int(v) for k, v in ckpt["dims"].items()})
            return dims, ckpt["model_state_dict"], os.path.abspath(path)
    raise RuntimeError(
        f"b200_whisper: no checkpoint for model {model_size!r} (looked at {candidates}); set B200_WHISPER_MODEL_DIR "
        "or pass a .pt path, or use 'random:<name>' for random-init weights")


def get_engine(model_size: str, device_index: int, compute: str, **engine_kwargs) -> Engine:
    """One engine (= one weight copy, one KV pool, one scheduler) per (model, GPU, compute mode); every
    pool handle the reference creates with identical arguments (model_registry.py:230-247) shares it."""
    key = (model_size, device_index, compute)
    with _ENGINES_LOCK:
        eng = _ENGINES.get(key)
        if eng is None:
            dims, state, _ = load_checkpoint(model_size)
            eng = Engine(dims, state, device_index=device_index, compute=compute, **engine_kwargs)
            _ENGINES[key] = eng
        return eng


def compression_ratio(text: str) -> float:
    b = text.encode("utf-8")
    return len(b) / len(zlib.compress(b))


class B200WhisperBackend:
    """Backend wrapper for the B200-native engine (see module docstring)."""

    def __init__(self, model_size: str, device: str, compute_type: str, **engine_kwargs) -> None:
        self.model_size = model_size
        self.device = device
        self.compute_type = compute_type
        ct = (compute_type or "default").lower()
        if ct in FP32_ALIASES:
            self.compute = "fp32"
        elif ct in BF16_INT8KV_ALIASES:
            self.compute = "bf16_int8kv"
        else:
            if ct in REMAPPED_TO_BF16:
                if ct not in _REMAP_WARNED:
                    _REMAP_WARNED.add(ct)
                    LOGGER.warning("b200_whisper: compute_type=%s runs as bfloat16 (bf16 storage, fp32 accumulate); the engine has "
                                   "no fp16 / int8 mode -- pass float32 for the validation mode", compute_type)
            elif ct not in BF16_ALIASES:
                LOGGER.warning("Unsupported compute_type=%s for b200_whisper; using bfloat16", compute_type)
            self.compute = "bf16"
        self._instance = next(_INSTANCE_COUNTER)
        self.device_index = parse_device(device, self._instance)
        self.engine = get_engine(model_size, self.device_index, self.compute, **engine_kwargs)
        self.vocab: Vocab = self.engine.vocab
        # A real checkpoint without its tokenizer rank file would hand `<id>` placeholders to clients: refuse to load.
        # Random-init models (tests / bench) and an explicit opt-in keep the placeholder renderer.
        allow_placeholders = model_size.startswith("random:") or os.environ.get("B200_WHISPER_ALLOW_PLACEHOLDER_TEXT", "0") == "1"
        self.detok = Detokenizer(self.vocab, allow_placeholders=allow_placeholders)
        # decode_with_fallback's repetitiveness check (compression ratio of the TEXT) is meaningless on `<id>` placeholders
        self.check_compression_ratio = self.detok.has_text
        self.honor_without_timestamps = os.environ.get("B200_WHISPER_HONOR_WITHOUT_TIMESTAMPS", "0") == "1"
        self.report_language_probability = os.environ.get("B200_WHISPER_REPORT_LANGUAGE_PROB", "0") == "1"
        self.last_language_probability: Optional[float] = None
        # language unset: detect it inside the first window's decode (one encoder pass) where the engine can; False runs
        # upstream's separate detect_language pass first, as engines without that capability do
        self.detect_in_decode = bool(getattr(self.engine, "detects_in_decode", False))
        env_seed = os.environ.get("B200_WHISPER_SEED")
        self.base_seed = int(env_seed) & _M64 if env_seed else int.from_bytes(os.urandom(8), "little")
        self._call_counter = itertools.count()
        LOGGER.info("b200_whisper loaded model=%s device=cuda:%d compute=%s", model_size, self.device_index, self.compute)

    # ---- torch_whisper.py:78-110 ----
    def _normalize_options(self, options: Dict[str, Any]) -> Dict[str, Any]:
        opts = dict(options)
        if "log_prob_threshold" in opts and "logprob_threshold" not in opts:
            opts["logprob_threshold"] = opts.pop("log_prob_threshold")
        without_ts = False
        if "without_timestamps" in opts and "word_timestamps" not in opts:
            without_ts = bool(opts.pop("without_timestamps"))
            opts["word_timestamps"] = not without_ts
        dropped = {k: v for k, v in opts.items() if k not in SUPPORTED_OPTIONS}
        for key, value in dropped.items():
            LOGGER.warning("Dropping unsupported b200_whisper option %s=%s", key, value)
            opts.pop(key, None)
        if self.honor_without_timestamps and without_ts:
            opts["_without_timestamps"] = True
        return opts

    def transcribe(self, audio: Any, options: Dict[str, Any]) -> Tuple[List[Segment], BackendInfo]:
        opts = self._normalize_options(options)
        result = self.transcribe_raw(audio, **opts)
        return self._to_segments(result)

    def transcribe_pcm16(self, pcm: Any, sample_rate: int, options: Dict[str, Any]) -> Tuple[List[Segment], BackendInfo]:
        """Side door for the raw stream bytes (SURVEY 8(f).2): `pcm` = PCM16 LE mono bytes (or an int16 array) at
        `sample_rate` Hz, exactly what `ModelWorker._decode` receives (worker.py:98-121).  `pcm16_to_float32` and
        `ensure_16k` (utils/audio.py:6-30) run on the device in front of the log-mel kernel; results are the ones
        `transcribe(ensure_16k(pcm16_to_float32(pcm), sample_rate), options)` gives."""
        if int(sample_rate) != sample_rate or int(sample_rate) <= 0:
            raise ValueError(f"sample_rate must be a positive integer, got {sample_rate!r}")
        opts = self._normalize_options(options)
        result = self.transcribe_raw(pcm, _sample_rate=int(sample_rate), **opts)
        return self._to_segments(result)

    def transcribe_many(self, audios: Sequence[Any], options: Any, sample_rates: Optional[Sequence[Optional[int]]] = None
                        ) -> List[Tuple[List[Segment], BackendInfo]]:
        """Explicit cross-session batch at the registry seam (SURVEY 8(f).3): what the reference declares as
        `decode_batch_window_ms` / `max_decode_batch_size` (config/server.yaml:48-49) but never implements.  All
        calls are handed to the engine together, so their windows share encoder launches and every decoder step;
        one worker thread can serve a whole batch instead of one pool handle per concurrent decode.
        `options`: one dict for all, or one per audio.  `sample_rates[i]` not None -> audios[i] is PCM16 at that rate.
        Returns results in input order; the first failure is raised after all calls have finished."""
        n = len(audios)
        opt_list = [options] * n if isinstance(options, dict) else list(options)
        rates = [None] * n if sample_rates is None else list(sample_rates)
        if len(opt_list) != n or len(rates) != n:
            raise ValueError("options / sample_rates must match audios in length")
        results: List[Any] = [None] * n
        errors: List[Optional[BaseException]] = [None] * n
        gens: List[Any] = [None] * n
        pending: Dict[int, tuple] = {}

        def advance(i: int, step) -> None:
            """run item i's seek loop up to its next window; `step` starts / resumes the generator"""
            try:
                pending[i] = step()
            except StopIteration as stop:
                pending.pop(i, None)
                results[i] = self._to_segments(stop.value)
            except Exception as exc:  # noqa: BLE001 - re-raised below, after every item has finished
                pending.pop(i, None)
                errors[i] = exc

        for i in range(n):
            def start(i=i):
                opts = self._normalize_options(opt_list[i])
                if rates[i] is not None:
                    if int(rates[i]) != rates[i] or int(rates[i]) <= 0:
                        raise ValueError(f"sample_rate must be a positive integer, got {rates[i]!r}")
                    opts["_sample_rate"] = int(rates[i])
                gens[i] = self._transcribe_steps(audios[i], **opts)
                return next(gens[i])
            advance(i, start)
        # One host thread: every round hands the next window of every unfinished item to the engine in ONE blocking
        # bw_decode_many, so the windows share encoder launches and every decoder step (no thread per item).
        while pending:
            idx = sorted(pending)
            outs = self.engine.decode_many([pending[i] for i in idx])
            for i, out in zip(idx, outs):
                if isinstance(out, BaseException):
                    advance(i, lambda i=i, out=out: gens[i].throw(out))
                else:
                    advance(i, lambda i=i, out=out: gens[i].send(out))
        for exc in errors:
            if exc is not None:
                raise exc
        return results

    def _to_segments(self, result: dict) -> Tuple[List[Segment], BackendInfo]:
        segments: List[Segment] = []
        for seg in result.get("segments", []):  # same defensive mapping as torch_whisper.py:56-75
            if not isinstance(seg, dict):
                continue

            def as_float(value: Any) -> float:
                try:
                    return float(value)
                except (TypeError, ValueError):
                    return 0.0

            segments.append(Segment(as_float(seg.get("start", 0.0)), as_float(seg.get("end", 0.0)), str(seg.get("text", "") or "")))
        language = result.get("language") or ""
        if not isinstance(language, str):
            language = str(language)
        # parity with torch_whisper.py:76: the probability is reported as -1.0 ("unknown"); the detected
        # value stays available as `last_language_probability` (B200_WHISPER_REPORT_LANGUAGE_PROB=1 returns it)
        self.last_language_probability = result.get("language_probability")
        prob = -1.0
        if self.report_language_probability and self.last_language_probability is not None:
            prob = float(self.last_language_probability)
        return segments, BackendInfo(language, prob)

    def transcribe_raw(self, audio: Any, **opts) -> dict:
        """upstream whisper.transcribe() over the engine: one blocking bw_call_decode per window"""
        gen = self._transcribe_steps(audio, **opts)
        try:
            call, seek, kw = next(gen)
            while True:
                kw = dict(kw)
                res = call.decode_detect(seek, **kw) if kw.pop("detect", False) else call.decode(seek, **kw)
                call, seek, kw = gen.send(res)
        except StopIteration as stop:
            return stop.value

    # ---- upstream whisper/transcribe.py seek loop; a generator that yields one (call, seek, decode arguments) per window
    # and is sent the window's result, so that one thread can drive many calls in lockstep (transcribe_many) ----
    def _transcribe_steps(self, audio: Any, *, temperature: Any = 0.0, compression_ratio_threshold: Optional[float] = 2.4,
                       logprob_threshold: Optional[float] = -1.0, no_speech_threshold: Optional[float] = 0.6,
                       condition_on_previous_text: bool = True, initial_prompt: Optional[str] = None,
                       language: Optional[str] = None, task: Optional[str] = None, beam_size: Optional[int] = None,
                       best_of: Optional[int] = None, patience: Optional[float] = None,
                          length_penalty: Optional[float] = None, sample_len: Optional[int] = None, **ignored):
        v = self.vocab
        sample_rate = ignored.pop("_sample_rate", None)  # not None: `audio` is PCM16 at that rate (transcribe_pcm16)
        if sample_rate is None:
            if hasattr(audio, "detach"):
                audio = audio.detach().cpu().numpy()
            audio = np.ascontiguousarray(audio, dtype=np.float32).reshape(-1)
            n_in = audio.size
        else:
            n_in = len(audio) // 2 if isinstance(audio, (bytes, bytearray, memoryview)) else int(np.asarray(audio).size)
        if n_in == 0:
            return {"text": "", "segments": [], "language": language or "", "language_probability": None}
        temperatures = [float(t) for t in temperature] if isinstance(temperature, (list, tuple)) else [float(temperature or 0.0)]
        if not temperatures:
            temperatures = [0.0]
        if any(t < 0 or t != t for t in temperatures):
            raise ValueError(f"temperature must be >= 0, got {temperature!r}")
        seed = ignored.pop("_seed", None)
        # distinct calls of one backend draw from distinct streams; an explicit `_seed` (tests) pins the call
        call_seed = int(seed) & _M64 if seed is not None else (self.base_seed + 0xA0761D6478BD642F * (next(self._call_counter) + 1)) & _M64
        without_ts = bool(ignored.get("_without_timestamps", False))
        beam = int(beam_size) if beam_size is not None else None
        if beam is not None and not (1 <= beam <= 8):
            raise ValueError(f"beam_size must be in [1, 8], got {beam_size}")
        n_best = int(best_of) if best_of is not None else None
        if n_best is not None and not (1 <= n_best <= 8):
            raise ValueError(f"best_of must be in [1, 8], got {best_of}")

        with self.engine.open_call(audio, sample_rate) as call:
            content_frames = call.content_frames
            language_probability = None
            # Language unset on a multilingual model: upstream detects it once per call on the window at seek 0.  When
            # nothing precedes that window's <|sot|> (no initial_prompt), its first decode attempt detects the language
            # itself (Call.decode_detect: one encoder pass for both); otherwise -- or with detect_in_decode off -- a
            # separate detect_language pass runs first.
            detect_first = False
            if language is None:
                if not v.multilingual:
                    language = "en"
                elif initial_prompt is None and content_frames > 0 and self.detect_in_decode:
                    detect_first = True
                else:
                    tok, probs = call.detect_language(0)
                    language = v.language_of_token(tok)
                    language_probability = float(probs[tok - v.first_language_token])
            else:
                language = normalize_language(language)

            def sot_sequence_of(lang: Optional[str]) -> List[int]:
                seq = v.sot_sequence(lang, task)
                return seq + [v.no_timestamps] if without_ts else seq

            sot_sequence = sot_sequence_of(language)
            n_ctx = self.engine.dims.n_text_ctx

            all_tokens: List[int] = []
            if initial_prompt is not None:
                enc = self.detok.encode(" " + initial_prompt.strip())
                if enc is None:  # placeholder mode only (random-init models / explicit opt-in): there is no text codec
                    LOGGER.warning("b200_whisper: initial_prompt dropped (placeholder text mode, no tokenizer rank file)")
                else:
                    all_tokens.extend(enc)
            n_initial_prompt = len(all_tokens)
            all_segments: List[dict] = []
            prompt_reset_since = 0
            seek = 0
            input_stride = 2
            time_precision = 0.02
            while seek < content_frames:
                time_offset = float(seek * HOP_LENGTH / SAMPLE_RATE)
                segment_size = min(N_FRAMES, content_frames - seek)
                segment_duration = segment_size * HOP_LENGTH / SAMPLE_RATE
                prompt = all_tokens[prompt_reset_since:]
                initial = list(sot_sequence)
                if prompt:
                    initial = [v.sot_prev] + prompt[-(n_ctx // 2 - 1):] + initial
                # sample_len: upstream DecodingOptions.sample_len (default n_text_ctx // 2); not reachable through
                # transcribe() -- torch_whisper.py:78-110 drops it -- but tools use it to bound synthetic decodes
                # decode_with_fallback (upstream transcribe.py): walk the temperature ladder until a rung passes the
                # compression-ratio / log-probability checks; beam search at T = 0, best_of samples above it
                for attempt, t in enumerate(temperatures):
                    kw = dict(initial=initial, sot_index=initial.index(v.sot), beam_size=beam, patience=patience,
                              length_penalty=length_penalty, sample_len=int(sample_len or 0), without_timestamps=without_ts)
                    if t > 0:
                        kw.update(beam_size=None, patience=None, temperature=t, best_of=n_best, seed=window_seed(call_seed, seek, attempt))
                    if detect_first:  # the first window has no prompt: initial == sot_sequence, sot at index 0
                        kw.update(initial=[v.sot, LANGUAGE_PLACEHOLDER] + initial[2:], detect=True)
                    res = dict((yield call, seek, kw))
                    if detect_first:  # later rungs and windows decode with the detected language, as upstream's
                        detect_first = False
                        tok = res.pop("language_token")
                        language = v.language_of_token(tok)
                        language_probability = float(res.pop("language_probs")[tok - v.first_language_token])
                        sot_sequence = sot_sequence_of(language)
                        initial = list(sot_sequence)
                    res["temperature"] = t
                    text_all = self.detok.decode([tk for tk in res["tokens"] if tk < v.eot]).strip()
                    res["compression_ratio"] = compression_ratio(text_all)
                    needs_fallback = False
                    # (placeholder renderer: `<id>` strings say nothing about repetitiveness -- the check needs real text)
                    if (compression_ratio_threshold is not None and self.check_compression_ratio
                            and res["compression_ratio"] > compression_ratio_threshold):
                        needs_fallback = True  # too repetitive
                    if logprob_threshold is not None and res["avg_logprob"] < logprob_threshold:
                        needs_fallback = True  # average log probability is too low
                    if (no_speech_threshold is not None and res["no_speech_prob"] > no_speech_threshold
                            and logprob_threshold is not None and res["avg_logprob"] < logprob_threshold):
                        needs_fallback = False  # silence
                    if not needs_fallback:
                        break
                tokens: List[int] = res["tokens"]
                if no_speech_threshold is not None:
                    should_skip = res["no_speech_prob"] > no_speech_threshold
                    if logprob_threshold is not None and res["avg_logprob"] > logprob_threshold:
                        should_skip = False
                    if should_skip:
                        seek += segment_size
                        continue
                cr = res["compression_ratio"]

                def new_segment(start: float, end: float, toks: Sequence[int]) -> dict:
                    return {"seek": seek, "start": start, "end": end,
                            "text": self.detok.decode([t for t in toks if t < v.eot]), "tokens": list(toks),
                            "temperature": res["temperature"], "avg_logprob": res["avg_logprob"], "compression_ratio": cr,
                            "no_speech_prob": res["no_speech_prob"]}

                current: List[dict] = []
                is_ts = [t >= v.timestamp_begin for t in tokens]
                single_timestamp_ending = is_ts[-2:] == [False, True]
                consecutive = [i + 1 for i in range(len(tokens) - 1) if is_ts[i] and is_ts[i + 1]]
                if consecutive:
                    slices = list(consecutive)
                    if single_timestamp_ending:
                        slices.append(len(tokens))
                    last_slice = 0
                    for cur_slice in slices:
                        sliced = tokens[last_slice:cur_slice]
                        start_pos = sliced[0] - v.timestamp_begin
                        end_pos = sliced[-1] - v.timestamp_begin
                        current.append(new_segment(time_offset + start_pos * time_precision,
                                                   time_offset + end_pos * time_precision, sliced))
                        last_slice = cur_slice
                    if single_timestamp_ending:
                        seek += segment_size
                    else:
                        seek += (tokens[last_slice - 1] - v.timestamp_begin) * input_stride
                else:
                    duration = segment_duration
                    stamps = [t for t in tokens if t >= v.timestamp_begin]
                    if stamps and stamps[-1] != v.timestamp_begin:
                        duration = (stamps[-1] - v.timestamp_begin) * time_precision
                    current.append(new_segment(time_offset, time_offset + duration, tokens))
                    seek += segment_size
                for seg in current:
                    if seg["start"] == seg["end"] or seg["text"].strip() == "":
                        seg["text"] = ""
                        seg["tokens"] = []
                all_segments.extend({"id": i, **seg} for i, seg in enumerate(current, start=len(all_segments)))
                all_tokens.extend(t for seg in current for t in seg["tokens"])
                if not condition_on_previous_text or res["temperature"] > 0.5:
                    prompt_reset_since = len(all_tokens)  # do not feed the prompt tokens if a high temperature was used
        return {"text": self.detok.decode(all_tokens[n_initial_prompt:]), "segments": all_segments, "language": language,
                "language_probability": language_probability}
