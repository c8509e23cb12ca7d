"""Shared plumbing of the CLI shells: model/tokenizer loading, transcript source, batching."""
from __future__ import annotations

import datetime
import json
import os
import time

import torch

from .. import audio, whisper_model
from ..retokenize import encode, remove_punctuation
from ..tokenizer import get_tokenizer as byte_tokenizer

MAX_FRAMES = 1500  # reference infer_ali.py:25
MAX_LENGTH = 448   # reference infer_ali.py:26
AUDIO_SAMPLES_PER_TOKEN = audio.N_SAMPLES_PER_TOKEN  # reference infer_ali.py:179

def load_model_and_tokenizer(name: str, device, qk_gain: float = 4.0):
    """Stock `openai-whisper` when it is installed (real checkpoints, real tokenizer, greedy decode available).
    Otherwise `name` must be a checkpoint file or an explicit `random:<size>` (seeded random init, offline byte
    tokenizer) -- a bare size name such as `medium` raises instead of silently aligning with random weights.
    Returns (model, tokenizer, whisper package or None, model_source)."""
    try:
        import whisper  # noqa: F401
        from whisper.tokenizer import get_tokenizer

        if not (hasattr(whisper, "decode") and hasattr(whisper, "DecodingOptions")):
            raise ImportError("a `whisper` module without decode() is not openai-whisper")
        model = whisper.load_model(name).to(device)
        return model, get_tokenizer(model.is_multilingual, language="English"), whisper, f"openai-whisper:{name}"
    except ImportError:
        model = whisper_model.load_model(name, device, qk_gain=qk_gain)
        # the reference leaves num_languages at 99 (infer_ali.py:41), which is off by one for large-v3's
        # vocabulary; the offline tokenizer takes the model's own count
        tk = byte_tokenizer(model.is_multilingual, language="English", num_languages=model.num_languages)
        return model, tk, None, model.model_source


TRANSCRIBE = os.environ.get("WCA_TRANSCRIBE", "reference")  # offline default: align the reference transcript
#: tokens the built-in greedy decoder may generate per utterance (whisper's DecodingOptions.sample_len default)
DECODE_TOKENS = 224


def transcript_source(whisper_pkg) -> str:
    if whisper_pkg is not None:
        return "whisper.decode"
    return "greedy_decode" if TRANSCRIBE == "greedy" else "ground-truth transcript (no ASR step)"


def transcribe(whisper_pkg, model, mel, reference_text: str, tokenizer=None) -> str:
    """The reference transcribes with whisper.decode (infer_ali.py:60).  With openai-whisper installed
    that call is used as is; offline the reference transcript is force-aligned (a random-init model
    transcribes noise), or, with WCA_TRANSCRIBE=greedy and a checkpoint, the built-in greedy decoder."""
    if whisper_pkg is not None:
        return whisper_pkg.decode(model, mel, whisper_pkg.DecodingOptions(language="en")).text
    if TRANSCRIBE == "greedy" and tokenizer is not None:
        return tokenizer.decode(whisper_model.greedy_decode(model, mel, tokenizer, DECODE_TOKENS))
    return reference_text


def prepare(record, tokenizer, unit, device, whisper_pkg, model):
    """One dataset record -> dict with tokens and frame count, or None when the reference would skip it
    (infer_ali.py:78-81)."""
    mel = record[1].to(device)
    return _item(record, mel, transcribe(whisper_pkg, model, mel, remove_punctuation(record[3]), tokenizer), tokenizer,
                 unit, device)


def prepare_window(records, tokenizer, unit, device, whisper_pkg, model, batch_size):
    """prepare() for a window of records, in order.  With WCA_TRANSCRIBE=greedy on a CUDA device (and no
    openai-whisper) the records are transcribed `batch_size` at a time: one encoder pass per chunk, whose output
    greedy_decode_cached transcribes and each item keeps (`audio_features`, a view of the chunk's output) for its
    alignment.  Every other mode transcribes record by record, and its items carry no features."""
    if not (whisper_pkg is None and TRANSCRIBE == "greedy" and torch.device(device).type == "cuda"):
        return [prepare(r, tokenizer, unit, device, whisper_pkg, model) for r in records]
    out = []
    for chunk in batches(records, batch_size):
        mels = torch.stack([r[1] for r in chunk]).to(device)
        with torch.no_grad():
            xa = model.embed_audio(mels)
        texts = whisper_model.greedy_decode_cached(model, xa, tokenizer, DECODE_TOKENS)
        out += [_item(r, mels[i], tokenizer.decode(texts[i]), tokenizer, unit, device, xa[i]) for i, r in enumerate(chunk)]
    return out


def _item(record, mel, transcription, tokenizer, unit, device, audio_features=None):
    _, _, duration, text, starts, ends, fid = record
    text = remove_punctuation(text)
    # an empty transcription stays empty, as in the reference (its `len(transcription) == ''` guard at
    # infer_ali.py:65 never fires): force_align then returns the EOT-only sentinel and 0 predictions
    transcription = remove_punctuation(transcription)
    text_tokens = encode(transcription, tokenizer, unit)
    tokens = torch.tensor([*tokenizer.sot_sequence, tokenizer.no_timestamps, *text_tokens, tokenizer.eot], device=device)
    max_frames = int(duration) // AUDIO_SAMPLES_PER_TOKEN
    if max_frames > MAX_FRAMES or len(tokens) > MAX_LENGTH or max_frames < 1:
        print(fid)
        return None
    return dict(mel=mel, tokens=tokens, text_tokens=text_tokens, max_frames=max_frames, text=text, starts=starts,
                ends=ends, fid=fid, audio_features=audio_features)


def batches(items, size):
    for i in range(0, len(items), size):
        yield items[i:i + size]


def dump_results(args, results: dict, suffix: str = ""):
    """<output_dir>/<%Y-%m-%d-%H:%M:%S><suffix>.json = flags merged with metrics (reference infer_ali.py:139-146)."""
    stamp = datetime.datetime.fromtimestamp(time.time()).strftime("%Y-%m-%d-%H:%M:%S")
    os.makedirs(args.output_dir, exist_ok=True)
    path = os.path.join(args.output_dir, stamp + suffix + ".json")
    with open(path, "w") as f:
        json.dump({**vars(args), **results}, f)
    return path, stamp
