"""Text to audio from the command line: the reference's text-to-audio and text-to-audio-batch tasks
(streamlit/tasks/text_to_audio.py, text_to_audio_batch.py) without the streamlit UI.

    python -m riffusion.text_to_audio text-to-audio --prompt "church bells" --checkpoint ckpt --output-dir out \
        [--negative-prompt drums] [--seed 42] [--num-clips 4] [--num-inference-steps 30] [--guidance 7] [--width 768] \
        [--scheduler PNDMScheduler] [--use-20k]
    python -m riffusion.text_to_audio text-to-audio-batch --input-json prompts.json --output-dir out [--num-seeds 2]

Each clip is a txt2img image (`RiffusionPipeline.txt2img`, height 512) written as PNG with the spectrogram parameters in
its EXIF block (so `python -m riffusion.cli image-to-audio` reads it back), and the audio the reference derives from
that image (`SpectrogramImageConverter.audio_from_spectrogram_image`, filters included) as WAV.  The clips of one
command (the seeds of text-to-audio, every entry x seed of one parameter set in the batch) run as batched denoising
loops of up to MAX_BATCH clips.

File names carry the seed.  The reference's batch task names files by parameter set and prompts only, so its outputs
for different seeds overwrite each other; here each seed keeps its files.
"""
from __future__ import annotations

import json
import sys
import typing as T
from pathlib import Path

from riffusion.cli import _store_image, build_parser
from riffusion.scheduler_b200 import SCHEDULER_OPTIONS
from riffusion.spectrogram_image_converter import SpectrogramImageConverter
from riffusion.spectrogram_params import SpectrogramParams

DEFAULT_CHECKPOINT = "riffusion/riffusion-model-v1"
HEIGHT = 512
MAX_BATCH = 32          # clips per batched denoising loop (CFG batch 64, the size bench.py measures)


def _load_pipeline(checkpoint: str, device: str):
    from riffusion.riffusion_pipeline import RiffusionPipeline

    return RiffusionPipeline.load_checkpoint(checkpoint, device=device)


def _slug(text: str) -> str:
    return text.replace(" ", "_")


def _chunks(items: T.Sequence, size: int = MAX_BATCH) -> T.Iterator[T.Sequence]:
    for i in range(0, len(items), size):
        yield items[i:i + size]


def _write_clip(image, params: SpectrogramParams, converter: SpectrogramImageConverter, image_path: Path,
                audio_path: Path) -> None:
    image.getexif().update(params.to_exif().items())
    _store_image(image, image_path, "PNG")
    converter.audio_from_spectrogram_image(image).export(str(audio_path), format="wav")
    print(f"Wrote {image_path} and {audio_path}")


def text_to_audio(*, prompt: str, checkpoint: str, output_dir: str, negative_prompt: str = "", seed: int = 42,
                  num_clips: int = 1, num_inference_steps: int = 30, guidance: float = 7.0, width: int = 512,
                  scheduler: str = SCHEDULER_OPTIONS[0], use_20k: bool = False, device: str = "cuda"):
    """Generate audio clips from a text prompt, seeds seed, seed + 1, ..."""
    if use_20k:
        params = SpectrogramParams(min_frequency=10, max_frequency=20000, sample_rate=44100, stereo=True)
    else:
        params = SpectrogramParams(min_frequency=0, max_frequency=10000, stereo=False)
    pipe = _load_pipeline(checkpoint, device)
    converter = SpectrogramImageConverter(params=params, device=device)
    target = Path(output_dir)
    target.mkdir(parents=True, exist_ok=True)
    for seeds in _chunks(list(range(seed, seed + num_clips))):
        out = pipe.txt2img(prompt, negative_prompt=negative_prompt or None, seed=list(seeds),
                           num_inference_steps=num_inference_steps, guidance_scale=guidance, width=width, height=HEIGHT,
                           scheduler=scheduler)
        for s, image in zip(seeds, out["images"]):
            stem = f"{_slug(prompt)}_{s}"
            _write_clip(image, params, converter, target / f"{stem}.png", target / f"{stem}.wav")


def text_to_audio_batch(*, input_json: str, output_dir: str, num_seeds: int = 1, device: str = "cuda"):
    """Generate audio for every entry x seed x parameter set of a JSON file (the reference's batch format:
    {"params": {...} or [{...}, ...], "entries": [{"prompt", "negative_prompt", "seed"}, ...]}); writes index.json."""
    data = json.loads(Path(input_json).read_text())
    param_sets = data["params"] if isinstance(data["params"], list) else [data["params"]]
    entries = data["entries"]
    target = Path(output_dir)
    target.mkdir(parents=True, exist_ok=True)
    spec = SpectrogramParams(min_frequency=0, max_frequency=10000)
    converter = SpectrogramImageConverter(params=spec, device=device)
    pipes: T.Dict[str, T.Any] = {}
    for i, params in enumerate(param_sets):
        params.setdefault("name", f"params[{i}]")
        ckpt = params.get("checkpoint", DEFAULT_CHECKPOINT)
        if ckpt not in pipes:
            pipes[ckpt] = _load_pipeline(ckpt, device)
        jobs = [(entry, s) for entry in entries for s in range(entry.get("seed", 42), entry.get("seed", 42) + num_seeds)]
        for chunk in _chunks(jobs):
            out = pipes[ckpt].txt2img(
                [e["prompt"] for e, _ in chunk], negative_prompt=[e.get("negative_prompt") for e, _ in chunk],
                seed=[s for _, s in chunk], num_inference_steps=params.get("num_inference_steps", 50),
                guidance_scale=params.get("guidance", 7.0), width=params.get("width", 512), height=HEIGHT,
                scheduler=params.get("scheduler", SCHEDULER_OPTIONS[0]))
            for (entry, s), image in zip(chunk, out["images"]):
                stem = f"{i}_{_slug(entry['prompt'])}_neg_{_slug(entry.get('negative_prompt') or '')}_seed_{s}"
                image_path, audio_path = target / f"image_{stem}.png", target / f"audio_{stem}.wav"
                _write_clip(image, spec, converter, image_path, audio_path)
                # the reference's keys (the last clip written for the entry), plus every clip
                entry["image_path"], entry["audio_path"] = str(image_path), str(audio_path)
                entry.setdefault("outputs", []).append(dict(params=params["name"], seed=s, image_path=str(image_path),
                                                            audio_path=str(audio_path)))
    (target / "index.json").write_text(json.dumps(data, indent=4))
    print(f"Output written to {target}")


COMMANDS = [text_to_audio, text_to_audio_batch]


def main(argv: T.Optional[T.Sequence[str]] = None) -> None:
    args = vars(build_parser(COMMANDS, prog="riffusion.text_to_audio", description=__doc__).parse_args(argv))
    fn = args.pop("_fn")
    args.pop("command")
    fn(**args)


if __name__ == "__main__":
    main(sys.argv[1:])
