"""Command line front end: the six commands of the reference's `python -m riffusion.cli` (riffusion/cli.py:21-278) with
the same names, flags and defaults:

    python -m riffusion.cli audio-to-image --audio clip.wav --image clip.png [--stereo] [--device cuda]
    python -m riffusion.cli image-to-audio --image clip.png --audio clip.wav
    python -m riffusion.cli print-exif --image clip.png
    python -m riffusion.cli sample-clips --audio song.wav --output-dir clips --num-clips 4
    python -m riffusion.cli audio-to-images-batch --audio-dir clips --output-dir images
    python -m riffusion.cli sample-clips-batch --audio-dir songs --output-dir clips

Each command is a keyword-only function (callable from Python exactly like the reference's); `argh`, which the reference
uses to turn those functions into sub-commands, is not installed on the B200 image, so `build_parser` derives an
argparse sub-command per function from its signature instead.  Audio I/O goes through riffusion.util.audio_util
(pydub when present, else the WAV-only stand-in).
"""
from __future__ import annotations

import argparse
import inspect
import random
import sys
import typing as T
from multiprocessing.pool import ThreadPool
from pathlib import Path

import numpy as np
from PIL import Image

from riffusion.spectrogram_image_converter import SpectrogramImageConverter
from riffusion.spectrogram_params import SpectrogramParams
from riffusion.util import image_util
from riffusion.util.audio_util import AudioSegment

_PIL_FORMAT = {"jpg": "JPEG", "jpeg": "JPEG", "png": "PNG"}


# ------------------------------------------------------------------------------------------------ shared pieces
def _store_image(picture: Image.Image, path, fmt: str) -> None:
    """Save with the EXIF block (conversion parameters + MAX_VALUE) that image-to-audio reads back."""
    picture.save(path, exif=picture.getexif(), format=fmt)


def _files_in(folder: str, pattern: str = "*", limit: int = -1) -> T.List[Path]:
    found = sorted(p for p in Path(folder).glob(pattern) if p.is_file())
    return found[:limit] if limit > 0 else found


def _try_load(path: Path):
    """Unreadable / non-audio files in a batch directory are skipped, as in the reference (cli.py:176-179, 247-250)."""
    try:
        return AudioSegment.from_file(str(path))
    except Exception:  # noqa: BLE001
        return None


def _run_pool(worker: T.Callable[[Path], None], items: T.Sequence[Path], num_threads: T.Optional[int]) -> None:
    with ThreadPool(processes=num_threads) as pool:
        for _ in pool.imap_unordered(worker, items):
            pass


# ------------------------------------------------------------------------------------------------ commands
def audio_to_image(*, audio: str, image: str, step_size_ms: int = 10, num_frequencies: int = 512,
                   min_frequency: int = 0, max_frequency: int = 10000, window_duration_ms: int = 100,
                   padded_duration_ms: int = 400, power_for_image: float = 0.25, stereo: bool = False,
                   device: str = "cuda"):
    """Compute a spectrogram image from a waveform."""
    clip = AudioSegment.from_file(audio)
    spec = SpectrogramParams(sample_rate=clip.frame_rate, stereo=stereo, step_size_ms=step_size_ms,
                             window_duration_ms=window_duration_ms, padded_duration_ms=padded_duration_ms,
                             num_frequencies=num_frequencies, min_frequency=min_frequency, max_frequency=max_frequency,
                             power_for_image=power_for_image)
    picture = SpectrogramImageConverter(params=spec, device=device).spectrogram_image_from_audio(clip)
    _store_image(picture, image, "PNG")
    print(f"Wrote {image}")


def print_exif(*, image: str) -> None:
    """Print the params of a spectrogram image as saved in the exif data."""
    for tag, value in image_util.exif_from_image(Image.open(image)).items():
        print(f"{tag:<20} = {value:>15}")


def image_to_audio(*, image: str, audio: str, device: str = "cuda"):
    """Reconstruct an audio clip from a spectrogram image."""
    picture = Image.open(image)
    tags = picture.getexif()
    assert tags is not None
    try:
        spec = SpectrogramParams.from_exif(exif=tags)
    except KeyError:       # an image without our tags: the reference falls back to the defaults with this message
        print("WARNING: Could not find spectrogram parameters in exif data. Using defaults.")
        spec = SpectrogramParams()
    clip = SpectrogramImageConverter(params=spec, device=device).audio_from_spectrogram_image(picture)
    clip.export(audio, format=Path(audio).suffix[1:])
    print(f"Wrote {audio} ({clip.duration_seconds:.2f} seconds)")


def sample_clips(*, audio: str, output_dir: str, num_clips: int = 1, duration_ms: int = 5120, mono: bool = False,
                 extension: str = "wav", seed: int = -1):
    """Slice an audio file into clips of the given duration."""
    if seed >= 0:
        np.random.seed(seed)
    source = AudioSegment.from_file(audio)
    if mono:
        source = source.set_channels(1)
    target = Path(output_dir)
    target.mkdir(parents=True, exist_ok=True)
    total_ms = int(source.duration_seconds * 1000)
    for index in range(num_clips):
        begin = np.random.randint(0, total_ms - duration_ms)
        out_path = target / f"clip_{index}_start_{begin}_ms_duration_{duration_ms}_ms.{extension}"
        source[begin: begin + duration_ms].export(out_path, format=extension)
        print(f"Wrote {out_path}")


def audio_to_images_batch(*, audio_dir: str, output_dir: str, image_extension: str = "jpg", step_size_ms: int = 10,
                          num_frequencies: int = 512, min_frequency: int = 0, max_frequency: int = 10000,
                          power_for_image: float = 0.25, mono: bool = False, sample_rate: int = 44100,
                          device: str = "cuda", num_threads: T.Optional[int] = None, limit: int = -1):
    """Process audio clips into spectrograms in batch, multi-threaded (one converter shared by all threads)."""
    target = Path(output_dir)
    target.mkdir(parents=True, exist_ok=True)
    spec = SpectrogramParams(sample_rate=sample_rate, stereo=not mono, step_size_ms=step_size_ms,
                             num_frequencies=num_frequencies, min_frequency=min_frequency, max_frequency=max_frequency,
                             power_for_image=power_for_image)
    shared = SpectrogramImageConverter(params=spec, device=device)
    want_channels = 1 if mono else 2

    def convert_one(path: Path) -> None:
        clip = _try_load(path)
        if clip is None:
            return
        if clip.channels != want_channels:
            clip = clip.set_channels(want_channels)
        if clip.frame_rate != spec.sample_rate:
            clip = clip.set_frame_rate(spec.sample_rate)
        _store_image(shared.spectrogram_image_from_audio(clip), target / f"{path.stem}.{image_extension}",
                     _PIL_FORMAT[image_extension])

    _run_pool(convert_one, _files_in(audio_dir, limit=limit), num_threads)


def sample_clips_batch(*, audio_dir: str, output_dir: str, num_clips_per_file: int = 1, duration_ms: int = 5120,
                       mono: bool = False, extension: str = "mp3", num_threads: T.Optional[int] = None, glob: str = "*",
                       limit: int = -1, seed: int = -1):
    """Sample short clips from a directory of audio files, multi-threaded."""
    sources = [p for p in _files_in(audio_dir, pattern=glob) if p.suffix != ".json"]      # metadata files never count (:219-220)
    if limit > 0:
        sources = sources[:limit]
    if seed >= 0:
        random.seed(seed)
    target = Path(output_dir)
    target.mkdir(parents=True, exist_ok=True)

    def cut_one(path: Path) -> None:
        source = _try_load(path)
        if source is None:
            return
        if mono:
            source = source.set_channels(1)
        total_ms = int(source.duration_seconds * 1000)
        for index in range(num_clips_per_file):
            try:        # a source no longer than the clip duration yields nothing, as in the reference (:247-250)
                begin = int(np.random.randint(0, total_ms - duration_ms))
            except ValueError:
                continue
            name = f"{path.stem}_{index}_start_{begin}_ms_dur_{duration_ms}_ms.{extension}"
            source[begin: begin + duration_ms].export(target / name, format=extension)

    _run_pool(cut_one, sources, num_threads)


COMMANDS = [audio_to_image, image_to_audio, sample_clips, print_exif, audio_to_images_batch, sample_clips_batch]


# ------------------------------------------------------------------------------------------------ argparse front end
def _str2bool(v: str) -> bool:
    if v.lower() in ("1", "true", "yes", "y"):
        return True
    if v.lower() in ("0", "false", "no", "n"):
        return False
    raise argparse.ArgumentTypeError(f"expected a boolean, got {v!r}")


def build_parser(commands: T.Optional[T.Sequence[T.Callable]] = None, prog: str = "riffusion.cli",
                 description: T.Optional[str] = __doc__) -> argparse.ArgumentParser:
    """argh-style front end: one sub-command per function (underscores -> dashes), one --flag per keyword-only arg.
    `commands` defaults to this module's six commands."""
    parser = argparse.ArgumentParser(prog=prog, description=description)
    sub = parser.add_subparsers(dest="command", required=True)
    for fn in (COMMANDS if commands is None else commands):
        sp = sub.add_parser(fn.__name__.replace("_", "-"), help=(fn.__doc__ or "").strip())
        sp.set_defaults(_fn=fn)
        for name, prm in inspect.signature(fn).parameters.items():
            flag = "--" + name.replace("_", "-")
            if prm.default is inspect.Parameter.empty:
                sp.add_argument(flag, dest=name, required=True)
            elif isinstance(prm.default, bool):
                sp.add_argument(flag, dest=name, nargs="?", const=True, default=prm.default, type=_str2bool)
            elif prm.default is None:
                sp.add_argument(flag, dest=name, default=None, type=int)
            else:
                sp.add_argument(flag, dest=name, default=prm.default, type=type(prm.default))
    return parser


def main(argv: T.Optional[T.Sequence[str]] = None) -> None:
    args = vars(build_parser().parse_args(argv))
    fn = args.pop("_fn")
    args.pop("command")
    fn(**args)


if __name__ == "__main__":
    main(sys.argv[1:])
