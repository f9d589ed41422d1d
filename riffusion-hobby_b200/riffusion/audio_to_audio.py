"""Audio to audio from the command line: the reference's audio-to-audio task (streamlit/tasks/audio_to_audio.py) without
the streamlit UI.

    python -m riffusion.audio_to_audio audio-to-audio --audio in.wav --prompt "jazz piano" --checkpoint ckpt \
        --output out.wav [--negative-prompt drums] [--seed 42] [--denoising 0.55] [--num-inference-steps 25] \
        [--guidance 7] [--scheduler PNDMScheduler] [--start-time-s 0] [--duration-s 20] [--clip-duration-s 5] \
        [--overlap-duration-s 0.2] [--prompt-b "rock" --seed-b 7 --denoising-b 0.6] [--image-dir clips]

The track is cut into overlapping clips (`clip_start_times`, `slice_audio_into_clips`), every clip is riffed with the
same prompt, seed and denoising strength, and the clips are joined again with crossfades over the overlap.  The clips
of a track share everything but their audio, so they run as batched img2img loops of up to MAX_BATCH clips on the
device (`RiffusionPipeline.audio_to_audio_clips`) rather than one clip at a time.

Giving --prompt-b turns on the reference's interpolation mode: clip i runs `riffuse` with alpha = linspace(0, 1, n)[i]
between (prompt, seed, denoising) and (prompt-b, seed-b, denoising-b), on the host-made 32-stride spectrogram image;
riffuse uses its own PNDM scheduler, so --scheduler does not apply there.

Input is WAV at 44100 Hz.  The reference resamples other rates with pydub, which this build does not have.  Spectrograms
are mono 0-10 kHz; the reference's 20 kHz stereo option and its magic-mix pipeline are not available.
"""
from __future__ import annotations

import sys
import typing as T
from pathlib import Path

import numpy as np
from PIL import Image

from riffusion.cli import _store_image, build_parser
from riffusion.datatypes import InferenceInput, PromptInput
from riffusion.scheduler_b200 import SCHEDULER_OPTIONS
from riffusion.spectrogram_converter import SpectrogramConverter
from riffusion.spectrogram_image_converter import SpectrogramImageConverter, _conform_channels
from riffusion.spectrogram_params import SpectrogramParams
from riffusion.util import audio_util

DEFAULT_CHECKPOINT = "riffusion/riffusion-model-v1"
SAMPLE_RATE = 44100
MAX_BATCH = 32          # clips per batched denoising loop (CFG batch 64, as text_to_audio)


def _load_pipeline(checkpoint: str, device: str):
    from riffusion.riffusion_pipeline import RiffusionPipeline

    return RiffusionPipeline.load_checkpoint(checkpoint, device=device)


def _chunks(n: int, size: int = MAX_BATCH) -> T.Iterator[range]:
    for i in range(0, n, size):
        yield range(i, min(i + size, n))


def clip_start_times(start_time_s: float, duration_s: float, clip_duration_s: float = 5.0,
                     overlap_duration_s: float = 0.2) -> np.ndarray:
    """Clip starts of the reference: start + arange(0, duration - clip, clip - overlap) (no clip starts in the last
    clip's worth of the duration)."""
    return start_time_s + np.arange(0, duration_s - clip_duration_s, clip_duration_s - overlap_duration_s)


def slice_audio_into_clips(segment, clip_start_times: T.Sequence[float], clip_duration_s: float) -> T.List:
    """Clips of `clip_duration_s` at the given start times, cut in whole milliseconds as the reference cuts them.  The
    last clip is padded with silence to the full clip length if the track ends inside it.  (The reference appends the
    silence with pydub's default 100 ms crossfade, which shortens the clip or fails; here it is appended as is.)"""
    clip_duration_ms = int(clip_duration_s * 1000)
    clips = []
    for i, t in enumerate(clip_start_times):
        start_ms = int(t * 1000)
        clip = segment[start_ms:start_ms + clip_duration_ms]
        if i == len(clip_start_times) - 1:
            silence_ms = clip_duration_ms - int(clip.duration_seconds * 1000)
            if silence_ms > 0:
                silence = audio_util.AudioSegment.silent(duration=silence_ms, frame_rate=segment.frame_rate)
                clip = clip.append(silence, crossfade=0)
        clips.append(clip)
    return clips


def scale_image_to_32_stride(image: Image.Image) -> Image.Image:
    """BICUBIC resize to the next multiples of 32 (what rf_resample_u8 does on the device path)."""
    return image.resize((int(np.ceil(image.width / 32) * 32), int(np.ceil(image.height / 32) * 32)), Image.BICUBIC)


def _segment_from_waveform(wave: np.ndarray):
    """host end of `audio_from_spectrogram`: peak-normalised int16, then the loudness filters"""
    segment = audio_util.audio_from_waveform(samples=wave[None].astype(np.float32), sample_rate=SAMPLE_RATE, normalize=True)
    return audio_util.apply_filters(segment, compression=False)


def audio_to_audio(segment, *, pipe, prompt: str, negative_prompt: T.Optional[str] = None, seed: int = 42,
                   denoising: float = 0.55, num_inference_steps: int = 25, guidance: float = 7.0,
                   scheduler: str = SCHEDULER_OPTIONS[0], start_time_s: float = 0.0, duration_s: float = 20.0,
                   clip_duration_s: float = 5.0, overlap_duration_s: float = 0.2, prompt_b: T.Optional[str] = None,
                   seed_b: T.Optional[int] = None, denoising_b: T.Optional[float] = None, device: str = "cuda"):
    """Riff `segment` (an AudioSegment at 44100 Hz) clip by clip and stitch the result.  `prompt_b` turns on
    interpolation (seed_b / denoising_b default to seed / denoising).  Returns (stitched segment, clip start times,
    source images, riffed images), the images as PIL images of the clips' spectrograms."""
    if int(segment.frame_rate) != SAMPLE_RATE:
        raise ValueError(f"audio must be sampled at {SAMPLE_RATE} Hz, got {segment.frame_rate} Hz "
                         "(resampling needs pydub, which is not installed)")
    params = SpectrogramParams(min_frequency=0, max_frequency=10000, stereo=False)
    duration_s = min(duration_s, segment.duration_seconds - start_time_s)
    starts = clip_start_times(start_time_s, duration_s, clip_duration_s, overlap_duration_s)
    if len(starts) == 0:
        raise ValueError(f"{duration_s:.2f} s of audio after {start_time_s} s hold no clip of {clip_duration_s} s")
    clips = [_conform_channels(c, False) for c in slice_audio_into_clips(segment, starts, clip_duration_s)]
    n = len(clips)
    sources: T.List[Image.Image] = []
    riffed: T.List[Image.Image] = []
    segments = []
    if prompt_b:
        converter = SpectrogramImageConverter(params=params, device=device)
        alphas = np.linspace(0, 1, n)
        start = PromptInput(prompt=prompt, seed=seed, denoising=denoising, guidance=guidance)
        end = PromptInput(prompt=prompt_b, seed=seed if seed_b is None else seed_b,
                          denoising=denoising if denoising_b is None else denoising_b, guidance=guidance)
        sources = [converter.spectrogram_image_from_audio(c) for c in clips]
        for idx in _chunks(n):
            inputs = [InferenceInput(alpha=float(alphas[i]), num_inference_steps=num_inference_steps,
                                     seed_image_id="og_beat", start=start, end=end) for i in idx]
            images = pipe.riffuse_batch(inputs, init_images=[scale_image_to_32_stride(sources[i]) for i in idx])
            for i, image in zip(idx, images):
                image = image.resize(sources[i].size, Image.BICUBIC)
                image.getexif().update(params.to_exif().items())
                riffed.append(image)
                segments.append(converter.audio_from_spectrogram_image(image))
    else:
        import torch

        converter = SpectrogramConverter(params=params, device=device)
        waves = np.stack([np.asarray(c.get_array_of_samples(), dtype=np.float32) for c in clips])
        for idx in _chunks(n):
            out = pipe.audio_to_audio_clips(torch.from_numpy(waves[idx.start:idx.stop]).to(device), converter=converter,
                                            prompt=prompt, negative_prompt=negative_prompt or None, seed=seed,
                                            strength=denoising, num_inference_steps=num_inference_steps,
                                            guidance_scale=guidance, scheduler=scheduler)
            for k, name in ((0, "source_images"), (1, "images")):
                for im in out[name].cpu().numpy():
                    image = Image.fromarray(im)
                    image.getexif().update(params.to_exif().items())
                    (sources, riffed)[k].append(image)
            segments.extend(_segment_from_waveform(w) for w in out["waveform"].cpu().numpy())
    return audio_util.stitch_segments(segments, crossfade_s=overlap_duration_s), starts, sources, riffed


def audio_to_audio_command(*, audio: str, prompt: str, output: str, checkpoint: str = DEFAULT_CHECKPOINT,
                           negative_prompt: str = "", seed: int = 42, denoising: float = 0.55,
                           num_inference_steps: int = 25, guidance: float = 7.0, scheduler: str = SCHEDULER_OPTIONS[0],
                           start_time_s: float = 0.0, duration_s: float = 20.0, clip_duration_s: float = 5.0,
                           overlap_duration_s: float = 0.2, prompt_b: str = "", seed_b: T.Optional[int] = None,
                           denoising_b: float = -1.0, image_dir: str = "", device: str = "cuda"):
    """Riff a WAV track with a text prompt in overlapping clips and write the stitched result as WAV.  --prompt-b
    (with --seed-b, --denoising-b; a negative --denoising-b means --denoising) interpolates between two prompts along the
    track.  --image-dir writes each clip's source and riffed spectrogram as PNG."""
    segment = audio_util.AudioSegment.from_file(audio)
    if int(segment.frame_rate) != SAMPLE_RATE:
        raise ValueError(f"{audio}: audio must be sampled at {SAMPLE_RATE} Hz, got {segment.frame_rate} Hz "
                         "(resampling needs pydub, which is not installed)")
    pipe = _load_pipeline(checkpoint, device)
    result, starts, sources, riffed = audio_to_audio(
        segment, pipe=pipe, prompt=prompt, negative_prompt=negative_prompt or None, seed=seed, denoising=denoising,
        num_inference_steps=num_inference_steps, guidance=guidance, scheduler=scheduler, start_time_s=start_time_s,
        duration_s=duration_s, clip_duration_s=clip_duration_s, overlap_duration_s=overlap_duration_s,
        prompt_b=prompt_b or None, seed_b=seed_b, denoising_b=None if denoising_b < 0 else denoising_b, device=device)
    print(f"Riffed {len(starts)} clips of {clip_duration_s} s with {overlap_duration_s} s overlap, starting at "
          + ", ".join(f"{t:.2f}" for t in starts) + " s")
    if image_dir:
        target = Path(image_dir)
        target.mkdir(parents=True, exist_ok=True)
        for i, (src, out) in enumerate(zip(sources, riffed)):
            _store_image(src, target / f"clip_{i}_source.png", "PNG")
            _store_image(out, target / f"clip_{i}_riffed.png", "PNG")
    Path(output).parent.mkdir(parents=True, exist_ok=True)
    result.export(output, format="wav")
    print(f"Wrote {output} ({result.duration_seconds:.3f} s)")


audio_to_audio_command.__name__ = "audio_to_audio"     # the sub-command name: audio-to-audio
COMMANDS = [audio_to_audio_command]


def main(argv: T.Optional[T.Sequence[str]] = None) -> None:
    args = vars(build_parser(COMMANDS, prog="riffusion.audio_to_audio", description=__doc__).parse_args(argv))
    fn = args.pop("_fn")
    args.pop("command")
    fn(**args)


if __name__ == "__main__":
    main(sys.argv[1:])
