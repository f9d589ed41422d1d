"""Audio-to-audio timing on one GPU; prints one JSON line.

  (a) a 20 s track as the reference's audio-to-audio task cuts it: 4 clips of 5 s, DPM-Solver++ 25 steps at denoising
      0.55 (13 UNet evaluations at CFG batch 8), guidance 7, one batched loop on the device path
      (riffusion.audio_to_audio.audio_to_audio: slicing, audio_to_audio_clips, host int16 + filters, stitching)
  (b) a ~3 min track (180 s: 37 clips, loops of 32 + 5), clips/s over the whole track
  (c) rf_resample_u8 alone on 32 clip images, 512 x 501 -> 512 x 512 and back, CUDA events over 200 graph-replayed
      launches each.  The kernel is there to keep the batch on the device, not for its rate.

Random-init SD-1.5 UNet / VAE and ClipTextB200.random_init, as bench.py --workload riffuse; the track is seeded
synthetic audio.  Card name, power limit and SM clock are read in the same run.
    python scratch/bench_audio_to_audio.py [--reps 3]
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT, ROOT / "riffusion-hobby_b200", ROOT / "tests" / "golden", ROOT / "scratch"):
    sys.path.insert(0, str(p))

from bench_text_to_audio import gpu_info  # noqa: E402


def timed(fn, reps: int) -> float:
    import torch

    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def kernel_us(fn, launches: int = 200) -> float:
    import torch

    for _ in range(10):
        fn()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(launches):
            fn()
    graph.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / launches


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import numpy as np
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    from prompt_stub import StubTokenizer
    from riffusion import tc_ops as ops
    from riffusion.audio_to_audio import audio_to_audio
    from riffusion.clip_b200 import ClipTextB200
    from riffusion.riffusion_pipeline import RiffusionPipeline
    from riffusion.util.audio_util import AudioSegment

    info_before = gpu_info()
    pipe = RiffusionPipeline.random_init(seed=0, device="cuda")
    pipe.text_encoder, pipe.tokenizer = ClipTextB200.random_init(seed=2, device="cuda"), StubTokenizer()
    rng = np.random.default_rng(0)

    def track(seconds: float) -> AudioSegment:
        t = np.arange(int(seconds * 44100)) / 44100.0
        x = 6000 * np.sin(2 * np.pi * 220 * t) * np.sin(2 * np.pi * 0.5 * t) + rng.normal(0, 500, t.size)
        return AudioSegment(x.astype(np.int16)[:, None], 44100)

    kw = dict(pipe=pipe, prompt="jazz with piano", seed=42, denoising=0.55, num_inference_steps=25, guidance=7.0)
    t20, t180 = track(20.0), track(180.0)
    counts = {}

    def run(seg, duration):
        result, starts, _, _ = audio_to_audio(seg, duration_s=duration, **kw)
        counts[duration] = (len(starts), result.duration_seconds)

    run(t20, 20.0)                                           # warm-up: graph capture, plans, allocator, resize tables
    t_20 = timed(lambda: run(t20, 20.0), args.reps)
    run(t180, 180.0)
    t_180 = timed(lambda: run(t180, 180.0), max(1, args.reps - 1))

    src = torch.from_numpy(rng.integers(0, 256, (32, 512, 501, 3), dtype=np.uint8)).cuda()
    up = ops.resample_u8(src, 512, 512)
    us_up = kernel_us(lambda: ops.resample_u8(src, 512, 512))
    us_down = kernel_us(lambda: ops.resample_u8(up, 512, 501))

    print(json.dumps(dict(
        workload="audio_to_audio", weights="random-init SD-1.5 (BASELINE config 4)",
        track_20s=dict(clips=counts[20.0][0], output_s=round(counts[20.0][1], 3), steps=25, denoising=0.55,
                       unet_evals=13, cfg_batch=2 * counts[20.0][0], seconds=round(t_20, 4)),
        track_180s=dict(clips=counts[180.0][0], output_s=round(counts[180.0][1], 3), loops=[32, counts[180.0][0] - 32],
                        seconds=round(t_180, 4), clips_per_s=round(counts[180.0][0] / t_180, 3)),
        resample_kernel=dict(batch=32, up_512x501_to_512x512_us=round(us_up, 2), down_512x512_to_512x501_us=round(us_down, 2)),
        gpu_before=info_before, gpu_after=gpu_info())))


if __name__ == "__main__":
    main()
