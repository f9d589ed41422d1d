"""Text-to-audio timing on one GPU; prints one JSON line.

  (a) one request as the reference's text-to-audio task makes it: 30 DPM-Solver++ steps, width 512, guidance 7, one clip
      - device path: RiffusionPipeline.text_to_audio_clips (latents -> VAE -> uint8 -> mel -> Griffin-Lim on the device)
      - PIL path: txt2img -> PIL image -> SpectrogramImageConverter.audio_from_spectrogram_image (what the CLI runs)
  (b) 32 clips in one batched loop (text_to_audio_clips, CFG batch 64), clips/s
  (c) rf_cfg_dpmpp_step_f16 alone at B = 32 (second order, 524288 elements), CUDA events over 2000 launches (graph
      replays of 100 launches each), against its
      12 B/element of traffic (eps pair 4, sample 2, x0 history 2 read; x0 and x_t 2 + 2 written).  The 6.3 MB working
      set stays in L2, so the rate is an L2 rate, not an HBM rate.

Random-init SD-1.5 UNet / VAE and ClipTextB200.random_init, as bench.py --workload riffuse.  Card name, power limit and
SM clock are read in the same run.
    python scratch/bench_text_to_audio.py [--reps 5]
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT, ROOT / "riffusion-hobby_b200", ROOT / "tests" / "golden"):
    sys.path.insert(0, str(p))


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                              capture_output=True, text=True, check=True).stdout.strip()
        name, power, sm, sm_max = [v.strip() for v in line.split(",")]
        return dict(gpu=name, power_limit_w=float(power), sm_mhz=int(sm), sm_max_mhz=int(sm_max))
    except Exception as e:  # noqa: BLE001
        return dict(gpu=None, error=str(e))


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


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    from prompt_stub import StubTokenizer
    from riffusion import tc_ops as ops
    from riffusion.clip_b200 import ClipTextB200
    from riffusion.riffusion_pipeline import RiffusionPipeline
    from riffusion.spectrogram_converter import SpectrogramConverter
    from riffusion.spectrogram_image_converter import SpectrogramImageConverter
    from riffusion.spectrogram_params import SpectrogramParams

    info_before = gpu_info()
    pipe = RiffusionPipeline.random_init(seed=0, device="cuda")
    pipe.text_encoder, pipe.tokenizer = ClipTextB200.random_init(seed=2, device="cuda"), StubTokenizer()
    params = SpectrogramParams(min_frequency=0, max_frequency=10000, stereo=False)
    conv = SpectrogramConverter(params, device="cuda")
    img_conv = SpectrogramImageConverter(params, device="cuda")
    kw = dict(num_inference_steps=30, guidance_scale=7.0, width=512)

    # (a) one request
    def device_one():
        pipe.text_to_audio_clips("church bells on sunday", converter=conv, seed=42, **kw)

    def pil_one():
        image = pipe.txt2img("church bells on sunday", seed=42, height=512, **kw)["images"][0]
        img_conv.audio_from_spectrogram_image(image)

    device_one(), pil_one()                                  # warm-up: graph capture, plans, allocator
    t_dev = timed(device_one, args.reps)
    t_pil = timed(pil_one, args.reps)

    # (b) 32 clips, one batched loop
    prompts = [f"church bells on sunday take {i}" for i in range(32)]

    def batch32():
        pipe.text_to_audio_clips(prompts, converter=conv, seed=list(range(100, 132)), **kw)

    batch32()
    t_b32 = timed(batch32, max(2, args.reps // 2))

    # (c) the fused step alone
    n = 32 * 4 * 64 * 64
    eps_pair = torch.randn(2 * n, device="cuda").half()
    x, m1, m0 = (torch.randn(n, device="cuda").half() for _ in range(3))
    out = torch.empty_like(x)
    co = dict(sigma_s=0.9965558648109436, alpha_s=0.08292368054389954, c_x=0.998393177986145, c_0=-0.01753595843911171,
              inv_r0=0.9819893836975098, c_d1=-0.008767979219555855)
    for _ in range(50):
        ops.cfg_dpmpp_step(eps_pair, 7.0, x, m1, x0_out=m0, out=out, **co)
    # 100 launches captured in one CUDA graph, replayed 20 times: kernel time without the Python launch overhead
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(100):
            ops.cfg_dpmpp_step(eps_pair, 7.0, x, m1, x0_out=m0, out=out, **co)
    graph.replay()
    launches = 2000
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches // 100):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / launches
    gbs = 12 * n / (us * 1e-6) / 1e9

    print(json.dumps(dict(
        workload="text_to_audio", weights="random-init SD-1.5 (BASELINE config 4)",
        single_request=dict(steps=30, width=512, guidance=7.0, device_path_s=round(t_dev, 4), pil_path_s=round(t_pil, 4)),
        batch32=dict(steps=30, width=512, seconds=round(t_b32, 4), clips_per_s=round(32 / t_b32, 3)),
        dpmpp_step_kernel=dict(batch=32, elements=n, launches=launches, us_per_launch=round(us, 3),
                               bytes_per_element=12, gb_per_s=round(gbs, 1), working_set="L2-resident (6.3 MB)"),
        gpu_before=info_before, gpu_after=gpu_info())))


if __name__ == "__main__":
    main()
