#!/usr/bin/env python
"""bench.py — throughput of the hot path on N B200s of one node (driver contract).

Two workloads:
  --workload clip (default): BASELINE's metric — clips/sec of a full 512x512 clip: 50 UNet evaluations (img2img with
      denoising 1.0, classifier-free guidance, PNDM) + VAE decode + image -> mel -> inverse mel -> 32-iteration
      Griffin-Lim, random-init SD-1.5 weights (BASELINE config 4: no network for the checkpoint), `--clips` clips
      per GPU per step.  roofline = the tcgen05 GEMM/conv kernel (tensor bound).  The Griffin-Lim sub-benchmark of
      configs[1] is run too and reported under "griffinlim" (its own HBM roofline = "GL HBM GB/s" of the metric).
  --workload gl: only BASELINE configs[1] — inverse-mel + 32-iteration Griffin-Lim, 512x512 mel, batch 64 per GPU.
  --workload riffuse: BASELINE configs[2] — ONE request through RiffusionPipeline.riffuse() (PIL in -> PIL out, seed image
      og_beat, alpha 0.5, 50 scheduler steps, --denoising 0.75 -> 38 CFG evaluations; 1.0 -> 50): latency per request.
  --workload roundtrip: BASELINE configs[4] — audio -> image -> audio: STFT + mel + image quantisation of 16 waveforms per
      GPU, VAE encode, 50-step denoise, VAE decode, image -> mel -> inverse mel + Griffin-Lim -> int16.

gl workload: one "step" = one pass of the hot path over one batch of 64 synthetic clips per GPU.
  value  : clips/s, whole job, inputs (mel amplitudes + initial phases) resident in HBM
  e2e    : clips/s through SpectrogramConverter.waveform_from_mel_amplitudes with HOST buffers:
           pinned mel -> H2D, torch.rand phase init (as the reference does per call), kernels,
           waveform D2H — all inside the timed region
  roofline: dominant Griffin-Lim kernel, algorithmic bytes (SURVEY §8d: 36 B per live bin x frame x
           iteration, split 12 B iSTFT / 24 B STFT) over its CUDA-event duration, vs MEASURED_PEAKS
  cpu_baseline / --impl reference: the reference's own CPU arithmetic (installed torchaudio
           transforms built with the reference's arguments, oracle/torchaudio_ref.py) on all host
           cores, on a bounded sample (one clip per step).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for _p in (str(ROOT), str(ROOT / "riffusion-hobby_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np
import torch

N_FFT, WIN, HOP, N_MELS, T_FRAMES, F_LIVE, N_ITER = 17640, 4410, 441, 512, 512, 4000, 32
BATCH_PER_GPU = 64
L_WAVE = HOP * (T_FRAMES - 1)


def algorithmic_bytes_per_clip() -> float:
    """SURVEY §8(d): n_iter*36*F_live*T + 12*F_live*T + (2 n_iter+1)*4*hop*(T-1)"""
    return N_ITER * 36 * F_LIVE * T_FRAMES + 12 * F_LIVE * T_FRAMES + (2 * N_ITER + 1) * 4 * L_WAVE


def synthetic_mel(batch: int, seed: int) -> torch.Tensor:
    """SURVEY §8(d) config 2: og_beat amplitudes perturbed per clip, mel_b = mel * exp(0.1 N(0,1))."""
    g = np.load(ROOT / "tests" / "golden" / "og_beat.npz")
    rgb = g["rgb"]
    data = rgb[::-1].transpose(2, 0, 1)[0:1].astype(np.float32)
    data = np.power((255 - data) / 255, 4.0).astype(np.float32) * np.float32(30e6)
    base = torch.from_numpy(data)  # (1, 512, 512)
    gen = torch.Generator().manual_seed(seed)
    noise = torch.randn((batch, N_MELS, T_FRAMES), generator=gen)
    return (base * torch.exp(0.1 * noise)).contiguous()


def peaks() -> dict:
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "source": "fallback"}


DUMP_BYTES = 60 << 20      # --dump-outputs: array data in all; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: write each tensor the timed path returned in its last step as DIR/<name>.npy, in float32 (float64
    tensors stay float64), DUMP_BYTES at most in all.  Arrays are taken smallest first, each against an equal share of
    what is left: one that fits is written whole with its shape, a larger one as the flattened elements at a sample of
    indices drawn from a fixed seed and sorted, the same for every run with the same arguments, so that two builds of the
    project can be compared output for output."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left = DUMP_BYTES
    for i, (name, t) in enumerate(items):
        a = t.detach().cpu().numpy()
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32, copy=False)
        k = left // (len(items) - i) // a.itemsize
        if a.size > k:
            idx = np.sort(np.random.default_rng(0).choice(a.size, size=k, replace=False, shuffle=False))
            a = a.reshape(-1)[idx]
        np.save(d / f"{name}.npy", a)
        left -= a.nbytes


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def time_reference(steps: int, warmup: int, host_cores: int) -> dict:
    """The reference's CPU path (torchaudio transforms with the reference's arguments), one clip per
    step.  torch's CPU FFT path does not scale with threads (measured on the 128-core GPU host:
    ~50 s/clip with 128 threads vs a few s with 8-32), so one clip is timed at 8, 16 and 32 threads
    (capped at the host's core count) and the fastest setting is used and reported as `cores`."""
    from oracle.torchaudio_ref import TorchaudioConverter

    conv = TorchaudioConverter(n_iter=N_ITER)
    mel = synthetic_mel(1, seed=0)
    torch.manual_seed(0)
    best = None
    for th in sorted({min(host_cores, 8), min(host_cores, 16), min(host_cores, 32)}):
        torch.set_num_threads(th)
        if best is None:
            for _ in range(max(warmup, 1)):
                conv.waveform_from_mel_amplitudes(mel)
        t0 = time.perf_counter()
        conv.waveform_from_mel_amplitudes(mel)
        dt = time.perf_counter() - t0
        if best is None or dt < best[1]:
            best = (th, dt)
    threads = best[0]
    torch.set_num_threads(threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        w = conv.waveform_from_mel_amplitudes(mel)
    dt = time.perf_counter() - t0
    assert w.shape == (1, L_WAVE)
    return {"value": steps / dt, "seconds_per_clip": dt / steps, "cores": threads,
            "sample": f"{steps} x 1 clip (512x512 mel, inverse-mel lstsq + 32-iter Griffin-Lim), torchaudio "
                      f"{__import__('torchaudio').__version__} fp32, {threads} threads (fastest of 8/16/32; host has "
                      f"{host_cores} cores)"}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="clips per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="clip", choices=["clip", "gl", "riffuse", "roundtrip"])
    ap.add_argument("--denoising", type=float, default=0.75, help="riffuse workload: img2img strength (0.75 -> 38 of 50 evals)")
    ap.add_argument("--clips", type=int, default=32, help="clips per GPU per step (clip workload)")
    ap.add_argument("--evals", type=int, default=50, help="scheduler steps = UNet evaluations per clip (denoising 1.0)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (B200 arm, rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 arm's timed path; the reference arm has none")
    if args.workload == "roundtrip" and args.clips == 32:
        args.clips = 16                      # BASELINE configs[4]: batch 128 on 8 GPUs
    if args.workload in ("clip", "roundtrip") and args.impl == "b200":
        return main_clip(args)
    if args.workload == "riffuse" and args.impl == "b200":
        return main_riffuse(args)
    if args.workload in ("clip", "roundtrip", "riffuse") and args.impl == "reference":
        return main_clip_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = os.cpu_count() or 1
    workload = (f"configs[1]: inverse-mel + Griffin-Lim {N_ITER}-iter reconstruction of {N_MELS}x{T_FRAMES} mel "
                f"spectrograms, batch {args.batch} per GPU")
    config = {"workload": workload, "includes_denoise": False, "n_fft": N_FFT, "win": WIN, "hop": HOP,
              "live_bins": F_LIVE, "batch_per_gpu": args.batch,
              "l2": "inputs+state (2.9 GB per step) larger than L2; no explicit flush",
              "sharding": "independent clips per rank, no collective in the step"}

    if args.impl == "reference":
        if rank != 0:
            return
        steps = max(1, min(args.steps, 6))
        r = time_reference(steps, max(1, min(args.warmup, 1)), cores)
        line = {"impl": "reference", "metric": "clips/sec", "value": r["value"], "unit": "clips/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": 1e3 * r["seconds_per_clip"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": "clips/s", "cores": r["cores"], "kind": "reference",
                                 "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    from riffusion import _native
    from riffusion.spectrogram_converter import SpectrogramConverter, get_plan
    from riffusion.spectrogram_params import SpectrogramParams

    params = SpectrogramParams()
    conv = SpectrogramConverter(params, device=str(dev))
    plan = get_plan(params, full_band=False)
    B = args.batch
    F = plan.info.n_freq
    mel_host = synthetic_mel(B, seed=rank).pin_memory()
    mel = mel_host.to(dev)
    torch.manual_seed(rank)
    angles = torch.rand((B, F, T_FRAMES), dtype=torch.complex64, device=dev)
    wave = torch.empty((B, L_WAVE), dtype=torch.float32, device=dev)
    wave_host = torch.empty((B, L_WAVE), dtype=torch.float32).pin_memory()
    lib = _native.lib()
    nbytes = lib.rf_griffinlim_workspace_bytes(plan.handle, B, T_FRAMES)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)

    def step_device():
        _native.check(lib.rf_mel_to_wave(plan.handle, mel.data_ptr(), angles.data_ptr(), B, T_FRAMES, N_ITER,
                                         0.99, wave.data_ptr(), ws.data_ptr(), nbytes, stream.cuda_stream))

    def step_e2e():
        m = mel_host.to(dev, non_blocking=True)
        w = conv.waveform_from_mel_amplitudes(m)      # draws torch.rand phases like the reference
        wave_host.copy_(w, non_blocking=True)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """milliseconds of `steps` calls of fn, and what the last call returned"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = None
        for _ in range(steps):
            out = fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    for _ in range(max(args.warmup, 3)):
        step_device()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total, _ = timed(step_device, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"waveform": wave})      # step_device writes its result into `wave`

    # per-kernel CUDA-event timing of the same step (rank 0 reports)
    ms_cls = (ctypes.c_float * 3)()
    n_cls = (ctypes.c_int * 3)()
    acc = np.zeros(3)
    prof_steps = min(args.steps, 3)
    for _ in range(prof_steps):
        _native.check(lib.rf_mel_to_wave_profiled(plan.handle, mel.data_ptr(), angles.data_ptr(), B, T_FRAMES, N_ITER,
                                                  0.99, wave.data_ptr(), ws.data_ptr(), nbytes, stream.cuda_stream,
                                                  ms_cls, n_cls))
        acc += np.array(list(ms_cls))
    acc /= prof_steps
    launches = list(n_cls)

    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    ms_step = ms_total / args.steps
    clips = B * world
    value = clips / (ms_step / 1e3)
    pk = peaks()
    names = ["k_istft_chunk", "k_ola_assemble", "k_stft_pair"]     # kernel classes: iSTFT (k_istft_half in the loop — every chunk
    # at half rate plus the edge chunks on the other sample parity — and k_istft_chunk for the last full-rate pass), overlap-add
    # assembly (k_ola_assemble_dec + k_ola_assemble_strips), STFT (k_stft_edge + k_stft_half)
    per_launch_bytes = [B * 12.0 * F_LIVE * T_FRAMES + B * 4.0 * L_WAVE, 0.0, B * 24.0 * F_LIVE * T_FRAMES + B * 4.0 * L_WAVE]
    dom = int(np.argmax(acc))
    dom_ms = acc[dom] / max(launches[dom], 1)
    achieved = per_launch_bytes[dom] / (dom_ms / 1e3) / 1e9 if dom_ms > 0 else 0.0
    loop_ms = float(acc.sum())
    loop_gbs = B * algorithmic_bytes_per_clip() / (loop_ms / 1e3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
        "frac": achieved / pk["hbm_gbs"], "traffic": None, "peak_source": pk["source"] + " (burst copy)",
        "kernel_ms_per_launch": dom_ms, "kernel_share_of_step": acc[dom] / (ms_step),
        "algorithmic_bytes_per_launch": per_launch_bytes[dom],
        "per_kernel_ms_per_step": dict(zip(names, [float(a) for a in acc])),
        "loop": {"achieved": loop_gbs, "frac": loop_gbs / pk["hbm_gbs"], "unit": "GB/s",
                 "algorithmic_bytes_per_step": B * algorithmic_bytes_per_clip(), "ms": loop_ms},
    }
    traffic_file = ROOT / "profiles" / "traffic_latest.json"
    if traffic_file.exists():
        try:
            roofline["traffic"] = json.loads(traffic_file.read_text()).get(names[dom])
        except (ValueError, OSError):
            pass
    ms_e2e_step = ms_e2e / args.steps
    e2e = {"value": clips / (ms_e2e_step / 1e3), "unit": "clips/s", "ms_per_step": ms_e2e_step,
           "h2d_bytes_per_step": int(B * N_MELS * T_FRAMES * 4), "d2h_bytes_per_step": int(B * L_WAVE * 4),
           "api": "SpectrogramConverter.waveform_from_mel_amplitudes (pinned host mel in, pinned host waveform out)"}
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        r = time_reference(3, 1, cores)
        cpu_baseline = {"value": r["value"], "unit": "clips/s", "cores": r["cores"], "kind": "reference",
                        "sample": r["sample"]}
    line = {
        "metric": "clips/sec", "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "clocks": clocks,
        # kernels per step of the hybrid loop: one iSTFT launch per pass, two assembly launches (one on the last, full-rate
        # pass), edge + half-rate STFT launches, plus envelope, inverse mel and the angle gather
        "e2e": e2e, "gpu_launches": int((launches[0] + 2 * launches[1] - 1 + 2 * launches[2] + 3) * args.steps),
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
    }
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


# =============================================================================== clip workload
UNET_TFLOP_PER_SAMPLE = 0.803     # SURVEY 8(a) b-4: 401.6 GMAC per sample-forward
VAE_DEC_TFLOP = 2.515


def tensor_peaks() -> dict:
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return {"burst": float(d["bf16_tflops"]), "sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "source": "measured"}
    return {"burst": 1590.0, "sustained": 1400.0, "source": "fallback"}


def time_reference_clip(host_cores: int, budget_s: float = 25.0) -> dict:
    """CPU baseline for the clip workload on a bounded sample: the reference's arithmetic for one clip is
    n_evals x (CFG UNet forward, fp32 on CPU as riffusion_pipeline.py:88-90 forces) + VAE decode + torchaudio
    inverse-mel/Griffin-Lim.  diffusers is not installable, so the UNet/VAE are the torch-eager restatement
    (oracle/unet_oracle.py, kind = "port"); ONE CFG UNet evaluation and the torchaudio audio path are timed and the
    per-clip time is n_evals * t_unet + t_audio (the VAE decode, ~3 % of the FLOPs, is extrapolated from the UNet
    rate) — stated in `sample`."""
    from oracle import unet_oracle as uo

    with torch.no_grad():
        unet = uo.init_weights_(uo.UNet2DConditionOracle()).eval()
        x = torch.randn(2, 4, 64, 64)
        ctx = torch.randn(2, 77, 768)
        t_unet, threads = None, None
        for th in sorted({min(host_cores, 32), host_cores}):      # fastest of 32 threads and all cores (BASELINE.md 4)
            torch.set_num_threads(th)
            t0 = time.perf_counter()
            unet(x, 741, ctx)
            dt = time.perf_counter() - t0
            if t_unet is None or dt < t_unet:
                t_unet, threads = dt, th
    audio = time_reference(1, 1, host_cores)
    return {"t_unet_cfg_eval_s": t_unet, "t_audio_s": audio["seconds_per_clip"], "threads": threads,
            "audio_threads": audio["cores"]}


def clip_config(n_steps: int, n_evals: int, clips_per_gpu: int, workload: str = "clip", denoising: float = 1.0) -> dict:
    """`config` of the clip-type workloads: shared by the B200 arm and the reference arm (the driver compares them)"""
    if workload == "roundtrip":
        name = (f"configs[4] audio->image->audio round trip: STFT + mel + uint8 image of {L_WAVE}-sample waveforms, VAE encode, "
                f"{n_steps}-step img2img (denoising 1.0 -> {n_evals} CFG UNet evaluations, guidance 7, PNDM), VAE decode, image->mel + "
                f"inverse-mel + Griffin-Lim {N_ITER} it -> int16, 512x512, {clips_per_gpu} clips per GPU per step")
    elif workload == "riffuse":
        name = (f"configs[2] RiffusionPipeline.riffuse(): one request, seed image og_beat 512x512, alpha 0.5, {n_steps} scheduler steps, "
                f"denoising {denoising} -> {n_evals} CFG UNet evaluations, guidance 7, PIL image in -> PIL image out")
    else:
        name = (f"full clip: {n_steps}-step img2img (denoising 1.0 -> {n_evals} CFG UNet evaluations, guidance 7, PNDM) + VAE "
                f"decode + image->mel + inverse-mel + Griffin-Lim {N_ITER} it, 512x512, {clips_per_gpu} clips per GPU per step")
    return {"workload": name,
            "includes_denoise": True, "n_unet_evals": n_evals, "weights": "random-init SD-1.5 (N(0,0.02^2)), broadcast from rank 0 at init",
            "clips_per_gpu": clips_per_gpu, "cuda_graph": True,
            "l2": "UNet weights 1.7 GB + activations larger than L2; no explicit flush",
            "sharding": "independent clips per rank; NCCL broadcast of weights at init only"}


VAE_ENC_TFLOP = 1.117            # SURVEY 8(a): VAE encoder, 512x512 image


def n_evals_for(n_steps: int, denoising: float) -> int:
    """UNet evaluations of the reference's img2img loop (riffusion_pipeline.py:358-396, PNDM table, steps_offset 1)"""
    init = min(int(n_steps * denoising) + 1, n_steps)
    return (n_steps + 1) - max(n_steps - init + 1, 0)


def main_clip_reference(args) -> None:
    """`--impl reference`: the reference's CPU arithmetic for one unit of the workload on the host cores.  diffusers is not
    installable here, so the UNet / VAE are the torch-eager fp32 restatement (oracle/unet_oracle.py: kind "port");
    torchaudio is the reference's own audio path.  Each step is a bounded sample: ONE CFG UNet evaluation (+ one clip of
    torchaudio inverse-mel + Griffin-Lim, + one forward STFT/mel for the round trip), extrapolated to the workload's n_evals
    evaluations and its VAE passes at the UNet's measured FLOP rate (stated in `sample`)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import unet_oracle as uo
    from oracle.torchaudio_ref import TorchaudioConverter

    cores = os.cpu_count() or 1
    wl = args.workload
    n_evals = n_evals_for(args.evals, args.denoising) if wl == "riffuse" else args.evals
    steps = max(1, min(args.steps, 20))
    warm = max(0, min(args.warmup, 1))
    audio = time_reference(1, 1, cores)                  # picks the fastest thread count for torch's CPU FFT path
    audio_threads = audio["cores"]
    # UNet leg: the fastest of 32 threads and all cores (BASELINE.md 4 asks for all host cores; torch's CPU conv does not
    # always scale past a socket) — one evaluation each, then the timed steps with the winner
    conv = TorchaudioConverter(n_iter=N_ITER)
    mel = synthetic_mel(1, seed=0)
    wave = torch.randn(1, L_WAVE) * 3000.0
    with torch.no_grad():
        unet = uo.init_weights_(uo.UNet2DConditionOracle()).eval()
        x, ctx = torch.randn(2, 4, 64, 64), torch.randn(2, 77, 768)
        cand = sorted({min(cores, 32), cores})
        best = None
        for th in cand:
            torch.set_num_threads(th)
            t0 = time.perf_counter()
            unet(x, 741, ctx)
            dt = time.perf_counter() - t0
            if best is None or dt < best[1]:
                best = (th, dt)
        unet_threads = best[0]
        t_unet = t_audio = t_fwd = 0.0
        for it in range(warm + steps):
            torch.set_num_threads(unet_threads)
            t0 = time.perf_counter()
            unet(x, 741, ctx)
            t1 = time.perf_counter()
            torch.set_num_threads(audio_threads)
            if wl != "riffuse":
                conv.waveform_from_mel_amplitudes(mel)
            t2 = time.perf_counter()
            if wl == "roundtrip":
                conv.mel_amplitudes_from_waveform(wave)
            t3 = time.perf_counter()
            if it >= warm:
                t_unet += t1 - t0
                t_audio += t2 - t1
                t_fwd += t3 - t2
    t_unet /= steps
    t_audio /= steps
    t_fwd /= steps
    vae_tflop = VAE_DEC_TFLOP + (VAE_ENC_TFLOP if wl in ("riffuse", "roundtrip") else 0.0)
    sec = n_evals * t_unet * (1 + vae_tflop / (n_evals * 2 * UNET_TFLOP_PER_SAMPLE)) + t_audio + t_fwd
    value = 1.0 / sec
    sample = (f"{steps} x [1 CFG UNet evaluation ({t_unet:.1f} s, torch-eager fp32 restatement, {unet_threads} threads = fastest of "
              f"{cand}) extrapolated to {n_evals} evals + VAE {'encode + ' if vae_tflop > VAE_DEC_TFLOP else ''}decode at the same FLOP rate"
              + (f", plus 1 clip of torchaudio inverse-mel + Griffin-Lim ({t_audio:.1f} s, {audio_threads} threads)" if wl != "riffuse" else "")
              + (f", plus 1 forward STFT + mel ({t_fwd:.2f} s)" if wl == "roundtrip" else "") + f"]; host has {cores} cores")
    line = {"impl": "reference", "metric": "clips/sec", "value": value, "unit": "clips/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": clip_config(args.evals, n_evals, 1 if wl == "riffuse" else args.clips, wl, args.denoising),
            "cpu_baseline": {"value": value, "unit": "clips/s", "cores": unet_threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def load_frozen_weights(rank: int, dist, dev):
    """random-init SD-1.5 UNet + VAE state dicts (BASELINE config 4): created on rank 0, broadcast ONCE as two flat NCCL
    buffers through the library helper (riffusion/distributed.py) — the only collective of a run."""
    from riffusion import sd15_spec
    from riffusion.distributed import broadcast_state_dict

    out = []
    for spec, seed in ((sd15_spec.unet_spec(), 0), (sd15_spec.vae_spec(), 1)):
        sd = {k: v.to(dev) for k, v in sd15_spec.random_state_dict(spec, seed).items()} if rank == 0 else None
        if dist is not None:
            sd = broadcast_state_dict(spec, sd, src=0, device=dev)
        out.append(sd)
    return out


def main_clip(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = os.cpu_count() or 1
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    from riffusion import _native, sd15_spec, tc_ops
    from riffusion.riffusion_pipeline import RiffusionPipeline, VAE_SCALE
    from riffusion.spectrogram_converter import SpectrogramConverter
    from riffusion.spectrogram_params import SpectrogramParams
    from riffusion.unet_b200 import UNetB200
    from riffusion.vae_b200 import VaeB200

    lib = _native.lib()
    # frozen weights: created on rank 0 and broadcast once over NCCL (init only; no collective in the step loop)
    unet_sd, vae_sd = load_frozen_weights(rank, dist, dev)
    pipe = RiffusionPipeline(vae=VaeB200(vae_sd, device=str(dev)), unet=UNetB200(unet_sd, device=str(dev)), device=str(dev))
    del unet_sd, vae_sd
    params = SpectrogramParams()
    conv = SpectrogramConverter(params, device=str(dev))

    B, n_steps = args.clips, args.evals
    roundtrip = args.workload == "roundtrip"
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    text = torch.randn((B, 77, 768), generator=g, device=dev, dtype=torch.float16)      # SURVEY 8(d) config 4: N(0,1) embeddings
    uncond = torch.randn((1, 77, 768), generator=g, device=dev, dtype=torch.float16)
    seed_rgb = torch.from_numpy(np.load(ROOT / "tests" / "golden" / "og_beat.npz")["rgb"].copy())   # (512,512,3) u8
    seed_host = seed_rgb.pin_memory()
    text_host, uncond_host = text.cpu().pin_memory(), uncond.cpu().pin_memory()
    alphas = torch.linspace(0, 1, B).tolist()
    img = (seed_rgb.to(dev).permute(2, 0, 1)[None].half() / 255.0) * 2 - 1
    mean, logvar = pipe.vae.encode_moments(img)                                          # cacheable per seed image
    std = torch.exp(0.5 * logvar.float().clamp(-30, 20))

    def make_inputs(mean_=None, std_=None):
        """per-request tensors the reference draws from its generators: posterior noise + noise_a/noise_b -> slerp.
        mean_/std_: per-clip posterior moments (B,4,64,64) of the round-trip workload, else the cached seed-image moments"""
        lat, nas, nbs = [], [], []
        shape = mean.shape
        for i in range(B):
            ga = torch.Generator(device=dev).manual_seed(i + 1000 * rank)
            gb = torch.Generator(device=dev).manual_seed(10_000 + i + 1000 * rank)
            eps = torch.randn(shape, generator=ga, device=dev)
            m_i = mean.float() if mean_ is None else mean_[i:i + 1].float()
            s_i = std if std_ is None else std_[i:i + 1]
            lat.append((VAE_SCALE * (m_i + s_i * eps)).half())
            nas.append(torch.randn(shape, generator=ga, device=dev, dtype=torch.float16))
            nbs.append(torch.randn(shape, generator=gb, device=dev, dtype=torch.float16))
        noise = tc_ops.slerp(alphas, torch.cat(nas), torch.cat(nbs))       # per-request slerp on the device (rf_slerp_f16)
        return torch.cat(lat), noise

    lat0, noise0 = make_inputs()
    # round trip (configs[4]): int16-scaled band-limited noise of exactly 512 frames per clip (SURVEY 8d config 5)
    waves_host = wave_dev = None
    if roundtrip:
        from riffusion.util import image_util

        gw = torch.Generator().manual_seed(77 + rank)
        w = torch.randn((B, L_WAVE + 16), generator=gw)
        w = torch.nn.functional.avg_pool1d(w[:, None], 9, stride=1, padding=4)[:, 0, : L_WAVE] * 9000.0
        waves_host = w.contiguous().pin_memory()
        wave_dev = waves_host.to(dev)

        def audio_to_latents(wav):
            """waveform -> mel (rf_stft_mel) -> uint8 spectrogram image (rf_mel_to_image, per-clip max) -> VAE posterior"""
            mel_in = conv.mel_amplitudes_from_waveform(wav)                          # (B, 512, 512)
            imgs = torch.stack([image_util.image_from_spectrogram_device(mel_in[i:i + 1], power=0.25)[0] for i in range(B)])
            x = (imgs.permute(0, 3, 1, 2).half() / 255.0) * 2 - 1                  # preprocess_image (:439-452)
            m_, lv_ = pipe.vae.encode_moments(x)
            return make_inputs(m_, torch.exp(0.5 * lv_.float().clamp(-30, 20)))
    F = 8821
    torch.manual_seed(rank)
    angles = torch.rand((B, F, T_FRAMES), dtype=torch.complex64, device=dev)
    pcm_host = torch.empty((B, L_WAVE), dtype=torch.int16).pin_memory()
    img_host = torch.empty((B, 512, 512, 3), dtype=torch.uint8).pin_memory()
    stream = torch.cuda.current_stream(dev)

    def step_device():
        if roundtrip:
            lat, nz = audio_to_latents(wave_dev)
            return pipe.generate_clips(text, uncond, lat, nz, 1.0, n_steps, 7.0, conv, init_angles=angles)
        return pipe.generate_clips(text, uncond, lat0, noise0, 1.0, n_steps, 7.0, conv, init_angles=angles)

    def step_e2e():
        # host buffers in: seed image + text embeddings; out: uint8 image + int16 pcm
        t_emb = text_host.to(dev, non_blocking=True)
        u_emb = uncond_host.to(dev, non_blocking=True)
        if roundtrip:
            lat, nz = audio_to_latents(waves_host.to(dev, non_blocking=True))
        else:
            rgb = seed_host.to(dev, non_blocking=True)
            im = (rgb.permute(2, 0, 1)[None].half() / 255.0) * 2 - 1
            m_, lv_ = pipe.vae.encode_moments(im)            # the reference re-encodes the seed image on every request
            lat, nz = make_inputs()
        out = pipe.generate_clips(t_emb, u_emb, lat, nz, 1.0, n_steps, 7.0, conv)      # random GL phases like the reference
        w = out["waveform"]
        pcm = torch.empty((B, L_WAVE), dtype=torch.int16, device=dev)
        scratch = torch.zeros(1, dtype=torch.float32, device=dev)
        for i in range(B):                               # per-clip peak normalisation (audio_util.py:24)
            _native.check(lib.rf_wave_to_int16(w[i].data_ptr(), 1, L_WAVE, 1, pcm[i].data_ptr(), scratch.data_ptr(),
                                               stream.cuda_stream))
        pcm_host.copy_(pcm, non_blocking=True)
        img_host.copy_(out["images"], non_blocking=True)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """milliseconds of `steps` calls of fn, and what the last call returned"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = None
        for _ in range(steps):
            out = fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    warm = max(args.warmup, 3)
    for _ in range(warm):
        out = step_device()
    n_evals = out["n_unet_evals"]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total, out = timed(step_device, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v for k, v in out.items() if isinstance(v, torch.Tensor)})
    step_e2e()
    e2e_steps = min(args.steps, 5)       # the e2e loop repeats the whole step with host I/O: bounded so a large --steps stays within minutes
    ms_e2e, _ = timed(step_e2e, e2e_steps)

    # live tensor-core measurement: one eager (non-graph) step with CUDA events around every tcgen05 launch
    pipe.use_cuda_graph = False
    step_device()
    lib.rf_tc_profile_begin()
    step_device()
    tc_ms, tc_fl, tc_n = ctypes.c_double(), ctypes.c_double(), ctypes.c_long()
    lib.rf_tc_profile_end(ctypes.byref(tc_ms), ctypes.byref(tc_fl), ctypes.byref(tc_n))
    pipe.use_cuda_graph = True
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    ms_step = ms_total / args.steps
    clips = B * world
    value = clips / (ms_step / 1e3)
    pk = tensor_peaks()
    achieved = tc_fl.value / (tc_ms.value / 1e3) / 1e12
    alg_tflop_step = B * (n_evals * 2 * UNET_TFLOP_PER_SAMPLE + VAE_DEC_TFLOP + (VAE_ENC_TFLOP if roundtrip else 0.0))
    roofline = {
        "bound": "tensor", "kernel": "k_tc_gemm (tcgen05 GEMM / implicit-GEMM conv)", "achieved": achieved,
        "peak": pk["sustained"], "unit": "TFLOP/s", "frac": achieved / pk["sustained"], "traffic": gemm_traffic(),
        "traffic_detail": gemm_traffic(detail=True),
        "peak_source": pk["source"] + " (sustained cuBLAS bf16: kernel timed inside a long step)",
        "kernel_ms_per_step": tc_ms.value, "kernel_launches_per_step": tc_n.value,
        "kernel_flops_per_step": tc_fl.value, "kernel_share_of_step": tc_ms.value / ms_step,
        "note": "kernel time and FLOPs (2MNK, true extents, fused-attention MMAs not included) measured live with "
                "CUDA events around every launch of one eager step; share is vs the CUDA-graph step",
        "step": {"algorithmic_tflop": alg_tflop_step, "achieved": alg_tflop_step / (ms_step / 1e3),
                 "frac": alg_tflop_step / (ms_step / 1e3) / pk["sustained"], "unit": "TFLOP/s",
                 "formula": "B*(n_evals*2*0.803 + 2.515" + (" + 1.117" if roundtrip else "") + ") TFLOP (SURVEY 8d)"},
    }
    ms_e2e_step = ms_e2e / e2e_steps
    e2e = {"value": clips / (ms_e2e_step / 1e3), "unit": "clips/s", "ms_per_step": ms_e2e_step,
           "h2d_bytes_per_step": int((waves_host.numel() * 4 if roundtrip else seed_host.numel()) + text_host.numel() * 2 +
                                     uncond_host.numel() * 2),
           "d2h_bytes_per_step": int(pcm_host.numel() * 2 + img_host.numel()),
           "steps": e2e_steps,
           "api": ("SpectrogramConverter.mel_amplitudes_from_waveform + image_from_spectrogram_device + " if roundtrip else "") +
                  "VaeB200.encode_moments + RiffusionPipeline.generate_clips + rf_wave_to_int16: pinned host " +
                  ("waveforms" if roundtrip else "seed image") + " and text embeddings in, uint8 images and int16 PCM out"}
    # Griffin-Lim sub-benchmark (BASELINE configs[1]) in a child process so that its memory does not add to ours
    gl = None
    cpu_baseline = None
    if world == 1 and not roundtrip:
        try:
            r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "gl", "--steps", "5", "--warmup", "3",
                                "--no-cpu-baseline"], capture_output=True, text=True, timeout=600)
            gl_line = json.loads(r.stdout.strip().splitlines()[-1])
            gl = {"value": gl_line["value"], "unit": gl_line["unit"], "ms_per_step": gl_line["ms_per_step"],
                  "workload": gl_line["config"]["workload"], "roofline": gl_line["roofline"], "e2e": gl_line["e2e"]}
        except Exception as exc:  # noqa: BLE001
            gl = {"error": repr(exc)}
    if world == 1:
        if not args.no_cpu_baseline:
            r = time_reference_clip(cores)
            vae_tf = VAE_DEC_TFLOP + (VAE_ENC_TFLOP if roundtrip else 0.0)
            per_clip = n_evals * r["t_unet_cfg_eval_s"] * (1 + vae_tf / (n_evals * 2 * UNET_TFLOP_PER_SAMPLE)) + r["t_audio_s"]
            cpu_baseline = {"value": 1.0 / per_clip, "unit": "clips/s", "cores": r["threads"], "kind": "port",
                            "sample": f"1 CFG UNet evaluation ({r['t_unet_cfg_eval_s']:.1f} s, torch-eager fp32 restatement, "
                                      f"{r['threads']} threads) extrapolated to {n_evals} evals + VAE decode at the same FLOP rate, plus 1 clip of "
                                      f"torchaudio inverse-mel + Griffin-Lim ({r['t_audio_s']:.1f} s, {r['audio_threads']} threads); host has {cores} cores"}
    config = clip_config(n_steps, n_evals, B, args.workload)
    line = {
        "metric": "clips/sec", "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
        "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e,
        "gpu_launches": int(args.steps * (n_evals * 442 + 400)), "roofline": roofline, "cpu_baseline": cpu_baseline,
        "griffinlim": gl,
    }
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


class _BenchTokenizer:
    """whitespace tokenizer stand-in (no CLIP vocabulary files offline); ids feed the random-init text encoder"""
    model_max_length = 77
    bos_token_id = 49406
    eos_token_id = 49407

    def __call__(self, text, padding=None, max_length=None, truncation=False, return_tensors=None):
        import types
        import zlib

        single = isinstance(text, str)
        rows = []
        for t in ([text] if single else text):
            ids = [self.bos_token_id] + [1 + zlib.crc32(w.lower().encode()) % 49000 for w in t.split()] + [self.eos_token_id]
            if truncation and max_length and len(ids) > max_length:
                ids = ids[: max_length - 1] + [self.eos_token_id]
            if padding == "max_length":
                ids = ids + [self.eos_token_id] * (max_length - len(ids))
            rows.append(ids)
        if return_tensors == "pt":
            return types.SimpleNamespace(input_ids=torch.tensor(rows, dtype=torch.long))
        return types.SimpleNamespace(input_ids=rows[0] if single else rows)


def main_riffuse(args) -> None:
    """BASELINE configs[2]: one request through RiffusionPipeline.riffuse() — PIL seed image in, PIL image out, alpha 0.5,
    50 scheduler steps; `--denoising 0.75` (the reference default: 38 CFG evaluations) or 1.0 (50).  Each rank serves its own
    request (weak scaling).  value = requests/s with the seed image's VAE moments cached and latents resident (the loop +
    decode + uint8); e2e = riffuse() itself, PIL -> PIL (host image in, VAE encode on a cache miss excluded by the moment
    cache exactly as in serving, uint8 image back to the host)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    from PIL import Image

    from riffusion import _native, sd15_spec
    from riffusion.clip_b200 import ClipTextB200
    from riffusion.datatypes import InferenceInput, PromptInput
    from riffusion.riffusion_pipeline import RiffusionPipeline
    from riffusion.unet_b200 import UNetB200
    from riffusion.vae_b200 import VaeB200

    lib = _native.lib()
    unet_sd, vae_sd = load_frozen_weights(rank, dist, dev)
    text_encoder = ClipTextB200.random_init(seed=2, device=str(dev))
    pipe = RiffusionPipeline(vae=VaeB200(vae_sd, device=str(dev)), unet=UNetB200(unet_sd, device=str(dev)),
                             text_encoder=text_encoder, tokenizer=_BenchTokenizer(), device=str(dev))
    del unet_sd, vae_sd
    rgb = np.load(ROOT / "tests" / "golden" / "og_beat.npz")["rgb"]
    init_image = Image.fromarray(rgb, mode="RGB")
    n_steps = args.evals
    n_evals = n_evals_for(n_steps, args.denoising)

    def request(i: int) -> InferenceInput:
        return InferenceInput(alpha=0.5, num_inference_steps=n_steps, seed_image_id="og_beat",
                              start=PromptInput(prompt="church bells on sunday", seed=42 + i + 1000 * rank, denoising=args.denoising),
                              end=PromptInput(prompt="jazz with piano", seed=123 + i + 1000 * rank, denoising=args.denoising))

    stream = torch.cuda.current_stream(dev)
    counter = [0]

    def step_e2e():
        counter[0] += 1
        return pipe.riffuse(request(counter[0]), init_image)

    # device-resident variant: embeddings + latents prepared once, the timed part is loop + decode + uint8 on the device
    inp = request(0)
    e0, e1 = pipe.embed_text_weighted(inp.start.prompt), pipe.embed_text_weighted(inp.end.prompt)
    text = (e0 + 0.5 * (e1 - e0)).half()
    lat0 = pipe.encode_image(init_image, torch.Generator(device=dev).manual_seed(42))
    noise0 = torch.randn(lat0.shape, generator=torch.Generator(device=dev).manual_seed(7), device=dev, dtype=torch.float16)
    uncond = pipe.embed_text("").half()

    def step_device():
        from riffusion import tc_ops

        out = pipe.interpolate_img2img(text_embeddings=text, init_latents=lat0, generator_a=None, generator_b=None,
                                       interpolate_alpha=0.0, strength_a=args.denoising, strength_b=args.denoising,
                                       num_inference_steps=n_steps, guidance_scale=7.0, uncond_embeddings=uncond, noise=noise0,
                                       output_type="latent")
        return tc_ops.vae_image_to_u8(pipe.vae.decode(out["latents"]).sample), out["n_unet_evals"]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """milliseconds of `steps` calls of fn, and what the last call returned"""
        barrier()
        e0_, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0_.record(stream)
        out = None
        for _ in range(steps):
            out = fn()
        e1_.record(stream)
        barrier()
        ms = torch.tensor([e0_.elapsed_time(e1_)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    warm = max(args.warmup, 3)
    for _ in range(warm):
        _, got_evals = step_device()
    assert got_evals == n_evals, (got_evals, n_evals)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total, (image_u8, _) = timed(step_device, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"images": image_u8})
    step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    pipe.use_cuda_graph = False
    step_device()
    lib.rf_tc_profile_begin()
    step_device()
    tc_ms, tc_fl, tc_n = ctypes.c_double(), ctypes.c_double(), ctypes.c_long()
    lib.rf_tc_profile_end(ctypes.byref(tc_ms), ctypes.byref(tc_fl), ctypes.byref(tc_n))
    pipe.use_cuda_graph = True
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    ms_step, ms_e2e_step = ms_total / args.steps, ms_e2e / args.steps
    pk = tensor_peaks()
    achieved = tc_fl.value / (tc_ms.value / 1e3) / 1e12
    alg = n_evals * 2 * UNET_TFLOP_PER_SAMPLE + VAE_DEC_TFLOP
    roofline = {"bound": "tensor", "kernel": "k_tc_gemm (tcgen05 GEMM / implicit-GEMM conv)", "achieved": achieved,
                "peak": pk["sustained"], "unit": "TFLOP/s", "frac": achieved / pk["sustained"], "traffic": gemm_traffic(),
                "peak_source": pk["source"] + " (sustained cuBLAS bf16)", "kernel_ms_per_step": tc_ms.value,
                "kernel_launches_per_step": tc_n.value, "kernel_share_of_step": tc_ms.value / ms_step,
                "note": "batch 2 (one CFG pair): sub-wave problems, split-K on the 8x8 / 16x16 levels",
                "step": {"algorithmic_tflop": alg, "achieved": alg / (ms_step / 1e3), "frac": alg / (ms_step / 1e3) / pk["sustained"],
                         "unit": "TFLOP/s"}}
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        r = time_reference_clip(os.cpu_count() or 1)
        per = n_evals * r["t_unet_cfg_eval_s"] * (1 + (VAE_DEC_TFLOP + VAE_ENC_TFLOP) / (n_evals * 2 * UNET_TFLOP_PER_SAMPLE))
        cpu_baseline = {"value": 1.0 / per, "unit": "clips/s", "cores": r["threads"], "kind": "port",
                        "sample": f"1 CFG UNet evaluation ({r['t_unet_cfg_eval_s']:.1f} s, torch-eager fp32 restatement, {r['threads']} "
                                  f"threads) extrapolated to {n_evals} evals + VAE encode + decode at the same FLOP rate"}
    line = {"metric": "clips/sec", "value": world / (ms_step / 1e3), "unit": "clips/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_step, "latency_ms": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": clip_config(n_steps, n_evals, 1, "riffuse", args.denoising), "clocks": clocks,
            "e2e": {"value": world / (ms_e2e_step / 1e3), "unit": "clips/s", "ms_per_step": ms_e2e_step, "latency_ms": ms_e2e_step,
                    "h2d_bytes_per_step": int(rgb.size + 2 * 77 * 4), "d2h_bytes_per_step": int(512 * 512 * 3),
                    "api": "RiffusionPipeline.riffuse(InferenceInput, PIL.Image) -> PIL.Image (tokenise + CLIP text encoder "
                           "(lru-cached per prompt), cached VAE moments of the seed image, generator draws, loop, decode, uint8)"},
            "gpu_launches": int(args.steps * (n_evals * 460 + 250)), "roofline": roofline, "cpu_baseline": cpu_baseline}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def gemm_traffic(detail: bool = False):
    """ncu dram__bytes_read + dram__bytes_write of the tensor-core kernel, average per launch over the 236 launches of one
    CFG evaluation at the benchmarked batch (profiles/traffic_latest.json, from profiles/r02_eval32_launches_dram.csv);
    detail=True: the whole record (bytes per evaluation, algorithmic bytes)"""
    f = ROOT / "profiles" / "traffic_latest.json"
    try:
        rec = json.loads(f.read_text()).get("k_tc_gemm")
    except (OSError, ValueError):
        return None
    if not isinstance(rec, dict):
        return rec
    return rec if detail else rec.get("dram_bytes_per_launch_avg")


if __name__ == "__main__":
    main()
