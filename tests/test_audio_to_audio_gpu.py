"""Audio to audio on the B200: rf_resample_u8 against Pillow, the uint8 -> fp16 input conversion against
`preprocess_image(...).half()`, rf_add_noise_f16_seq against torch's own fp16 op sequence, the img2img loop against the
fp32 oracle loop and its fp16-storage emulation (tests/img2img_oracle.py), CUDA-graph replay, clip batching,
`audio_to_audio_clips` against the host PIL path, and the `riffusion.audio_to_audio` command end to end on a small
random-init pipeline."""
import numpy as np
import pytest
import torch
from PIL import Image

pytestmark = pytest.mark.gpu

DPM = "DPMSolverMultistepScheduler"
WIDTHS = [(301, 320), (401, 416), (501, 512), (601, 608), (701, 704), (1001, 1024)]


def rel_l2(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm())


def _check_vs_floor(got, ref32, emul, what, floor_factor=1.25):
    """tests/test_parity_bench_gpu.py's bars: kernels vs fp32 oracle within floor_factor x the fp16-storage floor
    (emulation vs fp32), kernels vs emulation within 1.25 x the spread of two independent fp16 evaluations"""
    e_k, e_f, e_o = rel_l2(got, emul), rel_l2(emul, ref32), rel_l2(got, ref32)
    print(f"{what}: kernels vs fp32 oracle {e_o:.3e} | fp16-storage floor (emulation vs fp32) {e_f:.3e} | "
          f"kernels vs emulation {e_k:.3e}")
    assert torch.isfinite(got.float()).all()
    assert e_o <= floor_factor * e_f + 1e-4, f"{what}: kernels vs fp32 {e_o:.3e}, floor {e_f:.3e}"
    spread = 2 ** 0.5 * floor_factor * e_f
    assert e_k <= 1.25 * spread + 1e-4, f"{what}: kernels vs emulation {e_k:.3e}, spread {spread:.3e}"


@pytest.fixture(scope="module", autouse=True)
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


def _round_params(m):
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(p.half().float())
    return m


@pytest.fixture(scope="module")
def sd15(native_lib):
    from oracle import unet_oracle as uo
    from riffusion.unet_b200 import UNetB200

    oracle = _round_params(uo.init_weights_(uo.UNet2DConditionOracle(), seed=0)).cuda().eval()
    return oracle, UNetB200(oracle.state_dict(), device="cuda")


@pytest.fixture(scope="module")
def small_unet(native_lib):
    from oracle import unet_oracle as uo
    from riffusion.unet_b200 import UNetB200

    cfg = dict(block_out_channels=(64, 128, 128, 128), heads=4, cross_attention_dim=64)
    oracle = _round_params(uo.init_weights_(uo.UNet2DConditionOracle(**cfg), seed=21)).cuda().eval()
    return oracle, UNetB200(oracle.state_dict(), device="cuda", block_out_channels=cfg["block_out_channels"], heads=4)


@pytest.fixture(scope="module")
def vae_pair(native_lib):
    from oracle.unet_oracle import init_weights_
    from oracle.vae_oracle import AutoencoderKLOracle
    from riffusion.vae_b200 import VaeB200

    oracle = _round_params(init_weights_(AutoencoderKLOracle(), seed=5, std=0.03)).cuda().eval()
    return oracle, VaeB200(oracle.state_dict(), device="cuda")


class _StubTextEncoder:
    def __init__(self, dim=64):
        g = torch.Generator().manual_seed(123)
        self.table = torch.randn(49408, dim, generator=g).cuda()
        self.pos = torch.randn(77, dim, generator=g).cuda() * 0.3

    def __call__(self, ids):
        return ((self.table[ids.cuda()] + self.pos[None]).half(),)


def _small_pipe(small_unet, vae_pair):
    import sys
    from pathlib import Path

    from riffusion.riffusion_pipeline import RiffusionPipeline

    sys.path.insert(0, str(Path(__file__).parent / "golden"))
    from prompt_stub import StubTokenizer

    return RiffusionPipeline(vae=vae_pair[1], unet=small_unet[1], text_encoder=_StubTextEncoder(), tokenizer=StubTokenizer(),
                             device="cuda")


def _spectrogram_like(rng, B, H, W):
    """smooth dark images with bright streaks, like spectrogram images, plus full-range noise in a corner"""
    y = np.linspace(0, 1, H)[:, None]
    x = np.linspace(0, 1, W)[None, :]
    out = []
    for _ in range(B):
        base = 255 * np.clip(np.sin(rng.uniform(5, 40) * x) * np.cos(rng.uniform(5, 60) * y), 0, 1) ** 3
        img = np.repeat(base[..., None], 3, axis=2).astype(np.uint8)
        img[: H // 8, : W // 8] = rng.integers(0, 256, (H // 8, W // 8, 3))
        out.append(img)
    return np.stack(out)


# ----------------------------------------------------------------------------------------------- kernels
def test_resample_u8_equals_pillow(native_lib):
    from riffusion import tc_ops as ops

    rng = np.random.default_rng(0)
    for w_in, w_up in WIDTHS:
        a = _spectrogram_like(rng, 3, 512, w_in)
        up = ops.resample_u8(torch.from_numpy(a).cuda(), 512, w_up).cpu().numpy()
        want_up = np.stack([np.asarray(Image.fromarray(im).resize((w_up, 512), Image.BICUBIC)) for im in a])
        down = ops.resample_u8(torch.from_numpy(want_up).cuda(), 512, w_in).cpu().numpy()
        want_down = np.stack([np.asarray(Image.fromarray(im).resize((w_in, 512), Image.BICUBIC)) for im in want_up])
        bad_up, bad_down = int((up != want_up).sum()), int((down != want_down).sum())
        print(f"rf_resample_u8 3 x 512 x {w_in} -> {w_up} -> {w_in}: {bad_up} / {bad_down} bytes differ from Pillow")
        assert bad_up == 0 and bad_down == 0
    a = rng.integers(0, 256, (2, 500, 301, 3), dtype=np.uint8)        # both passes, and the same-size copy
    for w, h in ((320, 512), (301, 250), (301, 500)):
        got = ops.resample_u8(torch.from_numpy(a).cuda(), h, w).cpu().numpy()
        want = np.stack([np.asarray(Image.fromarray(im).resize((w, h), Image.BICUBIC)) for im in a])
        assert np.array_equal(got, want), (w, h)


def test_image_u8_to_f16_equals_preprocess(native_lib):
    from riffusion import tc_ops as ops
    from riffusion.riffusion_pipeline import preprocess_image

    rng = np.random.default_rng(1)
    a = rng.integers(0, 256, (2, 512, 512, 3), dtype=np.uint8)
    a[0, 0, :256, 0] = np.arange(256)
    got = ops.image_u8_to_f16(torch.from_numpy(a).cuda())
    want = torch.cat([preprocess_image(Image.fromarray(im)).half() for im in a]).cuda()
    assert got.shape == want.shape and torch.equal(got.view(torch.int16), want.view(torch.int16))


@torch.no_grad()
def test_add_noise_f16_seq_bit_exact_vs_torch_ops(native_lib):
    from riffusion import tc_ops as ops
    from riffusion.scheduler_b200 import DPMSolverMultistepSchedulerB200

    s = DPMSolverMultistepSchedulerB200()
    ac = s.alphas_cumprod.to("cuda", torch.float16)                   # add_noise: alphas_cumprod.to(sample dtype)
    torch.manual_seed(2)
    for n in (4 * 64 * 64 * 3, 4 * 64 * 63 + 5):
        x = (torch.randn(n, device="cuda") * 2).half()
        nz = torch.randn(n, device="cuda").half()
        for t in (999, 559, 519, 40, 0):
            tt = torch.tensor([t], device="cuda")
            want = (ac[tt] ** 0.5) * x + ((1 - ac[tt]) ** 0.5) * nz
            got = s.add_noise_fp16(x, nz, t)
            bad = int((got.view(torch.int16) != want.view(torch.int16)).sum())
            once = ops.axpby(x, nz, float(s.alphas_cumprod[t]) ** 0.5, (1 - float(s.alphas_cumprod[t])) ** 0.5)
            print(f"rf_add_noise_f16_seq n={n} t={t}: {bad} differing elements; single-rounding axpby differs in "
                  f"{int((once != want).sum())}")
            assert bad == 0


# ----------------------------------------------------------------------------------------------- loop parity
def _img2img_case(oracle, unet, vae, scheduler, steps, strength, width, ctx_dim, seed):
    from oracle import unet_oracle as uo
    from img2img_oracle import img2img_loop, img2img_loop_emul
    from riffusion import tc_ops as ops
    from riffusion.riffusion_pipeline import VAE_SCALE, RiffusionPipeline
    from riffusion.scheduler_b200 import get_scheduler
    from riffusion.vae_b200 import _Posterior
    from txt2img_oracle import DPMSolverMultistepSchedulerOracle

    pipe = RiffusionPipeline(vae=vae, unet=unet, device="cuda")
    rng = np.random.default_rng(seed)
    u8 = torch.from_numpy(_spectrogram_like(rng, 1, 512, width)).cuda()
    torch.manual_seed(seed)
    text = torch.randn(1, 77, ctx_dim, device="cuda").half()
    uncond = torch.randn(1, 77, ctx_dim, device="cuda").half()
    out = pipe.img2img(init_images_u8=u8, seed=seed, strength=strength, num_inference_steps=steps, guidance_scale=7.0,
                       scheduler=scheduler, text_embeddings=text, uncond_embeddings=uncond, output_type="latent")
    sched = get_scheduler(scheduler)
    t_start, ts, t_noise = sched.img2img_timesteps(steps, strength)
    mean, logvar = vae.encode_moments(ops.image_u8_to_f16(u8))
    g = torch.Generator(device="cuda").manual_seed(seed)
    lat = VAE_SCALE * _Posterior(mean, logvar).sample(generator=g)
    x0 = sched.add_noise_fp16(lat, torch.randn(lat.shape, generator=g, device="cuda", dtype=torch.float16), t_noise)
    sch = DPMSolverMultistepSchedulerOracle() if scheduler == DPM else uo.PNDMSchedulerOracle()
    ref, n = img2img_loop(oracle, sch, text.float(), uncond.float(), x0.float(), steps, t_start, 7.0)
    emul, n2 = img2img_loop_emul(oracle, scheduler, text, uncond, x0, steps, t_start, 7.0)
    assert out["n_unet_evals"] == n == n2 == len(ts)
    return pipe, out, ref, emul, dict(init_images_u8=u8, seed=seed, strength=strength, num_inference_steps=steps,
                                      guidance_scale=7.0, scheduler=scheduler, text_embeddings=text,
                                      uncond_embeddings=uncond, output_type="latent")


@torch.no_grad()
def test_img2img_small_unet_25_dpm_steps_and_graph_replay(small_unet, vae_pair):
    oracle, unet = small_unet
    pipe, out, ref, emul, kw = _img2img_case(oracle, unet, vae_pair[1], DPM, 25, 0.55, 512, 64, 25)
    assert out["n_unet_evals"] == 13
    _check_vs_floor(out["latents_unscaled"], ref, emul, "img2img small UNet 64x64 latents, 25 DPM steps, strength 0.55")
    pipe.use_cuda_graph = False
    eager = pipe.img2img(**kw)
    assert torch.equal(eager["latents_unscaled"], out["latents_unscaled"]), "CUDA-graph replay differs from eager"


@torch.no_grad()
def test_img2img_small_unet_50_pndm_steps(small_unet, vae_pair):
    oracle, unet = small_unet
    _, out, ref, emul, _ = _img2img_case(oracle, unet, vae_pair[1], "PNDMScheduler", 50, 0.75, 704, 64, 50)
    assert out["n_unet_evals"] == 38
    _check_vs_floor(out["latents_unscaled"], ref, emul, "img2img small UNet 64x88 latents, 50 PNDM steps, strength 0.75")


@torch.no_grad()
def test_img2img_full_size_dpm(sd15, vae_pair):
    oracle, unet = sd15
    _, out, ref, emul, _ = _img2img_case(oracle, unet, vae_pair[1], DPM, 25, 0.55, 512, 768, 7)
    _check_vs_floor(out["latents_unscaled"], ref, emul, "img2img SD-1.5 64x64 latents, 25 DPM steps, strength 0.55")


@torch.no_grad()
def test_img2img_clip_batch_equals_single_calls(small_unet, vae_pair):
    pipe = _small_pipe(small_unet, vae_pair)
    rng = np.random.default_rng(3)
    u8 = torch.from_numpy(_spectrogram_like(rng, 3, 512, 512)).cuda()
    kw = dict(strength=0.55, num_inference_steps=25, guidance_scale=7.0, negative_prompt="drums")
    batch = pipe.img2img("church bells", init_images_u8=u8, seed=42, **kw)
    for i in range(3):
        single = pipe.img2img("church bells", init_images_u8=u8[i:i + 1], seed=42, **kw)
        e = rel_l2(batch["latents_unscaled"][i], single["latents_unscaled"][0])
        d = np.abs(np.array(batch["images"][i]).astype(np.int16) - np.array(single["images"][0]).astype(np.int16))
        print(f"img2img clip batch, clip {i}: latents vs single call rel L2 {e:.2e}; image mean |diff| {d.mean():.4f} LSB, "
              f"max {d.max()}, within 1 LSB {100 * (d <= 1).mean():.2f} %")
        assert e < 5e-3 and d.mean() < 0.25 and (d <= 1).mean() >= 0.98
    pil = pipe.img2img("church bells", init_image=[Image.fromarray(im) for im in u8.cpu().numpy()], seed=42, **kw)
    assert torch.equal(pil["latents_unscaled"], batch["latents_unscaled"]), "PIL input and uint8 input differ"


# ----------------------------------------------------------------------------------------------- audio chain
@torch.no_grad()
def test_audio_to_audio_clips_equals_host_pil_path(small_unet, vae_pair):
    """device chain vs the reference's per-clip chain on the host (32-stride PIL resize -> img2img PIL output -> PIL resize
    back), same seed, so the same latents: identical uint8 images; the waveform against torchaudio on our uint8 image"""
    from oracle import audio_oracle as ao
    from oracle.torchaudio_ref import TorchaudioConverter
    from riffusion.spectrogram_converter import SpectrogramConverter, mel_filterbank
    from riffusion.spectrogram_params import SpectrogramParams

    pipe = _small_pipe(small_unet, vae_pair)
    conv = SpectrogramConverter(SpectrogramParams(), device="cuda")
    g = torch.Generator(device="cuda").manual_seed(11)
    t = torch.arange(220500, device="cuda") / 44100.0
    waves = torch.stack([8000 * torch.sin(2 * np.pi * f * t) * torch.sin(2 * np.pi * 0.7 * t) for f in (220.0, 523.0)])
    waves = (waves + 500 * torch.randn(waves.shape, generator=g, device="cuda")).round()
    angles = torch.rand(2, 8821, 501, dtype=torch.complex64, device="cuda")
    kw = dict(seed=7, strength=0.55, num_inference_steps=10, guidance_scale=7.0)
    out = pipe.audio_to_audio_clips(waves, converter=conv, prompt="jazz", init_angles=angles, **kw)
    src, u8, wave = out["source_images"], out["images"], out["waveform"]
    assert src.shape == u8.shape == (2, 512, 501, 3) and wave.shape == (2, 441 * 500) and out["n_unet_evals"] == 5
    srcn = src.cpu().numpy()
    host = pipe.img2img("jazz", init_image=[Image.fromarray(im).resize((512, 512), Image.BICUBIC) for im in srcn], **kw)
    assert torch.equal(host["latents_unscaled"], out["latents_unscaled"])
    want = np.stack([np.asarray(im.resize((501, 512), Image.BICUBIC)) for im in host["images"]])
    assert np.array_equal(u8.cpu().numpy(), want)
    u8n = u8.cpu().numpy()
    mel_ref = np.concatenate([ao.spectrogram_from_image_array(u8n[i], power=0.25, stereo=False, max_value=30e6)
                              for i in range(2)])
    wave_ref = TorchaudioConverter().waveform_from_mel_amplitudes(torch.from_numpy(mel_ref), angles.cpu())
    w = wave.cpu()

    def nrms(a, b):
        return float((((a - b) / b.abs().amax(dim=-1, keepdim=True)) ** 2).mean().sqrt())

    rms = nrms(w, wave_ref)
    print(f"audio_to_audio_clips: waveform vs torchaudio on our uint8 image: normalised RMS {rms:.3e}")
    if rms >= 1e-4:            # ill-conditioned Griffin-Lim input: the fp64 recurrence referees (test_parity_bench_gpu)
        fb = mel_filterbank(8821, 0.0, 10000.0, 512, 44100).numpy()
        o64 = torch.from_numpy(ao.waveform_from_mel_amplitudes(mel_ref[:1], fb, 17640, 441, ao.hann_window(4410).double().numpy(),
                                                               32, angles[:1].cpu().numpy())).float()
        e_ta, e_us = nrms(wave_ref[:1], o64), nrms(w[:1], o64)
        print(f"audio_to_audio_clips: vs the fp64 recurrence: torchaudio {e_ta:.3e}, kernels {e_us:.3e}")
        assert e_us <= max(2 * e_ta, 2e-5)


def test_audio_to_audio_command_end_to_end(small_unet, vae_pair, tmp_path, monkeypatch):
    from scipy.io import wavfile

    from riffusion import audio_to_audio
    from riffusion.riffusion_pipeline import RiffusionPipeline
    from riffusion.spectrogram_params import SpectrogramParams

    pipe = _small_pipe(small_unet, vae_pair)
    monkeypatch.setattr(RiffusionPipeline, "load_checkpoint", classmethod(lambda cls, *a, **k: pipe))
    rng = np.random.default_rng(5)
    tt = np.arange(int(10.2 * 44100)) / 44100.0
    track = 6000 * np.sin(2 * np.pi * 330 * tt)[:, None] + rng.normal(0, 300, (tt.size, 2))
    wavfile.write(tmp_path / "in.wav", 44100, track.astype(np.int16))
    for extra, name in (([], "a2a"), (["--prompt-b", "rock", "--seed-b", "3", "--denoising-b", "0.6"], "interp")):
        out = tmp_path / f"{name}.wav"
        audio_to_audio.main(["audio-to-audio", "--audio", str(tmp_path / "in.wav"), "--prompt", "jazz", "--output",
                             str(out), "--num-inference-steps", "6", "--image-dir", str(tmp_path / name)] + extra)
        rate, data = wavfile.read(out)
        print(f"audio-to-audio {name}: {data.shape[0] / rate:.4f} s, peak {np.abs(data).max()}")
        assert rate == 44100 and data.ndim == 1 and data.shape[0] == 2 * 220500 - 8820
        assert np.abs(data).max() > 1000
        for i in range(2):
            for kind in ("source", "riffed"):
                img = Image.open(tmp_path / name / f"clip_{i}_{kind}.png")
                assert img.size == (501, 512)
                assert SpectrogramParams.from_exif(img.getexif()).max_frequency == 10000
